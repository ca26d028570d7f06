"""`rsicnv rsi -unsorted` / `rsicnv stat -unsorted`: a BAM in any record order gives what the same file gives through the sorted
route after a stable coordinate sort -- the table, the .log (but for the command echo), the `-s` dumps and the `stat` lines."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from bind import REF_BAMTOOL, REF_BIN
from rsicnv_b200 import api, synth
from test_sim_unsorted import stable_sorted

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rsicnv_b200", "bin", "rsicnv")


@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.run(["make", "-s", "cli"], cwd=ROOT, check=True)
    return CLI


def _rsi(bam, fasta, *extra):
    return ["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np", *extra]


def _run(cli, args, out, env=None):
    return subprocess.run([cli] + args + ["-o", out], capture_output=True, text=True, env=dict(os.environ, **(env or {})))


def _table(path):
    return [ln for ln in open(path).read().splitlines() if not ln.startswith("#input")]


def _log(path):
    """the .log but for the command echo and the input file; the output's directory written as DIR"""
    text = open(path).read().replace(os.path.dirname(path), "DIR")
    return [ln for ln in text.splitlines() if not ln.startswith(("#command:", "#bamfile:"))]


def shuffle_files(d, contigs, reads, seed, n_unplaced=40):
    """every record of `reads` ({tid: position-sorted reads}) shuffled, with unplaced records among them -> (shuffled BAM, the
    same records after a stable coordinate sort written as a sorted BAM)"""
    rng = np.random.default_rng(seed)
    units = [(t, i) for t in reads for i in range(len(reads[t]["pos"]))] + [(-1, 0)] * n_unplaced
    units = [units[i] for i in rng.permutation(len(units))]
    order = np.array([t for t, _ in units])
    file_reads = {t: synth.take_reads(reads[t], np.array([i for u, i in units if u == t])) for t in reads}
    shuffled, srt = str(d / "u.bam"), str(d / "s.bam")
    synth.write_bam_unsorted(shuffled, contigs, file_reads, order, random_seq=seed, threads=32)
    synth.write_bam(srt, contigs, {t: stable_sorted(R) for t, R in file_reads.items()}, random_seq=seed, unmapped_tail=n_unplaced, threads=32)
    return shuffled, srt


def test_unsorted_flag_listed_and_refused_combinations(cli, tmp_path):
    out = subprocess.run([cli], capture_output=True, text=True)
    assert "-unsorted" in out.stderr, out.stderr
    bam, fa, cnv = str(tmp_path / "x.bam"), str(tmp_path / "x.fa"), str(tmp_path / "x.txt")
    for args in (_rsi(bam, fa, "-unsorted", "-split", "2"), _rsi(bam, fa, "-unsorted", "-hostdecode"),
                 ["stat", "-b", bam, "-v", cnv, "-unsorted", "-hostdecode"]):
        r = subprocess.run([cli] + args, capture_output=True, text=True)
        assert r.returncode == 2 and "-unsorted" in r.stderr, (args, r.returncode, r.stderr)


@pytest.fixture(scope="module")
def two_contigs(tmp_path_factory):
    d = tmp_path_factory.mktemp("unsorted")
    contigs = [("1", 4_300_000), ("2", 4_200_000), ("MT", 16_000)]
    fas = {t: synth.make_fasta(contigs[t][1], 60 + t) for t in (0, 1)}
    reads = {t: synth.make_reads(contigs[t][1], 60 + t, fas[t], coverage=8, n_events=4, lens=(4000, 9000, 20000), tid=t)[0] for t in (0, 1)}
    shuffled, srt = shuffle_files(d, contigs, reads, 61)
    fasta = str(d / "t.fa")
    synth.write_fasta_multi(fasta, [("1", fas[0]), ("2", fas[1])])
    return d, shuffled, srt, fasta


def _same_outputs(cli, d, shuffled, srt, fasta, tmp_path, *extra):
    a, b = tmp_path / "a", tmp_path / "b"
    a.mkdir(); b.mkdir()
    ra = _run(cli, _rsi(srt, fasta, "-s", *extra), str(a / "o.txt"))
    rb = _run(cli, _rsi(shuffled, fasta, "-s", "-unsorted", *extra), str(b / "o.txt"))
    assert ra.returncode == 0 and rb.returncode == 0, (ra.stderr, rb.stderr)
    assert _table(str(b / "o.txt")) == _table(str(a / "o.txt")) and len(_table(str(a / "o.txt"))) > 2
    assert _log(str(b / "o.txt.log")) == _log(str(a / "o.txt.log"))
    dumps = sorted(f for f in os.listdir(a) if f.endswith("_rd"))
    assert dumps == sorted(f for f in os.listdir(b) if f.endswith("_rd")) and len(dumps) == 2
    for f in dumps:
        assert open(a / f, "rb").read() == open(b / f, "rb").read(), f
    return str(a / "o.txt")


@pytest.mark.gpu
def test_cli_rsi_unsorted_equals_sorted(cli, two_contigs, tmp_path):
    d, shuffled, srt, fasta = two_contigs
    _same_outputs(cli, d, shuffled, srt, fasta, tmp_path)


@pytest.mark.gpu
def test_cli_rsi_unsorted_two_gpus(cli, two_contigs, tmp_path):
    if api.load_library().rsigpu_num_devices() < 2:
        pytest.skip("one GPU")
    d, shuffled, srt, fasta = two_contigs
    _same_outputs(cli, d, shuffled, srt, fasta, tmp_path, "-gpus", "2")


@pytest.mark.gpu
def test_cli_unsorted_ignores_the_bai_and_needs_the_flag(cli, two_contigs, tmp_path):
    d, shuffled, srt, fasta = two_contigs
    bam = str(tmp_path / "u.bam")
    shutil.copy(shuffled, bam)
    r = _run(cli, _rsi(bam, fasta), str(tmp_path / "plain.txt"))
    assert r.returncode != 0, "an unsorted file without -unsorted must still fail"
    synth.write_bai(srt)
    shutil.copy(srt + ".bai", bam + ".bai")           # an index of another file: -unsorted must not read it
    want = _run(cli, _rsi(srt, fasta), str(tmp_path / "want.txt"))
    got = _run(cli, _rsi(bam, fasta, "-unsorted"), str(tmp_path / "got.txt"))
    os.remove(srt + ".bai")
    assert want.returncode == 0 and got.returncode == 0, (want.stderr, got.stderr)
    assert _table(str(tmp_path / "got.txt")) == _table(str(tmp_path / "want.txt"))


@pytest.mark.gpu
def test_cli_stat_unsorted_equals_sorted(cli, two_contigs, tmp_path):
    d, shuffled, srt, fasta = two_contigs
    calls = str(tmp_path / "calls.txt")
    assert _run(cli, _rsi(srt, fasta), calls).returncode == 0
    ra = _run(cli, ["stat", "-b", srt, "-v", calls], str(tmp_path / "a.stat"))
    rb = _run(cli, ["stat", "-b", shuffled, "-v", calls, "-unsorted"], str(tmp_path / "b.stat"))
    assert ra.returncode == 0 and rb.returncode == 0, (ra.stderr, rb.stderr)
    a, b = open(tmp_path / "a.stat").read(), open(tmp_path / "b.stat").read()
    assert a == b and "RP=" in a


@pytest.mark.gpu
def test_cli_unsorted_many_contigs(cli, tmp_path):
    """a GRCh38-style header: 300 eligible contigs with reads among 2700 names containing '.' (never processed)"""
    n_el, n_dot, L = 300, 2700, 20_000
    contigs, reads, fas = [], {}, []
    for k in range(n_el + n_dot):
        if k % 10 == 3:
            t = len(contigs)
            name = f"c{t}"
            contigs.append((name, L))
            fa = synth.make_fasta(L, 1000 + t)
            fas.append((name, fa))
            reads[t] = synth.make_reads(L, 1000 + t, fa, coverage=12, n_events=0, tid=t)[0]
        else:
            contigs.append((f"chrUn_KI{k}v1.1", 4000 + k))
    assert len(reads) == n_el
    shuffled, srt = shuffle_files(tmp_path, contigs, reads, 62, n_unplaced=100)
    fasta = str(tmp_path / "m.fa")
    synth.write_fasta_multi(fasta, fas)
    (tmp_path / "a").mkdir(); (tmp_path / "b").mkdir()
    ra = _run(cli, _rsi(srt, fasta), str(tmp_path / "a" / "o.txt"))
    rb = _run(cli, _rsi(shuffled, fasta, "-unsorted"), str(tmp_path / "b" / "o.txt"))
    assert rb.returncode == ra.returncode, (ra.stderr[-2000:], rb.stderr[-2000:])
    assert _table(str(tmp_path / "b" / "o.txt")) == _table(str(tmp_path / "a" / "o.txt"))
    assert _log(str(tmp_path / "b" / "o.txt.log")) == _log(str(tmp_path / "a" / "o.txt.log"))
    assert rb.stderr.count("#processing") == n_el


@pytest.mark.gpu
def test_cli_unsorted_chr19_sized(cli, tmp_path):
    """a fully shuffled chr19-sized 30x file: the table is byte-identical to the stably sorted file's"""
    L = synth.CHR19_LEN
    fa = synth.make_fasta(L, 19)
    reads = synth.make_reads(L, 19, fa, coverage=30, n_events=20)[0]
    shuffled, srt = shuffle_files(tmp_path, [("19", L)], {0: reads}, 63, n_unplaced=1000)
    del reads
    fasta = str(tmp_path / "19.fa")
    synth.write_fasta_multi(fasta, [("19", fa)])
    ra = _run(cli, _rsi(srt, fasta), str(tmp_path / "a.txt"))
    rb = _run(cli, _rsi(shuffled, fasta, "-unsorted"), str(tmp_path / "b.txt"))
    assert ra.returncode == 0 and rb.returncode == 0, (ra.stderr[-2000:], rb.stderr[-2000:])
    assert open(tmp_path / "b.txt").read().split("\n", 1)[1] == open(tmp_path / "a.txt").read().split("\n", 1)[1]
    assert len(_table(str(tmp_path / "a.txt"))) > 5


@pytest.mark.gpu
def test_cli_unsorted_against_reference_on_its_own_sort(cli, two_contigs, tmp_path):
    """the unmodified reference CLI on samtools-0.1.18's sort of the shuffled file gives our -unsorted table"""
    if not (os.path.exists(REF_BIN) and os.path.exists(REF_BAMTOOL)):
        pytest.skip("oracle/_ref not built")
    d, shuffled, srt, fasta = two_contigs
    prefix = str(tmp_path / "ref_sorted")
    subprocess.run([REF_BAMTOOL, "sort", shuffled, prefix], check=True, capture_output=True)
    subprocess.run([REF_BAMTOOL, "index", prefix + ".bam"], check=True, capture_output=True)
    subprocess.run([REF_BIN] + _rsi(prefix + ".bam", fasta) + ["-o", str(tmp_path / "ref.txt")], check=True, capture_output=True)
    assert _run(cli, _rsi(shuffled, fasta, "-unsorted"), str(tmp_path / "ours.txt")).returncode == 0
    assert _table(str(tmp_path / "ours.txt")) == _table(str(tmp_path / "ref.txt"))
