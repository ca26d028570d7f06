"""`rsicnv index`: the BAI index written on the GPU, byte for byte synth.write_bai's; `rsi` and `stat` give the same tables on
it as on write_bai's index and without an index; a corrupt BAM leaves no index behind."""
import os
import subprocess

import numpy as np
import pytest

from bind import REF_BAMTOOL, have_ref
from rsicnv_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rsicnv_b200", "bin", "rsicnv")


@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.run(["make", "-s", "cli"], cwd=ROOT, check=True)
    return CLI


def _table(path):
    return [ln for ln in open(path).read().splitlines() if not ln.startswith("#input")]


def _run(args, env=None):
    return subprocess.run(args, capture_output=True, text=True, env=dict(os.environ, **(env or {})))


def test_index_is_listed_and_needs_a_bam(cli):
    out = _run([cli])
    assert "rsicnv index -b BAM" in out.stderr
    out = _run([cli, "index"])
    assert "need input file" in out.stderr


@pytest.fixture(scope="module")
def two_contigs(tmp_path_factory):
    d = tmp_path_factory.mktemp("ix")
    L1, L2 = 2_400_000, 2_100_000
    fa1 = synth.make_fasta(L1, 61); fa2 = synth.make_fasta(L2, 62)
    r1, _ = synth.make_reads(L1, 61, fa1, coverage=10, n_events=4, lens=(3000, 8000, 20000), tid=0)
    r2, _ = synth.make_reads(L2, 62, fa2, coverage=10, n_events=4, lens=(3000, 8000, 20000), tid=1)
    bam = str(d / "t.bam"); fasta = str(d / "t.fa")
    synth.write_bam(bam, [("1", L1), ("2", L2), ("MT", 16569)], {0: r1, 1: r2}, level=6, block_size=20000, unmapped_tail=9)
    synth.write_fasta_multi(fasta, [("1", fa1), ("2", fa2)])
    synth.write_bai(bam)
    want = open(bam + ".bai", "rb").read()
    os.remove(bam + ".bai")
    return bam, fasta, want


@pytest.mark.gpu
def test_index_bytes_and_tables(cli, two_contigs, tmp_path):
    bam, fasta, want = two_contigs
    out = _run([cli, "index", "-b", bam])
    assert out.returncode == 0, out.stderr
    assert open(bam + ".bai", "rb").read() == want
    out = _run([cli, "index", "-b", bam, "-o", str(tmp_path / "x.bai"), "-crc"])
    assert out.returncode == 0, out.stderr
    assert open(str(tmp_path / "x.bai"), "rb").read() == want
    common = [cli, "rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"]
    tables = {}
    for key, env in (("ours", {}), ("one_pass", {"RSICNV_NO_INDEX": "1"})):
        o = str(tmp_path / f"{key}.txt")
        r = _run(common + ["-o", o], env)
        assert r.returncode == 0, r.stderr
        tables[key] = _table(o)
    with open(bam + ".bai", "wb") as f:          # write_bai's index in its place: the same table
        f.write(want)
    o = str(tmp_path / "wb.txt")
    r = _run(common + ["-o", o])
    assert r.returncode == 0, r.stderr
    tables["write_bai"] = _table(o)
    assert tables["ours"] == tables["one_pass"] == tables["write_bai"]
    assert len(tables["ours"]) > 2
    # stat with the table as its list of calls: the GPU-built index, write_bai's, none
    calls = str(tmp_path / "ours.txt")
    _run([cli, "index", "-b", bam])
    res = []
    for env in ({}, "write_bai", {"RSICNV_NO_INDEX": "1"}):
        if env == "write_bai":
            with open(bam + ".bai", "wb") as f:
                f.write(want)
            env = {}
        o = str(tmp_path / "stat.txt")
        r = _run([cli, "stat", "-b", bam, "-v", calls, "-o", o], env)
        assert r.returncode == 0, r.stderr
        res.append(open(o).read())
    assert "RP=" in res[0] and res[0] == res[1] == res[2]


@pytest.mark.gpu
def test_corrupt_bam_leaves_no_index(cli, two_contigs, tmp_path):
    bam, _, _ = two_contigs
    data = np.fromfile(bam, np.uint8)
    bad = str(tmp_path / "bad.bam")
    d = data.copy(); d[len(d) // 2] ^= 0xff; d[len(d) // 2 + 7] ^= 0x5a
    d.tofile(bad)
    r = _run([cli, "index", "-b", bad])
    assert r.returncode != 0
    assert not os.path.exists(bad + ".bai")
    assert not [f for f in os.listdir(str(tmp_path)) if ".bai" in f]
    # a file cut in the middle of a block
    cut = str(tmp_path / "cut.bam")
    data[:len(data) // 3].tofile(cut)
    r = _run([cli, "index", "-b", cut])
    assert r.returncode != 0 and not os.path.exists(cut + ".bai")


@pytest.mark.gpu
def test_two_gpus_on_the_gpu_built_index(cli, two_contigs, tmp_path):
    if int(subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.count("GPU ")) < 2:
        pytest.skip("needs two GPUs")
    bam, fasta, _ = two_contigs
    assert _run([cli, "index", "-b", bam]).returncode == 0
    common = [cli, "rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"]
    a = _run(common + ["-o", str(tmp_path / "a.txt")], {"RSICNV_NO_INDEX": "1"})
    b = _run(common + ["-gpus", "2", "-o", str(tmp_path / "b.txt")])
    assert a.returncode == 0 and b.returncode == 0, (a.stderr, b.stderr)
    assert _table(str(tmp_path / "a.txt")) == _table(str(tmp_path / "b.txt"))


@pytest.mark.gpu
def test_same_bytes_as_samtools(cli, tmp_path):
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    L = synth.CHR19_LEN
    reads, _ = synth.make_reads(L, 19, None, coverage=30, n_events=0)
    big = str(tmp_path / "chr19.bam")
    synth.write_bam(big, [("19", L)], {0: reads}, level=1, random_seq=7, threads=32)
    r0, _ = synth.make_reads(300_000, 1, None, coverage=6, n_events=0, tid=0)
    r2, _ = synth.make_reads(250_000, 2, None, coverage=5, n_events=0, tid=2, frac_indel=0.3)
    rich = str(tmp_path / "rich.bam")
    synth.write_bam(rich, [("1", 300_000), ("2", 1000), ("3", 250_000)], {0: r0, 2: r2}, level=6, rich=5, unmapped_tail=11, block_size=20000)
    for bam in (big, rich):
        assert _run([cli, "index", "-b", bam, "-o", bam + ".gpu.bai"]).returncode == 0
        subprocess.run([REF_BAMTOOL, "index", bam], check=True)
        assert open(bam + ".gpu.bai", "rb").read() == open(bam + ".bai", "rb").read(), bam
