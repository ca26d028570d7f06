"""The C++ host program (rsicnv_b200/bin/rsicnv): BGZF/BAM decoding and argument handling without a GPU;
with a GPU, the whole CLI against the unmodified reference CLI on the same files (tables must be identical
apart from the `#input` line, which echoes the path)."""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

from bind import REF_BAMTOOL, REF_BIN, have_ref
from rsicnv_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rsicnv_b200", "bin", "rsicnv")
FIELDS = (("pos", np.int32), ("mpos", np.int32), ("isize", np.int32), ("mtid", np.int32), ("flag", np.uint16), ("mapq", np.uint8),
          ("cigar_off", np.uint32), ("cigar", np.uint32), ("qual_off", np.uint64), ("qual", np.uint8))


@pytest.fixture(scope="module")
def cli():
    if not os.path.exists(CLI):
        subprocess.run(["make", "-s", "cli"], cwd=ROOT, check=True)
    return CLI


def test_bam_decoder_round_trip(cli, tmp_path):
    r1, _ = synth.make_reads(400_000, 3, None, coverage=6, n_events=0, tid=0)
    r2, _ = synth.make_reads(500_000, 4, None, coverage=3, n_events=0, tid=1, frac_indel=0.3)
    bam = str(tmp_path / "t.bam")
    synth.write_bam(bam, [("1", 400_000), ("2", 500_000), ("MT", 1000)], {0: r1, 1: r2})
    for name, want in (("1", r1), ("2", r2)):
        out = subprocess.run([cli, "decode", "-b", bam, "-c", name, "-o", str(tmp_path / "d")], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        for f, dt in FIELDS:
            assert np.array_equal(np.fromfile(str(tmp_path / ("d." + f)), dtype=dt), want[f]), (name, f)
    out = subprocess.run([cli, "decode", "-b", bam, "-c", "7", "-o", str(tmp_path / "d")], capture_output=True, text=True)
    assert out.returncode != 0 and "doesn't have 7" in out.stderr


def test_argument_errors(cli, tmp_path):
    for args, msg in ((["rsi"], "need input file"), (["rsi", "-b", "x.bam"], "need reference file"), (["rsi", "-d", "x.rd", "-f", "x.fa"], "must be specified together"),
                      (["rsi", "-b", "x.bam", "-f", "x.fa", "-bogus"], "unknown option -bogus"), (["plot", "-b", "x.bam"], "no such function")):
        out = subprocess.run([cli] + args, capture_output=True, text=True)
        assert msg in out.stderr, (args, out.stderr)


def _table(path):
    return [ln for ln in open(path).read().splitlines() if not ln.startswith("#input")]


def log_lines(path, outname):
    """<out>.log without what no other implementation can reproduce: the Vm* lines of /proc/<pid>/status and the command line
    (it names the binary); the output file's name is normalised"""
    out = []
    for ln in open(path, newline="\n").read().split("\n"):
        if ln.startswith("Vm") or ln.startswith("#command:"):
            continue
        out.append(ln.replace(outname, "OUT"))
    return out


@pytest.mark.gpu
def test_cli_bam_two_contigs_matches_reference(cli, tmp_path):
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    L1, L2 = 10_600_000, 10_450_000
    fa1 = synth.make_fasta(L1, 3); fa2 = synth.make_fasta(L2, 4)
    r1, _ = synth.make_reads(L1, 3, fa1, coverage=12, n_events=6, lens=(3000, 8000, 20000), tid=0)
    r2, _ = synth.make_reads(L2, 4, fa2, coverage=10, n_events=5, lens=(3000, 8000, 20000), tid=1)
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_bam(bam, [("1", L1), ("2", L2), ("MT", 16569), ("GL000207.1", 4262)], {0: r1, 1: r2})
    synth.write_fasta_multi(fasta, [("1", fa1), ("2", fa2)])
    subprocess.run([REF_BAMTOOL, "index", bam], check=True)
    common = ["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"]
    subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / "ref.txt")], check=True, capture_output=True)
    out = subprocess.run([cli] + common + ["-gpus", "2", "-o", str(tmp_path / "ours.txt")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert _table(str(tmp_path / "ours.txt")) == _table(str(tmp_path / "ref.txt")), out.stderr
    assert len(_table(str(tmp_path / "ours.txt"))) > 6
    # <out>.log: parameter echo, BAM header check, per contig the loaders' and the detector's lines (per-L DEL-/DUP+ counts, level table ...)
    assert log_lines(str(tmp_path / "ours.txt.log"), str(tmp_path / "ours.txt")) == log_lines(str(tmp_path / "ref.txt.log"), str(tmp_path / "ref.txt"))
    # the host decoder (zlib on threads) instead of the GPU one: same table
    out = subprocess.run([cli] + common + ["-hostdecode", "-o", str(tmp_path / "ours_h.txt")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert _table(str(tmp_path / "ours_h.txt")) == _table(str(tmp_path / "ref.txt"))
    # one chromosome only, other knobs
    common = ["rsi", "-b", bam, "-f", fasta, "-c", "2", "-m", "51", "-NOGC", "-MED", "-np"]
    subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / "ref2.txt")], check=True, capture_output=True)
    out = subprocess.run([cli] + common + ["-o", str(tmp_path / "ours2.txt")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert _table(str(tmp_path / "ours2.txt")) == _table(str(tmp_path / "ref2.txt"))
    assert log_lines(str(tmp_path / "ours2.txt.log"), str(tmp_path / "ours2.txt")) == log_lines(str(tmp_path / "ref2.txt.log"), str(tmp_path / "ref2.txt"))
    common = ["rsi", "-b", bam, "-f", fasta, "-c", "1", "-ALL", "-q", "0", "-Q", "10", "-np"]
    subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / "ref3.txt")], check=True, capture_output=True)
    out = subprocess.run([cli] + common + ["-o", str(tmp_path / "ours3.txt")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert _table(str(tmp_path / "ours3.txt")) == _table(str(tmp_path / "ref3.txt"))
    assert log_lines(str(tmp_path / "ours3.txt.log"), str(tmp_path / "ours3.txt")) == log_lines(str(tmp_path / "ref3.txt.log"), str(tmp_path / "ref3.txt"))


@pytest.mark.gpu
def test_cli_depth_file_matches_reference(cli, tmp_path):
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    L = 3_000_017
    fa = synth.make_fasta(L, 5)
    d, _ = synth.make_depth(L, 5, fa, n_events=12, lens=(2000, 5000, 10000, 30000))
    fasta = str(tmp_path / "c.fa"); rd = str(tmp_path / "c.rd")
    synth.write_fasta(fasta, "19", fa)
    synth.write_depth_file(rd, d)
    with open(rd, "a") as f:
        f.write("# a comment\n\n12\tjunk\nnot a number\n")     # parser corner cases of loaddata.cpp:506-517
    common = ["rsi", "-d", rd, "-c", "19", "-f", fasta, "-m", "101", "-np"]
    subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / "ref.txt")], check=True, capture_output=True)
    out = subprocess.run([cli] + common + ["-o", str(tmp_path / "ours.txt")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert open(str(tmp_path / "ours.txt")).read() == open(str(tmp_path / "ref.txt")).read()
    assert log_lines(str(tmp_path / "ours.txt.log"), str(tmp_path / "ours.txt")) == log_lines(str(tmp_path / "ref.txt.log"), str(tmp_path / "ref.txt"))


GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_vectors.json")))


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


CLI_FLAGS = {"m": lambda v: ["-m", str(v)], "trans": lambda v: ["-" + v], "gcadjust": lambda v: [] if v else ["-NOGC"],
             "cap": lambda v: ["-cap", str(v)], "merge": lambda v: [] if v else ["-nomerge"]}


@pytest.mark.gpu
@pytest.mark.parametrize("g", GOLD["depth_cases"], ids=lambda g: f"L{g['L']}-s{g['seed']}-{'-'.join(f'{k}{v}' for k, v in g['kw'].items()) or 'default'}")
def test_cli_depth_file_matches_stored_reference_rows(g, cli, tmp_path):
    """the CLI on a depth file of every stored case gives the rows the unmodified reference computed for it
    (tests/golden/reference_vectors.json, tests/golden/make_golden.py)"""
    from common import make_case
    fa, d, _ = make_case(g["L"], g["seed"], stress=g["stress"])
    assert _sha(d) + _sha(fa) == g["input_sha"], "synthetic input generator drifted"
    fasta = str(tmp_path / "c.fa"); rd = str(tmp_path / "c.rd")
    synth.write_fasta(fasta, "19", fa)
    synth.write_depth_file_fast(rd, d)
    flags = [f for k, v in g["kw"].items() for f in CLI_FLAGS[k](v)]
    out = subprocess.run([cli, "rsi", "-d", rd, "-c", "19", "-f", fasta, "-np", "-o", str(tmp_path / "ours.txt")] + flags, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    rows = [ln for ln in _table(str(tmp_path / "ours.txt")) if not ln.startswith("#")]
    assert rows == g["rows"], out.stderr


@pytest.mark.gpu
def test_cli_bam_matches_stored_reference_table(cli, tmp_path):
    """the stored BAM case (the reference CLI's `rsi -b ... -q 0 -Q 10 -np -s` table and the hash of its `-s` depth dump) through the
    CLI on every decode route: per-GPU decoders from the index, one pass without it, host zlib"""
    b = GOLD["bam_case"]
    fa = synth.make_fasta(b["L"], b["seed"])
    reads, _ = synth.make_reads(b["L"], b["seed"], fa, coverage=b["coverage"], n_events=b["n_events"], lens=tuple(b["lens"]))
    assert _sha(reads["pos"]) + _sha(reads["qual"]) == b["reads_sha"], "synthetic read generator drifted"
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_fasta(fasta, "1", fa)
    synth.write_bam(bam, [("1", b["L"])], {0: reads})
    synth.write_bai(bam)
    for extra, env in (([], {}), ([], {"RSICNV_NO_INDEX": "1"}), (["-hostdecode"], {})):
        o = str(tmp_path / "ours.txt")
        out = subprocess.run([cli, "rsi", "-b", bam, "-f", fasta, "-q", str(b["minq"]), "-Q", str(b["min_baseQ"]), "-np", "-s", "-o", o] + extra,
                             capture_output=True, text=True, env=dict(os.environ, **env))
        assert out.returncode == 0, (extra, env, out.stderr)
        assert _table(o) == b["table"], (extra, env, out.stderr)
        a = np.fromfile(o + ".1_rd", dtype=np.int64, sep=" ").reshape(-1, 2)
        rd = np.zeros(b["L"], np.int32); rd[a[:, 0] - 1] = a[:, 1]
        assert _sha(rd) == b["raw_depth_sha"], (extra, env)


def _read_bai(path):
    """per reference ({bin: [(beg, end), ...]}, linear index), and the trailing count of unplaced records (None if absent)"""
    import struct
    ix = open(path, "rb").read()
    assert ix[:4] == b"BAI\x01"
    o = 8; refs = []
    for _ in range(struct.unpack_from("<i", ix, 4)[0]):
        bins = {}
        nbin = struct.unpack_from("<i", ix, o)[0]; o += 4
        for _ in range(nbin):
            b, nc = struct.unpack_from("<Ii", ix, o); o += 8
            bins[b] = [struct.unpack_from("<QQ", ix, o + 16 * i) for i in range(nc)]; o += 16 * nc
        ni = struct.unpack_from("<i", ix, o)[0]; o += 4
        refs.append((bins, list(struct.unpack_from("<%dQ" % ni, ix, o)))); o += 8 * ni
    return refs, (struct.unpack_from("<Q", ix, o)[0] if o + 8 <= len(ix) else None)


def test_write_bai_indexes_every_record(tmp_path):
    """synth.write_bai against the records of the file, walked here independently: every record lies in a chunk of its own bin,
    the linear index never starts past a record of its window, the pseudo-bin holds the reference's file range and mapped /
    unmapped counts, unplaced records are counted; where the reference's samtools is built, its index has the same content"""
    import bisect
    import struct
    import zlib
    r0, _ = synth.make_reads(300_000, 1, None, coverage=6, n_events=0, tid=0)
    r2, _ = synth.make_reads(250_000, 2, None, coverage=5, n_events=0, tid=2, frac_indel=0.3)
    bam = str(tmp_path / "t.bam")
    synth.write_bam(bam, [("1", 300_000), ("2", 1000), ("3", 250_000)], {0: r0, 2: r2}, level=6, rich=5, unmapped_tail=11, block_size=20000)
    synth.write_bai(bam)
    refs, n_no_coor = _read_bai(bam + ".bai")
    raw = open(bam, "rb").read(); dec = b""; fo, ds = [], []
    off = 0
    while off < len(raw):
        xlen = struct.unpack_from("<H", raw, off + 10)[0]; bs = struct.unpack_from("<H", raw, off + 16)[0] + 1
        fo.append(off); ds.append(len(dec)); dec += zlib.decompress(raw[off + 12 + xlen:off + bs - 8], -15); off += bs

    def voff(x):
        k = bisect.bisect_right(ds, x) - 1
        return fo[k] << 16 | (x - ds[k])
    lt = struct.unpack_from("<i", dec, 4)[0]; q = 12 + lt
    for _ in range(struct.unpack_from("<i", dec, 8 + lt)[0]):
        q += 8 + struct.unpack_from("<i", dec, q)[0]
    recs = []
    while q < len(dec):
        bsz, tid, pos, bmn, fnc = struct.unpack_from("<iiiII", dec, q)
        recs.append((tid, pos, bmn >> 16, fnc >> 16, voff(q), voff(q + 4 + bsz))); q += 4 + bsz
    assert len(refs) == 3 and refs[1] == ({}, []) and n_no_coor == 11
    for t, src in ((0, r0), (2, r2)):
        mine = [r for r in recs if r[0] == t]
        assert len(mine) == len(src["pos"])
        bins, lin = refs[t]
        for _, pos, b, flag, a, e in mine:
            assert any(u <= a and e <= v for u, v in bins[b]), (t, pos, b)
            assert lin[pos >> 14] <= a, (t, pos)
        nmap = sum(1 for r in mine if not r[3] & 4)
        assert bins[37450] == [(mine[0][4], mine[-1][5]), (nmap, len(mine) - nmap)]
        assert min(u for b, ch in bins.items() if b != 37450 for u, _ in ch) == mine[0][4]
    if have_ref():
        ours = _read_bai(bam + ".bai")
        subprocess.run([REF_BAMTOOL, "index", bam], check=True)
        assert _read_bai(bam + ".bai") == ours


def test_host_decoder_real_looking_records(cli, tmp_path):
    """the zlib reader on records with names, bases, optional fields and an unmapped tail"""
    r1, _ = synth.make_reads(120_000, 5, None, coverage=6, n_events=0, tid=0)
    bam = str(tmp_path / "t.bam")
    synth.write_bam(bam, [("1", 120_000)], {0: r1}, level=6, rich=3, unmapped_tail=10)
    out = subprocess.run([cli, "decode", "-b", bam, "-c", "1", "-o", str(tmp_path / "d")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    for f, dt in FIELDS:
        assert np.array_equal(np.fromfile(str(tmp_path / ("d." + f)), dtype=dt), r1[f]), f


@pytest.mark.gpu
def test_cli_real_looking_bam_matches_reference(cli, tmp_path):
    """records as real files carry them (names, bases, optional fields, unmapped reads at the end): GPU decode, host decode and
    the unmodified reference CLI give the same table"""
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    L = 10_400_000
    fa = synth.make_fasta(L, 6)
    r, _ = synth.make_reads(L, 6, fa, coverage=12, n_events=5, lens=(3000, 8000, 20000), tid=0)
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_bam(bam, [("7", L), ("MT", 16569)], {0: r}, level=6, rich=11, unmapped_tail=100)
    synth.write_fasta_multi(fasta, [("7", fa)])
    subprocess.run([REF_BAMTOOL, "index", bam], check=True)
    common = ["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"]
    subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / "ref.txt")], check=True, capture_output=True)
    for extra, name in (([], "gpu.txt"), (["-hostdecode"], "host.txt")):
        out = subprocess.run([cli] + common + extra + ["-o", str(tmp_path / name)], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        assert _table(str(tmp_path / name)) == _table(str(tmp_path / "ref.txt")), name
    assert len(_table(str(tmp_path / "ref.txt"))) > 3
    # -s: the per-base depth dump <out>.<chr>_rd (write_rd_to_file, loaddata.cpp:464-470) is byte-identical, and so is the table
    subprocess.run([REF_BIN] + common + ["-s", "-o", str(tmp_path / "refs.txt")], check=True, capture_output=True)
    out = subprocess.run([cli] + common + ["-s", "-o", str(tmp_path / "gpus.txt")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert open(str(tmp_path / "gpus.txt.7_rd"), "rb").read() == open(str(tmp_path / "refs.txt.7_rd"), "rb").read()
    assert _table(str(tmp_path / "gpus.txt")) == _table(str(tmp_path / "refs.txt"))
    assert log_lines(str(tmp_path / "gpus.txt.log"), str(tmp_path / "gpus.txt")) == log_lines(str(tmp_path / "refs.txt.log"), str(tmp_path / "refs.txt"))


@pytest.mark.gpu
def test_cli_six_contigs_streamed(cli, tmp_path):
    """a small 'whole genome': six contigs of different lengths plus MT and an unplaced scaffold, decoded on the GPU in
    chunks that cut through contigs, dealt to the GPUs longest first; rows must come out in header order, equal to the reference's"""
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    lens = [10_900_000, 10_300_000, 10_700_000, 10_250_000, 10_500_000, 10_400_000]
    names = ["1", "2", "3", "4", "X", "Y"]
    fas = [synth.make_fasta(L, 30 + i) for i, L in enumerate(lens)]
    reads = {}
    for i, L in enumerate(lens):
        reads[i], _ = synth.make_reads(L, 30 + i, fas[i], coverage=6, n_events=3, lens=(4000, 9000, 20000), tid=i)
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_bam(bam, [(n, L) for n, L in zip(names, lens)] + [("MT", 16569), ("GL000192.1", 547496)], reads, level=1, rich=23, unmapped_tail=50)
    synth.write_fasta_multi(fasta, list(zip(names, fas)))
    subprocess.run([REF_BAMTOOL, "index", bam], check=True)
    common = ["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"]
    subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / "ref.txt")], check=True, capture_output=True)
    out = subprocess.run([cli] + common + ["-gpus", "8", "-o", str(tmp_path / "ours.txt")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    ours, ref = _table(str(tmp_path / "ours.txt")), _table(str(tmp_path / "ref.txt"))
    assert ours == ref, out.stderr
    assert len({ln.split("\t")[0] for ln in ref if not ln.startswith("#")}) >= 4


@pytest.mark.gpu
def test_cli_explicit_contig_and_decode_paths(cli, tmp_path):
    """-c with a name the default list would skip ("MT", a name with a dot) is processed like any other (rsi.cpp:2137-2143 resets
    the list to the named target); the default run skips both (rsi.cpp:2119-2120).  Every decode route gives the same table:
    per-GPU decoders started from the .bai offsets (default), one sequential pass without the index, host zlib."""
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    lens = [10_350_000, 10_450_000, 10_550_000]
    names = ["1", "MT", "GL000207.1"]
    fas = [synth.make_fasta(L, 60 + i) for i, L in enumerate(lens)]
    reads = {i: synth.make_reads(L, 60 + i, fas[i], coverage=8, n_events=4, lens=(4000, 9000, 20000), tid=i)[0] for i, L in enumerate(lens)}
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_bam(bam, list(zip(names, lens)), reads, level=1, rich=29, unmapped_tail=20)
    synth.write_fasta_multi(fasta, list(zip(names, fas)))
    subprocess.run([REF_BAMTOOL, "index", bam], check=True)
    for k, sel in enumerate((["-c", "MT"], ["-c", "GL000207.1"], [])):
        common = ["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"] + sel
        subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / f"ref{k}.txt")], check=True, capture_output=True)
        ref = _table(str(tmp_path / f"ref{k}.txt"))
        for extra, env in (([], {}), ([], {"RSICNV_NO_INDEX": "1"}), (["-hostdecode"], {}), (["-gpus", "2"], {})):
            out = subprocess.run([cli] + common + extra + ["-o", str(tmp_path / "ours.txt")], capture_output=True, text=True, env=dict(os.environ, **env))
            assert out.returncode == 0, out.stderr
            assert _table(str(tmp_path / "ours.txt")) == ref, (sel, extra, env, out.stderr)
        chroms = {ln.split("\t")[0] for ln in ref if not ln.startswith("#")}
        assert chroms == ({"MT"}, {"GL000207.1"}, {"1"})[k], chroms


@pytest.mark.gpu
def test_cli_corrupt_bam_is_an_error_not_a_table(cli, tmp_path):
    """a deflate stream damaged in the middle of the second contig: the first contig's rows are written, the damaged contig's are NOT
    (no calls from partial depth) and the exit status is non-zero -- on every decode route"""
    lens = [10_300_000, 10_400_000]
    fas = [synth.make_fasta(L, 70 + i) for i, L in enumerate(lens)]
    reads = {i: synth.make_reads(L, 70 + i, fas[i], coverage=8, n_events=4, lens=(4000, 9000, 20000), tid=i)[0] for i, L in enumerate(lens)}
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_bam(bam, [("1", lens[0]), ("2", lens[1])], reads, level=1, random_seq=5)
    synth.write_fasta_multi(fasta, [("1", fas[0]), ("2", fas[1])])
    synth.write_bai(bam)
    good = subprocess.run([cli, "rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np", "-o", str(tmp_path / "good.txt")], capture_output=True, text=True)
    assert good.returncode == 0, good.stderr
    rows = [ln for ln in _table(str(tmp_path / "good.txt")) if not ln.startswith("#")]
    assert {ln.split("\t")[0] for ln in rows} == {"1", "2"}
    data = bytearray(open(bam, "rb").read())
    at = int(len(data) * 0.8)                    # well inside contig 2
    for k in range(64):
        data[at + k] ^= 0x5a
    open(bam, "wb").write(bytes(data))
    for extra, env in (([], {}), ([], {"RSICNV_NO_INDEX": "1"}), (["-hostdecode"], {})):
        out = subprocess.run([cli, "rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np", "-o", str(tmp_path / "bad.txt")] + extra,
                             capture_output=True, text=True, env=dict(os.environ, **env))
        assert out.returncode != 0, (extra, env, out.stderr)
        bad = [ln for ln in _table(str(tmp_path / "bad.txt")) if not ln.startswith("#")]
        first = [ln for ln in rows if ln.split("\t")[0] == "1"]
        if env or extra:   # sequential readers: the chunk / block group that holds the damage may also hold the end of contig 1, which then fails as well
            assert bad in ([], first), (extra, env, out.stderr)
        else:              # per-contig byte ranges from the index: contig 1 is untouched by the damage
            assert bad == first, (extra, env, out.stderr)


def test_header_reader_agrees_with_the_python_one(cli, tmp_path):
    """read_bam_header (what the CLI hands to the GPU decoder) vs api.parse_bam_header: ordinary file, header ending exactly at a
    block boundary, header spanning many blocks"""
    from rsicnv_b200 import api
    r1, _ = synth.make_reads(60_000, 7, None, coverage=3, n_events=0, tid=0)
    text = "@HD\tVN:1.0\tSO:coordinate\n@SQ\tSN:19\tLN:60000\n"
    hdr_len = 12 + len(text) + 4 + len("19") + 1 + 4
    for k, (contigs, bs) in enumerate(([[("19", 60_000)], 65280], [[("19", 60_000)], hdr_len], [[("19", 60_000)] + [("c%d" % i, 1000) for i in range(400)], 211])):
        bam = str(tmp_path / ("t%d.bam" % k))
        synth.write_bam(bam, contigs, {0: r1}, level=6, block_size=bs)
        h = api.parse_bam_header(np.fromfile(bam, np.uint8))
        out = subprocess.run([cli, "decode", "-b", bam, "-c", "19", "-o", str(tmp_path / "d")], capture_output=True, text=True)
        assert out.returncode == 0, out.stderr
        assert "records start at file offset %d + %d decoded bytes, %d references" % (h["coff"], h["skip"], len(contigs)) in out.stdout, out.stdout


@pytest.mark.gpu
def test_cli_stat_matches_reference(cli, tmp_path):
    """`rsicnv stat -b BAM -v CALLS -o OUT` (rsi.cpp:2235-2249): the reference's own table goes in, every call line comes back with
    RP= / Q0= appended; also lines the reader skips (comments, short lines, < 4 fields), and the route without the index"""
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    lens = [10_600_000, 10_450_000]
    fas = [synth.make_fasta(L, 40 + i) for i, L in enumerate(lens)]
    reads = {i: synth.make_reads(L, 40 + i, fas[i], coverage=10, n_events=5, lens=(3000, 8000, 20000), tid=i)[0] for i, L in enumerate(lens)}
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_bam(bam, [("1", lens[0]), ("2", lens[1])], reads, level=1, rich=17, unmapped_tail=10)
    synth.write_fasta_multi(fasta, [("1", fas[0]), ("2", fas[1])])
    subprocess.run([REF_BAMTOOL, "index", bam], check=True)
    subprocess.run([REF_BIN, "rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np", "-o", str(tmp_path / "calls.txt")], check=True, capture_output=True)
    calls = str(tmp_path / "calls.txt")
    with open(calls, "a") as f:
        f.write("# comment\n1 2\n2\t5000000\t5003000\tgain\textra\n1\t7000000\t6990000\tloss\n2 x y\n")
    subprocess.run([REF_BIN, "stat", "-b", bam, "-v", calls, "-o", str(tmp_path / "ref_stat.txt")], check=True, capture_output=True)
    ref = open(str(tmp_path / "ref_stat.txt")).read().splitlines()
    assert len(ref) > 8
    for env in ({}, {"RSICNV_NO_INDEX": "1"}):
        out = subprocess.run([cli, "stat", "-b", bam, "-v", calls, "-o", str(tmp_path / "our_stat.txt")], capture_output=True, text=True, env=dict(os.environ, **env))
        assert out.returncode == 0, out.stderr
        ours = open(str(tmp_path / "our_stat.txt")).read().splitlines()
        assert ours == ref, (env, out.stderr)
