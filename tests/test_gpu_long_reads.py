"""The long / spliced / many-op read cases of test_sim_long_reads.py on the B200, plus what only the GPU runs at its size: a
60 Mbp contig with 30x short and 10x long reads (pileup, whole BAM path, decode), records larger than the carry buffer, and
the CLI's raw-depth dump of a long/spliced BAM against the unmodified reference where that is built."""
import os
import subprocess

import numpy as np
import pytest

from bind import REF_BAMTOOL, REF_BIN, have_ref, oracle_pileup
from common import run_bam_case
from rsicnv_b200 import api, synth
from test_sim_bam_decode import assert_same_reads, decode_file
from test_sim_bam_index import build_index, expected
from test_cli import _table
from test_sim_long_reads import (EQ, M, MODES, THRESHOLDS, assert_depth, check_pileup, edge_reads, eq_reach_reads, explicit_reads,
                                 long_and_spliced, long_bam, pileup)  # noqa: F401  (long_bam: the module's BAM fixture)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rsicnv_b200", "bin", "rsicnv")


@THRESHOLDS
@pytest.mark.parametrize("L,n,seed,kw", [(2_000_000, 300, 1, {}), (300_000, 200, 2, dict(max_len=20_000, max_skip=100_000)),
                                         (20_000_000, 3000, 11, {})], ids=["2Mbp", "300kbp-dense", "20Mbp"])
def test_pileup_random_long_reads(gpu_lib, oracle, L, n, seed, kw, minq, Q):
    reads = synth.make_long_reads(L, n, seed, **kw)
    assert check_pileup(gpu_lib, oracle, L, reads, minq, Q, seed).sum() > 0


@THRESHOLDS
@pytest.mark.parametrize("L", [12 * 8192, 12 * 8192 + 77])
def test_pileup_chunk_and_tile_edges(gpu_lib, oracle, L, minq, Q):
    assert check_pileup(gpu_lib, oracle, L, edge_reads(L), minq, Q, 3).sum() > 0


@THRESHOLDS
def test_pileup_reach_of_eq_ops(gpu_lib, oracle, minq, Q):
    L, reads = eq_reach_reads()
    assert check_pileup(gpu_lib, oracle, L, reads, minq, Q, 4)[40_000] > 0


def test_bam_path_with_long_and_spliced_reads(gpu_lib, oracle):
    fa, reads = long_and_spliced(10_600_000, 5)
    calls, st = run_bam_case(gpu_lib, oracle, fa, reads, n_batches=5, minq=0, min_baseQ=13)
    assert len(calls) > 0 and st.isize_mean > 0


@pytest.mark.parametrize("mode", MODES, ids=["lane-per-block", "warp-per-block"])
@pytest.mark.parametrize("chunk", [None, 30_000, 70_001, 1 << 20])
def test_decode_long_records(gpu_lib, long_bam, monkeypatch, mode, chunk):
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    monkeypatch.setenv("RSIGPU_BGZF_CRC", "1" if chunk == 30_000 else "0")
    path, reads = long_bam
    got, _ = decode_file(gpu_lib, path, chunk)
    assert_same_reads(got[0], reads)


@pytest.mark.parametrize("mode", MODES, ids=["lane-per-block", "warp-per-block"])
@pytest.mark.parametrize("chunk,crc", [(None, False), (30_000, False), (70_001, True)])
def test_index_long_records(gpu_lib, long_bam, mode, chunk, crc):
    path, _ = long_bam
    assert build_index(gpu_lib, path, mode, chunk, crc=crc) == expected(path)


def _one_big_record(tmp_path, ops):
    """short reads with one huge record among them (random qualities: the file does not compress, so the record spans many
    1 MiB feeds)"""
    L = 2_000_000
    bg, _ = synth.make_reads(L, 13, None, coverage=1, n_events=0)
    lq = sum(l for l, _ in ops)
    reads = synth.merge_reads(bg, explicit_reads([(1_000_000, ops, np.random.default_rng(1).integers(0, 256, lq), 0, 60)]))
    path = str(tmp_path / "big.bam")
    synth.write_bam(path, [("1", L)], {0: reads}, level=1)
    return path, reads, 4 + 32 + 2 + 4 * len(ops) + (lq + 1) // 2 + lq


@pytest.mark.parametrize("mode", MODES, ids=["lane-per-block", "warp-per-block"])
def test_record_of_16_mib_is_carried_across_many_feeds(gpu_lib, tmp_path, monkeypatch, mode):
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    path, reads, size = _one_big_record(tmp_path, [(5_592_390, M), (5_592_390, M)])
    assert size == 16 << 20
    got, _ = decode_file(gpu_lib, path, 1 << 20)
    assert_same_reads(got[0], reads)


def test_record_over_16_mib_is_refused(gpu_lib, tmp_path):
    path, _, size = _one_big_record(tmp_path, [(7_000_000, M), (7_000_000, EQ)])
    assert size > (16 << 20) + (4 << 20)
    with pytest.raises(api.RsiGpuError) as e:
        decode_file(gpu_lib, path, 1 << 20)
    assert e.value.code == 3 and f"record of {size} bytes" in str(e.value)


# ---- a 60 Mbp contig: 30x short reads and 10x long reads of 10-100 kb
@pytest.fixture(scope="module")
def big_case(tmp_path_factory):
    L = 60_000_000
    fa = synth.make_fasta(L, 17)
    short, _ = synth.make_reads(L, 17, fa, coverage=30, n_events=12, lens=(3000, 8000, 20000, 50000))
    cand = synth.make_long_reads(L, 70_000, 18, max_ops=60, min_len=300, max_len=8000, max_skip=3000, max_other=50)
    ql = np.diff(cand["qual_off"].astype(np.int64))
    keep = np.flatnonzero((ql >= 10_000) & (ql <= 100_000))
    keep = keep[np.cumsum(ql[keep]) <= 10 * L]
    long = synth.take_reads(cand, keep)
    assert int(np.diff(long["qual_off"].astype(np.int64)).sum()) > 9 * L
    reads = synth.merge_reads(short, long)
    path = str(tmp_path_factory.mktemp("big") / "big.bam")
    synth.write_bam(path, [("1", L)], {0: reads}, level=1)
    return fa, reads, path


def test_60mbp_pileup_and_bam_path(gpu_lib, oracle, big_case):
    fa, reads, _ = big_case
    oracle.set_params(minq=1, min_baseQ=20)
    want = oracle_pileup(oracle, reads, len(fa))
    assert_depth(pileup(gpu_lib, fa, reads, 1, 20), want, "60 Mbp")
    calls, st = run_bam_case(gpu_lib, oracle, fa, reads, n_batches=4, minq=0, min_baseQ=13)
    assert len(calls) > 0 and st.isize_mean > 0


@pytest.mark.parametrize("chunk", [None, 1 << 20])
def test_60mbp_decode(gpu_lib, big_case, chunk):
    _, reads, path = big_case
    got, _ = decode_file(gpu_lib, path, chunk)
    assert_same_reads(got[0], reads)


def test_cli_depth_dump_of_long_reads_matches_reference(tmp_path):
    if not have_ref():
        pytest.skip("oracle/_ref not built")
    if not os.path.exists(CLI):
        subprocess.run(["make", "-s", "cli"], cwd=ROOT, check=True)
    fa, reads = long_and_spliced(10_600_000, 5)
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_bam(bam, [("7", len(fa))], {0: reads}, level=1)
    synth.write_fasta_multi(fasta, [("7", fa)])
    subprocess.run([REF_BAMTOOL, "index", bam], check=True)
    common = ["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "13", "-np", "-s"]
    subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / "ref.txt")], check=True, capture_output=True)
    out = subprocess.run([CLI] + common + ["-o", str(tmp_path / "gpu.txt")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert open(str(tmp_path / "gpu.txt.7_rd"), "rb").read() == open(str(tmp_path / "ref.txt.7_rd"), "rb").read()
    assert _table(str(tmp_path / "gpu.txt")) == _table(str(tmp_path / "ref.txt"))
