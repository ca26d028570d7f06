"""Multi-GPU paths (need >= 2 devices: `gpurun --gpus 2 -- python -m pytest tests/test_gpu_multi.py -m gpu`; skipped on a
one-GPU box).  Contigs are independent units (rsi.cpp:2189-2217), so every multi-GPU run must reproduce the one-GPU table
byte for byte:
  * the C ABI: a decoder context on GPU 0 hands its runs to a contig context on GPU 1 (rsigpu_bam_take across devices);
  * the CLI with `-gpus 2`: per-GPU decoders started from the .bai offsets, and the one-pass route without the index whose
    decoder sits on GPU 0 and feeds the contexts of both GPUs;
  * bench.py's whole-genome workload under torchrun with 2 ranks: same table hash as with 1 rank.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from bind import REF_BIN, have_ref
from rsicnv_b200 import api, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "rsicnv_b200", "bin", "rsicnv")


def _ndev():
    return api.load_library().rsigpu_num_devices()


def _table(path):
    return [ln for ln in open(path).read().splitlines() if not ln.startswith("#input")]


@pytest.fixture(scope="module")
def two_gpus():
    if _ndev() < 2:
        pytest.skip("needs two GPUs")


def test_bam_take_across_gpus(two_gpus, gpu_lib, tmp_path):
    L = 10_400_000
    fa = synth.make_fasta(L, 81)
    reads, _ = synth.make_reads(L, 81, fa, coverage=10, n_events=5, lens=(3000, 8000, 20000))
    bam = str(tmp_path / "t.bam")
    synth.write_bam(bam, [("1", L)], {0: reads}, level=1, random_seq=3)
    data = np.fromfile(bam, np.uint8)
    h = api.parse_bam_header(data)
    outs = []
    for dst_dev in (0, 1):
        with api.Context(device=0, lib=gpu_lib) as dec, api.Context(device=dst_dev, lib=gpu_lib, minq=0, min_baseQ=10) as ctx:
            ctx.set_reference(fa); ctx.pileup_begin()
            dec.bam_begin(1)
            consumed, runs = dec.bam_feed(data[h["coff"]:], skip=h["skip"])
            for i, (tid, n) in enumerate(runs):
                if tid == 0:
                    dec.bam_take(i, ctx)
            dec.bam_end(); ctx.pileup_end()
            raw = ctx.array(api.ARR_RAW_DEPTH).copy()
            calls = ctx.run()
            outs.append((raw.tobytes(), b"".join(bytes(c) for c in calls)))
    assert outs[0] == outs[1] and len(outs[0][1]) > 0


def test_cli_two_gpus_equals_one(two_gpus, tmp_path):
    if not os.path.exists(CLI):
        subprocess.run(["make", "-s", "cli"], cwd=ROOT, check=True)
    lens = [10_900_000, 10_300_000, 10_700_000, 10_250_000]
    names = ["1", "2", "3", "X"]
    fas = [synth.make_fasta(L, 90 + i) for i, L in enumerate(lens)]
    reads = {i: synth.make_reads(L, 90 + i, fas[i], coverage=8, n_events=3, lens=(4000, 9000, 20000), tid=i)[0] for i, L in enumerate(lens)}
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa")
    synth.write_bam(bam, list(zip(names, lens)), reads, level=1, rich=31, unmapped_tail=30)
    synth.write_fasta_multi(fasta, list(zip(names, fas)))
    common = ["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"]
    tables = {}
    synth.write_bai(bam)
    if have_ref():
        subprocess.run([REF_BIN] + common + ["-o", str(tmp_path / "ref.txt")], check=True, capture_output=True)
        tables["reference"] = _table(str(tmp_path / "ref.txt"))
    for key, extra, env in (("1gpu", ["-gpus", "1"], {}), ("2gpu_indexed", ["-gpus", "2"], {}), ("2gpu_one_pass", ["-gpus", "2"], {"RSICNV_NO_INDEX": "1"}),
                            ("2gpu_hostdecode", ["-gpus", "2", "-hostdecode"], {})):
        out = subprocess.run([CLI] + common + extra + ["-o", str(tmp_path / (key + ".txt"))], capture_output=True, text=True, env=dict(os.environ, **env))
        assert out.returncode == 0, (key, out.stderr)
        tables[key] = _table(str(tmp_path / (key + ".txt")))
        if "2gpu" in key:
            assert "on GPU 1" in out.stderr, (key, out.stderr)        # the second GPU really took contigs
    first = tables["1gpu"]
    assert len(first) > 4
    for key, t in tables.items():
        assert t == first, key


def test_bench_whole_genome_two_ranks_same_table(two_gpus, tmp_path):
    """bench.py --workload wg at 1 and 2 ranks (small genome scale): identical table hash, i.e. LPT sharding + the ordered gather
    change nothing"""
    env = dict(os.environ)
    args = ["--workload", "wg", "--genome-scale", "0.05", "--steps", "1", "--warmup", "1", "--no-cli", "--profile-steps", "1"]
    r1 = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, env=env, cwd=ROOT, timeout=900)
    assert r1.returncode == 0, r1.stderr[-2000:]
    r2 = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29571",
                         os.path.join(ROOT, "bench.py"), "--gpus", "2"] + args, capture_output=True, text=True, env=env, cwd=ROOT, timeout=900)
    assert r2.returncode == 0, r2.stderr[-2000:]
    j1 = json.loads([ln for ln in r1.stdout.splitlines() if ln.startswith("{")][-1])
    j2 = json.loads([ln for ln in r2.stdout.splitlines() if ln.startswith("{")][-1])
    assert j1["table_sha1"] == j2["table_sha1"] and j1["calls"] == j2["calls"] and j1["calls"] > 0
    assert j2["n_gpus"] == 2 and j2["scaling"] == "strong"


def _snap(ctx, calls):
    st = ctx.chr_stats()
    return dict(calls=[bytes(c) for c in calls], depth=ctx.array(api.ARR_DEPTH).tobytes(), nbn=ctx.array(api.ARR_BIN_NBN).tobytes(),
                status=ctx.array(api.ARR_BIN_STATUS).tobytes(), stats=(st.rdmedian, st.rdsd, st.rdmad, st.isize_mean, st.isize_sd, st.nbins, st.compact_len))


def test_split_chr1_sized_contig_two_gpus_equals_one(two_gpus, gpu_lib):
    """config 5's building block: a chr1-sized contig (249,250,621 bp) split over two GPUs by base range -- per-base passes on each
    half, integer tables added on the lead over NVLink peer copies, halo of the bins that straddle the cut -- gives the one-GPU
    result bit for bit"""
    L = synth.B37_LENS["1"]
    fa = synth.make_fasta(L, 1)
    d, _ = synth.make_depth(L, 1, fa, n_events=40, lens=(2000, 5000, 10000, 30000, 100000))
    with api.Context(device=0, lib=gpu_lib) as c0:
        c0.set_reference(fa); c0.set_depth(d)
        c0.run()                                   # warm-up (allocations)
        want = _snap(c0, c0.run())
        one_ms = c0.stage_ms()["total"]
    parts = [api.Context(device=g, lib=gpu_lib) for g in range(2)]
    try:
        for p in parts:
            p.set_reference(fa); p.set_depth(d)
        api.split_run(parts)                       # warm-up (allocations)
        got = _snap(parts[0], api.split_run(parts))
        split_ms = parts[0].stage_ms()["total"]
        p2p = parts[0].lib.rsigpu_split_p2p_bytes(parts[0].h)
    finally:
        for p in parts:
            p.close()
    assert got == want and len(want["calls"]) >= 20
    assert p2p > 0.4 * 4 * L          # about half of the compacted depth crosses to the lead, plus tables and bins
    print(f"chr1-sized contig: one GPU {one_ms:.2f} ms, split over two {split_ms:.2f} ms, {p2p / 1e6:.1f} MB peer-to-peer")


def test_split_bam_contig_two_gpus_and_cli(two_gpus, gpu_lib, tmp_path):
    L = 10_600_000
    fa = synth.make_fasta(L, 83)
    reads, _ = synth.make_reads(L, 83, fa, coverage=12, n_events=6, lens=(3000, 8000, 20000))
    kw = dict(minq=0, min_baseQ=10)
    with api.Context(device=0, lib=gpu_lib, **kw) as c0:
        c0.set_reference(fa); c0.pileup_begin(); c0.pileup_push(reads); c0.have_reads()
        want = _snap(c0, c0.run())
    parts = [api.Context(device=g, lib=gpu_lib, **kw) for g in range(2)]
    try:
        for g, p in enumerate(parts):
            b, e, halo = api.split_range(p.lib, L, 2, g)
            p.set_reference(fa); p.pileup_begin(); p.pileup_push(api.split_reads(reads, b, e, halo)); p.have_reads()
        got = _snap(parts[0], api.split_run(parts))
    finally:
        for p in parts:
            p.close()
    assert got == want and len(want["calls"]) >= 3 and any(api.Cnv.from_buffer_copy(c).rp > 0 for c in want["calls"])
    # the CLI: -split 2 against one GPU, BAM and depth-file input
    if not os.path.exists(CLI):
        subprocess.run(["make", "-s", "cli"], cwd=ROOT, check=True)
    bam = str(tmp_path / "t.bam"); fasta = str(tmp_path / "t.fa"); rd = str(tmp_path / "t.rd")
    synth.write_bam(bam, [("7", L)], {0: reads}, level=1, random_seq=9)
    synth.write_fasta(fasta, "7", fa)
    synth.write_bai(bam)
    depth, _ = synth.make_depth(L, 83, fa, n_events=6, lens=(3000, 8000, 20000))
    synth.write_depth_file_fast(rd, depth)
    for common in (["rsi", "-b", bam, "-f", fasta, "-q", "0", "-Q", "10", "-np"], ["rsi", "-d", rd, "-c", "7", "-f", fasta, "-np"]):
        outs = []
        for extra, env in (([], {}), (["-split", "2"], {}), (["-split", "2"], {"RSICNV_NO_INDEX": "1"})):
            o = str(tmp_path / f"o{len(outs)}.txt")
            r = subprocess.run([CLI] + common + extra + ["-o", o], capture_output=True, text=True, env=dict(os.environ, **env))
            assert r.returncode == 0, r.stderr
            outs.append(_table(o))
        assert outs[0] == outs[1] == outs[2] and len(outs[0]) > 3
