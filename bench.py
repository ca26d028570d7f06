#!/usr/bin/env python
"""bench.py -- Gbases/s of the B200-native `rsicnv rsi` depth -> CNV-call path.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload wg|chr19_bam|chr19_depth] [--dump-outputs DIR]

Workloads (BASELINE.json configs):
  wg          (default; configs[2]) a b37-shaped genome -- 24 contigs in b37 proportions at --genome-scale (default 1/4: 774 Mbp,
              every contig > 12 Mbp), 30x 2x100 bp read pairs, -q 0 -Q 10 -m 101.  One "step" = the whole genome through the hot
              path.  N GPUs: contigs are dealt to ranks longest first (LPT, rsicnv_b200/shard.py), no data-path collective,
              rows gathered in header order => STRONG scaling (total work fixed).
  chr19_bam   (configs[1]) --inflight independent chr19-shaped contigs (59,128,983 bp, 30x) per GPU and step => weak scaling.
  chr19_depth (configs[0]) the same from a depth array (no pileup).

`value` = reference bases of all contigs processed per second with the inputs already resident in HBM (reads staged in the
contexts; each step = pileup -> GC adjust -> cap -> bins -> RSI scan -> candidates -> RP/Q0 -> calls on the host), wall time of
the K timed steps bracketed by barrier + torch.cuda.synchronize on both sides, max over ranks.  `e2e` = the same work starting
from the BAM FILE's bytes in pinned host memory (H2D + BGZF inflate + record decode on the GPU inside the timed region) through
the C ABI: the rank's contigs go to the decoder in batches of --e2e-batch-mb compressed bytes (rsigpu_bam_feed_parts: the byte
ranges of several contigs inflated by one launch), then every contig is taken and run on its own.  `--impl reference` times the unmodified reference CLI (oracle/_ref/rsicnv, built from /root/reference by
oracle/Makefile.ref) on the box's host cores on a bounded sample of the same workload.

The whole-genome inputs are built from ONE seeded master contig (the longest): contig i is the master truncated to its length
(FASTA prefix, reads that start before L_i - 700), i.e. 24 per-chromosome inputs; the master's BAM image is written with BGZF
blocks that end at record boundaries, so a byte-range prefix of it IS the BAM of the truncated contig (synth.write_bam_aligned).
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from rsicnv_b200 import shard, synth  # noqa: E402

CHR19 = synth.CHR19_LEN
METRIC = "Gbases/s depth->RSI CNV calls"
READ_FIELDS = ("pos", "mpos", "isize", "mtid", "flag", "mapq", "cigar_off", "cigar", "qual_off", "qual")
SEED = 19


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, gpu_index: int):
        self.idx = gpu_index; self.proc = None; self.lines = []

    def start(self):
        q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
            "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True); self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def genome_contigs(scale: float):
    names = list(synth.B37_LENS)
    return names, [int(round(synth.B37_LENS[n] * scale)) for n in names]


# algorithmic HBM bytes of one launch of each streaming kernel (DESIGN.md section 4); L = contig, Lc = after N removal
def kernel_bytes(name: str, L: int, Lc: int, reads_bytes: int = 0, qual_bytes: int = 0):
    name = name.split("<")[0]
    if name == "k_bins_warp":
        name = "k_bins"           # the warp-pipelined form of pass C (bins of <= 127 bases)
    return {
        "k_qual_mask": qual_bytes,        # every base quality once (the 1-bit-per-base mask it writes is overhead, not counted)
        "k_gc_table": 5 * L,          # depth 4 + FASTA 1, read once
        "k_gc_adjust": 9 * L,         # depth 4 + FASTA 1 read, adjusted depth 4 written
        "k_bins": 4 * Lc,             # compacted depth read once
        "k_pileup_tile": reads_bytes - qual_bytes + 4 * L,   # every read record's core fields + CIGAR once + depth written once
    }.get(name, 0)


# DRAM traffic per launch on a chr19-sized contig, from the ncu --set full captures kept under profiles/ (bytes); None = not captured for this build
NCU_TRAFFIC_FILE = os.path.join(ROOT, "profiles", "ncu_traffic.json")


def ncu_traffic():
    try:
        return json.load(open(NCU_TRAFFIC_FILE))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------------------------------
# reference arm (CPU): the unmodified reference on bounded samples of the workload
def ref_worker(args):
    """one reference-CPU process on the depth path: the reference's own functions on an in-memory contig (oracle/_ref/libref_harness.so)"""
    seed, L, kind = args
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from bind import Lib
    fa = synth.make_fasta(L, seed)
    depth, _ = synth.make_depth(L, seed, fa, n_events=20)
    r = Lib(kind); r.set_params()
    t0 = time.perf_counter()
    res = r.depth_path(depth, fa, 3)
    return time.perf_counter() - t0, len(res["calls"])


def ref_bam_worker(args):
    """one reference-CPU process on the BAM path: the UNMODIFIED reference CLI on its own sorted + indexed synthetic BAM"""
    seed, L, workdir = args[:3]
    with_ours = len(args) > 3 and args[3]
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from bind import REF_BAMTOOL, REF_BIN
    d = os.path.join(workdir, f"s{seed}")
    os.makedirs(d, exist_ok=True)
    fa = synth.make_fasta(L, seed)
    reads, _ = synth.make_reads(L, seed, fa, coverage=30.0, n_events=20)
    synth.write_fasta(os.path.join(d, "t.fa"), "19", fa)
    synth.write_bam(os.path.join(d, "t.bam"), [("19", L)], {0: reads})
    subprocess.run([REF_BAMTOOL, "index", os.path.join(d, "t.bam")], check=True)
    t0 = time.perf_counter()
    subprocess.run([REF_BIN, "rsi", "-b", os.path.join(d, "t.bam"), "-f", os.path.join(d, "t.fa"), "-q", "0", "-Q", "10", "-np", "-o", os.path.join(d, "out.txt")],
                   check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    dt = time.perf_counter() - t0
    ncalls = sum(1 for ln in open(os.path.join(d, "out.txt")) if not ln.startswith("#"))
    ours = None
    cli = os.path.join(ROOT, "rsicnv_b200", "bin", "rsicnv")
    if with_ours and os.path.exists(cli):
        # the same files through this repo's CLI; second run = CUDA context and page cache warm
        ts = []; notes = []
        for extra in ([], [], ["-hostdecode"]):
            t0 = time.perf_counter()
            r = subprocess.run([cli, "rsi", "-b", os.path.join(d, "t.bam"), "-f", os.path.join(d, "t.fa"), "-q", "0", "-Q", "10", "-np", "-o", os.path.join(d, "ours.txt")] + extra,
                               check=True, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=dict(os.environ, RSICNV_TIMING="1"))
            ts.append(time.perf_counter() - t0)
            notes += [ln for ln in r.stderr.splitlines() if ln.startswith("#timing")]
        ours = {"first_s": ts[0], "second_s": ts[1], "hostdecode_s": ts[2], "timing": notes,
                "identical_table": [ln for ln in open(os.path.join(d, "ours.txt")) if not ln.startswith("#input")] ==
                                   [ln for ln in open(os.path.join(d, "out.txt")) if not ln.startswith("#input")]}
    return dt, ncalls, ours


def ref_bam_port_worker(args):
    """fallback when oracle/_ref is absent: the oracle restatement of the same path on the read SoA"""
    seed, L = args[:2]
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from bind import Lib, oracle_bam_path
    fa = synth.make_fasta(L, seed)
    reads, _ = synth.make_reads(L, seed, fa, coverage=30.0, n_events=20)
    o = Lib("oracle")
    t0 = time.perf_counter()
    res = oracle_bam_path(o, reads, fa, minq=0, min_baseQ=10)
    return time.perf_counter() - t0, len(res["calls"]), None


def ref_kind():
    """"reference" = the unmodified reference objects built into oracle/_ref; "port" = the oracle restatement"""
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_harness.so")):
        return "ref", "reference"
    if not os.path.exists(os.path.join(ROOT, "oracle", "librsi_oracle.so")):
        subprocess.run(["make", "-s", "oracle"], cwd=ROOT, check=True)
    return "oracle", "port"


def time_reference_bam(sample_len: int, procs: int, seed0: int, with_ours: bool = False):
    import multiprocessing as mp
    import tempfile
    ctx = mp.get_context("spawn")
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "rsicnv"))
    if not have_ref:
        ref_kind()
    with tempfile.TemporaryDirectory() as td, ctx.Pool(procs) as pool:
        out = pool.map(ref_bam_worker if have_ref else ref_bam_port_worker, [(seed0 + i, sample_len, td, with_ours) for i in range(procs)])
    return max(o[0] for o in out), out, ("reference" if have_ref else "port")


def time_reference(sample_len: int, procs: int, seed0: int):
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    lib_kind = ref_kind()[0]
    with ctx.Pool(procs) as pool:
        out = pool.map(ref_worker, [(seed0 + i, sample_len, lib_kind) for i in range(procs)])
    return max(o[0] for o in out), out


def run_reference_arm(a, config, bam):
    procs = min(os.cpu_count() or 1, 32)
    sample = a.cpu_sample
    kind = ref_kind()[1]
    times = []
    for s in range(a.warmup + a.steps):
        if 0 < s < a.warmup:
            continue  # one warm-up pass is enough for a CPU job (page cache / import)
        if bam:
            cpu, out, kind = time_reference_bam(sample, procs, 1000 + 97 * s)
        else:
            cpu, out = time_reference(sample, procs, 1000 + 97 * s)
        if s >= a.warmup:
            times.append((cpu, float(np.mean([o[0] for o in out]))))
    ms = 1e3 * float(np.mean([t[0] for t in times]))
    val = procs * sample / (ms / 1e3) / 1e9
    per_core = sample / float(np.mean([t[1] for t in times])) / 1e9
    what = (f"{procs} processes x one {sample} bp 30x synthetic contig each: BAM + FASTA files through the unmodified `rsicnv rsi -b ... -q 0 -Q 10 -np` CLI "
            f"(BGZF/BAM decode included)" if bam else
            f"{procs} processes x one {sample} bp synthetic contig each through the reference's own checkgccontent..detectcnv..sd_filters "
            f"(in-memory depth array, same boundary as the C ABI; text parsing excluded)")
    cfg = dict(config)
    # the arm runs a BOUNDED SAMPLE of the workload: contigs of `sample` bp (the workload's contigs are 12-62 Mbp at genome scale 1/4), one per host core
    cfg["reference_sample"] = {"contig_bp": sample, "contigs_per_step": procs, "bases_per_step": procs * sample, "same_config": False,
                               "why": "the reference is single-threaded and needs ~290 s per Gbase per core: the whole workload per step would take an hour"}
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "Gbases/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": config["scaling"], "vs_baseline": None, "dtype": "int32/f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": val, "unit": "Gbases/s", "cores": procs, "kind": kind, "sample": what, "per_core_value": per_core},
            "e2e": {"value": val, "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


DUMP_CAP_BYTES = 64 << 20


def dump_outputs(path: str, per_contig: list) -> None:
    """per_contig[i] = (statistics, calls) of contig i in header order -> DIR/contig_<statistic>.npy (one value per contig),
    DIR/call_<field>.npy (one value per call, contigs in header order) and DIR/call_contig.npy (each call's contig index).
    Above DUMP_CAP_BYTES in all, the call files hold a fixed seeded sample of the calls (same rows in every file, in order)."""
    from rsicnv_b200 import api
    os.makedirs(path, exist_ok=True)
    for k in per_contig[0][0]:
        np.save(os.path.join(path, f"contig_{k}.npy"), np.array([s[k] for s, _ in per_contig], np.float64))
    calls = [(i, c) for i, (_, cs) in enumerate(per_contig) for c in cs]
    fields = [n for n, _ in api.Cnv._fields_ if n != "pad_"]
    room = (DUMP_CAP_BYTES - (1 << 16) - 8 * len(per_contig) * len(per_contig[0][0])) // (8 * (len(fields) + 1))
    if len(calls) > room:
        keep = np.sort(np.random.default_rng(0).choice(len(calls), room, replace=False))
        calls = [calls[j] for j in keep]
    np.save(os.path.join(path, "call_contig.npy"), np.array([i for i, _ in calls], np.float64))
    for k in fields:
        np.save(os.path.join(path, f"call_{k}.npy"), np.array([c[k] for _, c in calls], np.float64))


# ------------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="wg", choices=["wg", "chr19_bam", "chr19_depth"])
    ap.add_argument("--genome-scale", type=float, default=0.25, help="wg: contig lengths = b37 lengths x this (1/4 keeps every contig > 12 Mbp)")
    ap.add_argument("--len", type=int, default=CHR19, help="chr19_*: contig length (debug; the contract uses the default)")
    ap.add_argument("--cpu-sample", type=int, default=12_000_000, help="contig length of the bounded CPU-reference sample (> 10 Mbp for the BAM path)")
    ap.add_argument("--profile-steps", type=int, default=2)
    ap.add_argument("--inflight", "--contigs-per-step", type=int, default=4, dest="inflight",
                    help="contigs in flight per GPU (one context + stream + host thread each, as the CLI runs them)")
    ap.add_argument("--e2e-batch-mb", type=int, default=1000, help="e2e leg: compressed MiB of BAM one decoder feed takes (the contigs of a batch are inflated by one launch; "
                                                                      "a feed holds at most 2 GiB compressed and, here, 10 GiB decoded)")
    ap.add_argument("--no-cli", action="store_true", help="skip the CLI / one-core reference comparison at the end (N=1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step of the device-resident leg returned as DIR/<name>.npy "
                                                          "(float64): every call's fields, in header order, and each contig's statistics")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes what this project's path computed: it needs --impl ours")
    rank =int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    bam = a.workload != "chr19_depth"
    K = max(1, a.inflight)
    if a.workload == "wg":
        names, lens = genome_contigs(a.genome_scale)
        scaling = "strong"
        workload = (f"wg (BASELINE.json configs[2]): b37-shaped genome at scale {a.genome_scale:g} -- {len(lens)} contigs, {sum(lens)} bp "
                    f"(chr1 {lens[0]} .. chr21 {lens[20]}), 30x 2x100bp pairs, 20 planted DEL/DUP on the longest; rsicnv rsi -b <BAM> -f <FASTA> -q 0 -Q 10 -m 101 -np "
                    f"per contig (full pileup + RP/Q0 path), contigs LPT-sharded over the GPUs")
    else:
        names = [f"19_{i}" for i in range(K * world)]; lens = [a.len] * (K * world)
        scaling = "weak"
        workload = ((f"chr19_bam (BASELINE.json configs[1]): rsicnv rsi -b <simulated sorted chr19-shaped BAM, {a.len} bp, 30x 2x100bp pairs, 20 planted DEL/DUP> "
                     f"-f <synthetic FASTA> -q 0 -Q 10 -m 101 -np (full pileup + RP/Q0 path)") if bam else
                    f"chr19_depth (BASELINE.json configs[0]): rsicnv rsi -d <synthetic chr19-shaped depth, {a.len} bp, 30x NB-like, 20 planted DEL/DUP> -c 19 -f <synthetic FASTA> -m 101 -np")
        workload += f"; {K} independent contigs per GPU and step"
    owner = shard.lpt_assign(lens, world)
    mine = [i for i in range(len(lens)) if owner[i] == rank]
    mine.sort(key=lambda i: -lens[i])          # longest first inside a rank too
    Lmax = max(lens)
    config = {"workload": workload, "contigs": len(lens), "genome_bp": int(sum(lens)), "m": 101, "scaling": scaling,
              "contigs_in_flight_per_gpu": K,
              "parallelism": f"contig-sharded (LPT) x{world} GPUs, imbalance {shard.imbalance(lens, world):.4f}, no data-path collective; {K} contigs in flight per GPU",
              "l2": "inputs per contig (read records ~40 B/base + FASTA 1 B/base, >= 0.5 GB) are far larger than the 126 MB L2"}

    if a.impl == "reference":
        if rank != 0:
            return 0
        return run_reference_arm(a, config, bam)

    import torch
    import torch.distributed as dist
    from rsicnv_b200 import api

    if not torch.cuda.is_available():
        print(json.dumps({"error": "no CUDA device: the product has no CPU path"}))
        return 2
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    nthreads = max(4, min(32, (os.cpu_count() or 8) // world))

    # ---- inputs: ONE seeded master contig of the longest length; contig i = the master truncated to lens[i]
    t_gen = time.perf_counter()
    fa = synth.make_fasta(Lmax, SEED)
    fa_pin = torch.from_numpy(fa).pin_memory()
    n_reads = [0] * len(lens); bam_bytes = [0] * len(lens)
    reads_bytes_of = [0] * len(lens); qual_bytes_of = [0] * len(lens)
    if bam:
        reads, events = synth.make_reads(Lmax, SEED, fa, coverage=30.0, n_events=20)
        import tempfile
        with tempfile.TemporaryDirectory() as td:
            t0 = time.perf_counter()
            # BGZF level 1, random bases so that it compresses like a real file; blocks end at record boundaries
            bix = synth.write_bam_aligned(os.path.join(td, "t.bam"), "19", Lmax, reads, level=1, random_seq=7, threads=nthreads)
            bam_np = np.fromfile(os.path.join(td, "t.bam"), np.uint8)
        config["bam_file_bytes"] = int(bam_np.size); config["bam_write_s"] = round(time.perf_counter() - t0, 1)
        bam_pin = torch.from_numpy(bam_np).pin_memory()
        rec_off = int(bix["rec_off"])
        pins = {k: torch.from_numpy(reads[k]).pin_memory() for k in READ_FIELDS}
        co = reads["cigar_off"].astype(np.int64); qo = reads["qual_off"].astype(np.int64)
        for i, L in enumerate(lens):
            want = int(np.searchsorted(reads["pos"], L - 700)) if L < Lmax else len(reads["pos"])
            k = int(np.searchsorted(bix["blk_rec_end"], want, side="right")) - 1      # whole record blocks only
            n_reads[i] = int(bix["blk_rec_end"][k]) if k >= 0 else 0
            bam_bytes[i] = int(bix["blk_end"][k]) - rec_off if k >= 0 else 0
            n = n_reads[i]
            qual_bytes_of[i] = int(qo[n])
            # bytes the pileup kernels read once: pos 4, flag 2, mapq 1, CIGAR offsets 4 + ops, quality offsets 8 + qualities
            reads_bytes_of[i] = n * (4 + 2 + 1 + 4 + 8) + 4 * int(co[n]) + int(qo[n])
        config["reads"] = int(sum(n_reads))
    else:
        depth, events = synth.make_depth(Lmax, SEED, fa, n_events=20)
        dp_pin = torch.from_numpy(depth).pin_memory()
    config["input_build_s"] = round(time.perf_counter() - t_gen, 1)

    def batch_for(i):
        b = api.ReadBatch()
        b.n_reads = n_reads[i]; b.tid = 0
        for k in READ_FIELDS:
            setattr(b, k, pins[k].data_ptr())
        return b

    mk = (lambda: api.Context(device=local, minq=0, min_baseQ=10)) if bam else (lambda: api.Context(device=local))
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(K)
    ctx_of = {i: mk() for i in mine}
    bufs = {i: (api.Cnv * 65536)() for i in mine}

    def stage_one(cx, i):
        cx.set_reference_ptr(fa_pin.data_ptr(), lens[i])
        if bam:
            cx.pileup_begin()
            b = batch_for(i)
            cx._ck(cx.lib.rsigpu_pileup_push(cx.h, C.byref(b)))
            cx.have_reads()
        else:
            cx.set_depth_ptr(dp_pin.data_ptr(), lens[i])

    def run_all():
        """one step: this rank's contigs go through the hot path, K in flight (ctypes releases the GIL)"""
        return dict(zip(mine, pool.map(lambda i: ctx_of[i].run_count(bufs[i], 65536), mine)))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident leg: inputs staged once, each step = the whole hot path on this rank's contigs
    for i in mine:
        stage_one(ctx_of[i], i)
    for _ in range(a.warmup):
        ncalls = run_all()
    sampler = ClockSampler(local); sampler.start()
    barrier()
    l0 = sum(cx.launch_count() for cx in ctx_of.values())
    t0 = time.perf_counter()
    for _ in range(a.steps):
        ncalls = run_all()
        torch.cuda.synchronize()
    barrier()
    dev_ms = 1e3 * (time.perf_counter() - t0)
    clocks = sampler.stop()
    launches = sum(cx.launch_count() for cx in ctx_of.values()) - l0
    big = mine[0] if mine else None
    stages = ctx_of[big].stage_ms() if big is not None else {}
    # the table (rows of every contig, header order) -> one hash: equal at every N, since sharding must not change a single byte
    rows = {}
    outputs = {}
    for i in mine:
        st = ctx_of[i].chr_stats()
        rows[i] = [api.format_row(ctx_of[i].lib, bufs[i][j], names[i], st.rdmedian, st.rdsd) for j in range(ncalls[i])]
        if a.dump_outputs:
            outputs[i] = [({n: getattr(st, n) for n, _ in api.ChrStats._fields_ if n != "reserved_"}, [bufs[i][j].as_dict() for j in range(ncalls[i])])]
    table = shard.gather_rows(rows, len(lens), rank, world)
    if a.dump_outputs:
        dump = shard.gather_rows(outputs, len(lens), rank, world)
        if rank == 0:
            dump_outputs(a.dump_outputs, dump)
    # ---- per-kernel device times on this rank's largest contig (extra profiled steps, CUDA events around every launch on the context's stream)
    prof = []
    if big is not None:
        cx = ctx_of[big]
        cx.set_profile(True)
        for _ in range(a.profile_steps):
            cx.run_count(bufs[big], 65536)
        prof = cx.profile()
        cx.set_profile(False)
        big_st = cx.chr_stats()
    staged_calls = dict(ncalls)
    for cx in ctx_of.values():
        cx.close()
    ctx_of.clear()
    torch.cuda.empty_cache()

    # ---- end-to-end leg: host bytes -> H2D -> (BGZF inflate + record decode) -> hot path -> calls on the host, every step.
    # BAM: the rank's contigs are grouped into batches of <= --e2e-batch-mb of compressed bytes; a worker (host thread + one
    # decoder context + one contig context) decodes a batch with ONE rsigpu_bam_feed_parts call -- one inflate launch over the
    # blocks of all its contigs, which is what the GPU decodes efficiently -- then takes and runs the contigs one by one while
    # the other workers decode.  Depth files: one contig per work item.
    import queue
    if bam:
        limit = int(a.e2e_batch_mb) << 20
        batches = []                                  # first-fit decreasing
        for i in sorted(mine, key=lambda i: -bam_bytes[i]):
            for b in batches:
                if sum(bam_bytes[j] for j in b) + bam_bytes[i] <= limit:
                    b.append(i); break
            else:
                batches.append([i])
        items = batches
    else:
        items = [[i] for i in mine]
    nwork = min(K, max(1, len(items)))
    decoders = [mk() for _ in range(nwork)] if bam else []
    for d in decoders:
        d.set_feed_limit(10 << 30)          # decoded bytes one feed may produce (level-1 BGZF of BAM records inflates ~4.9x)
    workers = [mk() for _ in range(nwork)]
    wbufs = [(api.Cnv * 65536)() for _ in workers]
    phase_s = [[0.0, 0.0, 0.0, 0.0] for _ in workers]      # host wall time per worker: feed_parts, set_reference, take, run

    def batch_one(w, batch):
        """BAM file bytes (pinned host memory) of every contig of the batch -> BGZF inflate + record decode on the GPU (one chunk) ->
        per contig: pileup -> ... -> calls on the host"""
        dec, cx, out = decoders[w], workers[w], wbufs[w]
        ph = phase_s[w]
        t0 = time.perf_counter()
        dec.bam_begin(1)
        runs = dec.bam_feed_parts([(bam_pin.data_ptr() + rec_off, bam_bytes[i]) for i in batch])
        t1 = time.perf_counter(); ph[0] += t1 - t0
        res = {}
        for r, (tid, nr, part) in enumerate(runs):
            i = batch[part]
            t1 = time.perf_counter()
            cx.set_reference_ptr(fa_pin.data_ptr(), lens[i])
            cx.pileup_begin()
            t2 = time.perf_counter(); ph[1] += t2 - t1
            dec.bam_take(r, cx)
            cx.have_reads()
            t3 = time.perf_counter(); ph[2] += t3 - t2
            res[i] = cx.run_count(out, 65536)
            ph[3] += time.perf_counter() - t3
        dec.bam_end()
        return res

    def depth_one(w, batch):
        cx, i = workers[w], batch[0]
        cx.set_reference_ptr(fa_pin.data_ptr(), lens[i])
        cx.set_depth_ptr(dp_pin.data_ptr(), lens[i])
        return {i: cx.run_count(wbufs[w], 65536)}

    one = batch_one if bam else depth_one

    def e2e_pass(nsteps):
        q = queue.Queue()
        for _ in range(nsteps):
            for b in sorted(items, key=lambda b: -sum((bam_bytes[j] if bam else lens[j]) for j in b)):
                q.put(b)
        got = {}

        def work(w):
            while True:
                try:
                    b = q.get_nowait()
                except queue.Empty:
                    return
                got.update(one(w, b))
        ths = [threading.Thread(target=work, args=(w,)) for w in range(nwork)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        return got

    # warm-up: every worker takes the largest work item once (its device buffers then fit any item: no cudaMalloc / cudaFree,
    # which synchronise the whole device, inside the timed region), then one untimed pass
    if items:
        biggest = max(items, key=lambda b: sum((bam_bytes[j] if bam else lens[j]) for j in b))
        for w in range(nwork):
            one(w, biggest)
            if big is not None and big not in biggest:
                one(w, [big])
    got = e2e_pass(1)
    assert all(got[i] == staged_calls[i] for i in mine), "the path from BAM bytes disagrees with the staged-reads path"
    barrier()
    for ph in phase_s:
        ph[:] = [0.0, 0.0, 0.0, 0.0]
    t0 = time.perf_counter()
    pass_ms = []
    for _ in range(a.steps):
        tp = time.perf_counter()
        e2e_pass(1)
        torch.cuda.synchronize()
        pass_ms.append(1e3 * (time.perf_counter() - tp))
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - t0)
    dprof = []; dprof_batch = None
    if bam and items:
        biggest = max(items, key=lambda b: sum(bam_bytes[j] for j in b))
        decoders[0].set_profile(True)
        batch_one(0, biggest)
        dprof = [(nm, ms, n) for nm, ms, n in decoders[0].profile() if nm.startswith("k_bgzf") or nm.startswith("k_bam")]
        decoders[0].set_profile(False)
        dprof_batch = {"contigs": len(biggest), "compressed_bytes": int(sum(bam_bytes[j] for j in biggest)), "bases": int(sum(lens[j] for j in biggest))}
    for cx in workers + decoders:
        cx.close()

    t = torch.tensor([dev_ms, e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms = [float(x) for x in t.tolist()]
    tl = torch.tensor([launches], dtype=torch.int64, device="cuda")
    if world > 1:
        dist.all_reduce(tl, op=dist.ReduceOp.SUM)
    launches = int(tl.item())
    if rank == 0:
        peak, peak_src = peaks()
        step_bases = int(sum(lens))
        value = step_bases * a.steps / (dev_ms / 1e3) / 1e9
        L = lens[big]; Lc = big_st.compact_len
        kern = []
        for name, ms, n in prof:
            b = kernel_bytes(name, L, Lc, reads_bytes_of[big], qual_bytes_of[big])
            avg = ms / max(n, 1)
            kern.append({"kernel": name, "launches_per_step": n / a.profile_steps, "avg_ms": avg, "ms_per_step": ms / a.profile_steps,
                         "algorithmic_bytes": b, "gbs": (b / 1e9) / (avg / 1e3) if b and avg > 0 else None})
        kern.sort(key=lambda k: -k["ms_per_step"])
        stream = [k for k in kern if k["algorithmic_bytes"]]
        # algorithmic bytes of the WHOLE path per step (SURVEY 8d: 18 B/base depth path + read records once + 4 B/base depth written)
        path_bytes = sum(18 * lens[i] + (reads_bytes_of[i] + 4 * lens[i] if bam else 0) for i in range(len(lens)))
        path_gbs = path_bytes * a.steps / (dev_ms / 1e3) / 1e9
        top = stream[0] if stream else (kern[0] if kern else None)
        roof = None
        if top:
            ach = top["gbs"] or 0.0
            tot_ms = max(sum(k["ms_per_step"] for k in kern), 1e-9)
            roof = {"bound": "hbm", "kernel": top["kernel"], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": ncu_traffic().get(top["kernel"]),
                    "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum per launch on a chr19-sized contig, ncu --set full (profiles/ncu_traffic.json)",
                    "peak_source": peak_src, "share_of_step": top["ms_per_step"] / tot_ms,
                    "how": "dominant streaming kernel (largest time among the HBM-bound kernels): algorithmic bytes per launch / average launch duration "
                           "(CUDA events on the context's stream, %d extra profiled steps on the rank's largest contig, %d bp)" % (a.profile_steps, L),
                    "top_kernel_by_time": kern[0]["kernel"], "top_kernel_ms": kern[0]["avg_ms"],
                    "streaming_kernels": [{"kernel": k["kernel"], "gbs": k["gbs"], "frac": (k["gbs"] or 0) / peak, "ms": k["avg_ms"], "share_of_step": k["ms_per_step"] / tot_ms,
                                           "traffic": ncu_traffic().get(k["kernel"])} for k in stream],
                    "streaming_share_of_step": sum(k["ms_per_step"] for k in stream) / tot_ms,
                    # the whole hot path against the same peak: algorithmic bytes of every stage / step time, all GPUs (per GPU: / n_gpus)
                    "path_achieved": path_gbs, "path_frac": path_gbs / (peak * world), "path_bytes_per_base": path_bytes / step_bases}
        d2h = int(sum(staged_calls.values())) * 128 + 53000 * len(mine)
        line = {"metric": METRIC, "value": value, "unit": "Gbases/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
                "dtype": "u8 qualities -> int32 depth / f64 statistics" if bam else "int32 depth / f64 statistics", "data": "synthetic", "config": config, "clocks": clocks,
                "e2e": {"value": step_bases * a.steps / (e2e_ms / 1e3) / 1e9, "unit": "Gbases/s",
                        "h2d_bytes_per_step": int(sum((bam_bytes[i] if bam else 4 * lens[i]) + lens[i] for i in range(len(lens)))),
                        "d2h_bytes_per_step": d2h * world if scaling == "weak" else d2h, "ms_per_step": e2e_ms / a.steps,
                        "pass_ms_rank0": [round(x, 1) for x in pass_ms], "workers": nwork, "work_items": len(items),
                        "worker_wall_ms_per_step_rank0": [dict(zip(("feed_parts", "set_reference", "take", "run"), [round(1e3 * x / a.steps, 1) for x in ph])) for ph in phase_s],
                        "input": ("BAM file images (BGZF) + FASTA contigs in pinned host memory -> rsigpu_bam_feed_parts (the contigs of a batch decoded as one chunk) / take -> rsigpu_run per contig -> calls on the host" if bam else
                                  "depth arrays + FASTA contigs in pinned host memory -> rsigpu_set_depth -> rsigpu_run -> calls on the host")},
                "gpu_launches": launches, "calls": int(len(table)), "table_sha1": hashlib.sha1("\n".join(table).encode()).hexdigest(), "roofline": roof,
                "largest_contig_stage_ms": stages,
                "timing": "value: wall time of the K timed steps, barrier + torch.cuda.synchronize on both sides (the contexts run on their own streams, "
                          "so the step is bracketed on the host; max over ranks); e2e: same bracket around `steps` passes over the rank's contigs from host bytes; "
                          "kernels: CUDA events around every launch of one context in extra profiled steps",
                "kernels": kern[:14]}
        if dprof:
            line["decode_kernels"] = [{"kernel": nm, "launches": nl, "ms": ms} for nm, ms, nl in sorted(dprof, key=lambda x: -x[1])]
            line["decode_batch"] = dict(dprof_batch, what="the largest e2e work item: the record blocks of these contigs decoded by one rsigpu_bam_feed_parts call "
                                                         "(decode_kernels = CUDA-event times of that call's kernels)")
        if world == 1 and not a.no_cli:
            # release this process's pinned buffers before other processes (the CLIs) are timed
            if bam:
                del pins, bam_pin
            del fa_pin
            torch.cuda.empty_cache()
            sample = a.cpu_sample
            if bam:
                cpu, out, kind = time_reference_bam(sample, 1, 19, with_ours=True)
                if len(out[0]) > 2 and out[0][2]:
                    o = out[0][2]
                    line["cli_e2e"] = {"sample_bp": sample, "reference_cli_s": cpu, "this_cli_first_s": o["first_s"], "this_cli_second_s": o["second_s"],
                                       "this_cli_hostdecode_s": o["hostdecode_s"], "this_cli_timing": o["timing"], "identical_table": o["identical_table"],
                                       "speedup_second": cpu / o["second_s"],
                                       "what": "BAM + FASTA files -> CNV table through each CLI (process start and CUDA context creation included; this CLI decodes "
                                               "the BAM on the GPU, -hostdecode on host threads)"}
                line["cpu_baseline"] = {"value": sample / cpu / 1e9, "unit": "Gbases/s", "cores": 1, "kind": kind,
                                        "sample": f"one {sample} bp 30x synthetic contig: BAM + FASTA files through the unmodified `rsicnv rsi -b ... -q 0 -Q 10 -np` CLI on one host core "
                                                  f"(the reference is single-threaded; BGZF/BAM decode included, files in page cache)"}
            else:
                cpu, out = time_reference(sample, 1, 19)
                line["cpu_baseline"] = {"value": sample / cpu / 1e9, "unit": "Gbases/s", "cores": 1, "kind": ref_kind()[1],
                                        "sample": f"one {sample} bp synthetic contig through checkgccontent..detectcnv..sd_filters on one host core "
                                                  f"(the reference is single-threaded; in-memory depth array, text parsing excluded)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
