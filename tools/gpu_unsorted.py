"""manual measurement: what grouping a feed's records by refID (rsigpu_set_bam_by_ref) adds to rsigpu_bam_feed, and the time of
rsigpu_pileup_sort on a chr19-sized contig's reads (k_sort.cuh).

A chr19-shaped 30x BAM (synth, level 1) under a 25-reference header (the reads on refID 18) is fed whole, from pinned memory,
with by-ref off and on alternately, for both inflate kernels, in one process; every by-ref feed must give the same single run.
Then the contig's reads, shuffled by a seeded permutation, are staged in one context and sorted; the sorted reads must equal the
stable sort by position.  Prints the GPU's name and power limit, median wall times, the added time, and per-kernel CUDA-event
times of a separate profiled call.  argv: [repetitions [output json]]."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

from rsicnv_b200 import api, synth  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("gpu:", gpu, flush=True)
L = synth.CHR19_LEN
fa = synth.make_fasta(L, 19)
reads, _ = synth.make_reads(L, 19, fa, coverage=30, n_events=20, tid=18)
n_rec = len(reads["pos"])
contigs = [(f"c{k}", 1_000_000) for k in range(25)]
contigs[18] = ("19", L)
result = {"gpu": gpu, "records": n_rec}


def prof_of(ctx):
    return {nm: round(ms, 3) for nm, ms, _ in ctx.profile()}


with tempfile.TemporaryDirectory() as td:
    path = os.path.join(td, "t.bam")
    synth.write_bam(path, contigs, {18: reads}, level=1, random_seq=7, threads=32)
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    body_len = len(data) - h["coff"]
    lib = api.load_library()
    pin = C.c_void_p()
    assert lib.rsigpu_pinned_alloc(C.c_size_t(len(data)), C.byref(pin)) == 0
    C.memmove(pin, data.ctypes.data, len(data))
    result["file_bytes"] = len(data)

    def one_feed(dec, by_ref):
        dec.set_bam_by_ref(by_ref)
        dec.bam_begin(len(contigs))
        t0 = time.perf_counter()
        consumed, runs = dec.bam_feed(pin.value + h["coff"], body_len, skip=h["skip"])
        t1 = time.perf_counter()
        assert consumed == body_len and runs == [(18, n_rec)], runs
        dec.bam_end()
        return 1e3 * (t1 - t0)

    for mode, name in ((1, "lane-per-block"), (2, "warp-per-block")):
        dec = api.Context()
        dec.set_inflate_mode(mode)
        dec.set_feed_limit(10 << 30)
        one_feed(dec, False); one_feed(dec, True)          # warm-up: buffers, modules
        t = {False: [], True: []}
        for r in range(REPS):
            for on in ((False, True) if r % 2 == 0 else (True, False)):
                t[on].append(one_feed(dec, on))
        dec.set_profile(True)
        one_feed(dec, True)
        prof = prof_of(dec)
        dec.close()
        off_ms, on_ms = statistics.median(t[False]), statistics.median(t[True])
        sort_k = {k: v for k, v in prof.items() if k.startswith(("k_sort", "k_off"))}
        result[name] = {"feed_off_ms": off_ms, "feed_on_ms": on_ms, "added_ms": on_ms - off_ms, "added_pct": 100.0 * (on_ms - off_ms) / off_ms,
                        "sort_kernels_ms": sort_k, "off_all_ms": t[False], "on_all_ms": t[True]}
        print(f"by-ref feed, {name}: {n_rec} records; off {off_ms:.2f} ms, on {on_ms:.2f} ms (median of {REPS}); added {on_ms - off_ms:.2f} ms "
              f"= {100.0 * (on_ms - off_ms) / off_ms:.1f} %; sort kernels {sort_k}", flush=True)
    lib.rsigpu_pinned_free(pin)

# pileup_sort on the contig's reads: shuffled, and already sorted (the check alone)
perm = np.random.default_rng(19).permutation(n_rec)
shuffled = synth.take_reads(reads, perm)
want_pos = shuffled["pos"][np.argsort(shuffled["pos"], kind="stable")]
staged_bytes = sum(int(np.asarray(v).nbytes) for v in shuffled.values())
result["staged_bytes"] = staged_bytes
ctx = api.Context()
ctx.reads_begin(18, L)


def timed_sort(R, profile=False):
    ctx.reads_begin(18, L)
    ctx.pileup_push(R)
    ctx.set_profile(profile)
    t0 = time.perf_counter()
    ctx.pileup_sort()
    return 1e3 * (time.perf_counter() - t0)


timed_sort(shuffled)                                   # warm-up
got = ctx.reads()
assert np.array_equal(got["pos"], want_pos)
assert np.array_equal(got["qual_off"], synth.take_reads(shuffled, np.argsort(shuffled["pos"], kind="stable"))["qual_off"])
ts = [timed_sort(shuffled) for _ in range(REPS)]
tc = [timed_sort(reads) for _ in range(REPS)]
timed_sort(shuffled, profile=True)
prof = prof_of(ctx)
ctx.close()
result["pileup_sort"] = {"shuffled_ms": ts, "sorted_check_ms": tc, "kernels_ms": prof}
print(f"pileup_sort: {n_rec} reads, {staged_bytes / 1e9:.2f} GB staged; shuffled {statistics.median(ts):.2f} ms, already sorted "
      f"{statistics.median(tc):.3f} ms (medians of {REPS}, host clock, includes the allocation of the sorted copy); kernels {prof}", flush=True)
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as f:
        json.dump(result, f, indent=1)
