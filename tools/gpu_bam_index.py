"""manual measurement: what building the BAI index on the GPU (rsigpu_bam_index_begin, k_bam_index.cuh) adds to rsigpu_bam_feed,
and the wall time of `rsicnv index` on the same file.

One chr19-shaped 30x BAM (synth, level 1) is fed whole, from pinned memory, with indexing off and on alternately, for both
inflate kernels, in one process; the index of every indexed feed must equal synth.write_bai's.  Prints the GPU's name and power
limit, the median wall time of the feed each way, the added time, and the index kernels' own CUDA-event time in a separate
profiled feed.  Then `rsicnv index` runs on the file (and the reference's `bamtool index` where it is built).
argv: [repetitions [output json]]."""
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

from bind import REF_BAMTOOL  # noqa: E402
from rsicnv_b200 import api, synth  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 7
CLI = os.path.join(ROOT, "rsicnv_b200", "bin", "rsicnv")
KERNELS = ("k_bam_index_rec", "k_bam_index_scan", "k_bam_index_emit")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("gpu:", gpu, flush=True)
L = synth.CHR19_LEN
fa = synth.make_fasta(L, 19)
reads, _ = synth.make_reads(L, 19, fa, coverage=30, n_events=20)
result = {"gpu": gpu}
with tempfile.TemporaryDirectory() as td:
    path = os.path.join(td, "t.bam")
    synth.write_bam(path, [("19", L)], {0: reads}, level=1, random_seq=7, threads=32)
    t0 = time.perf_counter(); synth.write_bai(path); t_py = time.perf_counter() - t0
    want = open(path + ".bai", "rb").read(); os.remove(path + ".bai")
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    body_len = len(data) - h["coff"]
    lib = api.load_library()
    pin = C.c_void_p()
    assert lib.rsigpu_pinned_alloc(C.c_size_t(len(data)), C.byref(pin)) == 0
    C.memmove(pin, data.ctypes.data, len(data))
    n_rec = len(reads["pos"])
    result.update(file_bytes=len(data), records=n_rec, write_bai_python_s=t_py)

    def one_feed(dec, ix):
        dec.bam_begin(1)
        if ix:
            dec.bam_index_begin(h["coff"])
        t0 = time.perf_counter()
        consumed, runs = dec.bam_feed(pin.value + h["coff"], body_len, skip=h["skip"])
        t1 = time.perf_counter()
        assert consumed == body_len and runs == [(0, n_rec)], runs
        dec.bam_end()
        if ix:
            assert dec.bam_index() == want
        return 1e3 * (t1 - t0)

    for mode, name in ((1, "lane-per-block"), (2, "warp-per-block")):
        dec = api.Context()
        dec.set_inflate_mode(mode)
        dec.set_feed_limit(10 << 30)
        one_feed(dec, False); one_feed(dec, True)          # warm-up: buffers, modules
        t = {False: [], True: []}
        for r in range(REPS):
            for ix in ((False, True) if r % 2 == 0 else (True, False)):
                t[ix].append(one_feed(dec, ix))
        dec.set_profile(True)                               # a separate feed: per-kernel CUDA-event time (serialises the launches)
        one_feed(dec, True)
        prof = {nm: (ms, n) for nm, ms, n in dec.profile()}
        dec.close()
        kern = {k: prof[k][0] / prof[k][1] for k in KERNELS}
        off_ms, on_ms = statistics.median(t[False]), statistics.median(t[True])
        row = {"inflate": name, "feed_off_ms": off_ms, "feed_on_ms": on_ms, "added_ms": on_ms - off_ms,
               "added_pct": 100.0 * (on_ms - off_ms) / off_ms, "kernel_ms": kern, "kernels_total_ms": sum(kern.values()),
               "off_all_ms": t[False], "on_all_ms": t[True]}
        result[name] = row
        print(f"{name}: {n_rec} records; feed off {off_ms:.2f} ms, on {on_ms:.2f} ms (median of {REPS}); added {on_ms - off_ms:.2f} ms = "
              f"{row['added_pct']:.1f} %; kernels " + ", ".join(f"{k} {v:.3f} ms" for k, v in kern.items()), flush=True)
    lib.rsigpu_pinned_free(pin)
    # the CLI, and the reference's samtools where it is built
    walls = []
    for _ in range(3):
        t0 = time.perf_counter()
        r = subprocess.run([CLI, "index", "-b", path], capture_output=True, text=True, env=dict(os.environ, RSICNV_TIMING="1"))
        walls.append(time.perf_counter() - t0)
        assert r.returncode == 0, r.stderr
        assert open(path + ".bai", "rb").read() == want
    result["rsicnv_index_wall_s"] = walls
    result["rsicnv_index_timing"] = r.stderr.strip()
    print(f"rsicnv index: wall {min(walls):.3f} s (best of 3: {', '.join(f'{w:.3f}' for w in walls)}); {r.stderr.strip()}", flush=True)
    if os.path.exists(REF_BAMTOOL):
        os.remove(path + ".bai")
        t0 = time.perf_counter(); subprocess.run([REF_BAMTOOL, "index", path], check=True); tb = time.perf_counter() - t0
        result["reference_bamtool_index_s"] = tb
        result["reference_same_bytes"] = open(path + ".bai", "rb").read() == want
        print(f"reference bamtool index: {tb:.3f} s, same bytes: {result['reference_same_bytes']}", flush=True)
    else:
        result["reference_bamtool_index_s"] = None
        print("reference bamtool not built (oracle/_ref): its time is not measured", flush=True)
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as f:
        json.dump(result, f, indent=1)
