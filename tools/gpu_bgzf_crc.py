"""manual measurement: what the CRC32 check of BGZF blocks (rsigpu_set_bgzf_crc, k_bgzf_crc32) adds to rsigpu_bam_feed.

One chr19-shaped 30x BAM (synth, level 1) is fed whole, from pinned memory, with the check off and on alternately, for both
inflate kernels, in one process.  Prints the GPU's name and power limit, the median wall time of the feed each way, the
added time per feed, and the check's rate in decoded GB/s (from the added wall time, and from the kernel's own CUDA-event
time in a separate profiled feed).  argv: [repetitions [output json]]."""
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
import numpy as np  # noqa: E402

from rsicnv_b200 import api, synth  # noqa: E402

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 7
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
print("gpu:", gpu, flush=True)
L = synth.CHR19_LEN
fa = synth.make_fasta(L, 19)
reads, _ = synth.make_reads(L, 19, fa, coverage=30, n_events=20)
with tempfile.TemporaryDirectory() as td:
    path = os.path.join(td, "t.bam")
    synth.write_bam(path, [("19", L)], {0: reads}, level=1, random_seq=7, threads=32)
    data = np.fromfile(path, np.uint8)
h = api.parse_bam_header(data)
body_len = len(data) - h["coff"]
lib = api.load_library()
pin = C.c_void_p()
assert lib.rsigpu_pinned_alloc(C.c_size_t(len(data)), C.byref(pin)) == 0
C.memmove(pin, data.ctypes.data, len(data))
n_rec = len(reads["pos"])


def one_feed(dec, crc):
    dec.set_bgzf_crc(crc)
    dec.bam_begin(1)
    t0 = time.perf_counter()
    consumed, runs = dec.bam_feed(pin.value + h["coff"], body_len, skip=h["skip"])
    t1 = time.perf_counter()
    assert consumed == body_len and runs == [(0, n_rec)], runs
    dec.bam_end()
    return 1e3 * (t1 - t0)


result = {"gpu": gpu, "file_bytes": len(data), "records": n_rec}
for mode, name in ((1, "lane-per-block"), (2, "warp-per-block")):
    dec = api.Context()
    dec.set_inflate_mode(mode)
    dec.set_feed_limit(10 << 30)
    one_feed(dec, False); one_feed(dec, True)          # warm-up: buffers, modules
    t = {False: [], True: []}
    for r in range(REPS):
        for crc in ((False, True) if r % 2 == 0 else (True, False)):
            t[crc].append(one_feed(dec, crc))
    dec.set_profile(True)                               # a separate feed: per-kernel CUDA-event time (serialises the launches)
    one_feed(dec, True)
    prof = {nm: (ms, n) for nm, ms, n in dec.profile()}
    dec.close()
    ms_k, n_k = prof["k_bgzf_crc32"]
    kern = ms_k / n_k
    blk = []; off = h["coff"]; dec_bytes = 0
    while off + 18 <= len(data):
        bsize = int(data[off + 16]) + (int(data[off + 17]) << 8) + 1
        dec_bytes += int(data[off + bsize - 4]) | int(data[off + bsize - 3]) << 8 | int(data[off + bsize - 2]) << 16 | int(data[off + bsize - 1]) << 24
        blk.append(off); off += bsize
    off_ms, on_ms = statistics.median(t[False]), statistics.median(t[True])
    row = {"inflate": name, "blocks": len(blk), "decoded_bytes": dec_bytes, "feed_off_ms": off_ms, "feed_on_ms": on_ms,
           "added_ms": on_ms - off_ms, "added_pct": 100.0 * (on_ms - off_ms) / off_ms, "kernel_ms": kern,
           "rate_gbs_added": dec_bytes / 1e6 / max(on_ms - off_ms, 1e-9), "rate_gbs_kernel": dec_bytes / 1e6 / kern,
           "off_all_ms": t[False], "on_all_ms": t[True]}
    result[name] = row
    print(f"{name}: {len(blk)} blocks, {dec_bytes / 1e9:.2f} GB decoded; feed off {off_ms:.2f} ms, on {on_ms:.2f} ms "
          f"(median of {REPS}); added {on_ms - off_ms:.2f} ms = {row['added_pct']:.1f} %; k_bgzf_crc32 {kern:.3f} ms = "
          f"{row['rate_gbs_kernel']:.0f} GB/s", flush=True)
lib.rsigpu_pinned_free(pin)
if len(sys.argv) > 2:
    with open(sys.argv[2], "w") as f:
        json.dump(result, f, indent=1)
