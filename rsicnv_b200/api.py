"""Python host-side mirror of the reference's seams for the `rsicnv rsi` path, over the C ABI in
include/rsigpu.h (ctypes; no torch types cross the boundary).

The method names follow the reference functions they stand for (file:line relative to the reference's
src/): `load_finish` = checkgccontent + apply_cap + concatenate_data + the chromosome statistics of
main() (gccontent.cpp:95, loaddata.cpp:229, 48, rsi.cpp:2202), `detectcnv` (rsi.cpp:1795),
`sd_filters` (rsi.cpp:1753), `cnv_stat` (pairrd.cpp:622), `write_cnv_to_file` (rsi.cpp:1592).

There is no CPU implementation behind this module: the shared library is built by nvcc for sm_100a and
`load_library()` raises if it is missing; `Context()` raises if there is no CUDA device.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(_HERE, "librsigpu.so")

TYPE_NAMES = ("DEL", "DUP", "UNKNOWN")
TRANS = {"NBN": 0, "NB": 0, "MED": 1, "ALL": 2}

ARR_RAW_DEPTH, ARR_DEPTH, ARR_BIN_MED, ARR_BIN_NBN, ARR_BIN_MEDINT, ARR_BIN_STATUS, ARR_NOSEQ_BEG, ARR_NOSEQ_END, \
    ARR_BIN_STATUS1, ARR_SEGMENTS, ARR_BLOCKS, ARR_PREMERGE, ARR_MERGED, ARR_DETECTED = range(14)
_ARR_DTYPE = {ARR_RAW_DEPTH: np.int32, ARR_DEPTH: np.int32, ARR_BIN_MED: np.float32, ARR_BIN_NBN: np.float32,
              ARR_BIN_MEDINT: np.int32, ARR_BIN_STATUS: np.int32, ARR_NOSEQ_BEG: np.int32, ARR_NOSEQ_END: np.int32,
              ARR_BIN_STATUS1: np.int32}

ERRORS = {1: "CUDA error", 2: "bad argument / call order", 3: "input outside the supported range", 4: "output buffer too small",
          5: "no CUDA device (there is no CPU fallback)"}


class RsiGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"rsigpu error {code} ({ERRORS.get(code, '?')}): {msg}")
        self.code = code


class Params(C.Structure):
    """rsigpu_params: the tunables get_parameters() fills (rsi.cpp:1986-2068)"""
    _fields_ = [("m", C.c_int32), ("minq", C.c_int32), ("min_baseQ", C.c_int32), ("gcadjust", C.c_int32), ("trans", C.c_int32),
                ("merge", C.c_int32), ("maxchkbp", C.c_int32), ("reserved_", C.c_int32), ("cap", C.c_double),
                ("threshold", C.c_double), ("epsilon", C.c_double), ("chklen", C.c_double)]


class Cnv(C.Structure):
    """rsigpu_cnv: flat mirror of cnv_st (rsi.h:8-51)"""
    _fields_ = [(n, C.c_int32) for n in ("tid", "type", "geno", "status", "start", "end", "length", "sc1", "sc2", "pair")] + \
               [(n, C.c_double) for n in ("score", "p1", "p2", "cnvmed", "cnvsd", "cnviqr", "refmed", "refsd", "refiqr", "q0")] + \
               [("rp", C.c_int32), ("pad_", C.c_int32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_ if n != "pad_"}


class ReadBatch(C.Structure):
    _fields_ = [("n_reads", C.c_int64), ("tid", C.c_int32), ("reserved_", C.c_int32), ("pos", C.c_void_p), ("mpos", C.c_void_p),
                ("isize", C.c_void_p), ("mtid", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p), ("cigar_off", C.c_void_p),
                ("cigar", C.c_void_p), ("qual_off", C.c_void_p), ("qual", C.c_void_p)]


class ChrStats(C.Structure):
    _fields_ = [("rdmedian", C.c_double), ("rdsd", C.c_double), ("tmedian", C.c_double), ("tlamda", C.c_double), ("rdmad", C.c_double),
                ("target_len", C.c_int32), ("compact_len", C.c_int32), ("nbins", C.c_int32), ("lmax", C.c_int32),
                ("isize_mean", C.c_int32), ("isize_sd", C.c_int32), ("n_noseq", C.c_int32), ("reserved_", C.c_int32)]


EXPORTS = ("rsigpu_default_params", "rsigpu_create", "rsigpu_destroy", "rsigpu_last_error", "rsigpu_num_devices", "rsigpu_set_reference",
           "rsigpu_set_depth", "rsigpu_pileup_begin", "rsigpu_pileup_push", "rsigpu_pileup_end", "rsigpu_load_finish", "rsigpu_detectcnv",
           "rsigpu_sd_filters", "rsigpu_cnv_stat", "rsigpu_get_calls", "rsigpu_run", "rsigpu_get_chr_stats", "rsigpu_get_array",
           "rsigpu_format_row", "rsigpu_launch_count", "rsigpu_last_stage_ms", "rsigpu_set_profile", "rsigpu_get_profile",
           "rsigpu_get_log", "rsigpu_reads_begin", "rsigpu_stat_calls", "rsigpu_bam_take_range", "rsigpu_split_range", "rsigpu_split_run", "rsigpu_split_p2p_bytes", "rsigpu_set_level0_mode", "rsigpu_set_feed_limit", "rsigpu_set_inflate_mode", "rsigpu_set_bgzf_crc", "rsigpu_set_cand_threads", "rsigpu_debug_state", "rsigpu_pileup_commit", "rsigpu_bam_begin", "rsigpu_bam_feed", "rsigpu_bam_feed_parts", "rsigpu_bam_take",
           "rsigpu_bam_end", "rsigpu_bam_run_field", "rsigpu_bam_index_begin", "rsigpu_bam_index_get", "rsigpu_pinned_alloc", "rsigpu_pinned_free",
           "rsigpu_set_bam_by_ref", "rsigpu_pileup_sort", "rsigpu_reads_take", "rsigpu_reads_field")

_libs: dict[str, C.CDLL] = {}


def load_library(path: str | None = None) -> C.CDLL:
    path = os.path.abspath(path or DEFAULT_LIB)
    if path in _libs:
        return _libs[path]
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with `make lib` (nvcc, sm_100a). There is no CPU fallback.")
    lib = C.CDLL(path)
    lib.rsigpu_last_error.restype = C.c_char_p
    lib.rsigpu_launch_count.restype = C.c_int64
    lib.rsigpu_split_p2p_bytes.restype = C.c_longlong
    lib.rsigpu_destroy.restype = None
    lib.rsigpu_pinned_free.restype = None
    lib.rsigpu_pinned_free.argtypes = [C.c_void_p]
    lib.rsigpu_pinned_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
    for name in EXPORTS:
        getattr(lib, name)  # raises AttributeError if the ABI is incomplete
    _libs[path] = lib
    return lib


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


class BamRun(C.Structure):
    _fields_ = [("tid", C.c_int32), ("part", C.c_int32), ("n_reads", C.c_int64)]


def parse_bam_header(data) -> dict:
    """BAM header from the first BGZF blocks of a file (bam_header_read, samtools-0.1.18/bam.c:69-110), inflated on the
    host with zlib -- a few KiB.  Returns names, lengths and where the alignment records start: `coff` = file offset of the
    BGZF block that holds the first record, `skip` = decoded bytes of that block in front of it."""
    import struct
    import zlib
    mv = memoryview(data)
    dec = b""; starts = []          # (file offset of block, decoded offset of its first byte)
    off = 0

    def more():
        nonlocal off, dec
        if off + 18 > len(mv):
            raise ValueError("truncated BAM header")
        h = bytes(mv[off:off + 18])
        if h[:4] != b"\x1f\x8b\x08\x04":
            raise ValueError("not a BGZF file")
        bsize = struct.unpack_from("<H", h, 16)[0] + 1
        xlen = struct.unpack_from("<H", h, 10)[0]
        starts.append((off, len(dec)))
        dec += zlib.decompress(bytes(mv[off + 12 + xlen:off + bsize - 8]), -15)
        off += bsize

    def need(n):
        while len(dec) < n:
            more()
    need(12)
    if dec[:4] != b"BAM\x01":
        raise ValueError("not a BAM file")
    l_text = struct.unpack_from("<i", dec, 4)[0]
    need(12 + l_text)
    n_ref = struct.unpack_from("<i", dec, 8 + l_text)[0]
    p = 12 + l_text
    names, lens = [], []
    for _ in range(n_ref):
        need(p + 4)
        ln = struct.unpack_from("<i", dec, p)[0]
        need(p + 8 + ln)
        names.append(dec[p + 4:p + 4 + ln - 1].decode()); lens.append(struct.unpack_from("<i", dec, p + 4 + ln)[0])
        p += 8 + ln
    # the block that holds decoded offset p (the first record); if the header ends exactly at a block end, the next block
    coff, skip = off, 0
    for i, (fo, do) in enumerate(starts):
        hi = starts[i + 1][1] if i + 1 < len(starts) else len(dec)
        if do <= p < hi:
            coff, skip = fo, p - do
    return {"names": names, "lens": lens, "coff": coff, "skip": skip}


class Context:
    """One contig on one GPU: what one iteration of the reference's chromosome loop owns (rsi.cpp:2189-2217)."""

    def __init__(self, device: int = 0, lib: str | None = None, m=101, minq=0, min_baseQ=13, cap=4.0, gcadjust=True, trans="NBN",
                 merge=True, threshold=-1.0, epsilon=1.5, chklen=2.5, maxchkbp=100000):
        self.lib = load_library(lib)
        p = Params()
        self.lib.rsigpu_default_params(C.byref(p))
        p.m = m; p.minq = minq; p.min_baseQ = min_baseQ; p.cap = cap; p.gcadjust = 1 if gcadjust else 0
        p.trans = TRANS[trans] if isinstance(trans, str) else int(trans)
        p.merge = 1 if merge else 0; p.threshold = threshold; p.epsilon = epsilon; p.chklen = chklen; p.maxchkbp = maxchkbp
        self.params = p
        self.m = m if m % 2 == 1 else m + 1
        h = C.c_void_p()
        rc = self.lib.rsigpu_create(C.c_int(device), C.byref(p), C.byref(h))
        if rc != 0:
            raise RsiGpuError(rc, "rsigpu_create failed")
        self.h = h
        self._keep = []
        mode = int(os.environ.get("RSIGPU_INFLATE_MODE", "0") or 0)      # test hook: force one of the two inflate kernels (rsigpu_set_inflate_mode)
        if mode:
            self.set_inflate_mode(mode)
        if int(os.environ.get("RSIGPU_BGZF_CRC", "0") or 0):           # run any decode with the CRC32 check on (rsigpu_set_bgzf_crc)
            self.set_bgzf_crc(True)

    def close(self):
        if getattr(self, "h", None):
            self.lib.rsigpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise RsiGpuError(rc, (self.lib.rsigpu_last_error(self.h) or b"").decode())

    # ---- inputs
    def set_reference(self, fasta: np.ndarray, tid: int = 0):
        """read_fasta output for one contig (readref.cpp:10-86): uint8 ASCII, newlines stripped"""
        fasta = np.ascontiguousarray(fasta, dtype=np.uint8)
        self._ck(self.lib.rsigpu_set_reference(self.h, _ptr(fasta), C.c_int32(len(fasta)), C.c_int32(tid)))
        self.L = len(fasta)

    def set_reference_ptr(self, ptr: int, n: int, tid: int = 0):
        self._ck(self.lib.rsigpu_set_reference(self.h, C.c_void_p(ptr), C.c_int32(n), C.c_int32(tid)))
        self.L = n

    def set_depth(self, depth: np.ndarray):
        """the array load_data_from_text builds (loaddata.cpp:496-517)"""
        depth = np.ascontiguousarray(depth, dtype=np.int32)
        self._keep = [depth]
        self._ck(self.lib.rsigpu_set_depth(self.h, _ptr(depth), C.c_int32(len(depth))))

    def set_depth_ptr(self, ptr: int, n: int):
        self._ck(self.lib.rsigpu_set_depth(self.h, C.c_void_p(ptr), C.c_int32(n)))

    def pileup_begin(self):
        self._ck(self.lib.rsigpu_pileup_begin(self.h, C.c_int32(self.L)))

    def pileup_push(self, reads: dict, tid: int = 0):
        """reads: dict of numpy arrays pos, mpos, isize, mtid (int32), flag (uint16), mapq (uint8), cigar_off (uint32, n+1),
        cigar (uint32), qual_off (uint64, n+1), qual (uint8) -- one position-sorted batch of one contig"""
        b = ReadBatch()
        keep = {}
        for name, dt in (("pos", np.int32), ("mpos", np.int32), ("isize", np.int32), ("mtid", np.int32), ("flag", np.uint16),
                         ("mapq", np.uint8), ("cigar_off", np.uint32), ("cigar", np.uint32), ("qual_off", np.uint64), ("qual", np.uint8)):
            keep[name] = np.ascontiguousarray(reads[name], dtype=dt)
            setattr(b, name, keep[name].ctypes.data)
        b.n_reads = len(keep["pos"]); b.tid = tid
        self._ck(self.lib.rsigpu_pileup_push(self.h, C.byref(b)))

    # ---- BAM bytes decoded on the GPU (k_bam.cuh): begin / feed / take / end
    def bam_begin(self, n_ref: int):
        self._ck(self.lib.rsigpu_bam_begin(self.h, C.c_int32(n_ref)))

    RUN_CAP = 65536      # the decoder's own limit of refID runs per feed: nothing is ever truncated

    def _run_buf(self):
        if getattr(self, "_runs", None) is None:
            self._runs = (BamRun * self.RUN_CAP)()
        return self._runs

    def bam_feed(self, data, nbytes: int | None = None, skip: int = 0):
        """data: uint8 numpy array (or an integer host address with nbytes) that starts at a BGZF block boundary.
        Returns (bytes consumed, [(tid, n_reads), ...]) -- the runs stay valid until the next feed."""
        if isinstance(data, int):
            ptr, n = C.c_void_p(data), int(nbytes)
        else:
            data = np.ascontiguousarray(data, dtype=np.uint8)
            self._keep = [data]
            ptr, n = _ptr(data), (len(data) if nbytes is None else int(nbytes))
        runs = self._run_buf()
        consumed = C.c_int64(0); nr = C.c_int32(0)
        self._ck(self.lib.rsigpu_bam_feed(self.h, ptr, C.c_int64(n), C.c_int64(skip), C.byref(consumed), runs, C.c_int32(self.RUN_CAP), C.byref(nr)))
        return int(consumed.value), [(runs[i].tid, int(runs[i].n_reads)) for i in range(nr.value)]

    def bam_feed_parts(self, parts: list):
        """parts: [(host address, nbytes), ...] or uint8 arrays -- whole BGZF blocks each, record-aligned at both ends -- decoded as
        ONE chunk (rsigpu_bam_feed_parts).  Returns [(tid, n_reads, part), ...]"""
        keep = []; ptrs = (C.c_void_p * len(parts))(); sizes = (C.c_int64 * len(parts))()
        for j, pt in enumerate(parts):
            if isinstance(pt, tuple):
                ptrs[j] = C.c_void_p(pt[0]); sizes[j] = int(pt[1])
            else:
                a = np.ascontiguousarray(pt, dtype=np.uint8); keep.append(a)
                ptrs[j] = a.ctypes.data; sizes[j] = len(a)
        self._keep = keep
        runs = self._run_buf(); nr = C.c_int32(0)
        self._ck(self.lib.rsigpu_bam_feed_parts(self.h, C.c_int32(len(parts)), ptrs, sizes, runs, C.c_int32(self.RUN_CAP), C.byref(nr)))
        return [(runs[i].tid, int(runs[i].n_reads), int(runs[i].part)) for i in range(nr.value)]

    def bam_take(self, run: int, dst: "Context"):
        rc = self.lib.rsigpu_bam_take(self.h, C.c_int32(run), dst.h)
        if rc != 0:
            raise RsiGpuError(rc, (self.lib.rsigpu_last_error(dst.h) or self.lib.rsigpu_last_error(self.h) or b"").decode())

    def bam_take_range(self, run: int, dst: "Context", pos_lo: int, pos_hi: int):
        rc = self.lib.rsigpu_bam_take_range(self.h, C.c_int32(run), dst.h, C.c_int32(pos_lo), C.c_int32(pos_hi))
        if rc != 0:
            raise RsiGpuError(rc, (self.lib.rsigpu_last_error(dst.h) or self.lib.rsigpu_last_error(self.h) or b"").decode())

    def bam_end(self):
        self._ck(self.lib.rsigpu_bam_end(self.h))

    def bam_index_begin(self, file_offset: int):
        """build the file's .bai while it is decoded (rsigpu_bam_index_begin): call after bam_begin, before the first feed;
        file_offset = offset in the file of the first byte fed, and every feed must continue where the last one's consumed ended"""
        self._ck(self.lib.rsigpu_bam_index_begin(self.h, C.c_int64(file_offset)))

    def bam_index(self) -> bytes:
        """the .bai bytes after a successful bam_end (rsigpu_bam_index_get)"""
        nb = C.c_int64(0)
        self._ck(self.lib.rsigpu_bam_index_get(self.h, None, C.c_int64(0), C.byref(nb)))
        buf = (C.c_uint8 * max(nb.value, 1))()
        self._ck(self.lib.rsigpu_bam_index_get(self.h, buf, C.c_int64(nb.value), C.byref(nb)))
        return bytes(buf[:nb.value])

    _BAM_FIELDS = (("pos", np.int32), ("mpos", np.int32), ("isize", np.int32), ("mtid", np.int32), ("flag", np.uint16), ("mapq", np.uint8),
                   ("cigar_off", np.uint32), ("cigar", np.uint32), ("qual_off", np.uint64), ("qual", np.uint8))

    def bam_run_reads(self, run: int) -> dict:
        """the decoded records of one run as the read dict pileup_push takes (parity tests)"""
        out = {}
        for f, (name, dt) in enumerate(self._BAM_FIELDS):
            nb = C.c_int64(0)
            self._ck(self.lib.rsigpu_bam_run_field(self.h, C.c_int32(run), C.c_int32(f), None, C.c_int64(0), C.byref(nb)))
            a = np.empty(nb.value // np.dtype(dt).itemsize, dt)
            if nb.value:
                self._ck(self.lib.rsigpu_bam_run_field(self.h, C.c_int32(run), C.c_int32(f), _ptr(a), C.c_int64(nb.value), C.byref(nb)))
            out[name] = a
        return out

    def reads(self) -> dict:
        """every staged read as the read dict pileup_push takes (rsigpu_reads_field)"""
        out = {}
        for f, (name, dt) in enumerate(self._BAM_FIELDS):
            nb = C.c_int64(0)
            self._ck(self.lib.rsigpu_reads_field(self.h, C.c_int32(f), None, C.c_int64(0), C.byref(nb)))
            a = np.empty(nb.value // np.dtype(dt).itemsize, dt)
            if nb.value:
                self._ck(self.lib.rsigpu_reads_field(self.h, C.c_int32(f), _ptr(a), C.c_int64(nb.value), C.byref(nb)))
            out[name] = a
        return out

    def reads_take(self, r0: int, r1: int, dst: "Context"):
        """append this context's staged reads [r0, r1) to dst's (rsigpu_reads_take)"""
        before = (self.lib.rsigpu_last_error(self.h), self.lib.rsigpu_last_error(dst.h))
        rc = self.lib.rsigpu_reads_take(self.h, C.c_int64(r0), C.c_int64(r1), dst.h)
        if rc != 0:   # the message of whichever context the failure was recorded on (a stale one on the other is ignored)
            src_e, dst_e = self.lib.rsigpu_last_error(self.h), self.lib.rsigpu_last_error(dst.h)
            msg = src_e if src_e and src_e != before[0] else dst_e if dst_e and dst_e != before[1] else src_e or dst_e or b""
            raise RsiGpuError(rc, msg.decode())

    def pileup_sort(self):
        """sort the staged reads by position on the GPU, stable (rsigpu_pileup_sort)"""
        self._ck(self.lib.rsigpu_pileup_sort(self.h))

    def set_bam_by_ref(self, on: bool):
        """group each bam_feed's records by refID, -1 last, stable in file order (rsigpu_set_bam_by_ref)"""
        self._ck(self.lib.rsigpu_set_bam_by_ref(self.h, C.c_int(1 if on else 0)))

    def reads_begin(self, tid: int, target_len: int):
        """`stat`: stage reads of one contig without a reference (then pileup_push / bam_take)"""
        self._ck(self.lib.rsigpu_reads_begin(self.h, C.c_int32(tid), C.c_int32(target_len)))
        self.L = target_len

    def stat_calls(self, calls: list) -> list:
        """RP / Q0 (cnv_stat, pairrd.cpp:622-748) for a list of calls (the whole file's list, in order); returns the annotated copies"""
        buf = (Cnv * max(len(calls), 1))()
        for i, c in enumerate(calls):
            C.memmove(C.byref(buf[i]), C.byref(c), C.sizeof(Cnv))
        self._ck(self.lib.rsigpu_stat_calls(self.h, buf, C.c_int32(len(calls))))
        return [_copy_cnv(buf[i]) for i in range(len(calls))]

    def pileup_end(self):
        """runs the pileup kernels now (so that the raw depth can be read back); `run()` re-runs them as its first stage"""
        self._ck(self.lib.rsigpu_pileup_end(self.h))

    def have_reads(self):
        """marks the staged batches as complete WITHOUT running the pileup yet (rsigpu_run does it as its first stage)"""
        self._ck(self.lib.rsigpu_pileup_commit(self.h))

    # ---- the seams, in the order main() calls them (rsi.cpp:2197-2211)
    def load_finish(self):
        self._ck(self.lib.rsigpu_load_finish(self.h))

    def detectcnv(self):
        self._ck(self.lib.rsigpu_detectcnv(self.h))

    def sd_filters(self):
        self._ck(self.lib.rsigpu_sd_filters(self.h))

    def cnv_stat(self):
        self._ck(self.lib.rsigpu_cnv_stat(self.h))

    def calls(self, cap: int = 65536) -> list[Cnv]:
        n = C.c_int32(0)
        buf = (Cnv * cap)()
        self._ck(self.lib.rsigpu_get_calls(self.h, buf, C.c_int32(cap), C.byref(n)))
        return [_copy_cnv(buf[i]) for i in range(n.value)]

    def run(self, cap: int = 65536) -> list[Cnv]:
        n = C.c_int32(0)
        buf = (Cnv * cap)()
        self._ck(self.lib.rsigpu_run(self.h, buf, C.c_int32(cap), C.byref(n)))
        return [_copy_cnv(buf[i]) for i in range(n.value)]

    def run_count(self, buf, cap: int) -> int:
        """rsigpu_run into a caller-owned (Cnv * cap) buffer; returns the number of calls (bench hot loop)"""
        n = C.c_int32(0)
        self._ck(self.lib.rsigpu_run(self.h, buf, C.c_int32(cap), C.byref(n)))
        return n.value

    # ---- outputs
    def chr_stats(self) -> ChrStats:
        s = ChrStats()
        self._ck(self.lib.rsigpu_get_chr_stats(self.h, C.byref(s)))
        return s

    def array(self, which: int):
        cnt = C.c_int64(0)
        self._ck(self.lib.rsigpu_get_array(self.h, C.c_int32(which), None, C.c_int64(0), C.byref(cnt)))
        n = cnt.value
        if which >= ARR_SEGMENTS:
            buf = (Cnv * max(n, 1))()
            self._ck(self.lib.rsigpu_get_array(self.h, C.c_int32(which), buf, C.c_int64(n), C.byref(cnt)))
            return [_copy_cnv(buf[i]) for i in range(n)]
        out = np.zeros(max(n, 1), _ARR_DTYPE[which])
        self._ck(self.lib.rsigpu_get_array(self.h, C.c_int32(which), _ptr(out), C.c_int64(n), C.byref(cnt)))
        return out[:n]

    def log_text(self, chrom: str, text_input: bool) -> str:
        """the deterministic part of <out>.log for the contig just processed (rsigpu_get_log)"""
        n = C.c_int64(0)
        self._ck(self.lib.rsigpu_get_log(self.h, C.c_char_p(chrom.encode()), C.c_int32(1 if text_input else 0), None, C.c_int64(0), C.byref(n)))
        buf = C.create_string_buffer(n.value + 1)
        self._ck(self.lib.rsigpu_get_log(self.h, C.c_char_p(chrom.encode()), C.c_int32(1 if text_input else 0), buf, C.c_int64(n.value), C.byref(n)))
        return buf.raw[:n.value].decode()

    def launch_count(self) -> int:
        return int(self.lib.rsigpu_launch_count(self.h))

    def stage_ms(self):
        a = (C.c_float * 6)()
        self._ck(self.lib.rsigpu_last_stage_ms(self.h, a))
        return dict(zip(("pileup", "load_finish", "detect", "candidates", "stat", "total"), [float(x) for x in a]))

    def set_profile(self, on: bool):
        self._ck(self.lib.rsigpu_set_profile(self.h, C.c_int(1 if on else 0)))

    def profile(self):
        cap, stride = 128, 48
        names = C.create_string_buffer(cap * stride)
        ms = (C.c_float * cap)(); ln = (C.c_int32 * cap)()
        k = self.lib.rsigpu_get_profile(self.h, names, C.c_int32(stride), ms, ln, C.c_int32(cap))
        out = []
        for i in range(min(k, cap)):
            nm = names.raw[i * stride:(i + 1) * stride].split(b"\0", 1)[0].decode()
            out.append((nm, float(ms[i]), int(ln[i])))
        return out

    DEBUG_FIELDS = ("err", "rd_min", "rd_max", "pos_sum", "pos_cnt", "rdmean", "cap_median", "cap_thr", "capv", "hist_base", "chist_R", "rdmedian",
                    "rdsd", "rdmad", "max_binsum", "gstar", "gc_tab80", "gc_tab90", "gc_tab100", "gc_cnt90", "tmedian", "tsigma", "tlamda", "Lmax",
                    "lbreak_del", "lbreak_dup", "n_runs", "n_nonzero", "st_lo", "st_hi", "lvl0_sum", "filt_on", "cand_redone",
                    "cp_tests", "cp_left", "cp_reverse", "cp_right", "cp_prefix", "cp_runmean", "cp_hist_ref", "cp_hist_cnv", "cp_sums", "cp_edge_refine",
                    "cp_merge", "cp_final", "cp_blocks", "cp_sort", "cp_cnvlen_total", "cp_nref_total", "bam_rewalked")

    def debug_state(self) -> dict:
        a = (C.c_double * 64)()
        n = self.lib.rsigpu_debug_state(self.h, a, C.c_int32(64))
        return dict(zip(self.DEBUG_FIELDS, [float(a[i]) for i in range(n)]))

    def set_level0_mode(self, mode: int):
        self._ck(self.lib.rsigpu_set_level0_mode(self.h, C.c_int(mode)))

    def set_inflate_mode(self, mode: int):
        """0 = by chunk size, 1 = one lane per BGZF block, 2 = one warp per BGZF block"""
        self._ck(self.lib.rsigpu_set_inflate_mode(self.h, C.c_int(mode)))

    def set_bgzf_crc(self, on: bool):
        """check the CRC32 of every BGZF block bam_feed / bam_feed_parts decode (off by default, like the reference's reader)"""
        self._ck(self.lib.rsigpu_set_bgzf_crc(self.h, C.c_int(1 if on else 0)))

    def set_feed_limit(self, decoded_bytes: int):
        """test hook: decoded bytes one bam_feed may produce"""
        self._ck(self.lib.rsigpu_set_feed_limit(self.h, C.c_int64(decoded_bytes)))

    def set_cand_threads(self, threads: int):
        self._ck(self.lib.rsigpu_set_cand_threads(self.h, C.c_int(threads)))


def split_range(lib: C.CDLL, target_len: int, n_parts: int, part: int):
    """(beg, end, read_halo) of one part of a contig split over several GPUs (rsigpu_split_range)"""
    b = C.c_int32(0); e = C.c_int32(0); h = C.c_int32(0)
    rc = lib.rsigpu_split_range(C.c_int32(target_len), C.c_int32(n_parts), C.c_int32(part), C.byref(b), C.byref(e), C.byref(h))
    if rc != 0:
        raise RsiGpuError(rc, "split_range")
    return b.value, e.value, h.value


def split_reads(reads: dict, beg: int, end: int, halo: int) -> dict:
    """the reads a part of a split contig stages: pos in [beg - halo, end), offsets rebased (position-sorted SoA in, SoA out)"""
    pos = reads["pos"]
    lo = int(np.searchsorted(pos, beg - halo, side="left")); hi = int(np.searchsorted(pos, end, side="left"))
    co = reads["cigar_off"].astype(np.int64); qo = reads["qual_off"].astype(np.int64)
    d = {k: reads[k][lo:hi] for k in ("pos", "mpos", "isize", "mtid", "flag", "mapq")}
    d["cigar_off"] = (co[lo:hi + 1] - co[lo]).astype(np.uint32); d["cigar"] = reads["cigar"][co[lo]:co[hi]]
    d["qual_off"] = (qo[lo:hi + 1] - qo[lo]).astype(np.uint64); d["qual"] = reads["qual"][qo[lo]:qo[hi]]
    return d


def split_run(parts: list, cap: int = 65536) -> list:
    """rsigpu_split_run: parts[0] is the lead; returns the calls"""
    arr = (C.c_void_p * len(parts))(*[p.h for p in parts])
    n = C.c_int32(0)
    buf = (Cnv * cap)()
    rc = parts[0].lib.rsigpu_split_run(arr, C.c_int32(len(parts)), buf, C.c_int32(cap), C.byref(n))
    if rc != 0:
        raise RsiGpuError(rc, (parts[0].lib.rsigpu_last_error(parts[0].h) or b"").decode())
    return [_copy_cnv(buf[i]) for i in range(n.value)]


def _copy_cnv(src: Cnv) -> Cnv:
    c = Cnv()
    C.memmove(C.byref(c), C.byref(src), C.sizeof(Cnv))
    return c


def format_row(lib: C.CDLL, cnv: Cnv | None, chrom: str, rdmedian: float, rdsd: float) -> str:
    """cnv_format1 (rsi.cpp:581-631); cnv=None gives the column header"""
    buf = C.create_string_buffer(1024)
    rc = lib.rsigpu_format_row(C.byref(cnv) if cnv is not None else None, C.c_char_p(chrom.encode()), C.c_double(rdmedian),
                               C.c_double(rdsd), buf, C.c_int32(1024))
    if rc != 0:
        raise RsiGpuError(rc, "format_row")
    return buf.value.decode()


def write_cnv_to_file(path: str, lib: C.CDLL, calls: list[Cnv], chrom: str, rdmedian: float, rdsd: float, input_name: str,
                      gcadjusted: bool, append: bool):
    """write_cnv_to_file (rsi.cpp:1592-1616): header lines once, then one row per call, appended per contig"""
    with open(path, "a" if append else "w") as f:
        if not append:
            f.write(f"#input {input_name}\n")
            if gcadjusted:
                f.write("#GC adjusted\n")
            f.write(format_row(lib, None, "", 0, 0) + "\n")
        for c in calls:
            f.write(format_row(lib, c, chrom, rdmedian, rdsd) + "\n")
