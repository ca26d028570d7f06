"""The BAI index built while the GPU decodes a BAM (k_bam_index.cuh, rsigpu_bam_index_begin / rsigpu_bam_index_get) in the CPU
emulator, with both inflate kernels: byte for byte what synth.write_bai writes for the same file."""
import os
import struct
import zlib

import numpy as np
import pytest

from rsicnv_b200 import api, synth

MODES = pytest.mark.parametrize("mode", [1, 2], ids=["lane-per-block", "warp-per-block"])


def build_index(lib, path, mode, chunk=None, feed_limit=None, crc=False):
    """feed the file from its first record block in `chunk`-byte pieces with indexing on; returns the index bytes"""
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    ctx = api.Context(lib=lib)
    try:
        ctx.set_inflate_mode(mode); ctx.set_bgzf_crc(crc)
        if feed_limit:
            ctx.set_feed_limit(feed_limit)
        ctx.bam_begin(len(h["names"]))
        ctx.bam_index_begin(h["coff"])
        off = h["coff"]; pending = np.zeros(0, np.uint8); first = True
        step = chunk or len(data)
        while off < len(data) or len(pending):
            piece = data[off:off + step]; off += len(piece)
            buf = np.concatenate((pending, piece))
            consumed, _ = ctx.bam_feed(buf, skip=h["skip"] if first else 0)
            if consumed:
                first = False
            pending = buf[consumed:]
            if off >= len(data) and consumed == 0:
                break
        assert len(pending) == 0
        ctx.bam_end()
        return ctx.bam_index()
    finally:
        ctx.close()


def expected(path):
    synth.write_bai(path)
    with open(path + ".bai", "rb") as f:
        return f.read()


def three_contigs(tmp_path, unmapped_tail=7, **kw):
    """contigs 1 and 3 with reads, 2 empty, plus an unmapped tail"""
    r0, _ = synth.make_reads(90_000, 21, None, coverage=5, n_events=0, tid=0)
    r2, _ = synth.make_reads(70_000, 22, None, coverage=4, n_events=0, tid=2, frac_indel=0.3)
    path = str(tmp_path / "t.bam")
    synth.write_bam(path, [("1", 90_000), ("2", 1000), ("3", 70_000)], {0: r0, 2: r2}, unmapped_tail=unmapped_tail, **kw)
    return path


def long_span_reads(L, seed, n_long=40):
    """normal reads plus reads whose CIGAR spans several 16 kbp windows (long D / N ops: large bins), reads without a CIGAR and
    placed reads with flag 0x4 -- sorted by position"""
    R, _ = synth.make_reads(L, seed, None, coverage=3, n_events=0)
    rng = np.random.default_rng(seed)
    n = len(R["pos"])
    co = R["cigar_off"].astype(np.int64); qo = R["qual_off"].astype(np.int64)
    cig = [R["cigar"][co[i]:co[i + 1]] for i in range(n)]
    qual = [R["qual"][qo[i]:qo[i + 1]] for i in range(n)]
    pos = R["pos"].astype(np.int64).tolist(); flag = R["flag"].astype(np.int64).tolist()
    for k in range(n_long):                                    # 50M <gap>D|N 50M: spans up to ~12 windows
        gap = int(rng.integers(10_000, 200_000)); op = 2 if k % 2 else 3
        cig.append(np.array([50 << 4, (gap << 4) | op, 50 << 4], np.uint32)); qual.append(np.full(100, 30, np.uint8))
        pos.append(int(rng.integers(0, L - gap - 200))); flag.append(0)
    for k in range(30):                                        # no CIGAR, some of them placed but unmapped
        cig.append(np.zeros(0, np.uint32)); qual.append(np.full(20, 30, np.uint8))
        pos.append(int(rng.integers(0, L - 100))); flag.append(4 if k % 3 else 0)
    for i in rng.choice(n, 25, replace=False):                 # placed reads with flag 0x4 that keep their CIGAR
        flag[int(i)] |= 4
    order = np.argsort(np.asarray(pos), kind="stable")
    m = len(pos)
    out = {"pos": np.asarray(pos, np.int32)[order], "flag": np.asarray(flag, np.uint16)[order]}
    for k, v in (("mpos", R["mpos"]), ("isize", R["isize"]), ("mtid", R["mtid"]), ("mapq", R["mapq"])):
        ext = np.concatenate((np.asarray(v), np.zeros(m - n, np.asarray(v).dtype)))
        out[k] = ext[order]
    cs = [cig[i] for i in order]; qs = [qual[i] for i in order]
    out["cigar_off"] = np.concatenate(([0], np.cumsum([len(c) for c in cs]))).astype(np.uint32)
    out["cigar"] = np.concatenate(cs).astype(np.uint32)
    out["qual_off"] = np.concatenate(([0], np.cumsum([len(q) for q in qs]))).astype(np.uint64)
    out["qual"] = np.concatenate(qs).astype(np.uint8)
    return out


# ---- 1. three contigs (one empty), unmapped tail; fed whole and in pieces that cut records
@MODES
@pytest.mark.parametrize("chunk", [None, 70_001])
def test_three_contigs_unmapped_tail(sim_lib, tmp_path, mode, chunk):
    path = three_contigs(tmp_path, level=6, block_size=20000)
    want = expected(path)
    assert struct.unpack_from("<Q", want, len(want) - 8)[0] == 7        # n_no_coor is written
    assert build_index(sim_lib, path, mode, chunk) == want


# ---- 2. real-looking records, indels, reads over many windows / in large bins, no CIGAR, placed unmapped
@MODES
def test_rich_records_long_spans_no_cigar(sim_lib, tmp_path, mode):
    L = 400_000
    r0 = long_span_reads(L, 31)
    r1, _ = synth.make_reads(120_000, 32, None, coverage=4, n_events=0, tid=1, frac_indel=0.3)
    path = str(tmp_path / "t.bam")
    synth.write_bam(path, [("1", L), ("2", 120_000)], {0: r0, 1: r1}, level=1, block_size=4000, rich=9)
    assert build_index(sim_lib, path, mode, 50_000) == expected(path)


# ---- 3. compression levels, fixed Huffman, block sizes; the CRC check does not change a byte
CASES = [(0, 0, 4000), (1, 0, 97), (6, 0, 20000), (9, 0, 65280), (9, zlib.Z_FIXED, 4000)]


@MODES
@pytest.mark.parametrize("level,strategy,block_size", CASES)
def test_levels_and_block_sizes(sim_lib, tmp_path, mode, level, strategy, block_size):
    path = three_contigs(tmp_path, unmapped_tail=3, level=level, strategy=strategy, block_size=block_size, random_seq=4)
    want = expected(path)
    assert build_index(sim_lib, path, mode, 90_001, crc=False) == want
    assert build_index(sim_lib, path, mode, 90_001, crc=True) == want


# ---- 4. blocks that end exactly at record ends (a record's end voffset is the next block's offset << 16)
@MODES
def test_records_ending_on_block_ends(sim_lib, tmp_path, mode):
    r, _ = synth.make_reads(150_000, 41, None, coverage=6, n_events=0)
    path = str(tmp_path / "a.bam")
    synth.write_bam_aligned(path, "19", 150_000, r, level=1, threads=1, block_size=8000)
    want = expected(path)
    assert build_index(sim_lib, path, mode) == want
    assert build_index(sim_lib, path, mode, 30_000) == want


# ---- 5. a small feed limit: records carried across feeds, runs of one bin cut by feed boundaries
@MODES
def test_small_feed_limit(sim_lib, tmp_path, mode):
    path = three_contigs(tmp_path, level=1, block_size=20000)
    assert build_index(sim_lib, path, mode, feed_limit=70_000) == expected(path)


# ---- 6. errors: unsorted files, feed_parts while indexing, positions past 2^29; the index is then refused
def write_records(path, contigs, recs):
    """a BAM of explicit (tid, pos, cigar) records"""
    reads_by_tid = {}
    for tid in sorted({t for t, _, _ in recs}):
        mine = [(p, c) for t, p, c in recs if t == tid]
        n = len(mine)
        reads_by_tid[tid] = {"pos": np.array([p for p, _ in mine], np.int32), "mpos": np.full(n, -1, np.int32), "isize": np.zeros(n, np.int32),
                             "mtid": np.full(n, -1, np.int32), "flag": np.zeros(n, np.uint16), "mapq": np.full(n, 30, np.uint8),
                             "cigar_off": np.concatenate(([0], np.cumsum([len(c) for _, c in mine]))).astype(np.uint32),
                             "cigar": np.concatenate([np.asarray(c, np.uint32) for _, c in mine]).astype(np.uint32),
                             "qual_off": np.arange(0, 10 * n + 1, 10, dtype=np.uint64), "qual": np.full(10 * n, 30, np.uint8)}
    synth.write_bam(path, contigs, reads_by_tid, level=1, block_size=4000)


def index_error(lib, path, mode, chunk=None):
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    ctx = api.Context(lib=lib)
    try:
        ctx.set_inflate_mode(mode)
        ctx.bam_begin(len(h["names"])); ctx.bam_index_begin(h["coff"])
        with pytest.raises(api.RsiGpuError) as e:
            off = h["coff"]; first = True; pending = np.zeros(0, np.uint8)
            while off < len(data) or len(pending):
                piece = data[off:off + (chunk or len(data))]; off += len(piece)
                buf = np.concatenate((pending, piece))
                consumed, _ = ctx.bam_feed(buf, skip=h["skip"] if first else 0)
                first = False if consumed else first
                pending = buf[consumed:]
                if off >= len(data) and consumed == 0:
                    break
        msg = str(e.value)
        ctx.bam_end()
        with pytest.raises(api.RsiGpuError):
            ctx.bam_index()
        return e.value.code, msg
    finally:
        ctx.close()


M10 = [10 << 4]


@MODES
def test_unsorted_position(sim_lib, tmp_path, mode):
    path = str(tmp_path / "u.bam")
    recs = [(0, 100 + 7 * i, M10) for i in range(500)]
    recs[321] = (0, 50, M10)
    write_records(path, [("1", 100_000)], recs)
    code, msg = index_error(sim_lib, path, mode)
    assert code == 2 and "bam_index: records not sorted: record 321 of this feed (tid 0, pos 50) follows tid 0, pos 2340" in msg, msg


@MODES
def test_unsorted_refid(sim_lib, tmp_path, mode):
    path = str(tmp_path / "u.bam")
    a, _ = synth.make_reads(30_000, 5, None, coverage=3, n_events=0)
    b, _ = synth.make_reads(30_000, 6, None, coverage=3, n_events=0)
    synth.write_bam(path, [("1", 30_000), ("2", 30_000)], {1: a, 0: b}, level=1, block_size=4000)   # written 0 first: swap the ids
    raw = np.fromfile(path, np.uint8)
    # rewrite as tid 1 then tid 0: decode, swap the refIDs of every record, re-compress
    h = api.parse_bam_header(raw)
    dec = bytearray()
    off = 0
    while off < len(raw):
        xlen = int(raw[off + 10]) | int(raw[off + 11]) << 8; bs = (int(raw[off + 16]) | int(raw[off + 17]) << 8) + 1
        dec += zlib.decompress(raw[off + 12 + xlen:off + bs - 8].tobytes(), -15); off += bs
    lt = struct.unpack_from("<i", dec, 4)[0]; p = 12 + lt
    for _ in range(2):
        p += 8 + struct.unpack_from("<i", dec, p)[0]
    n0 = len(b["pos"])
    q = p; k = 0
    while q < len(dec):
        struct.pack_into("<i", dec, q + 4, 1 if k < n0 else 0); q += 4 + struct.unpack_from("<i", dec, q)[0]; k += 1
    out = bytearray()
    for s in range(0, len(dec), 4000):
        blk = bytes(dec[s:s + 4000]); co = zlib.compressobj(1, zlib.DEFLATED, -15); comp = co.compress(blk) + co.flush()
        out += b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(comp) + 25) + comp + struct.pack("<II", zlib.crc32(blk) & 0xffffffff, len(blk))
    out += bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
    open(path, "wb").write(bytes(out))
    assert h["names"] == ["1", "2"]
    code, msg = index_error(sim_lib, path, mode)
    last = int(b["pos"][-1]); first = int(a["pos"][0])
    assert code == 2 and f"bam_index: records not sorted: record {n0} of this feed (tid 0, pos {first}) follows tid 1, pos {last}" in msg, msg


@MODES
def test_unsorted_across_feeds(sim_lib, tmp_path, mode):
    """the first record of a feed is checked against the last one of the previous feed"""
    path = str(tmp_path / "u.bam")
    recs = [(0, 1000 + 3 * i, M10) for i in range(3000)]
    recs[2000:] = [(0, 10 + i, M10) for i in range(1000)]
    write_records(path, [("1", 100_000)], recs)
    code, msg = index_error(sim_lib, path, mode, chunk=20_000)
    assert code == 2 and "bam_index: records not sorted: record " in msg and "(tid 0, pos 10) follows tid 0, pos 6997" in msg, msg


@MODES
def test_position_past_2_29(sim_lib, tmp_path, mode):
    path = str(tmp_path / "r.bam")
    recs = [(0, 100 + i, M10) for i in range(300)] + [(0, (1 << 29) - 5, M10)]
    write_records(path, [("1", (1 << 29) + 100)], recs)
    code, msg = index_error(sim_lib, path, mode)
    assert code == 3 and f"bam_index: record 300 of this feed (tid 0, pos {(1 << 29) - 5}) ends past 2^29" in msg, msg


def test_feed_parts_refused_while_indexing(sim_lib, tmp_path):
    r, _ = synth.make_reads(40_000, 43, None, coverage=4, n_events=0)
    path = str(tmp_path / "p.bam")
    ix = synth.write_bam_aligned(path, "19", 40_000, r, level=1, threads=1, block_size=8000)
    data = np.fromfile(path, np.uint8)
    part = data[int(ix["rec_off"]):int(ix["blk_end"][-1])]
    ctx = api.Context(lib=sim_lib)
    ctx.bam_begin(1); ctx.bam_index_begin(int(ix["rec_off"]))
    for parts in ([part, part], [part]):
        with pytest.raises(api.RsiGpuError) as e:
            ctx.bam_feed_parts(parts)
        assert e.value.code == 2 and "bam_feed_parts: not available while a BAM index is built" in str(e.value)
    ctx.bam_end()
    with pytest.raises(api.RsiGpuError) as e:
        ctx.bam_index()
    assert "bam_index_get: no index" in str(e.value)
    # without indexing the same context decodes the parts as before
    ctx.bam_begin(1)
    assert [(t, p) for t, n, p in ctx.bam_feed_parts([part, part])] == [(0, 0), (0, 1)]
    ctx.bam_end()
    ctx.close()


def test_index_begin_after_the_first_feed_is_refused(sim_lib, tmp_path):
    path = three_contigs(tmp_path, level=1, block_size=20000)
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    ctx = api.Context(lib=sim_lib)
    ctx.bam_begin(3)
    ctx.bam_feed(data[h["coff"]:h["coff"] + 60_000], skip=h["skip"])
    with pytest.raises(api.RsiGpuError) as e:
        ctx.bam_index_begin(h["coff"])
    assert "bam_index_begin: call it after rsigpu_bam_begin and before the first feed" in str(e.value)
    ctx.close()
