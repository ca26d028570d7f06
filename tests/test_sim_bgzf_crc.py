"""The CRC32 check of BGZF blocks on the GPU decode path (k_crc32.cuh, rsigpu_set_bgzf_crc) in the CPU emulator, with both
inflate kernels.  The kernel's CRC is pinned to zlib.crc32 through the error precedence (inflate, then CRC, then record):
a file whose blocks all carry the right CRC but whose bytes are no BAM records must fail with a RECORD error."""
import hashlib
import struct
import zlib

import numpy as np
import pytest

import test_sim_bam_decode as T
import test_sim_inflate_fuzz as F
from rsicnv_b200 import api, synth

MODES = pytest.mark.parametrize("mode", [1, 2], ids=["lane-per-block", "warp-per-block"])
EOF_BLOCK = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def bgzf_block(data, crc=None):
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    comp = co.compress(data) + co.flush()
    assert len(comp) + 26 <= 65536
    crc = zlib.crc32(data) & 0xffffffff if crc is None else crc
    return b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(comp) + 25) + comp + struct.pack("<II", crc, len(data))


def blocks(b):
    """(file offset, xlen, bsize) of every BGZF block"""
    b = bytes(b); off = 0; out = []
    while off + 18 <= len(b):
        xlen = struct.unpack_from("<H", b, off + 10)[0]; bsize = struct.unpack_from("<H", b, off + 16)[0] + 1
        out.append((off, xlen, bsize)); off += bsize
    return out


def feed(lib, mode, body, skip=0, crc=True):
    """one feed of `body`: (True, signature of the decoded runs) or (False, error message)"""
    ctx = api.Context(lib=lib); ctx.set_inflate_mode(mode); ctx.set_bgzf_crc(crc); ctx.bam_begin(1)
    try:
        consumed, runs = ctx.bam_feed(body, skip=skip)
        sig = [consumed, runs]
        for i in range(len(runs)):
            r = ctx.bam_run_reads(i)
            sig.append(hashlib.sha1(b"".join(np.ascontiguousarray(r[k]).tobytes() for k in sorted(r))).hexdigest())
        return True, sig
    except api.RsiGpuError as e:
        return False, str(e)
    finally:
        ctx.close()


def crc_message(k, off):
    return f"CRC32 mismatch in BGZF block {k} of this feed (compressed offset {off} of the bytes passed)"


def small_file(tmp_path, level, block_size=4000, strategy=0, L=30000, seed=77):
    fa = synth.make_fasta(L, seed)
    reads, _ = synth.make_reads(L, seed, fa, coverage=4, n_events=2)
    path = str(tmp_path / "t.bam")
    synth.write_bam(path, [("1", L)], {0: reads}, level=level, strategy=strategy, block_size=block_size)
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    return data[h["coff"]:], h["skip"]


# ---- 1. every length 0..300, around 4 KiB and up to 64 KiB, at every alignment of the decoded buffer
def every_length_and_alignment(lib, mode):
    rng = np.random.default_rng(7)
    lens = [7, 1] + list(range(0, 301)) + [4095, 13, 4096, 5, 4097, 3, 65535, 9, 65536, 1, 65536]
    payloads = []
    for i, n in enumerate(lens):
        hi = 256 if n <= 4097 else 4       # the 64 KiB blocks must compress to fit a BGZF block
        p = rng.integers(0, hi, n, dtype=np.uint8).tobytes()
        if i == 0:
            p = b"\x00" * 4 + p[4:]        # a first record of block_size 0: the bytes are no BAM records
        payloads.append(p)
    good = b"".join(bgzf_block(p) for p in payloads) + EOF_BLOCK
    ok, msg = feed(lib, mode, np.frombuffer(good, np.uint8))
    assert not ok and "corrupt BAM record" in msg and "CRC32" not in msg, msg
    offs = np.cumsum([0] + [len(bgzf_block(p)) for p in payloads])
    nblk = len(payloads) + 1
    picks = [[2], [1 + 300], [len(lens) - 1], [len(lens) - 3, len(lens) - 1], [nblk - 1]] + \
            [sorted(rng.choice(nblk, 3, replace=False).tolist()) for _ in range(4)]
    for pick in picks:
        parts = []
        for k, p in enumerate(payloads):
            crc = zlib.crc32(p) & 0xffffffff
            parts.append(bgzf_block(p, crc ^ (1 << int(rng.integers(0, 32))) if k in pick else crc))
        eof = EOF_BLOCK if nblk - 1 not in pick else EOF_BLOCK[:-8] + struct.pack("<I", 1 << int(rng.integers(0, 32))) + EOF_BLOCK[-4:]
        ok, msg = feed(lib, mode, np.frombuffer(b"".join(parts) + eof, np.uint8))
        k = min(pick)
        assert not ok and crc_message(k, int(offs[k])) in msg, (pick, msg)


@MODES
def test_every_length_and_alignment(sim_lib, mode):
    every_length_and_alignment(sim_lib, mode)


# ---- 2. valid files pass and decode to the same reads, fed in pieces that cut records
VALID = [(0, 0, 4000, 50000), (1, 0, 65280, 70000), (6, 0, 97, 30000), (9, 0, 4000, 90001), (9, zlib.Z_FIXED, 65280, 60000)]


def valid_files_decode_identically(lib, tmp_path, monkeypatch, level, strategy, block_size, chunk):
    contigs = [("1", 60000), ("2", 5000), ("3", 40000)]
    rb = {0: T.make_reads(60000, 11)[1], 2: T.make_reads(40000, 12)[1]}
    path = str(tmp_path / "t.bam")
    synth.write_bam(path, contigs, rb, level=level, strategy=strategy, block_size=block_size, random_seq=5)
    monkeypatch.setenv("RSIGPU_BGZF_CRC", "0")
    off, _ = T.decode_file(lib, path, chunk)
    monkeypatch.setenv("RSIGPU_BGZF_CRC", "1")
    on, _ = T.decode_file(lib, path, chunk)
    assert sorted(on) == sorted(off) == [0, 2]
    for tid in on:
        T.assert_same_reads(on[tid], off[tid])
        T.assert_same_reads(on[tid], rb[tid])


@MODES
@pytest.mark.parametrize("level,strategy,block_size,chunk", VALID)
def test_valid_files_decode_identically(sim_lib, tmp_path, monkeypatch, mode, level, strategy, block_size, chunk):
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    valid_files_decode_identically(sim_lib, tmp_path, monkeypatch, level, strategy, block_size, chunk)


# ---- 3. only a footer CRC changed: accepted unchanged without the check, refused with it
def footer_only_damage(lib, tmp_path, mode):
    body, skip = small_file(tmp_path, 6)
    ok, want = feed(lib, mode, body, skip, crc=False)
    assert ok
    assert feed(lib, mode, body, skip, crc=True) == (True, want)
    bl = blocks(body)
    rng = np.random.default_rng(3)
    for k in [0, 1, len(bl) // 2, len(bl) - 2] + rng.choice(len(bl) - 1, 3, replace=False).tolist():
        off, xlen, bsize = bl[k]
        b = body.copy(); b[off + bsize - 8 + int(rng.integers(0, 4))] ^= 1 << int(rng.integers(0, 8))
        assert feed(lib, mode, b, skip, crc=False) == (True, want), k
        ok, msg = feed(lib, mode, b, skip, crc=True)
        assert not ok and crc_message(k, off) in msg, (k, msg)


@MODES
def test_footer_only_damage(sim_lib, tmp_path, mode):
    footer_only_damage(sim_lib, tmp_path, mode)


# ---- 4. one bit of a stored block's payload: the check refuses every flip; without it nothing changes
def stored_payload_flips(lib, tmp_path, mode):
    body, skip = small_file(tmp_path, 0)
    ok, want = feed(lib, mode, body, skip, crc=False)
    assert ok
    bl = blocks(body)
    rng = np.random.default_rng(5)
    silently_different = 0
    for _ in range(30):
        k = int(rng.integers(1, len(bl) - 2))
        off, xlen, bsize = bl[k]
        p = off + 12 + xlen + 5 + int(rng.integers(0, bsize - 12 - xlen - 8 - 5))    # past the 5-byte stored-block header
        b = body.copy(); b[p] ^= 1 << int(rng.integers(0, 8))
        ok, msg = feed(lib, mode, b, skip, crc=True)
        assert not ok and crc_message(k, off) in msg, (k, msg)
        off_ok, off_sig = feed(lib, mode, b, skip, crc=False)
        silently_different += off_ok and off_sig != want
    assert silently_different > 0          # what the check is for: without it, damaged records decode without an error


@MODES
def test_stored_payload_flips(sim_lib, tmp_path, mode):
    stored_payload_flips(sim_lib, tmp_path, mode)


# ---- 5. random bit flips: accepted iff every block passes zlib's raw inflate, ISIZE and CRC32; both kernels agree
def zlib_crc_verdict(b):
    v = F.zlib_verdict(b)
    if not v:
        return v
    b = bytes(b)
    for off, xlen, bsize in blocks(b):
        data = zlib.decompress(b[off + 12 + xlen:off + bsize - 8], -15)
        if zlib.crc32(data) & 0xffffffff != struct.unpack_from("<I", b, off + bsize - 8)[0]:
            return False
    return True


def fuzz_against_zlib(lib, tmp_path, level):
    body, skip = small_file(tmp_path, level)
    rng = np.random.default_rng(200 + level)
    checked = refused = 0
    for it in range(14):
        b = body.copy()
        for _ in range(int(rng.integers(1, 3))):
            b[int(rng.integers(18, len(b) - 8))] ^= 1 << int(rng.integers(0, 8))
        z = zlib_crc_verdict(b)
        if z is None:
            continue
        lane = feed(lib, 1, b, skip, crc=True)
        warp = feed(lib, 2, b, skip, crc=True)
        assert lane == warp, (it, lane, warp)
        assert lane[0] == z, (it, z, lane)
        checked += 1; refused += not z
    assert checked >= 10 and refused > 0


@pytest.mark.parametrize("level", [1, 6, 9])
def test_fuzz_against_zlib_with_crc(sim_lib, tmp_path, level):
    fuzz_against_zlib(sim_lib, tmp_path, level)


# ---- 6. feed_parts: the failing part is named with the offset inside it; intact parts decode as separate feeds do
def feed_parts(lib, tmp_path, mode):
    files = []
    for k, (L, seed) in enumerate(((40000, 41), (30000, 42), (50000, 43))):
        fa, reads = T.make_reads(L, seed, cov=5)
        path = str(tmp_path / f"p{k}.bam")
        ix = synth.write_bam_aligned(path, "19", L, reads, level=1, random_seq=3, threads=1, block_size=8000)
        data = np.fromfile(path, np.uint8)
        files.append((data[int(ix["rec_off"]):int(ix["blk_end"][-1])], reads))
    ctx = api.Context(lib=lib); ctx.set_inflate_mode(mode); ctx.set_bgzf_crc(True)
    ctx.bam_begin(1)
    runs = ctx.bam_feed_parts([f[0] for f in files])
    assert [(t, p) for t, n, p in runs] == [(0, 0), (0, 1), (0, 2)]
    for i, (tid, n, part) in enumerate(runs):
        T.assert_same_reads(ctx.bam_run_reads(i), files[part][1])
    ctx.bam_end()
    for j in (0, 1, 2):
        bl = blocks(files[j][0])
        k = len(bl) // 2
        off, xlen, bsize = bl[k]
        bad = [f[0] for f in files]; bad[j] = bad[j].copy(); bad[j][off + bsize - 6] ^= 0x10
        ctx.bam_begin(1)
        with pytest.raises(api.RsiGpuError) as e:
            ctx.bam_feed_parts(bad)
        assert f"CRC32 mismatch in BGZF block {k} of part {j} (compressed offset {off} of that part)" in str(e.value), str(e.value)
        ctx.bam_end()
        ctx.set_bgzf_crc(False)        # the same parts without the check: accepted, same reads
        ctx.bam_begin(1)
        assert [(t, p) for t, n, p in ctx.bam_feed_parts(bad)] == [(0, 0), (0, 1), (0, 2)]
        T.assert_same_reads(ctx.bam_run_reads(j), files[j][1])
        ctx.bam_end()
        ctx.set_bgzf_crc(True)
    ctx.close()


@MODES
def test_feed_parts(sim_lib, tmp_path, mode):
    feed_parts(sim_lib, tmp_path, mode)
