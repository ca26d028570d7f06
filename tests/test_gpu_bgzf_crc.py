"""The CRC32 check of BGZF blocks (k_crc32.cuh, rsigpu_set_bgzf_crc) on the GPU: the emulator's cases through the real library,
a 12 Mbp / 30x file fed in 32 MiB pieces, and one feed large enough that the lane-per-block inflate kernel is picked by size."""
import numpy as np
import pytest

import test_sim_bam_decode as T
import test_sim_bgzf_crc as S
from rsicnv_b200 import api, synth

pytestmark = pytest.mark.gpu


@S.MODES
def test_every_length_and_alignment(gpu_lib, mode):
    S.every_length_and_alignment(gpu_lib, mode)


@S.MODES
@pytest.mark.parametrize("level,strategy,block_size,chunk", S.VALID)
def test_valid_files_decode_identically(gpu_lib, tmp_path, monkeypatch, mode, level, strategy, block_size, chunk):
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    S.valid_files_decode_identically(gpu_lib, tmp_path, monkeypatch, level, strategy, block_size, chunk)


@S.MODES
def test_footer_only_damage(gpu_lib, tmp_path, mode):
    S.footer_only_damage(gpu_lib, tmp_path, mode)


@S.MODES
def test_stored_payload_flips(gpu_lib, tmp_path, mode):
    S.stored_payload_flips(gpu_lib, tmp_path, mode)


@pytest.mark.parametrize("level", [1, 6, 9])
def test_fuzz_against_zlib_with_crc(gpu_lib, tmp_path, level):
    S.fuzz_against_zlib(gpu_lib, tmp_path, level)


@S.MODES
def test_feed_parts(gpu_lib, tmp_path, mode):
    S.feed_parts(gpu_lib, tmp_path, mode)


@S.MODES
def test_large_file_all_fields(gpu_lib, tmp_path, monkeypatch, mode):
    """12 Mbp at 30x (3.6 M records, ~13 k BGZF blocks), fed in 32 MiB pieces with the check on"""
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    monkeypatch.setenv("RSIGPU_BGZF_CRC", "1")
    L = 12_000_000
    fa = synth.make_fasta(L, 19)
    reads, _ = synth.make_reads(L, 19, fa, coverage=30, n_events=6)
    path = str(tmp_path / "t.bam")
    synth.write_bam(path, [("19", L), ("20", 1000)], {0: reads}, level=1, random_seq=3)
    got, h = T.decode_file(gpu_lib, path, 32 << 20)
    assert sorted(got) == [0]
    T.assert_same_reads(got[0], reads)


def test_one_feed_of_many_blocks(gpu_lib, tmp_path):
    """more than 28 k blocks in one feed: the inflate kernel is chosen by size (a lane per block), then the check; a footer
    changed in the last data block is found"""
    L = 2_000_000
    fa = synth.make_fasta(L, 23)
    reads, _ = synth.make_reads(L, 23, fa, coverage=8, n_events=2)
    path = str(tmp_path / "t.bam")
    synth.write_bam(path, [("19", L)], {0: reads}, level=6, block_size=1000, random_seq=3)
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    body = data[h["coff"]:]
    bl = S.blocks(body)
    assert len(bl) > 28000
    ctx = api.Context(lib=gpu_lib); ctx.set_bgzf_crc(True)
    ctx.bam_begin(1)
    consumed, runs = ctx.bam_feed(body, skip=h["skip"])
    assert consumed == len(body) and runs == [(0, len(reads["pos"]))]
    T.assert_same_reads(ctx.bam_run_reads(0), reads)
    ctx.bam_end()
    k = len(bl) - 2
    off, xlen, bsize = bl[k]
    bad = body.copy(); bad[off + bsize - 5] ^= 0x80
    ctx.bam_begin(1)
    with pytest.raises(api.RsiGpuError) as e:
        ctx.bam_feed(bad, skip=h["skip"])
    assert S.crc_message(k, off) in str(e.value), str(e.value)
    ctx.close()
