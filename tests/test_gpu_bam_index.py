"""The BAI index built while the GPU decodes (k_bam_index.cuh, rsigpu_bam_index_begin / rsigpu_bam_index_get) on the device: the
emulator's cases through the real library, and a 12 Mbp / 30x file fed whole and in 32 MiB pieces, byte-compared to
synth.write_bai."""
import numpy as np
import pytest

import test_sim_bam_index as S
from rsicnv_b200 import synth

pytestmark = pytest.mark.gpu


@S.MODES
@pytest.mark.parametrize("chunk", [None, 70_001])
def test_three_contigs_unmapped_tail(gpu_lib, tmp_path, mode, chunk):
    S.test_three_contigs_unmapped_tail(gpu_lib, tmp_path, mode, chunk)


@S.MODES
def test_rich_records_long_spans_no_cigar(gpu_lib, tmp_path, mode):
    S.test_rich_records_long_spans_no_cigar(gpu_lib, tmp_path, mode)


@S.MODES
@pytest.mark.parametrize("level,strategy,block_size", S.CASES)
def test_levels_and_block_sizes(gpu_lib, tmp_path, mode, level, strategy, block_size):
    S.test_levels_and_block_sizes(gpu_lib, tmp_path, mode, level, strategy, block_size)


@S.MODES
def test_records_ending_on_block_ends(gpu_lib, tmp_path, mode):
    S.test_records_ending_on_block_ends(gpu_lib, tmp_path, mode)


@S.MODES
def test_small_feed_limit(gpu_lib, tmp_path, mode):
    S.test_small_feed_limit(gpu_lib, tmp_path, mode)


@S.MODES
def test_unsorted_position(gpu_lib, tmp_path, mode):
    S.test_unsorted_position(gpu_lib, tmp_path, mode)


@S.MODES
def test_unsorted_refid(gpu_lib, tmp_path, mode):
    S.test_unsorted_refid(gpu_lib, tmp_path, mode)


@S.MODES
def test_unsorted_across_feeds(gpu_lib, tmp_path, mode):
    S.test_unsorted_across_feeds(gpu_lib, tmp_path, mode)


@S.MODES
def test_position_past_2_29(gpu_lib, tmp_path, mode):
    S.test_position_past_2_29(gpu_lib, tmp_path, mode)


def test_feed_parts_refused_while_indexing(gpu_lib, tmp_path):
    S.test_feed_parts_refused_while_indexing(gpu_lib, tmp_path)


def test_index_begin_after_the_first_feed_is_refused(gpu_lib, tmp_path):
    S.test_index_begin_after_the_first_feed_is_refused(gpu_lib, tmp_path)


@pytest.fixture(scope="module")
def large_bam(tmp_path_factory):
    L = 12_000_000
    reads, _ = synth.make_reads(L, 12, None, coverage=30, n_events=0, frac_indel=0.1)
    path = str(tmp_path_factory.mktemp("large") / "t.bam")
    synth.write_bam(path, [("19", L), ("20", 5000)], {0: reads}, level=1, random_seq=3, threads=16, unmapped_tail=5)
    return path, S.expected(path)


@S.MODES
@pytest.mark.parametrize("chunk", [None, 32 << 20])
def test_large_file(gpu_lib, large_bam, mode, chunk):
    path, want = large_bam
    assert S.build_index(gpu_lib, path, mode, chunk) == want
