"""BAM files that are not coordinate-sorted on the B200: the emulator's cases of test_sim_unsorted.py through the real library,
and a shuffled 12 Mbp 30x file through by-ref decode, staging, reads_take and pileup_sort against the sorted file."""
import numpy as np
import pytest

from rsicnv_b200 import api, synth
import test_sim_unsorted as T

pytestmark = pytest.mark.gpu


def test_sort_short_and_long_reads(gpu_lib):
    T.check_sort(gpu_lib, T.short_and_long(4_000_000, 3, cov=10, n_long=600), 3)


def test_sort_is_stable_on_one_position(gpu_lib):
    T.test_sort_is_stable_on_one_position(gpu_lib)


def test_sort_positions_up_to_2_31(gpu_lib):
    T.test_sort_positions_up_to_2_31(gpu_lib)


def test_sort_empty_one_and_sorted(gpu_lib):
    T.test_sort_empty_one_and_sorted(gpu_lib)


def test_reads_take_between_contexts(gpu_lib):
    T.test_reads_take_between_contexts(gpu_lib)


@pytest.mark.parametrize("mode", T.MODES, ids=T.MODE_IDS)
@pytest.mark.parametrize("kind,rich,n_mid,n_tail", [("pairs", None, 0, 0), ("shuffled", None, 40, 25), ("pairs", 3, 7, 0)],
                         ids=["pairs", "shuffled-unplaced", "pairs-rich"])
@pytest.mark.parametrize("feed_limit,crc", [(None, False), (1 << 16, False), (3 << 16, True)], ids=["whole", "carried", "carried-crc"])
def test_decode_by_ref(gpu_lib, tmp_path, monkeypatch, mode, kind, rich, n_mid, n_tail, feed_limit, crc):
    T.test_decode_by_ref(gpu_lib, tmp_path, monkeypatch, mode, kind, rich, n_mid, n_tail, feed_limit, crc)


def test_decode_by_ref_3000_references(gpu_lib, tmp_path):
    T.test_decode_by_ref_3000_references(gpu_lib, tmp_path)


def test_without_by_ref_an_unsorted_file_still_fails(gpu_lib, tmp_path):
    T.test_without_by_ref_an_unsorted_file_still_fails(gpu_lib, tmp_path)


def test_by_ref_refusals(gpu_lib, tmp_path):
    T.test_by_ref_refusals(gpu_lib, tmp_path)


def test_whole_path_shuffled_equals_sorted(gpu_lib, whole_files):
    T.check_whole_path(gpu_lib, whole_files)


whole_files = T.whole_files


@pytest.mark.parametrize("mode", T.MODES, ids=T.MODE_IDS)
def test_shuffled_12mbp_30x(gpu_lib, tmp_path, monkeypatch, mode):
    """one 12 Mbp contig at 30x plus unplaced reads, every record shuffled: by-ref decode in 32 MiB feeds, staging, reads_take,
    pileup_sort; depth, calls, RP / Q0, arrays and log equal the sorted file's through the existing route"""
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    L = 12_000_000
    contigs = [("12", L), ("x", 5000)]
    fa = synth.make_fasta(L, 31)
    reads = synth.make_reads(L, 31, fa, coverage=30, n_events=8, lens=(3000, 8000, 20000))[0]
    sorted_path, shuffled_path = str(tmp_path / "s.bam"), str(tmp_path / "u.bam")
    n = len(reads["pos"])
    perm = np.random.default_rng(31).permutation(n)
    order = np.zeros(n + 100, np.int64)
    order[np.random.default_rng(32).choice(n + 100, 100, replace=False)] = -1
    synth.write_bam_unsorted(shuffled_path, contigs, {0: synth.take_reads(reads, perm)}, order, random_seq=4, threads=32)
    synth.write_bam(sorted_path, contigs, {0: T.stable_sorted(synth.take_reads(reads, perm))}, random_seq=4, unmapped_tail=100, threads=32)
    kw = dict(minq=0, min_baseQ=10)
    stage, seg = T.stage_by_ref(gpu_lib, shuffled_path, feed_limit=32 << 20)
    try:
        def from_stage(ctx):
            for r0, r1 in seg[0]:
                stage.reads_take(r0, r1, ctx)
            ctx.pileup_sort()
        got, calls = T.run_contig(gpu_lib, fa, 0, "12", from_stage, kw)
        want, _ = T.run_contig(gpu_lib, fa, 0, "12", lambda ctx: T.take_sorted(gpu_lib, sorted_path, 0, ctx), kw)
        assert len(seg[0]) > 1 and got == want and len(calls) >= 3
    finally:
        stage.close()
