"""BAM files that are not coordinate-sorted, in the CPU emulator: the stable GPU sort of staged reads (rsigpu_pileup_sort,
k_sort.cuh), the decoder grouping each feed's records by refID (rsigpu_set_bam_by_ref), moving staged reads between contexts
(rsigpu_reads_take), and the whole path on a shuffled file against the same file sorted through the existing route."""
import numpy as np
import pytest

from bind import oracle_bam_decode
from common import split_reads
from rsicnv_b200 import api, synth
from test_sim_bam_decode import assert_same_reads
from test_sim_long_reads import uneven_cuts
from test_sim_split import _snapshot

MODES = [1, 2]
MODE_IDS = ["lane-per-block", "warp-per-block"]


def stable_sorted(R):
    return synth.take_reads(R, np.argsort(R["pos"], kind="stable"))


def sort_staged(lib, R, batches=None, L=None):
    """push R (in batches), pileup_sort, read every staged field back; returns (reads, launches of pileup_sort)"""
    with api.Context(lib=lib) as ctx:
        ctx.reads_begin(0, L or int(max(int(R["pos"].max(initial=0)) + 1, 1000)))
        for b in batches if batches is not None else [R]:
            if len(b["pos"]):
                ctx.pileup_push(b)
        n0 = ctx.launch_count()
        ctx.pileup_sort()
        return ctx.reads(), ctx.launch_count() - n0


def short_and_long(L, seed, cov=4, n_long=60):
    fa = synth.make_fasta(L, seed)
    short, _ = synth.make_reads(L, seed, fa, coverage=cov, n_events=2, lens=(3000, 8000))
    return synth.merge_reads(short, synth.make_long_reads(L, n_long, seed + 1, max_ops=60, max_len=3000, max_skip=20_000))


# ---- the sort of staged reads
def check_sort(lib, R, seed, L=None):
    """R shuffled by a seeded permutation, pushed whole and in uneven batches, sorted: every field must equal the stable sort"""
    perm = np.random.default_rng(seed).permutation(len(R["pos"]))
    S = synth.take_reads(R, perm)
    want = stable_sorted(S)
    for batches in (None, split_reads(S, uneven_cuts(len(S["pos"]), seed))):
        got, _ = sort_staged(lib, S, batches, L)
        assert_same_reads(got, want)


def test_sort_short_and_long_reads(sim_lib):
    check_sort(sim_lib, short_and_long(400_000, 3), 3)


def test_sort_is_stable_on_one_position(sim_lib):
    """5000 reads on one position, distinct flag and isize, among reads elsewhere: ties keep their staging order"""
    R = short_and_long(200_000, 4, cov=1, n_long=10)
    n = 5000
    stack = synth.make_long_reads(200_000, n, 9, max_ops=3, max_len=150)
    stack["pos"][:] = 77_777
    stack["flag"] = np.arange(n, dtype=np.uint16)
    stack["isize"] = np.arange(n, dtype=np.int32) * 7 - 3
    S = synth.take_reads(synth.merge_reads(stack, R), np.random.default_rng(4).permutation(n + len(R["pos"])))
    got, _ = sort_staged(sim_lib, S)
    assert_same_reads(got, stable_sorted(S))
    at = got["pos"] == 77_777
    assert np.array_equal(got["flag"][at], S["flag"][S["pos"] == 77_777])


def test_sort_positions_up_to_2_31(sim_lib):
    """a long, sparse contig: positions up to 2^31 - 2 need every radix pass"""
    L = (1 << 31) - 1
    rng = np.random.default_rng(6)
    R = synth.make_long_reads(1_000_000, 3000, 6, max_ops=4, max_len=200, max_skip=1000)
    pos = rng.integers(0, L, len(R["pos"])).astype(np.int64)
    pos[:4] = [L - 1, 0, L - 1, (1 << 24) + 5]
    pos[4:40] = rng.integers(0, 256, 36)            # differ only in the low byte
    pos[40:80] = (rng.integers(0, 128, 40) << 24) | 0x00abcdef   # differ only in the high byte
    R["pos"] = pos.astype(np.int32)
    got, _ = sort_staged(sim_lib, R, L=L)
    assert_same_reads(got, stable_sorted(R))


def test_sort_empty_one_and_sorted(sim_lib):
    R = short_and_long(300_000, 5, cov=2, n_long=20)
    for n in (0, 1):
        one = synth.take_reads(R, np.arange(n))
        got, launches = sort_staged(sim_lib, one, L=300_000)
        assert_same_reads(got, one)
        assert launches == 0
    got, launches = sort_staged(sim_lib, R, split_reads(R, uneven_cuts(len(R["pos"]), 5)))
    assert_same_reads(got, R)
    assert launches == 1, "already-sorted reads must cost only the sortedness check"


def test_reads_take_between_contexts(sim_lib):
    R = short_and_long(300_000, 6, cov=2, n_long=20)
    fa = synth.make_fasta(300_000, 6)
    n = len(R["pos"])
    cuts = [0, 7, n // 3, n // 3, n - 1, n]
    with api.Context(lib=sim_lib) as src, api.Context(lib=sim_lib) as dst:
        src.reads_begin(5, 300_000)
        src.pileup_push(R)
        dst.set_reference(fa); dst.pileup_begin()
        for a, b in reversed(list(zip(cuts[:-1], cuts[1:]))):
            src.reads_take(a, b, dst)
        want = synth.take_reads(R, np.concatenate([np.arange(a, b) for a, b in reversed(list(zip(cuts[:-1], cuts[1:])))]))
        assert_same_reads(dst.reads(), want)
        with pytest.raises(api.RsiGpuError) as e:
            src.reads_take(0, n + 1, dst)
        assert e.value.code == 2 and "outside" in str(e.value)
        with pytest.raises(api.RsiGpuError) as e:
            src.reads_take(0, 1, src)
        assert e.value.code == 2 and "same context" in str(e.value)


# ---- the decoder grouping records by refID
CONTIGS = [("1", 60_000), ("2", 5_000), ("3", 90_000), ("MT", 20_000)]


def unsorted_file(path, kind, seed, rich=None, contigs=CONTIGS, tids=(0, 2, 3), covs=(6, 6, 3), n_mid=0, n_tail=0):
    """the reads of several contigs interleaved: kind "pairs" keeps two consecutive reads of a contig together and shuffles
    those pairs (like a name-ordered file's mates), "shuffled" shuffles every record; n_mid unplaced records anywhere in
    the file, n_tail at its end.  Returns {tid: that contig's reads in file order}."""
    rng = np.random.default_rng(seed)
    units = []
    src = {}
    for t, cov in zip(tids, covs):
        L = contigs[t][1]
        R = synth.make_reads(L, seed + t, synth.make_fasta(L, seed + t), coverage=cov, n_events=1, lens=(1000,), tid=t)[0]
        src[t] = R
        n = len(R["pos"])
        step = 2 if kind == "pairs" else 1
        units += [(t, np.arange(i, min(n, i + step))) for i in range(0, n, step)]
    units += [(-1, np.zeros(1, np.int64))] * n_mid
    units = [units[i] for i in rng.permutation(len(units))]
    order = np.concatenate([np.full(len(ix), t) for t, ix in units] + [np.full(n_tail, -1)])
    file_reads = {t: synth.take_reads(src[t], np.concatenate([ix for u, ix in units if u == t])) for t in src}
    synth.write_bam_unsorted(path, contigs, file_reads, order, random_seq=seed, rich=rich)
    return file_reads


def decode_by_ref(lib, path, feed_limit=None, crc=False):
    """feed the whole file with records grouped by refID; returns ({tid: reads over all feeds}, [[tids of each feed's runs]])"""
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    parts, feeds = {}, []
    with api.Context(lib=lib) as ctx:
        ctx.set_bam_by_ref(True)
        if crc:
            ctx.set_bgzf_crc(True)
        if feed_limit:
            ctx.set_feed_limit(feed_limit)
        ctx.bam_begin(len(h["names"]))
        off, first = h["coff"], True
        while off < len(data):
            consumed, runs = ctx.bam_feed(data[off:], skip=h["skip"] if first else 0)
            assert consumed > 0
            first = False; off += consumed
            feeds.append([t for t, _ in runs])
            for i, (t, n) in enumerate(runs):
                r = ctx.bam_run_reads(i)
                assert len(r["pos"]) == n
                parts.setdefault(t, []).append(r)
        ctx.bam_end()
    return {t: concat_reads(v) for t, v in parts.items()}, feeds


def concat_reads(rs):
    out = {k: np.concatenate([r[k] for r in rs]) for k in ("pos", "mpos", "isize", "mtid", "flag", "mapq", "cigar", "qual")}
    co, qo = [np.zeros(1, np.int64)], [np.zeros(1, np.int64)]
    for r in rs:
        co.append(r["cigar_off"][1:].astype(np.int64) + co[-1][-1]); qo.append(r["qual_off"][1:].astype(np.int64) + qo[-1][-1])
    out["cigar_off"] = np.concatenate(co).astype(np.uint32); out["qual_off"] = np.concatenate(qo).astype(np.uint64)
    return out


def check_by_ref(lib, path, feed_limit=None, crc=False):
    got, feeds = decode_by_ref(lib, path, feed_limit, crc)
    want = oracle_bam_decode(np.fromfile(path, np.uint8))["reads"]
    assert sorted(got) == sorted(want)
    for t in want:
        assert_same_reads(got[t], want[t])
    for f in feeds:     # one run per refID present, ascending, unplaced last
        key = [t if t >= 0 else 1 << 30 for t in f]
        assert key == sorted(set(key)), f
    return feeds


@pytest.mark.parametrize("mode", MODES, ids=MODE_IDS)
@pytest.mark.parametrize("kind,rich,n_mid,n_tail", [("pairs", None, 0, 0), ("shuffled", None, 40, 25), ("pairs", 3, 7, 0)],
                         ids=["pairs", "shuffled-unplaced", "pairs-rich"])
@pytest.mark.parametrize("feed_limit,crc", [(None, False), (1 << 16, False), (3 << 16, True)], ids=["whole", "carried", "carried-crc"])
def test_decode_by_ref(sim_lib, tmp_path, monkeypatch, mode, kind, rich, n_mid, n_tail, feed_limit, crc):
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    path = str(tmp_path / "u.bam")
    unsorted_file(path, kind, 11, rich=rich, n_mid=n_mid, n_tail=n_tail)
    feeds = check_by_ref(sim_lib, path, feed_limit, crc)
    assert (len(feeds) > 3) == (feed_limit is not None)


def test_decode_by_ref_3000_references(sim_lib, tmp_path):
    contigs = [(f"chrUn_{k}.1", 3000 + k) for k in range(3000)]
    contigs[17] = ("17", 40_000); contigs[2999] = ("last", 30_000); contigs[1500] = ("mid", 20_000)
    path = str(tmp_path / "many.bam")
    unsorted_file(path, "shuffled", 12, contigs=contigs, tids=(17, 1500, 2999), covs=(3, 3, 3), n_mid=5, n_tail=2)
    feeds = check_by_ref(sim_lib, path, 1 << 16)
    assert any(len(f) >= 3 for f in feeds)


def test_without_by_ref_an_unsorted_file_still_fails(sim_lib, tmp_path):
    path = str(tmp_path / "u.bam")
    unsorted_file(path, "shuffled", 13, covs=(200, 200, 200))
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    with api.Context(lib=sim_lib) as ctx:
        ctx.bam_begin(len(h["names"]))
        with pytest.raises(api.RsiGpuError) as e:
            ctx.bam_feed(data[h["coff"]:], skip=h["skip"])
        assert e.value.code == 3 and "not coordinate-sorted" in str(e.value)


# ---- refusals
def test_by_ref_refusals(sim_lib, tmp_path):
    path = str(tmp_path / "u.bam")
    unsorted_file(path, "pairs", 14)
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    with api.Context(lib=sim_lib) as ctx, api.Context(lib=sim_lib) as dst:
        ctx.set_bam_by_ref(True)
        ctx.bam_begin(len(h["names"]))
        with pytest.raises(api.RsiGpuError) as e:
            ctx.bam_index_begin(h["coff"])
        assert e.value.code == 2 and "grouped by refID" in str(e.value)
        with pytest.raises(api.RsiGpuError) as e:
            ctx.bam_feed_parts([data[h["coff"]:]])
        assert e.value.code == 2 and "grouped by refID" in str(e.value)
        _, runs = ctx.bam_feed(data[h["coff"]:], skip=h["skip"])
        dst.reads_begin(0, 60_000)
        with pytest.raises(api.RsiGpuError) as e:
            ctx.bam_take_range(0, dst, 0, 1000)
        assert e.value.code == 2 and "positions are not sorted" in str(e.value)
        ctx.bam_take(0, dst)           # a whole run is fine
        assert len(dst.reads()["pos"]) == runs[0][1]
        ctx.bam_end()
    with api.Context(lib=sim_lib) as ctx:   # indexing first, by-ref second
        ctx.bam_begin(3); ctx.bam_index_begin(0)
        with pytest.raises(api.RsiGpuError) as e:
            ctx.set_bam_by_ref(True)
        assert e.value.code == 2 and "index" in str(e.value)
    with api.Context(lib=sim_lib) as ctx:   # more than 65535 references, either order
        ctx.set_bam_by_ref(True)
        with pytest.raises(api.RsiGpuError) as e:
            ctx.bam_begin(65_536)
        assert e.value.code == 2 and "65535" in str(e.value)
        ctx.set_bam_by_ref(False); ctx.bam_begin(65_536)
        with pytest.raises(api.RsiGpuError) as e:
            ctx.set_bam_by_ref(True)
        assert e.value.code == 2 and "65535" in str(e.value)
        ctx.bam_begin(65_535); ctx.set_bam_by_ref(True)


# ---- the whole path: shuffled file -> by-ref decode -> staging -> reads_take -> pileup_sort -> run, against the sorted file
WHOLE = [("1", 10_600_000), ("2", 3_000), ("3", 1_200_000)]


def stage_by_ref(lib, path, feed_limit=None):
    """decode with records grouped by refID into one staging context; returns (staging context, {tid: [(r0, r1)]})"""
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    stage = api.Context(lib=lib)
    seg = {}
    with api.Context(lib=lib) as dec:
        dec.set_bam_by_ref(True)
        if feed_limit:
            dec.set_feed_limit(feed_limit)
        stage.reads_begin(0, 1000)
        dec.bam_begin(len(h["names"]))
        off, first = h["coff"], True
        while off < len(data):
            consumed, runs = dec.bam_feed(data[off:], skip=h["skip"] if first else 0)
            first = False; off += consumed
            for i, (t, n) in enumerate(runs):
                if t >= 0:
                    r0 = stage_count(stage)
                    dec.bam_take(i, stage)
                    seg.setdefault(t, []).append((r0, r0 + n))
        dec.bam_end()
    return stage, seg


def stage_count(ctx):
    """number of staged reads: the size of field 0 (pos)"""
    import ctypes as C
    nb = C.c_int64(0)
    ctx._ck(ctx.lib.rsigpu_reads_field(ctx.h, C.c_int32(0), None, C.c_int64(0), C.byref(nb)))
    return nb.value // 4


def take_sorted(lib, path, tid, dst):
    """the existing route: the coordinate-sorted file decoded in file order, the runs of `tid` taken into dst"""
    data = np.fromfile(path, np.uint8)
    h = api.parse_bam_header(data)
    with api.Context(lib=lib) as dec:
        dec.bam_begin(len(h["names"]))
        _, runs = dec.bam_feed(data[h["coff"]:], skip=h["skip"])
        for i, (t, _) in enumerate(runs):
            if t == tid:
                dec.bam_take(i, dst)
        dec.bam_end()


def run_contig(lib, fa, tid, name, fill, kw):
    with api.Context(lib=lib, **kw) as ctx:
        ctx.set_reference(fa, tid); ctx.pileup_begin()
        fill(ctx)
        ctx.pileup_end()
        raw = ctx.array(api.ARR_RAW_DEPTH).tobytes()
        calls = ctx.run()
        snap = _snapshot(ctx, calls)
        snap["raw"] = raw
        snap["log"] = ctx.log_text(name, False)
        return snap, calls


@pytest.fixture(scope="module")
def whole_files(tmp_path_factory):
    d = tmp_path_factory.mktemp("whole")
    rng = np.random.default_rng(21)
    reads, fas = {}, {}
    for t, (name, L) in enumerate(WHOLE):
        if L < 10_000:
            continue
        fas[t] = synth.make_fasta(L, 21 + t)
        reads[t] = synth.make_reads(L, 21 + t, fas[t], coverage=8 if t == 0 else 5, n_events=5 if t == 0 else 1,
                                    lens=(3000, 8000, 20000), tid=t)[0]
    units = [(t, i) for t in reads for i in range(len(reads[t]["pos"]))] + [(-1, 0)] * 30
    units = [units[i] for i in rng.permutation(len(units))]
    order = np.array([t for t, _ in units])
    file_reads = {t: synth.take_reads(reads[t], np.array([i for u, i in units if u == t])) for t in reads}
    shuffled_path = str(d / "shuffled.bam")
    synth.write_bam_unsorted(shuffled_path, WHOLE, file_reads, order, random_seq=3)
    # the reference: the shuffled file after a stable coordinate sort (ties in shuffled-file order), through the sorted route
    sorted_path = str(d / "sorted.bam")
    synth.write_bam(sorted_path, WHOLE, {t: stable_sorted(R) for t, R in file_reads.items()}, random_seq=3, unmapped_tail=30)
    return sorted_path, shuffled_path, fas, reads


def test_whole_path_shuffled_equals_sorted(sim_lib, whole_files):
    check_whole_path(sim_lib, whole_files)


def check_whole_path(lib, whole_files):
    sorted_path, shuffled_path, fas, reads = whole_files
    kw = dict(minq=0, min_baseQ=10)
    stage, seg = stage_by_ref(lib, shuffled_path, feed_limit=8 << 20)
    try:
        for t, fa in fas.items():
            def from_stage(ctx):
                for r0, r1 in seg[t]:
                    stage.reads_take(r0, r1, ctx)
                ctx.pileup_sort()
            got, calls = run_contig(lib, fa, t, WHOLE[t][0], from_stage, kw)
            want, _ = run_contig(lib, fa, t, WHOLE[t][0], lambda ctx: take_sorted(lib, sorted_path, t, ctx), kw)
            assert got == want, f"contig {t}"
            if t == 0:
                assert len(calls) >= 3 and any(c.rp > 0 for c in calls)
        # `stat`: RP / Q0 of a call list on the sorted staged reads
        with api.Context(lib=lib) as ctx:
            ctx.reads_begin(0, WHOLE[0][1])
            for r0, r1 in seg[0]:
                stage.reads_take(r0, r1, ctx)
            ctx.pileup_sort()
            got = [bytes(c) for c in ctx.stat_calls(calls)]
        with api.Context(lib=lib) as ctx:
            ctx.reads_begin(0, WHOLE[0][1]); take_sorted(lib, sorted_path, 0, ctx)
            assert got == [bytes(c) for c in ctx.stat_calls(calls)]
    finally:
        stage.close()
