"""The read path on reads that do not look like make_reads' 2x100 bp pairs, in the CPU emulator: long reads, spliced reads
(RNA-seq style N gaps), reads with hundreds of CIGAR ops of every type.  Pileup (k_pileup.cuh) against oracle_pileup at the
edges of its 128-base mask chunks and 8192-base tiles, the whole BAM path with a reach (max_extent) of hundreds of kb, the
BAM decoder on records of hundreds of KB carried across many feeds, and the read halo of split mode at its exact bound."""
import numpy as np
import pytest

from bind import oracle_pileup
from common import run_bam_case, split_reads
from rsicnv_b200 import api, synth
from test_sim_bam_decode import assert_same_reads, decode_file
from test_sim_bam_index import build_index, expected
from test_sim_split import _snapshot

M, I, D, N, S, H, P, EQ, X = range(9)
THRESHOLDS = pytest.mark.parametrize("minq,Q", [(0, 0), (0, 13), (20, 0), (1, 128), (0, 255)])
MODES = [1, 2]


def explicit_reads(items, tid=0):
    """[(pos, [(len, op), ...], qualities (an int for all of them, or an array), flag, mapq)] in the given order -> read SoA"""
    pos, flag, mapq, cig, qual, co, qo = [], [], [], [], [], [0], [0]
    for p, ops, q, fl, mq in items:
        nq = sum(l for l, o in ops if o in (M, I, S, EQ, X))
        qa = np.full(nq, q, np.uint8) if np.isscalar(q) else np.asarray(q, np.uint8)
        assert len(qa) == nq
        pos.append(p); flag.append(fl); mapq.append(mq); qual.append(qa)
        cig += [(l << 4) | o for l, o in ops]; co.append(len(cig)); qo.append(qo[-1] + nq)
    n = len(pos)
    return dict(pos=np.asarray(pos, np.int32), mpos=np.asarray(pos, np.int32), isize=np.zeros(n, np.int32), mtid=np.full(n, tid, np.int32),
                flag=np.asarray(flag, np.uint16), mapq=np.asarray(mapq, np.uint8), cigar_off=np.asarray(co, np.uint32),
                cigar=np.asarray(cig, np.uint32), qual_off=np.asarray(qo, np.uint64),
                qual=np.concatenate(qual) if qual else np.zeros(0, np.uint8))


def uneven_cuts(n, seed):
    """batch boundaries: a few random ones, the first and the last read alone, and a run of 1-read batches"""
    rng = np.random.default_rng(seed)
    cuts = set(int(x) for x in rng.integers(1, n, 6)) | {1, n - 1}
    k = int(rng.integers(1, max(2, n - 8)))
    cuts |= set(range(k, min(n, k + 8)))
    return sorted(c for c in cuts if 0 < c < n)


def pileup(lib, fa, reads, minq, Q, batches=None):
    with api.Context(lib=lib, minq=minq, min_baseQ=Q) as ctx:
        ctx.set_reference(fa); ctx.pileup_begin()
        for b in batches if batches is not None else [reads]:
            ctx.pileup_push(b)
        ctx.pileup_end()
        return ctx.array(api.ARR_RAW_DEPTH)


def assert_depth(got, want, what):
    bad = np.flatnonzero(got != want)
    assert len(bad) == 0, f"{what}: {len(bad)} positions differ, first {bad[:5].tolist()}: got {got[bad[:5]].tolist()} want {want[bad[:5]].tolist()}"


def check_pileup(lib, oracle, L, reads, minq, Q, seed=0):
    """whole and in uneven batches, against the oracle; returns the oracle's depth"""
    fa = synth.make_fasta(L, 8)
    oracle.set_params(minq=minq, min_baseQ=Q)
    want = oracle_pileup(oracle, reads, L)
    assert_depth(pileup(lib, fa, reads, minq, Q), want, "pushed whole")
    assert_depth(pileup(lib, fa, reads, minq, Q, split_reads(reads, uneven_cuts(len(reads["pos"]), seed))), want, "pushed in batches")
    return want


# ---- pileup: random long / spliced / many-op reads
@THRESHOLDS
@pytest.mark.parametrize("L,n,seed,kw", [(2_000_000, 300, 1, {}), (300_000, 200, 2, dict(max_len=20_000, max_skip=100_000))],
                         ids=["2Mbp", "300kbp-dense"])
def test_pileup_random_long_reads(sim_lib, oracle, L, n, seed, kw, minq, Q):
    reads = synth.make_long_reads(L, n, seed, **kw)
    ops = reads["cigar"] & 15
    assert set(np.unique(ops).tolist()) == set(range(9)) and np.any((reads["cigar"] >> 4) == 0)
    assert np.any(reads["pos"] == 0) and np.any(reads["pos"] == L - 1)
    want = check_pileup(sim_lib, oracle, L, reads, minq, Q, seed)
    assert want.sum() > 0


# ---- pileup: deterministic edges of the mask chunks (128 bases) and tiles (8192 bases)
def edge_reads(L):
    T = 8192
    items = []                                  # (pos, ops, qualities, flag, mapq, residue of the quality offset mod 32 or None)
    p = 1000
    for ln in (127, 128, 129, 255, 256, 8193):   # runs crossing chunk ends, the quality offset at every residue mod 32
        for res in range(32):
            items.append((p, [(ln, M)], 255, 0, 60, res)); p += 301
    for k in range(1, L // T + 1):              # ops ending exactly at a tile end, one op covering a whole tile and one base on each side
        for ln in (1, 100, T):
            if k * T - ln > 0:
                items.append((k * T - ln, [(ln, M)], 255, 0, 60, None))
        if (k + 1) * T + 1 <= L:
            items.append((k * T - 1, [(T + 2, M)], 255, 0, 60, None))
            items.append((k * T - 1, [(3, S), (T + 2, EQ), (2, S)], 255, 0, 60, None))
        if k * T - 2050 > 0:
            items.append((k * T - 2050, [(3, H), (7, S), (50, M), (1000, N), (1000, M)], 255, 0, 60, None))
            items.append((k * T - 2000, [(2, P), (1, I), (1000, M), (4, S), (996, M), (5, D), (0, M)], 255, 0, 60, None))
    for ln in (1, 100, 129):                    # ending at L, and one base past it
        items.append((L - ln, [(ln, M)], 255, 0, 60, None)); items.append((L - ln + 1, [(ln, M)], 255, 0, 60, None))
    items.append((L - 1, [(4, S), (1, M), (300, N), (1, M)], 255, 0, 60, None))
    rng = np.random.default_rng(5)
    for r in range(5000):                       # 5000 reads stacked on one position
        ops = [(120, M)] if r % 3 else [(int(rng.integers(0, 30)), S), (60, M), (2, I), (58, M)]
        nq = sum(l for l, o in ops if o in (M, I, S, EQ, X))
        items.append((30_001, ops, rng.integers(0, 256, nq), int(rng.choice([0, 0, 0, 1024, 256])), int(rng.integers(0, 61)), None))
    items.sort(key=lambda t: t[0])
    out, q = [], 0
    for p, ops, qv, fl, mq, res in items:
        if res is not None:                     # a spacer read in front: only a soft clip, nothing counted
            k = (res - q) % 32
            out.append((p, [(k, S)], 255, 0, 60)); q += k
        out.append((p, ops, qv, fl, mq)); q += sum(l for l, o in ops if o in (M, I, S, EQ, X))
    return explicit_reads(out)


@THRESHOLDS
@pytest.mark.parametrize("L", [12 * 8192, 12 * 8192 + 77])
def test_pileup_chunk_and_tile_edges(sim_lib, oracle, L, minq, Q):
    reads = edge_reads(L)
    assert np.all(np.diff(reads["pos"]) >= 0)
    want = check_pileup(sim_lib, oracle, L, reads, minq, Q, 3)
    assert want.sum() > 0


def eq_reach_reads():
    """'=' ops count bases without advancing the reference coordinate: a read's reach is its M/D/N/S span from the first
    M/D/=/X op plus its longest '=' op.  Here only '=' ops reach past the next tile; the other reads are 50 bases long."""
    items = [(100, [(1, M), (30_000, EQ)], 255, 0, 60), (200, [(4, S), (20_000, EQ)], 255, 0, 60),
             (9000, [(10, EQ), (3, I), (25_000, EQ), (2, M)], 255, 0, 60), (9100, [(5, X), (40_000, EQ), (1, S)], 255, 0, 60)]
    items += [(p, [(50, M)], 30, 0, 60) for p in range(300, 70_000 - 100, 997)]
    items.sort(key=lambda t: t[0])
    return 70_000, explicit_reads(items)


@THRESHOLDS
def test_pileup_reach_of_eq_ops(sim_lib, oracle, minq, Q):
    L, reads = eq_reach_reads()
    assert check_pileup(sim_lib, oracle, L, reads, minq, Q, 4)[40_000] > 0


# ---- the whole BAM path with long and spliced reads among the short ones
def long_and_spliced(L, seed):
    """short read pairs with 5 % more reads: spliced ones (N gaps up to 500 kb) and long ones with up to 40 ops"""
    fa = synth.make_fasta(L, seed)
    short, _ = synth.make_reads(L, seed, fa, coverage=12, n_events=6, lens=(3000, 8000, 20000))
    n_long = len(short["pos"]) // 20
    spliced = synth.make_long_reads(L, n_long * 4 // 5, seed + 1, max_ops=8, max_len=300, max_skip=500_000, min_len=20)
    long = synth.make_long_reads(L, n_long // 5, seed + 2, max_ops=40, max_len=3000, max_skip=20_000)
    return fa, synth.merge_reads(short, spliced, long)


def test_bam_path_with_long_and_spliced_reads(sim_lib, oracle):
    fa, reads = long_and_spliced(10_600_000, 5)
    calls, st = run_bam_case(sim_lib, oracle, fa, reads, n_batches=5, minq=0, min_baseQ=13)
    assert len(calls) > 0 and st.isize_mean > 0


# ---- decode: records of hundreds of KB with hundreds of ops, carried across many feeds
@pytest.fixture(scope="module")
def long_bam(tmp_path_factory):
    L = 400_000
    bg, _ = synth.make_reads(L, 3, None, coverage=0.5, n_events=0)
    reads = synth.merge_reads(bg, synth.make_long_reads(L, 10, 3))
    path = str(tmp_path_factory.mktemp("long") / "long.bam")
    synth.write_bam(path, [("1", L)], {0: reads}, level=1, random_seq=7)
    size = 36 + 2 + 4 * np.diff(reads["cigar_off"].astype(np.int64)) + np.diff(reads["qual_off"].astype(np.int64)) * 3 // 2
    assert size.max() > 300_000 and np.diff(reads["cigar_off"].astype(np.int64)).max() > 150
    return path, reads


@pytest.mark.parametrize("mode", MODES, ids=["lane-per-block", "warp-per-block"])
@pytest.mark.parametrize("chunk", [None, 30_000, 70_001, 1 << 20])
def test_decode_long_records(sim_lib, long_bam, monkeypatch, mode, chunk):
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    path, reads = long_bam
    got, _ = decode_file(sim_lib, path, chunk)
    assert sorted(got) == [0]
    assert_same_reads(got[0], reads)


@pytest.mark.parametrize("mode", MODES, ids=["lane-per-block", "warp-per-block"])
def test_decode_long_records_with_crc(sim_lib, long_bam, monkeypatch, mode):
    monkeypatch.setenv("RSIGPU_INFLATE_MODE", str(mode))
    monkeypatch.setenv("RSIGPU_BGZF_CRC", "1")
    path, reads = long_bam
    got, _ = decode_file(sim_lib, path, 30_000)
    assert_same_reads(got[0], reads)


@pytest.mark.parametrize("mode", MODES, ids=["lane-per-block", "warp-per-block"])
@pytest.mark.parametrize("chunk,crc", [(None, False), (30_000, False), (70_001, True)])
def test_index_long_records(sim_lib, long_bam, mode, chunk, crc):
    """the begin offset of a record carried across several feeds is the one of the feed it started in"""
    path, _ = long_bam
    assert build_index(sim_lib, path, mode, chunk, crc=crc) == expected(path)


# ---- split mode: the read halo of 65536 bases is an exact bound
def halo_reads(cuts, reach):
    """reads of M and N ops only (their reach is exactly their M + N span) placed so that they end just before, at and just
    after each cut"""
    items = []
    for c in cuts:
        for d in (0, 1, 2, 700):
            p = c - 65_536 + d
            for ops in ([(reach, M)], [(100, M), (reach - 200, N), (100, M)], [(1, M), (reach - 2, N), (1, M)],
                        [(30_000, M), (reach - 60_000, N), (30_000, M)]):
                items.append((p, ops, 30, 0, 60))
    items.sort(key=lambda t: t[0])
    return explicit_reads(items)


def _split_vs_whole(lib, fa, reads, nparts, kw):
    with api.Context(lib=lib, **kw) as c0:
        c0.set_reference(fa); c0.pileup_begin(); c0.pileup_push(reads); c0.have_reads()
        want = _snapshot(c0, c0.run())
    parts = [api.Context(lib=lib, **kw) for _ in range(nparts)]
    try:
        for g, p in enumerate(parts):
            b, e, halo = api.split_range(p.lib, len(fa), nparts, g)
            p.set_reference(fa); p.pileup_begin(); p.pileup_push(api.split_reads(reads, b, e, halo)); p.have_reads()
        calls = api.split_run(parts)
        return _snapshot(parts[0], calls), want
    finally:
        for p in parts:
            p.close()


def test_split_reads_reaching_the_halo(sim_lib):
    L = 1_000_003
    fa = synth.make_fasta(L, 9)
    short, _ = synth.make_reads(L, 9, fa, coverage=6, n_events=4, lens=(3000, 8000, 20000))
    kw = dict(minq=0, min_baseQ=10)
    with api.Context(lib=sim_lib) as c:
        rng = [api.split_range(c.lib, L, 3, g) for g in range(3)]
    assert all(h == 65_536 for _, _, h in rng)
    reads = synth.merge_reads(short, halo_reads([rng[1][0], rng[2][0]], 65_536))
    got, want = _split_vs_whole(sim_lib, fa, reads, 3, kw)
    assert got == want and len(want["calls"]) >= 2
    # one base further and the halo no longer covers the read: refused, not a silently different depth
    reads = synth.merge_reads(short, halo_reads([rng[1][0]], 65_537))
    with pytest.raises(api.RsiGpuError) as e:
        _split_vs_whole(sim_lib, fa, reads, 3, kw)
    assert e.value.code == 3 and "65536" in str(e.value)
