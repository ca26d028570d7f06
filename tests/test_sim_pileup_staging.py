"""Pileup (k_pileup.cuh) against oracle_pileup on the inputs that any staging of k_pileup_tile's reads in shared memory
(fields, CIGAR words and pass-mask words copied per chunk of a tile's reads) has to get right, in the CPU emulator: tiles
whose reads span many 256-read chunks, reads whose CIGAR or mask words exceed 4 KB among short reads, quality offsets that
are not monotonic, array ranges starting at every residue mod 16 bytes, a contig length that is not a multiple of the
tile, reads at the edges of 4096-base tiles, and a split run."""
import numpy as np
import pytest

from bind import oracle_pileup
from test_sim_long_reads import EQ, I, M, S, _split_vs_whole, assert_depth, explicit_reads, pileup
from rsicnv_b200 import synth

L_ODD = 100_003          # not a multiple of the 4096- or 8192-base tile
MINQ, Q = 0, 13


def short_reads(L, seed, coverage=30.0):
    fa = synth.make_fasta(L, seed)
    reads, _ = synth.make_reads(L, seed, fa, coverage=coverage, events=[])
    return fa, reads


def overflow_reads(L, seed):
    """reads with more than 1024 CIGAR words or 1024 mask words (4 KB each), one with 282 mask words, one reaching past L"""
    rng = np.random.default_rng(seed)
    q = lambda n: rng.integers(0, 40, n)
    items = [(L // 3, [(40_000, M)], q(40_000), 0, 60),                                  # 1250 mask words
             (L // 3 + 5, [(3, S)] + [(1, M), (1, I)] * 750 + [(20, EQ)], q(1523), 0, 60),  # 1502 CIGAR words
             (L // 2 + 17, [(9_000, M)], q(9_000), 0, 60),                               # 282 mask words
             (L - 50, [(60, M)], q(60), 0, 60)]                                           # reaches past L
    return explicit_reads(items)


def want_depth(oracle, reads, L):
    oracle.set_params(minq=MINQ, min_baseQ=Q)
    return oracle_pileup(oracle, reads, L)


def check(lib, oracle, fa, reads, what):
    assert_depth(pileup(lib, fa, reads, MINQ, Q), want_depth(oracle, reads, len(fa)), what)


def case_many_chunks(lib, oracle, L=L_ODD):
    fa, reads = short_reads(L, 31)
    assert len(reads["pos"]) / ((L + 4095) // 4096) > 2 * 256    # every 4096-base tile has more than 512 reads
    check(lib, oracle, fa, reads, "30x short reads")


def case_overflow(lib, oracle, L=L_ODD):
    fa, short = short_reads(L, 32)
    check(lib, oracle, fa, synth.merge_reads(short, overflow_reads(L, 32)), "short reads + reads larger than a stage")


def case_nonmonotonic_qual_offsets(lib, oracle, L=L_ODD):
    """the reads' quality blocks laid out in a shuffled order: qual_off[r] still starts read r's block, but qual_off[b] of a
    chunk's end no longer bounds the blocks of the chunk's reads"""
    fa, short = short_reads(L, 33)
    reads = synth.merge_reads(short, overflow_reads(L, 33))
    qo = reads["qual_off"].astype(np.int64)
    n = len(reads["pos"])
    order = np.random.default_rng(33).permutation(n)
    ln = qo[1:] - qo[:-1]
    start = np.zeros(n, np.int64)
    start[order] = np.concatenate(([0], np.cumsum(ln[order])[:-1]))
    reads = dict(reads)
    reads["qual"] = np.concatenate([reads["qual"][qo[r]:qo[r + 1]] for r in order])
    reads["qual_off"] = np.concatenate((start, [qo[-1]])).astype(np.uint64)
    assert np.any(np.diff(reads["qual_off"].astype(np.int64)) < 0)
    check(lib, oracle, fa, reads, "shuffled quality blocks")


def case_residues(lib, oracle, L=20_011):
    """k unplaced reads (pos 0: not counted) in front shift the field, CIGAR and quality ranges by k elements, k CIGAR words
    and 37k quality bytes: every start residue mod 16 bytes of every staged array"""
    fa, short = short_reads(L, 34, coverage=40)
    for k in range(16):
        pad = explicit_reads([(0, [(37, S)], 20, 0, 60)] * k) if k else None
        reads = synth.merge_reads(pad, short) if k else short
        check(lib, oracle, fa, reads, f"{k} reads in front")


def case_tile_edges(lib, oracle, L=L_ODD, T=4096):
    """ops ending exactly at a 4096-base tile end, one op covering a whole tile and one base on each side, among short reads"""
    fa, short = short_reads(L, 36, coverage=10)
    items = []
    for k in range(1, L // T + 1):
        for ln in (1, 100, T):
            if k * T - ln > 0:
                items.append((k * T - ln, [(ln, M)], 30, 0, 60))
        if (k + 1) * T + 1 <= L:
            items.append((k * T - 1, [(T + 2, M)], 30, 0, 60))
            items.append((k * T - 1, [(3, S), (T + 2, EQ), (2, S)], 30, 0, 60))
    items.sort(key=lambda t: t[0])
    check(lib, oracle, fa, synth.merge_reads(short, explicit_reads(items)), "reads at 4096-base tile edges")


def case_split(lib, nparts):
    L = 1_000_003
    fa, short = short_reads(L, 35, coverage=6)
    got, want = _split_vs_whole(lib, fa, synth.merge_reads(short, overflow_reads(L, 35)), nparts, dict(minq=MINQ, min_baseQ=Q))
    assert got == want


def test_many_chunks(sim_lib, oracle):
    case_many_chunks(sim_lib, oracle)


def test_overflow_among_short_reads(sim_lib, oracle):
    case_overflow(sim_lib, oracle)


def test_nonmonotonic_qual_offsets(sim_lib, oracle):
    case_nonmonotonic_qual_offsets(sim_lib, oracle)


def test_start_residues(sim_lib, oracle):
    case_residues(sim_lib, oracle)


def test_tile_edges(sim_lib, oracle):
    case_tile_edges(sim_lib, oracle)


@pytest.mark.parametrize("nparts", [2, 3])
def test_split_run(sim_lib, nparts):
    case_split(sim_lib, nparts)
