"""Seeded synthetic inputs for the rsicnv `rsi` hot path (no network: every input is simulated).

Shapes follow SURVEY.md §8(d): a b37-shaped contig (uppercase ACGT with N blocks), an NB-like
per-base depth track with planted DEL/DUP segments, and 2x100 bp FR read pairs for the BAM path.
Nothing here is on the measured path; it only fabricates inputs for tests and bench.py.
"""
from __future__ import annotations

import numpy as np

CHR19_LEN = 59_128_983
B37_LENS = {
    "1": 249250621, "2": 243199373, "3": 198022430, "4": 191154276, "5": 180915260, "6": 171115067,
    "7": 159138663, "8": 146364022, "9": 141213431, "10": 135534747, "11": 135006516, "12": 133851895,
    "13": 115169878, "14": 107349540, "15": 102531392, "16": 90354753, "17": 81195210, "18": 78077248,
    "19": 59128983, "20": 63025520, "21": 48129895, "22": 51304566, "X": 155270560, "Y": 59373566,
}
EVENT_LENS = (2_000, 5_000, 10_000, 30_000, 100_000)


def n_blocks_for(L: int) -> list[tuple[int, int]]:
    """N blocks shaped like b37 chr19: telomere gap, centromere, tail (scaled for small L)."""
    if L >= 40_000_000:
        return [(0, 60_000), (int(L * 0.41657), int(L * 0.41657) + 3_100_000), (L - 10_000, L)]
    a = max(1000, L // 1000)
    c0 = int(L * 0.41657)
    return [(0, a), (c0, c0 + max(2000, L // 20)), (L - max(500, a // 6), L)]


def make_fasta(L: int, seed: int, n_blocks=None) -> np.ndarray:
    """uint8 ASCII contig; GC fraction drifts regionally (0.30..0.60) so that GC strata are populated."""
    rng = np.random.default_rng(seed)
    if n_blocks is None:
        n_blocks = n_blocks_for(L)
    seg = 5_000
    nseg = (L + seg - 1) // seg
    gcf = 0.45 + 0.15 * np.sin(np.arange(nseg) * 0.37 + seed) * rng.uniform(0.3, 1.0, nseg)
    p = np.repeat(gcf, seg)[:L].astype(np.float32)
    u = rng.random(L, dtype=np.float32)
    v = rng.integers(0, 2, L, dtype=np.uint8)
    is_gc = u < p
    out = np.where(is_gc, np.where(v == 0, ord("G"), ord("C")), np.where(v == 0, ord("A"), ord("T"))).astype(np.uint8)
    for a, b in n_blocks:
        out[a:b] = ord("N")
    return out


def plant_events(L: int, seed: int, n_events: int, n_blocks, lens=EVENT_LENS, margin=None):
    """Alternating DEL (x0.5) / DUP (x1.5) events away from N blocks and contig ends."""
    rng = np.random.default_rng(seed + 7)
    ev = []
    if n_events == 0:
        return ev
    margin = margin if margin is not None else max(3 * max(lens), L // 200)
    slots = np.linspace(margin, L - margin, n_events + 2)[1:-1]
    for k, c in enumerate(slots):
        ln = int(lens[k % len(lens)])
        s = int(c + rng.integers(-ln, ln))
        e = s + ln
        bad = any(s < b + 3 * ln and e > a - 3 * ln for a, b in n_blocks)
        if bad or s < margin or e > L - margin:
            continue
        ev.append((s, e, 0.5 if k % 2 == 0 else 1.5))
    return ev


def make_depth(L: int, seed: int, fasta: np.ndarray | None = None, n_events: int = 20, mean: float = 30.0,
               shape: float = 40.0, lens=EVENT_LENS, gc_bias: float = 0.25, events=None, block: int = 100):
    """NB-like depth: moving-average(100) of Poisson(Gamma(shape, mean) per `block` bases) with a mild GC bias,
    0 inside N blocks, planted copy-number events.  Returns (int32 depth, events)."""
    rng = np.random.default_rng(seed)
    if fasta is None:
        fasta = make_fasta(L, seed)
    n_blocks = _n_runs(fasta)
    if events is None:
        events = plant_events(L, seed, n_events, n_blocks, lens)
    nblk = (L + block - 1) // block
    lam = np.repeat(rng.gamma(shape, mean / shape, nblk).astype(np.float32), block)[:L].copy()
    cn = np.ones(L, np.float32)
    for s, e, f in events:
        cn[s:e] = f
    # regional GC effect (201-bp window GC fraction), multiplicative
    gc = ((fasta == ord("G")) | (fasta == ord("C"))).astype(np.float32)
    cs = np.concatenate(([0.0], np.cumsum(gc, dtype=np.float64)))
    w = 201
    lo = np.clip(np.arange(L) - w // 2, 0, max(L - w, 0))
    frac = ((cs[np.minimum(lo + w, L)] - cs[lo]) / w).astype(np.float32)
    lam *= cn * (1.0 + gc_bias * (frac - 0.45) / 0.15)
    np.maximum(lam, 0, out=lam)
    raw = rng.poisson(lam).astype(np.float64)
    k = 100
    c2 = np.concatenate(([0.0], np.cumsum(raw)))
    hi = np.minimum(np.arange(L) + k // 2, L)
    lo2 = np.maximum(np.arange(L) - k // 2, 0)
    d = np.rint((c2[hi] - c2[lo2]) / (hi - lo2)).astype(np.int32)
    d[fasta == ord("N")] = 0
    return d, events


def _n_runs(fasta: np.ndarray) -> list[tuple[int, int]]:
    isn = (fasta == ord("N")).astype(np.int8)
    d = np.diff(np.concatenate(([0], isn, [0])))
    return list(zip(np.flatnonzero(d == 1).tolist(), np.flatnonzero(d == -1).tolist()))


# --------------------------------------------------------------------------------------------
# files
def write_fasta(path: str, name: str, seq: np.ndarray, width: int = 60) -> None:
    L = len(seq)
    header = f">{name}\n".encode()
    nfull = L // width
    body = np.empty(L + nfull + (1 if L % width else 0), np.uint8)
    if nfull:
        blk = body[: nfull * (width + 1)].reshape(nfull, width + 1)
        blk[:, :width] = seq[: nfull * width].reshape(nfull, width)
        blk[:, width] = 10
    if L % width:
        body[nfull * (width + 1):-1] = seq[nfull * width:]
        body[-1] = 10
    with open(path, "wb") as f:
        f.write(header)
        f.write(body.tobytes())
    with open(path + ".fai", "w") as f:
        f.write(f"{name}\t{L}\t{len(header)}\t{width}\t{width + 1}\n")


def write_fasta_multi(path: str, contigs: list[tuple[str, np.ndarray]], width: int = 60) -> None:
    off = 0
    fai = []
    with open(path, "wb") as f:
        for name, seq in contigs:
            L = len(seq)
            header = f">{name}\n".encode()
            f.write(header)
            off += len(header)
            fai.append(f"{name}\t{L}\t{off}\t{width}\t{width + 1}\n")
            nfull = L // width
            body = np.empty(L + nfull + (1 if L % width else 0), np.uint8)
            if nfull:
                blk = body[: nfull * (width + 1)].reshape(nfull, width + 1)
                blk[:, :width] = seq[: nfull * width].reshape(nfull, width)
                blk[:, width] = 10
            if L % width:
                body[nfull * (width + 1):-1] = seq[nfull * width:]
                body[-1] = 10
            f.write(body.tobytes())
            off += len(body)
    with open(path + ".fai", "w") as f:
        f.writelines(fai)


def write_depth_file(path: str, depth: np.ndarray, chunk: int = 4_000_000) -> None:
    """`pos<TAB>depth` lines, 1-based (what `rsicnv rsi -s` writes: loaddata.cpp:464-470)."""
    with open(path, "wb") as f:
        for a in range(0, len(depth), chunk):
            d = depth[a:a + chunk]
            pos = np.arange(a + 1, a + 1 + len(d))
            f.write("\n".join(f"{p}\t{v}" for p, v in zip(pos.tolist(), d.tolist())).encode())
            f.write(b"\n")


def write_depth_file_fast(path: str, depth: np.ndarray, chunk: int = 8_000_000) -> None:
    """the same `pos<TAB>depth` file written with vectorised digit arithmetic (a chr19-sized file in seconds); the depth column is
    zero-padded to the width of the largest value -- `istream >> int` (loaddata.cpp:509) reads "030" as 30"""
    depth = np.asarray(depth)
    wd = max(1, len(str(int(depth.max(initial=0)))))
    assert depth.min(initial=0) >= 0
    with open(path, "wb") as f:
        L = len(depth)
        a = 0
        while a < L:
            # positions a+1 .. with the same number of digits
            p0 = a + 1
            wp = len(str(p0))
            b = min(L, a + chunk, 10 ** wp - 1)
            n = b - a
            pos = np.arange(p0, p0 + n, dtype=np.int64)
            d = depth[a:b].astype(np.int64)
            line = np.empty((n, wp + 1 + wd + 1), np.uint8)
            for k in range(wp):
                line[:, wp - 1 - k] = 48 + (pos // 10 ** k) % 10
            line[:, wp] = 9
            for k in range(wd):
                line[:, wp + wd - k] = 48 + (d // 10 ** k) % 10
            line[:, -1] = 10
            f.write(line.tobytes())
            a = b


def stress_events(L: int, seed: int, n_blocks) -> list[tuple[int, int, float]]:
    """Adversarial event layout for the candidate stage: same-type neighbours separated by short gaps
    (merge paths), nested copy-number levels (multi-level RSI status -> multisegments), weak events
    that fail the depth test, events hugging contig ends and N blocks."""
    rng = np.random.default_rng(seed + 101)
    ev: list[tuple[int, int, float]] = []
    free = []
    prev = 0
    for a, b in sorted(n_blocks) + [(L, L)]:
        if a - prev > 60_000:
            free.append((prev + 3_000, a - 3_000))
        prev = b
    factors = [0.5, 1.5, 0.0, 2.0, 0.8, 1.2, 0.65, 1.35]
    for lo, hi in free:
        p = lo + int(rng.integers(500, 4_000))
        while p < hi - 40_000:
            kind = int(rng.integers(0, 5))
            f = factors[int(rng.integers(0, len(factors)))]
            ln = int(rng.choice([600, 1200, 2500, 5000, 9000, 20000]))
            if kind == 0:      # isolated
                ev.append((p, p + ln, f)); p += ln
            elif kind == 1:    # two same-type events with a short gap
                g = int(rng.choice([150, 400, 900, 2500]))
                ev.append((p, p + ln, f)); ev.append((p + ln + g, p + 2 * ln + g, f)); p += 2 * ln + g
            elif kind == 2:    # nested: outer mild, inner strong
                inner = ln // 3
                ev.append((p, p + ln, 0.6 if f < 1 else 1.4))
                ev.append((p + inner, p + 2 * inner, 0.1 if f < 1 else 2.2)); p += ln
            elif kind == 3:    # staircase of three levels
                ev.append((p, p + ln, 0.75 if f < 1 else 1.25)); ev.append((p + ln, p + 2 * ln, 0.5 if f < 1 else 1.5))
                ev.append((p + 2 * ln, p + 3 * ln, 0.25 if f < 1 else 1.75)); p += 3 * ln
            else:              # opposite types back to back
                ev.append((p, p + ln, 0.5)); ev.append((p + ln + 300, p + 2 * ln + 300, 1.5)); p += 2 * ln + 300
            p += int(rng.integers(3_000, 60_000))
    return [(s, e, f) for s, e, f in ev if e < L]


def apply_events(cn: np.ndarray, events) -> None:
    for s, e, f in events:
        cn[s:e] = f


# --------------------------------------------------------------------------------------------
# reads (BAM path).  Structure-of-arrays exactly as include/rsigpu.h's rsigpu_read_batch takes them.
READ_LEN = 100
F_PAIRED, F_PROPER, F_REV, F_MREV, F_R1, F_R2, F_SECONDARY, F_DUP = 1, 2, 16, 32, 64, 128, 256, 1024


def make_reads(L: int, seed: int, fasta: np.ndarray | None = None, coverage: float = 30.0, events=None, n_events: int = 8,
               lens=EVENT_LENS, tid: int = 0, discordant_per_edge: int = 12, frac_clip=0.15, frac_indel=0.03, frac_lowq=0.09,
               frac_dup=0.01, frac_mapq0=0.02, frac_secondary=0.002):
    """2x100 bp FR pairs, insert ~ N(400,30), copy-number-thinned starts for the planted events, spanning
    discordant pairs at DEL edges and everted pairs at DUP edges.  Returns (dict of numpy arrays sorted by pos, events)."""
    rng = np.random.default_rng(seed + 1000)
    if fasta is None:
        fasta = make_fasta(L, seed)
    n_blocks = _n_runs(fasta)
    if events is None:
        events = plant_events(L, seed, n_events, n_blocks, lens)
    RL = READ_LEN
    n_pairs = int(coverage * L / (2 * RL))
    # candidate fragment starts, thinned by copy number (max factor 1.5 -> oversample by 1.5)
    n_try = int(n_pairs * 1.5)
    start = rng.integers(2, L - 700, n_try, dtype=np.int64)
    cn = np.ones(L, np.float32)
    for s, e, f in events:
        cn[s:e] = f
    isn = fasta == ord("N")
    cn[isn] = 0
    keep = rng.random(n_try, dtype=np.float32) * 1.5 < cn[start]
    start = start[keep]
    ins = np.clip(np.rint(rng.normal(400, 30, len(start))), 250, 650).astype(np.int64)
    # drop fragments that touch N
    cs = np.concatenate(([0], np.cumsum(isn, dtype=np.int64)))
    ok = (cs[np.minimum(start + ins, L)] - cs[start]) == 0
    start, ins = start[ok], ins[ok]
    p1 = start; p2 = start + ins - RL
    extra = []
    # discordant pairs supporting the events
    for s, e, f in events:
        k = discordant_per_edge
        if f < 1:   # deletion: pairs spanning it, mates ~ (e - s) + 400 apart
            a = s - rng.integers(120, 300, k); b = e + rng.integers(20, 200, k)
            extra.append((a, b, np.full(k, 0)))
        else:       # duplication: everted pairs (read 1 near the end, mate near the start)
            a = e - rng.integers(120, 300, k); b = s + rng.integers(20, 200, k)
            extra.append((a, b, np.full(k, 1)))
    n_norm = len(p1)
    pos1 = [p1]; pos2 = [p2]; kind = [np.full(n_norm, -1)]
    for a, b, kk in extra:
        pos1.append(a.astype(np.int64)); pos2.append(b.astype(np.int64)); kind.append(kk)
    p1 = np.concatenate(pos1); p2 = np.concatenate(pos2); kind = np.concatenate(kind)
    n = len(p1)
    # per-read arrays: read 1 (forward) and read 2 (reverse)
    pos = np.concatenate((p1, p2)).astype(np.int32)
    mpos = np.concatenate((p2, p1)).astype(np.int32)
    isz = (p2 + RL - p1)
    isize = np.concatenate((isz, -isz)).astype(np.int32)
    proper = np.concatenate((kind < 0, kind < 0))
    flag = np.concatenate((np.full(n, F_PAIRED | F_MREV | F_R1), np.full(n, F_PAIRED | F_REV | F_R2))).astype(np.uint16)
    flag[proper] |= F_PROPER
    nr = 2 * n
    u = rng.random(nr)
    flag[u < frac_dup] |= F_DUP
    flag[(u >= frac_dup) & (u < frac_dup + frac_secondary)] |= F_SECONDARY
    mapq = np.full(nr, 60, np.uint8)
    mapq[rng.random(nr) < frac_mapq0] = 0
    mtid = np.full(nr, tid, np.int32)
    # CIGARs: 100M | xS yM | yM xS | 50M 2D 50M | 50M 2I 48M
    u = rng.random(nr)
    ctype = np.zeros(nr, np.int8)
    ctype[u < frac_clip / 2] = 1
    ctype[(u >= frac_clip / 2) & (u < frac_clip)] = 2
    ctype[(u >= frac_clip) & (u < frac_clip + frac_indel / 2)] = 3
    ctype[(u >= frac_clip + frac_indel / 2) & (u < frac_clip + frac_indel)] = 4
    x = rng.integers(5, 31, nr).astype(np.uint32)
    ncig = np.where(ctype == 0, 1, np.where(ctype <= 2, 2, 3)).astype(np.uint32)
    order = np.argsort(pos, kind="stable")
    pos, mpos, isize, flag, mapq, mtid, ctype, x, ncig = (a[order] for a in (pos, mpos, isize, flag, mapq, mtid, ctype, x, ncig))
    cigar_off = np.concatenate(([0], np.cumsum(ncig, dtype=np.uint64))).astype(np.uint32)
    cigar = np.zeros(int(cigar_off[-1]), np.uint32)
    o = cigar_off[:-1]
    M, I, D, S = 0, 1, 2, 4
    m0 = ctype == 0; cigar[o[m0]] = (RL << 4) | M
    m1 = ctype == 1; cigar[o[m1]] = (x[m1] << 4) | S; cigar[o[m1] + 1] = ((RL - x[m1]) << 4) | M
    m2 = ctype == 2; cigar[o[m2]] = ((RL - x[m2]) << 4) | M; cigar[o[m2] + 1] = (x[m2] << 4) | S
    m3 = ctype == 3; cigar[o[m3]] = (50 << 4) | M; cigar[o[m3] + 1] = (2 << 4) | D; cigar[o[m3] + 2] = (50 << 4) | M
    m4 = ctype == 4; cigar[o[m4]] = (50 << 4) | M; cigar[o[m4] + 1] = (2 << 4) | I; cigar[o[m4] + 2] = (48 << 4) | M
    qual_off = (np.arange(nr + 1, dtype=np.uint64) * RL)
    qual = np.full(nr * RL, 30, np.uint8)
    lowq = np.flatnonzero(rng.random(nr) < frac_lowq)
    st = rng.integers(0, RL - 10, len(lowq))
    idx = (lowq[:, None] * RL + st[:, None] + np.arange(10)[None, :]).ravel()
    qual[idx] = 2
    reads = dict(pos=pos, mpos=mpos, isize=isize, mtid=mtid, flag=flag, mapq=mapq, cigar_off=cigar_off, cigar=cigar,
                 qual_off=qual_off, qual=qual)
    return reads, events


def make_long_reads(L: int, n: int, seed: int, tid: int = 0, max_ops: int = 200, max_len: int = 50_000, max_skip: int = 500_000,
                    max_other: int = 300, min_len: int = 0):
    """Long, spliced and many-op reads, unlike make_reads' 2x100 bp pairs: 1..max_ops CIGAR ops of every type 0-8 in any order
    (so I/S/N/H/P can precede the first M/D/=/X op and S can sit between M ops), lengths log-uniform -- M/=/X in
    [min_len, max_len], N up to max_skip, the rest up to max_other; zero-length ops included when min_len is 0.  Qualities
    0-255, mapq 0-60, FR / proper / duplicate / secondary flags at random.  Positions uniform in [0, L), plus reads at 0 and at
    L - 1; many reads reach past L.  Each read has exactly as many qualities as its CIGAR consumes query bases (M/I/S/=/X).
    Returns the position-sorted SoA dict that pileup_push, write_bam and the oracle bindings take."""
    rng = np.random.default_rng(seed + 7000)

    def logu(lo, hi, size):        # integers in [lo, hi], log-uniform: mostly short, a few near hi
        return np.minimum(lo + np.floor(np.expm1(rng.random(size) * np.log1p(hi - lo + 1))).astype(np.int64), hi)
    nops = rng.integers(1, max_ops + 1, n)
    op = rng.integers(0, 9, int(nops.sum()))
    ln = np.where(np.isin(op, (0, 7, 8)), logu(min_len, max_len, len(op)),
                  np.where(op == 3, logu(0, max_skip, len(op)), logu(0, max_other, len(op))))
    cigar_off = np.concatenate(([0], np.cumsum(nops))).astype(np.uint32)
    cigar = ((ln.astype(np.uint32) << 4) | op.astype(np.uint32)).astype(np.uint32)
    qcons = np.where(np.isin(op, (0, 1, 4, 7, 8)), ln, 0)
    qlen = np.add.reduceat(qcons, cigar_off[:-1].astype(np.int64))
    qual_off = np.concatenate(([0], np.cumsum(qlen))).astype(np.uint64)
    pos = rng.integers(0, L, n).astype(np.int64)
    pos[:min(n, 2)] = 0
    if n > 2:
        pos[2] = L - 1
    order = np.argsort(pos, kind="stable")
    flag = (rng.choice(np.array([F_PAIRED | F_MREV | F_R1, F_PAIRED | F_REV | F_R2], np.uint16), n) |
            np.where(rng.random(n) < 0.5, F_PROPER, 0)).astype(np.uint16)
    u = rng.random(n)
    flag[u < 0.05] |= F_DUP
    flag[(u >= 0.05) & (u < 0.08)] |= F_SECONDARY
    isize = rng.integers(-2000, 2000, n).astype(np.int32)
    R = dict(pos=pos.astype(np.int32), mpos=(pos + rng.integers(-5000, 5000, n)).clip(0, L - 1).astype(np.int32), isize=isize,
             mtid=np.full(n, tid, np.int32), flag=flag, mapq=rng.integers(0, 61, n).astype(np.uint8), cigar_off=cigar_off,
             cigar=cigar, qual_off=qual_off, qual=rng.integers(0, 256, int(qual_off[-1])).astype(np.uint8))
    return take_reads(R, order)


def take_reads(R: dict, idx) -> dict:
    """the reads R[idx] (any order) as a new SoA dict with its own CIGAR / quality offsets"""
    idx = np.asarray(idx, np.int64)
    co = R["cigar_off"].astype(np.int64); qo = R["qual_off"].astype(np.int64)
    nc = co[idx + 1] - co[idx]; nq = qo[idx + 1] - qo[idx]
    out = {k: np.asarray(R[k])[idx] for k in ("pos", "mpos", "isize", "mtid", "flag", "mapq")}
    out["cigar_off"] = np.concatenate(([0], np.cumsum(nc))).astype(np.uint32)
    out["qual_off"] = np.concatenate(([0], np.cumsum(nq))).astype(np.uint64)
    ci = np.repeat(co[idx], nc) + (np.arange(int(nc.sum())) - np.repeat(np.cumsum(nc) - nc, nc))
    qi = np.repeat(qo[idx], nq) + (np.arange(int(nq.sum())) - np.repeat(np.cumsum(nq) - nq, nq))
    out["cigar"] = R["cigar"][ci]; out["qual"] = R["qual"][qi]
    return out


def merge_reads(*sets: dict) -> dict:
    """several read SoA dicts of one contig as one, sorted by position (stable: equal positions keep the order of `sets`)"""
    keys = ("pos", "mpos", "isize", "mtid", "flag", "mapq", "cigar", "qual")
    cat = {k: np.concatenate([s[k] for s in sets]) for k in keys}
    nco = [0]; nqo = [0]
    for s in sets:
        nco.append(nco[-1] + int(s["cigar_off"][-1])); nqo.append(nqo[-1] + int(s["qual_off"][-1]))
    cat["cigar_off"] = np.concatenate([s["cigar_off"][:-1].astype(np.int64) + b for s, b in zip(sets, nco)] + [[nco[-1]]]).astype(np.uint32)
    cat["qual_off"] = np.concatenate([s["qual_off"][:-1].astype(np.int64) + b for s, b in zip(sets, nqo)] + [[nqo[-1]]]).astype(np.uint64)
    return take_reads(cat, np.argsort(cat["pos"], kind="stable"))


def _fill_var(buf, starts, lens, values):
    """buf[starts[r] + k] = values[...] for k < lens[r], all records at once"""
    lens = np.asarray(lens, np.int64)
    tot = int(lens.sum())
    if tot == 0:
        return
    idx = np.repeat(np.asarray(starts, np.int64), lens) + (np.arange(tot) - np.repeat(np.cumsum(lens) - lens, lens))
    buf[idx] = values


def _bam_records(R: dict, tid: int, lo: int, hi: int, random_seq, rich=None, want_offsets: bool = False):
    """records lo..hi of one contig's reads as BAM bytes (bam1_core_t layout, bam.h:131-155).  rich=SEED: what real files
    carry and the path must skip -- read names of varying length, random bases, optional fields after the qualities."""
    nr = hi - lo
    co_all = R["cigar_off"].astype(np.int64); qo_all = R["qual_off"].astype(np.int64)
    co = co_all[lo:hi]; ncig = co_all[lo + 1:hi + 1] - co; qo = qo_all[lo:hi]; lq = qo_all[lo + 1:hi + 1] - qo
    rs = np.random.default_rng([rich if rich is not None else (random_seq or 0), tid, lo])
    if rich is not None:
        lname = rs.integers(2, 25, nr).astype(np.int64)          # incl. the NUL
        laux = np.where(rs.random(nr) < 0.7, rs.integers(4, 64, nr), 0).astype(np.int64)
    else:
        lname = np.full(nr, 2, np.int64)  # "r\0"
        laux = np.zeros(nr, np.int64)
    nseq = (lq + 1) // 2
    size = 32 + lname + 4 * ncig + nseq + lq + laux   # block_size payload (without the 4-byte length)
    offs = np.concatenate(([0], np.cumsum(size + 4)))
    buf = np.zeros(int(offs[-1]), np.uint8)
    o = offs[:-1]

    def put32(off, val):
        v = np.ascontiguousarray(np.asarray(val).astype("<u4")).view(np.uint8).reshape(-1, 4)
        for k in range(4):
            buf[o + off + k] = v[:, k]
    pos = R["pos"][lo:hi].astype(np.int64)
    # reg2bin needs the alignment end: sum of M/D/N lengths
    cig = R["cigar"][int(co_all[lo]):int(co_all[hi])]
    cl = (cig >> 4).astype(np.int64); cop = cig & 15
    refl = np.where((cop == 0) | (cop == 2) | (cop == 3), cl, 0)
    csum = np.concatenate(([0], np.cumsum(refl)))
    c0 = co - co_all[lo]
    end = pos + (csum[c0 + ncig] - csum[c0])
    b = _reg2bin(pos, np.maximum(end, pos + 1))
    put32(0, size)
    put32(4, np.full(nr, tid)); put32(8, R["pos"][lo:hi])
    put32(12, (b.astype(np.uint32) << 16) | (R["mapq"][lo:hi].astype(np.uint32) << 8) | lname.astype(np.uint32))
    put32(16, (R["flag"][lo:hi].astype(np.uint32) << 16) | ncig.astype(np.uint32))
    put32(20, lq); put32(24, R["mtid"][lo:hi]); put32(28, R["mpos"][lo:hi]); put32(32, R["isize"][lo:hi])
    # read name: printable characters, NUL-terminated
    if rich is not None:
        _fill_var(buf, o + 36, lname - 1, rs.integers(33, 127, int((lname - 1).sum())).astype(np.uint8))
    else:
        buf[o + 36] = ord("r")
    # CIGAR words
    _fill_var(buf, o + 36 + lname, 4 * ncig, np.ascontiguousarray(cig.astype("<u4")).view(np.uint8))
    # packed sequence (all 'A' = 1, or random bases) and qualities
    soff = o + 36 + lname + 4 * ncig
    nib = np.array([1, 2, 4, 8], np.uint8)
    nst = int(nseq.sum())
    if random_seq is None and rich is None:
        seqb = np.full(nst, 0x11, np.uint8)
    else:
        seqb = ((nib[rs.integers(0, 4, nst)] << 4) | nib[rs.integers(0, 4, nst)]).astype(np.uint8)
    _fill_var(buf, soff, nseq, seqb)
    odd = np.flatnonzero(lq % 2 == 1)
    buf[soff[odd] + nseq[odd] - 1] &= 0xf0
    _fill_var(buf, soff + nseq, lq, R["qual"][int(qo_all[lo]):int(qo_all[hi])])
    # optional fields: "XA:Z:<text>\0"-shaped bytes (never parsed on this path)
    if rich is not None and int(laux.sum()):
        aux = rs.integers(33, 127, int(laux.sum())).astype(np.uint8)
        _fill_var(buf, soff + nseq + lq, laux, aux)
        has = np.flatnonzero(laux > 0)
        a0 = (soff + nseq + lq)[has]
        buf[a0] = ord("X"); buf[a0 + 1] = ord("A"); buf[a0 + 2] = ord("Z"); buf[a0 + laux[has] - 1] = 0
    if want_offsets:
        return buf.tobytes(), offs
    return buf.tobytes()


def _bam_header(contigs: list[tuple[str, int]], sort_order: str) -> bytes:
    import struct
    text = f"@HD\tVN:1.0\tSO:{sort_order}\n" + "".join(f"@SQ\tSN:{n}\tLN:{l}\n" for n, l in contigs)
    hdr = bytearray(b"BAM\x01") + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", len(contigs))
    for n, l in contigs:
        hdr += struct.pack("<i", len(n) + 1) + n.encode() + b"\x00" + struct.pack("<i", l)
    return bytes(hdr)


def _unplaced_record(u: int) -> bytes:
    """an unplaced, unmapped read: refID -1, pos -1, flag 4, no CIGAR"""
    import struct
    name = b"unm%d\x00" % u
    body = struct.pack("<iiIIiiii", -1, -1, (4680 << 16) | len(name), (4 << 16), 10, -1, -1, 0) + name + b"\x11" * 5 + b"\x1e" * 10
    return struct.pack("<I", len(body)) + body


def _write_bgzf(path: str, pieces, level: int, strategy: int, block_size: int, threads: int) -> None:
    """the concatenated pieces as BGZF blocks of block_size decoded bytes, then the EOF marker"""
    import struct
    import zlib
    from concurrent.futures import ThreadPoolExecutor

    def bgzf(blk: bytes) -> bytes:
        co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, strategy)
        comp = co.compress(blk) + co.flush()
        return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(comp) + 25) + comp +
                struct.pack("<II", zlib.crc32(blk) & 0xffffffff, len(blk)))
    BS = block_size
    with open(path, "wb") as f, ThreadPoolExecutor(threads) as pool:
        carry = b""
        for piece in pieces:
            data = carry + piece
            nfull = len(data) // BS * BS
            for out in pool.map(bgzf, (data[a:a + BS] for a in range(0, nfull, BS))):
                f.write(out)
            carry = data[nfull:]
        if carry:
            f.write(bgzf(carry))
        f.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))


def write_bam(path: str, contigs: list[tuple[str, int]], reads_by_tid: dict[int, dict], level: int = 1, strategy: int = 0,
              block_size: int = 65280, random_seq: int | None = None, threads: int = 8, rich: int | None = None,
              unmapped_tail: int = 0) -> None:
    """Minimal BAM (BGZF) writer for the synthetic reads: one record per read, name 'r', sequence all 'A'
    (the path never looks at bases; random_seq=SEED writes random bases instead, which makes the file compress like a
    real one), qualities as given.  strategy: zlib strategy (zlib.Z_FIXED forces fixed-Huffman blocks), level 0 writes
    stored blocks; records are NOT aligned to BGZF blocks.  Reads are serialised in slabs and the blocks compressed on a
    thread pool, so a chr19-sized file takes about a minute.  rich=SEED writes real-looking records (names, bases, optional
    fields); unmapped_tail appends that many refID -1 records.  Layout: SURVEY.md Appendix B."""
    def pieces():
        yield _bam_header(contigs, "coordinate")
        for tid in sorted(reads_by_tid):
            R = reads_by_tid[tid]
            nr = len(R["pos"])
            for lo in range(0, nr, 1 << 19):
                yield _bam_records(R, tid, lo, min(nr, lo + (1 << 19)), random_seq, rich)
        for u in range(unmapped_tail):
            yield _unplaced_record(u)
    _write_bgzf(path, pieces(), level, strategy, block_size, threads)


def write_bam_unsorted(path: str, contigs: list[tuple[str, int]], reads_by_tid: dict[int, dict], order, level: int = 1,
                       strategy: int = 0, block_size: int = 65280, random_seq: int | None = None, threads: int = 8,
                       rich: int | None = None) -> None:
    """write_bam with the records in any interleaving, header `@HD SO:unsorted`.  order: a sequence of refIDs, one per record;
    the k-th occurrence of refID t writes reads_by_tid[t]'s read k (so each contig's reads appear in the order of its dict,
    which need not be by position), and each -1 writes the next unplaced, unmapped record (refID -1, pos -1, flag 4)."""
    order = np.asarray(order, np.int64)
    tids = sorted(reads_by_tid)
    for t in tids:
        assert int(np.count_nonzero(order == t)) == len(reads_by_tid[t]["pos"]), f"order must name refID {t} once per read"
    assert set(np.unique(order).tolist()) <= set(tids) | {-1}
    bufs, starts, lens, base = [], {}, {}, 0
    for t in tids:
        b, offs = _bam_records(reads_by_tid[t], t, 0, len(reads_by_tid[t]["pos"]), random_seq, rich, want_offsets=True)
        bufs.append(np.frombuffer(b, np.uint8)); starts[t] = base + offs[:-1]; lens[t] = np.diff(offs); base += len(b)
    n_un = int(np.count_nonzero(order == -1))
    un = [_unplaced_record(u) for u in range(n_un)]
    ul = np.array([len(r) for r in un], np.int64)
    bufs.append(np.frombuffer(b"".join(un), np.uint8)); starts[-1] = base + np.concatenate(([0], np.cumsum(ul)[:-1])) if n_un else np.zeros(0, np.int64); lens[-1] = ul
    src = np.concatenate(bufs) if bufs else np.zeros(0, np.uint8)
    rec_start = np.zeros(len(order), np.int64); rec_len = np.zeros(len(order), np.int64)
    for t in list(tids) + [-1]:
        at = np.flatnonzero(order == t)
        rec_start[at] = starts[t]; rec_len[at] = lens[t]
    body = src[np.repeat(rec_start, rec_len) + (np.arange(int(rec_len.sum())) - np.repeat(np.cumsum(rec_len) - rec_len, rec_len))]

    def pieces():
        yield _bam_header(contigs, "unsorted")
        for a in range(0, len(body), 1 << 26):
            yield body[a:a + (1 << 26)].tobytes()
    _write_bgzf(path, pieces(), level, strategy, block_size, threads)


def write_bam_aligned(path: str, name: str, L: int, reads: dict, level: int = 1, random_seq: int | None = None, threads: int = 8,
                      block_size: int = 65280):
    """One-contig BAM whose BGZF blocks END AT RECORD BOUNDARIES (valid BGZF/BAM: writers may flush anywhere), the header in
    blocks of its own.  Any prefix of the record blocks is then itself a complete record stream, so the byte range
    [rec_off, blk_end[k]) of this ONE image is the BAM of the contig truncated after record blk_rec_end[k] -- what bench.py's
    whole-genome workload uses to present 24 per-chromosome files without compressing 24 images.
    Returns dict(rec_off=file offset of the first record block, blk_end=int64[nblk] file offset after each record block,
    blk_rec_end=int64[nblk] number of records in blocks 0..k)."""
    import struct
    import zlib
    from concurrent.futures import ThreadPoolExecutor
    text = "@HD\tVN:1.0\tSO:coordinate\n" + f"@SQ\tSN:{name}\tLN:{L}\n"
    hdr = bytearray(b"BAM\x01") + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", 1)
    hdr += struct.pack("<i", len(name) + 1) + name.encode() + b"\x00" + struct.pack("<i", L)

    def bgzf(blk: bytes) -> bytes:
        co = zlib.compressobj(level, zlib.DEFLATED, -15, 8, 0)
        comp = co.compress(blk) + co.flush()
        return (b"\x1f\x8b\x08\x04\x00\x00\x00\x00\x00\xff\x06\x00BC\x02\x00" + struct.pack("<H", len(comp) + 25) + comp +
                struct.pack("<II", zlib.crc32(blk) & 0xffffffff, len(blk)))
    nr = len(reads["pos"])
    blk_end, blk_rec_end = [], []
    with open(path, "wb") as f, ThreadPoolExecutor(threads) as pool:
        f.write(bgzf(bytes(hdr)))
        rec_off = foff = f.tell()
        for lo in range(0, nr, 1 << 19):
            hi = min(nr, lo + (1 << 19))
            data, offs = _bam_records(reads, 0, lo, hi, random_seq, None, want_offsets=True)
            cuts = [0]                       # indices into offs: greedy blocks of whole records
            while cuts[-1] < hi - lo:
                k = int(np.searchsorted(offs, offs[cuts[-1]] + block_size, side="right")) - 1
                cuts.append(max(k, cuts[-1] + 1))
            for a, b, out in zip(cuts[:-1], cuts[1:], pool.map(bgzf, (data[int(offs[a]):int(offs[b])] for a, b in zip(cuts[:-1], cuts[1:])))):
                f.write(out)
                foff += len(out)
                blk_end.append(foff); blk_rec_end.append(lo + b)
        f.write(bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000"))
    return dict(rec_off=rec_off, blk_end=np.asarray(blk_end, np.int64), blk_rec_end=np.asarray(blk_rec_end, np.int64))


def write_bai(bam_path: str) -> None:
    """<bam_path>.bai for a coordinate-sorted BGZF/BAM file (SAM spec 5.2, laid out as samtools-0.1.18's bam_index_build
    writes it): per reference one chunk per run of records with the same bin (adjacent chunks of a bin that meet in one BGZF
    block merged), the pseudo-bin 37450 (file range of the reference, mapped / unmapped counts) and the 16 kbp linear index;
    the count of unplaced records at the end.  Lets the indexed routes of the CLI run on the files write_bam produces."""
    import struct
    import zlib
    raw = np.fromfile(bam_path, np.uint8)
    blocks, foffs, dstarts = [], [], []
    off = dlen = 0
    while off < len(raw):
        xlen = int(raw[off + 10]) | int(raw[off + 11]) << 8
        bsize = (int(raw[off + 16]) | int(raw[off + 17]) << 8) + 1
        blk = zlib.decompress(raw[off + 12 + xlen:off + bsize - 8].tobytes(), -15)
        blocks.append(blk); foffs.append(off); dstarts.append(dlen)
        off += bsize; dlen += len(blk)
    dec = b"".join(blocks)
    d = np.frombuffer(dec, np.uint8)
    foffs = np.asarray(foffs, np.int64); dstarts = np.asarray(dstarts, np.int64)

    def i32(at):
        return (d[at].astype(np.int64) | d[at + 1].astype(np.int64) << 8 | d[at + 2].astype(np.int64) << 16 |
                d[at + 3].astype(np.int64) << 24).astype(np.uint32).astype(np.int64)

    l_text = struct.unpack_from("<i", dec, 4)[0]
    n_ref = struct.unpack_from("<i", dec, 8 + l_text)[0]
    p = 12 + l_text
    for _ in range(n_ref):
        p += 8 + struct.unpack_from("<i", dec, p)[0]
    starts = []
    while p < len(dec):
        starts.append(p)
        p += 4 + struct.unpack_from("<i", dec, p)[0]
    s = np.asarray(starts + [len(dec)], np.int64)
    k = np.searchsorted(dstarts, s, side="right") - 1           # the block a decoded offset lies in (its end: the next block)
    voff = (foffs[k] << 16) | (s - dstarts[k])
    s = s[:-1]
    tid = i32(s + 4).astype(np.int32).astype(np.int64); pos = i32(s + 8).astype(np.int32).astype(np.int64)
    bmn = i32(s + 12); fnc = i32(s + 16)
    rbin = bmn >> 16; l_name = bmn & 0xff; flag = fnc >> 16; ncig = fnc & 0xffff
    # alignment end (bam_calend): sum of M / D / N lengths; an end <= pos counts as pos + 1
    cs = s + 36 + l_name
    tot = int(ncig.sum())
    ci = np.repeat(cs, ncig) + 4 * (np.arange(tot) - np.repeat(np.cumsum(ncig) - ncig, ncig))
    cw = i32(ci) if tot else np.zeros(0, np.int64)
    rl = np.where(np.isin(cw & 15, (0, 2, 3)), cw >> 4, 0)
    end = pos + np.add.reduceat(rl, np.minimum(np.cumsum(ncig) - ncig, tot - 1)) * (ncig > 0) if tot else pos.copy()
    end = np.maximum(end, pos + 1)
    out = bytearray(b"BAI\x01") + struct.pack("<i", n_ref)
    for r in range(n_ref):
        idx = np.flatnonzero(tid == r)
        if not len(idx):
            out += struct.pack("<ii", 0, 0)
            continue
        beg, fin = voff[idx], voff[idx + 1]
        cut = np.flatnonzero(np.diff(rbin[idx]) != 0) + 1       # runs of records with the same bin
        rs = np.concatenate(([0], cut)); re = np.concatenate((cut, [len(idx)])) - 1
        chunks: dict[int, list[list[int]]] = {}
        for a, b in zip(rs, re):
            lst = chunks.setdefault(int(rbin[idx[a]]), [])
            u, v = int(beg[a]), int(fin[b])
            if lst and lst[-1][1] >> 16 == u >> 16:
                lst[-1][1] = v
            else:
                lst.append([u, v])
        nmap = int(((flag[idx] & 4) == 0).sum())
        chunks[37450] = [[int(beg[0]), int(fin[-1])], [nmap, len(idx) - nmap]]
        out += struct.pack("<i", len(chunks))
        for b in sorted(chunks):
            out += struct.pack("<Ii", b, len(chunks[b]))
            for u, v in chunks[b]:
                out += struct.pack("<QQ", u, v)
        w0 = pos[idx] >> 14; w1 = (end[idx] - 1) >> 14
        nw = int(w1.max()) + 1
        lin = np.full(nw, np.iinfo(np.int64).max, np.int64)
        nwr = w1 - w0 + 1
        np.minimum.at(lin, np.repeat(w0, nwr) + (np.arange(int(nwr.sum())) - np.repeat(np.cumsum(nwr) - nwr, nwr)), np.repeat(beg, nwr))
        lin[lin == np.iinfo(np.int64).max] = 0
        for j in range(1, nw):
            if lin[j] == 0:
                lin[j] = lin[j - 1]
        out += struct.pack("<i", nw) + lin.astype("<u8").tobytes()
    n_no_coor = int((tid < 0).sum())
    if n_no_coor:
        out += struct.pack("<Q", n_no_coor)
    with open(bam_path + ".bai", "wb") as f:
        f.write(bytes(out))


def _reg2bin(beg, end):
    """UCSC binning (samtools bam.h:bam_reg2bin), vectorised"""
    end = end - 1
    out = np.zeros(len(beg), np.int64)
    done = np.zeros(len(beg), bool)
    for shift, base in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        m = ~done & ((beg >> shift) == (end >> shift))
        out[m] = base + (beg[m] >> shift)
        done |= m
    return out
