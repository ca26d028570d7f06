// k_pileup.cuh -- BAM-input kernels on position-sorted read batches staged in HBM as SoA.
//
// Replaces (reference file:line relative to src/):
//   load_data_from_bam hot loop  loaddata.cpp:312-335  +  resolve_cigar_pos  samfunctions.cpp:38-100   k_read_ends, k_pileup_tile
//   bam_calend                   samtools-0.1.18/bam.c:17-27                                            k_read_ends
//   bam_rd_pr_stats (insert-size sample)  pairrd.cpp:112-260 (order of tests: SURVEY.md A.2)            k_isize_stats
//   cnv_stat                     pairrd.cpp:622-748                                                     k_cnv_stat
//
// Pileup design: (1) k_qual_mask streams the quality bytes once and leaves one pass bit per base
// (quality >= Q); (2) in k_pileup_tile a block OWNS a tile of reference positions: the reads that can
// touch it come from a precomputed binary search of the sorted read starts, every thread walks the
// CIGAR of its reads and turns each maximal stretch of passing M/= bases (bit tricks on the pass mask)
// into +1/-1 events in a shared-memory difference array (clipped to the tile), a block-wide scan turns
// events into depth and the tile is stored once with 16-byte stores: no global atomics, no zero-fill,
// no read-modify-write.
#pragma once
#include "k_seg.cuh"

namespace rsigpu {

struct ReadSoA {
  i64 n;
  int tid;
  const int* pos; const int* mpos; const int* isize; const int* mtid;
  const u16* flag; const u8* mapq;
  const u32* cigar_off; const u32* cigar;
  const u64* qual_off; const u8* qual;
  int* calend;   // bam_calend per read (pos + 1 for reads without CIGAR)
  u16* ncig;     // n_cigar per read (clamped to 65535), written by k_read_ends; when cigar_off is null (the read summaries of a
                 // split contig, rsigpu_split_run) the kernels that only need the NUMBER of ops read it from here
};
__device__ __forceinline__ int read_ncig(const ReadSoA& R, i64 r) { return R.cigar_off ? (int)(R.cigar_off[r + 1] - R.cigar_off[r]) : (int)R.ncig[r]; }
enum { BF_PROPER = 2, BF_REV = 16, BF_MREV = 32, BF_SECONDARY = 256, BF_DUP = 1024 };
// PU_T: positions per tile of k_pileup_tile.  4096 keeps the shared difference array at 17 KB, so 8 blocks of PU_NT
// threads fit an SM (full occupancy at 32 registers; 8192 held it to 6 blocks).  PU_ENDS_PER_SM: read-end blocks per SM
// in k_qual_mask.
enum { PU_T = 4096, PU_NT = 256, PU_ENDS_PER_SM = 4 };

// per read: bam_calend, and the largest reference extent any of its counted bases can reach
// (reference coordinates advance on M, D, N and S from the first M/D/=/X op: samfunctions.cpp:59-100).
// Reads r0, r0 + stride, ...: the body of k_read_ends and of the read-end blocks of k_qual_mask.
__device__ __forceinline__ void read_ends_body(const ReadSoA& R, i64 r0, i64 stride, int* max_extent, int* sorted_bad) {
  int mx = 0, bad = 0;
  for (i64 r = r0; r < R.n; r += stride) {
    const u32 c0 = R.cigar_off[r], c1 = R.cigar_off[r + 1];
    u32 end = (u32)R.pos[r], ext = 0; bool anchored = false;
    for (u32 k = c0; k < c1; ++k) {
      const u32 op = R.cigar[k] & 15u, l = R.cigar[k] >> 4;
      if (op == 0 || op == 2 || op == 3) end += l;
      if (op == 0 || op == 2 || op == 7 || op == 8) anchored = true;
      if (anchored && (op == 0 || op == 2 || op == 3 || op == 4)) ext += l;
    }
    // an '=' op does not advance the reference coordinate but its bases are counted from there on
    u32 eqmax = 0;
    for (u32 k = c0; k < c1; ++k) { const u32 op = R.cigar[k] & 15u, l = R.cigar[k] >> 4; if (op == 7 && l > eqmax) eqmax = l; }
    ext += eqmax;
    R.calend[r] = c1 > c0 ? (int)end : R.pos[r] + 1;
    R.ncig[r] = (u16)(c1 - c0 > 65535u ? 65535u : c1 - c0);
    mx = imax(mx, (int)ext);
    if (r > 0 && R.pos[r] < R.pos[r - 1]) bad = 1;
  }
  if (mx) atomicMax(max_extent, mx);
  if (bad) atomicOr(sorted_bad, 1);
}
__global__ void k_read_ends(ReadSoA R, int* max_extent, int* sorted_bad) {
  read_ends_body(R, (i64)blockIdx.x * blockDim.x + threadIdx.x, (i64)gridDim.x * blockDim.x, max_extent, sorted_bad);
}

// Base-quality filter as a pure streaming pass: one bit per quality byte (bit i of word w = byte 32w+i has
// quality >= Q), 32 bytes per thread, SWAR byte compare (exact for any Q in [0, 255]; Q > 255 passes nothing).
// Reads every quality byte exactly once at HBM speed and leaves an 8x smaller array for the pileup proper.
__device__ __forceinline__ u32 qual_pass_nibble(u32 w, u32 qlow4, bool qhigh) {
  const u32 t = ((w & 0x7f7f7f7fu) | 0x80808080u) - qlow4;
  const u32 m7 = (qhigh ? (w & t) : (w | t)) & 0x80808080u;
  return ((m7 >> 7) * 0x01020408u) >> 24;
}
// Blocks [0, nb_ends) run the read-end pass (read_ends_body) over all reads, the others stream the quality bytes: the
// latency-bound CIGAR walk runs on the same SMs as the bandwidth-bound stream instead of alone before it.
__global__ void __launch_bounds__(256) k_qual_mask(const u8* __restrict__ qual, u64 nbytes, int min_baseQ, u32* __restrict__ mask,
                                                   ReadSoA R, int* max_extent, int* sorted_bad, int nb_ends) {
  if ((int)blockIdx.x < nb_ends) {
    read_ends_body(R, (i64)blockIdx.x * blockDim.x + threadIdx.x, (i64)nb_ends * blockDim.x, max_extent, sorted_bad);
    return;
  }
  const int Qc = min_baseQ < 0 ? 0 : min_baseQ;
  const bool q_none = Qc > 255, qhigh = Qc > 128;
  const u32 qlow4 = (u32)(qhigh ? Qc - 128 : Qc) * 0x01010101u;
  const u64 nwords = (nbytes + 31) >> 5;
  const u64 stride = (u64)(gridDim.x - nb_ends) * blockDim.x;
  for (u64 w = (u64)(blockIdx.x - nb_ends) * blockDim.x + threadIdx.x; w < nwords; w += stride) {
    const uint4 a = reinterpret_cast<const uint4*>(qual)[2 * w], b = reinterpret_cast<const uint4*>(qual)[2 * w + 1];
    u32 m = qual_pass_nibble(a.x, qlow4, qhigh) | (qual_pass_nibble(a.y, qlow4, qhigh) << 4) | (qual_pass_nibble(a.z, qlow4, qhigh) << 8) |
            (qual_pass_nibble(a.w, qlow4, qhigh) << 12) | (qual_pass_nibble(b.x, qlow4, qhigh) << 16) | (qual_pass_nibble(b.y, qlow4, qhigh) << 20) |
            (qual_pass_nibble(b.z, qlow4, qhigh) << 24) | (qual_pass_nibble(b.w, qlow4, qhigh) << 28);
    mask[w] = q_none ? 0u : m;
  }
}

#define PU_DI(i) ((i) + ((i) >> 5))
// One M/= op: maximal stretches of passing bases among quality bytes [qb, qb + len) (global byte indices into the
// quality array = bit indices into the pass mask) become +1 / -1 events at tile offsets dbase + j.  Chunks of 128
// bases: five mask words, funnel shifts, then run starts / ends by bit tricks.
__device__ __forceinline__ void pu_mask_runs(const u32* __restrict__ mask, u64 qb, int len_total, int dbase0, int* diff) {
  for (int cb = 0; cb < len_total; cb += 128) {
    const int len = imin(128, len_total - cb);
    const u64 bit0 = qb + (u64)cb;
    const u32* mw = mask + (bit0 >> 5);
    const u32 sh = (u32)(bit0 & 31);
    const int nwd = (len + 31) >> 5;
    u32 mk[4];
    u32 lo = mw[0];
#pragma unroll
    for (int wd = 0; wd < 4; ++wd) {
      mk[wd] = 0u;
      if (wd < nwd) {
        const u32 hi = mw[wd + 1];                     // one word past the op at most: the mask array is padded
        mk[wd] = sh ? ((lo >> sh) | (hi << (32 - sh))) : lo;
        lo = hi;
        const int nbits = len - 32 * wd;
        if (nbits < 32) mk[wd] &= (1u << nbits) - 1u;
      }
    }
    u32 prev = 0u;
    const int dbase = dbase0 + cb;
#pragma unroll
    for (int wd = 0; wd < 4; ++wd) {
      const u32 cur = mk[wd];
      const u32 shf = (cur << 1) | prev;
      u32 st_ = cur & ~shf, en = ~cur & shf;
      while (st_) { const int bbit = __ffs((int)st_) - 1; atomicAdd(&diff[PU_DI(dbase + 32 * wd + bbit)], 1); st_ &= st_ - 1u; }
      while (en) { const int bbit = __ffs((int)en) - 1; atomicAdd(&diff[PU_DI(dbase + 32 * wd + bbit)], -1); en &= en - 1u; }
      prev = cur >> 31;
    }
    if (prev) atomicAdd(&diff[PU_DI(dbase + 128)], -1);
  }
}

// first / one-past-last read that can touch each position tile (reads with pos in [t0 - max_extent, t1))
__global__ void k_tile_ranges(ReadSoA R, int L, const int* max_extent, int2* __restrict__ range) {
  const int ntiles = (L + PU_T - 1) / PU_T;
  const int ext = *max_extent;
  for (int tile = (int)(blockIdx.x * blockDim.x + threadIdx.x); tile < ntiles; tile += (int)(gridDim.x * blockDim.x)) {
    const int t0 = tile * PU_T, t1 = imin(t0 + PU_T, L);
    i64 lo = 0, hi = R.n; const int want = t0 - ext;
    while (lo < hi) { i64 mid = (lo + hi) >> 1; if (R.pos[mid] < want) lo = mid + 1; else hi = mid; }
    const i64 r0 = lo;
    hi = R.n;
    while (lo < hi) { i64 mid = (lo + hi) >> 1; if (R.pos[mid] < t1) lo = mid + 1; else hi = mid; }
    range[tile] = make_int2((int)r0, (int)lo);
  }
}

// tile0 .. tile1: the position tiles this launch covers (all of them, or one part of a contig split over several GPUs)
__global__ void __launch_bounds__(PU_NT) k_pileup_tile(ReadSoA R, const u32* __restrict__ qmask, int* __restrict__ rd, int L, int minq,
                                                        const int2* __restrict__ range, int tile0, int tile1) {
  RSI_CTA_SETUP(c);
  __shared__ int diff[PU_T + 1 + (PU_T + 1) / 32 + 1];   // entry i lives at i + i/32: conflict-free 32-per-thread scan
  const int ntiles = imin((L + PU_T - 1) / PU_T, tile1);
  for (int tile = tile0 + (int)blockIdx.x; tile < ntiles; tile += (int)gridDim.x) {
    const int t0 = tile * PU_T, t1 = imin(t0 + PU_T, L);
    c.sync();
    for (int k = c.tid; k < PU_T + 1 + (PU_T + 1) / 32 + 1; k += PU_NT) diff[k] = 0;
    const int2 rr = range[tile];
    c.sync();
    for (int r = rr.x + c.tid; r < rr.y; r += PU_NT) {
      const int pos = R.pos[r], fl = R.flag[r], mq = (int)R.mapq[r];
      const u32 c0 = R.cigar_off[r], c1 = R.cigar_off[r + 1];
      const u64 qoff = R.qual_off[r];
      u32 cg[3] = {0u, 0u, 0u};
#pragma unroll
      for (int k = 0; k < 3; ++k) if (c0 + k < c1) cg[k] = R.cigar[c0 + k];
      if (pos == 0 || mq < minq || (fl & (BF_SECONDARY | BF_DUP))) continue;
      // reference / query coordinate at the start of each op
      u32 k = c0, q = 0;
      while (k < c1) { const u32 cgk = k - c0 < 3 ? cg[k - c0] : R.cigar[k]; const u32 op = cgk & 15u; if (op == 0 || op == 2 || op == 7 || op == 8) break; if (op == 1 || op == 4) q += cgk >> 4; ++k; }
      u32 e = (u32)pos + 1;
      for (; k < c1; ++k) {      // (no M/D/=/X op: k == c1, nothing is counted)
        const u32 cgk = k - c0 < 3 ? cg[k - c0] : R.cigar[k];
        const u32 op = cgk & 15u, l = cgk >> 4;
        if (op == 0 || op == 7) {
          const int p = (int)e - 1;                      // 0-based position of the op's first base
          const int jb = imax(0, t0 - p), je = imin((int)l, imin(t1, L) - p);   // clipped to the tile and to L
          if (jb < je) pu_mask_runs(qmask, qoff + q + (u32)jb, je - jb, p + jb - t0, diff);
        }
        if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) q += l;
        if (op == 0 || op == 2 || op == 3 || op == 4) e += l;
      }
    }
    c.sync();
    // difference array -> depth, PU_T / PU_NT consecutive positions per thread
    const int per = PU_T / PU_NT;
    int loc[PU_T / PU_NT]; int s = 0;
#pragma unroll
    for (int j = 0; j < per; ++j) { s += diff[PU_DI(c.tid * per + j)]; loc[j] = s; }
    int tot;
    const int ex = c.scan_excl(s, &tot);
#pragma unroll
    for (int j = 0; j < per; j += 4) {
      const int p = t0 + c.tid * per + j;
      if (p < L) *reinterpret_cast<int4*>(rd + p) = make_int4(loc[j] + ex, loc[j + 1] + ex, loc[j + 2] + ex, loc[j + 3] + ex);
    }
  }
}
#undef PU_DI

// ---------------------------------------------------------------------------------------------
// Insert-size sample.  `keep`-filtered reads in file order from the first one overlapping 10 Mbp;
// sums run up to and including the read that trips a stop rule.
enum { IS_K = 8 };   // consecutive reads per thread and iteration
__global__ void __launch_bounds__(1024) k_isize_stats(ReadSoA R, int tid_len, const int* max_extent, int* __restrict__ out2) {
  RSI_CTA_SETUP(c);
  __shared__ int s_lastpos, s_segstart, s_segidx;
  const u32 beg = 10000000u, end = 349250621u;
  i64 lo = 0, hi = R.n;
  { const int want = (int)beg - *max_extent - 1; while (lo < hi) { i64 mid = (lo + hi) >> 1; if (R.pos[mid] < want) lo = mid + 1; else hi = mid; } }
  const i64 r_first = lo;
  if (c.tid == 0) { s_lastpos = -10000; s_segstart = 0; s_segidx = 0; }
  c.sync();
  const int lane = c.tid & 31, warp = c.tid >> 5;
  double s = 0, s2 = 0, cn = 0;
  i64 kept_before = 0;   // kept reads before this chunk
  for (i64 r0 = r_first; r0 < R.n; r0 += (i64)c.nthr * IS_K) {
    const i64 rb = r0 + (i64)c.tid * IS_K;
    int pos[IS_K], isz[IS_K]; bool kept[IS_K], prop[IS_K], stopA[IS_K], past[IS_K];
    int nkept = 0, lastkept = -0x7fffffff;
#pragma unroll
    for (int k = 0; k < IS_K; ++k) {
      const i64 r = rb + k;
      kept[k] = prop[k] = stopA[k] = past[k] = false; pos[k] = 0; isz[k] = 0;
      if (r < R.n) {
        pos[k] = R.pos[r];
        const u32 re = (u32)R.calend[r];
        const bool overl = (u32)pos[k] < end && re > beg;
        const int mt = R.mtid[r]; const int fl = R.flag[r];
        kept[k] = overl && !(mt != R.tid && mt > 0) && !(fl & BF_SECONDARY) && !(fl & BF_DUP);
        prop[k] = kept[k] && (fl & BF_PROPER) && mt == R.tid;
        isz[k] = R.isize[r];
        const int rpe = read_ncig(R, r) > 0 ? (int)re : pos[k];   // bam_calend proper
        stopA[k] = kept[k] && (pos[k] >= tid_len || rpe >= tid_len);
        past[k] = (u32)pos[k] >= end;          // the iterator stops at the first read with pos >= end
        if (kept[k]) { ++nkept; lastkept = pos[k]; }
      }
    }
    // exclusive sum-scan of kept counts and exclusive max-scan of the last kept position across threads
    int tot;
    const int ex = c.scan_excl(nkept, &tot);
    int prevpos;
    {
      int v = lastkept;
      for (int o = 1; o < 32; o <<= 1) { int u = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v = imax(v, u); }
      int* slots = reinterpret_cast<int*>(c.red);
      c.sync(); if (lane == 31) slots[warp] = v; c.sync();
      int pre = -0x7fffffff; for (int w = 0; w < warp; ++w) pre = imax(pre, slots[w]);
      int upv = __shfl_up_sync(0xffffffffu, v, 1);
      prevpos = imax(pre, lane ? upv : -0x7fffffff);
      c.sync();
    }
    prevpos = imax(prevpos, s_lastpos);
    // gaps inside the thread's reads; the most recent gap key = (kept rank << 32 | pos)
    i64 kidx[IS_K]; i64 key = -1; int pp = prevpos; i64 kk = kept_before + ex;
    i64 keyat[IS_K];
#pragma unroll
    for (int k = 0; k < IS_K; ++k) {
      kidx[k] = kk;
      if (kept[k]) { if (pos[k] > pp + 1000) key = (kk << 32) | (i64)(u32)pos[k]; pp = pos[k]; ++kk; }
      keyat[k] = key;    // latest gap at or before read k within this thread (or -1)
    }
    // inclusive max-scan of the threads' last keys -> exclusive prefix for this thread
    i64 prekey;
    {
      i64 v = key;
      for (int o = 1; o < 32; o <<= 1) { i64 u = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v = lmax(v, u); }
      i64* slots = reinterpret_cast<i64*>(c.red);
      c.sync(); if (lane == 31) slots[warp] = v; c.sync();
      i64 pre = -1; for (int w = 0; w < warp; ++w) pre = lmax(pre, slots[w]);
      i64 upv = __shfl_up_sync(0xffffffffu, v, 1);
      prekey = lmax(pre, lane ? upv : (i64)-1);
      c.sync();
    }
    // stop rules; first stopping read of the chunk
    int stop_at = 0x7fffffff;
#pragma unroll
    for (int k = 0; k < IS_K; ++k) {
      if (stop_at != 0x7fffffff) break;
      const i64 kf = lmax(keyat[k], prekey);
      int seg_idx, seg_pos;
      if (kf >= 0) { seg_idx = (int)(kf >> 32); seg_pos = (int)(kf & 0xffffffff); } else { seg_idx = s_segidx; seg_pos = s_segstart; }
      const i64 count = kidx[k] - seg_idx + 1;
      const bool stopB = kept[k] && !stopA[k] && (count > 1000000 || (pos[k] - seg_pos) > 1000000);
      if (stopA[k] || stopB || past[k]) stop_at = c.tid * IS_K + k;
    }
    const int first_stop = c.reduce(stop_at, MinOp());
#pragma unroll
    for (int k = 0; k < IS_K; ++k) {
      const int id = c.tid * IS_K + k;
      if (prop[k] && id <= first_stop && !(past[k] && id == first_stop)) {
        s += (double)(isz[k] < 0 ? -isz[k] : isz[k]);
        s2 += (double)(int)((u32)isz[k] * (u32)isz[k]);
        cn += 1;
      }
    }
    if (first_stop != 0x7fffffff) break;
    c.sync();
    if (c.tid == c.nthr - 1) {   // carry the running state to the next chunk
      s_lastpos = imax(s_lastpos, imax(prevpos, lastkept));
      const i64 kf = lmax(key, prekey);
      if (kf >= 0) { s_segidx = (int)(kf >> 32); s_segstart = (int)(kf & 0xffffffff); }
    }
    kept_before += tot;
    c.sync();
  }
  s = c.reduce(s, SumOp()); s2 = c.reduce(s2, SumOp()); cn = c.reduce(cn, SumOp());
  if (c.tid == 0) {
    int im = -1, isd = -1;
    if (cn > 2) {
      s /= cn;
      const double sd = sqrt((s2 - cn * s * s) / cn);
      im = (int)s; isd = (int)sd;
    }
    out2[0] = im; out2[1] = isd;
  }
}

// One block per call: Q0 fraction and supporting read pairs.  dis[k] = the carried DIS of call k.
__global__ void __launch_bounds__(1024) k_cnv_stat(ReadSoA R, Cnv* calls, int ncalls, const int* max_extent, const int* __restrict__ isz) {
  RSI_CTA_SETUP(c);
  const int im = isz[0], isd = isz[1];
  for (int k = (int)blockIdx.x; k < ncalls; k += (int)gridDim.x) {
    if (calls[k].tid != R.tid) continue;      // `stat` hands over the calls of every contig: DIS below runs over the whole list
    int DIS = 1000;
    for (int j = 0; j <= k; ++j) {   // DIS is carried from call to call (pairrd.cpp:655-656)
      int b = calls[j].start, e = calls[j].end; if (b > e) { int t = b; b = e; e = t; }
      DIS = imax(DIS, e - b + 1); DIS = imin(DIS, 5000);
    }
    int beg = calls[k].start, end = calls[k].end; if (beg > end) { int t = beg; beg = end; end = t; }
    const int type = calls[k].type;
    const int LEN = end - beg + 1;
    int p1e = beg - DIS; const int p2e = end + DIS;
    if (p1e < 1) p1e = 1;
    i64 lo = 0, hi = R.n;
    { const int want = p1e - *max_extent - 1; while (lo < hi) { i64 mid = (lo + hi) >> 1; if (R.pos[mid] < want) lo = mid + 1; else hi = mid; } }
    const i64 ra = lo;
    hi = R.n;
    while (lo < hi) { i64 mid = (lo + hi) >> 1; if ((u32)R.pos[mid] < (u32)p2e) lo = mid + 1; else hi = mid; }
    const i64 rb = lo;
    u32 qall = 0, q0 = 0, rp = 0;
    for (i64 r = ra + c.tid; r < rb; r += c.nthr) {
      const int nc = read_ncig(R, r);
      const int rbeg = R.pos[r], rend = R.calend[r];
      if (!((u32)rend > (u32)p1e && (u32)rbeg < (u32)p2e)) continue;
      if (nc <= 1) continue;
      if (rend > beg && rbeg < end) { ++qall; if (R.mapq[r] == 0) ++q0; }
      const int mt = R.mtid[r];
      if (mt != R.tid && mt > 0) continue;
      const int F = R.flag[r];
      if ((F & BF_REV) == 0 && (F & BF_MREV) == 0) continue;
      if ((F & BF_REV) > 0 && (F & BF_MREV) > 0) continue;
      int r1 = rend, r2 = R.mpos[r];
      if (type == RSIGPU_TYPE_DEL) {
        if (r2 - r1 < im + isd * 3) continue;
        const int ov = imin(r2, end) - imax(r1, beg);
        if (ov < 0) continue;
        if (abs(r1 - beg) + abs(r2 - end) < im + isd * 3) { ++rp; continue; }
        if ((double)ov < LEN * 0.5) continue;
        if ((double)ov < (r2 - r1) * 0.5) continue;
        ++rp;
      } else if (type == RSIGPU_TYPE_DUP) {
        if (r2 - r1 > im - isd * 3) continue;
        if (abs(r1 - beg) + abs(r2 - end) < im + isd * 3) { ++rp; continue; }
        if (r1 > r2) { int t = r1; r1 = r2; r2 = t; }
        const int ov = imin(r2, end) - imax(r1, beg);
        if ((double)ov < LEN * 0.5) continue;
        if ((double)ov < (r2 - r1) * 0.5) continue;
        ++rp;
      }
    }
    qall = c.reduce_ol(qall, SumOp()); q0 = c.reduce_ol(q0, SumOp()); rp = c.reduce_ol(rp, SumOp());
    if (c.tid == 0) { calls[k].q0 = (double)q0 / ((double)qall + 0.00001); calls[k].rp = (int)rp; }
    c.sync();
  }
}

}  // namespace rsigpu
