// k_sort.cuh -- a stable GPU sort of read records: an LSD radix sort of (u32 key, u32 index) pairs and the gathers that apply
// its permutation to a read SoA.  Two users:
//   rsigpu_bam_feed with rsigpu_set_bam_by_ref: a feed's records by refID (key = tid, refID -1 last), stable in file order,
//     before the payload is copied out of the inflated bytes -- so only the fixed fields and the offsets are gathered and
//     k_bam_payload writes every record's CIGAR / qualities straight to its sorted place;
//   rsigpu_pileup_sort: a context's staged reads by pos + 1, stable in staging order, fixed fields and payload.
//
// Radix pass over 8 bits (k_sort_hist, k_sort_scan_rows, k_sort_scatter): a tile of SRT_TILE keys per block.  The per-tile
// digit counts are stored digit-major, hist[d * ntile + t], so an exclusive scan of each digit's row plus an exclusive scan
// of the digit totals gives every (digit, tile) its first output slot in stable order.  The scatter walks its tile in index
// order, SRT_NT keys at a time: a key's rank among equal digits of its warp comes from __match_any_sync, the earlier warps'
// counts of that digit from shared memory.  Only warp collectives, shared atomics, plain loads and one global atomicMax per warp
// (the largest key, k_sort_key_pos): all of which the CPU emulator runs.
#pragma once
#include "rt.cuh"

namespace rsigpu {

enum { SRT_NT = 256, SRT_CHUNKS = 16, SRT_TILE = SRT_NT * SRT_CHUNKS, SRT_RADIX = 256, SRT_BITS = 8 };
enum { OFS_NT = 256, OFS_ITEMS = 8, OFS_TILE = OFS_NT * OFS_ITEMS };

// exclusive prefix sum over the block (blockDim.x a multiple of 32, at most 32 warps); ws: one slot per warp
template <class T>
__device__ __forceinline__ T srt_scan_excl(T v, T* ws, T* total) {
  const int lane = (int)(threadIdx.x & 31), w = (int)(threadIdx.x >> 5), nw = (int)(blockDim.x >> 5);
  T inc = v;
  for (int o = 1; o < 32; o <<= 1) { const T up = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += up; }
  __syncthreads();                  // the previous call's readers of ws are done
  if (lane == 31) ws[w] = inc;
  __syncthreads();
  T base = 0, tot = 0;
  for (int k = 0; k < nw; ++k) { const T s = ws[k]; if (k < w) base += s; tot += s; }
  *total = tot;
  return base + inc - v;
}

// keys of the decoder's records: refID, with refID -1 (unplaced) mapped past every reference so that it sorts last
__global__ void k_sort_key_tid(const int* __restrict__ tid, u32 n, u32 n_ref, u32* __restrict__ key) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) key[i] = tid[i] < 0 ? n_ref : (u32)tid[i];
}
// keys of staged reads: pos + 1 (pos >= -1); *kmax = the largest key, which sets the number of passes
__global__ void k_sort_key_pos(const int* __restrict__ pos, u32 n, u32* __restrict__ key, u32* __restrict__ kmax) {
  u32 mx = 0;
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) { const u32 k = (u32)(pos[i] + 1); key[i] = k; mx = max(mx, k); }
  mx = __reduce_max_sync(0xffffffffu, mx);
  if ((threadIdx.x & 31) == 0 && mx) atomicMax(kmax, mx);
}

// per tile: how many keys have each digit
__global__ void __launch_bounds__(SRT_NT) k_sort_hist(const u32* __restrict__ key, u32 n, int shift, u32* __restrict__ hist, u32 ntile) {
  __shared__ u32 h[SRT_RADIX];
  h[threadIdx.x] = 0;
  __syncthreads();
  const u32 base = blockIdx.x * (u32)SRT_TILE;
  for (int c = 0; c < SRT_CHUNKS; ++c) {
    const u32 i = base + (u32)c * SRT_NT + threadIdx.x;
    if (i < n) atomicAdd(&h[(key[i] >> shift) & (SRT_RADIX - 1)], 1u);
  }
  __syncthreads();
  hist[(size_t)threadIdx.x * ntile + blockIdx.x] = h[threadIdx.x];
}

// one block per digit: exclusive scan of its row of tile counts in place, the row's total to dtot[digit]
__global__ void __launch_bounds__(SRT_NT) k_sort_scan_rows(u32* __restrict__ hist, u32 ntile, u32* __restrict__ dtot) {
  __shared__ u32 ws[SRT_NT / 32];
  u32* row = hist + (size_t)blockIdx.x * ntile;
  u32 carry = 0;
  for (u32 b = 0; b < ntile; b += SRT_NT) {
    const u32 i = b + threadIdx.x;
    const u32 v = i < ntile ? row[i] : 0u;
    u32 tot;
    const u32 ex = srt_scan_excl(v, ws, &tot);
    if (i < ntile) row[i] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) dtot[blockIdx.x] = carry;
}

// stable scatter of one tile; idx_in == nullptr: the first pass, the index is the position itself
__global__ void __launch_bounds__(SRT_NT) k_sort_scatter(const u32* __restrict__ key_in, const u32* __restrict__ idx_in, u32 n, int shift,
                                                         const u32* __restrict__ hist, const u32* __restrict__ dtot, u32 ntile,
                                                         u32* __restrict__ key_out, u32* __restrict__ idx_out) {
  __shared__ u32 run[SRT_RADIX];                  // next output slot of each digit
  __shared__ u32 cnt[SRT_NT / 32][SRT_RADIX];     // this chunk's count of each digit per warp
  __shared__ u32 ws[SRT_NT / 32];
  const int t = (int)threadIdx.x, lane = t & 31, w = t >> 5;
  {
    u32 tot;
    const u32 db = srt_scan_excl(dtot[t], ws, &tot);
    run[t] = db + hist[(size_t)t * ntile + blockIdx.x];
  }
  const u32 base = blockIdx.x * (u32)SRT_TILE;
  for (int c = 0; c < SRT_CHUNKS; ++c) {
    for (int k = 0; k < SRT_NT / 32; ++k) cnt[k][t] = 0;
    __syncthreads();
    const u32 i = base + (u32)c * SRT_NT + (u32)t;
    const bool ok = i < n;
    const u32 k = ok ? key_in[i] : 0u, d = ok ? (k >> shift) & (SRT_RADIX - 1) : (u32)SRT_RADIX;
    const unsigned m = __match_any_sync(0xffffffffu, d);
    const unsigned before = m & ((1u << lane) - 1u);
    if (ok && before == 0) cnt[w][d] = (u32)__popc(m);
    __syncthreads();
    if (ok) {
      u32 r = run[d] + (u32)__popc(before);
      for (int q = 0; q < w; ++q) r += cnt[q][d];
      key_out[r] = k;
      idx_out[r] = idx_in ? idx_in[i] : i;
    }
    __syncthreads();
    u32 s = 0;
    for (int q = 0; q < SRT_NT / 32; ++q) s += cnt[q][t];
    run[t] += s;
  }
}

// ---- applying the permutation
struct SortFields {   // any pointer may be null (that field is not carried); cigar_off / qual_off: n + 1 entries
  i64* rec; int* tid; int* pos; int* mpos; int* isize; int* mtid; u16* flag; u8* mapq; u32* cigar_off; u64* qual_off;
};

// out[i] = in[perm[i]] for the fixed fields; out.cigar_off / out.qual_off receive the LENGTHS (k_off_* turn them into offsets)
__global__ void k_sort_gather(const u32* __restrict__ perm, u32 n, SortFields in, SortFields out) {
  for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const u32 j = perm[i];
    if (in.rec) out.rec[i] = in.rec[j];
    if (in.tid) out.tid[i] = in.tid[j];
    out.pos[i] = in.pos[j]; out.mpos[i] = in.mpos[j]; out.isize[i] = in.isize[j]; out.mtid[i] = in.mtid[j];
    out.flag[i] = in.flag[j]; out.mapq[i] = in.mapq[j];
    out.cigar_off[i] = in.cigar_off[j + 1] - in.cigar_off[j];
    out.qual_off[i] = in.qual_off[j + 1] - in.qual_off[j];
  }
}

// exclusive scan of the lengths in place (n entries), the totals to entry n: tile sums, one block over the tile sums, tiles
__global__ void __launch_bounds__(OFS_NT) k_off_tile_sums(const u32* __restrict__ lc, const u64* __restrict__ lq, u32 n, u64* __restrict__ ts, u32 ntile) {
  __shared__ u64 ws[OFS_NT / 32];
  u64 c = 0, q = 0;
  const u32 base = blockIdx.x * (u32)OFS_TILE;
  for (int k = 0; k < OFS_ITEMS; ++k) { const u32 i = base + (u32)k * OFS_NT + threadIdx.x; if (i < n) { c += lc[i]; q += lq[i]; } }
  u64 tc, tq;
  srt_scan_excl(c, ws, &tc);
  srt_scan_excl(q, ws, &tq);
  if (threadIdx.x == 0) { ts[blockIdx.x] = tc; ts[(size_t)ntile + blockIdx.x] = tq; }
}
__global__ void __launch_bounds__(1024) k_off_tile_scan(u64* __restrict__ ts, u32 ntile, u32* __restrict__ lc, u64* __restrict__ lq, u32 n) {
  __shared__ u64 ws[32];
  for (int part = 0; part < 2; ++part) {
    u64* a = ts + (size_t)part * ntile;
    u64 carry = 0;
    for (u32 b = 0; b < ntile; b += blockDim.x) {
      const u32 i = b + threadIdx.x;
      const u64 v = i < ntile ? a[i] : 0ull;
      u64 tot;
      const u64 ex = srt_scan_excl(v, ws, &tot);
      if (i < ntile) a[i] = carry + ex;
      carry += tot;
    }
    if (threadIdx.x == 0) { if (part == 0) lc[n] = (u32)carry; else lq[n] = carry; }
  }
}
__global__ void __launch_bounds__(OFS_NT) k_off_apply(u32* __restrict__ lc, u64* __restrict__ lq, u32 n, const u64* __restrict__ ts, u32 ntile) {
  __shared__ u64 ws[OFS_NT / 32];
  const u32 i0 = blockIdx.x * (u32)OFS_TILE + threadIdx.x * (u32)OFS_ITEMS;   // OFS_ITEMS consecutive entries per thread
  u64 c[OFS_ITEMS], q[OFS_ITEMS], sc = 0, sq = 0;
  for (int k = 0; k < OFS_ITEMS; ++k) {
    const u32 i = i0 + (u32)k;
    c[k] = i < n ? lc[i] : 0u; q[k] = i < n ? lq[i] : 0ull;
    sc += c[k]; sq += q[k];
  }
  u64 tot;
  u64 oc = srt_scan_excl(sc, ws, &tot) + ts[blockIdx.x];
  u64 oq = srt_scan_excl(sq, ws, &tot) + ts[(size_t)ntile + blockIdx.x];
  for (int k = 0; k < OFS_ITEMS; ++k) {
    const u32 i = i0 + (u32)k;
    if (i < n) { lc[i] = (u32)oc; lq[i] = oq; }
    oc += c[k]; oq += q[k];
  }
}

// CIGAR words and quality bytes of read perm[i] to its new offsets; eight lanes per read (as k_bam_payload)
__global__ void k_sort_gather_payload(const u32* __restrict__ perm, u32 n, const u32* __restrict__ coff_in, const u32* __restrict__ cig_in,
                                      const u64* __restrict__ qoff_in, const u8* __restrict__ qual_in, const u32* __restrict__ coff_out,
                                      u32* __restrict__ cig_out, const u64* __restrict__ qoff_out, u8* __restrict__ qual_out) {
  const u32 sub = threadIdx.x & 7u;
  const u32 gid = (blockIdx.x * blockDim.x + threadIdx.x) >> 3, ng = (gridDim.x * blockDim.x) >> 3;
  for (u32 i = gid; i < n; i += ng) {
    const u32 j = perm[i];
    const u32 c0 = coff_in[j], nc = coff_in[j + 1] - c0;
    const u32* cs = cig_in + c0; u32* cd = cig_out + coff_out[i];
    for (u32 k = sub; k < nc; k += 8) cd[k] = cs[k];
    const u64 q0 = qoff_in[j], nq = qoff_in[j + 1] - q0;
    const u8* qs = qual_in + q0; u8* qd = qual_out + qoff_out[i];
    u64 k = sub;
    for (; k + 24 < nq; k += 32) {          // four independent bytes per lane and trip
      const u8 a0 = qs[k], a1 = qs[k + 8], a2 = qs[k + 16], a3 = qs[k + 24];
      qd[k] = a0; qd[k + 8] = a1; qd[k + 16] = a2; qd[k + 24] = a3;
    }
    for (; k < nq; k += 8) qd[k] = qs[k];
  }
}

}  // namespace rsigpu
