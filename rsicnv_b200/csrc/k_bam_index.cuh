// k_bam_index.cuh -- the BAI index (SAM spec 5.2, laid out as samtools-0.1.18's bam_index_build writes it) as a by-product of
// the GPU decode (rsigpu_bam_index_begin / rsigpu_bam_index_get).  Runs after k_bam_fields / k_bam_payload, on the records
// they decoded, only when indexing is on.
//
// What an index needs of every record: its begin virtual offset (BGZF block offset << 16 | offset inside the decoded
// block), its tid, the bin stored in the record, pos and the alignment end (bam_calend).  Records are contiguous, so a
// record's END virtual offset is the begin offset of the next record (the host resolves the last record of a feed from
// the next feed, or from where the stream ends).
//   chunks      one entry per run of consecutive records with the same (tid, bin), in file order: (tid, bin, begin voffset,
//               first record, unmapped records before it).  A run's end is the next run's begin.  The host merges them
//               (samtools' merge_chunks: u >> 16 == prev.v >> 16) -- which also joins a run that a feed boundary cut in two.
//   linear      the 16 kbp window w of a reference gets the smallest begin voffset of the records that cover it; voffsets
//               grow in file order, so that is the FIRST covering record.  With M = the largest last window of the earlier
//               records of the same reference (a running maximum), record r is the first to cover exactly the windows
//               (max(w0, M + 1) .. w1]: those ranges are disjoint, at most one per record, and their union is every covered
//               window.  They are appended in any order; the host writes them into the per-reference array.
// Three launches per feed: k_bam_index_rec (per record + per-tile totals), k_bam_index_scan (one CTA: exclusive prefix of
// the tile totals), k_bam_index_emit (per record: chunks at their scanned positions, linear-index ranges).
#pragma once
namespace rsigpu {

enum { BIX_NT = 256, BIX_SCAN_NT = 1024, BIX_SHIFT = 14, BIX_MAX_POS = 1 << 29 };
// cnt slots (u64): chunks, unmapped records, linear ranges, n - first unsorted record, n - first record past 2^29,
// last record's tid / pos / bin, the feed's largest (tid, last window) key
enum { BIX_C_CHUNKS = 0, BIX_C_UNMAP, BIX_C_LIN, BIX_C_UNSORTED, BIX_C_RANGE, BIX_C_LAST_TID, BIX_C_LAST_POS, BIX_C_LAST_BIN, BIX_C_MAXKEY, BIX_C_N };

struct BixChunk { u64 u; int tid; u32 bin; int rec; int unmap; };   // a run of records with one (tid, bin): begin voffset, first record, unmapped before it
struct BixLin { u64 voff; int tid, w0, w1; int pad_; };               // windows w0..w1 of reference tid: first covered by the record at voff

struct BixFeed {
  const u8* U; const i64* bound; const BgzfBlock* blk; int nblk;
  i64 base;                     // file offset of the feed's first byte
  u64 carry_voff;               // begin voffset of the record carried from the previous feed (it starts in front of bound[0])
  int n;                        // records of the feed
  const i64* rec; const int* tid; const int* pos; const u16* flag; const u32* cigar_off; const u32* cigar;
  int has_prev, prev_tid, prev_pos; u32 prev_bin; u64 prev_key;   // the last record of the previous feeds
  u64* beg; u64* key; u32* meta;                // per record: begin voffset, (tid, last window + 1), bin | run start << 16 | unmapped << 17
  int* t_start; int* t_unmap; u64* t_key;       // per tile: totals, replaced by their exclusive prefix in k_bam_index_scan
  BixChunk* chunk; BixLin* lin; u64* cnt;
};

__device__ __forceinline__ u32 bix_bin(const u8* U, i64 p) { return ld32u(U + p + 12) >> 16; }   // bin_mq_nl >> 16 as stored

// bam_calend (samtools-0.1.18/bam.c:17-27): pos + the reference length of the M / D / N ops
__device__ __forceinline__ i64 bix_calend(const u32* cigar, u32 c0, u32 c1, int pos) {
  i64 end = pos;
  for (u32 k = c0; k < c1; ++k) { const u32 op = cigar[k] & 15u; if (op == 0 || op == 2 || op == 3) end += cigar[k] >> 4; }
  return end;
}

__global__ void __launch_bounds__(BIX_NT) k_bam_index_rec(BixFeed F) {
  RSI_CTA_SETUP(c);
  const int r = (int)blockIdx.x * BIX_NT + (int)threadIdx.x;
  int start = 0, unm = 0; u64 key = 0;
  if (r < F.n) {
    const i64 p = F.rec[r];
    const int tid = F.tid[r], pos = F.pos[r];
    const u32 bin = bix_bin(F.U, p);
    // begin voffset: the last block that starts at or before p (a block that ends exactly at p gives way to the next one)
    u64 v = F.carry_voff;
    if (p >= F.bound[0]) {
      int lo = 0, hi = F.nblk - 1;
      while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (F.bound[mid] <= p) lo = mid; else hi = mid - 1; }
      const i64 coff = F.base + (lo ? (i64)F.blk[lo - 1].src + F.blk[lo - 1].src_len + 8 : 0);
      v = ((u64)coff << 16) | (u64)(p - F.bound[lo]);
    }
    // 16 kbp windows of [pos, end): an end <= pos counts as pos + 1
    key = (u64)(u32)tid << 32;
    if (tid >= 0 && pos >= 0) {
      i64 end = bix_calend(F.cigar, F.cigar_off[r], F.cigar_off[r + 1], pos);
      if (end <= pos) end = (i64)pos + 1;
      if (end > BIX_MAX_POS) atomicMax(F.cnt + BIX_C_RANGE, (u64)(F.n - r));
      key |= (u64)(u32)(((end - 1) >> BIX_SHIFT) + 1);
    }
    int pt = F.prev_tid, pp = F.prev_pos; u32 pb = F.prev_bin; bool hp = F.has_prev != 0;
    if (r > 0) { pt = F.tid[r - 1]; pp = F.pos[r - 1]; pb = bix_bin(F.U, F.rec[r - 1]); hp = true; }
    // sorted: refIDs never decrease (unplaced records, refID -1, last) and positions never decrease within a reference
    if (hp && ((u32)tid < (u32)pt || (tid == pt && tid >= 0 && pos < pp))) atomicMax(F.cnt + BIX_C_UNSORTED, (u64)(F.n - r));
    start = r == 0 || tid != pt || bin != pb;      // every feed opens a run: the host's merge joins it to the previous one
    unm = (F.flag[r] & 4) != 0;
    F.beg[r] = v; F.key[r] = key; F.meta[r] = bin | (u32)start << 16 | (u32)unm << 17;
    if (r == F.n - 1) { F.cnt[BIX_C_LAST_TID] = (u64)(u32)tid; F.cnt[BIX_C_LAST_POS] = (u64)(u32)pos; F.cnt[BIX_C_LAST_BIN] = bin; }
  }
  const int ts = c.reduce(start, SumOp()), tu = c.reduce(unm, SumOp());
  const u64 tk = c.reduce(key, MaxOp());
  if (threadIdx.x == 0) { F.t_start[blockIdx.x] = ts; F.t_unmap[blockIdx.x] = tu; F.t_key[blockIdx.x] = tk; }
}

// one CTA: exclusive prefix of the tile totals (run starts and unmapped records summed, keys by maximum from the previous feeds' key)
__global__ void __launch_bounds__(BIX_SCAN_NT) k_bam_index_scan(BixFeed F, int ntiles) {
  RSI_CTA_SETUP(c);
  const int per = (ntiles + c.nthr - 1) / c.nthr;
  const int k0 = imin(c.tid * per, ntiles), k1 = imin(k0 + per, ntiles);
  int ls = 0, lu = 0; u64 lk = 0;
  for (int k = k0; k < k1; ++k) { ls += F.t_start[k]; lu += F.t_unmap[k]; lk = F.t_key[k] > lk ? F.t_key[k] : lk; }
  int tots, totu; u64 totk;
  int bs = c.scan_excl(ls, &tots), bu = c.scan_excl(lu, &totu);
  u64 bk = c.scan_excl_op(lk, MaxOp(), F.prev_key, &totk);
  for (int k = k0; k < k1; ++k) {
    const int s = F.t_start[k], u = F.t_unmap[k]; const u64 kk = F.t_key[k];
    F.t_start[k] = bs; F.t_unmap[k] = bu; F.t_key[k] = bk;
    bs += s; bu += u; bk = kk > bk ? kk : bk;
  }
  if (c.tid == 0) { F.cnt[BIX_C_CHUNKS] = (u64)tots; F.cnt[BIX_C_UNMAP] = (u64)totu; F.cnt[BIX_C_MAXKEY] = totk > F.prev_key ? totk : F.prev_key; }
}

__global__ void __launch_bounds__(BIX_NT) k_bam_index_emit(BixFeed F) {
  RSI_CTA_SETUP(c);
  const int r = (int)blockIdx.x * BIX_NT + (int)threadIdx.x;
  const bool ok = r < F.n;
  const u32 m = ok ? F.meta[r] : 0u;
  const u64 key = ok ? F.key[r] : 0ull;
  const int start = (int)((m >> 16) & 1u), unm = (int)((m >> 17) & 1u);
  int tot; u64 totk;
  const int ci = F.t_start[blockIdx.x] + c.scan_excl(start, &tot);
  const int ub = F.t_unmap[blockIdx.x] + c.scan_excl(unm, &tot);
  u64 mk = c.scan_excl_op(key, MaxOp(), 0ull, &totk);
  mk = F.t_key[blockIdx.x] > mk ? F.t_key[blockIdx.x] : mk;      // the largest key of every earlier record
  if (!ok) return;
  const int tid = F.tid[r];
  if (start) { BixChunk ch; ch.u = F.beg[r]; ch.tid = tid; ch.bin = m & 0xffffu; ch.rec = r; ch.unmap = ub; F.chunk[ci] = ch; }
  if (tid >= 0 && (u32)key != 0u) {
    const int w1 = (int)(u32)key - 1, w0 = F.pos[r] >> BIX_SHIFT;
    const int before = (u32)(mk >> 32) == (u32)tid ? (int)(u32)mk - 1 : -1;   // last window an earlier record of this reference covers
    const int a = before + 1 > w0 ? before + 1 : w0;
    if (a <= w1) {
      BixLin L; L.voff = F.beg[r]; L.tid = tid; L.w0 = a; L.w1 = w1; L.pad_ = 0;
      F.lin[atomicAdd(F.cnt + BIX_C_LIN, 1ull)] = L;
    }
  }
}

}  // namespace rsigpu
