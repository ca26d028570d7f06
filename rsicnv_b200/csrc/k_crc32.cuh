// k_crc32.cuh -- CRC-32 of every decoded BGZF block against the CRC in its gzip footer (RFC 1952: the CRC-32 of zlib,
// reflected polynomial 0xEDB88320, init and final xor 0xFFFFFFFF).  Opt-in (rsigpu_set_bgzf_crc): the reference's
// samtools-0.1.18/bgzf.c:277-313 never checks it, htslib and the host route (host/bam_reader.cpp) always do.
//
// One warp per BGZF block, a separate pass after either inflate kernel has written the block's bytes to the decoded
// buffer (blocks are packed back to back there, so a block starts at any alignment and holds 0..65536 bytes).
// The block is treated as right-aligned in a virtual 64 KiB: leading zero bytes leave a CRC register that starts at 0
// unchanged, so lane l can own the fixed virtual slice [2048 l, 2048 (l + 1)) whatever the block's length, compute the
// raw CRC (no init, no final xor) of the real bytes in it, and move it to the end of the virtual 64 KiB by multiplying
// with x^(8 * 2048 * (31 - l)) mod P.  The XOR of the 32 products is the raw CRC of the block.  The init value is folded
// in by starting the register of the lane that holds the block's first byte at 0xFFFFFFFF.
// Each lane reads its slice sequentially, 16 bytes per load once aligned, with slicing-by-4 tables in shared memory.
// The tables are kept in one copy per lane (word (k * 256 + e) * 32 + lane), so the four look-ups of a step never
// meet a bank conflict: 128 KiB of shared memory, one CTA of 16 warps per SM.
#pragma once
namespace rsigpu {

enum {
  CRC_NT = 512, CRC_WARPS = CRC_NT / 32,
  CRC_SLICE = 2048,                                // virtual bytes per lane (32 x 2048 = 64 KiB, the largest BGZF block)
  CRC_SMEM = 4 * 256 * 32 * 4                      // slicing-by-4 tables, one copy per lane
};
#define CRC_POLY 0xEDB88320u

// a * b mod P in the reflected representation (bit 31 is x^0), as zlib's multmodp
__device__ __forceinline__ u32 crc_mulmod(u32 a, u32 b) {
  u32 p = 0;
  for (u32 m = 1u << 31; m; m >>= 1) {
    if (a & m) p ^= b;
    b = (b & 1u) ? (b >> 1) ^ CRC_POLY : b >> 1;
  }
  return p;
}

// err[1] |= BAM_ERR_CRC for a mismatch; err[3] = max(nblk - k) over the failing blocks k (the lowest failing block)
__global__ void __launch_bounds__(CRC_NT, 1) k_bgzf_crc32(const u8* __restrict__ U, const BgzfBlock* __restrict__ blk, int nblk, int* err) {
  RSI_DYN_SMEM(smem);
  u32* tab = reinterpret_cast<u32*>(smem);
  const int lane = (int)(threadIdx.x & 31), warp = (int)(threadIdx.x >> 5);
  // T0 is the byte-at-a-time table, Tk[e] = Tk-1[e] advanced by one zero byte; every entry written to all 32 copies
  for (int k = 0; k < 4; ++k) {
    for (int e = (int)threadIdx.x; e < 256; e += CRC_NT) {
      u32 c;
      if (k == 0) { c = (u32)e; for (int i = 0; i < 8; ++i) c = (c & 1u) ? (c >> 1) ^ CRC_POLY : c >> 1; }
      else { const u32 p = tab[((k - 1) * 256 + e) << 5]; c = (p >> 8) ^ tab[(p & 0xffu) << 5]; }
      for (int l = 0; l < 32; ++l) tab[((k * 256 + e) << 5) + l] = c;
    }
    __syncthreads();
  }
  // x^(8 * 2048 * (31 - lane)) mod P: x^16384 by 14 squarings of x, then a power of it
  u32 step = 1u << 30;
  for (int i = 0; i < 14; ++i) step = crc_mulmod(step, step);
  u32 K = 1u << 31;
  for (int e = 31 - lane; e; e >>= 1) { if (e & 1) K = crc_mulmod(K, step); step = crc_mulmod(step, step); }
  const u32* tl = tab + lane;
#define CRC_T(k, e) tl[((k) * 256 + (e)) << 5]
  for (int k = (int)blockIdx.x * CRC_WARPS + warp; k < nblk; k += (int)gridDim.x * CRC_WARPS) {
    const BgzfBlock B = blk[k];
    const u32 s = 65536u - B.dst_len;                              // the block's first byte in the virtual 64 KiB
    const u32 v0 = s > (u32)lane * CRC_SLICE ? s : (u32)lane * CRC_SLICE, v1 = (u32)(lane + 1) * CRC_SLICE;
    u32 c = 0;
    if (v0 < v1) {
      if (v0 == s) c = 0xffffffffu;
      const u8* p = U + B.dst + (v0 - s);
      const u8* const end = U + B.dst + (v1 - s);
      for (; p < end && (reinterpret_cast<uintptr_t>(p) & 15u); ++p) c = CRC_T(0, (c ^ *p) & 0xffu) ^ (c >> 8);
      for (; p + 16 <= end; p += 16) {
        const uint4 q = *reinterpret_cast<const uint4*>(p);
        c ^= q.x; c = CRC_T(3, c & 0xffu) ^ CRC_T(2, (c >> 8) & 0xffu) ^ CRC_T(1, (c >> 16) & 0xffu) ^ CRC_T(0, c >> 24);
        c ^= q.y; c = CRC_T(3, c & 0xffu) ^ CRC_T(2, (c >> 8) & 0xffu) ^ CRC_T(1, (c >> 16) & 0xffu) ^ CRC_T(0, c >> 24);
        c ^= q.z; c = CRC_T(3, c & 0xffu) ^ CRC_T(2, (c >> 8) & 0xffu) ^ CRC_T(1, (c >> 16) & 0xffu) ^ CRC_T(0, c >> 24);
        c ^= q.w; c = CRC_T(3, c & 0xffu) ^ CRC_T(2, (c >> 8) & 0xffu) ^ CRC_T(1, (c >> 16) & 0xffu) ^ CRC_T(0, c >> 24);
      }
      for (; p < end; ++p) c = CRC_T(0, (c ^ *p) & 0xffu) ^ (c >> 8);
    }
    c = crc_mulmod(K, c);
    for (int o = 16; o; o >>= 1) c ^= __shfl_xor_sync(0xffffffffu, c, o);
    const u32 crc = B.dst_len ? ~c : 0u;                           // the CRC of no bytes is 0
    if (lane == 0 && crc != B.crc) { atomicOr(err + 1, (int)BAM_ERR_CRC); atomicMax(err + 3, nblk - k); }
  }
#undef CRC_T
}

}  // namespace rsigpu
