// k_bam.cuh -- BGZF inflate and BAM record decoding on the GPU: compressed file bytes in, the
// position-sorted structure-of-arrays the pileup kernels read out (k_pileup.cuh: ReadSoA).
//
// Replaces, for the `rsicnv rsi -b` path (reference file:line relative to src/):
//   BGZF block inflate       samtools-0.1.18/bgzf.c:277-313 (inflate_block: raw deflate, -15 window, no CRC check)
//   block header             samtools-0.1.18/bgzf.c:56-70, 258-275 (check_header: gzip magic, FEXTRA, 'B','C' subfield)
//   bam_read1 / bam1_core_t  samtools-0.1.18/bam.c:179-210, bam.h:131-155 (32-byte core, name, CIGAR, 4-bit seq, qual)
//   the per-record fields load_data_from_bam and cnv_stat read  loaddata.cpp:312-335, pairrd.cpp:622-748
//
// Design.  A BGZF block (<= 64 KiB decoded) is an independent raw-deflate stream, and a chr19-sized BAM holds ~36 k of
// them.  Two inflate kernels, picked per feed by the number of blocks (rsigpu.cu): here one THREAD inflates one block --
// 32 unrelated streams per warp in lock-step, latency-bound, a launch costs 30-38 ms for anything up to a chr19-sized
// chunk and ~58 ms for an 80 k-block one -- and k_inflate_warp.cuh gives a block to a whole warp (time proportional to
// the bytes; better below ~28 k blocks).  This kernel's Huffman decode has three levels: a 6-bit direct table in shared
// memory (the frequent literal/length codes), 9/6-bit direct tables in global memory (per thread, warp-interleaved,
// L1/L2 resident) and the canonical count/symbol walk for longer codes.  The 32 lanes of a warp are kept converged -- a few
// symbols per lane per step, table construction as a separate phase -- and the LZ77 matches of all lanes are copied by
// the whole warp.
// BAM records are a linked list (each starts with its own length) and may straddle BGZF blocks, so their
// starts are found speculatively and then proven: every block guesses its first record start with a
// plausibility test and walks the list to the end of the block (k_bam_chain); one CTA checks that each
// guess equals the position the previous block's walk ended at, starting from the known first record --
// by induction every start is then exact -- and re-walks the rare block whose guess was wrong
// (k_bam_verify).  Records are then scattered field by field into arrays (k_bam_fields, k_bam_payload).
#pragma once
#include "k_pileup.cuh"

namespace rsigpu {

#ifndef INF_FB_BITS
#define INF_FB_BITS 9
#endif
#ifndef INF_SB_BITS
#define INF_SB_BITS 6
#endif
#ifndef INF_DB_BITS
#define INF_DB_BITS 6
#endif
enum {
  INF_NT = 64,                     // threads per CTA, one BGZF block per thread
  INF_SB = INF_SB_BITS,            // bits of the literal/length code's FIRST-level direct table, in shared memory (2^SB u16 per thread; >= 6)
  INF_FB = INF_FB_BITS, INF_DB = INF_DB_BITS,   // bits of the direct-lookup tables (literal/length, distance)
  INF_LF = 0,                      // per-thread table layout in GLOBAL memory, in u16 slots
  INF_LS = INF_LF + (1 << INF_FB), // literal/length symbols ordered by code
  INF_DF = INF_LS + 288,
  INF_DS = INF_DF + (1 << INF_DB),
  INF_GSLOTS = INF_DS + 32,
  INF_LC = 0, INF_DC = 16,         // code-length counts: shared memory, 16 u16 each per thread
  INF_NC = 32,                     // next code per length while a table is built (shared, 16 u16 per thread)
  INF_LX = 48, INF_DX = 50,        // canonical-decode state after the direct table's bits: first, index (2 u16 per table)
  INF_SSLOTS = 52                  // u16 slots of shared memory per thread; plus 128 bytes for the code-length code's direct table
};
// table scratch for n BGZF blocks (whole warps)
#define RSI_INFLATE_TAB_BYTES(nblk) ((size_t)(((nblk) + 31) / 32) * 32 * INF_GSLOTS * 2)

enum { BAM_HEAD = 16 << 20 };      // room in front of the decoded blocks for the partial record carried from the previous chunk
#define BAM_NONE (-1ll)
#define BAM_TAIL 0x7fffffffffffffffll
enum { BAM_ERR_INFLATE = 1, BAM_ERR_RECORD = 2, BAM_ERR_RUNS = 4, BAM_ERR_CRC = 8 };

struct BgzfBlock { u64 dst; u32 src, src_len, dst_len, crc; };   // payload offset/length in the compressed chunk, offset/length in the decoded buffer, footer CRC32

struct BitIn {
  const u8* base; u32 pos, end;   // word-aligned base, next byte to load, one past the payload (both relative to base)
  u64 buf; int cnt;
  u32 nextw;                      // the word at `pos`, loaded one refill ahead so that a refill never waits for memory
};
__device__ __forceinline__ u32 bits_word(const BitIn& b, u32 pos) { return pos < b.end + 8 ? *reinterpret_cast<const u32*>(b.base + pos) : 0u; }
// byte loads until the next load is word aligned (at most 3), then prime the look-ahead word
__device__ __forceinline__ void bits_align(BitIn& b) {
  while ((b.pos & 3u) && b.cnt <= 56) { b.buf |= (u64)(b.pos < b.end + 8 ? b.base[b.pos] : 0) << b.cnt; b.cnt += 8; b.pos++; }
  b.nextw = bits_word(b, b.pos);
}
// at least 33 valid bits afterwards; the payload is followed by the block's 8-byte footer, so the last word load stays inside the chunk
__device__ __forceinline__ void bits_refill(BitIn& b) {
  if (b.cnt <= 32) {
    b.buf |= (u64)b.nextw << b.cnt; b.cnt += 32; b.pos += 4;
    b.nextw = bits_word(b, b.pos);
  }
}
__device__ __forceinline__ u32 bits_take(BitIn& b, int n) { const u32 v = (u32)(b.buf & ((1ull << n) - 1)); b.buf >>= n; b.cnt -= n; return v; }

// Per-thread Huffman tables.  The big ones (9/6-bit direct tables, symbols by code) live in global memory and stay in L2:
// at 1.8 KB per thread, shared memory would hold a few warps per SM, and one thread's decode loop is a chain of dependent
// loads that only many resident warps can hide.  A 6-bit first level for the literal/length code (sf) is in shared memory.  Slot i of lane l is at g[i * 32 + l] (a warp's tables are interleaved, so
// the construction loops -- same i in every lane -- are coalesced).  The 2 x 16 code-length counts sit in shared memory.
struct InfTabs { u16* g; u16* s; u16* sf; u16* sd; int lane, stid; };   // sd: the distance code's first-level table in shared memory (INF_DSH bits, 0 = none)
#ifndef INF_DSH
#define INF_DSH 0
#endif
#define INF_SH(sh, i) (sh)[(i) * INF_NT + T.stid]
#define INF_G(i) T.g[(size_t)(i) * 32 + T.lane]
#define INF_C(i) T.s[(i) * INF_NT + T.stid]
#define INF_CL(i) reinterpret_cast<u8*>(&T.sf[((i) >> 1) * INF_NT + T.stid])[(i) & 1]   /* the code-length code's 128 one-byte entries live in 64 of the thread's own first-level slots while a header is parsed */
#define INF_SF(i) T.sf[(i) * INF_NT + T.stid]

// canonical code from code lengths (count/symbol form, plus a direct table for codes of <= fb bits whose
// entries are symbol << 4 | length).  Returns < 0 for an over-subscribed set, > 0 for an incomplete one.
// One pass over the symbols: codes are handed out in symbol order per length (next-code counters in shared memory), so the
// direct table is filled without reading back anything that was just written to global memory.
__device__ int inf_construct(const InfTabs& T, const u8* lens, int n, int fast, int fb, int cnts, int syms, int xs, int sfb, u16* sh) {
  for (int l = 0; l < 16; ++l) INF_C(cnts + l) = 0;
  for (int s = 0; s < n; ++s) INF_C(cnts + lens[s]) += 1;
  for (int i = 0; i < (1 << fb); ++i) INF_G(fast + i) = 0;
  for (int i = 0; i < (sfb ? (1 << sfb) : 0); ++i) INF_SH(sh, i) = 0;
  if (INF_C(cnts) == n) return 0;
  int left = 1;
  for (int l = 1; l <= 15; ++l) { left <<= 1; left -= (int)INF_C(cnts + l); if (left < 0) return left; }
  u16 offs[16];
  offs[1] = 0;
  for (int l = 1; l < 15; ++l) offs[l + 1] = (u16)(offs[l] + INF_C(cnts + l));
  { int code = 0; for (int l = 1; l <= 15; ++l) { INF_C(INF_NC + l) = (u16)code; code = (code + (int)INF_C(cnts + l)) << 1; } }
  { int first = 0, index = 0; for (int l = 1; l <= fb; ++l) { const int cn = (int)INF_C(cnts + l); index += cn; first += cn; first <<= 1; } INF_C(xs) = (u16)first; INF_C(xs + 1) = (u16)index; }
  for (int s = 0; s < n; ++s) {
    const int l = lens[s];
    if (!l) continue;
    INF_G(syms + offs[l]) = (u16)s; offs[l]++;
    const u32 code = INF_C(INF_NC + l); INF_C(INF_NC + l) = (u16)(code + 1);
    if (l <= fb) {
      const u32 rev = __brev(code) >> (32 - l);
      const u16 e = (u16)((s << 4) | l);
      for (u32 k = rev; k < (1u << fb); k += (1u << l)) INF_G(fast + k) = e;
      if (l <= sfb) for (u32 k = rev; k < (1u << sfb); k += (1u << l)) INF_SH(sh, k) = e;
    }
  }
  return left;
}
__device__ __forceinline__ int inf_decode(BitIn& b, const InfTabs& T, int fast, int fb, int cnts, int syms, int xs, int sfb, const u16* sh) {
  const u32 low = (u32)(b.buf & ((1u << fb) - 1));
  if (sfb) {   // codes of <= sfb bits (the frequent symbols): one shared-memory look-up, no trip to L1/L2
    const u32 e0 = INF_SH(sh, low & ((1u << sfb) - 1));
    if (e0) { const int l = (int)(e0 & 15u); b.buf >>= l; b.cnt -= l; return (int)(e0 >> 4); }
  }
  const u32 e = INF_G(fast + low);
  if (e) { const int l = (int)(e & 15u); b.buf >>= l; b.cnt -= l; return (int)(e >> 4); }
  // longer than fb bits: canonical walk (count / first / index per length), resumed after the fb bits already seen
  int code = (int)((__brev(low) >> (32 - fb)) << 1), first = (int)INF_C(xs), index = (int)INF_C(xs + 1);
  u64 bits = b.buf >> fb;
  for (int l = fb + 1; l <= 15; ++l) {
    code |= (int)(bits & 1); bits >>= 1;
    const int cn = (int)INF_C(cnts + l);
    if (code - cn < first) { b.buf >>= l; b.cnt -= l; return (int)INF_G(syms + index + (code - first)); }
    index += cn; first += cn; first <<= 1; code <<= 1;
  }
  return -1;
}
// the code-length code (19 symbols, codes of <= 7 bits): a 128-entry direct table in shared memory, entry = symbol << 3 | length
__device__ int inf_construct_cl(const InfTabs& T, const u8* lens) {
  for (int l = 0; l < 8; ++l) INF_C(INF_LC + l) = 0;
  for (int s = 0; s < 19; ++s) INF_C(INF_LC + (lens[s] & 7)) += 1;
  for (int i = 0; i < 128; ++i) INF_CL(i) = 0;
  int left = 1, code = 0;
  for (int l = 1; l < 8; ++l) { left <<= 1; left -= (int)INF_C(INF_LC + l); INF_C(INF_NC + l) = (u16)code; code = (code + (int)INF_C(INF_LC + l)) << 1; }
  if (left != 0) return left < 0 ? -1 : 1;
  for (int s = 0; s < 19; ++s) {
    const int l = lens[s];
    if (!l) continue;
    const u32 c = INF_C(INF_NC + l); INF_C(INF_NC + l) = (u16)(c + 1);
    const u32 rev = __brev(c) >> (32 - l);
    const u8 e = (u8)((s << 3) | l);
    for (u32 k = rev; k < 128u; k += (1u << l)) INF_CL(k) = e;
  }
  return 0;
}
__device__ __forceinline__ int inf_decode_cl(BitIn& b, const InfTabs& T) {
  const u32 e = INF_CL((u32)(b.buf & 127u));
  if (!e) return -1;
  const int l = (int)(e & 7u); b.buf >>= l; b.cnt -= l;
  return (int)(e >> 3);
}

// One raw-deflate stream -> dst[0, dst_len), as a stepper: the lanes of a warp work on 32 different streams, and a
// free-running per-lane loop lets the hardware serialise them (one lane runs its whole stream while the others wait).
// inf_step does ONE unit of work -- a block header with its tables, a stored block, or one literal/length symbol with
// its match copy -- and the kernel re-converges the warp after every step.
struct InfState {
  BitIn b; u32 o, dst_len; u8* dst;
  int phase;      // 0: at a block header, 1: inside a Huffman block, 2: finished (rc = 0 ok)
  int last, rc;
  u32 m_len, m_dist;   // match decoded by the last inf_symbol, not yet copied
};
enum { INF_HEADER = 0, INF_SYMS = 1, INF_DONE = 2 };

__device__ __forceinline__ void inf_fail(InfState& S, int rc) { S.rc = rc; S.phase = INF_DONE; }

__device__ __noinline__ void inf_block_header(InfState& S, const InfTabs& T) {
  BitIn& b = S.b;
  bits_refill(b);
  S.last = (int)bits_take(b, 1);
  const u32 type = bits_take(b, 2);
  if (type == 0) {   // stored
    bits_take(b, b.cnt & 7);
    bits_refill(b);
    const u32 len = bits_take(b, 16); bits_refill(b); const u32 nlen = bits_take(b, 16);
    if ((len ^ 0xffffu) != nlen) return inf_fail(S, 2);
    if (S.o + len > S.dst_len) return inf_fail(S, 3);
    u32 k = 0;      // bytes still in the bit buffer, then straight from memory
    while (k < len && b.cnt >= 8) { S.dst[S.o + k++] = (u8)bits_take(b, 8); }
    for (; k < len; ++k) { if (b.pos >= b.end) return inf_fail(S, 4); S.dst[S.o + k] = b.base[b.pos++]; }
    if (b.cnt == 0) bits_align(b);   // bytes were read straight from memory: get back to word loads (loaded-but-unused whole bytes stay in the buffer)
    S.o += len;
    if (S.last) { S.rc = S.o == S.dst_len ? 0 : 18; S.phase = INF_DONE; }
    return;
  }
  if (type == 3) return inf_fail(S, 1);
  u8 lens[320];
  if (type == 1) {
    for (int s = 0; s < 144; ++s) lens[s] = 8;
    for (int s = 144; s < 256; ++s) lens[s] = 9;
    for (int s = 256; s < 280; ++s) lens[s] = 7;
    for (int s = 280; s < 288; ++s) lens[s] = 8;
    inf_construct(T, lens, 288, INF_LF, INF_FB, INF_LC, INF_LS, INF_LX, INF_SB, T.sf);
    for (int s = 0; s < 30; ++s) lens[s] = 5;
    inf_construct(T, lens, 30, INF_DF, INF_DB, INF_DC, INF_DS, INF_DX, INF_DSH, T.sd);
  } else {
    bits_refill(b);
    const int nlen = (int)bits_take(b, 5) + 257, ndist = (int)bits_take(b, 5) + 1, ncode = (int)bits_take(b, 4) + 4;
    if (nlen > 286 || ndist > 30) return inf_fail(S, 5);
    const u8 order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    for (int i = 0; i < 19; ++i) lens[i] = 0;
    for (int i = 0; i < ncode; ++i) { bits_refill(b); lens[order[i]] = (u8)bits_take(b, 3); }
    if (inf_construct_cl(T, lens) != 0) return inf_fail(S, 6);   // the code-length code must be complete
    int idx = 0;
    while (idx < nlen + ndist) {
      bits_refill(b);
      const int sym = inf_decode_cl(b, T);
      if (sym < 0) return inf_fail(S, 7);
      if (sym < 16) lens[idx++] = (u8)sym;
      else {
        int rep; u8 v = 0;
        if (sym == 16) { if (idx == 0) return inf_fail(S, 8); v = lens[idx - 1]; rep = 3 + (int)bits_take(b, 2); }
        else if (sym == 17) rep = 3 + (int)bits_take(b, 3);
        else rep = 11 + (int)bits_take(b, 7);
        if (idx + rep > nlen + ndist) return inf_fail(S, 9);
        while (rep--) lens[idx++] = v;
      }
    }
    if (lens[256] == 0) return inf_fail(S, 10);
    int r = inf_construct(T, lens, nlen, INF_LF, INF_FB, INF_LC, INF_LS, INF_LX, INF_SB, T.sf);
    if (r < 0 || (r > 0 && nlen - (int)INF_C(INF_LC) != 1)) return inf_fail(S, 11);       // incomplete only allowed for a single code
    r = inf_construct(T, lens + nlen, ndist, INF_DF, INF_DB, INF_DC, INF_DS, INF_DX, INF_DSH, T.sd);
    if (r < 0 || (r > 0 && ndist - (int)INF_C(INF_DC) != 1)) return inf_fail(S, 12);
  }
  S.phase = INF_SYMS;
}

// One step of a lane: up to INF_LITS literals (most symbols of BAM data are literals: bases, names, fields), ended early by
// a length symbol -- whose match is then copied by the whole warp -- or by the end of the deflate block.  Several literals
// per step amortise the per-step costs of the warp (re-convergence, the search for pending matches, the copy rounds).
#ifndef INF_LITS
#define INF_LITS 4
#endif
__device__ __forceinline__ void inf_symbol(InfState& S, const InfTabs& T, const u16* tab) {
  BitIn& b = S.b;
  int sym = 0;
#pragma unroll 1
  for (int rep = 0; rep < INF_LITS; ++rep) {
    bits_refill(b);
    sym = inf_decode(b, T, INF_LF, INF_FB, INF_LC, INF_LS, INF_LX, INF_SB, T.sf);
    if (sym >= 256) break;
    if (sym < 0) return inf_fail(S, 13);
    if (S.o >= S.dst_len) return inf_fail(S, 3);
    S.dst[S.o++] = (u8)sym;
  }
  if (sym < 256) return;
  if (sym == 256) {
    if (b.pos > b.end + 16) return inf_fail(S, 17);
    if (S.last) { S.rc = S.o == S.dst_len ? 0 : 18; S.phase = INF_DONE; } else S.phase = INF_HEADER;
    return;
  }
  sym -= 257;
  if (sym >= 29) return inf_fail(S, 14);
  const u32 len = (u32)tab[sym] + bits_take(b, (int)tab[29 + sym]);
  bits_refill(b);
  const int ds = inf_decode(b, T, INF_DF, INF_DB, INF_DC, INF_DS, INF_DX, INF_DSH, T.sd);
  if (ds < 0 || ds >= 30) return inf_fail(S, 15);
  const u32 dist = (u32)tab[58 + ds] + bits_take(b, (int)tab[88 + ds]);
  if (dist > S.o) return inf_fail(S, 16);
  if (S.o + len > S.dst_len) return inf_fail(S, 3);
  S.m_len = len; S.m_dist = dist;      // copied by the whole warp (inf_warp_copy) before the next symbol
}

// The pending matches of all 32 lanes, copied by the whole warp.  A match byte i comes from i - dist, which for i >= dist is
// a byte of the same match: the source is periodic, out[i] = src[i mod dist], so every byte can be read from data that was
// complete before the copy began -- no byte depends on another one of this round.  The bytes of all lanes' matches are laid
// end to end and dealt to the lanes INF_CPB consecutive bytes each, 32 * INF_CPB per round (one round covers nearly every
// step: a match is ~10 bytes and about three lanes in four have one).  Who owns a flattened byte comes from shared memory
// instead of a search over shuffles: every lane posts its match (destination, first flattened byte, length, distance) and
// marks the byte where its match starts with its lane number; a running maximum over the marks, first inside the lane's
// INF_CPB bytes and then across the lanes, names the owner of every byte.  All loads of a round are independent and
// consecutive lanes touch consecutive addresses, instead of one lane copying byte by byte (a load -> store -> load chain
// through L2) while 31 wait.
#ifndef INF_CPB
#define INF_CPB 4
#endif
struct InfPending { u8* a[INF_CPB]; u32 v[INF_CPB]; };   // bytes loaded by the last round of inf_warp_copy, stored by the next call (a == nullptr: none)

__device__ __forceinline__ void inf_flush(InfPending& P) {
#pragma unroll
  for (int k = 0; k < INF_CPB; ++k) if (P.a[k]) { *P.a[k] = (u8)P.v[k]; P.a[k] = nullptr; }
}
// The loads of the LAST round are left in flight: their stores are issued by the next call (or by inf_flush), after the
// next symbols have been decoded, so the L2 round trip of the copy overlaps the table look-ups of the decode instead of
// adding to them.  Stores of a call are issued before its loads, with a warp barrier in between (memory ordering among the
// lanes), because a match may read what the previous one wrote.
// mrec: 32 x uint4 of the warp (destination low/high, first flattened byte, length << 16 | distance - 1); mhead: 32 * INF_CPB mark bytes
__device__ __forceinline__ void inf_warp_copy(InfState& S, int lane, InfPending& P, uint4* mrec, u8* mhead) {
  const u32 len = S.m_len;
  if (!__any_sync(0xffffffffu, len != 0)) return;
  u32 incl = len;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const u32 up = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += up; }
  const u32 total = __shfl_sync(0xffffffffu, incl, 31);
  const u32 excl = incl - len;
  {
    const u64 to_bits = (u64)(size_t)(S.dst + S.o);
    mrec[lane] = make_uint4((u32)to_bits, (u32)(to_bits >> 32), excl, (len << 16) | (S.m_dist - 1u));
  }
  for (u32 t0 = 0; t0 < total; t0 += 32 * INF_CPB) {
#pragma unroll
    for (int k = 0; k < INF_CPB; k += 4) *reinterpret_cast<u32*>(mhead + lane * INF_CPB + k) = 0u;
    __syncwarp();
    if (len != 0 && excl < t0 + 32 * INF_CPB && incl > t0) mhead[excl > t0 ? excl - t0 : 0u] = (u8)(lane + 1);   // the match that straddles t0 marks byte 0
    __syncwarp();
    u32 own[INF_CPB], m = 0;
#pragma unroll
    for (int k = 0; k < INF_CPB; k += 4) {
      const u32 hw = *reinterpret_cast<const u32*>(mhead + lane * INF_CPB + k);
#pragma unroll
      for (int q = 0; q < 4; ++q) { const u32 hq = (hw >> (8 * q)) & 255u; m = hq > m ? hq : m; own[k + q] = m; }
    }
    u32 sc = m;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const u32 up = __shfl_up_sync(0xffffffffu, sc, o); if (lane >= o) sc = up > sc ? up : sc; }
    u32 carry = __shfl_up_sync(0xffffffffu, sc, 1);
    if (lane == 0) carry = 0;
    inf_flush(P);
    __syncwarp();
#pragma unroll
    for (int k = 0; k < INF_CPB; ++k) {
      const u32 t = t0 + (u32)(lane * INF_CPB + k);
      if (t < total) {
        const u32 j1 = own[k] > carry ? own[k] : carry;      // owner's lane + 1
        const uint4 r = mrec[j1 - 1];
        u8* tj = reinterpret_cast<u8*>((size_t)(((u64)r.y << 32) | r.x));
        const u32 i = t - r.z, dist = (r.w & 0xffffu) + 1u;
        const u32 si = i < dist ? i : i % dist;
        P.a[k] = tj + i; P.v[k] = *(tj - dist + si);
      }
    }
  }
  S.o += len; S.m_len = 0;
}

// inflate: one thread per BGZF block of the chunk, the warp re-converged after every step
#ifndef INF_MINB
#define INF_MINB 16      // <= 64 registers: the inflate launches of several contigs fit an SM side by side
#endif
__global__ void __launch_bounds__(INF_NT, INF_MINB) k_bgzf_inflate(const u8* __restrict__ comp, const BgzfBlock* __restrict__ blk, int nblk, u8* __restrict__ U,
                                                         u16* __restrict__ tabs, int* __restrict__ err) {
  __shared__ u16 tab[120];
  __shared__ u16 cnts[INF_SSLOTS * INF_NT];
  __shared__ u16 sfast[(1 << INF_SB) * INF_NT];   // first-level literal/length table; doubles as the code-length code's table while a header is parsed
  __shared__ uint4 mrec[INF_NT];                  // the matches of a copy round, one per lane
  __shared__ __align__(8) u8 mhead[INF_NT * INF_CPB];   // who owns which flattened byte of the round
  __shared__ u16 sdist[(INF_DSH ? (1 << INF_DSH) : 1) * INF_NT];   // first-level distance table (optional; measured: 46.9 vs 48.0 ms with 6 bits, not worth the occupancy)
  {
    const u16 lbase[29] = {3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 15, 17, 19, 23, 27, 31, 35, 43, 51, 59, 67, 83, 99, 115, 131, 163, 195, 227, 258};
    const u16 lext[29] = {0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 2, 2, 2, 2, 3, 3, 3, 3, 4, 4, 4, 4, 5, 5, 5, 5, 0};
    const u16 dbase[30] = {1, 2, 3, 4, 5, 7, 9, 13, 17, 25, 33, 49, 65, 97, 129, 193, 257, 385, 513, 769, 1025, 1537, 2049, 3073, 4097, 6145, 8193, 12289, 16385, 24577};
    const u16 dext[30] = {0, 0, 0, 0, 1, 1, 2, 2, 3, 3, 4, 4, 5, 5, 6, 6, 7, 7, 8, 8, 9, 9, 10, 10, 11, 11, 12, 12, 13, 13};
    for (int i = (int)threadIdx.x; i < 29; i += INF_NT) { tab[i] = lbase[i]; tab[29 + i] = lext[i]; }
    for (int i = (int)threadIdx.x; i < 30; i += INF_NT) { tab[58 + i] = dbase[i]; tab[88 + i] = dext[i]; }
  }
  __syncthreads();
  const int k = (int)blockIdx.x * INF_NT + (int)threadIdx.x;
  InfTabs T; T.lane = (int)(threadIdx.x & 31); T.stid = (int)threadIdx.x; T.s = cnts; T.sf = sfast; T.sd = sdist;
  T.g = tabs + (size_t)(k >> 5) * 32 * INF_GSLOTS;
  InfState S;
  S.phase = INF_DONE; S.rc = 0; S.o = 0; S.dst_len = 0; S.dst = U; S.last = 0; S.m_len = 0; S.m_dist = 1;
  S.b.base = comp; S.b.pos = 0; S.b.end = 0; S.b.buf = 0; S.b.cnt = 0;
  if (k < nblk) {
    const BgzfBlock B = blk[k];
    if (B.dst_len) {
      const u8* src = comp + B.src;
      const u32 mis = (u32)((size_t)src & 3u);
      S.b.base = src - mis; S.b.pos = mis; S.b.end = B.src_len + mis;
      bits_align(S.b);
      S.dst = U + B.dst; S.dst_len = B.dst_len; S.phase = INF_HEADER;
    }
  }
  InfPending P;
#pragma unroll
  for (int k = 0; k < INF_CPB; ++k) { P.a[k] = nullptr; P.v[k] = 0; }
  uint4* const wrec = mrec + (threadIdx.x & ~31u);
  u8* const whead = mhead + (threadIdx.x & ~31u) * INF_CPB;
  while (__any_sync(0xffffffffu, S.phase != INF_DONE)) {
    // lanes that need a block header (table construction: long) go first and together; the others decode symbols
    if (__any_sync(0xffffffffu, S.phase == INF_HEADER)) { if (S.phase == INF_HEADER) { InfState H = S; inf_block_header(H, T); S = H; } }   // out of line: a copy keeps S in registers
    else {
#pragma unroll 1
      for (int it = 0; it < 8; ++it) { if (S.phase == INF_SYMS) inf_symbol(S, T, tab); __syncwarp(); inf_warp_copy(S, T.lane, P, wrec, whead); }
    }
  }
  inf_flush(P);
  if (S.rc) { atomicOr(err + 1, (int)BAM_ERR_INFLATE); atomicMax(err + 2, S.rc); }
}

}  // namespace rsigpu
#include "k_inflate_warp.cuh"
namespace rsigpu {

// ---------------------------------------------------------------------------------------------
// records
__device__ __forceinline__ u32 ld32u(const u8* p) { return (u32)p[0] | ((u32)p[1] << 8) | ((u32)p[2] << 16) | ((u32)p[3] << 24); }

struct BamChunk {
  const u8* U;          // decoded stream of this chunk; valid bytes [u_begin, u_end)
  i64 u_begin, u_end;   // u_begin = start of the first record (a carried partial record lies in front of BAM_HEAD)
  const i64* bound;     // nblk + 1 boundaries of the decoded BGZF blocks in U (bound[0] may be > u_begin)
  int nblk, n_ref;
};
struct BamChain {       // per BGZF block
  i64* first;           // first record start inside the block (BAM_NONE: none)
  i64* endp;            // where the walk from `first` stops: first record start at or after the block's end, BAM_TAIL if the walk met the chunk's incomplete last record
  i64* tailp;           // start of that incomplete record (valid when endp == BAM_TAIL)
  int* cnt; int* ncig; i64* nq;   // records started in the block, their CIGAR ops and quality bytes
};

// bam1_core_t sanity (bam.h:131-155): used to GUESS a record start, and as the corruption check of the walk
__device__ bool bam_core_ok(const BamChunk& C, i64 p, i64* next) {
  if (p + 36 > C.u_end) return false;
  const u8* r = C.U + p;
  const u32 bs = ld32u(r);
  if (bs < 32u || bs > (1u << 28)) return false;
  const int tid = (int)ld32u(r + 4), pos = (int)ld32u(r + 8);
  if (tid < -1 || tid >= C.n_ref || pos < -1) return false;
  const u32 l_name = r[12], n_cig = (u32)r[16] | ((u32)r[17] << 8);
  const int l_seq = (int)ld32u(r + 20);
  const int mtid = (int)ld32u(r + 24), mpos = (int)ld32u(r + 28);
  if (l_name < 1u || l_seq < 0 || mtid < -1 || mtid >= C.n_ref || mpos < -1) return false;
  const u64 need = 32ull + l_name + 4ull * n_cig + ((u64)l_seq + 1) / 2 + (u64)l_seq;
  if (need > (u64)bs) return false;
  if (p + 36 + (i64)l_name <= C.u_end && r[36 + l_name - 1] != 0) return false;
  *next = p + 4 + (i64)bs;
  return true;
}

// walk the record list from p while records START before `stop`; false if a record fails the core check (a wrong start,
// or a corrupt file).  The per-block results are written either way.
__device__ bool bam_walk(const BamChunk& C, i64 p, i64 stop, int k, const BamChain& H) {
  int cnt = 0, ncig = 0; i64 nq = 0, endp = 0, tailp = 0; bool clean = true;
  for (;;) {
    if (p >= stop) {                                                                  // the landing position must look like a record too
      i64 q = p, n2;
      for (int hop = 0; hop < 3 && clean && q + 36 <= C.u_end; ++hop) { if (!bam_core_ok(C, q, &n2)) clean = false; q = n2; }
      endp = p; break;
    }
    if (p + 4 > C.u_end) { endp = BAM_TAIL; tailp = p; break; }                       // the chunk ends inside the length field
    if (p + 36 > C.u_end) {                                                           // ... inside the fixed-size core
      const u32 bs = ld32u(C.U + p);
      clean = bs >= 32u && bs <= (1u << 28);
      endp = BAM_TAIL; tailp = p; break;
    }
    i64 nx;
    if (!bam_core_ok(C, p, &nx)) { clean = false; endp = BAM_TAIL; tailp = p; break; }
    if (nx > C.u_end) { endp = BAM_TAIL; tailp = p; break; }                          // ... inside the record: carried to the next chunk
    ++cnt; ncig += (int)((u32)C.U[p + 16] | ((u32)C.U[p + 17] << 8)); nq += (i64)(int)ld32u(C.U + p + 20);
    p = nx;
  }
  H.endp[k] = endp; H.tailp[k] = tailp; H.cnt[k] = cnt; H.ncig[k] = ncig; H.nq[k] = nq;
  return clean;
}
__device__ __forceinline__ void bam_no_start(int k, const BamChain& H) { H.first[k] = BAM_NONE; H.endp[k] = BAM_NONE; H.tailp[k] = 0; H.cnt[k] = 0; H.ncig[k] = 0; H.nq[k] = 0; }

// Guess: the first position of the block that passes the core check AND from which the list walks cleanly to the end of
// the block (a few hundred records) and lands on something that looks like a record -- wrong guesses that survive this are
// practically impossible, and k_bam_verify does not depend on it.  One thread per BGZF block; scanning and walking are
// written as a state machine advanced one unit per iteration of a warp-uniform loop, so that the 32 lanes (32 different
// blocks) stay converged instead of running their walks one after the other.
__global__ void k_bam_chain(BamChunk C, BamChain H) {
  const int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  enum { SCAN = 0, WALK = 1, DONE = 2 };
  int phase = DONE;
  i64 ub = 0, ue = 0, cand = 0, p = 0, nq = 0; int cnt = 0, ncig = 0;
  if (k < C.nblk) {
    ub = C.bound[k]; ue = C.bound[k + 1];
    if (k == 0) { if (C.u_begin < ue) { H.first[k] = C.u_begin; bam_walk(C, C.u_begin, ue, k, H); } else bam_no_start(k, H); }
    else { phase = SCAN; cand = ub; }
  }
  while (__any_sync(0xffffffffu, phase != DONE)) {
    if (phase == SCAN) {
      if (cand >= ue) { bam_no_start(k, H); phase = DONE; }
      else {
        i64 nx; bool ok = bam_core_ok(C, cand, &nx);
        if (ok) {   // a guess (only a guess) must not carry megabytes of optional fields: block_size close to what the core implies
          const u8* r = C.U + cand;
          const u64 need = 32ull + r[12] + 4ull * ((u32)r[16] | ((u32)r[17] << 8)) + ((u64)ld32u(r + 20) + 1) / 2 + (u64)ld32u(r + 20);
          ok = (u64)ld32u(r) - need <= 65536ull;
        }
        if (ok) { phase = WALK; p = cand; cnt = 0; ncig = 0; nq = 0; } else ++cand;
      }
    } else if (phase == WALK) {
      // one record per iteration: the same rules as bam_walk
      bool fail = false, fin = false; i64 endp = 0, tailp = 0;
      if (p >= ue) {
        i64 q = p, n2;
        for (int hop = 0; hop < 3 && !fail && q + 36 <= C.u_end; ++hop) { if (!bam_core_ok(C, q, &n2)) fail = true; q = n2; }
        endp = p; fin = true;
      } else if (p + 4 > C.u_end) { endp = BAM_TAIL; tailp = p; fin = true; }
      else if (p + 36 > C.u_end) { const u32 bs = ld32u(C.U + p); fail = !(bs >= 32u && bs <= (1u << 28)); endp = BAM_TAIL; tailp = p; fin = true; }
      else {
        i64 nx;
        if (!bam_core_ok(C, p, &nx)) fail = true;
        else if (nx > C.u_end) { endp = BAM_TAIL; tailp = p; fin = true; }
        else { ++cnt; ncig += (int)((u32)C.U[p + 16] | ((u32)C.U[p + 17] << 8)); nq += (i64)(int)ld32u(C.U + p + 20); p = nx; }
      }
      if (fail) { phase = SCAN; ++cand; }
      else if (fin) { H.first[k] = cand; H.endp[k] = endp; H.tailp[k] = tailp; H.cnt[k] = cnt; H.ncig[k] = ncig; H.nq[k] = nq; phase = DONE; }
    }
  }
}

// info (i64): [0] n records, [1] n cigar ops, [2] n quality bytes, [3] tail start, [4] repaired blocks.  cnt32: [0] n runs, [1] error bits, [2] inflate code
__global__ void __launch_bounds__(1024) k_bam_verify(BamChunk C, BamChain H, i64* __restrict__ in_pos, int* __restrict__ rbase, int* __restrict__ cbase,
                                                     i64* __restrict__ qbase, i64* __restrict__ info, int* __restrict__ err) {
  RSI_CTA_SETUP(c);
  const int n = C.nblk;
  const int per = (n + c.nthr - 1) / c.nthr;
  const int k0 = imin(c.tid * per, n), k1 = imin(k0 + per, n);
  const int lane = c.tid & 31, warp = c.tid >> 5;
  int fixed = 0;
  for (;;) {
    // in_pos[k] = position the list has reached when block k begins (exclusive max-scan of the walk ends)
    i64 loc = -1;
    for (int k = k0; k < k1; ++k) if (H.first[k] != BAM_NONE) loc = lmax(loc, H.endp[k]);
    i64 v = loc;
    for (int o = 1; o < 32; o <<= 1) { const i64 u = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v = lmax(v, u); }
    i64* slots = reinterpret_cast<i64*>(c.red);
    c.sync(); if (lane == 31) slots[warp] = v; c.sync();
    i64 pre = C.u_begin; for (int w = 0; w < warp; ++w) pre = lmax(pre, slots[w]);
    const i64 up = __shfl_up_sync(0xffffffffu, v, 1);
    i64 run = lmax(pre, lane ? up : -1);
    int bad = 0x7fffffff;
    for (int k = k0; k < k1; ++k) {
      in_pos[k] = run;
      const i64 ue = C.bound[k + 1], g = H.first[k];
      const bool ok = (run >= ue) ? (g == BAM_NONE) : (g == run);
      if (!ok && bad == 0x7fffffff) bad = k;
      if (g != BAM_NONE) run = lmax(run, H.endp[k]);
    }
    c.sync();
    const int firstbad = c.reduce(bad, MinOp());
    if (firstbad == 0x7fffffff) break;
    // Everything before the first mismatch is proven, so ITS incoming position is the true one and it is repaired whatever
    // it says.  A mismatch further on is usually an isolated wrong guess whose incoming position is already right, but it
    // can also be the shadow of an earlier wrong walk (the max-scan carries a wrong, far end over every later block): so
    // later blocks are only re-walked when the incoming position lies inside them, never emptied.  Each round settles at
    // least the first mismatch; the loop ends when every block matches, which is the proof.
    for (int k = k0; k < k1; ++k) {
      const i64 ue = C.bound[k + 1], g = H.first[k], cur = in_pos[k];
      const bool ok = (cur >= ue) ? (g == BAM_NONE) : (g == cur);
      if (ok) continue;
      if (cur >= ue) { if (k != firstbad) continue; bam_no_start(k, H); }
      else { H.first[k] = cur; bam_walk(C, cur, ue, k, H); }
      ++fixed;
    }
    c.sync();
  }
  fixed = c.reduce(fixed, SumOp());
  // all starts proven: a record that fails the core check inside a proven walk is a corrupt file
  i64 tail = -1, maxend = C.u_begin; int e = 0;
  for (int k = k0; k < k1; ++k) if (H.first[k] != BAM_NONE) {
    if (H.endp[k] == BAM_TAIL) {
      tail = H.tailp[k];
      i64 nx;
      if (tail + 36 <= C.u_end) { if (!bam_core_ok(C, tail, &nx) || nx <= C.u_end) e = 1; }      // complete but invalid: the walk stopped on it
      else if (tail + 4 <= C.u_end) { const u32 bs = ld32u(C.U + tail); if (bs < 32u || bs > (1u << 28)) e = 1; }
    } else maxend = lmax(maxend, H.endp[k]);
  }
  tail = c.reduce(tail, MaxOp()); maxend = c.reduce(maxend, MaxOp()); e = c.reduce(e, MaxOp());
  // exclusive sums -> where each block's records go
  int lc = 0, lg = 0; i64 lq = 0;
  for (int k = k0; k < k1; ++k) { lc += H.cnt[k]; lg += H.ncig[k]; lq += H.nq[k]; }
  int tc, tg; i64 tq;
  int bc = c.scan_excl(lc, &tc), bg = c.scan_excl(lg, &tg); i64 bq = c.scan_excl(lq, &tq);
  for (int k = k0; k < k1; ++k) { rbase[k] = bc; cbase[k] = bg; qbase[k] = bq; bc += H.cnt[k]; bg += H.ncig[k]; bq += H.nq[k]; }
  if (c.tid == 0) {
    info[0] = tc; info[1] = tg; info[2] = tq;
    info[3] = tail >= 0 ? tail : maxend; info[4] = fixed;
    if (e) atomicOr(err + 1, (int)BAM_ERR_RECORD);
    if (tail < 0 && maxend != C.u_end && n != 0) atomicOr(err + 1, (int)BAM_ERR_RECORD);
  }
}

struct BamSoA {
  i64* rec; int* tid; int* pos; int* mpos; int* isize; int* mtid; u16* flag; u8* mapq;
  u32* cigar_off; u32* cigar; u64* qual_off; u8* qual;
};

// fixed-size fields and offsets of every record (one thread walks the records of one BGZF block)
__global__ void k_bam_fields(BamChunk C, BamChain H, const int* __restrict__ rbase, const int* __restrict__ cbase, const i64* __restrict__ qbase,
                             const i64* __restrict__ info, BamSoA S) {
  const int k = (int)(blockIdx.x * blockDim.x + threadIdx.x);
  i64 p = k < C.nblk ? H.first[k] : BAM_NONE;
  const int n = p == BAM_NONE ? 0 : H.cnt[k];
  int r = n ? rbase[k] : 0; u32 co = n ? (u32)cbase[k] : 0u; u64 qo = n ? (u64)qbase[k] : 0ull;
  for (int i = 0; __any_sync(0xffffffffu, i < n); ++i) {      // warp-uniform trip count: the lanes walk 32 different blocks in step
    if (i < n) {
      // the 36 bytes of block_size + core as ten ALIGNED words and funnel shifts (records start at any byte; the lanes of a warp
      // read 32 different blocks, so every load instruction is 32 transactions: 10 instead of 36 byte loads)
      const u32* wq = reinterpret_cast<const u32*>(C.U + (p & ~3ll));
      const u32 sh = (u32)(p & 3ll) * 8u;
      u32 w[10];
#pragma unroll
      for (int k = 0; k < 10; ++k) w[k] = wq[k];
      u32 f[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) f[k] = __funnelshift_r(w[k], w[k + 1], sh);     // f[k] = the little-endian word at p + 4k
      const u32 bs = f[0], bmq = f[3], fnc = f[4];
      S.rec[r] = p; S.tid[r] = (int)f[1]; S.pos[r] = (int)f[2];
      S.mapq[r] = (u8)((bmq >> 8) & 0xffu); S.flag[r] = (u16)(fnc >> 16);
      S.mtid[r] = (int)f[6]; S.mpos[r] = (int)f[7]; S.isize[r] = (int)f[8];
      S.cigar_off[r] = co; S.qual_off[r] = qo;
      co += fnc & 0xffffu; qo += (u64)f[5];
      p += 4 + (i64)bs; ++r;
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) { S.cigar_off[info[0]] = (u32)info[1]; S.qual_off[info[0]] = (u64)info[2]; }
}

// CIGAR words and quality bytes: eight lanes per record, four records per warp at a time -- the per-record chain of
// dependent loads (record offset -> core fields -> payload) is latency, so four of them are kept in flight per warp
__global__ void k_bam_payload(const u8* __restrict__ U, const i64* __restrict__ info, BamSoA S) {
  const int n = (int)info[0];
  const int sub = (int)(threadIdx.x & 7);
  const int gid = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 3), ng = (int)((gridDim.x * blockDim.x) >> 3);
  for (int r = gid; r < n; r += ng) {
    const u8* q = U + S.rec[r];
    const u32 l_name = q[12], n_cig = (u32)q[16] | ((u32)q[17] << 8), l_seq = ld32u(q + 20);
    const u8* cg = q + 36 + l_name;
    u32* cd = S.cigar + S.cigar_off[r];
    for (u32 j = (u32)sub; j < n_cig; j += 8) cd[j] = ld32u(cg + 4 * j);
    const u8* qs = cg + 4 * n_cig + (l_seq + 1) / 2;
    u8* qd = S.qual + S.qual_off[r];
    u32 j = (u32)sub;
    for (; j + 24 < l_seq; j += 32) {          // four independent bytes per lane and trip
      const u8 a0 = qs[j], a1 = qs[j + 8], a2 = qs[j + 16], a3 = qs[j + 24];
      qd[j] = a0; qd[j + 8] = a1; qd[j + 16] = a2; qd[j + 24] = a3;
    }
    for (; j < l_seq; j += 8) qd[j] = qs[j];
  }
}

// runs of equal refID in record order (a coordinate-sorted BAM holds each contig's records contiguously)
__global__ void k_bam_runs(const int* __restrict__ tid, const i64* __restrict__ info, int* __restrict__ run_start, int cap, int* __restrict__ err) {
  const int n = (int)info[0];
  for (int r = (int)(blockIdx.x * blockDim.x + threadIdx.x); r < n; r += (int)(gridDim.x * blockDim.x)) {
    if (r == 0 || tid[r] != tid[r - 1]) {
      const int i = atomicAdd(err, 1);
      if (i < cap) run_start[i] = r; else atomicOr(err + 1, (int)BAM_ERR_RUNS);
    }
  }
}
// per run start r: tid, cigar offset, quality offset (for the host's run table)
__global__ void k_bam_run_info(const int* __restrict__ run_start, int nruns, BamSoA S, i64* __restrict__ out) {
  for (int i = (int)(blockIdx.x * blockDim.x + threadIdx.x); i < nruns; i += (int)(gridDim.x * blockDim.x)) {
    const int r = run_start[i];
    out[3 * i] = S.tid[r]; out[3 * i + 1] = S.cigar_off[r]; out[3 * i + 2] = (i64)S.qual_off[r];
  }
}

}  // namespace rsigpu
