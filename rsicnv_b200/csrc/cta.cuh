// cta.cuh -- cooperative-thread-array primitives used by the candidate stage (candidates.cuh).
//
// The candidate logic of the path (isitcnvwrap / areblockscnv / mergesegments ..., SURVEY.md §8a
// a19-a25) is list-sequential on the outside and data-parallel on the inside, so it runs as ONE
// thread block per contig: thread 0 does the list bookkeeping, all threads do the gathers, scans,
// histograms and reductions.  Everything here is written against `Cta`, which on the GPU wraps
// threadIdx / __syncthreads / warp shuffles.  When this header is compiled WITHOUT nvcc (only
// tests/hostsim/sim.cpp does that) `Cta` degenerates to a 1-thread block so the same control flow can be
// unit-tested against the oracle on a machine without a GPU.  The product never takes that path:
// librsigpu.so is built by nvcc only and there is no host entry into this code.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__) || defined(RSI_SIM)
#include "rt.cuh"
#define RSI_CTA_PARALLEL 1
#define RSI_DEV __device__ __forceinline__
#define RSI_DEVN __device__ __noinline__
#else
#define RSI_DEV inline
#define RSI_DEVN inline
#endif

namespace rsigpu {

struct MinOp { template <class T> RSI_DEV T operator()(T a, T b) const { return b < a ? b : a; } };
struct MaxOp { template <class T> RSI_DEV T operator()(T a, T b) const { return b > a ? b : a; } };
struct SumOp { template <class T> RSI_DEV T operator()(T a, T b) const { return a + b; } };

// (value, index) pair for arg-max / arg-min with "first index wins" ties
struct ValIdx { double v; long long i; };
struct ArgMaxFirst { RSI_DEV ValIdx operator()(ValIdx a, ValIdx b) const { return (b.v > a.v || (b.v == a.v && b.i < a.i)) ? b : a; } };
struct ArgMinFirst { RSI_DEV ValIdx operator()(ValIdx a, ValIdx b) const { return (b.v < a.v || (b.v == a.v && b.i < a.i)) ? b : a; } };

#if defined(RSI_CTA_PARALLEL)

template <class T>
RSI_DEV T shfl_xor_any(T v, int lane_mask) {
  static_assert(sizeof(T) % 4 == 0, "4-byte multiple");
  unsigned w[sizeof(T) / 4];
  memcpy(w, &v, sizeof(T));
#pragma unroll
  for (int k = 0; k < (int)(sizeof(T) / 4); ++k) w[k] = __shfl_xor_sync(0xffffffffu, w[k], lane_mask);
  memcpy(&v, w, sizeof(T));
  return v;
}

// cluster-level plumbing (a thread-block cluster of up to 8 CTAs can act as one big cooperative group)
#if defined(RSI_SIM)
RSI_DEV void cluster_barrier() { cusim::cluster_sync(); }
RSI_DEV int cluster_rank() { return (int)cusim::cluster_ctarank(); }
RSI_DEV int cluster_size() { return (int)cusim::cluster_nctarank(); }
#else
RSI_DEV void cluster_barrier() { asm volatile("barrier.cluster.arrive.release.aligned;\n barrier.cluster.wait.acquire.aligned;\n" ::: "memory"); }
RSI_DEV int cluster_rank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return (int)r; }
RSI_DEV int cluster_size() { unsigned r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return (int)r; }
#endif

enum { CTA_GX_BYTES = 2 * 16 * 16 + 256 * 16 };
// read a small value another CTA of the cluster wrote to global memory (word-wise volatile loads)
template <class T>
RSI_DEV T ld_xcta(const unsigned char* p) {
  unsigned w[sizeof(T) / 4];
#pragma unroll
  for (int k = 0; k < (int)(sizeof(T) / 4); ++k) w[k] = reinterpret_cast<const volatile unsigned*>(p)[k];
  T v; memcpy(&v, w, sizeof(T));
  return v;
}   // cluster exchange area: two generations of 16 partials + 256 warp slots

struct Cta {
  int tid, nthr;       // ids used to distribute work: block-local, or cluster-wide when nctas > 1
  unsigned char* red;  // shared scratch of THIS block, >= 33 * 16 bytes
  double* bc;          // broadcast area, >= 16 doubles: shared memory (one block) or global memory (cluster)
  int ltid = -1, lnthr = 0;   // block-local ids (default: same as tid / nthr)
  int nctas = 1, rank = 0;
  unsigned char* gx = nullptr;   // CTA_GX_BYTES of GLOBAL memory shared by the cluster (nctas > 1)
  mutable int xgen = 0;

  RSI_DEV int lt() const { return ltid < 0 ? tid : ltid; }
  RSI_DEV int ln() const { return ltid < 0 ? nthr : lnthr; }
  RSI_DEV void sync() const { if (nctas > 1) cluster_barrier(); else __syncthreads(); }
  // per-warp slots indexed by the (cluster-wide) warp id, 16 bytes each
  RSI_DEV unsigned char* wslots() const { return nctas > 1 ? gx + 2 * 16 * 16 : red; }

  // reduction over the whole group, result returned to every thread
  template <class T, class Op>
  RSI_DEV T reduce(T v, Op op) const {
    static_assert(sizeof(T) <= 16, "reduce payload");
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = op(v, shfl_xor_any(v, o));
    T* slots = reinterpret_cast<T*>(red);
    const int t = lt(), warp = t >> 5, lane = t & 31, nw = (ln() + 31) >> 5;
    __syncthreads();
    if (lane == 0) slots[warp] = v;
    __syncthreads();
    T r = slots[0];
    for (int w = 1; w < nw; ++w) r = op(r, slots[w]);
    if (nctas == 1) return r;
    T* ex = reinterpret_cast<T*>(gx + (xgen & 1) * 256);   // 16-byte stride per rank
    ++xgen;
    if (t == 0) *reinterpret_cast<T*>(reinterpret_cast<unsigned char*>(ex) + rank * 16) = r;
    cluster_barrier();
    T g = ld_xcta<T>(reinterpret_cast<unsigned char*>(ex));
    for (int k = 1; k < nctas; ++k) { T pk = ld_xcta<T>(reinterpret_cast<unsigned char*>(ex) + k * 16); g = op(g, pk); }
    return g;
  }
  // exclusive prefix sum of one value per thread (thread order over the whole group); *total to every thread
  template <class T>
  RSI_DEV T scan_excl(T v, T* total) const {
    const int t = lt(), warp = t >> 5, lane = t & 31, nw = (ln() + 31) >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      T up = shfl_up_any(inc, o);
      if (lane >= o) inc += up;
    }
    T* slots = reinterpret_cast<T*>(red);
    __syncthreads();
    if (lane == 31) slots[warp] = inc;
    __syncthreads();
    T base = 0, tot = 0;
    for (int w = 0; w < nw; ++w) { T sv = slots[w]; if (w < warp) base += sv; tot += sv; }
    if (nctas == 1) { *total = tot; return base + inc - v; }
    unsigned char* ex = gx + (xgen & 1) * 256;
    ++xgen;
    if (t == 0) *reinterpret_cast<T*>(ex + rank * 16) = tot;
    cluster_barrier();
    T before = 0, all = 0;
    for (int k = 0; k < nctas; ++k) { T pk = ld_xcta<T>(ex + k * 16); if (k < rank) before += pk; all += pk; }
    *total = all;
    return before + base + inc - v;
  }
  // exclusive scan under any associative, commutative op with identity `id` (one block: nctas == 1); *total to every thread
  template <class T, class Op>
  RSI_DEV T scan_excl_op(T v, Op op, T id, T* total) const {
    const int t = lt(), warp = t >> 5, lane = t & 31, nw = (ln() + 31) >> 5;
    T inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      T up = shfl_up_any(inc, o);
      if (lane >= o) inc = op(inc, up);
    }
    T ex = shfl_up_any(inc, 1);
    if (lane == 0) ex = id;
    T* slots = reinterpret_cast<T*>(red);
    __syncthreads();
    if (lane == 31) slots[warp] = inc;
    __syncthreads();
    T base = id, tot = id;
    for (int w = 0; w < nw; ++w) { T sv = slots[w]; if (w < warp) base = op(base, sv); tot = op(tot, sv); }
    *total = tot;
    return op(base, ex);
  }
  // out-of-line forms for the candidate kernels: their time is instruction FETCH (k_cand_a: 300 KB of SASS that one block runs
  // through once), and ~100 inlined copies of these two are a quarter of it.  The streaming kernels keep the inline forms: a
  // call inside their tile loops costs far more than it saves (k_pileup_tile 0.49 -> 1.48 ms when tried).
  template <class T, class Op>
  RSI_DEVN T reduce_ol(T v, Op op) const { return reduce(v, op); }
  template <class T>
  RSI_DEVN T scan_excl_ol(T v, T* total) const { return scan_excl(v, total); }
  template <class T>
  static RSI_DEV T shfl_up_any(T v, int d) {
    unsigned w[sizeof(T) / 4];
    memcpy(w, &v, sizeof(T));
#pragma unroll
    for (int k = 0; k < (int)(sizeof(T) / 4); ++k) w[k] = __shfl_up_sync(0xffffffffu, w[k], d);
    memcpy(&v, w, sizeof(T));
    return v;
  }
};

RSI_DEV void cta_atomic_inc(unsigned* p) { atomicAdd(p, 1u); }
// histogram increment called by ALL threads of a warp together (valid = this lane has a sample):
// lanes that hit the same bucket are merged into one atomic
RSI_DEV void cta_hist_add(unsigned* h, size_t b, bool valid) {
  const unsigned key = valid ? (unsigned)b : 0xffffffffu;     // bucket indices are far below 2^32
  const unsigned m = __match_any_sync(0xffffffffu, key);
  if (valid && (int)(threadIdx.x & 31) == __ffs((int)m) - 1) atomicAdd(&h[b], (unsigned)__popc(m));
}
RSI_DEV void cta_atomic_max(int* p, int v) { atomicMax(p, v); }
RSI_DEV void cta_atomic_min(int* p, int v) { atomicMin(p, v); }

#else  // ---- host simulation: a block of one thread (tests/hostsim only) ----

struct Cta {
  int tid = 0, nthr = 1;
  unsigned char* red = nullptr;
  double* bc = nullptr;
  int nctas = 1, rank = 0;
  void sync() const {}
  template <class T, class Op> T reduce(T v, Op) const { return v; }
  template <class T> T scan_excl(T v, T* total) const { *total = v; return T(0); }
  template <class T, class Op> T reduce_ol(T v, Op op) const { return reduce(v, op); }
  template <class T> T scan_excl_ol(T v, T* total) const { return scan_excl(v, total); }
};
inline void cta_atomic_inc(unsigned* p) { *p += 1u; }
inline void cta_hist_add(unsigned* h, size_t b, bool valid) { if (valid) h[b] += 1u; }
inline void cta_atomic_max(int* p, int v) { if (v > *p) *p = v; }
inline void cta_atomic_min(int* p, int v) { if (v < *p) *p = v; }

#endif

// thread 0 publishes a value (<= 8 bytes) to the whole block through the broadcast area
template <class T>
RSI_DEV T cta_bcast(const Cta& c, T v, int slot) {
#if defined(RSI_CTA_PARALLEL)
  static_assert(sizeof(T) <= 8, "bcast payload");
  c.sync();
  if (c.tid == 0) memcpy(&c.bc[slot], &v, sizeof(T));
  c.sync();
  T r;
  memcpy(&r, &c.bc[slot], sizeof(T));
  return r;
#else
  (void)c; (void)slot;
  return v;
#endif
}

}  // namespace rsigpu
