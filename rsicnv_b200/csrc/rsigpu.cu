// rsigpu.cu -- context, stream orchestration and the C ABI (include/rsigpu.h) of the B200-native
// `rsicnv rsi` hot path.  One context = one contig = what one iteration of the reference's chromosome
// loop owns (rsi.cpp:2189-2217).  Every stage is a short sequence of kernel launches on the context's
// stream; scalars travel between kernels in a device-resident DevState, so the host synchronises only
// (1) once after the per-base stage, to build the negative-binomial table with the box's libm
// (bit-exact by construction, SURVEY.md hard part 3), and (2) when results are copied back.
// There is NO CPU implementation behind this API: without a CUDA device every call fails.
#include <math.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <time.h>
#include <stdarg.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/rsigpu.h"
#include "k_bam.cuh"
#include "k_crc32.cuh"
#include "k_bam_index.cuh"
#include "k_sort.cuh"

using namespace rsigpu;

namespace {

#define CK(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess) { c->fail(std::string(#call) + ": " + cudaGetErrorString(e_)); return RSIGPU_E_CUDA; } \
    if (!c->launch_err.empty()) { c->fail("kernel launch failed: " + c->launch_err); c->launch_err.clear(); return RSIGPU_E_CUDA; } \
  } while (0)

template <class T>
struct DevBuf {
  T* p = nullptr; size_t cap = 0;
  cudaError_t ensure(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc((void**)&p, n * sizeof(T));
    if (e == cudaSuccess) cap = n;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};
template <class T>
struct DevVec {   // growable device array filled by appends from the host
  T* p = nullptr; size_t n = 0, cap = 0;
  // h: host memory, memory of the current device, or (src_dev >= 0) memory of another device
  cudaError_t append(const T* h, size_t cnt, cudaStream_t s, int src_dev = -1, int dst_dev = -1) {
    if (n + cnt > cap) {
      size_t ncap = std::max(n + cnt, cap * 2);
      T* q = nullptr;
      cudaError_t e = cudaMalloc((void**)&q, ncap * sizeof(T) + 64);
      if (e != cudaSuccess) return e;
      if (n) { e = cudaMemcpyAsync(q, p, n * sizeof(T), cudaMemcpyDeviceToDevice, s); if (e != cudaSuccess) return e; }
      cudaStreamSynchronize(s);
      if (p) cudaFree(p);
      p = q; cap = ncap;
    }
    cudaError_t e = (src_dev >= 0 && src_dev != dst_dev) ? cudaMemcpyPeerAsync(p + n, dst_dev, h, src_dev, cnt * sizeof(T), s)
                                                         : cudaMemcpyAsync(p + n, h, cnt * sizeof(T), cudaMemcpyDefault, s);   // host or device source
    n += cnt;
    return e;
  }
  void clear() { n = 0; }
  void release() { if (p) cudaFree(p); p = nullptr; n = cap = 0; }
  // a fresh array of exactly cnt elements (contents undefined), replacing this one
  cudaError_t alloc_exact(size_t cnt) {
    release();
    cudaError_t e = cudaMalloc((void**)&p, cnt * sizeof(T) + 64);
    if (e == cudaSuccess) { n = cnt; cap = cnt; }
    return e;
  }
};

const int LIST_CAP = 65536;          // runs / segments / calls per contig
const int CHIST_RCAP = 8192;         // value range of the class histograms
const size_t LUT_CAP = 1u << 24;

__global__ void k_add_u32(u32* a, size_t n, u32 v) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) a[i] += v;
}
__global__ void k_add_u64(u64* a, size_t n, u64 v) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) a[i] += v;
}

// ---- a contig split over several GPUs: partial tables of the parts are added on the lead
__global__ void k_vec_add_u32(u32* __restrict__ dst, const u32* __restrict__ src, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] += src[i];
}
// phase 0: after pass A (sums of positive depths, stratum tables, depth range); 1: after pass B; 2: after pass C (largest bin sum)
__global__ void k_split_reduce_state(DevState* lead, const DevState* parts, int nparts, int phase) {
  for (int g = 0; g < nparts; ++g) {
    const DevState* p = parts + g;
    if (phase == 0) {
      for (int k = (int)threadIdx.x; k < GC_STRATA; k += (int)blockDim.x) { lead->gc_sum[k] += p->gc_sum[k]; lead->gc_cnt[k] += p->gc_cnt[k]; }
      if (threadIdx.x == 0) {
        lead->pos_sum += p->pos_sum; lead->pos_cnt += p->pos_cnt;
        if (p->rd_min < lead->rd_min) lead->rd_min = p->rd_min;
        if (p->rd_max > lead->rd_max) lead->rd_max = p->rd_max;
      }
    }
    if (phase == 2 && threadIdx.x == 0 && p->max_binsum > lead->max_binsum) lead->max_binsum = p->max_binsum;
    if (threadIdx.x == 0) lead->err |= p->err;
  }
}
// number of reads that start before `key` (the reads a part shares with its left neighbour)
__global__ void k_count_before(const int* __restrict__ pos, long long n, int key, long long* out) {
  long long lo = 0, hi = n;
  while (lo < hi) { const long long mid = (lo + hi) >> 1; if (pos[mid] < key) lo = mid + 1; else hi = mid; }
  *out = lo;
}

}  // namespace

struct rsigpu_ctx {
  int device = 0, n_sm = 1;
  rsigpu_params P;
  cudaStream_t stream = nullptr, stream2 = nullptr;   // stream2: work that only depends on the staged reads (insert-size sample)
  cudaEvent_t ev_reads = nullptr, ev_isize = nullptr;
  bool isize_pending = false;
  std::string err;
  int L = 0, Lc = 0, nb = 0, tid = 0, gc_base = 0;
  bool have_ref = false, have_depth = false, have_reads = false, loaded = false, detected = false, filtered = false;
  bool pileup_fresh = false;   // rsigpu_pileup_end has just produced the depth of the staged reads: the next rsigpu_run does not redo it
  int cand_a_threads = 256;
  int level0_mode = 2;   // 2 = multi-block exact chain (default), 1 = one-block scan form, 0 = plain sequential FADD chain (cross-check)
  DevBuf<double> d_csum, d_clbc; DevBuf<i64> d_cchunk, d_clx; DevBuf<u32> d_clhist;
  // per-base
  DevBuf<u8> d_fasta; DevBuf<int> d_raw, d_rdc, d_nseq;  // d_nseq: nbeg | nend | ncum
  std::vector<int> h_nbeg, h_nend;
  DevState* d_st = nullptr; DevState* h_st = nullptr;
  DevBuf<u32> d_hist_all, d_chist, d_thist, d_tothist, d_fq_hist;
  // bins
  DevBuf<float> d_bin_med, d_bin_nbn, d_lut, d_nz_val; DevBuf<int> d_bin_medint, d_status, d_status1, d_tile, d_nz_idx, d_runs; DevBuf<i64> d_bin_sum, d_pfx, d_cprof, d_thr;
  DevBuf<u32> d_minl_del, d_minl_dup;
  float* h_lut = nullptr; size_t h_lut_cap = 0;
  // lists
  DevBuf<Cnv> d_lists;   // segs | tmp | ov(2) | segments | blocks | premerge | merged | detected | calls
  DevBuf<int> d_misc;    // n_dump[4] | cand_err | max_extent | sorted_bad | n_begN | n_endN
  DevBuf<int> d_ref, d_sub, d_spec_ref; DevBuf<i64> d_pref, d_spec_pref, d_spec_off; DevBuf<float> d_rm, d_spec_rm; DevBuf<u32> d_chist_c;
  DevBuf<int> d_nrun_beg, d_nrun_end, d_scan_scratch;
  std::vector<Cnv> h_detected, h_calls, h_dump[4];
  // reads
  DevVec<int> r_pos, r_mpos, r_isize, r_mtid; DevVec<u16> r_flag; DevVec<u8> r_mapq, r_qual; DevVec<u32> r_cigar_off, r_cigar; DevVec<u64> r_qual_off;
  DevBuf<int> r_calend, d_tile_range; DevBuf<u32> d_qmask; DevBuf<u16> r_ncig;
  // a contig split over several GPUs (rsigpu_split_run): on the lead, the read summaries of every part in position order
  // (what the insert-size sample and cnv_stat read), and staging space for the parts' partial tables
  DevBuf<int> s_pos, s_mpos, s_isize, s_mtid, s_calend; DevBuf<u16> s_flag; DevBuf<u8> s_mapq; DevBuf<u32> s_cigar_off;
  size_t s_n = 0; bool use_summary = false;
  DevBuf<DevState> d_part_st; DevBuf<u32> d_part_u32;
  cudaEvent_t ev_part = nullptr, ev_lead = nullptr;
  long long split_p2p_bytes = 0;
  // BAM decoder (k_bam.cuh): one chunk of BGZF blocks at a time
  DevBuf<u8> b_comp, b_U, b_carry, b_mapq, b_qual; DevBuf<BgzfBlock> b_blk; DevBuf<u16> b_flag, b_tabs; DevBuf<u32> b_cigoff, b_cig; DevBuf<u64> b_qoff;
  DevBuf<int> b_cnt, b_ncig, b_rbase, b_cbase, b_cnt32, b_runstart, b_tid, b_pos, b_mpos, b_isize, b_mtid;
  DevBuf<i64> b_bound, b_first, b_endp, b_tailp, b_in, b_info, b_rec, b_nq, b_qbase, b_runinfo;
  struct BamRun { int tid, part; i64 r0, r1, c0, c1, q0, q1; bool by_ref; };
  std::vector<BamRun> b_runs;
  int b_nref = 0, b_tail_len = 0, b_rewalked = 0; bool b_active = false, b_first_feed = true;
  size_t b_umax = (size_t)5 << 30;   // decoded bytes one feed may produce (test hook: rsigpu_set_feed_limit)
  int inflate_mode = 0;              // 0 = by chunk size, 1 = one lane per BGZF block, 2 = one warp per BGZF block (rsigpu_set_inflate_mode)
  bool bgzf_crc = false;             // check every block's CRC32 after inflate (rsigpu_set_bgzf_crc)
  bool bam_by_ref = false;           // group each feed's records by refID before the runs are found (rsigpu_set_bam_by_ref)
  DevBuf<i64> b2_rec; DevBuf<int> b2_tid, b2_pos, b2_mpos, b2_isize, b2_mtid; DevBuf<u16> b2_flag; DevBuf<u8> b2_mapq; DevBuf<u32> b2_cigoff; DevBuf<u64> b2_qoff;
  // radix sort scratch (k_sort.cuh): keys and indices ping-pong, per-tile digit counts, digit totals, offset-scan tile sums
  DevBuf<u32> t_key, t_key2, t_idx, t_idx2, t_hist, t_dtot; DevBuf<u64> t_ts;
  // BAI index built from the decoded records (k_bam_index.cuh, rsigpu_bam_index_begin / _get)
  struct IxChunk { u32 bin; u64 u, v; };
  struct IxRef { std::vector<IxChunk> ch; u64 n_map = 0, n_unmap = 0; std::vector<u64> lin; };
  bool ix_on = false, ix_failed = false, ix_ready = false, ix_has_prev = false;
  int64_t ix_off = 0;                // file offset of the next feed's first byte
  u64 ix_carry_voff = 0, ix_end_voff = 0, ix_prev_key = 0, ix_no_coor = 0;
  int ix_prev_tid = 0, ix_prev_pos = 0; u32 ix_prev_bin = 0;
  IxChunk ix_pend{}; int ix_pend_tid = -1; bool ix_pend_on = false;   // the last run seen: its end is the next run's begin
  std::vector<IxRef> ix_ref; std::vector<uint8_t> ix_out;
  DevBuf<u64> x_beg, x_key, x_cnt, x_tkey; DevBuf<u32> x_meta; DevBuf<int> x_tstart, x_tunmap; DevBuf<BixChunk> x_chunk; DevBuf<BixLin> x_lin;
  // accounting
  long long h_cprof[16] = {};
  int64_t launches = 0;
  float stage_ms[6] = {0, 0, 0, 0, 0, 0};
  cudaEvent_t ev[8] = {};
  bool profile = false;
  std::map<std::string, std::pair<float, int>> prof;
  std::vector<std::string> prof_order;

  std::string launch_err;
  void fail(const std::string& m) { err = m; }
  Cnv* list(int k) const { return d_lists.p + (size_t)k * LIST_CAP; }
};

namespace {

struct KTimer {
  rsigpu_ctx* c; const char* name; cudaEvent_t a, b;
  KTimer(rsigpu_ctx* c_, const char* n) : c(c_), name(n), a(nullptr), b(nullptr) {
    c->launches++;
    if (c->profile) { cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, c->stream); }
  }
  ~KTimer() {
    if (!c->profile) return;
    cudaEventRecord(b, c->stream); cudaEventSynchronize(b);
    float ms = 0; cudaEventElapsedTime(&ms, a, b);
    auto it = c->prof.find(name);
    if (it == c->prof.end()) { c->prof[name] = std::make_pair(ms, 1); c->prof_order.push_back(name); }
    else { it->second.first += ms; it->second.second += 1; }
    cudaEventDestroy(a); cudaEventDestroy(b);
  }
};
#define KL(name, grid, block, smem, ...)                                                          \
  do {                                                                                            \
    KTimer kt_(c, #name);                                                                         \
    RSI_LAUNCH(name, grid, block, smem, c->stream, __VA_ARGS__);                                  \
    cudaError_t le_ = cudaGetLastError();                                                         \
    if (le_ != cudaSuccess && c->launch_err.empty()) c->launch_err = std::string(#name) + ": " + cudaGetErrorString(le_); \
  } while (0)

#define KLC(name, grid, block, cluster, smem, ...)                                                \
  do {                                                                                            \
    KTimer kt_(c, #name);                                                                         \
    RSI_LAUNCH_CLUSTER(name, grid, block, cluster, smem, c->stream, __VA_ARGS__);                 \
    cudaError_t le_ = cudaGetLastError();                                                         \
    if (le_ != cudaSuccess && c->launch_err.empty()) c->launch_err = std::string(#name) + ": " + cudaGetErrorString(le_); \
  } while (0)

template <class T> T* field_ptr(DevState* base, T DevState::*m) { return &(base->*m); }

int map_dev_err(rsigpu_ctx* c, int e, int cand) {
  if (!e) return RSIGPU_OK;
  std::string m = "device-side range check failed:";
  if (e & ERR_DEPTH_RANGE) m += " depth outside [0, 2^24);";
  if (e & ERR_HIST_RANGE) m += " adjusted depth beyond the histogram range (65536 / class range 8192);";
  if (e & ERR_LMAX) m += " RSI Lmax above 2048;";
  if (e & ERR_FIXEDPOINT) m += " bin values make the reference's window sums inexact;";
  if (e & ERR_FQ_BINS) m += " float quantile needs more than 2^22 buckets;";
  if (e & ERR_LISTCAP) m += " more than 65536 runs;";
  if (e & ERR_CAND) m += " candidate-stage scratch overflow (code " + std::to_string(cand) + ");";
  if (e & ERR_DEGENERATE) m += " degenerate depth distribution (median or MAD is zero);";
  if (e & ERR_PILEUP) m += " malformed read batch;";
  c->fail(m);
  return RSIGPU_E_RANGE;
}

static double trace_now() { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec * 1e3 + 1e-6 * (double)t.tv_nsec; }
static bool trace_on() { static int on = -1; if (on < 0) on = getenv("RSIGPU_TRACE") ? 1 : 0; return on == 1; }
#define TRACE(c, what) do { if (trace_on()) fprintf(stderr, "[trace %p] %-28s %.3f ms\n", (void*)(c), what, trace_now()); } while (0)

int grid_for(int n_items, int per_block, int cap) { int g = (n_items + per_block - 1) / per_block; if (g < 1) g = 1; return g > cap ? cap : g; }

double nb_formula(double sum, double m2, double r) {  // rsi.cpp:1155-1156
  return 2.0 * sqrt(r) * log(sqrt((sum + 0.25) / (m2 * r - 0.5)) + sqrt(1.0 + (sum + 0.25) / (m2 * r - 0.5)));
}

// one histogram quantile of a bin array (k_quant.cuh)
void quantile(rsigpu_ctx* c, const float* x, const int* status, int masked, int mode, const double* center, int slot) {
  const int g = grid_for(c->nb, 256 * 8, c->n_sm * 4);
  KL(k_fq_minmax, g, 256, 0, x, status, masked, mode, center, c->d_st, slot);
  KL(k_fq_hist, g, 256, 0, x, status, masked, mode, center, c->d_fq_hist.p, c->d_st, slot);
  KL(k_fq_pick, 1, 1024, 0, c->d_fq_hist.p, c->d_st, slot);
}

// cudaFuncSetAttribute is per device: once for every device a context is created on (the current device is the context's)
int set_smem_attrs(int device) {
  static bool done[64] = {};
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  if (device < 0 || device >= 64 || done[device]) return 0;
  done[device] = true;
  cudaFuncSetAttribute(k_gc_table, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RSI_SMEM_A);
  cudaFuncSetAttribute(k_gc_adjust, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RSI_SMEM_B);
  cudaFuncSetAttribute(k_bins, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RSI_SMEM_C);
  cudaFuncSetAttribute(k_bins_warp<101>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(cw_nw(101) * cw_warp_bytes(101)));
  cudaFuncSetAttribute(k_bins_warp<51>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(cw_nw(51) * cw_warp_bytes(51)));
  cudaFuncSetAttribute(k_bins_warp<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(cw_nw(0) * cw_warp_bytes(0)));
  cudaFuncSetAttribute(k_cand_a, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RSI_SMEM_CAND_A);
  cudaFuncSetAttribute(k_cand_b, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(CAND_SHIST * 4));
  cudaFuncSetAttribute(k_cand_c, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(CAND_SHIST * 4));
  cudaFuncSetAttribute(k_cand_final, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RSI_SMEM_CAND_CL);
  cudaFuncSetAttribute(k_cand_edge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RSI_SMEM_CAND_CL);
  cudaFuncSetAttribute(k_rsi_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RSI_SCAN_SMEM);
  cudaFuncSetAttribute(k_rsi_scan_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RSI_SCAN_SMEM_T(LMAX_SMALL));
  // occupancy of these two is set by shared memory: ask for the largest shared-memory carve-out
  cudaFuncSetAttribute(k_rsi_scan_small, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  cudaFuncSetAttribute(k_bgzf_inflate, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
  cudaFuncSetAttribute(k_bgzf_crc32, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CRC_SMEM);
  return 0;
}

// ---- the RSI stage for one transformation (rsicnvnbn: which = 0, rsicnvmed: which = 1)
int run_rsi(rsigpu_ctx* c, int which, const float* t) {
  DevState* st = c->d_st;
  const int nb = c->nb, slot0 = which == 0 ? 0 : 4;
  const int gb = grid_for(nb, 1024, c->n_sm * 8);
  const size_t scan_smem = RSI_SCAN_SMEM;
  if (which == 0) quantile(c, t, nullptr, 0, QM_ID, nullptr, slot0);
  KL(k_rsi_params1, 1, 32, 0, t, st, which, c->P.threshold);
  quantile(c, t, nullptr, 0, QM_ABSDEV, field_ptr(st, &DevState::tmedian), slot0 + 1);
  KL(k_rsi_params2, 1, 32, 0, t, st, which, c->P.threshold, slot0 + 1);
  for (int pass = 0; pass < 2; ++pass) {
    KL(k_rsi_thresholds, (LMAX_CAP + 63) / 64, 64, 0, c->d_thr.p, st);
    KL(k_rsi_scan_small, (nb + S_T - 1) / S_T, S_NT, RSI_SCAN_SMEM_T(LMAX_SMALL), t, c->d_bin_medint.p, c->d_minl_del.p, c->d_minl_dup.p, c->d_scan_scratch.p, c->d_thr.p, st);
    KL(k_rsi_scan, (nb + S_T - 1) / S_T, S_NT, scan_smem, t, c->d_bin_medint.p, c->d_minl_del.p, c->d_minl_dup.p, c->d_scan_scratch.p, c->d_thr.p, st);
    KL(k_rsi_cnt_del, gb, 256, 0, c->d_minl_del.p, st);
    KL(k_rsi_cnt_dup, gb, 256, 0, c->d_minl_del.p, c->d_minl_dup.p, st);
    int* status = pass == 0 ? c->d_status1.p : c->d_status.p;
    KL(k_rsi_status, gb, 256, 0, c->d_minl_del.p, c->d_minl_dup.p, status, c->d_tile.p, st);
    KL(k_rsi_log_pass, 1, 256, 0, st, which, pass);
    if (pass == 1) break;
    // filterstatus (rsi.cpp:948-1057) on the first-pass status, in place via a second buffer
    KL(k_nz_scatter, gb, 256, 0, t, status, c->d_tile.p, c->d_nz_idx.p, c->d_nz_val.p, st);
    if (c->level0_mode == 2) {
      KL(k_chain_sums, CHN_N / 8, 256, 0, t, status, c->d_csum.p, st);
      KL(k_chain_compose, CHN_N / 8, 256, 0, t, status, c->d_csum.p, reinterpret_cast<ChainChunk*>(c->d_cchunk.p), st);
      KL(k_chain_resolve, 1, 32, 0, t, status, reinterpret_cast<const ChainChunk*>(c->d_cchunk.p), st);
    } else if (c->level0_mode == 1) KL(k_level0_chain_scan, 1, CH_NT, 0, t, status, st);
    else KL(k_level0_chain_seq, 1, 32, 0, t, status, st);
    KL(k_level_sums, (2 * LMAX_CAP + 3 + 127) / 128, 128, 0, c->d_nz_idx.p, c->d_nz_val.p, st);
    KL(k_filter_params, 1, 32, 0, st, which);
    CK(cudaMemcpyAsync(c->d_status.p, status, (size_t)nb * 4, cudaMemcpyDeviceToDevice, c->stream));
    KL(k_filter_trim, gb, 256, 0, t, c->d_status.p, status, st);
    quantile(c, t, status, 1, QM_ID, nullptr, slot0 + 2);
    quantile(c, t, status, 1, QM_ABSDEV, &(st->qj[slot0 + 2].q[1]), slot0 + 3);
    KL(k_rsi_params3, 1, 32, 0, st, slot0 + 2, slot0 + 3, which);
  }
  // get_rsi_segments on the second-pass status
  KL(k_runs_count, gb, 256, 0, c->d_status.p, c->d_tile.p, st);
  KL(k_runs_scatter, gb, 256, 0, c->d_status.p, c->d_tile.p, c->d_runs.p, LIST_CAP, st);
  KL(k_run_argmax, c->n_sm * 2, 1024, 0, t, c->d_status.p, c->d_runs.p, c->d_pfx.p, c->list(0), st);
  return RSIGPU_OK;
}

ReadSoA read_view(rsigpu_ctx* c) {
  ReadSoA R;
  if (c->use_summary) {   // the lead of a split contig: summaries of all parts (no CIGAR ops, no qualities: the pileup is done)
    R.n = (i64)c->s_n; R.tid = c->tid;
    R.pos = c->s_pos.p; R.mpos = c->s_mpos.p; R.isize = c->s_isize.p; R.mtid = c->s_mtid.p; R.flag = c->s_flag.p; R.mapq = c->s_mapq.p;
    R.cigar_off = nullptr; R.cigar = nullptr; R.qual_off = nullptr; R.qual = nullptr; R.calend = c->s_calend.p;
    R.ncig = reinterpret_cast<u16*>(c->s_cigar_off.p);
    return R;
  }
  R.n = (i64)c->r_pos.n; R.tid = c->tid;
  R.pos = c->r_pos.p; R.mpos = c->r_mpos.p; R.isize = c->r_isize.p; R.mtid = c->r_mtid.p; R.flag = c->r_flag.p; R.mapq = c->r_mapq.p;
  R.cigar_off = c->r_cigar_off.p; R.cigar = c->r_cigar.p; R.qual_off = c->r_qual_off.p; R.qual = c->r_qual.p; R.calend = c->r_calend.p;
  R.ncig = c->r_ncig.p;
  return R;
}

}  // namespace

extern "C" {

int rsigpu_default_params(rsigpu_params* p) {
  if (!p) return RSIGPU_E_ARG;
  memset(p, 0, sizeof *p);
  p->m = 101; p->minq = 0; p->min_baseQ = 13; p->gcadjust = 1; p->trans = RSIGPU_TRANS_NBN; p->merge = 1; p->maxchkbp = 100000;
  p->cap = 4.0; p->threshold = -1.0; p->epsilon = 1.5; p->chklen = 2.5;
  return RSIGPU_OK;
}

int rsigpu_num_devices(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

int rsigpu_create(int device, const rsigpu_params* p, rsigpu_ctx** out) {
  if (!p || !out) return RSIGPU_E_ARG;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return RSIGPU_E_NODEVICE;
  if (p->trans != RSIGPU_TRANS_NBN && p->trans != RSIGPU_TRANS_MED && p->trans != RSIGPU_TRANS_ALL) return RSIGPU_E_ARG;
  rsigpu_ctx* c = new rsigpu_ctx();
  c->device = device; c->P = *p;
  if (c->P.m % 2 != 1) c->P.m += 1;   // rsi.cpp:2061-2064
  if (c->P.m < 3 || c->P.m > C_TP) { delete c; return RSIGPU_E_ARG; }
  if (cudaSetDevice(device) != cudaSuccess) { delete c; return RSIGPU_E_CUDA; }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete c; return RSIGPU_E_CUDA; }
  c->n_sm = prop.multiProcessorCount;
  set_smem_attrs(device);
  bool ok = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) == cudaSuccess && cudaStreamCreateWithFlags(&c->stream2, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaEventCreate(&c->ev_reads) == cudaSuccess && cudaEventCreate(&c->ev_isize) == cudaSuccess;
  ok = ok && cudaEventCreate(&c->ev_part) == cudaSuccess && cudaEventCreate(&c->ev_lead) == cudaSuccess;
  ok = ok && cudaMalloc((void**)&c->d_st, sizeof(DevState)) == cudaSuccess;
  ok = ok && cudaMallocHost((void**)&c->h_st, sizeof(DevState)) == cudaSuccess;
  if (ok) memset(c->h_st, 0, sizeof(DevState));      // a context that only decodes never fills it; the debug / log getters read it
  for (int k = 0; k < 8 && ok; ++k) ok = cudaEventCreate(&c->ev[k]) == cudaSuccess;
  ok = ok && c->d_hist_all.ensure(HIST_ALL_BINS) == cudaSuccess && c->d_chist.ensure((size_t)MAD_CLASSES * CHIST_RCAP) == cudaSuccess;
  ok = ok && c->d_thist.ensure(CHIST_RCAP) == cudaSuccess && c->d_tothist.ensure(CHIST_RCAP) == cudaSuccess;
  ok = ok && c->d_fq_hist.ensure((size_t)FQ_BINS_CAP + 8) == cudaSuccess;
  ok = ok && c->d_lists.ensure((size_t)LIST_CAP * 11 + 8) == cudaSuccess && c->d_misc.ensure(64) == cudaSuccess;
  ok = ok && c->d_runs.ensure((size_t)LIST_CAP * 2 + 8) == cudaSuccess && c->d_cprof.ensure(16) == cudaSuccess && c->d_thr.ensure(2 * (LMAX_CAP + 2)) == cudaSuccess && c->d_csum.ensure(CHN_N + 8) == cudaSuccess
       && c->d_cchunk.ensure((size_t)(CHN_N + 8) * sizeof(ChainChunk) / 8 + 8) == cudaSuccess
       && c->d_clx.ensure((size_t)32 * CTA_GX_BYTES / 8 + 8) == cudaSuccess && c->d_clbc.ensure(32 * 32 + 8) == cudaSuccess
       && c->d_clhist.ensure((size_t)32 * CAND_CL_HIST + 8) == cudaSuccess;
  ok = ok && c->d_chist_c.ensure(1u << 22) == cudaSuccess && c->d_sub.ensure(((size_t)p->maxchkbp * 10 + 64) * 33) == cudaSuccess;
  ok = ok && c->d_nrun_beg.ensure(1 << 20) == cudaSuccess && c->d_nrun_end.ensure(1 << 20) == cudaSuccess;
  if (ok) ok = cudaMemsetAsync(c->d_fq_hist.p, 0, ((size_t)FQ_BINS_CAP + 8) * 4, c->stream) == cudaSuccess;
  if (!ok) { rsigpu_destroy(c); return RSIGPU_E_CUDA; }
  *out = c;
  return RSIGPU_OK;
}

void rsigpu_destroy(rsigpu_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream2) cudaStreamSynchronize(c->stream2);
  if (c->stream) cudaStreamSynchronize(c->stream);
  c->d_fasta.release(); c->d_raw.release(); c->d_rdc.release(); c->d_nseq.release();
  c->d_hist_all.release(); c->d_chist.release(); c->d_thist.release(); c->d_tothist.release(); c->d_fq_hist.release();
  c->d_bin_med.release(); c->d_bin_nbn.release(); c->d_lut.release(); c->d_bin_medint.release(); c->d_status.release(); c->d_status1.release();
  c->d_tile.release(); c->d_nz_idx.release(); c->d_nz_val.release(); c->d_runs.release(); c->d_bin_sum.release(); c->d_pfx.release(); c->d_cprof.release(); c->d_thr.release(); c->d_csum.release(); c->d_cchunk.release(); c->d_clx.release(); c->d_clbc.release(); c->d_clhist.release(); c->d_minl_del.release(); c->d_minl_dup.release();
  c->d_lists.release(); c->d_misc.release(); c->d_ref.release(); c->d_sub.release(); c->d_pref.release(); c->d_rm.release(); c->d_chist_c.release(); c->d_spec_ref.release(); c->d_spec_pref.release(); c->d_spec_off.release(); c->d_spec_rm.release();
  c->d_nrun_beg.release(); c->d_nrun_end.release(); c->d_scan_scratch.release(); c->d_tile_range.release(); c->d_qmask.release(); c->r_calend.release(); c->r_ncig.release();
  c->r_pos.release(); c->r_mpos.release(); c->r_isize.release(); c->r_mtid.release(); c->r_flag.release(); c->r_mapq.release(); c->r_qual.release();
  c->r_cigar_off.release(); c->r_cigar.release(); c->r_qual_off.release();
  c->b_carry.release(); c->b_tabs.release(); c->b_cnt32.release();
  c->b_comp.release(); c->b_U.release(); c->b_mapq.release(); c->b_qual.release(); c->b_blk.release(); c->b_flag.release(); c->b_cigoff.release(); c->b_cig.release(); c->b_qoff.release();
  c->b_bound.release(); c->b_first.release(); c->b_endp.release(); c->b_tailp.release(); c->b_cnt.release(); c->b_ncig.release(); c->b_in.release(); c->b_rbase.release(); c->b_cbase.release();
  c->b_info.release(); c->b_runstart.release(); c->b_rec.release(); c->b_tid.release(); c->b_pos.release(); c->b_mpos.release(); c->b_isize.release(); c->b_mtid.release();
  c->b_nq.release(); c->b_qbase.release(); c->b_runinfo.release();
  c->b2_rec.release(); c->b2_tid.release(); c->b2_pos.release(); c->b2_mpos.release(); c->b2_isize.release(); c->b2_mtid.release(); c->b2_flag.release(); c->b2_mapq.release(); c->b2_cigoff.release(); c->b2_qoff.release();
  c->t_key.release(); c->t_key2.release(); c->t_idx.release(); c->t_idx2.release(); c->t_hist.release(); c->t_dtot.release(); c->t_ts.release();
  c->x_beg.release(); c->x_key.release(); c->x_cnt.release(); c->x_tkey.release(); c->x_meta.release(); c->x_tstart.release(); c->x_tunmap.release(); c->x_chunk.release(); c->x_lin.release();
  if (c->d_st) cudaFree(c->d_st);
  if (c->h_st) cudaFreeHost(c->h_st);
  if (c->h_lut) cudaFreeHost(c->h_lut);
  for (int k = 0; k < 8; ++k) if (c->ev[k]) cudaEventDestroy(c->ev[k]);
  if (c->ev_reads) cudaEventDestroy(c->ev_reads);
  if (c->ev_isize) cudaEventDestroy(c->ev_isize);
  if (c->ev_part) cudaEventDestroy(c->ev_part);
  if (c->ev_lead) cudaEventDestroy(c->ev_lead);
  c->s_pos.release(); c->s_mpos.release(); c->s_isize.release(); c->s_mtid.release(); c->s_calend.release(); c->s_flag.release(); c->s_mapq.release(); c->s_cigar_off.release();
  c->d_part_st.release(); c->d_part_u32.release();
  if (c->stream2) cudaStreamDestroy(c->stream2);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

const char* rsigpu_last_error(const rsigpu_ctx* c) { return c ? c->err.c_str() : "null context"; }

// a3 + a4: N runs on the device, padding / merging of the few hundred intervals on the host
int rsigpu_set_reference(rsigpu_ctx* c, const uint8_t* fasta, int32_t len, int32_t tid) {
  if (!c || !fasta) return RSIGPU_E_ARG;
  if (len < 1000) { c->fail("contig shorter than 1000 bases"); return RSIGPU_E_RANGE; }
  cudaSetDevice(c->device);
  c->L = len; c->tid = tid;
  c->have_ref = true; c->have_depth = false; c->have_reads = false; c->loaded = false; c->detected = false; c->filtered = false;
  c->use_summary = false;
  const size_t padded = ((size_t)len + 15) / 16 * 16 + LD_T + 512;   // a whole tile beyond the last base is staged by the bulk copies
  CK(c->d_fasta.ensure(padded));
  CK(cudaMemsetAsync(c->d_fasta.p + len, 0, padded - (size_t)len, c->stream));
  CK(cudaMemcpyAsync(c->d_fasta.p, fasta, (size_t)len, cudaMemcpyHostToDevice, c->stream));
  int* n2 = c->d_misc.p + 8;     // n_begN | n_endN | (u64) number of G/C bases
  CK(cudaMemsetAsync(n2, 0, 16, c->stream));
  const int cap = 1 << 20;
  KL(k_n_runs, grid_for(len, 256 * 16, c->n_sm * 8), 256, 0, c->d_fasta.p, len, c->d_nrun_beg.p, c->d_nrun_end.p, n2, n2 + 1, cap, reinterpret_cast<u64*>(n2 + 2));
  int hn[4];
  CK(cudaMemcpyAsync(hn, n2, 16, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (hn[0] != hn[1] || hn[0] > cap) { c->fail("more than 2^20 N runs"); return RSIGPU_E_RANGE; }
  std::vector<int> b(hn[0]), e(hn[0]);
  if (hn[0]) {
    CK(cudaMemcpyAsync(b.data(), c->d_nrun_beg.p, (size_t)hn[0] * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaMemcpyAsync(e.data(), c->d_nrun_end.p, (size_t)hn[0] * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    std::sort(b.begin(), b.end()); std::sort(e.begin(), e.end());
  }
  // get_noseq_regions (loaddata.cpp:243-273): pad by max(50, m/4), clamp, re-merge overlapping or touching runs
  const int dx = std::max(50, c->P.m / 4);
  c->h_nbeg.clear(); c->h_nend.clear();
  for (int k = 0; k < hn[0]; ++k) {
    const int pb = std::max(b[k] - dx, 0), pe = std::min(e[k] + dx, len - 1);
    if (!c->h_nend.empty() && pb <= c->h_nend.back() + 1) c->h_nend.back() = std::max(c->h_nend.back(), pe);
    else { c->h_nbeg.push_back(pb); c->h_nend.push_back(pe); }
  }
  const int nn = (int)c->h_nbeg.size();
  std::vector<int> pack(3 * (size_t)nn + 4, 0);
  int removed = 0;
  for (int k = 0; k < nn; ++k) { pack[k] = c->h_nbeg[k]; pack[nn + k] = c->h_nend[k]; pack[2 * nn + k] = removed; removed += c->h_nend[k] - c->h_nbeg[k] + 1; }
  CK(c->d_nseq.ensure(3 * (size_t)nn + 4));
  CK(cudaMemcpyAsync(c->d_nseq.p, pack.data(), (3 * (size_t)nn + 4) * 4, cudaMemcpyHostToDevice, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  c->Lc = len - removed;
  {   // mean G/C count of a 201-base window of sequence: centre of the strata pass A keeps in its private tables
    u64 ngc; memcpy(&ngc, hn + 2, 8);
    long long nseq = 0; for (int k = 0; k < hn[0]; ++k) nseq += e[k] - b[k] + 1;
    nseq = (long long)len - nseq;
    const int centre = nseq > 0 ? (int)((double)GC_WIN * (double)ngc / (double)nseq + 0.5) : GC_WIN / 2;
    c->gc_base = std::max(0, std::min(centre - A_ROWS / 2, (int)GC_STRATA - A_ROWS));
  }
  c->nb = c->Lc / c->P.m;
  if (c->nb < 64) { c->fail("fewer than 64 bins after N removal"); return RSIGPU_E_RANGE; }
  return RSIGPU_OK;
}

int rsigpu_set_depth(rsigpu_ctx* c, const int32_t* depth, int32_t len) {
  if (!c || !depth) return RSIGPU_E_ARG;
  if (!c->have_ref || len != c->L) { c->fail("set_depth: call set_reference first with the same length"); return RSIGPU_E_ARG; }
  cudaSetDevice(c->device);
  const size_t padded = ((size_t)len + LD_TILE - 1) / LD_TILE * LD_TILE + 64;
  CK(c->d_raw.ensure(padded));
  CK(cudaMemcpyAsync(c->d_raw.p, depth, (size_t)len * 4, cudaMemcpyHostToDevice, c->stream));
  c->have_depth = true; c->have_reads = false; c->loaded = false; c->detected = false; c->filtered = false;
  return RSIGPU_OK;
}

int rsigpu_pileup_begin(rsigpu_ctx* c, int32_t target_len) {
  if (!c) return RSIGPU_E_ARG;
  if (!c->have_ref || target_len != c->L) { c->fail("pileup_begin: call set_reference first with the same length"); return RSIGPU_E_ARG; }
  c->r_pos.clear(); c->r_mpos.clear(); c->r_isize.clear(); c->r_mtid.clear(); c->r_flag.clear(); c->r_mapq.clear(); c->r_qual.clear();
  c->r_cigar_off.clear(); c->r_cigar.clear(); c->r_qual_off.clear();
  c->have_reads = false; c->have_depth = false; c->loaded = false; c->detected = false; c->filtered = false;
  return RSIGPU_OK;
}

// append one batch to the staged reads; the batch's pointers may be host or device memory, its offset arrays start
// at cig_first / q_first (0 for a caller's batch, the run's first offsets for records decoded on the GPU)
static int push_impl(rsigpu_ctx* c, const rsigpu_read_batch* b, size_t nc, size_t nq, u32 cig_first, u64 q_first, int src_dev = -1) {
  cudaSetDevice(c->device);
  const size_t n = (size_t)b->n_reads;
  const size_t r0 = c->r_pos.n, c0 = c->r_cigar.n, q0 = c->r_qual.n;
  const int sd = src_dev, dd = c->device;
  if (c0 + nc >= 0xffffffffull) { c->fail("more than 2^32 CIGAR ops in one contig"); return RSIGPU_E_RANGE; }
  CK(c->r_pos.append(b->pos, n, c->stream, sd, dd)); CK(c->r_mpos.append(b->mpos, n, c->stream, sd, dd)); CK(c->r_isize.append(b->isize, n, c->stream, sd, dd));
  CK(c->r_mtid.append(b->mtid, n, c->stream, sd, dd)); CK(c->r_flag.append(b->flag, n, c->stream, sd, dd)); CK(c->r_mapq.append(b->mapq, n, c->stream, sd, dd));
  CK(c->r_cigar.append(b->cigar, nc, c->stream, sd, dd)); CK(c->r_qual.append(b->qual, nq, c->stream, sd, dd));
  // offsets: entry r0 of the previous batch (its end) equals this batch's first entry after rebasing
  if (r0) { c->r_cigar_off.n = r0; c->r_qual_off.n = r0; }
  CK(c->r_cigar_off.append(b->cigar_off, n + 1, c->stream, sd, dd)); CK(c->r_qual_off.append(reinterpret_cast<const u64*>(b->qual_off), n + 1, c->stream, sd, dd));
  const u32 addc = (u32)c0 - cig_first; const u64 addq = (u64)q0 - q_first;
  if (addc) KL(k_add_u32, grid_for((int)std::min<size_t>(n + 1, 1u << 30), 1024, c->n_sm * 4), 256, 0, c->r_cigar_off.p + r0, n + 1, addc);
  if (addq) KL(k_add_u64, grid_for((int)std::min<size_t>(n + 1, 1u << 30), 1024, c->n_sm * 4), 256, 0, c->r_qual_off.p + r0, n + 1, addq);
  // the caller's buffers may be reused as soon as this returns
  CK(cudaStreamSynchronize(c->stream));
  return RSIGPU_OK;
}

int rsigpu_pileup_push(rsigpu_ctx* c, const rsigpu_read_batch* b) {
  if (!c || !b || b->n_reads < 0) return RSIGPU_E_ARG;
  if (b->n_reads == 0) return RSIGPU_OK;
  const size_t n = (size_t)b->n_reads;
  return push_impl(c, b, b->cigar_off[n], (size_t)b->qual_off[n], 0u, 0ull);
}

// ---------------------------------------------------------------------------------------------
// stable sort of read records (k_sort.cuh)
// LSD radix sort of the n keys in c->t_key over their low `bits` bits, stable in index order; *perm: the sorted order
static int sort_keys(rsigpu_ctx* c, u32 n, int bits, const u32** perm) {
  const u32 ntile = (n + SRT_TILE - 1) / SRT_TILE;
  CK(c->t_key2.ensure(n)); CK(c->t_idx.ensure(n)); CK(c->t_idx2.ensure(n)); CK(c->t_hist.ensure((size_t)SRT_RADIX * ntile)); CK(c->t_dtot.ensure(SRT_RADIX));
  u32 *ki = c->t_key.p, *ko = c->t_key2.p, *ii = nullptr, *io = c->t_idx.p;
  const int passes = std::max(1, (bits + SRT_BITS - 1) / SRT_BITS);
  for (int p = 0; p < passes; ++p) {
    KL(k_sort_hist, ntile, SRT_NT, 0, ki, n, p * SRT_BITS, c->t_hist.p, ntile);
    KL(k_sort_scan_rows, SRT_RADIX, SRT_NT, 0, c->t_hist.p, ntile, c->t_dtot.p);
    KL(k_sort_scatter, ntile, SRT_NT, 0, ki, ii, n, p * SRT_BITS, c->t_hist.p, c->t_dtot.p, ntile, ko, io);
    std::swap(ki, ko);
    ii = io; io = io == c->t_idx.p ? c->t_idx2.p : c->t_idx.p;
  }
  *perm = ii;
  return RSIGPU_OK;
}
// lc[0..n) / lq[0..n) hold lengths: exclusive prefix sums in place, the totals to lc[n] / lq[n] (n > 0)
static int lengths_to_offsets(rsigpu_ctx* c, u32* lc, u64* lq, u32 n) {
  const u32 ntile = (n + OFS_TILE - 1) / OFS_TILE;
  CK(c->t_ts.ensure(2 * (size_t)ntile));
  KL(k_off_tile_sums, ntile, OFS_NT, 0, lc, lq, n, c->t_ts.p, ntile);
  KL(k_off_tile_scan, 1, 1024, 0, c->t_ts.p, ntile, lc, lq, n);
  KL(k_off_apply, ntile, OFS_NT, 0, lc, lq, n, c->t_ts.p, ntile);
  return RSIGPU_OK;
}
static int bit_width(u32 v) { int b = 0; while (v) { ++b; v >>= 1; } return b; }

// ---------------------------------------------------------------------------------------------
// BAM bytes -> staged reads on the GPU (k_bam.cuh)
const int BY_REF_MAX_REFS = LIST_CAP - 1;   // with refID -1, one run per reference must fit a feed's run list

int rsigpu_bam_begin(rsigpu_ctx* c, int32_t n_ref) {
  if (!c || n_ref < 1) return RSIGPU_E_ARG;
  if (c->bam_by_ref && n_ref > BY_REF_MAX_REFS) {
    c->fail("bam_begin: " + std::to_string(n_ref) + " references, more than the 65535 that grouping records by refID (rsigpu_set_bam_by_ref) supports");
    return RSIGPU_E_ARG;
  }
  c->b_nref = n_ref; c->b_tail_len = 0; c->b_active = true; c->b_first_feed = true; c->b_runs.clear(); c->b_rewalked = 0;
  c->ix_on = false; c->ix_failed = false; c->ix_ready = false; c->ix_out.clear(); c->ix_ref.clear();
  return RSIGPU_OK;
}

int rsigpu_bam_index_begin(rsigpu_ctx* c, int64_t file_offset) {
  if (!c) return RSIGPU_E_ARG;
  if (c->bam_by_ref) { c->fail("bam_index_begin: not available while records are grouped by refID (rsigpu_set_bam_by_ref): the index needs them in file order"); return RSIGPU_E_ARG; }
  if (!c->b_active || !c->b_first_feed || file_offset < 0) { c->fail("bam_index_begin: call it after rsigpu_bam_begin and before the first feed, with the file offset of the first byte fed"); return RSIGPU_E_ARG; }
  c->ix_on = true; c->ix_failed = false; c->ix_ready = false; c->ix_has_prev = false; c->ix_off = file_offset;
  c->ix_carry_voff = 0; c->ix_end_voff = 0; c->ix_prev_key = 0; c->ix_no_coor = 0; c->ix_pend_on = false; c->ix_pend_tid = -1;
  c->ix_out.clear(); c->ix_ref.assign((size_t)c->b_nref, rsigpu_ctx::IxRef());
  return RSIGPU_OK;
}

// samtools-0.1.18's bam_index_save layout: per reference the bins in ascending order with their chunks (merge_chunks: a chunk
// whose begin lies in the BGZF block where the previous chunk of its bin ends is joined to it), the pseudo-bin 37450 (file
// range of the reference's records, mapped / unmapped counts), the 16 kbp linear index with uncovered windows taking the
// previous window's offset; the count of unplaced records last, when there are any
static void ix_serialize(rsigpu_ctx* c) {
  std::vector<uint8_t>& o = c->ix_out;
  o.clear();
  auto put32 = [&](u32 v) { for (int k = 0; k < 4; ++k) o.push_back((uint8_t)(v >> (8 * k))); };
  auto put64 = [&](u64 v) { for (int k = 0; k < 8; ++k) o.push_back((uint8_t)(v >> (8 * k))); };
  o.push_back('B'); o.push_back('A'); o.push_back('I'); o.push_back(1);
  put32((u32)c->ix_ref.size());
  for (rsigpu_ctx::IxRef& R : c->ix_ref) {
    if (R.ch.empty()) { put32(0); put32(0); continue; }
    const u64 first = R.ch.front().u, last = R.ch.back().v;
    std::stable_sort(R.ch.begin(), R.ch.end(), [](const rsigpu_ctx::IxChunk& a, const rsigpu_ctx::IxChunk& b) { return a.bin < b.bin; });
    std::vector<rsigpu_ctx::IxChunk> m;
    m.reserve(R.ch.size());
    int nbin = 1;
    for (const rsigpu_ctx::IxChunk& x : R.ch) {
      if (!m.empty() && m.back().bin == x.bin && m.back().v >> 16 == x.u >> 16) m.back().v = x.v;
      else { nbin += m.empty() || m.back().bin != x.bin; m.push_back(x); }
    }
    put32((u32)nbin);
    for (size_t i = 0; i < m.size();) {
      size_t j = i;
      while (j < m.size() && m[j].bin == m[i].bin) ++j;
      put32(m[i].bin); put32((u32)(j - i));
      for (; i < j; ++i) { put64(m[i].u); put64(m[i].v); }
    }
    put32(37450u); put32(2); put64(first); put64(last); put64(R.n_map); put64(R.n_unmap);
    for (size_t w = 1; w < R.lin.size(); ++w) if (!R.lin[w]) R.lin[w] = R.lin[w - 1];
    put32((u32)R.lin.size());
    for (u64 v : R.lin) put64(v);
  }
  if (c->ix_no_coor) put64(c->ix_no_coor);
}

int rsigpu_bam_index_get(rsigpu_ctx* c, uint8_t* out, int64_t cap, int64_t* nbytes) {
  if (!c || !nbytes) return RSIGPU_E_ARG;
  if (!c->ix_ready) { c->fail("bam_index_get: no index: rsigpu_bam_index_begin, feeds of the whole file and rsigpu_bam_end must all succeed first"); return RSIGPU_E_ARG; }
  *nbytes = (int64_t)c->ix_out.size();
  if (!out) return RSIGPU_OK;
  if (cap < *nbytes) { c->fail("bam_index_get: the buffer is smaller than the index"); return RSIGPU_E_CAPACITY; }
  memcpy(out, c->ix_out.data(), c->ix_out.size());
  return RSIGPU_OK;
}

// One feed over `nparts` byte ranges.  One range: the streaming form (a partial block at the end is left to the caller, a record
// cut by the end is carried).  Several ranges: each is a whole number of BGZF blocks that begins at a record start and ends at
// a record end (the records of one contig, say); they are decoded as ONE chunk -- one inflate launch over all their blocks --
// and every range starts a new run.
static int bam_feed_impl(rsigpu_ctx* c, int nparts, const uint8_t* const* ptrs, const int64_t* sizes, int64_t skip, int64_t* consumed, rsigpu_bam_run* runs, int32_t cap, int32_t* n_runs) {
  if (!c || nparts < 1 || !ptrs || !sizes || !n_runs || skip < 0) return RSIGPU_E_ARG;
  for (int j = 0; j < nparts; ++j) if (!ptrs[j] || sizes[j] < 0) return RSIGPU_E_ARG;
  const bool multi = nparts > 1;
  if (!multi && !consumed) return RSIGPU_E_ARG;
  if (!c->b_active) { c->fail("bam_feed: call rsigpu_bam_begin first"); return RSIGPU_E_ARG; }
  cudaSetDevice(c->device);
  if (consumed) *consumed = 0;
  *n_runs = 0; c->b_runs.clear();
  if (multi && c->b_tail_len) { c->fail("bam_feed_parts: a record of the previous feed is still incomplete"); return RSIGPU_E_ARG; }
  // BGZF block headers (bgzf.c:258-275): gzip magic, FEXTRA, the 'B','C' subfield carries the block size
  const size_t U_MAX = c->b_umax, C_MAX = (size_t)1 << 31;
  std::vector<BgzfBlock> blk; std::vector<i64> bound;
  size_t off = 0, utotal = 0;          // off: bytes of the packed compressed chunk so far (all parts)
  bound.push_back((i64)BAM_HEAD);
  std::vector<size_t> part_off((size_t)nparts + 1, 0); std::vector<int> part_blk((size_t)nparts, 0);
  for (int pj = 0; pj < nparts; ++pj) {
  const uint8_t* bgzf = ptrs[pj]; const size_t nbytes = (size_t)sizes[pj]; const size_t base = off;
  part_off[(size_t)pj] = base; part_blk[(size_t)pj] = (int)blk.size();
  while (off - base + 18 <= (size_t)nbytes) {
    const uint8_t* h = bgzf + (off - base);
    if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) { c->fail("bam_feed: not a BGZF block header"); return RSIGPU_E_ARG; }
    const size_t xlen = (size_t)h[10] | ((size_t)h[11] << 8);
    if (off - base + 12 + xlen > (size_t)nbytes) break;
    size_t bsize = 0; bool found = false;
    for (size_t x = 0; x + 4 <= xlen;) {
      const uint8_t* sf = h + 12 + x; const size_t sl = (size_t)sf[2] | ((size_t)sf[3] << 8);
      if (sf[0] == 'B' && sf[1] == 'C' && sl == 2 && x + 6 <= xlen) { bsize = ((size_t)sf[4] | ((size_t)sf[5] << 8)) + 1; found = true; break; }
      x += 4 + sl;
    }
    if (!found || bsize < 12 + xlen + 8) { c->fail("bam_feed: gzip member without a BGZF size field"); return RSIGPU_E_ARG; }
    if (off - base + bsize > (size_t)nbytes) break;
    const uint8_t* foot = h + bsize - 8;
    const size_t ulen = (size_t)foot[4] | ((size_t)foot[5] << 8) | ((size_t)foot[6] << 16) | ((size_t)foot[7] << 24);
    const u32 crc = (u32)foot[0] | ((u32)foot[1] << 8) | ((u32)foot[2] << 16) | ((u32)foot[3] << 24);
    if (ulen > 65536) { c->fail("bam_feed: BGZF block larger than 64 KiB"); return RSIGPU_E_ARG; }
    if (utotal + ulen > U_MAX || off + bsize > C_MAX) break;
    BgzfBlock B; B.src = (u32)(off + 12 + xlen); B.src_len = (u32)(bsize - 12 - xlen - 8); B.dst = (u64)BAM_HEAD + utotal; B.dst_len = (u32)ulen; B.crc = crc;
    blk.push_back(B);
    utotal += ulen; off += bsize;
    bound.push_back((i64)(BAM_HEAD + utotal));
  }
  if (multi && off - base != nbytes) { c->fail("bam_feed_parts: a part is not a whole number of BGZF blocks, or the parts exceed one feed's capacity"); return RSIGPU_E_RANGE; }
  }
  part_off[(size_t)nparts] = off;
  const int nblk = (int)blk.size();
  if (nblk == 0) {
    if ((size_t)sizes[0] >= ((size_t)1 << 17)) { c->fail("bam_feed: no whole BGZF block in 128 KiB"); return RSIGPU_E_ARG; }
    return RSIGPU_OK;
  }
  if (c->b_first_feed) { if ((size_t)skip > utotal) { c->fail("bam_feed: skip beyond the decoded chunk"); return RSIGPU_E_ARG; } }
  else if (skip != 0) { c->fail("bam_feed: skip is only meaningful on the first feed"); return RSIGPU_E_ARG; }
  CK(c->b_comp.ensure(off + 64)); CK(c->b_U.ensure((size_t)BAM_HEAD + utotal + 64)); CK(c->b_blk.ensure((size_t)nblk)); CK(c->b_bound.ensure((size_t)nblk + 1));
  CK(c->b_first.ensure(nblk)); CK(c->b_endp.ensure(nblk)); CK(c->b_tailp.ensure(nblk)); CK(c->b_cnt.ensure(nblk)); CK(c->b_ncig.ensure(nblk)); CK(c->b_nq.ensure(nblk));
  CK(c->b_in.ensure(nblk)); CK(c->b_rbase.ensure(nblk)); CK(c->b_cbase.ensure(nblk)); CK(c->b_qbase.ensure(nblk)); CK(c->b_info.ensure(8)); CK(c->b_cnt32.ensure(4));
  TRACE(c, "feed: start");
  for (int pj = 0; pj < nparts; ++pj) if (part_off[(size_t)pj + 1] > part_off[(size_t)pj])
    CK(cudaMemcpyAsync(c->b_comp.p + part_off[(size_t)pj], ptrs[pj], part_off[(size_t)pj + 1] - part_off[(size_t)pj], cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(c->b_blk.p, blk.data(), (size_t)nblk * sizeof(BgzfBlock), cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(c->b_bound.p, bound.data(), ((size_t)nblk + 1) * 8, cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemsetAsync(c->b_info.p, 0, 8 * 8, c->stream)); CK(cudaMemsetAsync(c->b_cnt32.p, 0, 4 * 4, c->stream));
  if (c->b_tail_len) CK(cudaMemcpyAsync(c->b_U.p + (BAM_HEAD - c->b_tail_len), c->b_carry.p, (size_t)c->b_tail_len, cudaMemcpyDeviceToDevice, c->stream));
  i64* info = c->b_info.p; int* err = c->b_cnt32.p;
  if (trace_on()) { cudaStreamSynchronize(c->stream); TRACE(c, "feed: H2D done"); }
  // two inflate kernels (k_inflate_warp.cuh): a warp per block costs time proportional to the chunk, a lane per block about
  // the same 30-38 ms for any chunk up to a chr19-sized one
  if (c->inflate_mode == 2 || (c->inflate_mode == 0 && nblk < (int)infw::INFW_MAX_BLOCKS))
    KL(k_bgzf_inflate_warp, (nblk + infw::INFW_WARPS - 1) / infw::INFW_WARPS, infw::INFW_NT, 0, c->b_comp.p, (u32)((off + 3) / 4), c->b_blk.p, nblk, c->b_U.p, err);
  else {
    CK(c->b_tabs.ensure(RSI_INFLATE_TAB_BYTES(nblk) / 2));
    KL(k_bgzf_inflate, (nblk + INF_NT - 1) / INF_NT, INF_NT, 0, c->b_comp.p, c->b_blk.p, nblk, c->b_U.p, c->b_tabs.p, err);
  }
  if (c->bgzf_crc) KL(k_bgzf_crc32, grid_for(nblk, CRC_WARPS, c->n_sm), CRC_NT, CRC_SMEM, c->b_U.p, c->b_blk.p, nblk, err);
  BamChunk C; C.U = c->b_U.p; C.u_begin = c->b_first_feed ? (i64)BAM_HEAD + skip : (i64)BAM_HEAD - c->b_tail_len; C.u_end = (i64)(BAM_HEAD + utotal);
  C.bound = c->b_bound.p; C.nblk = nblk; C.n_ref = c->b_nref;
  BamChain H; H.first = c->b_first.p; H.endp = c->b_endp.p; H.tailp = c->b_tailp.p; H.cnt = c->b_cnt.p; H.ncig = c->b_ncig.p; H.nq = c->b_nq.p;
  KL(k_bam_chain, (nblk + 127) / 128, 128, 0, C, H);
  KL(k_bam_verify, 1, 1024, 0, C, H, c->b_in.p, c->b_rbase.p, c->b_cbase.p, c->b_qbase.p, info, err);
  i64 hi[8]; int he[4];
  if (trace_on()) { cudaStreamSynchronize(c->stream); TRACE(c, "feed: inflate+chain done"); }
  CK(cudaMemcpyAsync(hi, info, 8 * 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(he, err, 4 * 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (he[1] & BAM_ERR_INFLATE) { c->fail("bam_feed: corrupt deflate stream in a BGZF block (code " + std::to_string(he[2]) + ")"); return RSIGPU_E_ARG; }
  if (he[1] & BAM_ERR_CRC) {           // he[3] = nblk - (lowest failing block)
    const int k = nblk - he[3];
    int pj = 0; while (pj + 1 < nparts && part_blk[(size_t)pj + 1] <= k) ++pj;
    // blocks of a part are contiguous: block k starts where block k - 1 of the same part ends
    const size_t start = k == part_blk[(size_t)pj] ? part_off[(size_t)pj] : (size_t)blk[(size_t)k - 1].src + blk[(size_t)k - 1].src_len + 8;
    if (multi) c->fail("bam_feed_parts: CRC32 mismatch in BGZF block " + std::to_string(k - part_blk[(size_t)pj]) + " of part " + std::to_string(pj) +
                       " (compressed offset " + std::to_string(start - part_off[(size_t)pj]) + " of that part)");
    else c->fail("bam_feed: CRC32 mismatch in BGZF block " + std::to_string(k) + " of this feed (compressed offset " + std::to_string(start) + " of the bytes passed)");
    return RSIGPU_E_ARG;
  }
  if (he[1] & BAM_ERR_RECORD) { c->fail("bam_feed: corrupt BAM record"); return RSIGPU_E_ARG; }
  const size_t n = (size_t)hi[0], ncg = (size_t)hi[1]; const i64 nq64 = hi[2];
  const i64 tail_start = hi[3];
  c->b_rewalked += (int)hi[4];
  c->b_first_feed = false;
  u64 xc[BIX_C_N] = {};
  std::vector<BixChunk> xchunk; std::vector<BixLin> xlin;
  if (n) {
    CK(c->b_rec.ensure(n)); CK(c->b_tid.ensure(n)); CK(c->b_pos.ensure(n)); CK(c->b_mpos.ensure(n)); CK(c->b_isize.ensure(n)); CK(c->b_mtid.ensure(n));
    CK(c->b_flag.ensure(n)); CK(c->b_mapq.ensure(n)); CK(c->b_cigoff.ensure(n + 1)); CK(c->b_qoff.ensure(n + 1)); CK(c->b_cig.ensure(ncg + 1)); CK(c->b_qual.ensure((size_t)nq64 + 16));
    CK(c->b_runstart.ensure(LIST_CAP)); CK(c->b_runinfo.ensure(3 * (size_t)LIST_CAP));
    BamSoA S; S.rec = c->b_rec.p; S.tid = c->b_tid.p; S.pos = c->b_pos.p; S.mpos = c->b_mpos.p; S.isize = c->b_isize.p; S.mtid = c->b_mtid.p; S.flag = c->b_flag.p;
    S.mapq = c->b_mapq.p; S.cigar_off = c->b_cigoff.p; S.cigar = c->b_cig.p; S.qual_off = c->b_qoff.p; S.qual = c->b_qual.p;
    KL(k_bam_fields, (nblk + 127) / 128, 128, 0, C, H, c->b_rbase.p, c->b_cbase.p, c->b_qbase.p, info, S);
    if (c->bam_by_ref) {
      // the records grouped by refID, stable in file order (k_sort.cuh): the fixed fields and the offsets move, and
      // k_bam_payload then copies every record's CIGAR and qualities from the inflated bytes straight to its sorted place
      CK(c->t_key.ensure(n)); CK(c->b2_rec.ensure(n)); CK(c->b2_tid.ensure(n)); CK(c->b2_pos.ensure(n)); CK(c->b2_mpos.ensure(n)); CK(c->b2_isize.ensure(n));
      CK(c->b2_mtid.ensure(n)); CK(c->b2_flag.ensure(n)); CK(c->b2_mapq.ensure(n)); CK(c->b2_cigoff.ensure(n + 1)); CK(c->b2_qoff.ensure(n + 1));
      const int g = grid_for((int)n, 1024, c->n_sm * 8);
      KL(k_sort_key_tid, g, 256, 0, c->b_tid.p, (u32)n, (u32)c->b_nref, c->t_key.p);
      const u32* perm = nullptr;
      int rc = sort_keys(c, (u32)n, bit_width((u32)c->b_nref), &perm);
      if (rc) return rc;
      SortFields fi{c->b_rec.p, c->b_tid.p, c->b_pos.p, c->b_mpos.p, c->b_isize.p, c->b_mtid.p, c->b_flag.p, c->b_mapq.p, c->b_cigoff.p, c->b_qoff.p};
      SortFields fo{c->b2_rec.p, c->b2_tid.p, c->b2_pos.p, c->b2_mpos.p, c->b2_isize.p, c->b2_mtid.p, c->b2_flag.p, c->b2_mapq.p, c->b2_cigoff.p, c->b2_qoff.p};
      KL(k_sort_gather, g, 256, 0, perm, (u32)n, fi, fo);
      if ((rc = lengths_to_offsets(c, c->b2_cigoff.p, c->b2_qoff.p, (u32)n))) return rc;
      std::swap(c->b_rec, c->b2_rec); std::swap(c->b_tid, c->b2_tid); std::swap(c->b_pos, c->b2_pos); std::swap(c->b_mpos, c->b2_mpos); std::swap(c->b_isize, c->b2_isize);
      std::swap(c->b_mtid, c->b2_mtid); std::swap(c->b_flag, c->b2_flag); std::swap(c->b_mapq, c->b2_mapq); std::swap(c->b_cigoff, c->b2_cigoff); std::swap(c->b_qoff, c->b2_qoff);
      S.rec = c->b_rec.p; S.tid = c->b_tid.p; S.pos = c->b_pos.p; S.mpos = c->b_mpos.p; S.isize = c->b_isize.p; S.mtid = c->b_mtid.p; S.flag = c->b_flag.p;
      S.mapq = c->b_mapq.p; S.cigar_off = c->b_cigoff.p; S.qual_off = c->b_qoff.p;
    }
    KL(k_bam_payload, c->n_sm * 8, 256, 0, c->b_U.p, info, S);
    KL(k_bam_runs, grid_for((int)std::min<size_t>(n, 1u << 30), 1024, c->n_sm * 8), 256, 0, c->b_tid.p, info, c->b_runstart.p, (int)LIST_CAP, err);
    if (c->ix_on) {          // the BAI index's share of this feed (k_bam_index.cuh); its counts travel with the error copy below
      const int ntile = (int)((n + BIX_NT - 1) / BIX_NT);
      CK(c->x_beg.ensure(n)); CK(c->x_key.ensure(n)); CK(c->x_meta.ensure(n)); CK(c->x_chunk.ensure(n)); CK(c->x_lin.ensure(n));
      CK(c->x_tstart.ensure((size_t)ntile)); CK(c->x_tunmap.ensure((size_t)ntile)); CK(c->x_tkey.ensure((size_t)ntile)); CK(c->x_cnt.ensure(BIX_C_N));
      CK(cudaMemsetAsync(c->x_cnt.p, 0, BIX_C_N * 8, c->stream));
      BixFeed F;
      F.U = c->b_U.p; F.bound = c->b_bound.p; F.blk = c->b_blk.p; F.nblk = nblk; F.base = (i64)c->ix_off; F.carry_voff = c->ix_carry_voff; F.n = (int)n;
      F.rec = c->b_rec.p; F.tid = c->b_tid.p; F.pos = c->b_pos.p; F.flag = c->b_flag.p; F.cigar_off = c->b_cigoff.p; F.cigar = c->b_cig.p;
      F.has_prev = c->ix_has_prev; F.prev_tid = c->ix_prev_tid; F.prev_pos = c->ix_prev_pos; F.prev_bin = c->ix_prev_bin; F.prev_key = c->ix_prev_key;
      F.beg = c->x_beg.p; F.key = c->x_key.p; F.meta = c->x_meta.p; F.t_start = c->x_tstart.p; F.t_unmap = c->x_tunmap.p; F.t_key = c->x_tkey.p;
      F.chunk = c->x_chunk.p; F.lin = c->x_lin.p; F.cnt = c->x_cnt.p;
      KL(k_bam_index_rec, ntile, BIX_NT, 0, F);
      KL(k_bam_index_scan, 1, BIX_SCAN_NT, 0, F, ntile);
      KL(k_bam_index_emit, ntile, BIX_NT, 0, F);
      CK(cudaMemcpyAsync(xc, c->x_cnt.p, BIX_C_N * 8, cudaMemcpyDeviceToHost, c->stream));
    }
    std::vector<int> part_rec;           // first record of every part (each part starts a run whatever its refID)
    if (multi) {
      part_rec.resize((size_t)nparts);
      for (int pj = 0; pj < nparts; ++pj) CK(cudaMemcpyAsync(&part_rec[(size_t)pj], c->b_rbase.p + part_blk[(size_t)pj], 4, cudaMemcpyDeviceToHost, c->stream));
    }
    CK(cudaMemcpyAsync(he, err, 4 * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (c->ix_on && xc[BIX_C_UNSORTED]) {
      const i64 k = (i64)n - (i64)xc[BIX_C_UNSORTED];
      int t[2] = {c->ix_prev_tid, 0}, q[2] = {c->ix_prev_pos, 0};
      if (k > 0) { CK(cudaMemcpyAsync(t, c->b_tid.p + k - 1, 8, cudaMemcpyDeviceToHost, c->stream)); CK(cudaMemcpyAsync(q, c->b_pos.p + k - 1, 8, cudaMemcpyDeviceToHost, c->stream)); }
      else { CK(cudaMemcpyAsync(t + 1, c->b_tid.p, 4, cudaMemcpyDeviceToHost, c->stream)); CK(cudaMemcpyAsync(q + 1, c->b_pos.p, 4, cudaMemcpyDeviceToHost, c->stream)); }
      CK(cudaStreamSynchronize(c->stream));
      c->fail("bam_index: records not sorted: record " + std::to_string(k) + " of this feed (tid " + std::to_string(t[1]) + ", pos " + std::to_string(q[1]) +
              ") follows tid " + std::to_string(t[0]) + ", pos " + std::to_string(q[0]));
      return RSIGPU_E_ARG;
    }
    if (c->ix_on && xc[BIX_C_RANGE]) {
      const i64 k = (i64)n - (i64)xc[BIX_C_RANGE];
      int t = 0, q = 0;
      CK(cudaMemcpyAsync(&t, c->b_tid.p + k, 4, cudaMemcpyDeviceToHost, c->stream)); CK(cudaMemcpyAsync(&q, c->b_pos.p + k, 4, cudaMemcpyDeviceToHost, c->stream));
      CK(cudaStreamSynchronize(c->stream));
      c->fail("bam_index: record " + std::to_string(k) + " of this feed (tid " + std::to_string(t) + ", pos " + std::to_string(q) +
              ") ends past 2^29, beyond what a BAI index can address");
      return RSIGPU_E_RANGE;
    }
    if (c->ix_on) {        // copied with the run starts below
      xchunk.resize((size_t)xc[BIX_C_CHUNKS]); xlin.resize((size_t)xc[BIX_C_LIN]);
      if (!xchunk.empty()) CK(cudaMemcpyAsync(xchunk.data(), c->x_chunk.p, xchunk.size() * sizeof(BixChunk), cudaMemcpyDeviceToHost, c->stream));
      if (!xlin.empty()) CK(cudaMemcpyAsync(xlin.data(), c->x_lin.p, xlin.size() * sizeof(BixLin), cudaMemcpyDeviceToHost, c->stream));
    }
    if (he[1] & BAM_ERR_RUNS) { c->fail("bam_feed: more than 65536 refID runs in one chunk (the BAM is not coordinate-sorted)"); return RSIGPU_E_RANGE; }
    int nr = he[0];
    std::vector<int> rs((size_t)nr);
    CK(cudaMemcpyAsync(rs.data(), c->b_runstart.p, (size_t)nr * 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (multi) { for (int pj = 0; pj < nparts; ++pj) if (part_blk[(size_t)pj] < (pj + 1 < nparts ? part_blk[(size_t)pj + 1] : nblk) && (size_t)part_rec[(size_t)pj] < n) rs.push_back(part_rec[(size_t)pj]); }
    std::sort(rs.begin(), rs.end());
    rs.erase(std::unique(rs.begin(), rs.end()), rs.end());
    if (rs.size() > (size_t)LIST_CAP) { c->fail("bam_feed: more than 65536 runs in one chunk"); return RSIGPU_E_RANGE; }
    nr = (int)rs.size();
    CK(cudaMemcpyAsync(c->b_runstart.p, rs.data(), (size_t)nr * 4, cudaMemcpyHostToDevice, c->stream));
    KL(k_bam_run_info, 1, 256, 0, c->b_runstart.p, nr, S, c->b_runinfo.p);
    std::vector<i64> ri(3 * (size_t)nr);
    CK(cudaMemcpyAsync(ri.data(), c->b_runinfo.p, ri.size() * 8, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < nr; ++i) {
      rsigpu_ctx::BamRun R; R.tid = (int)ri[3 * (size_t)i]; R.r0 = rs[(size_t)i]; R.c0 = ri[3 * (size_t)i + 1]; R.q0 = ri[3 * (size_t)i + 2];
      R.part = 0; R.by_ref = c->bam_by_ref;
      if (multi) { while (R.part + 1 < nparts && part_rec[(size_t)R.part + 1] <= rs[(size_t)i] && part_blk[(size_t)R.part + 1] < nblk) ++R.part; }
      R.r1 = i + 1 < nr ? rs[(size_t)i + 1] : (i64)n; R.c1 = i + 1 < nr ? ri[3 * (size_t)i + 4] : (i64)ncg; R.q1 = i + 1 < nr ? ri[3 * (size_t)i + 5] : nq64;
      c->b_runs.push_back(R);
    }
  }
  // the record cut by the end of this chunk is kept for the next feed (it goes in front of that chunk's first block); a record
  // that began in the carry and still does not end here (tail_start < BAM_HEAD) is carried again, however many feeds it spans
  const i64 tail_len = (i64)(BAM_HEAD + utotal) - tail_start;
  if (multi && tail_len > 0) { c->fail("bam_feed_parts: the last part ends inside a record"); return RSIGPU_E_ARG; }
  if (tail_len > 0) {
    if (tail_len > (i64)BAM_HEAD) {
      u32 bs = 0;                        // the record's block_size: its first 4 bytes are decoded
      CK(cudaMemcpyAsync(&bs, c->b_U.p + tail_start, 4, cudaMemcpyDeviceToHost, c->stream));
      CK(cudaStreamSynchronize(c->stream));
      c->fail("bam_feed: an alignment record of " + std::to_string((u64)bs + 4) + " bytes, longer than the decoder's carry buffer (16 MiB)");
      return RSIGPU_E_RANGE;
    }
    CK(c->b_carry.ensure((size_t)BAM_HEAD));
    CK(cudaMemcpyAsync(c->b_carry.p, c->b_U.p + tail_start, (size_t)tail_len, cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
  }
  c->b_tail_len = tail_len > 0 ? (int)tail_len : 0;
  if (c->ix_on) {
    // voffset of decoded position x: the last block that starts at or before it
    auto voff_at = [&](i64 x) {
      const int k = (int)(std::upper_bound(bound.begin(), bound.begin() + nblk, x) - bound.begin()) - 1;
      const u64 co = (u64)c->ix_off + (k ? (u64)blk[(size_t)k - 1].src + blk[(size_t)k - 1].src_len + 8 : 0ull);
      return (co << 16) | (u64)(x - bound[(size_t)k]);
    };
    for (size_t i = 0; i < xchunk.size(); ++i) {
      const BixChunk& h = xchunk[i];
      if (c->ix_pend_on && c->ix_pend_tid >= 0) { c->ix_pend.v = h.u; c->ix_ref[(size_t)c->ix_pend_tid].ch.push_back(c->ix_pend); }
      c->ix_pend.bin = h.bin; c->ix_pend.u = h.u; c->ix_pend.v = 0; c->ix_pend_tid = h.tid; c->ix_pend_on = true;
      const i64 nrec = (i + 1 < xchunk.size() ? (i64)xchunk[i + 1].rec : (i64)n) - h.rec;
      const i64 nun = (i + 1 < xchunk.size() ? (i64)xchunk[i + 1].unmap : (i64)xc[BIX_C_UNMAP]) - h.unmap;
      if (h.tid >= 0) { c->ix_ref[(size_t)h.tid].n_unmap += (u64)nun; c->ix_ref[(size_t)h.tid].n_map += (u64)(nrec - nun); }
      else c->ix_no_coor += (u64)nrec;
    }
    for (const BixLin& L : xlin) {
      std::vector<u64>& lin = c->ix_ref[(size_t)L.tid].lin;
      if (lin.size() < (size_t)L.w1 + 1) lin.resize((size_t)L.w1 + 1, 0);
      for (int w = L.w0; w <= L.w1; ++w) lin[(size_t)w] = L.voff;
    }
    if (n) { c->ix_has_prev = true; c->ix_prev_tid = (int)(u32)xc[BIX_C_LAST_TID]; c->ix_prev_pos = (int)(u32)xc[BIX_C_LAST_POS]; c->ix_prev_bin = (u32)xc[BIX_C_LAST_BIN]; c->ix_prev_key = xc[BIX_C_MAXKEY]; }
    if (tail_len > 0 && tail_start >= (i64)BAM_HEAD) c->ix_carry_voff = voff_at(tail_start);   // else: the carried record began in an earlier feed
    // where the stream stops if this is the last feed: an empty block at the end (the EOF marker) is that place, else the byte after the chunk
    const i64 u_end = (i64)(BAM_HEAD + utotal);
    c->ix_end_voff = bound[(size_t)nblk - 1] == u_end ? voff_at(u_end) : (u64)(c->ix_off + (int64_t)off) << 16;
    c->ix_off += (int64_t)off;
  }
  TRACE(c, "feed: end");
  if (consumed) *consumed = (int64_t)off;
  *n_runs = (int32_t)c->b_runs.size();
  for (int i = 0; i < (int)c->b_runs.size() && i < cap && runs; ++i) { runs[i].tid = c->b_runs[(size_t)i].tid; runs[i].part = c->b_runs[(size_t)i].part; runs[i].n_reads = c->b_runs[(size_t)i].r1 - c->b_runs[(size_t)i].r0; }
  return RSIGPU_OK;
}

int rsigpu_bam_feed(rsigpu_ctx* c, const uint8_t* bgzf, int64_t nbytes, int64_t skip, int64_t* consumed, rsigpu_bam_run* runs, int32_t cap, int32_t* n_runs) {
  if (!bgzf || !consumed) return RSIGPU_E_ARG;
  const uint8_t* p[1] = {bgzf}; const int64_t n[1] = {nbytes};
  const int rc = bam_feed_impl(c, 1, p, n, skip, consumed, runs, cap, n_runs);
  if (rc != RSIGPU_OK && c) c->ix_failed = true;     // an index missing this feed's records would be wrong: rsigpu_bam_index_get refuses
  return rc;
}
int rsigpu_bam_feed_parts(rsigpu_ctx* c, int32_t n_parts, const uint8_t* const* parts, const int64_t* nbytes, rsigpu_bam_run* runs, int32_t cap, int32_t* n_runs) {
  if (n_parts < 1) return RSIGPU_E_ARG;
  if (c && c->bam_by_ref) { c->fail("bam_feed_parts: not available while records are grouped by refID (rsigpu_set_bam_by_ref): each part already starts its own run"); return RSIGPU_E_ARG; }
  if (c && c->ix_on) { c->ix_failed = true; c->fail("bam_feed_parts: not available while a BAM index is built (rsigpu_bam_index_begin): its parts are not one contiguous file"); return RSIGPU_E_ARG; }
  if (n_parts == 1) { int64_t consumed = 0; const int rc = bam_feed_impl(c, 1, parts, nbytes, 0, &consumed, runs, cap, n_runs); if (rc == RSIGPU_OK && consumed != nbytes[0]) { c->fail("bam_feed_parts: a part is not a whole number of BGZF blocks"); return RSIGPU_E_RANGE; } return rc; }
  return bam_feed_impl(c, n_parts, parts, nbytes, 0, nullptr, runs, cap, n_runs);
}

int rsigpu_bam_take(rsigpu_ctx* c, int32_t run, rsigpu_ctx* dst) {
  if (!c || !dst || run < 0 || run >= (int)c->b_runs.size()) return RSIGPU_E_ARG;
  if (!dst->have_ref) { dst->fail("bam_take: call set_reference and pileup_begin on the destination first"); return RSIGPU_E_ARG; }
  const rsigpu_ctx::BamRun& R = c->b_runs[(size_t)run];
  rsigpu_read_batch b; memset(&b, 0, sizeof b);
  b.n_reads = R.r1 - R.r0; b.tid = R.tid;
  if (b.n_reads == 0) return RSIGPU_OK;
  b.pos = c->b_pos.p + R.r0; b.mpos = c->b_mpos.p + R.r0; b.isize = c->b_isize.p + R.r0; b.mtid = c->b_mtid.p + R.r0; b.flag = c->b_flag.p + R.r0; b.mapq = c->b_mapq.p + R.r0;
  b.cigar_off = c->b_cigoff.p + R.r0; b.cigar = c->b_cig.p + R.c0; b.qual_off = reinterpret_cast<const uint64_t*>(c->b_qoff.p + R.r0); b.qual = c->b_qual.p + R.q0;
  return push_impl(dst, &b, (size_t)(R.c1 - R.c0), (size_t)(R.q1 - R.q0), (u32)R.c0, (u64)R.q0, c->device);
}

// the records of a run whose pos lies in [pos_lo, pos_hi): what one part of a contig split over several GPUs stages
int rsigpu_bam_take_range(rsigpu_ctx* c, int32_t run, rsigpu_ctx* dst, int32_t pos_lo, int32_t pos_hi) {
  if (!c || !dst || run < 0 || run >= (int)c->b_runs.size()) return RSIGPU_E_ARG;
  if (!dst->have_ref) { dst->fail("bam_take: call set_reference and pileup_begin on the destination first"); return RSIGPU_E_ARG; }
  const rsigpu_ctx::BamRun& R = c->b_runs[(size_t)run];
  if (R.by_ref) { c->fail("bam_take_range: run " + std::to_string(run) + " was grouped by refID (rsigpu_set_bam_by_ref): its positions are not sorted"); return RSIGPU_E_ARG; }
  const long long n = R.r1 - R.r0;
  if (n == 0 || pos_hi <= pos_lo) return RSIGPU_OK;
  cudaSetDevice(c->device);
  long long* dcount = reinterpret_cast<long long*>(c->d_cprof.p);     // 16 x 8 bytes of scratch
  KL(k_count_before, 1, 1, 0, c->b_pos.p + R.r0, n, pos_lo, dcount);
  KL(k_count_before, 1, 1, 0, c->b_pos.p + R.r0, n, pos_hi, dcount + 1);
  long long h[2] = {0, 0};
  CK(cudaMemcpyAsync(h, dcount, 16, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const long long i0 = h[0], i1 = h[1];
  if (i1 <= i0) return RSIGPU_OK;
  u32 co[2]; u64 qo[2];
  CK(cudaMemcpyAsync(&co[0], c->b_cigoff.p + R.r0 + i0, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&co[1], c->b_cigoff.p + R.r0 + i1, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&qo[0], c->b_qoff.p + R.r0 + i0, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&qo[1], c->b_qoff.p + R.r0 + i1, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  rsigpu_read_batch b; memset(&b, 0, sizeof b);
  const long long a = R.r0 + i0;
  b.n_reads = i1 - i0; b.tid = R.tid;
  b.pos = c->b_pos.p + a; b.mpos = c->b_mpos.p + a; b.isize = c->b_isize.p + a; b.mtid = c->b_mtid.p + a; b.flag = c->b_flag.p + a; b.mapq = c->b_mapq.p + a;
  b.cigar_off = c->b_cigoff.p + a; b.cigar = c->b_cig.p + co[0]; b.qual_off = reinterpret_cast<const uint64_t*>(c->b_qoff.p + a); b.qual = c->b_qual.p + qo[0];
  return push_impl(dst, &b, (size_t)(co[1] - co[0]), (size_t)(qo[1] - qo[0]), co[0], qo[0], c->device);
}

int rsigpu_bam_end(rsigpu_ctx* c) {
  if (!c) return RSIGPU_E_ARG;
  const bool cut = c->b_active && c->b_tail_len > 0;
  c->b_active = false; c->b_runs.clear(); c->b_tail_len = 0;
  if (c->ix_on) {
    c->ix_on = false;
    if (!cut && !c->ix_failed) {
      if (c->ix_pend_on && c->ix_pend_tid >= 0) { c->ix_pend.v = c->ix_end_voff; c->ix_ref[(size_t)c->ix_pend_tid].ch.push_back(c->ix_pend); }
      c->ix_pend_on = false;
      ix_serialize(c);
      c->ix_ref.clear();
      c->ix_ready = true;
    }
  }
  if (cut) { c->fail("bam_end: the BAM stream stops inside an alignment record"); return RSIGPU_E_ARG; }
  return RSIGPU_OK;
}

int rsigpu_bam_run_field(rsigpu_ctx* c, int32_t run, int32_t field, void* out, int64_t cap_bytes, int64_t* nbytes) {
  if (!c || !nbytes || run < 0 || run >= (int)c->b_runs.size()) return RSIGPU_E_ARG;
  cudaSetDevice(c->device);
  const rsigpu_ctx::BamRun& R = c->b_runs[(size_t)run];
  const size_t n = (size_t)(R.r1 - R.r0);
  const void* src = nullptr; size_t bytes = 0;
  switch (field) {
    case 0: src = c->b_pos.p + R.r0; bytes = n * 4; break;
    case 1: src = c->b_mpos.p + R.r0; bytes = n * 4; break;
    case 2: src = c->b_isize.p + R.r0; bytes = n * 4; break;
    case 3: src = c->b_mtid.p + R.r0; bytes = n * 4; break;
    case 4: src = c->b_flag.p + R.r0; bytes = n * 2; break;
    case 5: src = c->b_mapq.p + R.r0; bytes = n; break;
    case 6: src = c->b_cigoff.p + R.r0; bytes = (n + 1) * 4; break;
    case 7: src = c->b_cig.p + R.c0; bytes = (size_t)(R.c1 - R.c0) * 4; break;
    case 8: src = c->b_qoff.p + R.r0; bytes = (n + 1) * 8; break;
    case 9: src = c->b_qual.p + R.q0; bytes = (size_t)(R.q1 - R.q0); break;
    default: return RSIGPU_E_ARG;
  }
  *nbytes = (int64_t)bytes;
  if (!out || cap_bytes < (int64_t)bytes) return RSIGPU_OK;
  if (bytes) { CK(cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToHost, c->stream)); CK(cudaStreamSynchronize(c->stream)); }
  if (field == 6) { u32* o = (u32*)out; const u32 b0 = (u32)R.c0; for (size_t i = 0; i <= n; ++i) o[i] -= b0; }
  if (field == 8) { u64* o = (u64*)out; const u64 b0 = (u64)R.q0; for (size_t i = 0; i <= n; ++i) o[i] -= b0; }
  return RSIGPU_OK;
}

int rsigpu_pinned_alloc(size_t nbytes, void** out) {
  if (!out) return RSIGPU_E_ARG;
  return cudaMallocHost(out, nbytes ? nbytes : 1) == cudaSuccess ? RSIGPU_OK : RSIGPU_E_CUDA;
}
void rsigpu_pinned_free(void* p) { if (p) cudaFreeHost(p); }

// the pileup kernels on the staged reads -> raw depth (a5)
static int run_pileup(rsigpu_ctx* c, int pt0 = 0, int pt1 = 0x7fffffff, bool with_isize = true) {
  cudaSetDevice(c->device);
  const size_t padded = ((size_t)c->L + LD_TILE - 1) / LD_TILE * LD_TILE + 64;
  CK(c->d_raw.ensure(padded));
  int* mx = c->d_misc.p + 5;   // max_extent, sorted_bad
  // a previous insert-size sample (second stream) may still be reading max_extent
  if (c->isize_pending) { CK(cudaStreamWaitEvent(c->stream, c->ev_isize, 0)); c->isize_pending = false; }
  CK(cudaMemsetAsync(mx, 0, 8, c->stream));
  if (c->r_pos.n == 0) {
    CK(cudaMemsetAsync(c->d_raw.p, 0, padded * 4, c->stream));
  } else {
    CK(c->r_calend.ensure(c->r_pos.n + 8)); CK(c->r_ncig.ensure(c->r_pos.n + 8));
    ReadSoA R = read_view(c);
    // one launch: the read-end pass (calend, ncig, max_extent, sortedness) in the first n_sm * PU_ENDS_PER_SM blocks, the
    // quality-mask stream in the rest
    const u64 nq = (u64)c->r_qual.n;
    CK(c->d_qmask.ensure((size_t)((nq + 31) >> 5) + 16));
    KL(k_qual_mask, c->n_sm * 16, 256, 0, c->r_qual.p, nq, c->P.min_baseQ, c->d_qmask.p, R, mx, mx + 1, c->n_sm * PU_ENDS_PER_SM);
    // the insert-size sample (bam_rd_pr_stats) needs only the reads: it runs beside the depth pipeline on a second stream
    if (with_isize) {
      CK(cudaEventRecord(c->ev_reads, c->stream));
      CK(cudaStreamWaitEvent(c->stream2, c->ev_reads, 0));
      {
        cudaStream_t main_s = c->stream; c->stream = c->stream2;
        KL(k_isize_stats, 1, 1024, 0, R, c->L, mx, c->d_misc.p + 16);
        c->stream = main_s;
      }
      CK(cudaEventRecord(c->ev_isize, c->stream2));
      c->isize_pending = true;
    }
    const int ntile = (c->L + PU_T - 1) / PU_T;
    CK(c->d_tile_range.ensure((size_t)ntile * 2 + 8));
    int2* tr = reinterpret_cast<int2*>(c->d_tile_range.p);
    KL(k_tile_ranges, grid_for(ntile, 128, c->n_sm * 8), 128, 0, R, c->L, mx, tr);
    const int npt = std::min(ntile, pt1) - pt0;
    // one block per tile: tiles differ in cost (read density, N runs), and the block scheduler hands out the next tile to
    // whichever SM frees up first (with 8192-base tiles, a fixed stride of n_sm * 6 blocks measured 0.49 ms against 0.43 ms
    // on a 59.1 Mbp contig)
    if (npt > 0) KL(k_pileup_tile, npt, PU_NT, 0, R, c->d_qmask.p, c->d_raw.p, c->L, c->P.minq, tr, pt0, pt1);
  }
  c->have_depth = true;
  return RSIGPU_OK;
}

int rsigpu_pileup_end(rsigpu_ctx* c) {
  if (!c) return RSIGPU_E_ARG;
  if (!c->have_ref) { c->fail("pileup_end: call set_reference / pileup_begin first"); return RSIGPU_E_ARG; }
  int rc = run_pileup(c);
  if (rc) return rc;
  int h[2] = {0, 0};
  CK(cudaMemcpyAsync(h, c->d_misc.p + 5, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (h[1]) { c->fail("read batch is not sorted by position"); return RSIGPU_E_ARG; }
  c->have_reads = true; c->loaded = false; c->detected = false; c->filtered = false;
  c->pileup_fresh = true;
  return RSIGPU_OK;
}

int rsigpu_pileup_commit(rsigpu_ctx* c) {
  if (!c) return RSIGPU_E_ARG;
  if (!c->have_ref) { c->fail("pileup_commit: call set_reference / pileup_begin first"); return RSIGPU_E_ARG; }
  c->have_reads = true; c->have_depth = false; c->loaded = false; c->detected = false; c->filtered = false;
  return RSIGPU_OK;
}

int rsigpu_pileup_sort(rsigpu_ctx* c) {
  if (!c) return RSIGPU_E_ARG;
  if (!c->have_ref) { c->fail("pileup_sort: call set_reference and pileup_begin (or reads_begin) first"); return RSIGPU_E_ARG; }
  const size_t n = c->r_pos.n;
  if (n < 2) return RSIGPU_OK;
  if (n > 0x7fffffffull) { c->fail("pileup_sort: more than 2^31 - 1 staged reads"); return RSIGPU_E_RANGE; }
  cudaSetDevice(c->device);
  // the check the pileup runs anyway (k_read_ends' sorted_bad): reads already in position order cost nothing more
  CK(c->r_calend.ensure(n + 8)); CK(c->r_ncig.ensure(n + 8));
  int* mx = c->d_misc.p + 5;   // max_extent, sorted_bad
  if (c->isize_pending) { CK(cudaStreamWaitEvent(c->stream, c->ev_isize, 0)); c->isize_pending = false; }
  CK(cudaMemsetAsync(mx, 0, 8, c->stream));
  KL(k_read_ends, grid_for((int)std::min<size_t>(n, 1u << 30), 256, c->n_sm * 16), 256, 0, read_view(c), mx, mx + 1);
  int bad = 0;
  CK(cudaMemcpyAsync(&bad, mx + 1, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (!bad) return RSIGPU_OK;
  // keys pos + 1; the passes cover the bits of the largest key
  CK(c->t_key.ensure(n)); CK(c->t_dtot.ensure(SRT_RADIX + 1));
  u32* kmax = c->t_dtot.p + SRT_RADIX;
  CK(cudaMemsetAsync(kmax, 0, 4, c->stream));
  const int g = grid_for((int)n, 1024, c->n_sm * 8);
  KL(k_sort_key_pos, g, 256, 0, c->r_pos.p, (u32)n, c->t_key.p, kmax);
  u32 hk = 0;
  CK(cudaMemcpyAsync(&hk, kmax, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  const u32* perm = nullptr;
  int rc = sort_keys(c, (u32)n, bit_width(hk), &perm);
  if (rc) return rc;
  // gather into fresh arrays, which then replace the staged ones
  DevVec<int> pos, mpos, isize, mtid; DevVec<u16> flag; DevVec<u8> mapq, qual; DevVec<u32> coff, cig; DevVec<u64> qoff;
  auto drop = [&]() { pos.release(); mpos.release(); isize.release(); mtid.release(); flag.release(); mapq.release(); qual.release(); coff.release(); cig.release(); qoff.release(); };
  cudaError_t e = pos.alloc_exact(n);
  if (e == cudaSuccess) e = mpos.alloc_exact(n);
  if (e == cudaSuccess) e = isize.alloc_exact(n);
  if (e == cudaSuccess) e = mtid.alloc_exact(n);
  if (e == cudaSuccess) e = flag.alloc_exact(n);
  if (e == cudaSuccess) e = mapq.alloc_exact(n);
  if (e == cudaSuccess) e = coff.alloc_exact(n + 1);
  if (e == cudaSuccess) e = qoff.alloc_exact(n + 1);
  if (e == cudaSuccess) e = cig.alloc_exact(c->r_cigar.n);
  if (e == cudaSuccess) e = qual.alloc_exact(c->r_qual.n);
  if (e != cudaSuccess) { drop(); c->fail(std::string("pileup_sort: no device memory for the sorted copy of the reads: ") + cudaGetErrorString(e)); return RSIGPU_E_CUDA; }
  SortFields fi{nullptr, nullptr, c->r_pos.p, c->r_mpos.p, c->r_isize.p, c->r_mtid.p, c->r_flag.p, c->r_mapq.p, c->r_cigar_off.p, c->r_qual_off.p};
  SortFields fo{nullptr, nullptr, pos.p, mpos.p, isize.p, mtid.p, flag.p, mapq.p, coff.p, qoff.p};
  KL(k_sort_gather, g, 256, 0, perm, (u32)n, fi, fo);
  if ((rc = lengths_to_offsets(c, coff.p, qoff.p, (u32)n))) { drop(); return rc; }
  KL(k_sort_gather_payload, c->n_sm * 8, 256, 0, perm, (u32)n, c->r_cigar_off.p, c->r_cigar.p, c->r_qual_off.p, c->r_qual.p, coff.p, cig.p, qoff.p, qual.p);
  e = cudaStreamSynchronize(c->stream);
  if (e != cudaSuccess || !c->launch_err.empty()) {
    drop();
    c->fail("pileup_sort: " + (e != cudaSuccess ? std::string(cudaGetErrorString(e)) : "kernel launch failed: " + c->launch_err));
    c->launch_err.clear();
    return RSIGPU_E_CUDA;
  }
  std::swap(c->r_pos, pos); std::swap(c->r_mpos, mpos); std::swap(c->r_isize, isize); std::swap(c->r_mtid, mtid); std::swap(c->r_flag, flag);
  std::swap(c->r_mapq, mapq); std::swap(c->r_cigar_off, coff); std::swap(c->r_qual_off, qoff); std::swap(c->r_cigar, cig); std::swap(c->r_qual, qual);
  drop();   // the unsorted arrays
  // the sort scratch (16 B per read and the digit counts) is not kept: a context holds one contig's reads at a time
  c->t_key.release(); c->t_key2.release(); c->t_idx.release(); c->t_idx2.release(); c->t_hist.release(); c->t_ts.release();
  c->pileup_fresh = false;
  return RSIGPU_OK;
}

int rsigpu_reads_take(rsigpu_ctx* src, int64_t r0, int64_t r1, rsigpu_ctx* dst) {
  if (!src || !dst) return RSIGPU_E_ARG;
  rsigpu_ctx* c = src;
  if (src == dst) { c->fail("reads_take: the source and the destination are the same context"); return RSIGPU_E_ARG; }
  if (r0 < 0 || r1 < r0 || (size_t)r1 > c->r_pos.n) {
    c->fail("reads_take: reads [" + std::to_string(r0) + ", " + std::to_string(r1) + ") outside the " + std::to_string(c->r_pos.n) + " staged reads");
    return RSIGPU_E_ARG;
  }
  if (!dst->have_ref) { dst->fail("reads_take: call set_reference and pileup_begin (or reads_begin) on the destination first"); return RSIGPU_E_ARG; }
  if (r1 == r0) return RSIGPU_OK;
  cudaSetDevice(c->device);
  u32 co[2]; u64 qo[2];
  CK(cudaMemcpyAsync(&co[0], c->r_cigar_off.p + r0, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&co[1], c->r_cigar_off.p + r1, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&qo[0], c->r_qual_off.p + r0, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&qo[1], c->r_qual_off.p + r1, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  rsigpu_read_batch b; memset(&b, 0, sizeof b);
  b.n_reads = r1 - r0; b.tid = c->tid;
  b.pos = c->r_pos.p + r0; b.mpos = c->r_mpos.p + r0; b.isize = c->r_isize.p + r0; b.mtid = c->r_mtid.p + r0; b.flag = c->r_flag.p + r0; b.mapq = c->r_mapq.p + r0;
  b.cigar_off = c->r_cigar_off.p + r0; b.cigar = c->r_cigar.p + co[0]; b.qual_off = reinterpret_cast<const uint64_t*>(c->r_qual_off.p + r0); b.qual = c->r_qual.p + qo[0];
  return push_impl(dst, &b, (size_t)(co[1] - co[0]), (size_t)(qo[1] - qo[0]), co[0], qo[0], c->device);
}

int rsigpu_reads_field(rsigpu_ctx* c, int32_t field, void* out, int64_t cap_bytes, int64_t* nbytes) {
  if (!c || !nbytes) return RSIGPU_E_ARG;
  cudaSetDevice(c->device);
  const size_t n = c->r_pos.n;
  const void* src = nullptr; size_t bytes = 0;
  switch (field) {
    case 0: src = c->r_pos.p; bytes = n * 4; break;
    case 1: src = c->r_mpos.p; bytes = n * 4; break;
    case 2: src = c->r_isize.p; bytes = n * 4; break;
    case 3: src = c->r_mtid.p; bytes = n * 4; break;
    case 4: src = c->r_flag.p; bytes = n * 2; break;
    case 5: src = c->r_mapq.p; bytes = n; break;
    case 6: src = c->r_cigar_off.p; bytes = (n + 1) * 4; break;
    case 7: src = c->r_cigar.p; bytes = c->r_cigar.n * 4; break;
    case 8: src = c->r_qual_off.p; bytes = (n + 1) * 8; break;
    case 9: src = c->r_qual.p; bytes = c->r_qual.n; break;
    default: return RSIGPU_E_ARG;
  }
  *nbytes = (int64_t)bytes;
  if (!out || cap_bytes < (int64_t)bytes) return RSIGPU_OK;
  if (n == 0 && (field == 6 || field == 8)) { memset(out, 0, bytes); return RSIGPU_OK; }   // nothing staged: the one offset is 0
  if (bytes) { CK(cudaMemcpyAsync(out, src, bytes, cudaMemcpyDeviceToHost, c->stream)); CK(cudaStreamSynchronize(c->stream)); }
  return RSIGPU_OK;
}

// a7 + a8 + a9 + chromosome statistics + bin arrays (median_transfer, negative_binomial_transfer), in phases: the per-base
// passes take a range so that one contig can be spread over several GPUs (rsigpu_split_run); rsigpu_load_finish is all
// phases over the whole contig on one context.
static int lf_prepare(rsigpu_ctx* c) {
  const int L = c->L, nb = c->nb, nn = (int)c->h_nbeg.size(), m = c->P.m;
  CK(c->d_rdc.ensure((size_t)c->Lc + 64));
  CK(c->d_bin_med.ensure(nb + 8)); CK(c->d_bin_nbn.ensure(nb + 8)); CK(c->d_bin_medint.ensure(nb + 8)); CK(c->d_bin_sum.ensure(nb + 8));
  CK(c->d_status.ensure(nb + 8)); CK(c->d_status1.ensure(nb + 8)); CK(c->d_nz_idx.ensure(nb + 8)); CK(c->d_nz_val.ensure(nb + 8)); CK(c->d_tile.ensure(nb / 1024 + 8));
  CK(c->d_scan_scratch.ensure((size_t)((nb + S_T - 1) / S_T) * 10 * S_NB + 64)); CK(c->d_minl_del.ensure(nb + 8)); CK(c->d_minl_dup.ensure(nb + 8)); CK(c->d_pfx.ensure((size_t)nb + LIST_CAP + 8));
  DevState* h = c->h_st;
  memset(h, 0, sizeof(DevState));
  h->L = L; h->Lc = c->Lc; h->nb = nb; h->m = m; h->n_noseq = nn; h->gc_on = c->P.gcadjust ? 1 : 0; h->cap_on = c->P.cap > 1 ? 1 : 0;
  h->gc_base = c->gc_base;
  h->trans = c->P.trans; h->cap = c->P.cap; h->rd_min = 0x7fffffff; h->rd_max = -0x7fffffff - 1;
  h->nb_tmin_ord = 0xffffffffu;
  h->factor = sqrt(2.0 * (1.0 + c->P.epsilon) * log(3.1E9));   // rsi.cpp:1829
  h->Lmax_base = std::max(10000 / m, 20);                        // rsi.cpp:1831
  h->isize_mean = -1; h->isize_sd = -1;
  CK(cudaEventRecord(c->ev[1], c->stream));
  CK(cudaMemcpyAsync(c->d_st, h, sizeof(DevState), cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemsetAsync(c->d_hist_all.p, 0, (size_t)HIST_ALL_BINS * 4, c->stream));
  CK(cudaMemsetAsync(c->d_chist.p, 0, (size_t)MAD_CLASSES * CHIST_RCAP * 4, c->stream));
  CK(cudaMemsetAsync(c->d_thist.p, 0, (size_t)CHIST_RCAP * 4, c->stream));
  CK(cudaMemsetAsync(c->d_misc.p, 0, 5 * 4, c->stream));
  return RSIGPU_OK;
}
static int lf_candidate_scratch(rsigpu_ctx* c) {   // what only the context that runs the candidate stage needs
  CK(c->d_ref.ensure((size_t)c->Lc + 64)); CK(c->d_pref.ensure((size_t)c->Lc + 64)); CK(c->d_rm.ensure((size_t)c->Lc + 64));
  CK(c->d_spec_ref.ensure(2 * (size_t)c->Lc + 128)); CK(c->d_spec_pref.ensure(2 * (size_t)c->Lc + LIST_CAP + 128)); CK(c->d_spec_rm.ensure(2 * (size_t)c->Lc + 128));
  CK(c->d_spec_off.ensure(LIST_CAP + 8));
  return RSIGPU_OK;
}
static int lf_pass_a(rsigpu_ctx* c, int wt0, int wt1) {
  const int nw = std::min((c->L + W_T - 1) / W_T, wt1) - wt0;
  if (nw > 0) KL(k_gc_table, std::min((nw + A_NW - 1) / A_NW, c->n_sm), A_NT, RSI_SMEM_A, c->d_raw.p, c->d_fasta.p, c->d_st, wt0, wt1);
  return RSIGPU_OK;
}
static int lf_finalize_a(rsigpu_ctx* c) { KL(k_gc_finalize, 1, 256, 0, c->d_fasta.p, c->d_st); return RSIGPU_OK; }
static int lf_pass_b(rsigpu_ctx* c, int wt0, int wt1) {
  const int nn = (int)c->h_nbeg.size();
  const int* nbeg = c->d_nseq.p; const int* nend = nbeg + nn; const int* ncum = nbeg + 2 * nn;
  const int nw = std::min((c->L + W_T - 1) / W_T, wt1) - wt0;
  if (nw > 0) KL(k_gc_adjust, std::min((nw + B_NW - 1) / B_NW, c->n_sm), B_NT, RSI_SMEM_B, c->d_raw.p, c->d_fasta.p, c->d_rdc.p, nbeg, nend, ncum, c->d_hist_all.p, c->d_st, wt0, wt1);
  return RSIGPU_OK;
}
static int lf_cap(rsigpu_ctx* c) { KL(k_cap_params, 1, 1024, 0, c->d_hist_all.p, c->d_st, CHIST_RCAP); return RSIGPU_OK; }
// pass C works on tiles of `unit` bins (lf_c_unit); the pseudo-tile after the last bin tile owns the bases beyond nb * m
static int lf_c_unit(const rsigpu_ctx* c) { return c->P.m <= 127 ? (int)CW_BINS : std::max(1, std::min((int)C_BINS, (C_CAP - 4) / c->P.m)); }
static int lf_c_tiles(const rsigpu_ctx* c) { const int u = lf_c_unit(c); return (c->nb + u - 1) / u + 1; }
static int lf_pass_c(rsigpu_ctx* c, int t0, int t1) {
  const int m = c->P.m, unit = lf_c_unit(c);
  const int nt = std::min(lf_c_tiles(c), t1) - t0;
  if (nt <= 0) return RSIGPU_OK;
  if (m <= 127) {   // every warp its own pipeline: warp-tiles of CW_BINS bins
#define RSI_BINS_WARP(M)                                                                                                                     \
  KL(k_bins_warp<M>, std::min((nt + cw_nw(M) - 1) / cw_nw(M), c->n_sm), cw_nw(M) * 32, cw_nw(M) * cw_warp_bytes(M), c->d_rdc.p, c->d_bin_med.p, \
     c->d_bin_medint.p, c->d_bin_sum.p, c->d_chist.p, c->d_thist.p, c->d_st, t0, t1)
    if (m == 101) RSI_BINS_WARP(101);
    else if (m == 51) RSI_BINS_WARP(51);
    else RSI_BINS_WARP(0);
#undef RSI_BINS_WARP
  } else {
    KL(k_bins, std::min(nt, c->n_sm), C_NT, RSI_SMEM_C, c->d_rdc.p, c->d_bin_med.p, c->d_bin_medint.p, c->d_bin_sum.p, c->d_chist.p,
       c->d_thist.p, c->d_st, unit, t0, t1);
  }
  return RSIGPU_OK;
}
static int lf_finish(rsigpu_ctx* c) {
  DevState* h = c->h_st;
  const int nb = c->nb, m = c->P.m;
  KL(k_chr_stats, 1, 1024, 0, c->d_chist.p, c->d_thist.p, c->d_tothist.p, c->d_st);
  CK(cudaMemcpyAsync(h, c->d_st, sizeof(DevState), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (c->have_reads && !c->use_summary) {
    int sb = 0;
    CK(cudaMemcpyAsync(&sb, c->d_misc.p + 6, 4, cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (sb) { c->fail("read batch is not sorted by position"); return RSIGPU_E_ARG; }
  }
  const bool low_depth = h->rdmedian < 5;   // "Read depths too low": detectcnv returns without calls (rsi.cpp:1809-1812)
  if (low_depth) h->err &= ~ERR_DEGENERATE;
  if (h->err) return map_dev_err(c, h->err, h->cand_err);
  if (low_depth) {
    CK(cudaEventRecord(c->ev[2], c->stream));
    c->loaded = true; c->detected = false; c->filtered = false;
    return RSIGPU_OK;
  }
  // negative_binomial_transfer's table over the bin sums, with the host's libm (rsi.cpp:1142-1163)
  const double rdmedian = h->rdmedian, r = rdmedian / h->rdmad;
  const size_t lut_n = (size_t)h->max_binsum + 1;
  if (lut_n > LUT_CAP) { c->fail("bin sums above 2^24: depth too high for the transform table"); return RSIGPU_E_RANGE; }
  if (lut_n > c->h_lut_cap) {
    if (c->h_lut) cudaFreeHost(c->h_lut);
    c->h_lut = nullptr; c->h_lut_cap = 0;
    CK(cudaMallocHost((void**)&c->h_lut, lut_n * 2 * sizeof(float)));
    c->h_lut_cap = lut_n * 2;
  }
  CK(c->d_lut.ensure(lut_n + 8));
  for (size_t s = 0; s < lut_n; ++s) c->h_lut[s] = (float)nb_formula((double)s, (double)m, r);
  double anchors[3];
  anchors[0] = nb_formula(rdmedian * m, (double)m, r);
  anchors[1] = nb_formula(rdmedian / 2.0 * (double)m, (double)m, r);
  anchors[2] = nb_formula(rdmedian * 1.5 * (double)m, (double)m, r);
  h->med_nbt_raw = anchors[0]; h->del_nbt_raw = anchors[1]; h->dup_nbt_raw = anchors[2];
  CK(cudaMemcpyAsync(c->d_lut.p, c->h_lut, lut_n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  CK(cudaMemcpyAsync(field_ptr(c->d_st, &DevState::med_nbt_raw), &h->med_nbt_raw, 3 * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  const int gb = grid_for(nb, 1024, c->n_sm * 8);
  KL(k_nb_gather, gb, 256, 0, c->d_bin_sum.p, c->d_lut.p, (int)lut_n, c->d_bin_nbn.p, c->d_st);
  KL(k_nb_scale, gb, 256, 0, c->d_bin_nbn.p, c->d_st);
  CK(cudaEventRecord(c->ev[2], c->stream));
  c->loaded = true; c->detected = false; c->filtered = false;
  return RSIGPU_OK;
}

int rsigpu_load_finish(rsigpu_ctx* c) {
  if (!c) return RSIGPU_E_ARG;
  if (c->have_ref && c->have_reads && !c->have_depth) { int rc = run_pileup(c); if (rc) return rc; }
  if (!c->have_ref || !c->have_depth) { c->fail("load_finish: no reference or depth staged"); return RSIGPU_E_ARG; }
  cudaSetDevice(c->device);
  int rc;
  if ((rc = lf_prepare(c)) || (rc = lf_candidate_scratch(c))) return rc;
  if ((rc = lf_pass_a(c, 0, 0x7fffffff)) || (rc = lf_finalize_a(c)) || (rc = lf_pass_b(c, 0, 0x7fffffff)) || (rc = lf_cap(c)) || (rc = lf_pass_c(c, 0, 0x7fffffff))) return rc;
  return lf_finish(c);
}

// detectcnv (rsi.cpp:1795-1945) incl. the list that sd_filters would keep
int rsigpu_detectcnv(rsigpu_ctx* c) {
  if (!c) return RSIGPU_E_ARG;
  if (!c->loaded) { c->fail("detectcnv: call load_finish first"); return RSIGPU_E_ARG; }
  cudaSetDevice(c->device);
  DevState* h = c->h_st;
  c->h_detected.clear(); c->h_calls.clear();
  for (int k = 0; k < 4; ++k) c->h_dump[k].clear();
  if (h->rdmedian < 5) {   // "Read depths too low", rsi.cpp:1809-1812
    CK(cudaEventRecord(c->ev[3], c->stream)); CK(cudaEventRecord(c->ev[4], c->stream));
    c->detected = true;
    return RSIGPU_OK;
  }
  const int nn = (int)c->h_nbeg.size();
  CandArgs A;
  A.all_phase = 0; A.saved = c->list(10); A.n_saved = c->d_misc.p + 14;
  const bool all = c->P.trans == RSIGPU_TRANS_ALL;
  const int which = c->P.trans == RSIGPU_TRANS_NBN ? 0 : 1;      // MED first for -MED and -ALL (rsi.cpp:1837-1840)
  int rc = run_rsi(c, which, which ? c->d_bin_med.p : c->d_bin_nbn.p);
  if (rc) return rc;
  if (!all) CK(cudaEventRecord(c->ev[3], c->stream));
  A.rdc = c->d_rdc.p; A.medint = c->d_bin_medint.p; A.status = c->d_status.p; A.nbeg = c->d_nseq.p; A.nend = c->d_nseq.p + nn;
  A.segs = c->list(0); A.tmp = c->list(1); A.ov = c->list(2);
  A.d_segments = c->list(3); A.d_blocks = c->list(4); A.d_premerge = c->list(5); A.d_merged = c->list(6); A.d_detected = c->list(7); A.d_calls = c->list(8);
  A.n_dump = c->d_misc.p; A.list_cap = LIST_CAP;
  A.S.ref = c->d_ref.p; A.S.ref_cap = (int)std::min<size_t>(c->d_ref.cap, 0x7fffffff); A.S.sub = c->d_sub.p; A.S.sub_cap = c->P.maxchkbp * 10 + 64;   // slice 0; the per-call cluster kernels use slice 1 + cluster id
  A.S.pref = c->d_pref.p; A.S.rm = c->d_rm.p; A.S.hist = c->d_chist_c.p; A.S.hist_cap = (int)c->d_chist_c.cap; A.S.err = c->d_misc.p + 4; A.S.prof = c->profile ? c->d_cprof.p : nullptr;
  if (c->profile) CK(cudaMemsetAsync(c->d_cprof.p, 0, 16 * 8, c->stream));
  A.maxchkbp = c->P.maxchkbp; A.merge = c->P.merge; A.tid = c->tid; A.chklen = c->P.chklen;
  CandSpec X;
  X.off = c->d_spec_off.p; X.res = c->list(9); X.on = c->d_misc.p + 12; X.nl = c->d_misc.p + 13;
  X.cap = (long long)c->d_spec_ref.cap - 64; X.ref = c->d_spec_ref.p; X.pref = c->d_spec_pref.p; X.rm = c->d_spec_rm.p;
  CK(cudaMemsetAsync(c->d_misc.p + 12, 0, 8, c->stream));
  if (all) {   // -ALL: MED segments are tested and parked, then the NBN pass is run and its segments appended
    A.all_phase = 1;
    KL(k_cand_a, 1, c->cand_a_threads, RSI_SMEM_CAND_A, A, X, c->d_st);
    if ((rc = run_rsi(c, 0, c->d_bin_nbn.p)) != RSIGPU_OK) return rc;
    CK(cudaEventRecord(c->ev[3], c->stream));
    A.all_phase = 2;
  }
  KL(k_cand_a, 1, c->cand_a_threads, RSI_SMEM_CAND_A, A, X, c->d_st);   // bin-level arrays are tiny: fewer threads = cheaper barriers
  ClusterArgs G; G.gx = reinterpret_cast<unsigned char*>(c->d_clx.p); G.gbc = c->d_clbc.p; G.ghist = c->d_clhist.p;
  const int ncl = std::max(1, std::min(c->n_sm / CAND_CL, 32));
  KLC(k_cand_edge, ncl * CAND_CL, CAND_CL_NT, CAND_CL, RSI_SMEM_CAND_CL, A, X, G, c->d_st);
  KL(k_cand_b, 1, 1024, (size_t)CAND_SHIST * 4, A, X, c->d_st);
  KLC(k_cand_final, ncl * CAND_CL, CAND_CL_NT, CAND_CL, RSI_SMEM_CAND_CL, A, X, G, c->d_st);
  KL(k_cand_c, 1, 1024, (size_t)CAND_SHIST * 4, A, X, c->d_st);
  CK(cudaEventRecord(c->ev[4], c->stream));
  CK(cudaMemcpyAsync(h, c->d_st, sizeof(DevState), cudaMemcpyDeviceToHost, c->stream));
  int nd[4];
  CK(cudaMemcpyAsync(nd, c->d_misc.p, 16, cudaMemcpyDeviceToHost, c->stream));
  if (c->profile) CK(cudaMemcpyAsync(c->h_cprof, c->d_cprof.p, 16 * 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (h->err) return map_dev_err(c, h->err, h->cand_err);
  c->h_detected.resize(h->n_detected); c->h_calls.resize(h->n_calls);
  if (h->n_detected) CK(cudaMemcpyAsync(c->h_detected.data(), c->list(7), sizeof(Cnv) * h->n_detected, cudaMemcpyDeviceToHost, c->stream));
  if (h->n_calls) CK(cudaMemcpyAsync(c->h_calls.data(), c->list(8), sizeof(Cnv) * h->n_calls, cudaMemcpyDeviceToHost, c->stream));
  for (int k = 0; k < 4; ++k) {
    const int n = std::min(nd[k], LIST_CAP);
    c->h_dump[k].resize(n);
    if (n) CK(cudaMemcpyAsync(c->h_dump[k].data(), c->list(3 + k), sizeof(Cnv) * n, cudaMemcpyDeviceToHost, c->stream));
  }
  CK(cudaStreamSynchronize(c->stream));
  c->detected = true; c->filtered = false;
  return RSIGPU_OK;
}

int rsigpu_sd_filters(rsigpu_ctx* c) {
  if (!c) return RSIGPU_E_ARG;
  if (!c->detected) { c->fail("sd_filters: call detectcnv first"); return RSIGPU_E_ARG; }
  c->filtered = true;   // k_candidates already produced the filtered list next to the unfiltered one
  return RSIGPU_OK;
}

// a26 + a27 on the read summaries kept by pileup_push
int rsigpu_cnv_stat(rsigpu_ctx* c) {
  if (!c) return RSIGPU_E_ARG;
  if (!c->detected) { c->fail("cnv_stat: call detectcnv first"); return RSIGPU_E_ARG; }
  if (!c->have_reads) { c->fail("cnv_stat: BAM input only (pairrd.cpp:622)"); return RSIGPU_E_ARG; }
  cudaSetDevice(c->device);
  std::vector<Cnv>& v = c->filtered ? c->h_calls : c->h_detected;
  Cnv* d = c->filtered ? c->list(8) : c->list(7);
  if (v.empty() || (c->use_summary ? c->s_n : c->r_pos.n) == 0) return RSIGPU_OK;
  ReadSoA R = read_view(c);
  int* mx = c->d_misc.p + 5;
  if (c->isize_pending) { CK(cudaStreamWaitEvent(c->stream, c->ev_isize, 0)); c->isize_pending = false; }
  KL(k_cnv_stat, std::min((int)v.size(), c->n_sm * 2), 1024, 0, R, d, (int)v.size(), mx, c->d_misc.p + 16);
  CK(cudaMemcpyAsync(v.data(), d, sizeof(Cnv) * v.size(), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&c->h_st->isize_mean, c->d_misc.p + 16, 8, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return RSIGPU_OK;
}

// `stat`: reads of one contig without a reference, then RP / Q0 for calls from a file
int rsigpu_reads_begin(rsigpu_ctx* c, int32_t tid, int32_t target_len) {
  if (!c || target_len < 1) return RSIGPU_E_ARG;
  c->L = target_len; c->tid = tid;
  c->have_ref = true;           // staging reads needs only the contig's length and id
  c->have_depth = false; c->have_reads = false; c->loaded = false; c->detected = false; c->filtered = false;
  return rsigpu_pileup_begin(c, target_len);
}

int rsigpu_stat_calls(rsigpu_ctx* c, rsigpu_cnv* list, int32_t n) {
  if (!c || !list || n < 0) return RSIGPU_E_ARG;
  if (n == 0 || c->r_pos.n == 0) return RSIGPU_OK;
  if (n > LIST_CAP * 8) { c->fail("stat_calls: more than 524288 calls"); return RSIGPU_E_RANGE; }
  cudaSetDevice(c->device);
  CK(c->r_calend.ensure(c->r_pos.n + 8)); CK(c->r_ncig.ensure(c->r_pos.n + 8));
  ReadSoA R = read_view(c);
  int* mx = c->d_misc.p + 5;
  if (c->isize_pending) { CK(cudaStreamWaitEvent(c->stream, c->ev_isize, 0)); c->isize_pending = false; }
  CK(cudaMemsetAsync(mx, 0, 8, c->stream));
  KL(k_read_ends, grid_for((int)std::min<size_t>(c->r_pos.n, 1u << 30), 256, c->n_sm * 16), 256, 0, R, mx, mx + 1);
  KL(k_isize_stats, 1, 1024, 0, R, c->L, mx, c->d_misc.p + 16);
  Cnv* d = c->list(0);          // lists 0..7 are contiguous: room for 8 * LIST_CAP entries
  CK(cudaMemcpyAsync(d, list, sizeof(Cnv) * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  KL(k_cnv_stat, std::min((int)n, c->n_sm * 2), 1024, 0, R, d, (int)n, mx, c->d_misc.p + 16);
  std::vector<Cnv> out((size_t)n);
  int sb = 0;
  CK(cudaMemcpyAsync(out.data(), d, sizeof(Cnv) * (size_t)n, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(&sb, mx + 1, 4, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (sb) { c->fail("read batch is not sorted by position"); return RSIGPU_E_ARG; }
  for (int32_t k = 0; k < n; ++k) if (list[k].tid == c->tid) { list[k].rp = out[(size_t)k].rp; list[k].q0 = out[(size_t)k].q0; }
  return RSIGPU_OK;
}

int rsigpu_get_calls(rsigpu_ctx* c, rsigpu_cnv* out, int32_t cap, int32_t* n) {
  if (!c || !n) return RSIGPU_E_ARG;
  if (!c->detected) { c->fail("get_calls: call detectcnv first"); return RSIGPU_E_ARG; }
  const std::vector<Cnv>& v = c->filtered ? c->h_calls : c->h_detected;
  *n = (int32_t)v.size();
  if ((int)v.size() > cap) return RSIGPU_E_CAPACITY;
  if (out && !v.empty()) memcpy(out, v.data(), sizeof(Cnv) * v.size());
  return RSIGPU_OK;
}

int rsigpu_run(rsigpu_ctx* c, rsigpu_cnv* out, int32_t cap, int32_t* n) {
  if (!c) return RSIGPU_E_ARG;
  cudaSetDevice(c->device);
  int rc;
  TRACE(c, "run: start");
  CK(cudaEventRecord(c->ev[0], c->stream));
  // BAM input: the pileup is the first stage of the path (already done when rsigpu_pileup_end has just run it, the -s path)
  if (c->have_reads && !(c->pileup_fresh && c->have_depth) && (rc = run_pileup(c)) != RSIGPU_OK) return rc;
  c->pileup_fresh = false;
  if ((rc = rsigpu_load_finish(c)) != RSIGPU_OK) return rc;
  if ((rc = rsigpu_detectcnv(c)) != RSIGPU_OK) return rc;
  if ((rc = rsigpu_sd_filters(c)) != RSIGPU_OK) return rc;
  if (c->have_reads && (rc = rsigpu_cnv_stat(c)) != RSIGPU_OK) return rc;
  CK(cudaEventRecord(c->ev[5], c->stream));
  CK(cudaStreamSynchronize(c->stream));
  TRACE(c, "run: end");
  float ms = 0;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]); c->stage_ms[0] = ms;
  cudaEventElapsedTime(&ms, c->ev[1], c->ev[2]); c->stage_ms[1] = ms;
  cudaEventElapsedTime(&ms, c->ev[2], c->ev[3]); c->stage_ms[2] = ms;
  cudaEventElapsedTime(&ms, c->ev[3], c->ev[4]); c->stage_ms[3] = ms;
  cudaEventElapsedTime(&ms, c->ev[4], c->ev[5]); c->stage_ms[4] = ms;
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[5]); c->stage_ms[5] = ms;
  return rsigpu_get_calls(c, out, cap, n);
}

// ---------------------------------------------------------------------------------------------
// One contig over several GPUs (north_star: "chromosomes larger than one shard are split with halo exchange ... over NVLink
// P2P").  Every part context holds the whole FASTA and full-length arrays but STAGES only the reads (or uses only the depth)
// of its own base range, and runs the per-base work -- pileup, passes A, B, C -- on that range.  What the passes accumulate
// is integer (sums and counts per GC stratum, the value histograms, bin sums): the parts' partial tables are copied to the
// lead over peer-to-peer and added there, which is exact, the lead derives the few scalars (stratum table, cap, medians) and
// sends the state back.  Halo: pass C works on whole bins of the N-compacted array, so a part needs the first few hundred
// compacted values of its right neighbour (the bins that straddle the cut).  After pass C the lead gathers the compacted
// depth, the bin arrays and the read summaries and runs the bin-level and candidate stages exactly as for an unsplit contig:
// the result is bit-identical.  Cuts are multiples of 57344 bases (whole pileup tiles and whole warp-tiles).
enum { SPLIT_ALIGN = 57344, SPLIT_HALO = 65536 };
static_assert(SPLIT_ALIGN % PU_T == 0, "a split part starts on a pileup tile");
static int split_point(int L, int n, int g) {
  if (g <= 0) return 0;
  if (g >= n) return L;
  const long long s = ((long long)L * g / n + SPLIT_ALIGN / 2) / SPLIT_ALIGN * SPLIT_ALIGN;
  return (int)std::min<long long>(s, (long long)L);
}
int rsigpu_split_range(int32_t L, int32_t n_parts, int32_t part, int32_t* beg, int32_t* end, int32_t* read_halo) {
  if (n_parts < 1 || part < 0 || part >= n_parts || L < 1 || !beg || !end) return RSIGPU_E_ARG;
  if ((long long)L < 2ll * SPLIT_ALIGN * n_parts) return RSIGPU_E_RANGE;
  *beg = split_point(L, n_parts, part); *end = split_point(L, n_parts, part + 1);
  if (read_halo) *read_halo = SPLIT_HALO;
  return RSIGPU_OK;
}

namespace {
// `dst`'s stream waits for everything queued so far on `src`'s stream (the two may sit on different devices)
int split_dep(rsigpu_ctx* src, rsigpu_ctx* dst) {
  rsigpu_ctx* c = src;
  cudaSetDevice(src->device);
  CK(cudaEventRecord(src->ev_part, src->stream));
  cudaSetDevice(dst->device);
  CK(cudaStreamWaitEvent(dst->stream, src->ev_part, 0));
  return RSIGPU_OK;
}
int split_copy(rsigpu_ctx* lead, rsigpu_ctx* dst, void* d, rsigpu_ctx* src, const void* s_, size_t bytes) {
  rsigpu_ctx* c = dst;
  if (!bytes) return RSIGPU_OK;
  cudaSetDevice(dst->device);
  CK(cudaMemcpyPeerAsync(d, dst->device, s_, src->device, bytes, dst->stream));
  if (dst->device != src->device) lead->split_p2p_bytes += (long long)bytes;
  return RSIGPU_OK;
}
// lead += the parts' DevState fields of `phase`, then every part gets the lead's state
int split_reduce_state(rsigpu_ctx** parts, int n, int phase, bool finalize_a, bool cap) {
  rsigpu_ctx* lead = parts[0]; rsigpu_ctx* c = lead;
  int rc;
  for (int g = 1; g < n; ++g) {
    if ((rc = split_dep(parts[g], lead))) return rc;
    if ((rc = split_copy(lead, lead, lead->d_part_st.p + (g - 1), parts[g], parts[g]->d_st, sizeof(DevState)))) return rc;
  }
  cudaSetDevice(lead->device);
  KL(k_split_reduce_state, 1, 256, 0, lead->d_st, lead->d_part_st.p, n - 1, phase);
  if (finalize_a && (rc = lf_finalize_a(lead))) return rc;
  if (cap && (rc = lf_cap(lead))) return rc;
  for (int g = 1; g < n; ++g) {
    if ((rc = split_dep(lead, parts[g]))) return rc;
    if ((rc = split_copy(lead, parts[g], parts[g]->d_st, lead, lead->d_st, sizeof(DevState)))) return rc;
  }
  return RSIGPU_OK;
}
int split_add_u32(rsigpu_ctx* lead, rsigpu_ctx* part, u32* dst, const u32* src, size_t n) {   // dst (lead) += src (part); the dependency is already in place
  rsigpu_ctx* c = lead;
  int rc;
  if ((rc = split_copy(lead, lead, lead->d_part_u32.p, part, src, n * 4))) return rc;
  cudaSetDevice(lead->device);
  KL(k_vec_add_u32, grid_for((int)n, 1024, lead->n_sm * 4), 256, 0, dst, lead->d_part_u32.p, n);
  return RSIGPU_OK;
}
long long compact_index(const rsigpu_ctx* c, int s) {   // number of non-N positions before s
  long long removed = 0;
  for (size_t k = 0; k < c->h_nbeg.size(); ++k) {
    if (c->h_nbeg[k] >= s) break;
    removed += (long long)std::min(c->h_nend[k], s - 1) - c->h_nbeg[k] + 1;
  }
  return (long long)s - removed;
}
}  // namespace

int rsigpu_split_run(rsigpu_ctx** parts, int32_t n, rsigpu_cnv* out, int32_t cap, int32_t* n_out) {
  if (!parts || n < 1 || !parts[0]) return RSIGPU_E_ARG;
  if (n == 1) return rsigpu_run(parts[0], out, cap, n_out);
  rsigpu_ctx* lead = parts[0]; rsigpu_ctx* c = lead;
  const int L = lead->L;
  for (int g = 0; g < n; ++g) {
    rsigpu_ctx* p = parts[g];
    if (!p || !p->have_ref || p->L != L || p->Lc != lead->Lc || p->P.m != lead->P.m) { lead->fail("split_run: every part needs the same reference and parameters"); return RSIGPU_E_ARG; }
    if (p->have_reads != lead->have_reads || (!p->have_reads && !p->have_depth)) { lead->fail("split_run: every part needs its reads (or the depth) staged"); return RSIGPU_E_ARG; }
    for (int q = 0; q < g; ++q) if (parts[q] == p) { lead->fail("split_run: a context appears twice"); return RSIGPU_E_ARG; }
  }
  if ((long long)L < 2ll * SPLIT_ALIGN * n) { lead->fail("split_run: contig too short for this many parts"); return RSIGPU_E_RANGE; }
  const bool reads = lead->have_reads;
  int rc;
  TRACE(lead, "split_run: start");
  // peer access (direct NVLink copies; without it the peer copies are staged through the host)
  for (int g = 0; g < n; ++g) for (int q = 0; q < n; ++q) if (parts[g]->device != parts[q]->device) {
    cudaSetDevice(parts[g]->device);
    int can = 0; cudaDeviceCanAccessPeer(&can, parts[g]->device, parts[q]->device);
    if (can) { cudaError_t e = cudaDeviceEnablePeerAccess(parts[q]->device, 0); if (e != cudaSuccess) cudaGetLastError(); }
  }
  cudaSetDevice(lead->device);
  lead->split_p2p_bytes = 0; lead->use_summary = false;
  CK(lead->d_part_st.ensure((size_t)n)); CK(lead->d_part_u32.ensure((size_t)MAD_CLASSES * CHIST_RCAP + 8));
  CK(cudaEventRecord(lead->ev[0], lead->stream));
  std::vector<int> cut((size_t)n + 1);
  for (int g = 0; g <= n; ++g) cut[(size_t)g] = split_point(L, n, g);
  // ---- pileup + pass A on every part's own range
  for (int g = 0; g < n; ++g) {
    rsigpu_ctx* p = parts[g]; c = p;
    cudaSetDevice(p->device);
    p->use_summary = false; p->pileup_fresh = false;
    if (reads && (rc = run_pileup(p, cut[(size_t)g] / PU_T, g + 1 < n ? cut[(size_t)g + 1] / PU_T : 0x7fffffff, false))) { if (p != lead) lead->fail(p->err); return rc; }
    if ((rc = lf_prepare(p)) || (rc = lf_pass_a(p, cut[(size_t)g] / W_T, g + 1 < n ? cut[(size_t)g + 1] / W_T : 0x7fffffff))) { if (p != lead) lead->fail(p->err); return rc; }
  }
  c = lead;
  if ((rc = split_reduce_state(parts, n, 0, true, false))) return rc;
  // ---- pass B
  for (int g = 0; g < n; ++g) {
    cudaSetDevice(parts[g]->device);
    if ((rc = lf_pass_b(parts[g], cut[(size_t)g] / W_T, g + 1 < n ? cut[(size_t)g + 1] / W_T : 0x7fffffff))) { if (parts[g] != lead) lead->fail(parts[g]->err); return rc; }
  }
  for (int g = 1; g < n; ++g) {
    if ((rc = split_dep(parts[g], lead))) return rc;
    if ((rc = split_add_u32(lead, parts[g], lead->d_hist_all.p, parts[g]->d_hist_all.p, (size_t)HIST_ALL_BINS))) return rc;
  }
  if ((rc = split_reduce_state(parts, n, 1, false, true))) return rc;
  // ---- pass C on whole tiles of bins; the bins that straddle a cut need the right neighbour's first compacted values
  const int unit = lf_c_unit(lead), ntile_c = lf_c_tiles(lead), m = lead->P.m;
  std::vector<int> ct((size_t)n + 1); std::vector<long long> cc((size_t)n + 1);
  for (int g = 0; g <= n; ++g) cc[(size_t)g] = g == n ? (long long)lead->Lc : compact_index(lead, cut[(size_t)g]);
  ct[0] = 0; ct[(size_t)n] = ntile_c;
  for (int g = 1; g < n; ++g) ct[(size_t)g] = (int)std::min<long long>((cc[(size_t)g] + (long long)unit * m - 1) / ((long long)unit * m), (long long)ntile_c - 1);
  for (int g = 0; g + 1 < n; ++g) {
    const long long a = cc[(size_t)g + 1], b = std::min<long long>((long long)ct[(size_t)g + 1] * unit * m, (long long)lead->Lc);
    if (b > cc[(size_t)g + 2]) { lead->fail("split_run: parts too small for the bin size"); return RSIGPU_E_RANGE; }
    if (b > a) {
      if ((rc = split_dep(parts[g + 1], parts[g]))) return rc;
      if ((rc = split_copy(lead, parts[g], parts[g]->d_rdc.p + a, parts[g + 1], parts[g + 1]->d_rdc.p + a, (size_t)(b - a) * 4))) return rc;
      // the neighbour must not start capping (pass C writes the capped values back) before its uncapped values have been copied
      if ((rc = split_dep(parts[g], parts[g + 1]))) return rc;
    }
  }
  for (int g = 0; g < n; ++g) {
    cudaSetDevice(parts[g]->device);
    if ((rc = lf_pass_c(parts[g], ct[(size_t)g], ct[(size_t)g + 1]))) { if (parts[g] != lead) lead->fail(parts[g]->err); return rc; }
  }
  // ---- gather on the lead: compacted depth, bin arrays, class histograms
  for (int g = 1; g < n; ++g) {
    rsigpu_ctx* p = parts[g];
    if ((rc = split_dep(p, lead))) return rc;
    const long long a = std::min<long long>((long long)ct[(size_t)g] * unit * m, (long long)lead->Lc), b = g + 1 < n ? std::min<long long>((long long)ct[(size_t)g + 1] * unit * m, (long long)lead->Lc) : (long long)lead->Lc;
    if ((rc = split_copy(lead, lead, lead->d_rdc.p + a, p, p->d_rdc.p + a, (size_t)std::max<long long>(b - a, 0) * 4))) return rc;
    const long long b0 = std::min<long long>((long long)ct[(size_t)g] * unit, (long long)lead->nb), b1 = std::min<long long>((long long)ct[(size_t)g + 1] * unit, (long long)lead->nb);
    if (b1 > b0) {
      if ((rc = split_copy(lead, lead, lead->d_bin_med.p + b0, p, p->d_bin_med.p + b0, (size_t)(b1 - b0) * 4))) return rc;
      if ((rc = split_copy(lead, lead, lead->d_bin_medint.p + b0, p, p->d_bin_medint.p + b0, (size_t)(b1 - b0) * 4))) return rc;
      if ((rc = split_copy(lead, lead, lead->d_bin_sum.p + b0, p, p->d_bin_sum.p + b0, (size_t)(b1 - b0) * 8))) return rc;
    }
    if ((rc = split_add_u32(lead, p, lead->d_chist.p, p->d_chist.p, (size_t)MAD_CLASSES * CHIST_RCAP))) return rc;
    if ((rc = split_add_u32(lead, p, lead->d_thist.p, p->d_thist.p, (size_t)CHIST_RCAP))) return rc;
  }
  if ((rc = split_reduce_state(parts, n, 2, false, false))) return rc;
  // ---- read summaries of the whole contig on the lead (insert-size sample, RP / Q0): a part owns the reads that start in its range
  cudaSetDevice(lead->device);
  if (reads) {
    std::vector<long long> skip((size_t)n, 0), cnt((size_t)n, 0);
    long long total = 0; int mxe[2] = {0, 0};
    for (int g = 0; g < n; ++g) {
      rsigpu_ctx* p = parts[g]; c = p;
      cudaSetDevice(p->device);
      long long h = 0; int pm[2] = {0, 0};
      if (p->r_pos.n) {
        if (g > 0) {
          long long* dcount = reinterpret_cast<long long*>(p->d_cprof.p);
          KL(k_count_before, 1, 1, 0, p->r_pos.p, (long long)p->r_pos.n, cut[(size_t)g], dcount);
          CK(cudaMemcpyAsync(&h, dcount, 8, cudaMemcpyDeviceToHost, p->stream));
        }
        CK(cudaMemcpyAsync(pm, p->d_misc.p + 5, 8, cudaMemcpyDeviceToHost, p->stream));
        CK(cudaStreamSynchronize(p->stream));
      }
      if (pm[1]) { lead->fail("read batch is not sorted by position"); return RSIGPU_E_ARG; }
      if (pm[0] > SPLIT_HALO) { lead->fail("split_run: a read reaches further than the halo of 65536 bases"); return RSIGPU_E_RANGE; }
      mxe[0] = std::max(mxe[0], pm[0]);
      skip[(size_t)g] = h; cnt[(size_t)g] = (long long)p->r_pos.n - h; total += cnt[(size_t)g];
    }
    c = lead;
    cudaSetDevice(lead->device);
    const size_t tn = (size_t)total;
    CK(lead->s_pos.ensure(tn + 8)); CK(lead->s_mpos.ensure(tn + 8)); CK(lead->s_isize.ensure(tn + 8)); CK(lead->s_mtid.ensure(tn + 8)); CK(lead->s_calend.ensure(tn + 8));
    CK(lead->s_flag.ensure(tn + 8)); CK(lead->s_mapq.ensure(tn + 8)); CK(lead->s_cigar_off.ensure(tn / 2 + 8));   // (holds the u16 n_cigar of every read)
    long long o = 0;
    for (int g = 0; g < n; ++g) {
      rsigpu_ctx* p = parts[g]; const size_t h = (size_t)skip[(size_t)g], k = (size_t)cnt[(size_t)g];
      if (p != lead && (rc = split_dep(p, lead))) return rc;
      if ((rc = split_copy(lead, lead, lead->s_pos.p + o, p, p->r_pos.p + h, k * 4)) || (rc = split_copy(lead, lead, lead->s_mpos.p + o, p, p->r_mpos.p + h, k * 4)) ||
          (rc = split_copy(lead, lead, lead->s_isize.p + o, p, p->r_isize.p + h, k * 4)) || (rc = split_copy(lead, lead, lead->s_mtid.p + o, p, p->r_mtid.p + h, k * 4)) ||
          (rc = split_copy(lead, lead, lead->s_calend.p + o, p, p->r_calend.p + h, k * 4)) || (rc = split_copy(lead, lead, lead->s_flag.p + o, p, p->r_flag.p + h, k * 2)) ||
          (rc = split_copy(lead, lead, lead->s_mapq.p + o, p, p->r_mapq.p + h, k)) ||
          (rc = split_copy(lead, lead, reinterpret_cast<u16*>(lead->s_cigar_off.p) + o, p, p->r_ncig.p + h, k * 2))) return rc;
      o += (long long)k;
    }
    lead->s_n = tn; lead->use_summary = true;
    CK(cudaMemcpyAsync(lead->d_misc.p + 5, mxe, 8, cudaMemcpyHostToDevice, lead->stream));
    CK(cudaStreamSynchronize(lead->stream));     // (mxe is a stack array)
    if (tn) {
      ReadSoA R = read_view(lead);
      KL(k_isize_stats, 1, 1024, 0, R, lead->L, lead->d_misc.p + 5, lead->d_misc.p + 16);
    }
  }
  // ---- from here on the lead alone, exactly as for an unsplit contig
  if ((rc = lf_candidate_scratch(lead)) || (rc = lf_finish(lead))) return rc;
  if ((rc = rsigpu_detectcnv(lead)) != RSIGPU_OK) return rc;
  if ((rc = rsigpu_sd_filters(lead)) != RSIGPU_OK) return rc;
  if (reads && (rc = rsigpu_cnv_stat(lead)) != RSIGPU_OK) return rc;
  CK(cudaEventRecord(lead->ev[5], lead->stream));
  CK(cudaStreamSynchronize(lead->stream));
  for (int g = 1; g < n; ++g) { cudaSetDevice(parts[g]->device); cudaStreamSynchronize(parts[g]->stream); }
  cudaSetDevice(lead->device);
  float ms = 0;
  cudaEventElapsedTime(&ms, lead->ev[0], lead->ev[5]); lead->stage_ms[5] = ms;
  TRACE(lead, "split_run: end");
  return rsigpu_get_calls(lead, out, cap, n_out);
}
long long rsigpu_split_p2p_bytes(const rsigpu_ctx* lead) { return lead ? lead->split_p2p_bytes : 0; }

int rsigpu_get_chr_stats(rsigpu_ctx* c, rsigpu_chr_stats* o) {
  if (!c || !o) return RSIGPU_E_ARG;
  if (!c->loaded) { c->fail("get_chr_stats: call load_finish first"); return RSIGPU_E_ARG; }
  const DevState* h = c->h_st;
  memset(o, 0, sizeof *o);
  o->rdmedian = h->rdmedian; o->rdsd = h->rdsd; o->tmedian = h->out_tmedian; o->tlamda = h->out_tlamda; o->rdmad = h->rdmad;
  o->target_len = c->L; o->compact_len = c->Lc; o->nbins = c->nb; o->lmax = h->Lmax; o->isize_mean = h->isize_mean; o->isize_sd = h->isize_sd;
  o->n_noseq = (int)c->h_nbeg.size();
  return RSIGPU_OK;
}

int rsigpu_get_array(rsigpu_ctx* c, int32_t which, void* out, int64_t cap, int64_t* count) {
  if (!c || !count) return RSIGPU_E_ARG;
  cudaSetDevice(c->device);
  const void* src = nullptr; size_t esz = 4; int64_t n = 0; bool host = false;
  switch (which) {
    case RSIGPU_ARR_RAW_DEPTH: if (!c->have_depth) return RSIGPU_E_ARG; src = c->d_raw.p; n = c->L; break;
    case RSIGPU_ARR_DEPTH: if (!c->loaded) return RSIGPU_E_ARG; src = c->d_rdc.p; n = c->Lc; break;
    case RSIGPU_ARR_BIN_MED: if (!c->loaded) return RSIGPU_E_ARG; src = c->d_bin_med.p; n = c->nb; break;
    case RSIGPU_ARR_BIN_NBN: if (!c->loaded) return RSIGPU_E_ARG; src = c->d_bin_nbn.p; n = c->nb; break;
    case RSIGPU_ARR_BIN_MEDINT: if (!c->loaded) return RSIGPU_E_ARG; src = c->d_bin_medint.p; n = c->nb; break;
    case RSIGPU_ARR_BIN_STATUS: if (!c->detected) return RSIGPU_E_ARG; src = c->d_status.p; n = c->nb; break;
    case RSIGPU_ARR_BIN_STATUS1: if (!c->detected) return RSIGPU_E_ARG; src = c->d_status1.p; n = c->nb; break;
    case RSIGPU_ARR_NOSEQ_BEG: src = c->h_nbeg.data(); n = (int64_t)c->h_nbeg.size(); host = true; break;
    case RSIGPU_ARR_NOSEQ_END: src = c->h_nend.data(); n = (int64_t)c->h_nend.size(); host = true; break;
    case RSIGPU_ARR_SEGMENTS: case RSIGPU_ARR_BLOCKS: case RSIGPU_ARR_PREMERGE: case RSIGPU_ARR_MERGED: {
      if (!c->detected) return RSIGPU_E_ARG;
      const std::vector<Cnv>& v = c->h_dump[which - RSIGPU_ARR_SEGMENTS];
      src = v.data(); n = (int64_t)v.size(); esz = sizeof(Cnv); host = true; break;
    }
    case RSIGPU_ARR_DETECTED: if (!c->detected) return RSIGPU_E_ARG; src = c->h_detected.data(); n = (int64_t)c->h_detected.size(); esz = sizeof(Cnv); host = true; break;
    default: return RSIGPU_E_ARG;
  }
  *count = n;
  const int64_t k = std::min(n, cap);
  if (!out || k <= 0) return RSIGPU_OK;
  if (host) { memcpy(out, src, (size_t)k * esz); return RSIGPU_OK; }
  CK(cudaMemcpyAsync(out, src, (size_t)k * esz, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return RSIGPU_OK;
}

// cnv_format1 (rsi.cpp:581-631); default ostream formatting of doubles = %g
int rsigpu_format_row(const rsigpu_cnv* cnv, const char* chrom, double rdmedian, double rdsd, char* buf, int32_t cap) {
  if (!buf || cap <= 0) return RSIGPU_E_ARG;
  if (!cnv) {
    int k = snprintf(buf, (size_t)cap, "#CHROM\tSTART\tEND\tTYPE\tSCORE\tLENGTH\tCNV_MED(CNV_SD);NEIGHBOR_MED(NEIGHBOR_RUNMEANSD);CHR_MED(CHR_SD)\tRP=#support_read_pairs;Q0=#fraction_of_Q0_reads\tMETHOD");
    return k < cap ? RSIGPU_OK : RSIGPU_E_CAPACITY;
  }
  static const char* T[] = {"DEL", "DUP", "UNKNOWN"};
  const double q1 = cnv->p1 < 1.0E-10 ? 99 : -10.0 * log(cnv->p1) / log(10.0);
  const int ty = cnv->type >= 0 && cnv->type <= 2 ? cnv->type : 2;
  int k = snprintf(buf, (size_t)cap, "%s\t%d\t%d\t%s\t%d\t%d\t%g(%g);%g(%g);%g(%g)\tRP=%d;Q0=%g\trsi", chrom ? chrom : "", cnv->start, cnv->end, T[ty],
                   (int)q1, cnv->end - cnv->start + 1, cnv->cnvmed, cnv->cnviqr / 1.349, cnv->refmed, cnv->refiqr / 1.349, rdmedian, rdsd, cnv->rp, cnv->q0);
  return k < cap ? RSIGPU_OK : RSIGPU_E_CAPACITY;
}

// The deterministic part of what the reference writes to <out>.log for one contig (rsi::dout tees to stderr and the log,
// rsi.cpp:86, 2079-2080), from "#Noseq regions excluded" to "Found n CNVs": loaddata.cpp:260-265, 315, 338, 349-356, 522-536,
// 234-236; gccontent.cpp:154, 181; rsi.cpp:1804-1813, 1140-1141, 1291-1298 / 1436-1448, 1221-1224, 1251-1254, 991-1002,
// 1320-1326 / 1472-1478, 1884, 1939-1942.  Doubles go through the default ostream formatting (= %g).
namespace {
struct LogBuf {
  std::string s;
  void add(const char* fmt, ...) {
    char tmp[512];
    va_list ap; va_start(ap, fmt); vsnprintf(tmp, sizeof tmp, fmt, ap); va_end(ap);
    s += tmp;
  }
};
void log_pass(LogBuf& o, const RsiLogT& g, int pass, int nb) {
  for (int sgn = 0; sgn < 2; ++sgn) {
    const int lb = sgn ? g.lbreak_dup[pass] : g.lbreak_del[pass];
    unsigned long long cum = 0;
    for (int L = 1; L <= g.lmax; ++L) {
      cum += g.cnt[pass][sgn][L];
      const double portion = (double)cum / (double)nb;
      o.add("%s\t%d\t%llu\t%d\t%g\n", sgn ? "DUP+" : "DEL-", L, cum, nb, portion);
      if (portion > 0.2 || L == lb) { if (portion > 0.2) break; }
    }
  }
}
void log_trans(LogBuf& o, const DevState* h, int which, int nb) {
  const RsiLogT& g = h->rlog[which];
  const char* name = which == 0 ? "Negative binormial transformation : " : "local median transformation : ";
  o.add("%s\n\tmedian of transformations : %g\n\tsigma : %g\n\tmedian/sigma : %g\n\trsifactor: %g\n\tlamda : %g\n\ttarget_tlamda : %g\n\tMax L needed  : %d\n",
        name, g.tmedian1, g.tsigma1, g.tmedian1 / g.tsigma1, h->factor, g.tlamda1, g.target, g.calmax);
  if (which == 1) {
    if (g.tlamda1 < g.tmedian1 * sqrt(2.5)) o.add("Warning : lamda might be low\n");
    if (g.tlamda1 > g.tmedian1 * sqrt(3.0)) o.add("Warning : lamda might be too large\n");
  }
  log_pass(o, g, 0, nb);
  const int nl = g.st_hi - g.st_lo + 1;
  for (int l = 0; l < nl; ++l) if (g.lvl_cnt[l]) o.add("%d\t%u\t%g\n", l + g.st_lo, g.lvl_cnt[l], (double)g.lvl_mean[l]);
  o.add("%d\t%g\n%d\t%g\n", g.leveldel, (double)g.lvl_mean[g.leveldel - g.st_lo], g.leveladd, (double)g.lvl_mean[g.leveladd - g.st_lo]);
  if (!g.filt_on) o.add("warning level error, status not filtered\n%d\t%d\nfilterstatus()\n", g.leveldel, g.leveladd);
  o.add("second pass\n%s\n\tmedian of transformations : %g\n\tsigma : %g\n\tmedian/sigma : %g\n\tlamda : %g\n\target_tlamda : %g\n",
        name, g.tmedian2, g.tsigma2, g.tmedian2 / g.tsigma2, g.tlamda2, g.target);
  log_pass(o, g, 1, nb);
}
}  // namespace

int rsigpu_get_log(rsigpu_ctx* c, const char* chrom, int32_t text_input, char* buf, int64_t cap, int64_t* nbytes) {
  if (!c || !nbytes) return RSIGPU_E_ARG;
  if (!c->loaded) { c->fail("get_log: call load_finish / run first"); return RSIGPU_E_ARG; }
  const DevState* h = c->h_st;
  const char* name = chrom ? chrom : "";
  LogBuf o;
  o.add("#Noseq regions excluded\n");
  for (size_t k = 0; k < c->h_nbeg.size(); ++k) o.add("%s\t%d\t%d\n", name, c->h_nbeg[k], c->h_nend[k]);
  const double L = (double)c->L;
  if (c->have_reads) {   // load_data_from_bam's progress marks (one per million records, carriage returns, one newline)
    const size_t nr = c->use_summary ? c->s_n : c->r_pos.n;
    for (size_t k = 1; k <= nr / 1000000; ++k) o.add("#processed %zuM reads\r", k);
    o.add("\n");
  }
  o.add("%d\t%g\n", c->L, (double)h->pos_sum / L);
  if (c->P.gcadjust) {
    o.add("RD mean before GC adjust = %g\n", h->rdmean);
    o.add("RD mean after GC adjust = %g\n", h->adj_sum / (double)h->adj_pos);
  }
  o.add("%d\t%g\n", c->L, h->adj_sum / L);
  if (c->P.cap > 1) o.add("applying cap %g times of mean %g\ncap = %g\n", c->P.cap, h->cap_median, c->P.cap * h->cap_median);
  if (text_input) o.add("%d\t%g\n", c->L, h->cap_sum / L);
  o.add("region  : %s:%d-%d\nmedian  : %g\nrs::m   : %d\nrs::cap : %g\n", name, 1, c->Lc, h->rdmedian, c->P.m, c->P.cap);
  if (h->rdmedian < 5) o.add("Read depths too low, cannot call\n");
  else {
    if (h->rdmedian < 10) o.add("Read depths low, not reliable\n");
    o.add("RD median : %g\nRD median absolute deviation : %g\n", h->rdmedian, h->rdmad);
    if (c->detected) {
      if (c->P.trans != RSIGPU_TRANS_NBN) log_trans(o, h, 1, c->nb);
      if (c->P.trans != RSIGPU_TRANS_MED) log_trans(o, h, 0, c->nb);
      int ndel = 0, nadd = 0;
      for (const Cnv& x : c->h_detected) { if (x.type == RSIGPU_TYPE_DUP) ++nadd; if (x.type == RSIGPU_TYPE_DEL) ++ndel; }
      o.add("Selected %zu segments for testing\n", c->h_dump[2].size());
      o.add("Done checking overlaps, after merging, %zu segments left\nFound %d CNVs : %d DEL + %d DUP\n", c->h_detected.size(), ndel + nadd, ndel, nadd);
    }
  }
  *nbytes = (int64_t)o.s.size();
  if (!buf || cap < (int64_t)o.s.size()) return buf ? RSIGPU_E_CAPACITY : RSIGPU_OK;
  memcpy(buf, o.s.data(), o.s.size());
  return RSIGPU_OK;
}

int64_t rsigpu_launch_count(const rsigpu_ctx* c) { return c ? c->launches : 0; }
int rsigpu_last_stage_ms(const rsigpu_ctx* c, float* ms6) {
  if (!c || !ms6) return RSIGPU_E_ARG;
  for (int k = 0; k < 6; ++k) ms6[k] = c->stage_ms[k];
  return RSIGPU_OK;
}
int rsigpu_set_profile(rsigpu_ctx* c, int on) {
  if (!c) return RSIGPU_E_ARG;
  c->profile = on != 0; c->prof.clear(); c->prof_order.clear();
  return RSIGPU_OK;
}
int rsigpu_get_profile(const rsigpu_ctx* c, char* names, int32_t name_stride, float* ms, int32_t* launches, int32_t cap) {
  if (!c) return 0;
  int k = 0;
  for (const std::string& nm : c->prof_order) {
    if (k < cap) {
      auto it = c->prof.find(nm);
      if (names && name_stride > 0) { strncpy(names + (size_t)k * name_stride, nm.c_str(), (size_t)name_stride - 1); names[(size_t)k * name_stride + name_stride - 1] = 0; }
      if (ms) ms[k] = it->second.first;
      if (launches) launches[k] = it->second.second;
    }
    ++k;
  }
  return k;
}

// test hook: selected device scalars of the last load_finish / detectcnv (host copy), as doubles
int rsigpu_debug_state(const rsigpu_ctx* c, double* out, int32_t cap) {
  if (!c || !out) return RSIGPU_E_ARG;
  const DevState* h = c->h_st;
  const double v[] = {(double)h->err, (double)h->rd_min, (double)h->rd_max, (double)h->pos_sum, (double)h->pos_cnt, h->rdmean, h->cap_median, h->cap_thr,
                      (double)h->capv, (double)h->hist_base, (double)h->chist_R, h->rdmedian, h->rdsd, h->rdmad, (double)h->max_binsum, (double)h->gstar,
                      h->gc_tab[80], h->gc_tab[90], h->gc_tab[100], (double)h->gc_cnt[90], h->tmedian, h->tsigma, h->tlamda, (double)h->Lmax,
                      (double)h->lbreak_del, (double)h->lbreak_dup, (double)h->n_runs, (double)h->n_nonzero, (double)h->st_lo, (double)h->st_hi,
                      (double)h->lvl_sum[(-h->st_lo < 0 || -h->st_lo >= 2 * LMAX_CAP + 3) ? 0 : -h->st_lo], (double)h->filt_on, (double)h->cand_redone};
  const int n = (int)(sizeof v / sizeof v[0]);
  for (int k = 0; k < n && k < cap; ++k) out[k] = v[k];
  for (int k = 0; k < 16 && n + k < cap; ++k) out[n + k] = (double)c->h_cprof[k];   // candidate-stage phase clocks (profile mode)
  if (n + 16 < cap) out[n + 16] = (double)c->b_rewalked;                              // BAM decoder: BGZF blocks whose speculative first record was wrong
  return n + 17;
}

// test hooks (see include/rsigpu.h): 0/1/2 = form of filterstatus' level-0 float sum (2 = multi-block, default)
int rsigpu_set_level0_mode(rsigpu_ctx* c, int mode) {
  if (!c || mode < 0 || mode > 2) return RSIGPU_E_ARG;
  c->level0_mode = mode;
  return RSIGPU_OK;
}
// test hook: decoded bytes one rsigpu_bam_feed may produce (partial-consumption path)
int rsigpu_set_inflate_mode(rsigpu_ctx* c, int mode) {
  if (!c || mode < 0 || mode > 2) return RSIGPU_E_ARG;
  c->inflate_mode = mode;
  return RSIGPU_OK;
}
int rsigpu_set_bgzf_crc(rsigpu_ctx* c, int on) {
  if (!c) return RSIGPU_E_ARG;
  c->bgzf_crc = on != 0;
  return RSIGPU_OK;
}
int rsigpu_set_bam_by_ref(rsigpu_ctx* c, int on) {
  if (!c) return RSIGPU_E_ARG;
  if (on && c->ix_on) { c->fail("set_bam_by_ref: not available while a BAM index is built (rsigpu_bam_index_begin): the index needs the records in file order"); return RSIGPU_E_ARG; }
  if (on && c->b_active && c->b_nref > BY_REF_MAX_REFS) {
    c->fail("set_bam_by_ref: " + std::to_string(c->b_nref) + " references, more than the 65535 that grouping records by refID supports");
    return RSIGPU_E_ARG;
  }
  c->bam_by_ref = on != 0;
  return RSIGPU_OK;
}
int rsigpu_set_feed_limit(rsigpu_ctx* c, int64_t decoded_bytes) {
  if (!c || decoded_bytes < 65536) return RSIGPU_E_ARG;
  c->b_umax = (size_t)decoded_bytes;
  return RSIGPU_OK;
}
// tuning hook: threads of the bin-level candidate kernel
int rsigpu_set_cand_threads(rsigpu_ctx* c, int threads) {
  if (!c || threads < 32 || threads > 1024 || threads % 32) return RSIGPU_E_ARG;
  c->cand_a_threads = threads;
  return RSIGPU_OK;
}

}  // extern "C"
