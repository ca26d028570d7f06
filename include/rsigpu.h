/* rsigpu.h -- C ABI of the B200-native `rsicnv rsi` read-depth -> CNV-call hot path.
 *
 * The reference (yhwu/rsicnv) has no plugin / FFI interface: the path sits behind its process
 * boundary and a handful of free functions that mutate a caller-owned depth array and talk through
 * `rsi::` globals (SURVEY.md §8b).  This header DEFINES the boundary a maintainer would bind
 * instead of those functions.  Each entry point names the reference seam it replaces (file:line
 * relative to the reference's src/).  Plain C types only; every call returns an int status and
 * never exits the process; all host buffers are caller-owned; one host thread per context; contexts
 * are independent (one per contig / GPU), unlike the reference's non-re-entrant globals.
 */
#ifndef RSIGPU_H
#define RSIGPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSIGPU_OK 0
#define RSIGPU_E_CUDA 1        /* a CUDA runtime call failed (see rsigpu_last_error) */
#define RSIGPU_E_ARG 2         /* bad argument / call order */
#define RSIGPU_E_RANGE 3       /* input outside what the kernels are sized for (see message) */
#define RSIGPU_E_CAPACITY 4    /* output buffer too small */
#define RSIGPU_E_NODEVICE 5    /* no CUDA device: there is NO CPU fallback */

#define RSIGPU_TYPE_DEL 0
#define RSIGPU_TYPE_DUP 1
#define RSIGPU_TYPE_UNKNOWN 2

#define RSIGPU_TRANS_NBN 0     /* -NB  (default)  rsi.cpp:51,2028 */
#define RSIGPU_TRANS_MED 1     /* -MED            rsi.cpp:2027    */
#define RSIGPU_TRANS_ALL 2     /* -ALL            rsi.cpp:2029    */

typedef struct rsigpu_ctx rsigpu_ctx;

/* The tunables get_parameters() fills (rsi.cpp:1986-2068); defaults = rsi.cpp:34-98. */
typedef struct rsigpu_params {
  int32_t m;          /* -m   bin size, forced odd (rsi.cpp:2061-2064)          default 101 */
  int32_t minq;       /* -q   minimum mapping quality                            default 0   */
  int32_t min_baseQ;  /* -Q   minimum base quality (code default 13, rsi.cpp:58) default 13  */
  int32_t gcadjust;   /* 0 = -NOGC                                               default 1   */
  int32_t trans;      /* RSIGPU_TRANS_*                                          default NBN */
  int32_t merge;      /* 0 = -nomerge                                            default 1   */
  int32_t maxchkbp;   /* -maxchkbp                                               default 100000 */
  int32_t reserved_;
  double cap;         /* -cap, <=1 disables                                      default 4.0 */
  double threshold;   /* -threshold (MED only), <=0 = unset                      default -1  */
  double epsilon;     /* -e                                                      default 1.5 */
  double chklen;      /* -reflen                                                 default 2.5 */
} rsigpu_params;

/* Flat mirror of cnv_st (rsi.h:8-51); both status (-9 = deleted) and geno are carried verbatim. */
typedef struct rsigpu_cnv {
  int32_t tid, type, geno, status, start, end, length, sc1, sc2, pair;
  double score, p1, p2, cnvmed, cnvsd, cnviqr, refmed, refsd, refiqr, q0;
  int32_t rp, pad_;
} rsigpu_cnv;

/* One batch of decoded BAM records of ONE contig, position-sorted, as structure-of-arrays.
 * Field meanings = bam1_core_t (samtools-0.1.18/bam.h:131-155).  HOST pointers. */
typedef struct rsigpu_read_batch {
  int64_t n_reads;
  int32_t tid;                /* core.tid of every read in the batch                       */
  int32_t reserved_;
  const int32_t* pos;         /* [n] core.pos, 0-based                                      */
  const int32_t* mpos;        /* [n] core.mpos                                              */
  const int32_t* isize;       /* [n] core.isize                                             */
  const int32_t* mtid;        /* [n] core.mtid                                              */
  const uint16_t* flag;       /* [n] core.flag                                              */
  const uint8_t* mapq;        /* [n] core.qual                                              */
  const uint32_t* cigar_off;  /* [n+1] offsets into cigar[] (n_cigar = difference)          */
  const uint32_t* cigar;      /* BAM-encoded ops, len<<4|op, ops MIDNSHP=X = 0..8           */
  const uint64_t* qual_off;   /* [n+1] offsets into qual[] (l_qseq = difference)            */
  const uint8_t* qual;        /* base qualities (Phred, 0xff = absent)                      */
} rsigpu_read_batch;

/* which-array selectors for rsigpu_get_array (parity tests, `-s`) */
#define RSIGPU_ARR_RAW_DEPTH 0   /* int32[L]   per-base depth before GC/cap (what `-s` dumps, loaddata.cpp:340-344) */
#define RSIGPU_ARR_DEPTH 1       /* int32[L']  after GC adjust, cap and N-compaction (RD as detectcnv sees it)    */
#define RSIGPU_ARR_BIN_MED 2     /* float[nb]  median_transfer output  (rsi.cpp:1363)                              */
#define RSIGPU_ARR_BIN_NBN 3     /* float[nb]  negative_binomial_transfer output (rsi.cpp:1120)                    */
#define RSIGPU_ARR_BIN_MEDINT 4  /* int32[nb]  RDmedint (rsi.cpp:1819)                                             */
#define RSIGPU_ARR_BIN_STATUS 5  /* int32[nb]  RSI status after the second rsistatus pass (rsi.cpp:1329/1482)      */
#define RSIGPU_ARR_NOSEQ_BEG 6   /* int32[k]   rsi::noncodelist starts, 0-based inclusive (loaddata.cpp:243)       */
#define RSIGPU_ARR_NOSEQ_END 7   /* int32[k]   rsi::noncodelist ends                                               */
#define RSIGPU_ARR_BIN_STATUS1 8 /* int32[nb]  status after pass 1 + filterstatus (rsi.cpp:1305/1455)              */
#define RSIGPU_ARR_SEGMENTS 9    /* rsigpu_cnv[k] candidates leaving rsicnvnbn/rsicnvmed (bin coordinates)         */
#define RSIGPU_ARR_BLOCKS 10     /* rsigpu_cnv[k] after areblockscnv (bin coordinates)                             */
#define RSIGPU_ARR_PREMERGE 11   /* rsigpu_cnv[k] after bins->bases + 2x optimize_with_derivative + sort           */
#define RSIGPU_ARR_MERGED 12     /* rsigpu_cnv[k] after mergesegments + sort                                       */
#define RSIGPU_ARR_DETECTED 13   /* rsigpu_cnv[k] detectcnv output (before sd_filters)                             */

/* chromosome-level scalars for the output row / log (rsi::RDmedian, rsi::RDsd, ...) */
typedef struct rsigpu_chr_stats {
  double rdmedian, rdsd;            /* rsi.cpp:2202-2203                                      */
  double tmedian, tlamda;           /* second-pass values (rsi::nbnmedian/nbnlamda or med*)   */
  double rdmad;                     /* negative_binomial_transfer's MAD (rsi.cpp:1138)        */
  int32_t target_len, compact_len;  /* L and L' (after N removal)                             */
  int32_t nbins, lmax;
  int32_t isize_mean, isize_sd;     /* bam_rd_pr_stats sample (pairrd.cpp:236-241), -1 if none */
  int32_t n_noseq, reserved_;
} rsigpu_chr_stats;

int rsigpu_default_params(rsigpu_params* p);

/* Context = what one iteration of the reference's chromosome loop owns (rsi.cpp:2189-2217). */
int rsigpu_create(int device, const rsigpu_params* p, rsigpu_ctx** out);
void rsigpu_destroy(rsigpu_ctx* c);
const char* rsigpu_last_error(const rsigpu_ctx* c);
int rsigpu_num_devices(void);

/* read_fasta output for one contig (readref.cpp:10-86): `len` ASCII bytes, newlines stripped.
 * Replaces the GC bitmap + get_noseq_regions steps (loaddata.cpp:290-295, 243-273).  HOST pointer. */
int rsigpu_set_reference(rsigpu_ctx* c, const uint8_t* fasta, int32_t len, int32_t tid);

/* Depth-file input: the array load_data_from_text builds (loaddata.cpp:496-517); the host parses
 * the text (rsicnv_parse_depth_text in the CLI).  HOST pointer, len must equal the reference length. */
int rsigpu_set_depth(rsigpu_ctx* c, const int32_t* depth, int32_t len);

/* BAM input: replaces the hot loop of load_data_from_bam (loaddata.cpp:312-335) and
 * resolve_cigar_pos (samfunctions.cpp:38-100).  push() only stages a batch in HBM (and keeps the
 * per-read summary cnv_stat needs); the pileup kernel runs in rsigpu_run / rsigpu_pileup_end. */
int rsigpu_pileup_begin(rsigpu_ctx* c, int32_t target_len);
int rsigpu_pileup_push(rsigpu_ctx* c, const rsigpu_read_batch* b);
int rsigpu_pileup_end(rsigpu_ctx* c);      /* runs the pileup kernels now: the raw depth becomes readable (-s) */
int rsigpu_pileup_commit(rsigpu_ctx* c);   /* only marks the staged batches complete; rsigpu_run runs the pileup as its first stage */
/* Reads that are not in position order (a BAM that is not coordinate-sorted, records gathered from several feeds):
 *   pileup_sort(c)               sorts the staged reads by pos on the GPU, stable (reads at one position keep their staging
 *                                order), fixed fields, CIGAR ops and qualities.  Reads already in position order cost only the
 *                                sortedness check the pileup runs anyway.  Afterwards rsigpu_run, rsigpu_pileup_end and
 *                                rsigpu_stat_calls take them as they take sorted input.  The sort needs a second copy of the
 *                                staged reads in HBM, plus 16 B per read of sort keys and indices, while it runs, and releases
 *                                both before it returns (RSIGPU_E_CUDA when there is no room: the reads are unchanged).
 *   reads_take(src, r0, r1, dst) appends src's staged reads [r0, r1) to dst's staged reads, exactly as rsigpu_pileup_push of the
 *                                same reads would (dst: set_reference + pileup_begin or reads_begin done; dst != src; dst may
 *                                be on another GPU).
 *   reads_field(c, field, ...)   one field of ALL staged reads copied to the host, numbered as in rsigpu_bam_run_field;
 *                                out == NULL or cap_bytes < *nbytes: only *nbytes. */
int rsigpu_pileup_sort(rsigpu_ctx* c);
int rsigpu_reads_take(rsigpu_ctx* src, int64_t r0, int64_t r1, rsigpu_ctx* dst);
int rsigpu_reads_field(rsigpu_ctx* c, int32_t field, void* out, int64_t cap_bytes, int64_t* nbytes);

/* BAM input straight from the file's bytes: BGZF inflate (samtools-0.1.18/bgzf.c:277-313 inflate_block,
 * 258-275 check_header) and bam_read1 (bam.c:179-210, core layout bam.h:131-155) on the GPU.  The caller
 * parses the BAM header itself (it needs the contig names anyway, bam.c:69-110) and then feeds the file from
 * the BGZF block that holds the first alignment record:
 *   begin(n_ref)                    n_ref = number of reference sequences in the header (record sanity bound)
 *   feed(bytes, n, skip, ...)       `bytes` must START at a BGZF block boundary; only whole blocks are taken and
 *                                   *consumed says how many bytes they covered (present the rest again, followed by
 *                                   more of the file).  `skip` = decoded bytes in front of the first record (first
 *                                   feed only).  Records are decoded into device arrays owned by the decoder and
 *                                   reported as runs of consecutive records with the same refID, in file order; a
 *                                   record cut by the end of the chunk is carried into the next feed, and on through
 *                                   as many feeds as it spans (a carried record may be up to 16 MiB: RSIGPU_E_RANGE,
 *                                   naming its size, beyond that).
 *   take(c, run, dst)               appends the run's records to dst's staged reads, exactly as rsigpu_pileup_push
 *                                   of the same records would (dst: set_reference + pileup_begin done; dst may be c
 *                                   itself or a context on another GPU).  Runs are valid until the next feed.
 *   end()                           fails if the file stopped inside a record.
 * HOST pointers (pinned memory from rsigpu_pinned_alloc makes the copy asynchronous and full speed). */
typedef struct rsigpu_bam_run { int32_t tid; int32_t part; int64_t n_reads; } rsigpu_bam_run;   /* part: which range of rsigpu_bam_feed_parts (0 for rsigpu_bam_feed) */
int rsigpu_bam_begin(rsigpu_ctx* c, int32_t n_ref);
int rsigpu_bam_feed(rsigpu_ctx* c, const uint8_t* bgzf, int64_t nbytes, int64_t skip, int64_t* consumed, rsigpu_bam_run* runs, int32_t cap,
                    int32_t* n_runs);
/* Several byte ranges decoded as ONE chunk (one inflate launch over all their blocks: the GPU decodes a large chunk far
 * more efficiently than several small ones).  Every range is a whole number of BGZF blocks that begins at a record start and
 * ends at a record end -- e.g. the records of one contig each, cut at the virtual offsets of the .bai when they fall on
 * block boundaries -- and starts a new run (runs[i].part says which range a run came from).  All or nothing: the ranges
 * must fit one feed (2 GiB compressed, 5 GiB decoded); nothing is carried over. */
int rsigpu_bam_feed_parts(rsigpu_ctx* c, int32_t n_parts, const uint8_t* const* parts, const int64_t* nbytes, rsigpu_bam_run* runs, int32_t cap,
                          int32_t* n_runs);
int rsigpu_bam_take(rsigpu_ctx* c, int32_t run, rsigpu_ctx* dst);
/* only the records of the run with pos in [pos_lo, pos_hi) (a part of a contig split over several GPUs, rsigpu_split_run) */
int rsigpu_bam_take_range(rsigpu_ctx* c, int32_t run, rsigpu_ctx* dst, int32_t pos_lo, int32_t pos_hi);
int rsigpu_bam_end(rsigpu_ctx* c);
/* one decoded field of a run copied to the host (parity tests): 0 pos, 1 mpos, 2 isize, 3 mtid (int32), 4 flag (uint16),
 * 5 mapq (uint8), 6 cigar_off (uint32, n+1, rebased to 0), 7 cigar (uint32), 8 qual_off (uint64, n+1, rebased), 9 qual (uint8) */
int rsigpu_bam_run_field(rsigpu_ctx* c, int32_t run, int32_t field, void* out, int64_t cap_bytes, int64_t* nbytes);
/* The BAI index of the file (SAM spec 5.2, byte for byte what samtools-0.1.18's bam_index_build writes) built on the GPU from
 * the records rsigpu_bam_feed decodes anyway: no second pass over the file.
 *   index_begin(file_offset)   after rsigpu_bam_begin, before the first feed.  file_offset = offset in the FILE of the first byte
 *                              the first feed receives (the BGZF block that holds the first record).  Every later feed must
 *                              continue the file where the previous one's *consumed ended; the offsets of the index follow.
 *   feeds as usual, then rsigpu_bam_end
 *   index_get(out, cap, &n)    the serialized .bai, valid after a successful rsigpu_bam_end; out == NULL: only *nbytes.
 * While indexing, a feed additionally fails
 *   with RSIGPU_E_ARG    "bam_index: records not sorted: record <k> of this feed (tid <t>, pos <p>) follows tid <t'>, pos <p'>"
 *                        (the lowest such record: refIDs must not decrease -- unplaced records, refID -1, come last -- and
 *                        positions must not decrease within a reference; reported after inflate, CRC and record errors)
 *   with RSIGPU_E_RANGE  "bam_index: record <k> of this feed (tid <t>, pos <p>) ends past 2^29, beyond what a BAI index can address"
 * and rsigpu_bam_feed_parts fails with RSIGPU_E_ARG (its parts are not one contiguous file):
 *   "bam_feed_parts: not available while a BAM index is built (rsigpu_bam_index_begin): its parts are not one contiguous file"
 * index_begin fails with RSIGPU_E_ARG after the first feed or without rsigpu_bam_begin:
 *   "bam_index_begin: call it after rsigpu_bam_begin and before the first feed, with the file offset of the first byte fed"
 * index_get fails with RSIGPU_E_ARG when any feed or rsigpu_bam_end failed, or indexing was never begun:
 *   "bam_index_get: no index: rsigpu_bam_index_begin, feeds of the whole file and rsigpu_bam_end must all succeed first"
 * and with RSIGPU_E_CAPACITY when cap < *nbytes: "bam_index_get: the buffer is smaller than the index".
 * Without index_begin nothing of this runs: no extra launch, no extra copy. */
int rsigpu_bam_index_begin(rsigpu_ctx* c, int64_t file_offset);
int rsigpu_bam_index_get(rsigpu_ctx* c, uint8_t* out, int64_t cap, int64_t* nbytes);
int rsigpu_pinned_alloc(size_t nbytes, void** out);
void rsigpu_pinned_free(void* p);

/* The seams, in the order main() calls them (rsi.cpp:2197-2211).  All asynchronous on the
 * context's stream except where a result is copied to the host. */
int rsigpu_load_finish(rsigpu_ctx* c);   /* checkgccontent + apply_cap + concatenate_data + RDmedian/RDsd: gccontent.cpp:95, loaddata.cpp:229, 48, rsi.cpp:2202 */
int rsigpu_detectcnv(rsigpu_ctx* c);     /* detectcnv, rsi.cpp:1795-1945 */
int rsigpu_sd_filters(rsigpu_ctx* c);    /* sd_filters, rsi.cpp:1753-1792.  The filter itself runs on the device at the end of detectcnv's last
                                            kernel (k_cand_c: sd_filter_list); this entry point only marks the filtered list as the one
                                            rsigpu_cnv_stat / rsigpu_get_calls use, so that the seams stay the reference's */
int rsigpu_cnv_stat(rsigpu_ctx* c);      /* cnv_stat + bam_rd_pr_stats, pairrd.cpp:622-748, 112-260 (BAM input only) */
int rsigpu_get_calls(rsigpu_ctx* c, rsigpu_cnv* out, int32_t cap, int32_t* n);  /* rows write_cnv_to_file would print */

/* `rsicnv stat` (rsi.cpp:2235-2249): RP / Q0 of calls that come from a file instead of detectcnv.
 *   reads_begin(tid, len)    stage reads of contig `tid` WITHOUT a reference (then rsigpu_pileup_push / rsigpu_bam_take as usual)
 *   stat_calls(list, n)      cnv_stat + bam_rd_pr_stats (pairrd.cpp:622-748, 112-260) on the staged reads for the entries of
 *                            `list` whose tid is this contig's; the list must be the WHOLE file's list in file order, because
 *                            the search distance DIS is carried from call to call (pairrd.cpp:655-656).  rp / q0 are filled in place. */
int rsigpu_reads_begin(rsigpu_ctx* c, int32_t tid, int32_t target_len);
int rsigpu_stat_calls(rsigpu_ctx* c, rsigpu_cnv* list, int32_t n);

/* Everything above on the staged inputs, one host synchronisation at the end. */
int rsigpu_run(rsigpu_ctx* c, rsigpu_cnv* out, int32_t cap, int32_t* n);

/* One contig over several GPUs (config 5; the reference is one thread on one array, rsi.cpp:2189-2217: there is nothing to
 * mirror, the result must simply be identical).  parts[0] is the lead (it ends up with the calls, the arrays and the stats);
 * every part context -- one per GPU -- gets the WHOLE reference (rsigpu_set_reference) and then either the whole depth array
 * (rsigpu_set_depth) or, for BAM input, only the reads with pos in [beg - read_halo, end) of ITS range as rsigpu_split_range
 * reports it (rsigpu_pileup_begin / push / commit or rsigpu_bam_take as usual).  rsigpu_split_run then does what rsigpu_run does:
 * pileup and the three per-base passes on each part's own range, the parts' integer tables added on the lead over peer-to-peer
 * copies, the bin-level and candidate stages on the lead.  rsigpu_split_p2p_bytes: bytes that crossed between devices. */
int rsigpu_split_range(int32_t target_len, int32_t n_parts, int32_t part, int32_t* beg, int32_t* end, int32_t* read_halo);
int rsigpu_split_run(rsigpu_ctx** parts, int32_t n_parts, rsigpu_cnv* out, int32_t cap, int32_t* n);
long long rsigpu_split_p2p_bytes(const rsigpu_ctx* lead);

int rsigpu_get_chr_stats(rsigpu_ctx* c, rsigpu_chr_stats* out);
/* copies min(count, cap) elements of the selected device array to `out`, *count = elements available */
int rsigpu_get_array(rsigpu_ctx* c, int32_t which, void* out, int64_t cap, int64_t* count);

/* cnv_format1 (rsi.cpp:581-631): one table row, or the column header when cnv == NULL. */
int rsigpu_format_row(const rsigpu_cnv* cnv, const char* chrom, double rdmedian, double rdsd, char* buf, int32_t cap);

/* The deterministic part of <out>.log for the contig just processed (what rsi::dout receives between "#processing <chr>" and
 * "output written to": N regions, depth means before / after GC adjust and cap, the transformation parameters of both passes,
 * the per-length DEL-/DUP+ lines of rsistatus, filterstatus' level table, segment counts; rsi.cpp:1221-1224, 1251-1254, 1291-1298,
 * 1884, 1939-1942, loaddata.cpp:260-265, 349-356).  text_input: 1 for a depth file (load_data_from_text prints a third mean).
 * Call with buf == NULL to get the size. */
int rsigpu_get_log(rsigpu_ctx* c, const char* chrom, int32_t text_input, char* buf, int64_t cap, int64_t* nbytes);

/* timing / accounting for bench.py: kernels launched by this context since creation, and the
 * device time (ms, CUDA events on the context's stream) of the last rsigpu_run by stage:
 * [0]=pileup [1]=load_finish [2]=detect bins+scan [3]=candidates [4]=sd_filters+cnv_stat [5]=total */
int64_t rsigpu_launch_count(const rsigpu_ctx* c);
int rsigpu_last_stage_ms(const rsigpu_ctx* c, float* ms6);
/* per-kernel device time of the last rsigpu_run when profiling is on (rsigpu_set_profile(c,1)):
 * writes up to cap (name, ms, launches) triples; returns the number of distinct kernels */
int rsigpu_set_profile(rsigpu_ctx* c, int on);
int rsigpu_get_profile(const rsigpu_ctx* c, char* names, int32_t name_stride, float* ms, int32_t* launches, int32_t cap);

/* test hook: filterstatus' level-0 float sum (rsi.cpp:967-974) as 0 = one sequential FADD chain,
 * 1 = the exact one-block scan form, 2 = the exact multi-block form (default); all must give identical bits. */
int rsigpu_set_level0_mode(rsigpu_ctx* c, int mode);
/* decoded bytes one rsigpu_bam_feed / rsigpu_bam_feed_parts may produce: bounds the decoder's buffers (5 GiB by default, >= 64 KiB;
 * the tests of the partial-consumption path set it small, bench.py raises it to batch more contigs per feed) */
int rsigpu_set_feed_limit(rsigpu_ctx* c, int64_t decoded_bytes);
/* tuning / test hook: which inflate kernel rsigpu_bam_feed uses: 0 = by chunk size (default: a warp per BGZF block below
 * 28,000 blocks, a lane per block above), 1 = always a lane per block, 2 = always a warp per block; same bytes either way */
int rsigpu_set_inflate_mode(rsigpu_ctx* c, int mode);
/* on != 0: rsigpu_bam_feed and rsigpu_bam_feed_parts check the CRC32 of every BGZF block they decode (zlib's crc32 of the
 * block's decoded bytes against the CRC in its gzip footer; a block with ISIZE 0 must carry CRC 0), on the GPU, after inflate.
 * Default 0, like the reference's samtools-0.1.18 reader: without it, damage that leaves the deflate stream and the record
 * cores valid (a changed quality byte or mate position, a bad footer) decodes without an error.  A mismatch fails the feed
 * with RSIGPU_E_ARG before any run is reported or carried, naming the lowest failing block:
 *   "bam_feed: CRC32 mismatch in BGZF block <k> of this feed (compressed offset <X> of the bytes passed)"
 *   "bam_feed_parts: CRC32 mismatch in BGZF block <k> of part <j> (compressed offset <X> of that part)"
 * A block whose deflate stream is corrupt is still reported as such; a CRC mismatch is reported before a corrupt record. */
int rsigpu_set_bgzf_crc(rsigpu_ctx* c, int on);
/* on != 0: every rsigpu_bam_feed sorts its complete records by refID on the GPU, stable in file order, before it reports the
 * runs: a feed then reports at most one run per refID present, in increasing refID order with the unplaced records (refID -1)
 * last, and each run holds its records in file order.  A record carried across feeds belongs to the feed it completes in.
 * This is what a file that is not coordinate-sorted needs (without it, such a file fails with "more than 65536 refID runs"):
 * gather each reference's runs over all feeds (rsigpu_bam_take into one staging context, rsigpu_reads_take), then
 * rsigpu_pileup_sort.  Default 0: nothing of this runs.  Refused with RSIGPU_E_ARG, naming the conflict:
 *   rsigpu_bam_index_begin while on, and set_bam_by_ref(c, 1) while an index is built (the index needs file order);
 *   rsigpu_bam_feed_parts while on (each part already starts its own run);
 *   rsigpu_bam_take_range on a run grouped by refID (its positions are not sorted);
 *   more than 65535 references (rsigpu_bam_begin, or set_bam_by_ref after it): one run per reference and refID -1 must fit
 *   the 65536 runs of a feed. */
int rsigpu_set_bam_by_ref(rsigpu_ctx* c, int on);
/* tuning hook: threads of the bin-level candidate kernel (multiple of 32, 32..1024) */
int rsigpu_set_cand_threads(rsigpu_ctx* c, int threads);
/* test hook: selected device-resident scalars of the last stage, as doubles; returns how many exist */
int rsigpu_debug_state(const rsigpu_ctx* c, double* out, int32_t cap);

#ifdef __cplusplus
}
#endif
#endif /* RSIGPU_H */
