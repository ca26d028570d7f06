// rsicnv (B200-native) -- host program of the `rsicnv rsi` path.
//
// Keeps the reference CLI (get_parameters, rsi.cpp:1986-2068: -f -b -d -c -m -q -Q -cap -NOGC -MED -NB -o, plus
// the flags the reference accepts and ignores) and the exact output table (cnv_format1 / write_cnv_to_file,
// rsi.cpp:581-631, 1592-1616).  The host side decodes BGZF/BAM (bam_reader.cpp), reads the FASTA through its
// .fai index (read_fasta, readref.cpp:10-86), parses depth files (load_data_from_text, loaddata.cpp:496-517) and
// writes the table; everything else runs on the GPU through the C ABI in include/rsigpu.h.  Contigs are
// independent units (rsi.cpp:2189-2217): with `-gpus N` they are dealt to N GPUs, longest first, one host
// thread and one context per GPU, and the rows are written in BAM-header order.
//
// Extra sub-command for the tests (no GPU needed):  rsicnv decode -b in.bam -c CHR -o prefix
//   writes the decoded structure-of-arrays of one contig as raw little-endian files prefix.<field>.
// `rsicnv index -b in.bam [-o out.bai]` writes the BAI index (default in.bam.bai, samtools' name), built on GPU 0 while it
//   decodes the file in one pass (rsigpu_bam_index_begin): what `rsi` and `stat` read to decode every contig from its own offset.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <fstream>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rsigpu.h"
#include "bam_reader.hpp"

using namespace rsihost;

namespace {

struct Opt {
  std::string function = "rsi", rdfile, bamfile, reffile, cnvfile, outfile = "rsiout.txt", chr = "1-22XY";
  bool saverd = false, hostdecode = false, crc = false, out_set = false, unsorted = false;
  int gpus = 1, threads = 8, split = 1;
  rsigpu_params P;
};

int usage() {
  fprintf(stderr,
          "Usage:\n  rsicnv rsi -f REF -b BAM [options]\n  rsicnv rsi -f REF -d RDFILE -c CHR [options]\n"
          "  rsicnv index -b BAM [-o OUT] [-crc]   write the BAI index (default BAM.bai), built on the GPU\n"
          "Options:\n   -o  STR  outputfile [rsiout.txt]\n   -c  STR  chromosome [1-22XY]\n   -m  INT  bin size, odd [101]\n"
          "   -q  INT  minimum mapping quality [0]\n   -Q  INT  minimum base quality [13]\n   -cap FLT cap depth at FLT x median, <=1 off [4]\n"
          "   -NOGC    no GC adjustment\n   -MED | -NB | -ALL  transformation [NB]\n   -s       save raw depth to <out>.<chr>_rd (BAM input)\n"
          "   -gpus INT  GPUs to shard contigs over [1]\n   -split INT  spread EVERY contig over INT GPUs instead (base ranges + halos, identical table) [1]\n   -hostdecode  inflate/parse the BAM on the host (zlib, -threads INT [8]) instead of on the GPU\n"
          "   -crc     check the CRC32 of every BGZF block the GPU decodes (the host decoder always does)\n"
          "   -unsorted  the BAM need not be coordinate-sorted (rsi, stat): records are grouped by contig while decoding and each contig's\n"
          "              reads sorted on the GPU; every contig's reads stay in GPU memory until the end of the file; the .bai is not read\n");
  return 0;
}

bool parse(int argc, char** argv, Opt* o) {
  rsigpu_default_params(&o->P);
  std::vector<std::string> a(argv, argv + argc);
  if (a.size() < 2) return false;
  if (a[1][0] != '-') {
    o->function = a[1]; a[1] = "";
    if (o->function != "rsi" && o->function != "decode" && o->function != "stat" && o->function != "index") { fprintf(stderr, "no such function %s (this build implements `rsi`, `stat` and `index`)\n", o->function.c_str()); return false; }
  }
  auto val = [&](size_t i) { return i + 1 < a.size() ? a[i + 1] : std::string(); };
  for (size_t i = 1; i < a.size(); ++i) {
    const std::string k = a[i];
    auto two = [&]() { a[i] = ""; if (i + 1 < a.size()) a[i + 1] = ""; };
    if (k == "-d") { o->rdfile = val(i); two(); continue; }
    if (k == "-b") { o->bamfile = val(i); two(); continue; }
    if (k == "-f") { o->reffile = val(i); two(); continue; }
    if (k == "-v") { o->cnvfile = val(i); two(); continue; }
    if (k == "-o") { o->outfile = val(i); o->out_set = true; two(); continue; }
    if (k == "-c") { o->chr = val(i); two(); continue; }
    if (k == "-s") { o->saverd = true; a[i] = ""; continue; }
    if (k == "-m") { o->P.m = atoi(val(i).c_str()); two(); continue; }
    if (k == "-q") { o->P.minq = atoi(val(i).c_str()); two(); continue; }
    if (k == "-Q") { o->P.min_baseQ = atoi(val(i).c_str()); two(); continue; }
    if (k == "-L" || k == "-p") { two(); continue; }                    // parsed and unused on this path (rsi.cpp:2018-2019)
    if (k == "-np" || k == "-debug" || k == "-hist" || k == "-overlap" || k == "-combine" || k == "-nocode") { a[i] = ""; continue; }
    if (k == "-threshold") { o->P.threshold = atof(val(i).c_str()); two(); continue; }
    if (k == "-e") { o->P.epsilon = atof(val(i).c_str()); two(); continue; }
    if (k == "-cap") { o->P.cap = atof(val(i).c_str()); two(); continue; }
    if (k == "-reflen") { o->P.chklen = atof(val(i).c_str()); two(); continue; }
    if (k == "-maxchkbp") { o->P.maxchkbp = atoi(val(i).c_str()); two(); continue; }
    if (k == "-MED") { o->P.trans = RSIGPU_TRANS_MED; a[i] = ""; continue; }
    if (k == "-NB") { o->P.trans = RSIGPU_TRANS_NBN; a[i] = ""; continue; }
    if (k == "-ALL") { o->P.trans = RSIGPU_TRANS_ALL; a[i] = ""; continue; }
    if (k == "-nomerge") { o->P.merge = 0; a[i] = ""; continue; }
    if (k == "-NOGC") { o->P.gcadjust = 0; a[i] = ""; continue; }
    if (k == "-gpus") { o->gpus = atoi(val(i).c_str()); two(); continue; }
    if (k == "-split") { o->split = atoi(val(i).c_str()); two(); continue; }
    if (k == "-threads") { o->threads = atoi(val(i).c_str()); two(); continue; }
    if (k == "-hostdecode") { o->hostdecode = true; a[i] = ""; continue; }
    if (k == "-crc") { o->crc = true; a[i] = ""; continue; }
    if (k == "-unsorted") { o->unsorted = true; a[i] = ""; continue; }
  }
  bool bad = false;
  for (size_t i = 1; i < a.size(); ++i) if (!a[i].empty()) { fprintf(stderr, "unknown option %s\n", a[i].c_str()); bad = true; }
  if (bad) return false;
  if (o->rdfile.empty() && o->bamfile.empty()) { fprintf(stderr, "need input file \n"); return false; }
  if (o->reffile.empty() && o->function == "rsi") { fprintf(stderr, "need reference file \n"); return false; }
  if (o->function == "stat" && (o->bamfile.empty() || o->cnvfile.empty())) { fprintf(stderr, "stat needs -b BAM and -v CNVFILE\n"); return false; }
  if (o->function == "index" && o->bamfile.empty()) { fprintf(stderr, "index needs -b BAM\n"); return false; }
  if (o->outfile == o->bamfile || o->outfile == o->rdfile) { fprintf(stderr, "output file is same as input file \n"); return false; }
  if (!o->rdfile.empty() && (o->chr.empty() || o->chr == "1-22XY")) { fprintf(stderr, "readdepth file and chromosome must be specified together\n"); return false; }
  if (o->P.m % 2 != 1) { o->P.m += 1; fprintf(stderr, "m is changed to %d\n", o->P.m); }
  return true;
}

// a context that only decodes BAM bytes (rsigpu_bam_feed), with the CRC32 check of -crc
int create_decoder(const Opt& o, int device, rsigpu_ctx** dec) {
  const int rc = rsigpu_create(device, &o.P, dec);
  if (rc) return rc;
  return rsigpu_set_bgzf_crc(*dec, o.crc ? 1 : 0);
}

// read_fasta (readref.cpp:10-86): contig `chr` or "chr"+chr through the .fai index, newlines stripped
bool read_fasta(const std::string& ref, const std::string& chr, std::string* out, std::string* err) {
  std::ifstream fai((ref + ".fai").c_str());
  if (!fai) { *err = "cannot open " + ref + ".fai"; return false; }
  std::string name; long long len = 0, off = 0, lb = 0, lw = 0; bool found = false;
  while (fai >> name >> len >> off >> lb >> lw) { if (name == chr || name == "chr" + chr) { found = true; break; } }
  if (!found) { *err = "reference has no contig " + chr; return false; }
  FILE* f = fopen(ref.c_str(), "rb");
  if (!f) { *err = "cannot open " + ref; return false; }
  const long long nbytes = len + (lb > 0 ? (len / lb) * (lw - lb) : 0);
  std::vector<char> raw((size_t)nbytes + 1);
  fseeko(f, (off_t)off, SEEK_SET);
  const size_t got = fread(raw.data(), 1, (size_t)nbytes, f);
  fclose(f);
  out->clear(); out->reserve((size_t)len);
  for (size_t i = 0; i < got && (long long)out->size() < len; ++i) if (raw[i] != '\n' && raw[i] != '\r') out->push_back(raw[i]);
  return true;
}

// load_data_from_text's parse loop (loaddata.cpp:496-517): `pos depth` lines, '#' and empty lines skipped,
// pos < 1 skipped, pos >= L ends the file, a token that is not a number reads as 0 (istream >> int)
bool parse_depth_text(const std::string& path, int L, std::vector<int32_t>* rd, std::string* err) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) { *err = "Cannot open file " + path; return false; }
  rd->assign((size_t)L, 0);
  std::vector<char> buf((size_t)64 << 20);
  std::string carry;
  bool done = false;
  auto take_int = [](const char*& p, const char* e) {
    while (p < e && (*p == ' ' || *p == '\t' || *p == '\r' || *p == '\v' || *p == '\f')) ++p;
    bool neg = false; const char* s = p;
    if (p < e && (*p == '-' || *p == '+')) { neg = *p == '-'; ++p; }
    long long v = 0; bool any = false;
    while (p < e && *p >= '0' && *p <= '9') { v = v * 10 + (*p - '0'); if (v > 0x7fffffffLL) v = 0x7fffffffLL; ++p; any = true; }
    if (!any) { p = s; return std::make_pair(0LL, false); }
    return std::make_pair(neg ? -v : v, true);
  };
  auto line = [&](const char* p, const char* e) {
    if (e - p < 1 || *p == '#') return;
    auto a = take_int(p, e);
    long long pos = a.first, d = 0;
    if (a.second) d = take_int(p, e).first;
    if (pos < 1) return;
    if (pos >= L) { done = true; return; }
    (*rd)[(size_t)pos - 1] = (int32_t)d;
  };
  while (!done) {
    const size_t got = fread(buf.data(), 1, buf.size(), f);
    if (got == 0) break;
    const char* p = buf.data(); const char* e = p + got;
    if (!carry.empty()) {
      const char* nl = (const char*)memchr(p, '\n', (size_t)(e - p));
      if (!nl) { carry.append(p, e); continue; }
      carry.append(p, nl);
      line(carry.data(), carry.data() + carry.size());
      carry.clear(); p = nl + 1;
    }
    while (!done && p < e) {
      const char* nl = (const char*)memchr(p, '\n', (size_t)(e - p));
      if (!nl) { carry.assign(p, e); break; }
      line(p, nl); p = nl + 1;
    }
  }
  if (!done && !carry.empty()) line(carry.data(), carry.data() + carry.size());
  fclose(f);
  return true;
}

struct ContigResult {
  std::string name; bool done = false; std::string err;
  std::vector<rsigpu_cnv> calls; double rdmedian = 0, rdsd = 0;
  std::string log;      // what the reference's <out>.log holds for this contig (rsigpu_get_log)
};

// <out>.log: the reference tees everything it says to stderr into it (rsi::dout, rsi.cpp:86, 2079-2098).  Reproduced: the parameter
// echo, the BAM header check, and per contig the deterministic lines of the loaders and the detector; not reproduced: the Vm*
// lines of /proc/<pid>/status.
std::string param_echo(const Opt& o, const std::string& command) {
  char tmp[64];
  std::string s = "#command:   " + command + "\n#bamfile:   " + o.bamfile + "\n#rdfile:    " + o.rdfile + "\n#reffile:   " + o.reffile + "\n#cnvfile:   " + o.cnvfile + "\n#chrom:     " + o.chr + "\n";
  snprintf(tmp, sizeof tmp, "#min_mapq:  %d\n#min_baseQ: %d\n#binsize:   %d\n#adjustGC:  %d\n", o.P.minq, o.P.min_baseQ, o.P.m, o.P.gcadjust ? 1 : 0); s += tmp;
  s += "#plots:     cnv_plots\n#output:    " + o.outfile + "\n";
  return s;
}
void contig_log(rsigpu_ctx* c, const Opt& o, const std::string& name, bool text_input, ContigResult* res) {
  int64_t n = 0;
  if (rsigpu_get_log(c, name.c_str(), text_input ? 1 : 0, nullptr, 0, &n) || n <= 0) return;
  std::string t((size_t)n, '\0');
  if (rsigpu_get_log(c, name.c_str(), text_input ? 1 : 0, &t[0], n, &n)) return;
  if (o.saverd && !text_input) {   // "RD of <chr> is saved to <file>" follows the progress line of the read loop (loaddata.cpp:338-342)
    size_t p = t.find('\n') + 1;                                  // after "#Noseq regions excluded"
    while (p < t.size() && t.compare(p, name.size() + 1, name + "\t") == 0) p = t.find('\n', p) + 1;
    p = t.find('\n', p) + 1;                                     // after the progress line
    t.insert(p, "RD of " + name + " is saved to " + o.outfile + "." + name + "_rd\n");
  }
  res->log = "#processing " + name + "\n" + t + "output written to " + o.outfile + "\n";
}

// set_reference + pileup_begin (BAM input) / set_depth (depth-file input)
bool begin_contig(rsigpu_ctx* c, int tid, const std::string& fasta, const std::vector<int32_t>* depth, ContigResult* res) {
  auto fail = [&](const char* what) { res->err = std::string(what) + ": " + rsigpu_last_error(c); return false; };
  if (rsigpu_set_reference(c, (const uint8_t*)fasta.data(), (int32_t)fasta.size(), tid)) return fail("set_reference");
  if (depth) { if (rsigpu_set_depth(c, depth->data(), (int32_t)depth->size())) return fail("set_depth"); }
  else if (rsigpu_pileup_begin(c, (int32_t)fasta.size())) return fail("pileup_begin");
  return true;
}

// everything after the inputs are staged: the body of the chromosome loop (rsi.cpp:2197-2211)
bool finish_contig(rsigpu_ctx* c, const Opt& o, const std::string& name, size_t fasta_len, bool bam, ContigResult* res) {
  auto fail = [&](const char* what) { res->err = std::string(what) + ": " + rsigpu_last_error(c); return false; };
  if (bam) {
    if (o.saverd) {
      if (rsigpu_pileup_end(c)) return fail("pileup_end");
      std::vector<int32_t> raw(fasta_len); int64_t cnt = 0;
      if (rsigpu_get_array(c, RSIGPU_ARR_RAW_DEPTH, raw.data(), (int64_t)raw.size(), &cnt)) return fail("get raw depth");
      const std::string fn = o.outfile + "." + name + "_rd";   // loaddata.cpp:340-344, 464-470
      FILE* f = fopen(fn.c_str(), "w");
      if (f) { for (size_t i = 0; i < raw.size(); ++i) fprintf(f, "%zu\t%d\n", i + 1, raw[i]); fclose(f); }
    } else if (rsigpu_pileup_commit(c)) return fail("pileup_commit");
  }
  int32_t n = 0;
  res->calls.resize(65536);
  if (rsigpu_run(c, res->calls.data(), (int32_t)res->calls.size(), &n)) return fail("run");
  res->calls.resize((size_t)n);
  rsigpu_chr_stats st;
  if (rsigpu_get_chr_stats(c, &st)) return fail("chr_stats");
  res->rdmedian = st.rdmedian; res->rdsd = st.rdsd;
  contig_log(c, o, name, !bam, res);
  return true;
}

bool run_contig(rsigpu_ctx* c, const Opt& o, const std::string& name, int tid, const std::string& fasta, const std::vector<int32_t>* depth,
                const ContigReads* reads, ContigResult* res) {
  if (!begin_contig(c, tid, fasta, depth, res)) return false;
  if (reads) {
    rsigpu_read_batch b; memset(&b, 0, sizeof b);
    b.n_reads = (int64_t)reads->n(); b.tid = tid;
    b.pos = reads->pos.data(); b.mpos = reads->mpos.data(); b.isize = reads->isize.data(); b.mtid = reads->mtid.data(); b.flag = reads->flag.data();
    b.mapq = reads->mapq.data(); b.cigar_off = reads->cigar_off.data(); b.cigar = reads->cigar.data(); b.qual_off = reads->qual_off.data(); b.qual = reads->qual.data();
    if (rsigpu_pileup_push(c, &b)) { res->err = std::string("pileup_push: ") + rsigpu_last_error(c); return false; }
  }
  return finish_contig(c, o, name, fasta.size(), reads != nullptr, res);
}

double now_s() { struct timespec t; clock_gettime(CLOCK_MONOTONIC, &t); return (double)t.tv_sec + 1e-9 * (double)t.tv_nsec; }

// which contigs of the header are processed (rsi.cpp:2116-2143): by default every contig whose name contains neither "MT"
// nor "." (and that has reads); with -c exactly the named one, whatever its name
bool eligible(const Opt& o, const std::string& name) {
  if (o.chr != "1-22XY") return name == o.chr;
  return name.find("MT") == std::string::npos && name.find(".") == std::string::npos;
}

// longest-processing-time assignment from the header lengths (SURVEY.md 8e: 1.038 imbalance for b37 on 8 GPUs)
std::vector<int> lpt_assign(const Opt& o, const BamHeader& h, int ng, const std::vector<BaiRef>* bai) {
  std::vector<int> gpu_of(h.name.size(), -1);
  std::vector<size_t> order;
  for (size_t i = 0; i < h.name.size(); ++i) if (eligible(o, h.name[i]) && (!bai || (*bai)[i].has_reads)) order.push_back(i);
  std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return h.len[a] > h.len[b]; });
  std::vector<long long> load((size_t)ng, 0);
  for (size_t i : order) { const int g = (int)(std::min_element(load.begin(), load.end()) - load.begin()); gpu_of[i] = g; load[(size_t)g] += h.len[i]; }
  return gpu_of;
}

// page-cache -> buffer with several threads (one memcpy stream of pread() tops out near 3 GB/s)
size_t parallel_pread(int fd, uint8_t* dst, size_t n, long long off, int nthreads = 4) {
  if (n < ((size_t)8 << 20)) nthreads = 1;
  std::vector<std::thread> th; std::vector<size_t> got((size_t)nthreads, 0);
  const size_t per = (n + (size_t)nthreads - 1) / (size_t)nthreads;
  for (int t = 0; t < nthreads; ++t)
    th.emplace_back([&, t]() {
      size_t a = (size_t)t * per, e = std::min(n, a + per), done = 0;
      while (a + done < e) {
        const ssize_t r = pread(fd, dst + a + done, e - a - done, (off_t)(off + (long long)(a + done)));
        if (r <= 0) break;
        done += (size_t)r;
      }
      got[(size_t)t] = done;
    });
  for (auto& x : th) x.join();
  size_t total = 0;
  for (int t = 0; t < nthreads; ++t) { total += got[(size_t)t]; if (got[(size_t)t] < std::min(n, ((size_t)t + 1) * per) - std::min(n, (size_t)t * per)) break; }
  return total;
}

// FASTA of the next contig read while the current one is being decoded
struct FastaPrefetch {
  std::string ref; std::thread th; std::string name, fasta, err; bool ok = false, busy = false;
  explicit FastaPrefetch(const std::string& r) : ref(r) {}
  ~FastaPrefetch() { if (th.joinable()) th.join(); }
  void request(const std::string& n) {
    if (th.joinable()) th.join();
    name = n; busy = true;
    th = std::thread([this]() { fasta.clear(); err.clear(); ok = read_fasta(ref, name, &fasta, &err); });
  }
  bool take(const std::string& n, std::string* out, std::string* e) {
    if (!busy || name != n) request(n);
    th.join(); busy = false;
    if (!ok) { *e = err; return false; }
    out->swap(fasta);
    return true;
  }
};

struct DecodeTiming { double feed = 0, take = 0, wait = 0, read = 0; };

// Streams a BAM file from file offset `coff` (a BGZF block boundary; `skip` decoded bytes of that block precede the first
// wanted record) through the decoder context `dec` in chunks of whole BGZF blocks read one chunk ahead.  on_run(i, run) is
// called for every run of records with one refID, in file order: 0 = go on, 1 = stop (the caller has what it wanted),
// < 0 = error.  Returns 0 (end of file or stopped), 1 on any error (message on stderr): the caller must NOT use the partial data.
template <class F>
int stream_bam(const std::string& path, long long coff, long long skip, long long end_off, rsigpu_ctx* dec, size_t chunk_bytes, F&& on_run, DecodeTiming* tm) {
  const int fd = open(path.c_str(), O_RDONLY);
  if (fd < 0) { fprintf(stderr, "cannot open %s\n", path.c_str()); return 1; }
  struct stat sb;
  if (fstat(fd, &sb) != 0 || (long long)sb.st_size < coff) { fprintf(stderr, "cannot read %s\n", path.c_str()); close(fd); return 1; }
  // end_off > 0: the BGZF block that starts there is the last one wanted (the contig's records end inside it)
  long long stop_at = (long long)sb.st_size;
  if (end_off > 0 && end_off + 18 <= (long long)sb.st_size) {
    uint8_t hb[18];
    if (pread(fd, hb, 18, (off_t)end_off) == 18 && hb[0] == 0x1f && hb[1] == 0x8b && hb[12] == 'B' && hb[13] == 'C')
      stop_at = std::min<long long>(stop_at, end_off + (long long)((unsigned)hb[16] | ((unsigned)hb[17] << 8)) + 1);
  }
  if (stop_at <= coff) stop_at = (long long)sb.st_size;
  const size_t remaining = (size_t)(stop_at - coff);
  const size_t CARRY = (size_t)1 << 20;
  const size_t CHUNK = std::max<size_t>(std::min(chunk_bytes, remaining + 1), (size_t)1 << 20);
  const bool two = remaining > CHUNK;
  uint8_t* buf[2] = {nullptr, nullptr};
  for (int k = 0; k < (two ? 2 : 1); ++k)
    if (rsigpu_pinned_alloc(CARRY + CHUNK, (void**)&buf[k])) { fprintf(stderr, "cannot allocate pinned staging memory\n"); close(fd); for (int j = 0; j < k; ++j) rsigpu_pinned_free(buf[j]); return 1; }
  auto cleanup = [&]() { for (int k = 0; k < 2; ++k) rsigpu_pinned_free(buf[k]); close(fd); };
  long long foff = coff;
  double t0 = now_s();
  size_t have = parallel_pread(fd, buf[0] + CARRY, std::min(CHUNK, remaining), foff);
  tm->read += now_s() - t0;
  foff += (long long)have;
  uint8_t* cur = buf[0] + CARRY;      // valid bytes: [cur, cur + have)
  int cb = 0; bool eof = (size_t)(foff - coff) >= remaining, first = true;
  std::vector<rsigpu_bam_run> runs(65536);          // the decoder's own limit of runs per feed
  std::thread reader; size_t next_got = 0;
  int status = 0; bool stop = false;
  while (have > 0 && !stop && !status) {
    const int nb = cb ^ 1;
    if (!eof) {
      const size_t want = std::min(CHUNK, remaining - (size_t)(foff - coff));
      reader = std::thread([&, nb, want]() { next_got = parallel_pread(fd, buf[nb] + CARRY, want, foff); });
    }
    size_t pos = 0;
    for (;;) {          // the decoder takes whole blocks up to its own limits: present the rest again until (less than) one block is left
      int64_t consumed = 0; int32_t nr = 0;
      t0 = now_s();
      const int rc = rsigpu_bam_feed(dec, cur + pos, (int64_t)(have - pos), first ? skip : 0, &consumed, runs.data(), (int32_t)runs.size(), &nr);
      tm->feed += now_s() - t0;
      if (rc) { fprintf(stderr, "%s\n", rsigpu_last_error(dec)); status = 1; break; }
      if (nr > (int32_t)runs.size()) { fprintf(stderr, "more than %zu reference runs in one chunk of %s\n", runs.size(), path.c_str()); status = 1; break; }
      if (consumed) first = false;
      t0 = now_s();
      for (int i = 0; i < nr && !stop && !status; ++i) {
        const int r = on_run(i, runs[(size_t)i]);
        if (r > 0) stop = true; else if (r < 0) status = 1;
      }
      tm->take += now_s() - t0;
      pos += (size_t)consumed;
      if (stop || status || consumed == 0 || have - pos < ((size_t)1 << 17)) break;
    }
    const size_t rest = have - pos;
    if (reader.joinable()) reader.join();
    if (stop || status) break;
    if (eof) {
      if (rest) { fprintf(stderr, "truncated BGZF block at the end of %s\n", path.c_str()); status = 1; }
      break;
    }
    if (rest > CARRY) { fprintf(stderr, "%s: a BGZF block sequence the decoder cannot take (%zu bytes left over)\n", path.c_str(), rest); status = 1; break; }
    memcpy(buf[nb] + CARRY - rest, cur + pos, rest);
    cur = buf[nb] + CARRY - rest; have = rest + next_got;
    foff += (long long)next_got;
    if ((size_t)(foff - coff) >= remaining || next_got == 0) eof = true;
    cb = nb;
  }
  if (reader.joinable()) reader.join();
  // the whole FILE was consumed without being stopped: it must not end inside a record (a bounded range ends where the index says)
  if (!status && !stop && stop_at == (long long)sb.st_size && rsigpu_bam_end(dec)) { fprintf(stderr, "%s\n", rsigpu_last_error(dec)); status = 1; }
  cleanup();
  return status;
}

// `-split N`: one contig over N GPUs (rsigpu_split_run).  parts[g] = the context on GPU g; every part gets the whole FASTA and
// the reads of its own base range (+ halo); the lead (GPU 0) ends up with the calls.
bool split_finish(const Opt& o, std::vector<rsigpu_ctx*>& parts, const std::string& name, bool bam, ContigResult* res) {
  auto fail = [&](const char* what) { res->err = std::string(what) + ": " + rsigpu_last_error(parts[0]); return false; };
  if (bam) for (rsigpu_ctx* p : parts) if (rsigpu_pileup_commit(p)) return fail("pileup_commit");
  int32_t n = 0;
  res->calls.resize(65536);
  if (rsigpu_split_run(parts.data(), (int32_t)parts.size(), res->calls.data(), (int32_t)res->calls.size(), &n)) return fail("split_run");
  res->calls.resize((size_t)n);
  rsigpu_chr_stats st;
  if (rsigpu_get_chr_stats(parts[0], &st)) return fail("chr_stats");
  res->rdmedian = st.rdmedian; res->rdsd = st.rdsd;
  contig_log(parts[0], o, name, !bam, res);
  if (getenv("RSICNV_TIMING")) fprintf(stderr, "#timing: %s split over %zu GPUs, %lld bytes crossed between devices\n", name.c_str(), parts.size(), rsigpu_split_p2p_bytes(parts[0]));
  return true;
}
int bam_split_on_gpu(const Opt& o, std::vector<rsigpu_ctx*>& parts, std::vector<ContigResult>* results_out) {
  std::string err; long long coff = 0, skip = 0;
  BamHeader h;
  if (!read_bam_header(o.bamfile, &h, &coff, &skip, &err)) { fprintf(stderr, "%s\n", err.c_str()); return 1; }
  std::vector<ContigResult>& results = *results_out;
  results.resize(h.name.size());
  for (size_t i = 0; i < h.name.size(); ++i) results[i].name = h.name[i];
  if (o.chr != "1-22XY" && std::find(h.name.begin(), h.name.end(), o.chr) == h.name.end()) { fprintf(stderr, "BAM file doesn't have %s\n", o.chr.c_str()); return 0; }
  const int n_ref = (int)h.name.size(), np = (int)parts.size();
  std::vector<BaiRef> bai;
  const bool indexed = !getenv("RSICNV_NO_INDEX") && read_bai(o.bamfile, h.name.size(), &bai);
  rsigpu_ctx* dec = nullptr;
  if (create_decoder(o, 0, &dec)) { fprintf(stderr, "cannot create the decoder context\n"); return 2; }
  DecodeTiming tm; int failed = 0;
  std::vector<int32_t> pbeg((size_t)np), pend((size_t)np); int32_t halo = 0;
  auto start = [&](int tid) -> bool {      // FASTA to every part, read staging opened
    ContigResult& r = results[(size_t)tid];
    fprintf(stderr, "#processing %s on %d GPUs\n", r.name.c_str(), np);
    std::string fasta, e2;
    if (!read_fasta(o.reffile, r.name, &fasta, &e2)) { r.err = e2; fprintf(stderr, "%s: %s\n", r.name.c_str(), e2.c_str()); ++failed; return false; }
    for (int g = 0; g < np; ++g) {
      if (rsigpu_split_range((int32_t)fasta.size(), np, g, &pbeg[(size_t)g], &pend[(size_t)g], &halo)) { fprintf(stderr, "%s: too short to be split over %d GPUs\n", r.name.c_str(), np); ++failed; return false; }
      if (!begin_contig(parts[(size_t)g], tid, fasta, nullptr, &r)) { fprintf(stderr, "%s: %s\n", r.name.c_str(), r.err.c_str()); ++failed; return false; }
    }
    return true;
  };
  auto take = [&](int i, int tid) -> bool {
    for (int g = 0; g < np; ++g)
      if (rsigpu_bam_take_range(dec, i, parts[(size_t)g], pbeg[(size_t)g] - halo, pend[(size_t)g])) { fprintf(stderr, "%s: %s\n", results[(size_t)tid].name.c_str(), rsigpu_last_error(parts[(size_t)g])); return false; }
    return true;
  };
  auto finish = [&](int tid) {
    ContigResult& r = results[(size_t)tid];
    r.done = split_finish(o, parts, r.name, true, &r);
    if (!r.done) { fprintf(stderr, "%s: %s\n", r.name.c_str(), r.err.c_str()); ++failed; }
  };
  if (indexed) {
    for (int tid = 0; tid < n_ref; ++tid) {
      if (!eligible(o, h.name[(size_t)tid]) || !bai[(size_t)tid].has_reads) continue;
      if (!start(tid) || rsigpu_bam_begin(dec, (int32_t)n_ref)) continue;
      const uint64_t v = bai[(size_t)tid].first_voff;
      uint64_t ve = bai[(size_t)tid].end_voff;
      if (!ve) for (int t = tid + 1; t < n_ref; ++t) if (bai[(size_t)t].has_reads) { ve = bai[(size_t)t].first_voff; break; }
      bool bad = false;
      const int rc = stream_bam(o.bamfile, (long long)(v >> 16), (long long)(v & 0xffff), ve ? (long long)(ve >> 16) : 0, dec, (size_t)1 << 30, [&](int i, const rsigpu_bam_run& run) {
        if (run.tid != tid) return 1;
        if (!take(i, tid)) { bad = true; return -1; }
        return 0;
      }, &tm);
      if (rc || bad) { fprintf(stderr, "%s: BAM decoding failed\n", h.name[(size_t)tid].c_str()); ++failed; continue; }
      finish(tid);
    }
  } else {
    if (rsigpu_bam_begin(dec, (int32_t)n_ref)) { fprintf(stderr, "%s\n", rsigpu_last_error(dec)); return 2; }
    int cur = -1; bool cur_ok = false;
    const int rc = stream_bam(o.bamfile, coff, skip, 0, dec, (size_t)256 << 20, [&](int i, const rsigpu_bam_run& run) {
      if (run.tid < 0) return 1;
      if (run.tid != cur) {
        if (cur >= 0 && cur_ok) finish(cur);
        cur = run.tid; cur_ok = eligible(o, h.name[(size_t)cur]) && start(cur);
      }
      if (cur_ok && !take(i, cur)) { cur_ok = false; ++failed; }
      return 0;
    }, &tm);
    if (rc) ++failed;
    else if (cur >= 0 && cur_ok) finish(cur);
  }
  rsigpu_destroy(dec);
  return failed ? 1 : 0;
}

// BAM input decoded on the GPU (rsigpu_bam_feed: BGZF inflate + record decoding, k_bam.cuh).
//   With the .bai index (which the reference requires, rsi.cpp:2112-2113): every GPU owns the contigs LPT gives it, seeks to the
//   first record of each (virtual offset from the index) and runs its OWN decoder -- reading, decoding and the hot path of
//   different GPUs never meet.  Per GPU two contig contexts alternate: contig k+1 is decoded while contig k is in the hot path,
//   and the FASTA of contig k+1 is read while contig k is decoded.
//   Without an index: one pass over the file with the decoder on GPU 0; each run of records is appended to the context of the
//   owning GPU (device-to-device, rsigpu_bam_take).
// Any decoder error fails the contig being decoded: its rows are not written and the exit status is non-zero.
int bam_on_gpu(const Opt& o, const std::vector<std::vector<rsigpu_ctx*>>& ctx, std::vector<ContigResult>* results_out) {
  const bool timing = getenv("RSICNV_TIMING") != nullptr;
  const double t_start = now_s();
  std::string err;
  long long coff = 0, skip = 0;
  BamHeader h;
  if (!read_bam_header(o.bamfile, &h, &coff, &skip, &err)) { fprintf(stderr, "%s\n", err.c_str()); return 1; }
  std::vector<ContigResult>& results = *results_out;
  results.resize(h.name.size());
  for (size_t i = 0; i < h.name.size(); ++i) results[i].name = h.name[i];
  if (o.chr != "1-22XY" && std::find(h.name.begin(), h.name.end(), o.chr) == h.name.end()) { fprintf(stderr, "BAM file doesn't have %s\n", o.chr.c_str()); return 0; }
  const int ng = (int)ctx.size(), n_ref = (int)h.name.size();
  std::vector<BaiRef> bai;
  const bool indexed = !getenv("RSICNV_NO_INDEX") && read_bai(o.bamfile, h.name.size(), &bai);
  const std::vector<int> gpu_of = lpt_assign(o, h, ng, indexed ? &bai : nullptr);
  std::mutex mu;
  std::atomic<int> failed(0);
  const size_t CHUNK = (size_t)1 << 30;
  auto fail_contig = [&](int tid, const std::string& what) {
    std::lock_guard<std::mutex> lk(mu);
    results[(size_t)tid].err = what; results[(size_t)tid].done = false;
    fprintf(stderr, "%s: %s\n", results[(size_t)tid].name.c_str(), what.c_str());
    failed++;
  };
  auto finish_async = [&](std::thread* slot, rsigpu_ctx* c, int tid, size_t flen) {
    *slot = std::thread([&, c, tid, flen]() {
      ContigResult& r = results[(size_t)tid];
      r.done = finish_contig(c, o, r.name, flen, true, &r);
      if (!r.done) { std::lock_guard<std::mutex> lk(mu); fprintf(stderr, "%s: %s\n", r.name.c_str(), r.err.c_str()); failed++; }
    });
  };
  std::vector<DecodeTiming> tms((size_t)ng);
  if (indexed) {
    std::vector<std::thread> lanes;
    for (int g = 0; g < ng; ++g)
      lanes.emplace_back([&, g]() {
        std::vector<int> tids;
        for (int t = 0; t < n_ref; ++t) if (gpu_of[(size_t)t] == g) tids.push_back(t);
        if (tids.empty()) return;
        rsigpu_ctx* dec = nullptr;
        if (create_decoder(o, g, &dec)) { for (int t : tids) fail_contig(t, "cannot create the decoder context"); return; }
        FastaPrefetch fp(o.reffile);
        fp.request(h.name[(size_t)tids[0]]);
        std::thread fin[2];
        for (size_t k = 0; k < tids.size(); ++k) {
          const int tid = tids[k]; const size_t slot = k % ctx[(size_t)g].size();
          rsigpu_ctx* c = ctx[(size_t)g][slot];
          double t0 = now_s();
          if (fin[slot & 1].joinable()) fin[slot & 1].join();
          tms[(size_t)g].wait += now_s() - t0;
          ContigResult& r = results[(size_t)tid];
          { std::lock_guard<std::mutex> lk(mu); fprintf(stderr, "#processing %s on GPU %d\n", r.name.c_str(), g); }
          std::string fasta, e2;
          const bool got = fp.take(r.name, &fasta, &e2);
          if (k + 1 < tids.size()) fp.request(h.name[(size_t)tids[k + 1]]);
          if (!got) { fail_contig(tid, e2); continue; }
          if ((int)fasta.size() != h.len[(size_t)tid]) fprintf(stderr, "reference and target not same size %zu\t%d\n", fasta.size(), h.len[(size_t)tid]);
          if (!begin_contig(c, tid, fasta, nullptr, &r)) { fail_contig(tid, r.err); continue; }
          if (rsigpu_bam_begin(dec, (int32_t)n_ref)) { fail_contig(tid, rsigpu_last_error(dec)); continue; }
          const uint64_t v = bai[(size_t)tid].first_voff;
          // the contig's byte range: up to the block where its last record ends (pseudo-bin), else where the next contig with reads starts
          uint64_t ve = bai[(size_t)tid].end_voff;
          if (!ve) for (int t = tid + 1; t < n_ref; ++t) if (bai[(size_t)t].has_reads) { ve = bai[(size_t)t].first_voff; break; }
          bool take_err = false;
          const int rc = stream_bam(o.bamfile, (long long)(v >> 16), (long long)(v & 0xffff), ve ? (long long)(ve >> 16) : 0, dec, CHUNK, [&](int i, const rsigpu_bam_run& run) {
            if (run.tid != tid) return 1;                         // the next contig (or the unplaced reads) begins: done
            if (rsigpu_bam_take(dec, i, c)) { take_err = true; return -1; }
            return 0;
          }, &tms[(size_t)g]);
          if (rc || take_err) { fail_contig(tid, take_err ? std::string("bam_take: ") + rsigpu_last_error(c) : "BAM decoding failed"); continue; }
          finish_async(&fin[slot & 1], c, tid, fasta.size());
        }
        for (auto& f : fin) if (f.joinable()) f.join();
        rsigpu_destroy(dec);
      });
    for (auto& l : lanes) l.join();
  } else {
    rsigpu_ctx* dec = nullptr;
    if (create_decoder(o, 0, &dec)) { fprintf(stderr, "cannot create the decoder context\n"); return 2; }
    if (rsigpu_bam_begin(dec, (int32_t)n_ref)) { fprintf(stderr, "%s\n", rsigpu_last_error(dec)); return 2; }
    std::vector<std::vector<std::thread>> fin((size_t)ng);
    for (int g = 0; g < ng; ++g) fin[(size_t)g].resize(ctx[(size_t)g].size());
    std::vector<size_t> next_slot((size_t)ng, 0);
    FastaPrefetch fp(o.reffile);
    int cur = -1; bool cur_ok = false; size_t cur_len = 0, cur_slot = 0;
    auto finish_cur = [&]() {
      if (cur >= 0 && cur_ok) { const int g = gpu_of[(size_t)cur]; finish_async(&fin[(size_t)g][cur_slot], ctx[(size_t)g][cur_slot], cur, cur_len); }
      cur = -1; cur_ok = false;
    };
    auto start = [&](int tid) {
      cur = tid; cur_ok = false;
      if (gpu_of[(size_t)tid] < 0) return;
      const int g = gpu_of[(size_t)tid];
      cur_slot = next_slot[(size_t)g]++ % ctx[(size_t)g].size();
      double t0 = now_s();
      if (fin[(size_t)g][cur_slot].joinable()) fin[(size_t)g][cur_slot].join();
      tms[0].wait += now_s() - t0;
      ContigResult& r = results[(size_t)tid];
      fprintf(stderr, "#processing %s on GPU %d\n", r.name.c_str(), g);
      std::string fasta, e2;
      const bool got = fp.take(r.name, &fasta, &e2);
      for (int t = tid + 1; t < n_ref; ++t) if (gpu_of[(size_t)t] >= 0) { fp.request(h.name[(size_t)t]); break; }   // the next eligible contig, in header order
      if (!got) { fail_contig(tid, e2); return; }
      if ((int)fasta.size() != h.len[(size_t)tid]) fprintf(stderr, "reference and target not same size %zu\t%d\n", fasta.size(), h.len[(size_t)tid]);
      cur_len = fasta.size();
      if (!begin_contig(ctx[(size_t)g][cur_slot], tid, fasta, nullptr, &r)) { fail_contig(tid, r.err); return; }
      cur_ok = true;
    };
    const int rc = stream_bam(o.bamfile, coff, skip, 0, dec, (size_t)256 << 20, [&](int i, const rsigpu_bam_run& run) {
      if (run.tid < 0) return 1;                                 // unplaced reads come last in a sorted BAM
      if (run.tid != cur) { finish_cur(); start(run.tid); }
      if (cur_ok && rsigpu_bam_take(dec, i, ctx[(size_t)gpu_of[(size_t)cur]][cur_slot])) {
        fail_contig(cur, std::string("bam_take: ") + rsigpu_last_error(ctx[(size_t)gpu_of[(size_t)cur]][cur_slot])); cur_ok = false;
      }
      return 0;
    }, &tms[0]);
    if (rc) {   // the contig being decoded is incomplete: never turn partial depth into calls
      if (cur >= 0 && cur_ok) fail_contig(cur, "BAM decoding failed inside this contig");
      else failed++;
      cur = -1; cur_ok = false;
    }
    finish_cur();
    for (auto& v : fin) for (auto& f : v) if (f.joinable()) f.join();
    rsigpu_destroy(dec);
  }
  if (timing) {
    DecodeTiming t;
    for (const DecodeTiming& x : tms) { t.feed += x.feed; t.take += x.take; t.wait += x.wait; t.read += x.read; }
    fprintf(stderr, "#timing: %s decode, header+index %.3f s, decode loop %.3f s (first read %.3f, bam_feed %.3f, take %.3f, waiting for the GPU %.3f; summed over %d lanes)\n",
            indexed ? "indexed per-GPU" : "sequential", 0.0, now_s() - t_start, t.read, t.feed, t.take, t.wait, indexed ? ng : 1);
  }
  return failed.load() ? 1 : 0;
}

// `-unsorted`: a BAM in any record order (an aligner's input or name order).  The decoder on GPU 0 groups every feed's records by
// refID (rsigpu_set_bam_by_ref); each run of an eligible contig is appended to one staging context on the contig's GPU and noted as a
// (r0, r1) segment of it.  At the end of the file every GPU runs its contigs, its two contexts alternating: the contig's segments
// are moved over (rsigpu_reads_take), sorted by position, stable in file order (rsigpu_pileup_sort), and run as usual -- what the
// sorted route computes on the same file after a stable coordinate sort.  Unlike the sorted route, every contig's reads stay in
// GPU memory until the end of the file.  A contig whose reads could not all be staged, or a file that cannot be read to its end,
// fails with its name on stderr and no rows: never calls from part of a contig's reads.  The .bai is not read.
int bam_unsorted_on_gpu(const Opt& o, const std::vector<std::vector<rsigpu_ctx*>>& ctx, std::vector<ContigResult>* results_out) {
  const bool timing = getenv("RSICNV_TIMING") != nullptr;
  const double t_start = now_s();
  std::string err;
  long long coff = 0, skip = 0;
  BamHeader h;
  if (!read_bam_header(o.bamfile, &h, &coff, &skip, &err)) { fprintf(stderr, "%s\n", err.c_str()); return 1; }
  std::vector<ContigResult>& results = *results_out;
  results.resize(h.name.size());
  for (size_t i = 0; i < h.name.size(); ++i) results[i].name = h.name[i];
  if (o.chr != "1-22XY" && std::find(h.name.begin(), h.name.end(), o.chr) == h.name.end()) { fprintf(stderr, "BAM file doesn't have %s\n", o.chr.c_str()); return 0; }
  const int ng = (int)ctx.size(), n_ref = (int)h.name.size();
  const std::vector<int> gpu_of = lpt_assign(o, h, ng, nullptr);
  std::mutex mu;
  std::atomic<int> failed(0);
  auto fail_contig = [&](int tid, const std::string& what) {
    std::lock_guard<std::mutex> lk(mu);
    results[(size_t)tid].err = what; results[(size_t)tid].done = false;
    fprintf(stderr, "%s: %s\n", results[(size_t)tid].name.c_str(), what.c_str());
    failed++;
  };
  std::vector<rsigpu_ctx*> stage((size_t)ng, nullptr);
  auto destroy_all = [&]() { for (rsigpu_ctx*& s : stage) { rsigpu_destroy(s); s = nullptr; } };
  for (int g = 0; g < ng; ++g)
    if (rsigpu_create(g, &o.P, &stage[(size_t)g]) || rsigpu_reads_begin(stage[(size_t)g], 0, 1)) {
      fprintf(stderr, "cannot create the staging context on GPU %d\n", g); destroy_all(); return 2;
    }
  rsigpu_ctx* dec = nullptr;
  if (create_decoder(o, 0, &dec) || rsigpu_set_bam_by_ref(dec, 1) || rsigpu_bam_begin(dec, (int32_t)n_ref)) {
    fprintf(stderr, "%s\n", dec ? rsigpu_last_error(dec) : "cannot create the decoder context"); rsigpu_destroy(dec); destroy_all(); return 2;
  }
  std::vector<std::vector<std::pair<int64_t, int64_t>>> seg((size_t)n_ref);
  std::vector<int64_t> staged((size_t)ng, 0);
  std::vector<std::string> stage_err((size_t)ng);   // non-empty: GPU g's staged reads are incomplete, every contig of it fails
  DecodeTiming tm;
  const int rc = stream_bam(o.bamfile, coff, skip, 0, dec, (size_t)256 << 20, [&](int i, const rsigpu_bam_run& run) {
    if (run.tid < 0 || gpu_of[(size_t)run.tid] < 0) return 0;    // unplaced, or not processed: the file goes on
    const int g = gpu_of[(size_t)run.tid];
    if (!stage_err[(size_t)g].empty()) return 0;
    if (rsigpu_bam_take(dec, i, stage[(size_t)g])) { stage_err[(size_t)g] = rsigpu_last_error(stage[(size_t)g]); return 0; }
    seg[(size_t)run.tid].emplace_back(staged[(size_t)g], staged[(size_t)g] + run.n_reads);
    staged[(size_t)g] += run.n_reads;
    return 0;
  }, &tm);
  rsigpu_destroy(dec);
  const double t_decoded = now_s();
  for (int t = 0; t < n_ref; ++t) {
    const int g = gpu_of[(size_t)t];
    if (g < 0) continue;
    if (rc) { if (!seg[(size_t)t].empty()) fail_contig(t, "the BAM file could not be decoded to its end: with -unsorted every contig may be incomplete"); }
    else if (!stage_err[(size_t)g].empty())
      fail_contig(t, "-unsorted keeps the reads of all contigs of GPU " + std::to_string(g) + " in one staging context until the end of the file, and staging them failed (" +
                     stage_err[(size_t)g] + "); more GPUs (-gpus) spread them");
  }
  if (rc) failed++;
  std::vector<std::thread> lanes;
  for (int g = 0; g < ng && !rc; ++g)
    lanes.emplace_back([&, g]() {
      std::vector<int> tids;
      if (stage_err[(size_t)g].empty()) for (int t = 0; t < n_ref; ++t) if (gpu_of[(size_t)t] == g && !seg[(size_t)t].empty()) tids.push_back(t);
      FastaPrefetch fp(o.reffile);
      if (!tids.empty()) fp.request(h.name[(size_t)tids[0]]);
      std::thread fin[2];
      for (size_t k = 0; k < tids.size(); ++k) {
        const int tid = tids[k]; const size_t slot = k % ctx[(size_t)g].size();
        rsigpu_ctx* c = ctx[(size_t)g][slot];
        if (fin[slot & 1].joinable()) fin[slot & 1].join();
        ContigResult& r = results[(size_t)tid];
        { std::lock_guard<std::mutex> lk(mu); fprintf(stderr, "#processing %s on GPU %d\n", r.name.c_str(), g); }
        std::string fasta, e2;
        const bool got = fp.take(r.name, &fasta, &e2);
        if (k + 1 < tids.size()) fp.request(h.name[(size_t)tids[k + 1]]);
        if (!got) { fail_contig(tid, e2); continue; }
        if ((int)fasta.size() != h.len[(size_t)tid]) fprintf(stderr, "reference and target not same size %zu\t%d\n", fasta.size(), h.len[(size_t)tid]);
        if (!begin_contig(c, tid, fasta, nullptr, &r)) { fail_contig(tid, r.err); continue; }
        std::string what;
        for (const auto& sg : seg[(size_t)tid])
          if (rsigpu_reads_take(stage[(size_t)g], sg.first, sg.second, c)) { what = std::string("reads_take: ") + rsigpu_last_error(c); break; }
        if (what.empty() && rsigpu_pileup_sort(c)) what = std::string("pileup_sort: ") + rsigpu_last_error(c);
        if (!what.empty()) { fail_contig(tid, what); continue; }
        const size_t flen = fasta.size();
        fin[slot & 1] = std::thread([&, c, tid, flen]() {
          ContigResult& rr = results[(size_t)tid];
          rr.done = finish_contig(c, o, rr.name, flen, true, &rr);
          if (!rr.done) { std::lock_guard<std::mutex> lk(mu); fprintf(stderr, "%s: %s\n", rr.name.c_str(), rr.err.c_str()); failed++; }
        });
      }
      for (auto& f : fin) if (f.joinable()) f.join();
    });
  for (auto& l : lanes) l.join();
  destroy_all();
  if (timing) {
    int64_t total = 0; for (int64_t x : staged) total += x;
    fprintf(stderr, "#timing: -unsorted decode + staging %.3f s (%lld reads staged; first read %.3f, bam_feed %.3f, take %.3f), contigs %.3f s\n",
            t_decoded - t_start, (long long)total, tm.read, tm.feed, tm.take, now_s() - t_decoded);
  }
  return failed.load() ? 1 : 0;
}

// `rsicnv stat -b BAM -v CNVFILE -o OUT` (rsi.cpp:2235-2249): every line of CNVFILE that names a call (read_cnvlist,
// loaddata.cpp:606-673: >= 5 characters, not a comment, >= 4 fields RNAME START END TYPE) is written back followed by
// RP=<supporting read pairs>;Q0=<fraction of mapq-0 reads> (cnv_stat, pairrd.cpp:622-748).  The reads of every contig that
// has calls are decoded on the GPU (from the .bai offset of the contig, or in one pass over the file without an index).
bool ci_has(const std::string& hay, const char* needle) {
  std::string h = hay; for (char& ch : h) ch = (char)tolower((unsigned char)ch);
  return h.find(needle) != std::string::npos;
}
int do_stat(const Opt& o, rsigpu_ctx* c) {
  std::string err; long long coff = 0, skip = 0;
  BamHeader h;
  if (!read_bam_header(o.bamfile, &h, &coff, &skip, &err)) { fprintf(stderr, "%s\n", err.c_str()); return 1; }
  std::ifstream in(o.cnvfile.c_str());
  if (!in) { fprintf(stderr, "File %s not exist\n", o.cnvfile.c_str()); return 0; }
  std::vector<rsigpu_cnv> list; std::vector<std::string> lines;
  std::string ln;
  while (std::getline(in, ln)) {
    if (ln.size() < 5 || ln[0] == '#') continue;
    std::vector<std::string> cell; { size_t p = 0; while (p < ln.size()) { while (p < ln.size() && isspace((unsigned char)ln[p])) ++p; size_t q = p; while (q < ln.size() && !isspace((unsigned char)ln[q])) ++q; if (q > p) cell.push_back(ln.substr(p, q - p)); p = q; } }
    if (cell.size() < 4) { fprintf(stderr, "skipping lines with less than 4 fields\nexpecting RNAME cnv_begin_pos cnv_end_pos cnv_type in each line\n"); continue; }
    rsigpu_cnv x; memset(&x, 0, sizeof x);
    x.tid = -1; x.type = RSIGPU_TYPE_UNKNOWN; x.p1 = x.p2 = 1.0; x.q0 = -1.0; x.rp = -1;
    for (size_t t = 0; t < h.name.size(); ++t) if (h.name[t] == cell[0]) { x.tid = (int32_t)t; break; }
    x.start = atoi(cell[1].c_str()); x.end = atoi(cell[2].c_str());
    if (ci_has(cell[3], "del")) x.type = RSIGPU_TYPE_DEL;
    if (ci_has(cell[3], "loss")) x.type = RSIGPU_TYPE_DEL;
    if (ci_has(cell[3], "dup")) x.type = RSIGPU_TYPE_DUP;
    if (ci_has(cell[3], "gain")) x.type = RSIGPU_TYPE_DUP;
    if (ci_has(cell[3], "add")) x.type = RSIGPU_TYPE_DUP;
    list.push_back(x); lines.push_back(ln);
  }
  if (list.empty()) { fprintf(stderr, "I can't find any CNV from %s\n", o.cnvfile.c_str()); return 0; }
  const int n_ref = (int)h.name.size();
  std::vector<char> wanted((size_t)n_ref, 0);
  for (const rsigpu_cnv& x : list) if (x.tid >= 0) wanted[(size_t)x.tid] = 1;
  rsigpu_ctx* dec = nullptr;
  if (create_decoder(o, 0, &dec)) { fprintf(stderr, "cannot create the decoder context\n"); return 2; }
  std::vector<BaiRef> bai;
  const bool indexed = !getenv("RSICNV_NO_INDEX") && read_bai(o.bamfile, h.name.size(), &bai);
  DecodeTiming tm;
  int failed = 0;
  auto stat_contig = [&](int tid) {
    if (rsigpu_stat_calls(c, list.data(), (int32_t)list.size())) { fprintf(stderr, "%s: %s\n", h.name[(size_t)tid].c_str(), rsigpu_last_error(c)); ++failed; }
  };
  if (o.unsorted) {   // records grouped by refID while decoding into one staging context, then per contig moved over and sorted
    rsigpu_ctx* stage = nullptr;
    if (rsigpu_create(0, &o.P, &stage) || rsigpu_reads_begin(stage, 0, 1) || rsigpu_set_bam_by_ref(dec, 1) || rsigpu_bam_begin(dec, (int32_t)n_ref)) {
      fprintf(stderr, "%s\n", stage ? rsigpu_last_error(dec) : "cannot create the staging context"); rsigpu_destroy(stage); rsigpu_destroy(dec); return 2;
    }
    std::vector<std::vector<std::pair<int64_t, int64_t>>> seg((size_t)n_ref);
    int64_t staged = 0; std::string stage_err;
    const int rc = stream_bam(o.bamfile, coff, skip, 0, dec, (size_t)256 << 20, [&](int i, const rsigpu_bam_run& run) {
      if (run.tid < 0 || !wanted[(size_t)run.tid] || !stage_err.empty()) return 0;
      if (rsigpu_bam_take(dec, i, stage)) { stage_err = rsigpu_last_error(stage); return 0; }
      seg[(size_t)run.tid].emplace_back(staged, staged + run.n_reads); staged += run.n_reads;
      return 0;
    }, &tm);
    if (rc) ++failed;
    else if (!stage_err.empty()) { fprintf(stderr, "-unsorted keeps the reads of every contig with calls in one staging context until the end of the file, and staging them failed (%s)\n", stage_err.c_str()); ++failed; }
    else
      for (int tid = 0; tid < n_ref; ++tid) {
        if (seg[(size_t)tid].empty()) continue;
        fprintf(stderr, "#sampling %s\n", h.name[(size_t)tid].c_str());
        bool ok = rsigpu_reads_begin(c, tid, h.len[(size_t)tid]) == 0;
        for (size_t k = 0; ok && k < seg[(size_t)tid].size(); ++k) ok = rsigpu_reads_take(stage, seg[(size_t)tid][k].first, seg[(size_t)tid][k].second, c) == 0;
        if (ok) ok = rsigpu_pileup_sort(c) == 0;
        if (!ok) { fprintf(stderr, "%s: %s\n", h.name[(size_t)tid].c_str(), rsigpu_last_error(c)); ++failed; continue; }
        stat_contig(tid);
      }
    rsigpu_destroy(stage);
  } else if (indexed) {
    for (int tid = 0; tid < n_ref; ++tid) {
      if (!wanted[(size_t)tid] || !bai[(size_t)tid].has_reads) continue;
      fprintf(stderr, "#sampling %s\n", h.name[(size_t)tid].c_str());
      if (rsigpu_reads_begin(c, tid, h.len[(size_t)tid]) || rsigpu_bam_begin(dec, (int32_t)n_ref)) { fprintf(stderr, "%s\n", rsigpu_last_error(c)); ++failed; continue; }
      const uint64_t v = bai[(size_t)tid].first_voff;
      uint64_t ve = bai[(size_t)tid].end_voff;
      if (!ve) for (int t = tid + 1; t < n_ref; ++t) if (bai[(size_t)t].has_reads) { ve = bai[(size_t)t].first_voff; break; }
      bool take_err = false;
      const int rc = stream_bam(o.bamfile, (long long)(v >> 16), (long long)(v & 0xffff), ve ? (long long)(ve >> 16) : 0, dec, (size_t)1 << 30, [&](int i, const rsigpu_bam_run& run) {
        if (run.tid != tid) return 1;
        if (rsigpu_bam_take(dec, i, c)) { take_err = true; return -1; }
        return 0;
      }, &tm);
      if (rc || take_err) { fprintf(stderr, "%s: BAM decoding failed\n", h.name[(size_t)tid].c_str()); ++failed; continue; }
      stat_contig(tid);
    }
  } else {
    if (rsigpu_bam_begin(dec, (int32_t)n_ref)) { fprintf(stderr, "%s\n", rsigpu_last_error(dec)); return 2; }
    int cur = -1; bool cur_ok = false;
    const int rc = stream_bam(o.bamfile, coff, skip, 0, dec, (size_t)256 << 20, [&](int i, const rsigpu_bam_run& run) {
      if (run.tid < 0) return 1;
      if (run.tid != cur) {
        if (cur >= 0 && cur_ok) stat_contig(cur);
        cur = run.tid; cur_ok = false;
        if (wanted[(size_t)cur]) { fprintf(stderr, "#sampling %s\n", h.name[(size_t)cur].c_str()); cur_ok = rsigpu_reads_begin(c, cur, h.len[(size_t)cur]) == 0; }
      }
      if (cur_ok && rsigpu_bam_take(dec, i, c)) { fprintf(stderr, "%s: %s\n", h.name[(size_t)cur].c_str(), rsigpu_last_error(c)); cur_ok = false; ++failed; }
      return 0;
    }, &tm);
    if (rc) ++failed;
    else if (cur >= 0 && cur_ok) stat_contig(cur);
  }
  rsigpu_destroy(dec);
  FILE* f = fopen(o.outfile.c_str(), "w");
  if (!f) { fprintf(stderr, "cannot write %s\n", o.outfile.c_str()); return 1; }
  for (size_t i = 0; i < list.size(); ++i) fprintf(f, "%s\tRP=%d;Q0=%g\n", lines[i].c_str(), list[i].rp, list[i].q0);
  fclose(f);
  return failed ? 1 : 0;
}

void write_table(const Opt& o, const std::vector<ContigResult>& all) {
  FILE* f = fopen(o.outfile.c_str(), "w");
  if (!f) { fprintf(stderr, "cannot write %s\n", o.outfile.c_str()); return; }
  char row[2048];
  bool header = false;
  for (const ContigResult& r : all) {
    if (!r.done) continue;
    if (!header) {   // write_cnv_to_file prints the header with the first processed contig (rsi.cpp:1598-1607)
      if (!o.rdfile.empty()) fprintf(f, "#input %s %s\n", o.rdfile.c_str(), r.name.c_str());
      if (!o.bamfile.empty()) fprintf(f, "#input %s\n", o.bamfile.c_str());
      if (o.P.gcadjust) fprintf(f, "#GC adjusted\n");
      rsigpu_format_row(nullptr, "", 0, 0, row, sizeof row);
      fprintf(f, "%s\n", row);
      header = true;
    }
    for (const rsigpu_cnv& c : r.calls) { rsigpu_format_row(&c, r.name.c_str(), r.rdmedian, r.rdsd, row, sizeof row); fprintf(f, "%s\n", row); }
  }
  fclose(f);
}

void write_log(const Opt& o, const std::string& command, const std::vector<ContigResult>& all, const std::string& bam_check) {
  FILE* f = fopen((o.outfile + ".log").c_str(), "w");
  if (!f) return;
  const std::string echo = param_echo(o, command);
  fputs(echo.c_str(), f);
  fputs(bam_check.c_str(), f);
  for (const ContigResult& r : all) if (r.done) fputs(r.log.c_str(), f);
  fprintf(f, "\n%s\n", echo.c_str());
  fputs("exit\n", f);
  fclose(f);
}

// `rsicnv index`: the file streamed through one decoder on GPU 0 with indexing on, the same chunks as the one-pass route.  The
// index goes to a temporary name first and is renamed into place only when every feed succeeded: a failed run leaves no .bai.
int do_index(const Opt& o) {
  if (o.hostdecode) { fprintf(stderr, "index: -hostdecode is not available (the index is built from the GPU decoder's records)\n"); return 2; }
  std::string err; long long coff = 0, skip = 0;
  BamHeader h;
  if (!read_bam_header(o.bamfile, &h, &coff, &skip, &err)) { fprintf(stderr, "%s\n", err.c_str()); return 1; }
  const std::string out = o.out_set ? o.outfile : o.bamfile + ".bai";
  const std::string tmp = out + ".tmp." + std::to_string((long long)getpid());
  rsigpu_ctx* dec = nullptr;
  if (create_decoder(o, 0, &dec)) { fprintf(stderr, "cannot create the decoder context\n"); return 2; }
  int rc = 1;
  const double t0 = now_s();
  DecodeTiming tm;
  if (rsigpu_bam_begin(dec, (int32_t)h.name.size()) || rsigpu_bam_index_begin(dec, (int64_t)coff)) fprintf(stderr, "%s\n", rsigpu_last_error(dec));
  else if (stream_bam(o.bamfile, coff, skip, 0, dec, (size_t)256 << 20, [](int, const rsigpu_bam_run&) { return 0; }, &tm) == 0) {
    int64_t nb = 0;
    std::vector<uint8_t> ix;
    if (rsigpu_bam_index_get(dec, nullptr, 0, &nb) == 0) { ix.resize((size_t)nb); if (rsigpu_bam_index_get(dec, ix.data(), nb, &nb)) ix.clear(); }
    if (ix.empty()) fprintf(stderr, "%s\n", rsigpu_last_error(dec));
    else {
      FILE* f = fopen(tmp.c_str(), "wb");
      const bool ok = f && fwrite(ix.data(), 1, ix.size(), f) == ix.size();
      if (f && fclose(f) != 0) rc = 1;
      if (ok && rename(tmp.c_str(), out.c_str()) == 0) rc = 0;
      else fprintf(stderr, "cannot write %s\n", out.c_str());
    }
  }
  if (rc) unlink(tmp.c_str());
  rsigpu_destroy(dec);
  if (getenv("RSICNV_TIMING")) fprintf(stderr, "#timing: index %.3f s (read %.3f, bam_feed %.3f)\n", now_s() - t0, tm.read, tm.feed);
  return rc;
}

int do_decode(const Opt& o) {
  BamReader br(o.threads); std::string err;
  {   // what the GPU decoder is given: where the alignment records start
    BamHeader h; long long coff = 0, skip = 0;
    if (read_bam_header(o.bamfile, &h, &coff, &skip, &err)) printf("records start at file offset %lld + %lld decoded bytes, %zu references\n", coff, skip, h.name.size());
  }
  if (!br.open(o.bamfile, &err)) { fprintf(stderr, "%s\n", err.c_str()); return 1; }
  ContigReads cr;
  while (br.next_contig(&cr, &err)) {
    if (br.header().name[(size_t)cr.tid] != o.chr) continue;
    auto dump = [&](const char* field, const void* p, size_t bytes) {
      FILE* f = fopen((o.outfile + "." + field).c_str(), "wb");
      if (f) { fwrite(p, 1, bytes, f); fclose(f); }
    };
    dump("pos", cr.pos.data(), cr.pos.size() * 4); dump("mpos", cr.mpos.data(), cr.mpos.size() * 4); dump("isize", cr.isize.data(), cr.isize.size() * 4);
    dump("mtid", cr.mtid.data(), cr.mtid.size() * 4); dump("flag", cr.flag.data(), cr.flag.size() * 2); dump("mapq", cr.mapq.data(), cr.mapq.size());
    dump("cigar_off", cr.cigar_off.data(), cr.cigar_off.size() * 4); dump("cigar", cr.cigar.data(), cr.cigar.size() * 4);
    dump("qual_off", cr.qual_off.data(), cr.qual_off.size() * 8); dump("qual", cr.qual.data(), cr.qual.size());
    printf("%s\t%zu reads\n", o.chr.c_str(), cr.n());
    return 0;
  }
  if (!err.empty()) fprintf(stderr, "%s\n", err.c_str());
  fprintf(stderr, "BAM file doesn't have %s\n", o.chr.c_str());
  return 1;
}

}  // namespace

int main(int argc, char** argv) {
  Opt o;
  if (!parse(argc, argv, &o)) return usage();
  if (o.function == "decode") return do_decode(o);
  if (o.unsorted && (o.split > 1 || o.hostdecode)) { fprintf(stderr, "-unsorted works with the GPU decoder and without -split\n"); return 2; }
  const double t_main = now_s();
  const int ndev = rsigpu_num_devices();
  if (ndev <= 0) { fprintf(stderr, "no CUDA device: this implementation has no CPU path\n"); return 2; }
  if (o.function == "index") return do_index(o);
  if (o.split > 1) {
    if (o.split > ndev) { fprintf(stderr, "-split %d: only %d GPUs\n", o.split, ndev); return 2; }
    if (o.hostdecode || o.saverd) { fprintf(stderr, "-split works with the GPU decoder and without -s\n"); return 2; }
    o.gpus = o.split;
  }
  const int ng = std::max(1, std::min(o.gpus, ndev));
  // per GPU: two contig contexts for BAM input decoded on the GPU (one is decoded into while the other runs the hot path), else one
  const int per_gpu = (!o.bamfile.empty() && !o.hostdecode && o.split <= 1) ? 2 : 1;
  std::vector<std::vector<rsigpu_ctx*>> ctx((size_t)ng);
  {
    std::vector<std::thread> th; std::atomic<int> bad(0);
    for (int g = 0; g < ng; ++g)
      th.emplace_back([&, g]() {
        for (int k = 0; k < per_gpu; ++k) { rsigpu_ctx* c = nullptr; if (rsigpu_create(g, &o.P, &c)) { bad++; return; } ctx[(size_t)g].push_back(c); }
      });
    for (auto& t : th) t.join();
    if (bad.load()) { fprintf(stderr, "cannot create a context on every GPU\n"); return 2; }
  }
  if (getenv("RSICNV_TIMING")) fprintf(stderr, "#timing: CUDA start-up + contexts %.3f s\n", now_s() - t_main);
  if (o.function == "stat") {
    const int rc = do_stat(o, ctx[0][0]);
    for (auto& v : ctx) for (rsigpu_ctx* c : v) rsigpu_destroy(c);
    return rc;
  }
  std::vector<ContigResult> results;
  std::string err;
  int rc_all = 0;
  if (!o.rdfile.empty()) {   // depth-file input: one contig (rsi.cpp:2133-2136, 2192-2195)
    results.resize(1); results[0].name = o.chr;
    std::string fasta; std::vector<int32_t> rd;
    if (!read_fasta(o.reffile, o.chr, &fasta, &err) || !parse_depth_text(o.rdfile, (int)fasta.size(), &rd, &err)) { fprintf(stderr, "%s\n", err.c_str()); return 0; }
    fprintf(stderr, "#processing %s\n", o.chr.c_str());
    if (o.split > 1) {
      std::vector<rsigpu_ctx*> parts;
      bool ok = true;
      for (int g = 0; g < ng && ok; ++g) { parts.push_back(ctx[(size_t)g][0]); ok = begin_contig(parts.back(), 0, fasta, &rd, &results[0]); }
      results[0].done = ok && split_finish(o, parts, o.chr, false, &results[0]);
    } else results[0].done = run_contig(ctx[0][0], o, o.chr, 0, fasta, &rd, nullptr, &results[0]);
    if (!results[0].done) { fprintf(stderr, "%s\n", results[0].err.c_str()); rc_all = 1; }
  } else if (o.split > 1) {
    std::vector<rsigpu_ctx*> parts;
    for (int g = 0; g < ng; ++g) parts.push_back(ctx[(size_t)g][0]);
    rc_all = bam_split_on_gpu(o, parts, &results);
    if (rc_all == 2) return 2;
  } else if (o.unsorted) {
    rc_all = bam_unsorted_on_gpu(o, ctx, &results);
    if (rc_all == 2) return 2;
  } else if (!o.hostdecode) {
    rc_all = bam_on_gpu(o, ctx, &results);
    if (rc_all == 2) return 2;
  } else {
    BamReader br(o.threads);
    if (!br.open(o.bamfile, &err)) { fprintf(stderr, "%s\n", err.c_str()); return 0; }
    const BamHeader& h = br.header();
    results.resize(h.name.size());
    for (size_t i = 0; i < h.name.size(); ++i) results[i].name = h.name[i];
    if (o.chr != "1-22XY" && std::find(h.name.begin(), h.name.end(), o.chr) == h.name.end()) { fprintf(stderr, "BAM file doesn't have %s\n", o.chr.c_str()); return 0; }
    // contigs stream out of the file in header order; each GPU has one worker thread that takes the next decoded contig
    std::mutex mu;
    std::vector<std::thread> workers((size_t)ng);
    ContigReads cr;
    const std::vector<int> gpu_of = lpt_assign(o, h, ng, nullptr);
    std::atomic<int> failed(0);
    while (br.next_contig(&cr, &err)) {
      const std::string& name = h.name[(size_t)cr.tid];
      if (!eligible(o, name)) continue;                       // rsi.cpp:2119-2120, 2137-2143
      const int g = gpu_of[(size_t)cr.tid];
      if (workers[(size_t)g].joinable()) workers[(size_t)g].join();
      fprintf(stderr, "#processing %s (%zu reads) on GPU %d\n", name.c_str(), cr.n(), g);
      ContigReads* mine = new ContigReads(std::move(cr));
      cr = ContigReads();
      const int tid = mine->tid;
      workers[(size_t)g] = std::thread([&, g, tid, mine]() {
        std::string fasta, e2;
        ContigResult& r = results[(size_t)tid];
        if (!read_fasta(o.reffile, r.name, &fasta, &e2)) r.err = e2;
        else {
          if ((int)fasta.size() != h.len[(size_t)tid]) fprintf(stderr, "reference and target not same size %zu\t%d\n", fasta.size(), h.len[(size_t)tid]);
          r.done = run_contig(ctx[(size_t)g][0], o, r.name, tid, fasta, nullptr, mine, &r);
        }
        if (!r.done) { std::lock_guard<std::mutex> lk(mu); fprintf(stderr, "%s: %s\n", r.name.c_str(), r.err.c_str()); failed++; }
        delete mine;
      });
    }
    for (auto& w : workers) if (w.joinable()) w.join();
    if (!err.empty()) { fprintf(stderr, "%s\n", err.c_str()); failed++; }   // the reader stopped on a corrupt block: the contig it was in is not reported
    if (failed.load()) rc_all = 1;
  }
  write_table(o, results);
  {
    std::string command, check;
    for (int i = 0; i < argc; ++i) command += std::string(argv[i]) + " ";
    if (!o.bamfile.empty()) {   // "#Check bam header for 1-22XY" (rsi.cpp:2114-2131): every target without "MT" / "." in its name, then those with reads
      BamHeader h; long long co = 0, sk = 0; std::string e3;
      if (read_bam_header(o.bamfile, &h, &co, &sk, &e3)) {
        std::vector<BaiRef> bai;
        const bool have_idx = !o.unsorted && read_bai(o.bamfile, h.name.size(), &bai);
        check = "#Check bam header for 1-22XY \n";
        std::string pop = "#BAM has reads on :";
        for (size_t i = 0; i < h.name.size(); ++i) {
          if (h.name[i].find("MT") != std::string::npos || h.name[i].find(".") != std::string::npos) continue;
          check += h.name[i] + "\t" + std::to_string(h.len[i]) + "\t" + std::to_string(i) + "\t0\t536870912\n";
          const bool has = have_idx ? bai[i].has_reads : (i < results.size() && (results[i].done || !results[i].err.empty()));
          if (has) pop += " " + h.name[i];
        }
        check += pop + "\n";
      }
    }
    write_log(o, command, results, check);
  }
  if (getenv("RSICNV_TIMING")) fprintf(stderr, "#timing: total %.3f s\n", now_s() - t_main);
  fprintf(stderr, "output written to %s\n", o.outfile.c_str());
  for (auto& v : ctx) for (rsigpu_ctx* c : v) rsigpu_destroy(c);
  return rc_all;
}
