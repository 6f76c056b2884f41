// malva-geno -- the MALVA genotyping CLI over the B200 hot path.
//
//   malva-geno index [flags] <reference.fa> <variants.vcf> <kmc_output_prefix>
//   malva-geno call  [flags] <reference.fa> <variants.vcf> <kmc_output_prefix>   > out.vcf
//   malva-geno call  [flags] <reference.fa> <variants.vcf> <db1> <db2> .. --out-dir DIR   (DIR/<basename>.vcf each)
//   malva-geno call  [flags] <reference.fa> <variants.vcf> <reads.fq|fa[.gz]> [<reads2> .. --out-dir DIR] --reads
//        genotype straight from reads: each sample is counted on the device, only the ref_k-mers the index can use
//        (mg_count_restrict), and scanned from the count table -- the VCFs of `count` + `call DB`, no database on disk
//
// Same sub-commands, flags (-k -r -e -s -f -c -b -p -u -v -1), index file name, stderr phase lines and VCF
// output as the reference (main.cpp:226-594, argument_parser.hpp:51-159).  The host keeps VCF/FASTA reading and
// var_block signature enumeration (signatures.hpp, vcf_io.hpp); everything the reference does through BF / KMAP /
// VB::genotype goes through the C ABI of include/malva_gpu.h into the sm_100a kernels.  There is no CPU path:
// without a usable CUDA device both sub-commands fail.
//
// What is organised differently from the reference's two loops:
//   * VCF lines are decoded and signatures enumerated in parallel (per variant, inside a block as well as across
//     blocks), in batches; a batch goes to the device in one call (mg_add_signatures_packed / mg_genotype_packed:
//     2-bit k-mer words) instead of one k-mer string at a time; the stages of consecutive batches overlap:
//     read (+ inflate, line cutting) | decode + group | enumerate | device | format + write each run on their own
//     thread, and a batch the last stage is done with goes back to the first (its buffers keep their pages);
//   * the KMC database is not decoded on the host: raw suffix records stream through pinned buffers into
//     mg_scan_kmc_records;
//   * with --reads there is no database: the reads are counted on the device and scanned from the count table;
//   * the index file holds sparse lists (index_file.hpp).
//
// Extra (non-reference) flags: --threads N, --device N, --devices, --out-dir, --sample-devices, --reads, --trace.
// Extra sub-commands:
//   malva-geno count [-k43 -ci2 -cs255 ...] <reads.fq|fa[.gz]> <kmc_output_prefix> [tmp_dir]
//        the `kmc` step of the MALVA wrapper (MALVA:107) on the GPU: same command-line shape as kmc, writes a KMC
//        database that `index` / `call` (and the reference) read
//   malva-geno kmc-dump <kmc_output_prefix>                 lists a database as text (no GPU involved)
//   malva-geno signatures [--index-blocks] [flags] <reference.fa> <variants.vcf>     (no GPU involved; CPU tests)
//   malva-geno format-selftest                              the output stage's number formatting against libc (CPU tests)
//   malva-geno container-selftest                           InlineVec / Chain against std::vector (CPU tests)
#include <getopt.h>
#include <sys/resource.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <cerrno>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <future>
#include <iostream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../../../include/malva_gpu.h"
#include "index_file.hpp"
#include "kmc_db.hpp"
#include "signatures.hpp"
#include "vcf_io.hpp"

namespace {

const char *USAGE =
    "Usage: malva-geno <index|call> [-k KMER-SIZE] [-r REF-KMER-SIZE] [-c MAX-COV] "
    "<reference.fa> <variants.vcf> <kmc_output_prefix>\n"
    "\n"
    "      -h, --help                        display this help and exit\n"
    "      -k, --kmer-size                   size of the kmers to index (default:35)\n"
    "      -r, --ref-kmer-size               size of the reference kmers to index (default:43)\n"
    "      -e, --error-rate                  expected sample error rate (default:0.001)\n"
    "      -s, --samples                     file containing the list of (VCF) samples to consider (default:-, i.e. all samples)\n"
    "      -f, --freq-key                    a priori frequency key in the INFO column of the input VCF (default:AF)\n"
    "      -c, --max-coverage                maximum coverage for variant alleles (default:200)\n"
    "      -b, --bf-size                     bloom filter size in GB (default:4)\n"
    "      -p, --strip-chr                   strip \"chr\" from sequence names (default:false)\n"
    "      -u, --uniform                     use uniform a priori probabilities (default:false)\n"
    "      -v, --verbose                     output COVS and GTS in INFO column (default: false)\n"
    "      -1, --haploid                     run MALVA in haploid mode (default: false)\n"
    "          --threads N                   host threads for VCF decoding / signature enumeration (default: all)\n"
    "          --device N                    CUDA device (default: 0)\n"
    "          --devices A,B,..              call: replicate the index on these devices, deal the KMC records\n"
    "                                        round-robin, add the counters up on the first one\n"
    "          --out-dir DIR                 call with several KMC databases (call [opts] ref.fa vars.vcf DB1 DB2 ..):\n"
    "                                        genotype every sample against one index, sample DB to DIR/basename(DB).vcf\n"
    "          --sample-devices A,B,..       call with --out-dir: replicate the index on these devices (a device may\n"
    "                                        repeat) and scan and genotype a share of every round's samples on each\n"
    "                                        (instead of --device / --devices)\n"
    "          --reads                       call: the samples are FASTA/FASTQ read files (plain or gz), not KMC\n"
    "                                        databases; each is counted on the device (as `count` -k<ref_k> -ci2\n"
    "                                        -cs255 would) and genotyped, no database is written (not with --devices)\n"
    "\n";

struct Options {
  unsigned k = 35, ref_k = 43;
  float error_rate = 0.001f;
  std::string samples = "-", freq_key = "AF";
  unsigned max_coverage = 200;
  uint64_t bf_size = 1ull << 35;
  bool strip_chr = false, uniform = false, verbose = false, haploid = false, index_blocks = false;
  int threads = 0, device = 0;
  bool trace = false;  // --trace: per-batch host/device timings on stderr
  std::vector<int> devices;  // --devices a,b,..: `call` replicates the index and deals the KMC records round-robin
  bool devices_given = false;  // --device or --devices was given
  std::vector<int> sample_devices;  // --sample-devices a,b,..: `call --out-dir` spreads the samples over replicas
  std::string fasta_path, vcf_path, kmc_path;
  std::vector<std::string> kmc_paths;  // call: one or more KMC databases (kmc_path = the first)
  std::string out_dir;                 // call with several databases: sample P is written to out_dir/basename(P).vcf
  bool reads = false;                  // --reads: call's samples (kmc_paths) are read files, counted on the device
};

// argument_parser.hpp:86-159; values are read like `istringstream >> x` reads them
// more_dbs: `call` takes one or more KMC databases after the VCF
bool parse_arguments(int argc, char **argv, Options &o, int n_positional, bool more_dbs = false) {
  static const option longopts[] = {{"kmer-size", required_argument, nullptr, 'k'},
                                    {"ref-kmer-size", required_argument, nullptr, 'r'},
                                    {"error-rate", required_argument, nullptr, 'e'},
                                    {"freq-key", required_argument, nullptr, 'f'},
                                    {"samples", required_argument, nullptr, 's'},
                                    {"max-coverage", required_argument, nullptr, 'c'},
                                    {"bf-size", required_argument, nullptr, 'b'},
                                    // the reference declares these two with required_argument (argument_parser.hpp:79-80)
                                    {"strip-chr", required_argument, nullptr, 'p'},
                                    {"uniform", required_argument, nullptr, 'u'},
                                    {"verbose", no_argument, nullptr, 'v'},
                                    {"haplod", no_argument, nullptr, '1'},  // sic (argument_parser.hpp:82)
                                    {"haploid", no_argument, nullptr, '1'},
                                    {"help", no_argument, nullptr, 'h'},
                                    {"threads", required_argument, nullptr, 1000},
                                    {"device", required_argument, nullptr, 1001},
                                    {"index-blocks", no_argument, nullptr, 1002},
                                    {"trace", no_argument, nullptr, 1003},
                                    {"devices", required_argument, nullptr, 1004},
                                    {"out-dir", required_argument, nullptr, 1005},
                                    {"sample-devices", required_argument, nullptr, 1006},
                                    {"reads", no_argument, nullptr, 1007},
                                    {nullptr, 0, nullptr, 0}};
  bool die = false;
  optind = 1;
  for (int c; (c = getopt_long(argc, argv, "k:r:e:s:f:c:b:hpuv1", longopts, nullptr)) != -1;) {
    std::istringstream arg(optarg ? optarg : "");
    switch (c) {
      case 'p': o.strip_chr = true; break;
      case 'u': o.uniform = true; break;
      case 'k': arg >> o.k; break;
      case 'r': arg >> o.ref_k; break;
      case 'e': arg >> o.error_rate; break;
      case 's': arg >> o.samples; break;
      case 'f': arg >> o.freq_key; break;
      case 'c': arg >> o.max_coverage; break;
      case 'b':
        arg >> o.bf_size;
        o.bf_size *= 1ull << 33;  // GB -> bits (argument_parser.hpp:119-123)
        break;
      case 'v': o.verbose = true; break;
      case '1': o.haploid = true; break;
      case 1000: arg >> o.threads; break;
      case 1001:
        arg >> o.device;
        o.devices_given = true;
        break;
      case 1002: o.index_blocks = true; break;
      case 1003: o.trace = true; break;
      case 1004:
      case 1006: {
        std::vector<int> &list = c == 1004 ? o.devices : o.sample_devices;
        std::string tok;
        while (std::getline(arg, tok, ','))
          if (!tok.empty()) list.push_back(atoi(tok.c_str()));
        o.devices_given = o.devices_given || c == 1004;
        break;
      }
      case 1005: o.out_dir = optarg ? optarg : ""; break;
      case 1007: o.reads = true; break;
      case '?': die = true; break;
      case 'h':
        std::cout << USAGE;
        exit(EXIT_SUCCESS);
    }
  }
  if (argc - optind < n_positional) {
    std::cerr << "malva : missing arguments\n";
    die = true;
  } else if (argc - optind > n_positional && !more_dbs) {
    std::cerr << "malva : too many arguments\n";
    die = true;
  }
  if (die) {
    std::cerr << "\n" << USAGE;
    return false;
  }
  o.fasta_path = argv[optind++];
  o.vcf_path = argv[optind++];
  if (n_positional > 2) o.kmc_path = argv[optind];
  while (n_positional > 2 && optind < argc) o.kmc_paths.push_back(argv[optind++]);
  if (o.threads <= 0) o.threads = (int)std::max(1u, std::thread::hardware_concurrency());
  mh::io_threads() = o.threads;
  if (o.devices.empty()) o.devices.push_back(o.device);
  o.device = o.devices[0];
  return true;
}

// ---- phase timers: the reference's pelapsed() lines (main.cpp:93-115), same labels, same layout ----
using Clock = std::chrono::high_resolution_clock;
Clock::time_point g_start = Clock::now(), g_last = g_start;
double cpu_seconds() {
  rusage u;
  getrusage(RUSAGE_SELF, &u);
  return (double)u.ru_utime.tv_sec + (double)u.ru_utime.tv_usec * 1e-6;
}
double g_cpu_start = cpu_seconds();
std::mutex g_pelapsed_mutex;  // (progress lines come from the reader thread as well)
void pelapsed(const std::string &s, bool rollback = false) {
  std::lock_guard<std::mutex> lock(g_pelapsed_mutex);
  auto now = Clock::now();
  char buf[512];
  rusage u;
  getrusage(RUSAGE_SELF, &u);
  snprintf(buf, sizeof(buf),
           "[malva-geno/%s] Execution Time %.4gs\n[malva-geno/%s] Time elapsed %.4gs\n"
           "[malva-geno/%s] Used CPU-time elapsed %.4gs\n[malva-geno/%s] Maximum memory used %ldMb\n%s",
           s.c_str(), std::chrono::duration<double>(now - g_last).count(), s.c_str(),
           std::chrono::duration<double>(now - g_start).count(), s.c_str(), cpu_seconds() - g_cpu_start, s.c_str(),
           u.ru_maxrss / 1024, rollback ? "\r" : "\n");
  std::cerr << buf;
  g_last = Clock::now();
}

struct Stopwatch {
  Clock::time_point t = Clock::now();
  double lap() {
    auto n = Clock::now();
    double s = std::chrono::duration<double>(n - t).count();
    t = n;
    return s * 1e3;
  }
};

// (A persistent worker pool and a malloc tuned to keep freed batches in the heap were both measured on the 16-core GPU
// box and were no faster than fresh threads per call -- 1.66 s against 1.51-1.56 s for the VCF pass of `call` at 6e6
// variants: with one shared queue the stages of the pipeline take turns instead of overlapping.)
void parallel_for(size_t n, int threads, const std::function<void(size_t)> &fn) {
  if (n == 0) return;
  int t = (int)std::min<size_t>((size_t)threads, n);
  if (t <= 1) {
    for (size_t i = 0; i < n; ++i) fn(i);
    return;
  }
  std::atomic<size_t> next{0};
  std::vector<std::exception_ptr> errs((size_t)t);
  std::vector<std::thread> pool;
  for (int w = 0; w < t; ++w)
    pool.emplace_back([&, w] {
      try {
        for (size_t i; (i = next.fetch_add(1)) < n;) fn(i);
      } catch (...) {
        errs[(size_t)w] = std::current_exception();
        next.store(n);
      }
    });
  for (auto &th : pool) th.join();
  for (auto &e : errs)
    if (e) std::rethrow_exception(e);
}

// Successful runs leave through here: everything that has to reach a file is flushed and closed by then, and tearing
// down gigabytes of device allocations and the CUDA context one by one only costs time (0.3-1 s) at exit.
[[noreturn]] void finish(int rc) {
  std::cout.flush();
  fflush(stdout);
  fflush(stderr);
  _exit(rc);
}

struct GpuError : std::runtime_error {
  using std::runtime_error::runtime_error;
};
void gpu(int rc, const char *what) {
  if (rc != MG_OK) throw GpuError(std::string(what) + ": " + mg_last_error());
}

// A bounded hand-over between two stages of the batch pipeline.
template <class T>
class Channel {
 public:
  explicit Channel(size_t cap) : cap_(cap) {}
  void push(T &&v) {
    std::unique_lock<std::mutex> l(m_);
    cv_.wait(l, [&] { return q_.size() < cap_ || closed_; });
    if (closed_) return;
    q_.push_back(std::move(v));
    cv_.notify_all();
  }
  bool pop(T &out) {  // false once the channel is closed and drained
    std::unique_lock<std::mutex> l(m_);
    cv_.wait(l, [&] { return !q_.empty() || closed_; });
    if (q_.empty()) return false;
    out = std::move(q_.front());
    q_.pop_front();
    cv_.notify_all();
    return true;
  }
  bool try_pop(T &out) {  // what is there right now, without waiting
    std::lock_guard<std::mutex> l(m_);
    if (q_.empty()) return false;
    out = std::move(q_.front());
    q_.pop_front();
    cv_.notify_all();
    return true;
  }
  bool try_push(T &&v) {  // dropped (false) if the channel is full or closed
    std::lock_guard<std::mutex> l(m_);
    if (closed_ || q_.size() >= cap_) return false;
    q_.push_back(std::move(v));
    cv_.notify_all();
    return true;
  }
  void close() {
    std::lock_guard<std::mutex> l(m_);
    closed_ = true;
    cv_.notify_all();
  }

 private:
  std::mutex m_;
  std::condition_variable cv_;
  std::deque<T> q_;
  size_t cap_;
  bool closed_ = false;
};

// ---- the VCF loop of index_main / call_main (main.cpp:309-370, 522-579) as a stream of batches of blocks ----
// A batch owns the records it was decoded into (`arena`, in file order, skipped records squeezed out) and the contig
// names its blocks refer to; the blocks are views into the arena.
struct BlockBatch {
  std::vector<mh::Variant> arena;
  std::vector<mh::VarBlock> blocks;
  std::vector<std::unique_ptr<std::string>> contigs;
  BlockBatch() = default;
  BlockBatch(BlockBatch &&) = default;
  BlockBatch &operator=(BlockBatch &&) = default;
  void clear() {
    arena.clear();
    blocks.clear();
    contigs.clear();
  }
};

class BlockStream {
 public:
  BlockStream(const Options &o, bool index_mode) : o_(o), index_mode_(index_mode), reader_(o.vcf_path) {
    is_file_ = o.samples != "-";
    samples_code = reader_.header.set_samples(o.samples);
    freq_declared_ = reader_.header.has_info(o.freq_key);
  }
  ~BlockStream() {
    text_.close();
    spare_.close();
    if (reader_thread_.joinable()) reader_thread_.join();
  }
  BlockStream(const BlockStream &) = delete;
  BlockStream &operator=(const BlockStream &) = delete;
  int samples_code = 0;
  double t_read = 0, t_decode = 0, t_group = 0;  // ms spent reading lines / decoding records / grouping blocks
  std::vector<std::string> used_seq_names;  // main.cpp:304-306, 323-328, 352-356
  uint64_t n_records = 0;
  const mh::VcfHeader &header() const { return reader_.header; }

  // up to `max_lines` more records; the blocks they complete go to `out`.  false when nothing is left.
  bool next_batch(BlockBatch &out, size_t max_lines) {
    out.blocks.clear();  // (the records of a recycled batch stay where they are: every one in use is assigned below)
    out.contigs.clear();
    if (done_) {
      out.arena.clear();
      return false;
    }
    // a block of whole lines (no per-line allocation; read ahead by the reader thread), decoded in parallel straight
    // into the batch's arena, behind the records of the block that was still open when the previous batch ended
    if (!reader_thread_.joinable()) start_reader(max_lines);
    std::unique_ptr<TextBlock> tb;
    if (!text_.pop(tb)) throw std::runtime_error("VCF reader thread ended early");
    if (tb->err) std::rethrow_exception(tb->err);
    const bool more = tb->more;
    const std::vector<mh::BlockLineReader::View> &lines_ = tb->lines;
    t_read += tb->read_ms;
    Stopwatch sw;
    std::vector<mh::Variant> &vars = out.arena;
    const size_t n_carry = carry_.size();
    vars.resize(n_carry + lines_.size());
    for (size_t i = 0; i < n_carry; ++i) vars[i] = std::move(carry_[i]);
    carry_.clear();
    // (a line of a 27,934-sample panel is 84 KB: a 12 MB block holds ~150 of them, so the grain follows the count)
    const size_t grain = std::max<size_t>(1, std::min<size_t>(256, lines_.size() / (4 * (size_t)o_.threads) + 1));
    const size_t n_tasks = (lines_.size() + grain - 1) / grain;
    parallel_for(n_tasks, o_.threads, [&](size_t t) {
      for (size_t i = t * grain; i < std::min(lines_.size(), (t + 1) * grain); ++i)
        vars[n_carry + i] = mh::parse_record(lines_[i].b, lines_[i].e, reader_.header, o_.freq_key, o_.uniform, freq_declared_);
    });
    t_decode += sw.lap();
    tb->lines.clear();
    spare_.try_push(std::move(tb));  // the text is not needed any more: its buffers go back to the reader
    // grouping (main.cpp:330-362): `open` = first record of the block being built, `w` = where the next kept record goes
    size_t w = n_carry, open = 0;
    bool have_open = n_carry > 0;
    auto flush = [&](size_t end) {  // (one name object per run of blocks on the same contig, not one per block)
      if (out.contigs.empty() || *out.contigs.back() != last_seq_name_)
        out.contigs.push_back(std::make_unique<std::string>(last_seq_name_));
      out.blocks.emplace_back((int)o_.k, vars.data() + open, end - open, out.contigs.back().get());
    };
    for (size_t r = n_carry; r < vars.size(); ++r) {
      mh::Variant &v = vars[r];
      ++n_records;
      if (n_records % 5000 == 0) pelapsed("Processed " + std::to_string(n_records) + " variants", true);
      if (last_seq_name_.empty()) {
        last_seq_name_ = v.seq_name;
        used_seq_names.push_back(last_seq_name_);
      }
      // index: variants with only symbolic ALTs or carried by no sample are skipped; call: the latter are kept
      // (they are genotyped 0/0, main.cpp:332 vs :538)
      if (!v.has_alts || (index_mode_ && !v.is_present)) continue;
      if (have_open && (!mh::variants_near(vars[w - 1], v, (int)o_.k, 0) || last_seq_name_ != v.seq_name)) {
        flush(w);
        have_open = false;
        if (last_seq_name_ != v.seq_name) {
          last_seq_name_ = v.seq_name;
          used_seq_names.push_back(last_seq_name_);
        }
      }
      if (!have_open) {
        open = w;
        have_open = true;
      }
      if (w != r) vars[w] = std::move(v);
      ++w;
    }
    if (!more) {  // end of file
      done_ = true;
      if (have_open) flush(w);
    } else if (have_open) {  // the open block continues in the next batch: its records travel on
      for (size_t i = open; i < w; ++i) carry_.push_back(std::move(vars[i]));
      w = open;
    }
    vars.resize(w);  // (shrinks: the blocks' views stay valid)
    t_group += sw.lap();
    return !out.blocks.empty() || !done_;
  }

 private:
  const Options &o_;
  bool index_mode_, is_file_ = false, freq_declared_ = false, done_ = false;
  mh::VcfReader reader_;
  std::vector<mh::Variant> carry_;  // the records of the block that is still open between two batches
  std::string last_seq_name_;

  // The file is read (and inflated, and cut into lines) by a thread of its own, one block of text ahead of the
  // decode: reading a block is serial work of the same order as decoding it on all threads.
  struct TextBlock {
    mh::TextBuf store;
    std::vector<mh::BlockLineReader::View> lines;
    bool more = false;
    double read_ms = 0;
    std::exception_ptr err;
  };
  void start_reader(size_t max_lines) {
    reader_thread_ = std::thread([this, max_lines] {
      while (true) {
        std::unique_ptr<TextBlock> tb;
        if (!spare_.try_pop(tb)) tb = std::make_unique<TextBlock>();
        Stopwatch sw;
        try {
          tb->more = reader_.next_lines(tb->store, tb->lines, max_lines, 12u << 20);
        } catch (...) {
          tb->err = std::current_exception();
          tb->more = false;
        }
        tb->read_ms = sw.lap();
        const bool last = !tb->more;
        text_.push(std::move(tb));
        if (last) break;
      }
    });
  }
  Channel<std::unique_ptr<TextBlock>> text_{1}, spare_{4};
  std::thread reader_thread_;
};

// Reads and decodes batch i+1 on a background thread while batch i is enumerated, sent to the device and printed.
class BatchPrefetcher {
 public:
  BatchPrefetcher(BlockStream &stream, size_t max_lines) : stream_(stream), max_lines_(max_lines) { launch(); }
  // false when the VCF is exhausted; otherwise `out` holds the next batch of flushed blocks (possibly empty).  What
  // `out` held before is taken in exchange and filled next: a batch that has been through the pipeline keeps its
  // buffers (25 MB of records), so in the steady state no batch touches fresh pages.
  bool next(BlockBatch &out) {
    if (!pending_.valid()) return false;
    if (!pending_.get()) return false;
    std::swap(out, filling_);
    launch();
    return true;
  }

 private:
  void launch() {
    pending_ = std::async(std::launch::async, [this] { return stream_.next_batch(filling_, max_lines_); });
  }
  BlockStream &stream_;
  size_t max_lines_;
  BlockBatch filling_;
  std::future<bool> pending_;
};

// signatures of a batch of blocks: tasks of ~64 consecutive variants (a block of thousands of variants is split,
// small blocks are grouped) enumerated in parallel, their parts then copied side by side into one CSR
void enumerate_batch(const std::vector<mh::VarBlock> &blocks, std::map<std::string, std::string> &refs, const Options &o,
                     mh::SignatureCsr &out) {
  for (const auto &b : blocks) refs[*b.contig];  // (the reference's refs[name] creates missing contigs as empty)
  struct Segment {
    uint32_t block, begin, end;
  };
  constexpr size_t TASK_VARIANTS = 64;
  std::vector<Segment> segs;
  std::vector<size_t> task_first{0};  // tasks = runs of segments
  size_t in_task = 0;
  for (size_t b = 0; b < blocks.size(); ++b)
    for (size_t v = 0; v < blocks[b].size();) {
      const size_t take = std::min(blocks[b].size() - v, TASK_VARIANTS - in_task);
      segs.push_back(Segment{(uint32_t)b, (uint32_t)v, (uint32_t)(v + take)});
      v += take;
      in_task += take;
      if (in_task == TASK_VARIANTS) {
        task_first.push_back(segs.size());
        in_task = 0;
      }
    }
  if (task_first.back() != segs.size()) task_first.push_back(segs.size());
  const size_t n_tasks = task_first.size() - 1;
  std::vector<mh::SignatureCsr> parts(n_tasks);
  std::vector<const std::string *> ref_of(blocks.size());
  for (size_t b = 0; b < blocks.size(); ++b) ref_of[b] = &refs.find(*blocks[b].contig)->second;
  parallel_for(n_tasks, o.threads, [&](size_t t) {
    static thread_local mh::VarBlock::Scratch sc;
    for (size_t i = task_first[t]; i < task_first[t + 1]; ++i)
      blocks[segs[i].block].enumerate(*ref_of[segs[i].block], o.haploid, segs[i].begin, segs[i].end, sc, parts[t]);
  });
  mh::SignatureCsr::concat(parts, out, [&](size_t n, const std::function<void(size_t)> &fn) { parallel_for(n, o.threads, fn); });
}

// one batch on its way through the pipeline
struct Batch {
  BlockBatch vb;
  mh::SignatureCsr sigs;
  double t_parse = 0, t_enum = 0, t_dev = 0;
  // results of the device stage (call)
  std::vector<uint64_t> lik_off;
  std::vector<uint32_t> cov;
  std::vector<int32_t> n_gts, status, best, gq;
  std::vector<double> lik;
};

// stage 1 + 2 of both sub-commands: batches of decoded blocks (read ahead by the BatchPrefetcher's own thread) with
// their signatures enumerated, handed over in order.  An exception ends the stream and is re-thrown by join().
class EnumeratedBatches {
 public:
  EnumeratedBatches(BatchPrefetcher &src, std::map<std::string, std::string> &refs, const Options &o)
      : out_(2), th_([this, &src, &refs, &o] {
          try {
            while (true) {
              std::unique_ptr<Batch> b;
              if (!spare_.try_pop(b)) b = std::make_unique<Batch>();
              Stopwatch sw;
              if (!src.next(b->vb)) break;
              b->t_parse = sw.lap();
              enumerate_batch(b->vb.blocks, refs, o, b->sigs);
              b->t_enum = sw.lap();
              out_.push(std::move(b));
            }
          } catch (...) {
            err_ = std::current_exception();
          }
          out_.close();
        }) {}
  ~EnumeratedBatches() {
    out_.close();
    if (th_.joinable()) th_.join();
  }
  bool next(std::unique_ptr<Batch> &b) { return out_.pop(b); }
  // a batch the last stage is done with: its buffers serve a later batch (no allocation, no page faults)
  void recycle(std::unique_ptr<Batch> &&b) {
    if (b) spare_.try_push(std::move(b));
  }
  void join() {
    if (th_.joinable()) th_.join();
    if (err_) std::rethrow_exception(err_);
  }

 private:
  Channel<std::unique_ptr<Batch>> out_, spare_{8};
  std::exception_ptr err_;
  std::thread th_;
};

constexpr size_t LINES_PER_BATCH = 1 << 17;  // (a batch is ~12 MB of VCF text, at most this many records)

struct Ctx {
  mg_ctx *c = nullptr;
  ~Ctx() { mg_destroy(c); }
};

// ------------------------------------------------------------------------------------------------
int index_main(int argc, char **argv) {
  Options o;
  if (!parse_arguments(argc, argv, o, 3)) return EXIT_FAILURE;
  // CUDA start-up and the empty index (allocation + clearing of the filters) overlap with the file reading
  Ctx g;
  Stopwatch sw;
  auto ctx_up = std::async(std::launch::async, [&]() -> std::string {
    if (mg_warmup(o.device) != MG_OK || mg_create(&g.c, o.device, (int)o.k, (int)o.ref_k, o.bf_size) != MG_OK) return mg_last_error();
    return std::string();
  });
  BlockStream stream(o, true);
  if (stream.samples_code != 0) {
    std::cerr << "ERROR: VCF samples subset (code: " << stream.samples_code << ")" << std::endl;
    return 1;
  }
  {
    mh::KmcDb db;  // opened and unused, like the reference (main.cpp:273-279)
    std::string why;
    if (!db.open(o.kmc_path, why)) {
      std::cerr << "ERROR: cannot open " << o.kmc_path << std::endl;
      return 1;
    }
  }
  // (the first batch of VCF records is read and decoded in the background while the reference is loaded and the
  // device starts up)
  BatchPrefetcher index_batches(stream, LINES_PER_BATCH);
  pelapsed("Reference parsing");
  std::map<std::string, std::string> refs = mh::read_fasta(o.fasta_path, o.strip_chr);
  pelapsed("Reference processed");

  pelapsed("VCF parsing (Bloom Filter construction)");
  {
    const double before = sw.lap();
    const std::string err = ctx_up.get();
    if (!err.empty()) throw GpuError("mg_create: " + err);
    if (o.trace)
      fprintf(stderr, "[trace] files read %.1f ms; then waited %.1f ms more for mg_create (CUDA start-up + empty index)\n", before,
              sw.lap());
  }
  {
    EnumeratedBatches batches(index_batches, refs, o);  // enumerates batch i+1 while batch i is inserted
    std::unique_ptr<Batch> b;
    std::vector<uint64_t> reg;  // the regular k-mers of a batch, and the text of the irregular ones
    std::vector<uint8_t> reg_is_ref, irr_is_ref;
    while (batches.next(b)) {
      sw.lap();
      const mh::SignatureCsr &sg = b->sigs;
      // add_kmers_to_bf (main.cpp:122-144): allele 0 -> ref_bf, others -> bf
      reg.clear();
      reg_is_ref.clear();
      irr_is_ref.clear();
      for (uint64_t i = 0; i < sg.n_kmers(); ++i) {
        if (sg.is_irregular(i)) continue;
        reg.push_back(sg.kmers[2 * i]);
        reg.push_back(sg.kmers[2 * i + 1] & ~(mh::SIG_REF_ALLELE | mh::SIG_IRREGULAR));
        reg_is_ref.push_back(sg.is_ref_kmer(i));
      }
      gpu(mg_add_signatures_packed(g.c, reg.data(), reg_is_ref.data(), reg_is_ref.size()), "mg_add_signatures_packed");
      if (sg.n_irregular()) {  // shorter than k / non-ACGT symbols: as text, hashed byte-exactly on the device
        for (uint64_t j = 0; j < sg.n_irregular(); ++j) irr_is_ref.push_back(sg.is_ref_kmer(sg.irr_kmer[j]));
        gpu(mg_add_signatures(g.c, sg.irr_pool.data(), sg.irr_off.data(), irr_is_ref.data(), sg.n_irregular()),
            "mg_add_signatures");
      }
      if (o.trace)
        fprintf(stderr, "[trace] index batch: %zu blocks, %llu k-mers (%llu irregular): read+decode wait %.1f ms, enumerate %.1f ms, device %.1f ms\n",
                b->vb.blocks.size(), (unsigned long long)sg.n_kmers(), (unsigned long long)sg.n_irregular(), b->t_parse,
                b->t_enum, sw.lap());
      batches.recycle(std::move(b));
    }
    batches.join();
  }
  pelapsed("Processed " + std::to_string(stream.n_records) + " variants");
  gpu(mg_finalize_alt(g.c), "mg_finalize_alt");  // bf.switch_mode()
  pelapsed("BF creation complete");

  pelapsed("Reference BF construction");
  for (const std::string &name : stream.used_seq_names) {
    const std::string &seq = refs[name];
    gpu(mg_scan_reference(g.c, seq.data(), seq.size()), "mg_scan_reference");
  }
  pelapsed("Reference BF creation complete");
  gpu(mg_finalize_context(g.c), "mg_finalize_context");  // context_bf.switch_mode()

  {
    sw.lap();
    mh::IndexWriter w(o.vcf_path + ".c" + std::to_string(o.ref_k) + ".k" + std::to_string(o.k) + ".malvax.zst", o.k,
                      o.ref_k, o.bf_size);
    for (int which : {1, 0}) {  // context_bf, then bf, then ref_bf (main.cpp:409-411)
      uint64_t n = 0;
      gpu(mg_export_set_bits(g.c, which, nullptr, 0, &n), "mg_export_set_bits");
      std::vector<uint64_t> idx(n);
      if (n) gpu(mg_export_set_bits(g.c, which, idx.data(), n, &n), "mg_export_set_bits");
      w.write_bits(idx);
    }
    uint64_t n = 0;
    gpu(mg_export_ref_keys(g.c, nullptr, 0, &n), "mg_export_ref_keys");
    std::vector<uint64_t> keys(2 * n);
    if (n) gpu(mg_export_ref_keys(g.c, keys.data(), n, &n), "mg_export_ref_keys");
    w.write_keys(keys);
    w.close();
    if (o.trace) fprintf(stderr, "[trace] index file (export from the device, compress, write) %.1f ms\n", sw.lap());
  }
  finish(0);
}

// ------------------------------------------------------------------------------------------------
// one VCF line per variant of the batch, VB::output_variants (var_block.hpp:337-396)
inline void append_int(std::string &out, long long x) {  // what std::to_string(int) appends, without the temporary
  char tmp[24];
  char *e = tmp + sizeof(tmp), *p = e;
  unsigned long long u = x < 0 ? 0ull - (unsigned long long)x : (unsigned long long)x;
  do {
    *--p = (char)('0' + u % 10);
    u /= 10;
  } while (u);
  if (x < 0) *--p = '-';
  out.append(p, (size_t)(e - p));
}

void format_variant(const mh::Variant &v, const uint32_t *cov, int n_gts, int status, int best, int gq, const double *lik,
                    const Options &o, std::string &out) {
  out += v.seq_name;
  out += '\t';
  append_int(out, (long long)v.ref_pos + 1);
  out += '\t';
  out += v.idx;
  out += '\t';
  out += v.ref_sub;
  out += '\t';
  for (size_t i = 0; i < v.alts.size(); ++i) {
    if (i) out += ',';
    out += v.alts[i];
  }
  out += '\t';
  if (std::isnan(v.quality)) {
    out += '.';
  } else if (v.quality >= 0.0f && v.quality < 1000000.0f && (float)(int)v.quality == v.quality && !std::signbit(v.quality)) {
    append_int(out, (int)v.quality);  // what %g prints for a whole number below 1e6
  } else {
    char num[64];
    snprintf(num, sizeof(num), "%g", (double)v.quality);  // ostream << float
    out += num;
  }
  const int n = v.n_alleles();
  // name of the i-th computed genotype: "g" / "g1/g2" in emission order, or the default for vetoed variants
  auto append_gt_name = [&](int i) {
    if (status != 0) {
      out += o.haploid ? "0" : "0/0";
      return;
    }
    if (o.haploid) {
      append_int(out, i);
      return;
    }
    int g1 = 0, left = i;
    while (left >= n - g1) {
      left -= n - g1;
      ++g1;
    }
    append_int(out, g1);
    out += '/';
    append_int(out, g1 + left);
  };
  out += "\tPASS\t";
  if (o.verbose) {
    out += "COVS=";
    for (int a = 0; a < n; ++a) {
      if (a) out += ',';
      append_int(out, (int)cov[a]);
    }
    out += ";GTS=";
    double total = 0.0;
    for (int i = 0; i < n_gts; ++i) total += lik[i];
    for (int i = 0; i < n_gts; ++i) {
      if (i) out += ',';
      append_gt_name(i);
      out += ':';
      volatile double q = lik[i] / total;  // 0/0 -> the machine's default NaN, printed "-nan" like the reference
      out += std::to_string((double)q);
    }
  } else {
    out += '.';
  }
  out += "\tGT:GQ\t";
  append_gt_name(best);
  out += ':';
  append_int(out, gq);
  out += '\n';
}

// CPU-only check of the formatting short cuts of format_variant against the library calls they stand in for
// (`malva-geno format-selftest`, run by tests/test_host_cpu.py): std::to_string for integers, "%g" for QUAL.
int format_selftest_main() {
  Options o;
  uint64_t bad = 0, n = 0;
  auto check_int = [&](long long x) {
    std::string a;
    append_int(a, x);
    ++n;
    if (a != std::to_string(x)) ++bad;
  };
  for (long long x = -70000; x <= 70000; ++x) check_int(x);
  for (int sh = 0; sh < 63; ++sh)
    for (long long d = -2; d <= 2; ++d) check_int((1ll << sh) + d), check_int(-((1ll << sh) + d));
  check_int(INT32_MAX), check_int(INT32_MIN), check_int(INT64_MAX), check_int(INT64_MIN + 1);
  auto check_qual = [&](float q) {
    mh::Variant v;
    v.seq_name = "1", v.idx = ".", v.ref_sub = "A", v.quality = q;
    v.alts.push_back("C");
    std::string line, want = "1\t1\t.\tA\tC\t";
    const uint32_t cov[2] = {0, 0};
    format_variant(v, cov, 0, 1, 0, 0, nullptr, o, line);
    char num[64];
    snprintf(num, sizeof(num), "%g", (double)q);
    want += std::isnan(q) ? "." : num;
    want += "\tPASS\t.\tGT:GQ\t0/0:0\n";
    ++n;
    if (line != want) {
      if (++bad <= 5) fprintf(stderr, "QUAL %a: got %s", (double)q, line.c_str());
    }
  };
  for (int i = -2000; i <= 2000000; ++i) check_qual((float)i);
  for (int i = 0; i <= 200000; ++i) check_qual((float)i * 0.25f), check_qual((float)i * 0.01f), check_qual(-(float)i * 0.5f);
  for (float q : {0.0f, -0.0f, 999999.0f, 999999.5f, 1e6f, 1e7f, 1e-5f, 3.4e38f, -3.4e38f, INFINITY, -INFINITY, NAN, 16777216.0f, 1e-40f})
    check_qual(q);
  uint32_t r = 12345;
  for (int i = 0; i < 2000000; ++i) {  // arbitrary bit patterns
    r = r * 1664525u + 1013904223u;
    float q;
    memcpy(&q, &r, 4);
    check_qual(q);
  }
  printf("format-selftest: %llu cases, %llu differ\n", (unsigned long long)n, (unsigned long long)bad);
  return bad ? 1 : 0;
}

// CPU-only check of the two small containers of signatures.hpp against std::vector under a random series of the
// operations the host code uses (`malva-geno container-selftest`, run by tests/test_host_cpu.py): growth past the
// inline capacity and back, copies and moves in both states, self-assignment, strings short and long.
int container_selftest_main() {
  uint32_t r = 2026;
  auto rnd = [&](uint32_t n) {
    r = r * 1664525u + 1013904223u;
    return (r >> 8) % n;
  };
  uint64_t checks = 0, bad = 0;
  auto word = [&]() { return std::string((size_t)rnd(40), (char)('A' + rnd(26))); };  // some beyond the SSO size
  {
    using V = mh::InlineVec<std::string, 2>;
    std::vector<V> a(6);
    std::vector<std::vector<std::string>> b(6);
    auto same = [&](size_t i) {
      ++checks;
      bool ok = a[i].size() == b[i].size() && a[i].empty() == b[i].empty();
      for (size_t j = 0; ok && j < b[i].size(); ++j) ok = a[i][j] == b[i][j];
      size_t n = 0;
      for (const std::string &x : a[i]) ok = ok && n < b[i].size() && x == b[i][n++];
      if (!ok || n != b[i].size()) ++bad;
    };
    for (int step = 0; step < 400000; ++step) {
      const size_t i = rnd(6), j = rnd(6);
      switch (rnd(10)) {
        case 0: case 1: case 2: { std::string w = word(); a[i].push_back(w); b[i].push_back(w); break; }
        case 3: { std::string w = word(); a[i].emplace_back(w.c_str()); b[i].emplace_back(w.c_str()); break; }
        case 4: a[i].clear(); b[i].clear(); break;
        case 5: { size_t n = rnd(7); a[i].resize(n); b[i].resize(n); break; }
        case 6: { size_t n = rnd(7); std::string w = word(); a[i].assign(n, w); b[i].assign(n, w); break; }
        case 7: a[i] = a[j]; b[i] = b[j]; break;
        case 8: if (i != j) { a[i] = std::move(a[j]); b[i] = std::move(b[j]); a[j].clear(); b[j].clear(); } break;
        default: { V c(a[j]); V d(std::move(c)); a[i] = d; b[i] = b[j]; if (!a[i].empty()) { a[i].back() += "x"; b[i].back() += "x"; } break; }
      }
      same(i);
      same(j);
    }
  }
  {
    std::vector<mh::Chain> a(5);
    std::vector<std::vector<int>> b(5);
    auto same = [&](size_t i) {
      ++checks;
      bool ok = a[i].size() == b[i].size() && a[i].empty() == b[i].empty() && (b[i].empty() || a[i].back() == b[i].back());
      for (size_t j = 0; ok && j < b[i].size(); ++j) ok = a[i][j] == b[i][j] && a[i].data()[j] == b[i][j];
      if (!ok) ++bad;
    };
    for (int step = 0; step < 400000; ++step) {
      const size_t i = rnd(5), j = rnd(5);
      switch (rnd(8)) {
        case 0: case 1: case 2: { int v = (int)rnd(1000); a[i].push_back(v); b[i].push_back(v); break; }
        case 3: if (!b[i].empty()) { a[i].pop_back(); b[i].pop_back(); } break;
        case 4: if (rnd(4) == 0) { a[i].clear(); b[i].clear(); } break;
        case 5: a[i] = a[j]; b[i] = b[j]; break;
        case 6: if (i != j && b[i].size() + b[j].size() < 300) { a[i].append(a[j].data(), a[j].size()); b[i].insert(b[i].end(), b[j].begin(), b[j].end()); } break;
        default: if (i != j) { mh::Chain c(std::move(a[j])); a[j].clear(); a[i] = mh::Chain(); a[i].append_reversed(c); a[j] = std::move(c);
                               b[i].assign(b[j].rbegin(), b[j].rend()); } break;
      }
      same(i);
      same(j);
    }
  }
  printf("container-selftest: %llu checks, %llu differ\n", (unsigned long long)checks, (unsigned long long)bad);
  return bad ? 1 : 0;
}

struct ReadFeeder {
  // sequences of a FASTA / FASTQ file (plain or gz), upper-cased, '\n' between records, in chunks of whole records.
  // Lines are taken block-wise as views (no per-line allocation); FASTQ records are four lines (header, sequence,
  // '+', qualities), FASTA sequences may span lines.
  explicit ReadFeeder(const std::string &path) : in_(path) {}
  bool next_chunk(std::string &out, size_t target) {
    out.clear();
    while (out.size() < target) {
      if (li_ == lines_.size()) {
        if (done_) break;
        li_ = 0;
        if (!in_.next_block(store_, lines_, 1u << 20, 32u << 20, true)) done_ = true;
        if (lines_.empty()) continue;
      }
      for (; li_ < lines_.size() && out.size() < target; ++li_) {
        const char *b = lines_[li_].b, *e = lines_[li_].e;
        if (format_ == 0) {
          if (b == e) continue;                   // blank lines before the first record
          format_ = *b == '>' ? 1 : 2;            // by the first byte of the file, whatever -f says
        }
        if (format_ == 1 && b == e) continue;     // blank line inside a FASTA file
        if (format_ == 2) {  // FASTQ
          if (phase_ == 1) {
            append_upper(out, b, e);
            out.push_back('\n');
          }
          phase_ = (phase_ + 1) & 3;
        } else if (*b == '>') {  // FASTA header: the previous record ends here
          if (open_) out.push_back('\n');
          open_ = true;
        } else {
          append_upper(out, b, e);
        }
      }
      if (format_ == 1 && open_ && out.size() >= target) {  // a FASTA record larger than a chunk is cut with k-mers
        // lost at the seam only if a chunk ends inside it: keep going to the end of the record instead
        while (true) {
          if (li_ == lines_.size()) {
            if (done_) break;
            li_ = 0;
            if (!in_.next_block(store_, lines_, 1u << 20, 32u << 20, true)) done_ = true;
            if (lines_.empty()) continue;
          }
          if (lines_[li_].b != lines_[li_].e && *lines_[li_].b == '>') break;
          append_upper(out, lines_[li_].b, lines_[li_].e);
          ++li_;
        }
      }
    }
    if (done_ && li_ == lines_.size() && open_) {
      out.push_back('\n');
      open_ = false;
    }
    return !out.empty();
  }

 private:
  static void append_upper(std::string &out, const char *b, const char *e) {
    const size_t o = out.size();
    out.resize(o + (size_t)(e - b));
    char *d = &out[o];
    for (const char *p = b; p < e; ++p) *d++ = (char)(*p & 0xDF);  // a-z -> A-Z; nothing else can become A, C, G or T
  }
  mh::BlockLineReader in_;
  mh::TextBuf store_;
  std::vector<mh::BlockLineReader::View> lines_;
  size_t li_ = 0;
  int format_ = 0, phase_ = 0;
  bool done_ = false, open_ = false;
};

struct Counter {
  mg_counter *c = nullptr;
  ~Counter() { mg_count_destroy(c); }
};

constexpr size_t READ_CHUNK = 64u << 20;  // read bytes per mg_count_add (count and call --reads)

// STEP 2 with --reads: the sample's reads counted on the device, restricted to the ref_k-mers the index of c can use,
// then scanned from there (mg_scan_counted).  The counters end up as they would after `count` (-ci2 -cs255 -cx1e9,
// its defaults and the MALVA wrapper's) and the scan of that database, with no database written.  A thread parses
// the next chunk of reads while the device counts this one.
void scan_reads(const Options &o, mg_ctx *c, mg_counter *cn, const std::string &path) {
  Stopwatch sw;
  uint64_t st0[6] = {}, st[6] = {};  // (the device time of the counting kernels adds up over the counter's life)
  if (o.trace) gpu(mg_count_stats(cn, st0, 6), "mg_count_stats");
  gpu(mg_count_reset(cn), "mg_count_reset");
  gpu(mg_count_restrict(cn, c), "mg_count_restrict");
  ReadFeeder feed(path);
  std::string cur, next;
  uint64_t bytes = 0;
  double t_read = 0, t_wait = 0, t_count = 0;
  bool more = feed.next_chunk(cur, READ_CHUNK);
  t_read += sw.lap();
  while (more) {
    std::future<bool> ahead = std::async(std::launch::async, [&] {
      Stopwatch r;
      const bool m = feed.next_chunk(next, READ_CHUNK);
      t_read += r.lap();
      return m;
    });
    bytes += cur.size();
    gpu(mg_count_add(cn, cur.data(), cur.size()), "mg_count_add");
    t_count += sw.lap();
    more = ahead.get();
    t_wait += sw.lap();
    std::swap(cur, next);
  }
  uint64_t n = 0;
  gpu(mg_count_finish(cn, 2, 255, 1000000000ull, &n), "mg_count_finish");
  gpu(mg_scan_counted(c, cn), "mg_scan_counted");
  t_count += sw.lap();
  if (o.trace) {
    gpu(mg_count_stats(cn, st, 6), "mg_count_stats");
    fprintf(stderr, "[trace] reads %s: %llu read bytes, %llu windows examined, %llu distinct kept (%llu seen twice or "
                    "more), table capacity %llu slots; reading %.1f ms (%.1f ms waited for), counting + scan %.1f ms "
                    "(counting kernels %.1f ms)\n",
            path.c_str(), (unsigned long long)bytes, (unsigned long long)st[5], (unsigned long long)st[0],
            (unsigned long long)n, (unsigned long long)st[2], t_read, t_wait, t_count, (double)(st[4] - st0[4]) * 1e-3);
  }
}

// Before every chunk, a counter's table grows to 2 x (distinct + chunk) slots, so that an insert never meets a full
// table: from the second 64 MB chunk of a sample on, 2^28 slots (8.6 GB).  Sample sets take the device memory left
// free, so a cohort grows its counters to that size before it plans them: one poly-A read and 128 MB of record
// separators.
void grow_counter(mg_counter *cn, unsigned k) {
  std::string warm(2 * READ_CHUNK, '\n');
  std::fill_n(warm.begin(), k, 'A');
  gpu(mg_count_add(cn, warm.data(), warm.size()), "mg_count_add");
}

// STEP 2: the sample k-mer scan (main.cpp:482-500) of one database.  Raw suffix records go through rings of pinned
// buffers, one ring per device, chunks dealt round-robin; the library copies and scans them asynchronously
// (double-buffered on its side), a buffer is refilled only after the event recorded behind its scan has completed.
// With several contexts the counters are then added up on the first one (all updates are commutative adds,
// main.cpp:495-499).
void scan_kmc(const Options &o, std::vector<mg_ctx *> gs, mh::KmcDb &db, const std::string &path) {
  const int n_dev = (int)gs.size();
  constexpr int RING = 4;
  constexpr uint64_t CHUNK = 1ull << 22;  // records per buffer
  std::vector<uint8_t *> buf((size_t)(n_dev * RING), nullptr);
  std::vector<char> used((size_t)(n_dev * RING), 0);
  Stopwatch sw;
  for (int d = 0; d < n_dev; ++d) {
    gpu(mg_kmc_open(gs[(size_t)d], db.lut.data(), db.lut.size(), db.lut_prefix_len, db.kmer_len, db.counter_size,
                    db.min_count, db.max_count),
        "mg_kmc_open");
    for (int s = 0; s < RING; ++s) gpu(mg_host_alloc((void **)&buf[(size_t)(d * RING + s)], CHUNK * db.record_bytes + 64), "mg_host_alloc");
  }
  uint64_t first = 0;
  double t_alloc = sw.lap(), t_wait = 0, t_read = 0, t_submit = 0;
  for (uint64_t chunk = 0;; ++chunk) {
    const int d = (int)(chunk % (uint64_t)n_dev), slot = d * RING + (int)((chunk / (uint64_t)n_dev) % RING);
    mg_ctx *c = gs[(size_t)d];
    if (used[(size_t)slot]) gpu(mg_event_sync(c, 32 + slot % RING), "mg_event_sync");
    t_wait += sw.lap();
    uint64_t n = db.read_records(buf[(size_t)slot], first, CHUNK);
    t_read += sw.lap();
    if (n == 0) break;
    gpu(mg_scan_kmc_records(c, buf[(size_t)slot], first, n), "mg_scan_kmc_records");
    gpu(mg_event_record(c, 32 + slot % RING), "mg_event_record");
    t_submit += sw.lap();
    used[(size_t)slot] = 1;
    first += n;
  }
  for (mg_ctx *x : gs) gpu(mg_sync(x), "mg_sync");
  const double t_drain = sw.lap();
  for (auto &b : buf) mg_host_free(b);
  if (o.trace)
    fprintf(stderr, "[trace] KMC scan: %llu records; pinned buffers %.1f ms, file reads %.1f ms, waiting for a free buffer "
                    "%.1f ms, submitting %.1f ms, draining %.1f ms, freeing %.1f ms\n",
            (unsigned long long)first, t_alloc, t_read, t_wait, t_submit, t_drain, sw.lap());
  if (first != db.total_kmers) throw std::runtime_error(path + ".kmc_suf is shorter than its header says");
  if (n_dev > 1) gpu(mg_reduce_counts(gs.data(), n_dev), "mg_reduce_counts");
}

// STEP 3: genotype (main.cpp:504-581), one pass over the VCF.  outs[s] receives the VCF body of output s.  Without
// sets: the live counters of gs[0] (mg_genotype_packed, one output).  With sets: context i holds a sample set of
// sets[i] samples, and they are the next sets[i] outputs after those of contexts 0..i-1 (mg_genotype_samples_packed,
// every context on its own worker, all on the same read-only batch).  Three stages on three threads: enumerate
// (EnumeratedBatches) | device (below) | format + write (this thread).
void genotype_pass(const Options &o, const std::vector<mg_ctx *> &gs, const std::vector<int> &sets,
                   EnumeratedBatches &batches, const std::vector<FILE *> &outs) {
  const size_t n_out = outs.size();
  std::vector<size_t> set_first(sets.size(), 0);
  for (size_t i = 1; i < sets.size(); ++i) set_first[i] = set_first[i - 1] + (size_t)sets[i - 1];
  Channel<std::unique_ptr<Batch>> done(2);
  std::exception_ptr dev_err;
  std::thread device([&] {
    try {
      std::unique_ptr<Batch> b;
      std::vector<mg_genotype_out> res(n_out);
      while (batches.next(b)) {
        Stopwatch sw;
        const mh::SignatureCsr &sg = b->sigs;
        const uint64_t nv = sg.n_variants(), na = sg.n_alleles();
        if (nv) {
          if (o.verbose) {
            b->lik_off.assign(nv + 1, 0);
            for (uint64_t i = 0; i < nv; ++i) {
              uint64_t n = sg.var_allele_off[i + 1] - sg.var_allele_off[i];
              b->lik_off[i + 1] = b->lik_off[i] + std::max<uint64_t>(n, o.haploid ? n : n * (n + 1) / 2);
            }
            b->lik.assign(b->lik_off[nv] * n_out, 0.0);
          }
          // (a recycled batch: nothing of its previous results may show through)
          b->cov.assign(na * n_out, 0);
          b->n_gts.assign(nv * n_out, 0), b->status.assign(nv * n_out, 0), b->best.assign(nv * n_out, 0);
          b->gq.assign(nv * n_out, 0);
          mg_packed_batch in = {nv,
                                sg.var_allele_off.data(),
                                sg.allele_sig_off.data(),
                                sg.sig_kmer_off.data(),
                                sg.kmers.data(),
                                sg.freq.data(),
                                sg.n_irregular(),
                                sg.irr_off.data(),
                                sg.irr_pool.data(),
                                sg.irr_kmer.data()};
          for (size_t s = 0; s < n_out; ++s)
            res[s] = {b->cov.data() + s * na, b->n_gts.data() + s * nv, b->status.data() + s * nv,
                      b->best.data() + s * nv, b->gq.data() + s * nv, o.verbose ? b->lik_off.data() : nullptr,
                      o.verbose ? b->lik.data() + s * b->lik_off[nv] : nullptr};
          if (sets.empty())
            gpu(mg_genotype_packed(gs[0], &in, res.data(), o.error_rate, (int)o.max_coverage, o.haploid ? 1 : 0),
                "mg_genotype_packed");
          else
            parallel_for(gs.size(), (int)gs.size(), [&](size_t i) {
              gpu(mg_genotype_samples_packed(gs[i], &in, res.data() + set_first[i], sets[i], o.error_rate,
                                             (int)o.max_coverage, o.haploid ? 1 : 0),
                  "mg_genotype_samples_packed");
            });
        }
        b->t_dev = sw.lap();
        done.push(std::move(b));
      }
    } catch (...) {
      dev_err = std::current_exception();
    }
    done.close();
  });
  struct Joiner {  // (an exception below must not leave the thread running)
    std::thread &t;
    Channel<std::unique_ptr<Batch>> &c;
    ~Joiner() {
      c.close();
      if (t.joinable()) t.join();
    }
  } joiner{device, done};
  std::vector<const mh::Variant *> order;
  std::vector<std::string> text;
  std::unique_ptr<Batch> b;
  Stopwatch sw;
  while (done.pop(b)) {
    sw.lap();
    const mh::SignatureCsr &sg = b->sigs;
    const uint64_t nv = sg.n_variants(), na = sg.n_alleles();
    if (nv == 0) {
      batches.recycle(std::move(b));
      continue;
    }
    order.clear();
    for (const auto &blk : b->vb.blocks)
      for (size_t i = 0; i < blk.size(); ++i) order.push_back(&blk[i]);
    const size_t chunk = 4096, n_chunks = (nv + chunk - 1) / chunk;
    if (text.size() < n_chunks * n_out) text.resize(n_chunks * n_out);
    for (size_t c = 0; c < n_chunks * n_out; ++c) text[c].clear();  // (capacity kept from batch to batch)
    parallel_for(n_chunks * n_out, o.threads, [&](size_t t) {
      const size_t s = t / n_chunks, c = t % n_chunks;
      const uint32_t *cov = b->cov.data() + s * na;
      const int32_t *n_gts = b->n_gts.data() + s * nv, *status = b->status.data() + s * nv,
                    *best = b->best.data() + s * nv, *gq = b->gq.data() + s * nv;
      const double *lik = o.verbose ? b->lik.data() + s * b->lik_off[nv] : nullptr;
      for (size_t i = c * chunk; i < std::min<size_t>(nv, (c + 1) * chunk); ++i)
        format_variant(*order[i], cov + sg.var_allele_off[i], n_gts[i], status[i], best[i], gq[i],
                       o.verbose ? lik + b->lik_off[i] : nullptr, o, text[t]);
    });
    for (size_t s = 0; s < n_out; ++s)
      for (size_t c = 0; c < n_chunks; ++c) fwrite(text[s * n_chunks + c].data(), 1, text[s * n_chunks + c].size(), outs[s]);
    if (o.trace)
      fprintf(stderr, "[trace] call batch: %llu variants, %llu k-mers: read+decode wait %.1f ms, enumerate %.1f ms, device %.1f ms, print %.1f ms\n",
              (unsigned long long)nv, (unsigned long long)sg.n_kmers(), b->t_parse, b->t_enum, b->t_dev, sw.lap());
    batches.recycle(std::move(b));
  }
  device.join();
  if (dev_err) std::rethrow_exception(dev_err);
  batches.join();
}

std::string base_name(const std::string &path) {
  const size_t p = path.find_last_of('/');
  return p == std::string::npos ? path : path.substr(p + 1);
}

int call_main(int argc, char **argv) {
  Options o;
  if (!parse_arguments(argc, argv, o, 3, true)) return EXIT_FAILURE;
  const size_t n_db = o.kmc_paths.size();
  if (!o.sample_devices.empty() && o.devices_given) {
    std::cerr << "ERROR: --sample-devices goes with neither --devices nor --device (--devices deals the records of one "
                 "KMC database over devices, --device picks the one device of a run, --sample-devices lists the "
                 "devices of several databases)"
              << std::endl;
    return 1;
  }
  if (!o.sample_devices.empty() && n_db == 1) {
    std::cerr << "ERROR: --sample-devices is for several KMC databases (call [opts] ref.fa vars.vcf DB1 DB2 .. --out-dir "
                 "DIR); one database goes over several devices with --devices"
              << std::endl;
    return 1;
  }
  if (n_db > 1 && o.out_dir.empty()) {
    std::cerr << "ERROR: several KMC databases need --out-dir DIR (sample P is written to DIR/basename(P).vcf)"
              << std::endl;
    return 1;
  }
  if (n_db == 1 && !o.out_dir.empty()) {
    std::cerr << "ERROR: --out-dir is for several KMC databases; with one the VCF goes to stdout" << std::endl;
    return 1;
  }
  if (n_db > 1 && o.devices.size() > 1) {
    std::cerr << "ERROR: --devices takes one KMC database; several databases run on one device (--device N) or are "
                 "spread over devices with --sample-devices A,B,.."
              << std::endl;
    return 1;
  }
  for (size_t i = 0; i < n_db; ++i)
    for (size_t j = 0; j < i; ++j)
      if (base_name(o.kmc_paths[i]) == base_name(o.kmc_paths[j])) {
        std::cerr << "ERROR: two KMC databases are named " << base_name(o.kmc_paths[i])
                  << ": both would be written to " << o.out_dir << "/" << base_name(o.kmc_paths[i]) << ".vcf (given twice)"
                  << std::endl;
        return 1;
      }
  if (o.reads) {
    if (o.devices.size() > 1) {
      std::cerr << "ERROR: --reads takes no --devices: the counts of one sample are complete only after all its reads "
                   "(k-mers seen once are dropped), so its reads cannot be dealt over devices; several read files go "
                   "over devices with --sample-devices A,B,.."
                << std::endl;
      return 1;
    }
    if (o.ref_k > 63) {
      std::cerr << "ERROR: --reads counts the ref k-mers on the device, which counts k <= 63 (-r " << o.ref_k << ")"
                << std::endl;
      return 1;
    }
    for (const std::string &path : o.kmc_paths) {
      FILE *f = fopen(path.c_str(), "rb");
      if (!f) {
        std::cerr << "ERROR: cannot open " << path << std::endl;
        return 1;
      }
      fclose(f);
    }
  }
  if (!o.sample_devices.empty()) {  // (before any file is read; without a usable driver mg_create fails as for --devices)
    const int visible = mg_device_count();
    for (int d : o.sample_devices)
      if (visible >= 0 && (d < 0 || d >= visible)) {
        std::cerr << "ERROR: --sample-devices: device " << d << " is not visible (" << visible << " visible)" << std::endl;
        return 1;
      }
  }
  // the contexts: one database is dealt over the --devices replicas, several databases over the --sample-devices ones
  // (a device may be listed more than once: one context each)
  const std::vector<int> &ctx_devices = o.sample_devices.empty() ? o.devices : o.sample_devices;
  std::vector<std::future<int>> cuda_up;  // CUDA start-up on every device, overlapped with the file reading
  for (int d : ctx_devices) cuda_up.push_back(std::async(std::launch::async, [d] { return mg_warmup(d); }));
  auto stream = std::make_unique<BlockStream>(o, false);
  if (stream->samples_code != 0) {
    std::cerr << "ERROR: VCF samples subset (code: " << stream->samples_code << ")" << std::endl;
    return 1;
  }
  std::vector<std::unique_ptr<mh::KmcDb>> dbs;  // every database is opened before any work
  for (const std::string &path : o.reads ? std::vector<std::string>() : o.kmc_paths) {
    dbs.push_back(std::make_unique<mh::KmcDb>());
    std::string why;
    if (!dbs.back()->open(path, why)) {
      std::cerr << "ERROR: cannot open " << path << std::endl;
      return 1;
    }
  }
  // first VCF batch decoded while the index loads and the scan runs
  auto call_batches = std::make_unique<BatchPrefetcher>(*stream, LINES_PER_BATCH);
  // the reference FASTA is read while CUDA starts and the index loads (host-only work, 1.4 s for 250 Mbp)
  std::future<std::map<std::string, std::string>> refs_ready =
      std::async(std::launch::async, [&o] { return mh::read_fasta(o.fasta_path, o.strip_chr); });
  const int n_ctx = (int)ctx_devices.size();
  std::vector<Ctx> gs((size_t)n_ctx);
  Ctx &g = gs[0];  // the context that answers after the reduce
  {  // load the index: context_bf, bf, ref_bf (main.cpp:455-461) -- from the file onto the first context, then
     // device-to-device copies of its image onto the others
    mh::IndexReader r(o.vcf_path + ".c" + std::to_string(o.ref_k) + ".k" + std::to_string(o.k) + ".malvax.zst");
    if (r.k != o.k || r.ref_k != o.ref_k)
      throw std::runtime_error("the index was built with -k " + std::to_string(r.k) + " -r " + std::to_string(r.ref_k));
    std::vector<uint64_t> ctx_bits = r.read_bits(), bf_bits = r.read_bits(), keys = r.read_keys();
    std::vector<uint8_t> flags(keys.size() / 2, 1);
    // the filter size travels with the index, like the reference's serialised bit vectors (-b matters at index time)
    gpu(mg_create(&g.c, ctx_devices[0], (int)o.k, (int)o.ref_k, r.bf_bits), "mg_create");
    gpu(mg_import_set_bits(g.c, 0, bf_bits.data(), bf_bits.size()), "mg_import_set_bits");
    gpu(mg_add_signatures_packed(g.c, keys.data(), flags.data(), flags.size()), "mg_add_signatures_packed");
    gpu(mg_finalize_alt(g.c), "mg_finalize_alt");
    gpu(mg_import_set_bits(g.c, 1, ctx_bits.data(), ctx_bits.size()), "mg_import_set_bits");
    gpu(mg_finalize_context(g.c), "mg_finalize_context");
    for (int i = 1; i < n_ctx; ++i) gpu(mg_replicate(&gs[(size_t)i].c, g.c, ctx_devices[(size_t)i]), "mg_replicate");
  }
  std::vector<mg_ctx *> cs;
  for (Ctx &x : gs) cs.push_back(x.c);
  // --reads: one counter per context, reset between its samples (its table keeps the size it grew to)
  std::vector<Counter> counters(o.reads ? (size_t)n_ctx : 0);
  for (size_t i = 0; i < counters.size(); ++i) {
    gpu(mg_count_create(&counters[i].c, ctx_devices[i], (int)o.ref_k), "mg_count_create");
    if (n_db > 1) grow_counter(counters[i].c, o.ref_k);
  }
  pelapsed("Reference parsing");
  std::map<std::string, std::string> refs = refs_ready.get();
  pelapsed("Reference processed");
  // (host only: the first batches are decoded and enumerated while the KMC records stream through the device)
  auto batches = std::make_unique<EnumeratedBatches>(*call_batches, refs, o);

  if (n_db == 1) {
    pelapsed("KMC output processing");
    if (o.reads)
      scan_reads(o, g.c, counters[0].c, o.kmc_path);
    else
      scan_kmc(o, cs, *dbs[0], o.kmc_path);
    for (size_t d = 1; d < gs.size(); ++d) {  // the replicas are no longer needed
      mg_destroy(gs[d].c);
      gs[d].c = nullptr;
    }
    pelapsed("BF weights created");
    std::cout << stream->header().cleaned(o.verbose);
    pelapsed("VCF parsing and genotyping");
    genotype_pass(o, {g.c}, {}, *batches, {stdout});
  } else {
    // several samples, in rounds: every context takes a sample set of up to MG_SAMPLE_SET_MAX (as many as device
    // memory holds), and a round's sets share one VCF pass.  Each context scans its samples one after the other into
    // its live counters and moves each into its column; the contexts scan at the same time, each on its own thread.
    // The index, the FASTA and the CUDA contexts serve every round.
    if (mkdir(o.out_dir.c_str(), 0777) != 0 && errno != EEXIST)
      throw std::runtime_error("cannot create " + o.out_dir + ": " + strerror(errno));
    const std::string header = stream->header().cleaned(o.verbose);
    for (size_t first = 0; first < n_db;) {
      // a round takes the next samples in command-line order: ceil(remaining / contexts) each, as far as they fit.
      // Planned one context after the other: contexts on one device share its memory.
      const size_t per_ctx = (n_db - first + (size_t)n_ctx - 1) / (size_t)n_ctx;
      std::vector<int> sets((size_t)n_ctx, 0);
      size_t n = 0;
      for (size_t i = 0; i < (size_t)n_ctx; ++i) {
        int fit = 0;
        gpu(mg_samples_capacity(cs[i], &fit), "mg_samples_capacity");
        sets[i] = (int)std::min({per_ctx, (size_t)fit, n_db - first - n});
        if (sets[i] > 0) gpu(mg_samples_begin(cs[i], sets[i]), "mg_samples_begin");
        n += (size_t)sets[i];
      }
      if (n == 0) throw std::runtime_error("not even one sample column fits in device memory next to the index");
      if (o.trace) {
        std::string plan;
        for (int x : sets) plan += " " + std::to_string(x);
        fprintf(stderr, "[trace] round of %zu samples, sets per context:%s\n", n, plan.c_str());
      }
      std::vector<mg_ctx *> set_ctx;  // the contexts with a set this round, and their sets
      std::vector<int> set_n;
      for (size_t i = 0; i < (size_t)n_ctx; ++i)
        if (sets[i] > 0) set_ctx.push_back(cs[i]), set_n.push_back(sets[i]);
      if (first > 0) {  // a fresh VCF pass (the previous group's has ended)
        batches.reset();
        call_batches.reset();
        stream = std::make_unique<BlockStream>(o, false);
        call_batches = std::make_unique<BatchPrefetcher>(*stream, LINES_PER_BATCH);
        batches = std::make_unique<EnumeratedBatches>(*call_batches, refs, o);
      }
      pelapsed("KMC output processing");
      std::vector<size_t> set_first(set_n.size(), first);
      for (size_t i = 1; i < set_n.size(); ++i) set_first[i] = set_first[i - 1] + (size_t)set_n[i - 1];
      parallel_for(set_ctx.size(), (int)set_ctx.size(), [&](size_t i) {
        mg_counter *cn = nullptr;
        for (size_t j = 0; j < (size_t)n_ctx && o.reads; ++j)
          if (cs[j] == set_ctx[i]) cn = counters[j].c;
        for (int s = 0; s < set_n[i]; ++s) {
          const size_t db = set_first[i] + (size_t)s;
          if (o.reads)
            scan_reads(o, set_ctx[i], cn, o.kmc_paths[db]);
          else
            scan_kmc(o, {set_ctx[i]}, *dbs[db], o.kmc_paths[db]);
          gpu(mg_samples_take(set_ctx[i], s), "mg_samples_take");
        }
      });
      pelapsed("BF weights created");
      std::vector<FILE *> outs;
      struct Files {  // (closed on every way out)
        std::vector<FILE *> &f;
        ~Files() {
          for (FILE *x : f) fclose(x);
        }
      } files{outs};
      for (size_t s = 0; s < n; ++s) {
        const std::string path = o.out_dir + "/" + base_name(o.kmc_paths[first + s]) + ".vcf";
        FILE *f = fopen(path.c_str(), "wb");
        if (!f) throw std::runtime_error("cannot write " + path + ": " + strerror(errno));
        outs.push_back(f);
        fwrite(header.data(), 1, header.size(), f);
      }
      pelapsed("VCF parsing and genotyping");
      genotype_pass(o, set_ctx, set_n, *batches, outs);
      for (FILE *f : outs)
        if (fflush(f) != 0) throw std::runtime_error("cannot write to " + o.out_dir + ": " + strerror(errno));
      for (mg_ctx *c : set_ctx) gpu(mg_samples_end(c), "mg_samples_end");
      first += n;
    }
  }
  pelapsed("Processed " + std::to_string(stream->n_records) + " variants");
  fflush(stdout);
  pelapsed("Execution completed");
  finish(0);
}

// ------------------------------------------------------------------------------------------------
// CPU-only: print the signatures of every block, for the parity tests of the host logic against the reference's
// VB::extract_kmers.  One line per signature: contig \t 1-based pos \t block-local variant index \t allele \t kmers
int signatures_main(int argc, char **argv) {
  Options o;
  if (!parse_arguments(argc, argv, o, 2)) return EXIT_FAILURE;
  mh::count_rows() = o.trace;
  BlockStream stream(o, o.index_blocks);
  if (stream.samples_code != 0) {
    std::cerr << "ERROR: VCF samples subset (code: " << stream.samples_code << ")" << std::endl;
    return 1;
  }
  std::map<std::string, std::string> refs = mh::read_fasta(o.fasta_path, o.strip_chr);
  BlockBatch batch;
  std::vector<mh::VarBlock> &blocks = batch.blocks;
  mh::SignatureCsr sigs;
  uint64_t block_no = 0;
  const bool quiet = getenv("MALVA_SIGNATURES_QUIET") != nullptr;  // (timing runs: enumerate, print nothing)
  Stopwatch sw;
  double t_batch = 0, t_enum = 0;
  BatchPrefetcher ahead(stream, LINES_PER_BATCH);
  while (true) {
    sw.lap();
    const bool more = ahead.next(batch);  // (decoded one batch ahead, like in index / call)
    t_batch += sw.lap();
    if (!more) {
      if (o.trace)
        fprintf(stderr, "[trace] fixed-stride GT decode: %llu of %llu rows with samples\n",
                (unsigned long long)mh::fast_gt_rows().load(), (unsigned long long)mh::sample_rows().load());
      break;
    }
    enumerate_batch(blocks, refs, o, sigs);
    t_enum += sw.lap();
    if (o.trace)
      fprintf(stderr, "[trace] read %.1f + decode %.1f + group %.1f ms, enumerate %.1f ms (cumulative)\n", stream.t_read,
              stream.t_decode, stream.t_group, t_enum);
    if (quiet) continue;
    uint64_t vi = 0;
    for (const auto &b : blocks) {
      for (size_t i = 0; i < b.size(); ++i, ++vi) {
        const uint64_t a0 = sigs.var_allele_off[vi], a1 = sigs.var_allele_off[vi + 1];
        for (uint64_t a = a0; a < a1; ++a)
          for (uint64_t s = sigs.allele_sig_off[a]; s < sigs.allele_sig_off[a + 1]; ++s) {
            std::cout << block_no << '\t' << *b.contig << '\t' << b[i].ref_pos + 1 << '\t' << i << '\t' << (a - a0) << '\t';
            for (uint64_t q = sigs.sig_kmer_off[s]; q < sigs.sig_kmer_off[s + 1]; ++q) {
              if (q != sigs.sig_kmer_off[s]) std::cout << ',';
              std::cout << sigs.text(q, (int)o.k);
            }
            std::cout << '\n';
          }
      }
      ++block_no;
    }
  }
  std::cout << "#used";
  for (const auto &n : stream.used_seq_names) std::cout << '\t' << n;
  std::cout << '\n';
  return 0;
}

// The 2-bit copy of the reads that `count` keeps while it counts (mg_count_add_keep): segments in host memory up to
// a budget, the rest in one spill file.  The file is unlinked as soon as it is created, so that it goes away with
// the process on every exit path.
class PackedStore {
 public:
  PackedStore(uint64_t budget, std::string dir) : budget_(budget), dir_(std::move(dir)) {}
  ~PackedStore() {
    if (fp_) fclose(fp_);
  }
  PackedStore(const PackedStore &) = delete;
  PackedStore &operator=(const PackedStore &) = delete;

  void add(const uint8_t *b, uint64_t nb, const uint32_t *l, uint64_t nr) {
    if (!nr) return;
    Seg g{nb, nr, -1, {}, {}};
    if (in_mem_ + nb + 4 * nr <= budget_) {
      g.bytes.assign(b, b + nb);
      g.lens.assign(l, l + nr);
      in_mem_ += nb + 4 * nr;
    } else {
      if (!fp_) open_spill();
      g.at = (int64_t)spilled_;
      if (fwrite(b, 1, nb, fp_) != nb || fwrite(l, 4, nr, fp_) != nr)
        throw std::runtime_error("short write on the spill file in " + dir_);
      spilled_ += nb + 4 * nr;
    }
    bytes_ += nb;
    runs_ += nr;
    segs_.push_back(std::move(g));
  }
  // f(packed, n_bytes, run_len, n_runs) over every segment, in the order they were added
  void each(const std::function<void(const uint8_t *, uint64_t, const uint32_t *, uint64_t)> &f) {
    if (fp_ && fflush(fp_) != 0) throw std::runtime_error("cannot flush the spill file in " + dir_);
    std::vector<uint8_t> buf;
    for (const Seg &g : segs_) {
      if (g.at < 0) {
        f(g.bytes.data(), g.nb, g.lens.data(), g.nr);
        continue;
      }
      buf.resize(g.nb + 4 * g.nr + 4);
      uint8_t *lens = buf.data() + ((g.nb + 3) & ~3ull);
      if (fseeko(fp_, (off_t)g.at, SEEK_SET) != 0 || fread(buf.data(), 1, g.nb, fp_) != g.nb ||
          fread(lens, 4, g.nr, fp_) != g.nr)
        throw std::runtime_error("cannot read back the spill file in " + dir_);
      f(buf.data(), g.nb, reinterpret_cast<const uint32_t *>(lens), g.nr);
    }
    if (fp_) fseeko(fp_, 0, SEEK_END);
  }
  uint64_t bytes() const { return bytes_; }
  uint64_t runs() const { return runs_; }
  uint64_t in_memory() const { return in_mem_; }
  uint64_t spilled() const { return spilled_; }
  const std::string &spill_path() const { return path_; }

 private:
  struct Seg {
    uint64_t nb, nr;
    int64_t at;  // offset in the spill file, -1: in memory
    std::vector<uint8_t> bytes;
    std::vector<uint32_t> lens;
  };
  void open_spill() {
    std::string t = dir_ + "/malva-count-XXXXXX";
    int fd = mkstemp(&t[0]);
    if (fd < 0) throw std::runtime_error("cannot create a spill file in " + dir_ + ": " + strerror(errno));
    unlink(t.c_str());
    fp_ = fdopen(fd, "w+b");
    if (!fp_) {
      close(fd);
      throw std::runtime_error("cannot open the spill file in " + dir_);
    }
    path_ = t;
  }
  uint64_t budget_, in_mem_ = 0, spilled_ = 0, bytes_ = 0, runs_ = 0;
  std::string dir_, path_;
  FILE *fp_ = nullptr;
  std::vector<Seg> segs_;
};

// half of MemAvailable: the host memory the packed copy may take before it goes to the spill file
uint64_t default_store_budget() {
  if (const char *e = getenv("MG_COUNT_HOST_BUDGET")) return strtoull(e, nullptr, 10);  // (tests force the spill)
  FILE *fp = fopen("/proc/meminfo", "r");
  unsigned long long kb = 0;
  if (fp) {
    char line[256];
    while (fgets(line, sizeof(line), fp))
      if (sscanf(line, "MemAvailable: %llu kB", &kb) == 1) break;
    fclose(fp);
  }
  return kb * 1024 / 2;
}

// a range of canonical k-mers: those whose top `bits` bits lie in [lo, hi) (bits = 0: all of them)
struct PrefixRange {
  int bits;
  uint32_t lo, hi;
};

// ------------------------------------------------------------------------------------------------
// `kmc -k43 -ci2 -cs255 -m4 -t1 -fm <sample> <out_prefix> <tmp>` (MALVA:107) on the GPU.  Flags come joined to their
// value like kmc's (-k43) or separated (-k 43); -m / -t / -f* are accepted and ignored (the file format is detected
// from its first byte).  The input is read once: while the device counts it, it also keeps a 2-bit copy of the
// countable bases (host memory up to half of what is available, then a spill file in tmp_dir, by default the
// directory of the output prefix).  When the k-mer table would outgrow the device, counting goes on in
// prefix-partitioned passes over that copy, in ascending prefix order; a range that still does not fit is split in
// two.  --passes N asks for N such passes from the start.
int count_main(int argc, char **argv) {
  unsigned k = 43, ci = 2, cs = 255, passes = 1;
  unsigned long long cx = 1000000000ull;
  int device = 0;
  bool trace = false;
  std::vector<std::string> pos;
  auto value = [&](const std::string &a, size_t skip, int &i) -> std::string {
    if (a.size() > skip) return a.substr(skip);
    if (i + 1 < argc) return argv[++i];
    throw std::runtime_error("missing value for " + a);
  };
  for (int i = 1; i < argc; ++i) {
    std::string a = argv[i];
    if (a == "--passes") passes = (unsigned)atoi(value(a, a.size(), i).c_str());
    else if (a == "--device") device = atoi(value(a, a.size(), i).c_str());
    else if (a == "--trace") trace = true;
    else if (a.compare(0, 3, "-ci") == 0) ci = (unsigned)atoi(value(a, 3, i).c_str());
    else if (a.compare(0, 3, "-cs") == 0) cs = (unsigned)atoi(value(a, 3, i).c_str());
    else if (a.compare(0, 3, "-cx") == 0) cx = strtoull(value(a, 3, i).c_str(), nullptr, 10);
    else if (a.compare(0, 2, "-k") == 0) k = (unsigned)atoi(value(a, 2, i).c_str());
    else if (a.compare(0, 2, "-m") == 0 || a.compare(0, 2, "-t") == 0) (void)value(a, 2, i);
    else if (a.compare(0, 2, "-f") == 0 || a == "-v" || a.compare(0, 2, "-p") == 0 || a.compare(0, 2, "-s") == 0 ||
             a.compare(0, 2, "-n") == 0 || a == "-r") continue;
    else if (a == "-b") throw std::runtime_error("-b (non-canonical counting) is not supported: MALVA needs canonical k-mers");
    else if (!a.empty() && a[0] == '-') throw std::runtime_error("unknown option " + a);
    else pos.push_back(a);
  }
  if (pos.size() < 2 || passes < 1 || passes > 256) {
    std::cerr << "Usage: malva-geno count [-k43] [-ci2] [-cs255] [-cx1000000000] [--passes N] [--device N] [--trace] "
                 "<reads.fq|fa[.gz]> <kmc_output_prefix> [tmp_dir]\n";
    return 1;
  }
  if (cs > 255) throw std::runtime_error("-cs above 255 is not supported (one counter byte per record)");
  std::string spill_dir = pos.size() > 2 ? pos[2] : pos[1].substr(0, pos[1].find_last_of('/') + 1);
  if (spill_dir.empty()) spill_dir = ".";
  pelapsed("k-mer counting");
  Counter cn;
  gpu(mg_count_create(&cn.c, device, (int)k), "mg_count_create");
  std::deque<PrefixRange> plan;
  for (unsigned p = 0; p < passes; ++p)
    plan.push_back(passes > 1 ? PrefixRange{8, p * 256 / passes, (p + 1) * 256 / passes} : PrefixRange{0, 0, 0});
  const PrefixRange first = plan.front();
  gpu(mg_count_set_partition(cn.c, first.bits, first.lo, first.hi), "mg_count_set_partition");

  // one read of the input: a thread parses the next chunk while the device counts and packs this one
  PackedStore store(default_store_budget(), spill_dir);
  ReadFeeder feed(pos[0]);
  std::string cur, next;
  std::vector<uint8_t> packed;
  std::vector<uint32_t> run_len;
  uint64_t total_bases = 0, st[9] = {}, at_overflow[9] = {};
  bool overflowed = false;
  Stopwatch sw;
  double t_read = 0, t_count = 0, t_wait = 0, t_passes = 0;
  bool more = feed.next_chunk(cur, READ_CHUNK);
  t_read += sw.lap();
  while (more) {
    std::future<bool> ahead = std::async(std::launch::async, [&] {
      Stopwatch r;
      const bool m = feed.next_chunk(next, READ_CHUNK);
      t_read += r.lap();
      return m;
    });
    packed.resize(cur.size() / 2 + 1);
    run_len.resize(cur.size() / (k + 1) + 2);
    uint64_t nb = 0, nr = 0;
    gpu(mg_count_add_keep(cn.c, cur.data(), cur.size(), packed.data(), packed.size(), run_len.data(), run_len.size(),
                          &nb, &nr),
        "mg_count_add_keep");
    store.add(packed.data(), nb, run_len.data(), nr);
    if (!overflowed) {
      gpu(mg_count_stats(cn.c, st, 9), "mg_count_stats");
      if (st[6]) {
        overflowed = true;
        memcpy(at_overflow, st, sizeof(st));
      }
    }
    total_bases += cur.size();
    t_count += sw.lap();
    more = ahead.get();
    t_wait += sw.lap();
    std::swap(cur, next);
  }
  std::string().swap(cur);
  std::string().swap(next);

  std::unique_ptr<mh::KmcWriter> w;
  std::vector<uint64_t> keys;
  std::vector<uint32_t> counts;
  uint64_t instances = 0, distinct = 0, n_passes = 0, n_splits = 0;
  auto write = [&](uint64_t n, uint64_t lut_n) {
    uint64_t s[4];
    gpu(mg_count_stats(cn.c, s, 4), "mg_count_stats");
    distinct += s[0];
    instances += s[1];
    keys.resize(2 * n);
    counts.resize(n);
    gpu(mg_count_download(cn.c, keys.data(), counts.data(), n), "mg_count_download");
    if (!w) w.reset(new mh::KmcWriter(pos[1], k, mh::KmcWriter::choose_prefix_len(k, lut_n), ci, cs));
    w->append(keys.data(), counts.data(), n);
  };
  if (!overflowed) {  // the first range is counted
    uint64_t n = 0;
    gpu(mg_count_finish(cn.c, ci, cs, cx, &n), "mg_count_finish");
    write(n, passes == 1 ? n : 1ull << 40);
    plan.pop_front();
  } else if (passes == 1) {
    // the first plan: the distinct k-mers per counted window so far, over all the windows, in ranges a quarter of
    // what the table held at the overflow; 4 ranges when it overflowed before it counted anything.  A range that
    // still does not fit is split below.
    const int bits = (int)std::min(30u, 2 * k);
    uint64_t n = 4;
    if (at_overflow[1]) {
      const double est = (double)at_overflow[0] / (double)at_overflow[1] * (double)total_bases;
      n = (uint64_t)std::ceil(est / (double)(at_overflow[2] / 4));
    }
    n = std::max<uint64_t>(4, std::min<uint64_t>(n, 1ull << bits));
    plan.clear();
    for (uint64_t p = 0; p < n; ++p)
      plan.push_back(PrefixRange{bits, (uint32_t)((p << bits) / n), (uint32_t)(((p + 1) << bits) / n)});
  }
  const uint64_t max_bits = std::min(30u, 2 * k);
  // the remaining ranges over the packed copy, in ascending order
  while (!plan.empty()) {
    const PrefixRange r = plan.front();
    plan.pop_front();
    Stopwatch pw;
    gpu(mg_count_reset(cn.c), "mg_count_reset");
    gpu(mg_count_set_partition(cn.c, r.bits, r.lo, r.hi), "mg_count_set_partition");
    int rc = MG_OK;
    store.each([&](const uint8_t *b, uint64_t nb, const uint32_t *l, uint64_t nr) {
      if (rc == MG_OK) rc = mg_count_add_packed(cn.c, b, nb, l, nr);
    });
    uint64_t n = 0;
    if (rc == MG_OK) rc = mg_count_finish(cn.c, ci, cs, cx, &n);
    t_passes += pw.lap();
    if (rc == MG_ERR_NOMEM) {  // split the range in two and count both halves, in order
      const std::string why = mg_last_error();
      PrefixRange a = r, b = r;
      if (r.hi - r.lo >= 2) {
        a.hi = b.lo = r.lo + (r.hi - r.lo) / 2;
      } else if ((uint64_t)r.bits < max_bits) {
        a = {r.bits + 1, 2 * r.lo, 2 * r.lo + 1};
        b = {r.bits + 1, 2 * r.lo + 1, 2 * r.lo + 2};
      } else {
        throw GpuError("the canonical k-mers of one " + std::to_string(r.bits) + "-bit prefix do not fit the k-mer "
                       "table: " + why);
      }
      plan.push_front(b);
      plan.push_front(a);
      ++n_splits;
      if (trace)
        fprintf(stderr, "[trace] count: prefix range %u..%u of %d bits split (%s)\n", r.lo, r.hi, r.bits, why.c_str());
      continue;
    }
    gpu(rc, "mg_count_add_packed / mg_count_finish");
    write(n, 1ull << 40);
    ++n_passes;
  }
  if (!w) w.reset(new mh::KmcWriter(pos[1], k, mh::KmcWriter::choose_prefix_len(k, 1ull << 40), ci, cs));
  w->close();
  if (trace) {
    gpu(mg_count_stats(cn.c, st, 9), "mg_count_stats");
    fprintf(stderr, "[trace] count: %llu read bytes, one read of the input; %s; packed copy %llu bytes in %llu runs "
                    "(%llu bytes in host memory, %llu bytes in %s); %llu passes over the copy, %llu splits; reading "
                    "%.1f ms (%.1f ms waited for), counting + packing %.1f ms, passes %.1f ms; device time: counting "
                    "kernels %.1f ms, host-to-device copies %.1f ms, packing %.1f ms\n",
            (unsigned long long)total_bases, overflowed ? "the table met its limit while reading" : "no overflow",
            (unsigned long long)store.bytes(), (unsigned long long)store.runs(), (unsigned long long)store.in_memory(),
            (unsigned long long)store.spilled(), store.spilled() ? store.spill_path().c_str() : "no spill file",
            (unsigned long long)n_passes, (unsigned long long)n_splits, t_read, t_wait, t_count, t_passes,
            st[4] * 1e-3, st[7] * 1e-3, st[8] * 1e-3);
  }
  std::cerr << "[malva-geno/count] " << total_bases << " read bytes, " << instances << " k-mer instances, " << distinct
            << " distinct, " << w->total() << " written (count >= " << ci << ", capped at " << cs << ")" << std::endl;
  pelapsed("k-mer counting complete");
  return 0;
}

// `kmc_dump`-like listing: "<k-mer>\t<count>" per record passing the database's count filter (host only)
int kmc_dump_main(int argc, char **argv) {
  if (argc != 2) {
    std::cerr << "Usage: malva-geno kmc-dump <kmc_output_prefix>\n";
    return 1;
  }
  mh::KmcDb db;
  std::string why;
  if (!db.open(argv[1], why)) {
    std::cerr << "ERROR: " << why << std::endl;
    return 1;
  }
  const uint32_t p = db.lut_prefix_len, sb = (db.kmer_len - p) / 4, single = 1u << (2 * p);
  constexpr uint64_t BLOCK = 1 << 16;
  std::vector<uint8_t> block(BLOCK * db.record_bytes);
  std::string kmer(db.kmer_len, 'A');
  size_t pi = 0;
  for (uint64_t i = 0; i < db.total_kmers; ++i) {
    while (pi + 1 < db.lut.size() && db.lut[pi + 1] <= i) ++pi;
    if (i % BLOCK == 0 && db.read_records(block.data(), i, BLOCK, 1) != std::min<uint64_t>(BLOCK, db.total_kmers - i))
      throw std::runtime_error("suffix file truncated");
    const uint8_t *rec = block.data() + (i % BLOCK) * db.record_bytes;
    uint64_t c = db.counter_size ? 0 : 1;
    for (uint32_t b = 0; b < db.counter_size; ++b) c |= (uint64_t)rec[sb + b] << (8 * b);
    if (c < db.min_count || c > db.max_count) continue;
    const uint32_t pfx = (uint32_t)(pi % single);
    for (uint32_t j = 0; j < p; ++j) kmer[j] = "ACGT"[(pfx >> (2 * (p - 1 - j))) & 3];
    for (uint32_t j = 0; j < 4 * sb; ++j) kmer[p + j] = "ACGT"[(rec[j >> 2] >> (2 * (3 - (j & 3)))) & 3];
    std::cout << kmer << '\t' << c << '\n';
  }
  return 0;
}

}  // namespace

int main(int argc, char **argv) {
  if (argc < 2) {
    std::cerr << "malva missing arguments" << std::endl << USAGE << std::endl;
    return 1;
  }
  try {
    if (strncmp(argv[1], "index", 5) == 0) return index_main(argc - 1, argv + 1);
    if (strncmp(argv[1], "call", 4) == 0) return call_main(argc - 1, argv + 1);
    if (strcmp(argv[1], "signatures") == 0) return signatures_main(argc - 1, argv + 1);
    if (strcmp(argv[1], "count") == 0) return count_main(argc - 1, argv + 1);
    if (strcmp(argv[1], "kmc-dump") == 0) return kmc_dump_main(argc - 1, argv + 1);
    if (strcmp(argv[1], "format-selftest") == 0) return format_selftest_main();
    if (strcmp(argv[1], "container-selftest") == 0) return container_selftest_main();
  } catch (const GpuError &e) {
    std::cerr << "malva-geno: GPU error: " << e.what() << " (there is no CPU fallback)" << std::endl;
    return 2;
  } catch (const std::exception &e) {
    std::cerr << "malva-geno: " << e.what() << std::endl;
    return 1;
  }
  std::cerr << "Could not interpret command " << argv[1] << "." << std::endl;
  std::cerr << "Accepted commands are index and call." << std::endl;
  return 1;
}
