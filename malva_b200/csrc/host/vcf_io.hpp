// Host-kept input side of malva-geno: gz-transparent line reader, FASTA reference, VCF header and record
// decoding with the htslib conventions the reference's output depends on (htslib itself is not part of this
// build: the records malva-geno needs are CHROM/POS/ID/REF/ALT/QUAL, one INFO float vector and the GT field):
//   * header lines are kept in file order, de-duplicated by key (+ID); `##FILTER=<ID=PASS,...>` always exists;
//     appending a line whose key/ID is already present is a no-op (bcf_hdr_append, main.cpp:190-204)
//   * sample subsetting (-s): kept samples stay in header order (bcf_hdr_set_samples, main.cpp:266,514)
//   * INFO floats are parsed with strtod and narrowed to float (variant.hpp:126-141)
//   * GT decode: allele index, '.' -> 0, phase taken from the separator before the second allele
//     (variant.hpp:158-211)
// Record decoding is a pure function of one text line, so that batches of lines are decoded in parallel.
#pragma once
#include <sys/stat.h>
#include <zlib.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "signatures.hpp"

namespace mh {

// A byte buffer whose resize() does not clear what it exposes (the readers overwrite it at once: clearing 12 MB per
// block first is a pass over memory for nothing).
template <class T>
struct NoInitAllocator : std::allocator<T> {
  template <class U>
  struct rebind {
    using other = NoInitAllocator<U>;
  };
  template <class U>
  void construct(U *p) noexcept(std::is_nothrow_default_constructible<U>::value) {
    ::new (static_cast<void *>(p)) U;
  }
  template <class U, class... A>
  void construct(U *p, A &&...a) {
    ::new (static_cast<void *>(p)) U(std::forward<A>(a)...);
  }
};
using TextBuf = std::vector<char, NoInitAllocator<char>>;

class LineReader {
 public:
  explicit LineReader(const std::string &path) : fp_(gzopen(path.c_str(), "r")) {
    if (!fp_) throw std::runtime_error("cannot open " + path);
    gzbuffer(fp_, 1 << 20);
    buf_.resize(1 << 20);
  }
  ~LineReader() {
    if (fp_) gzclose(fp_);
  }
  LineReader(const LineReader &) = delete;
  LineReader &operator=(const LineReader &) = delete;
  bool next(std::string &line) {
    line.clear();
    bool any = false;
    while (gzgets(fp_, buf_.data(), (int)buf_.size()) != nullptr) {
      any = true;
      size_t n = strlen(buf_.data());
      if (n && buf_[n - 1] == '\n') {
        line.append(buf_.data(), n - 1);
        if (!line.empty() && line.back() == '\r') line.pop_back();
        return true;
      }
      line.append(buf_.data(), n);
    }
    return any;
  }

 private:
  gzFile fp_;
  std::vector<char> buf_;
};

// MALVA_GENERAL_DECODE=1 in the environment switches the short cuts of this file off (block-parallel BGZF inflate,
// fixed-stride GT columns): the tests run both ways and compare.
inline bool general_decode_only() {
  static const bool on = getenv("MALVA_GENERAL_DECODE") != nullptr;
  return on;
}

// rows decoded by the fixed-stride GT short cut / rows with samples in all (reported by `signatures --trace`)
inline std::atomic<uint64_t> &fast_gt_rows() {
  static std::atomic<uint64_t> n{0};
  return n;
}
inline std::atomic<uint64_t> &sample_rows() {
  static std::atomic<uint64_t> n{0};
  return n;
}
inline bool &count_rows() {  // off unless tracing: the counters are shared by all decoding threads
  static bool on = false;
  return on;
}

// host threads the readers may use for block-parallel work (set once by the command-line driver; default: all)
inline int &io_threads() {
  static int n = (int)std::max(1u, std::thread::hardware_concurrency());
  return n;
}

// BGZF (bgzip / htslib: what .vcf.gz files in circulation are): a series of gzip members of at most 64 KB, each
// carrying its own compressed size in a "BC" extra field and its uncompressed size in its trailer -- so the members
// of a stretch of the file can be located without inflating anything and inflated side by side, each straight to its
// place in the caller's buffer.  (The reference reads through htslib, one member after the other on one thread.)
// CRC-32 and size of every member are checked, as zlib's gzread does for plain gzip.
class BgzfSource {
 public:
  // true if the file starts with a BGZF member header
  static bool is_bgzf(const std::string &path) {
    struct stat sb;  // (a pipe or FIFO is read once: no peeking at its first bytes)
    if (stat(path.c_str(), &sb) != 0 || !S_ISREG(sb.st_mode)) return false;
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) return false;
    unsigned char h[18];
    const size_t n = fread(h, 1, sizeof h, f);
    fclose(f);
    return n == sizeof h && header_ok(h);
  }
  explicit BgzfSource(const std::string &path) : f_(fopen(path.c_str(), "rb")) {
    if (!f_) throw std::runtime_error("cannot open " + path);
  }
  ~BgzfSource() {
    if (f_) fclose(f_);
  }
  BgzfSource(const BgzfSource &) = delete;
  BgzfSource &operator=(const BgzfSource &) = delete;

  // up to `want` bytes of the uncompressed stream; less only at the end of the file
  size_t read(char *dst, size_t want) {
    size_t done = 0;
    while (done < want) {
      if (spill_pos_ < spill_.size()) {  // what was left of a member that did not fit the previous request
        const size_t n = std::min(want - done, spill_.size() - spill_pos_);
        memcpy(dst + done, spill_.data() + spill_pos_, n);
        spill_pos_ += n;
        done += n;
        continue;
      }
      // the members of the next stretch that fit what is still wanted, whole
      struct Member {
        size_t in_off, in_len, out_off, out_len;
      };
      std::vector<Member> ms;
      size_t out = 0;
      bool full = false;
      while (!full && ms.size() < 8192) {
        // (refilling may move the buffer: only between stretches, never under members already picked)
        if (cend_ - cpos_ < 18) {
          if (!ms.empty()) break;
          if (!have(18)) break;
        }
        const unsigned char *h = cbuf_.data() + cpos_;
        if (!header_ok(h)) throw std::runtime_error("BGZF: bad member header");
        const size_t bsize = (size_t)(h[16] | (h[17] << 8)) + 1;
        if (bsize < 26) throw std::runtime_error("BGZF: bad member size");
        if (cend_ - cpos_ < bsize) {
          if (!ms.empty()) break;
          if (!have(bsize)) throw std::runtime_error("BGZF: truncated member");
          h = cbuf_.data() + cpos_;
        }
        const size_t isize = (size_t)h[bsize - 4] | ((size_t)h[bsize - 3] << 8) | ((size_t)h[bsize - 2] << 16) | ((size_t)h[bsize - 1] << 24);
        if (isize > want - done - out) {
          if (!ms.empty()) break;  // goes with the next stretch
          // a single member larger than the room left: inflate it aside, hand out its head
          spill_.resize(isize);
          spill_pos_ = 0;
          inflate_member(h, bsize, spill_.data(), isize);
          cpos_ += bsize;
          full = true;
          break;
        }
        ms.push_back(Member{cpos_, bsize, done + out, isize});
        out += isize;
        cpos_ += bsize;
      }
      if (full) continue;
      if (ms.empty()) break;  // end of the file
      const int t = (int)std::min<size_t>((size_t)io_threads(), (ms.size() + 15) / 16);
      if (t <= 1) {
        for (const Member &m : ms) inflate_member(cbuf_.data() + m.in_off, m.in_len, dst + m.out_off, m.out_len);
      } else {
        std::atomic<size_t> next{0};
        std::vector<std::exception_ptr> errs((size_t)t);
        std::vector<std::thread> pool;
        for (int w = 0; w < t; ++w)
          pool.emplace_back([&, w] {
            try {
              for (size_t i; (i = next.fetch_add(16)) < ms.size();)
                for (size_t j = i; j < std::min(ms.size(), i + 16); ++j)
                  inflate_member(cbuf_.data() + ms[j].in_off, ms[j].in_len, dst + ms[j].out_off, ms[j].out_len);
            } catch (...) {
              errs[(size_t)w] = std::current_exception();
              next.store(ms.size());
            }
          });
        for (auto &th : pool) th.join();
        for (auto &e : errs)
          if (e) std::rethrow_exception(e);
      }
      done += out;
    }
    return done;
  }

 private:
  static bool header_ok(const unsigned char *h) {
    return h[0] == 0x1f && h[1] == 0x8b && h[2] == 8 && h[3] == 4 && h[10] == 6 && h[11] == 0 && h[12] == 'B' && h[13] == 'C' &&
           h[14] == 2 && h[15] == 0;
  }
  // makes sure `n` bytes from cpos_ on are in cbuf_ (reading more of the file if need be); false at the end of the file
  bool have(size_t n) {
    if (cend_ - cpos_ >= n) return true;
    if (!eof_) {
      if (cpos_ > 0) {
        memmove(cbuf_.data(), cbuf_.data() + cpos_, cend_ - cpos_);
        cend_ -= cpos_;
        cpos_ = 0;
      }
      const size_t chunk = std::max<size_t>(n, (size_t)8 << 20);
      if (cbuf_.size() < cend_ + chunk) cbuf_.resize(cend_ + chunk);
      const size_t got = fread(cbuf_.data() + cend_, 1, chunk, f_);
      cend_ += got;
      if (got < chunk) eof_ = true;
    }
    if (cend_ - cpos_ >= n) return true;
    if (cend_ != cpos_) throw std::runtime_error("BGZF: truncated file");
    return false;
  }
  static void inflate_member(const unsigned char *h, size_t bsize, char *dst, size_t isize) {
    z_stream z;
    memset(&z, 0, sizeof z);
    if (inflateInit2(&z, -15) != Z_OK) throw std::runtime_error("BGZF: inflateInit2 failed");
    z.next_in = const_cast<unsigned char *>(h + 18);
    z.avail_in = (unsigned)(bsize - 18 - 8);
    z.next_out = reinterpret_cast<unsigned char *>(dst);
    z.avail_out = (unsigned)isize;
    const int rc = inflate(&z, Z_FINISH);
    const bool ok = rc == Z_STREAM_END && z.avail_out == 0;
    inflateEnd(&z);
    const unsigned long want_crc = (unsigned long)h[bsize - 8] | ((unsigned long)h[bsize - 7] << 8) |
                                   ((unsigned long)h[bsize - 6] << 16) | ((unsigned long)h[bsize - 5] << 24);
    if (!ok || crc32(crc32(0L, Z_NULL, 0), reinterpret_cast<const unsigned char *>(dst), (unsigned)isize) != want_crc)
      throw std::runtime_error("BGZF: corrupt member");
  }
  FILE *f_;
  std::vector<unsigned char> cbuf_;
  size_t cpos_ = 0, cend_ = 0;
  bool eof_ = false;
  std::vector<char> spill_;
  size_t spill_pos_ = 0;
};

// Block-wise reader: whole lines of a plain or gz file, many at a time, as views into one buffer (no per-line
// allocation; the VCF decode that follows runs on the views in parallel).
class BlockLineReader {
 public:
  struct View {
    const char *b, *e;
  };
  explicit BlockLineReader(const std::string &path) {
    if (!general_decode_only() && BgzfSource::is_bgzf(path)) {
      bgzf_.reset(new BgzfSource(path));
      return;
    }
    fp_ = gzopen(path.c_str(), "r");
    if (!fp_) throw std::runtime_error("cannot open " + path);
    gzbuffer(fp_, 1 << 20);
  }
  ~BlockLineReader() {
    if (fp_) gzclose(fp_);
  }
  BlockLineReader(const BlockLineReader &) = delete;
  BlockLineReader &operator=(const BlockLineReader &) = delete;
  // true when the file is not compressed (its size then bounds what is left to read)
  bool plain() { return fp_ && gzdirect(fp_) != 0; }

  // one line (header parsing); false at end of file
  bool next(std::string &line) {
    while (true) {
      const char *nl = pos_ < buf_.size() ? (const char *)memchr(buf_.data() + pos_, '\n', buf_.size() - pos_) : nullptr;
      if (nl || (eof_ && pos_ < buf_.size())) {
        const char *b = buf_.data() + pos_, *e = nl ? nl : buf_.data() + buf_.size();
        pos_ = nl ? (size_t)(nl - buf_.data()) + 1 : buf_.size();
        if (e > b && e[-1] == '\r') --e;
        line.assign(b, e);
        return true;
      }
      if (eof_) return false;
      fill(1 << 20);
    }
  }
  // whole lines, ~target bytes of them (at most max_lines; empty ones dropped unless keep_empty), read straight into
  // `store` (which keeps the views alive) -- one copy from the file, none per line; false when nothing is left
  bool next_block(TextBuf &store, std::vector<View> &lines, size_t max_lines, size_t target,
                  bool keep_empty = false) {
    lines.clear();
    // what next() left in its own buffer (header parsing) goes first
    store.assign(buf_.begin() + (long)pos_, buf_.end());
    buf_.clear();
    pos_ = 0;
    while (true) {
      while (!eof_ && store.size() < target) {
        const size_t old = store.size(), want = target - old + (1 << 16);
        store.resize(old + want);
        const size_t got = read_some(store.data() + old, want);
        store.resize(old + got);
        if (got < want) eof_ = true;
      }
      if (eof_ || memchr(store.data(), '\n', store.size())) break;
      target *= 2;  // one line longer than the target: keep reading
    }
    // cut after the last complete line; the rest waits in buf_ for the next call
    size_t end = store.size();
    if (!eof_) {
      while (end > 0 && store[end - 1] != '\n') --end;
    }
    const char *p = store.data(), *stop = store.data() + end;
    while (p < stop && lines.size() < max_lines) {
      const char *nl = (const char *)memchr(p, '\n', (size_t)(stop - p));
      const char *e = nl ? nl : stop;
      const char *next = nl ? nl + 1 : stop;
      if (e > p && e[-1] == '\r') --e;
      if (e > p || keep_empty) lines.push_back(View{p, e});
      p = next;
    }
    buf_.assign(p, (const char *)store.data() + store.size());  // unconsumed lines + the partial last one
    return !lines.empty() || !buf_.empty() || !eof_;
  }

 private:
  void fill(size_t want) {
    size_t old = buf_.size();
    buf_.resize(old + want);
    const size_t got = read_some(buf_.data() + old, want);
    buf_.resize(old + got);
    if (got < want) eof_ = true;
  }
  size_t read_some(char *dst, size_t want) {
    if (bgzf_) return bgzf_->read(dst, want);
    const int got = gzread(fp_, dst, (unsigned)want);
    if (got < 0) throw std::runtime_error("read error");
    return (size_t)got;
  }
  gzFile fp_ = nullptr;
  std::unique_ptr<BgzfSource> bgzf_;
  TextBuf buf_;
  size_t pos_ = 0;
  bool eof_ = false;
};

namespace detail {
// dst[i] = toupper(src[i]) (C locale) for i < n; returns whether any src[i] is white space (isspace, C locale)
inline bool upper_copy(char *dst, const char *src, size_t n) {
  size_t i = 0;
  bool space = false;
#if defined(__SSE2__)
  __m128i any = _mm_setzero_si128();
  const __m128i a_m1 = _mm_set1_epi8('a' - 1), z_p1 = _mm_set1_epi8('z' + 1), bit = _mm_set1_epi8(0x20),
                sp = _mm_set1_epi8(' '), t_m1 = _mm_set1_epi8(8), r_p1 = _mm_set1_epi8(14);
  for (; i + 16 <= n; i += 16) {
    const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(src + i));
    // (signed compares: bytes >= 0x80 are negative and fall outside both ranges, as they should)
    const __m128i lower = _mm_and_si128(_mm_cmpgt_epi8(c, a_m1), _mm_cmpgt_epi8(z_p1, c));
    const __m128i ws = _mm_or_si128(_mm_cmpeq_epi8(c, sp), _mm_and_si128(_mm_cmpgt_epi8(c, t_m1), _mm_cmpgt_epi8(r_p1, c)));
    any = _mm_or_si128(any, ws);
    _mm_storeu_si128(reinterpret_cast<__m128i *>(dst + i), _mm_sub_epi8(c, _mm_and_si128(lower, bit)));
  }
  space = _mm_movemask_epi8(any) != 0;
#endif
  for (; i < n; ++i) {
    const unsigned char c = (unsigned char)src[i];
    space |= (c == ' ') | ((unsigned)(c - 9u) < 5u);
    dst[i] = (char)((unsigned)(c - 'a') < 26u ? c - 32 : c);
  }
  return space;
}
}  // namespace detail

// whole reference, upper-cased, name = first word of the header line, optional "chr" strip (main.cpp:283-295).
// FASTA and FASTQ-style records are both accepted, like kseq does.
inline std::map<std::string, std::string> read_fasta(const std::string &path, bool strip_chr) {
  std::map<std::string, std::string> refs;
  BlockLineReader in(path);
  TextBuf store;
  std::vector<BlockLineReader::View> lines;
  std::string *cur = nullptr;
  bool in_qual = false;
  size_t qual_left = 0;
  size_t left = 0;  // bytes of an uncompressed file not yet seen (0: unknown)
  {
    struct stat st;
    if (in.plain() && stat(path.c_str(), &st) == 0) left = (size_t)st.st_size;
  }
  // lines are views into 16 MB blocks of the file: one copy from the file, one into the sequence
  while (in.next_block(store, lines, (size_t)1 << 22, (size_t)16 << 20, true)) {
    for (const BlockLineReader::View &ln : lines) {
      const size_t n = (size_t)(ln.e - ln.b);
      left = left > n + 1 ? left - n - 1 : 0;
      if (in_qual) {  // FASTQ quality lines: as many symbols as the sequence had
        qual_left = n >= qual_left ? 0 : qual_left - n;
        if (qual_left == 0) in_qual = false;
        continue;
      }
      if (n && (ln.b[0] == '>' || ln.b[0] == '@')) {
        const char *e = ln.b + 1;
        while (e < ln.e && *e != ' ' && *e != '\t') ++e;
        std::string name(ln.b + 1, e);
        if (strip_chr && name.compare(0, 3, "chr") == 0) name = name.substr(3);
        cur = &refs[name];
        cur->clear();
      } else if (n && ln.b[0] == '+' && cur) {
        in_qual = !cur->empty();
        qual_left = cur->size();
      } else if (cur && n) {  // sequence text: upper-cased, white space dropped (rare: noticed on the way, removed afterwards)
        const size_t old_size = cur->size();
        // growing a sequence copies it and touches fresh pages (several microseconds per page fault in a container):
        // an uncompressed file says how much can still come, so a contig is usually allocated once
        if (cur->capacity() < old_size + n)
          cur->reserve(std::max({old_size + n, 2 * cur->capacity(), std::min<size_t>(left, (size_t)1 << 29)}));
        cur->resize(old_size + n);
        char *q = &(*cur)[old_size];
        const bool space = detail::upper_copy(q, ln.b, n);
        if (space) {
          size_t w = 0;
          for (size_t i = 0; i < n; ++i)
            if (!isspace((unsigned char)q[i])) q[w++] = q[i];
          cur->resize(old_size + w);
        }
      }
    }
    if (lines.empty() && store.empty()) break;
  }
  return refs;
}

struct HeaderLine {
  std::string key, id, text;
};

class VcfHeader {
 public:
  std::vector<HeaderLine> lines;
  std::vector<std::string> samples;  // as in the file
  std::vector<int> keep;             // kept samples, header order
  std::vector<int32_t> kept_of_col;  // sample column -> its index in `keep`, -1 if dropped (filled by set_samples)

  static bool parse(const std::string &text, HeaderLine &h) {
    if (text.size() < 3 || text[0] != '#' || text[1] != '#') return false;
    size_t eq = text.find('=');
    if (eq == std::string::npos) return false;
    h.key = text.substr(2, eq - 2);
    h.text = text;
    h.id.clear();
    if (eq + 1 < text.size() && text[eq + 1] == '<') {
      size_t p = text.find("ID=", eq);
      if (p != std::string::npos) {
        size_t e = text.find_first_of(",>", p);
        h.id = text.substr(p + 3, e == std::string::npos ? std::string::npos : e - p - 3);
      }
    }
    return true;
  }
  void append(const std::string &text) {
    HeaderLine h;
    if (!parse(text, h)) return;
    for (const auto &o : lines) {
      if (o.key != h.key) continue;
      if (!h.id.empty() || !o.id.empty()) {
        if (o.id == h.id) return;
      } else if (o.text == h.text || h.key == "fileformat") {
        return;
      }
    }
    if (h.key == "fileformat")
      lines.insert(lines.begin(), h);
    else
      lines.push_back(h);
  }
  bool has_info(const std::string &id) const {
    for (const auto &l : lines)
      if (l.key == "INFO" && l.id == id) return true;
    return false;
  }
  // bcf_hdr_set_samples: "-" = all, otherwise a file with one name per line.
  // Returns 0, or (index of the first listed name that is absent) + 1, or -1 if the file cannot be read.
  int set_samples(const std::string &spec) {
    keep.clear();
    if (spec == "-") {
      for (size_t i = 0; i < samples.size(); ++i) keep.push_back((int)i);
      index_kept();
      return 0;
    }
    std::vector<std::string> names;
    try {
      LineReader in(spec);
      std::string l;
      while (in.next(l)) {
        size_t e = l.find_first_of(" \t");
        if (e != std::string::npos) l = l.substr(0, e);
        if (!l.empty()) names.push_back(l);
      }
    } catch (const std::exception &) {
      return -1;
    }
    std::vector<char> want(samples.size(), 0);
    int ret = 0;
    for (size_t i = 0; i < names.size(); ++i) {
      bool found = false;
      for (size_t j = 0; j < samples.size(); ++j)
        if (samples[j] == names[i]) {
          want[j] = 1;
          found = true;
        }
      if (!found && ret == 0) ret = (int)i + 1;
    }
    for (size_t j = 0; j < want.size(); ++j)
      if (want[j]) keep.push_back((int)j);
    index_kept();
    return ret;
  }
  void index_kept() {
    kept_of_col.assign(samples.size(), -1);
    for (size_t i = 0; i < keep.size(); ++i) kept_of_col[(size_t)keep[i]] = (int32_t)i;
  }
  // print_cleaned_header (main.cpp:190-219): GT/GQ (+COVS/GTS) appended if new, all samples replaced by DONOR
  std::string cleaned(bool verbose) const {
    VcfHeader h = *this;
    h.append("##FORMAT=<ID=GT,Number=1,Type=String,Description=\"Genotype\">");
    h.append("##FORMAT=<ID=GQ,Number=1,Type=Integer,Description=\"Genotype Quality\">");
    if (verbose) {
      h.append("##INFO=<ID=COVS,Number=R,Type=Integer,Description=\"Allele coverages\">");
      h.append("##INFO=<ID=GTS,Number=.,Type=String,Description=\"Genotypes Likelihood\">");
    }
    std::string out;
    for (const auto &l : h.lines) out += l.text + "\n";
    out += "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tDONOR\n";
    return out;
  }
};

// Opens a VCF (plain or gz), reads the header; data lines are then pulled in blocks with next_lines().
class VcfReader {
 public:
  VcfHeader header;

  explicit VcfReader(const std::string &path) : in_(path) {
    header.append("##FILTER=<ID=PASS,Description=\"All filters passed\">");
    std::string line;
    while (in_.next(line)) {
      if (line.size() >= 2 && line[0] == '#' && line[1] == '#') {
        header.append(line);
        continue;
      }
      if (!line.empty() && line[0] == '#') {
        size_t col = 0, p = 0;
        while (true) {
          size_t t = line.find('\t', p);
          std::string c = line.substr(p, t == std::string::npos ? std::string::npos : t - p);
          if (col >= 9 && !c.empty()) header.samples.push_back(c);
          ++col;
          if (t == std::string::npos) break;
          p = t + 1;
        }
        for (size_t i = 0; i < header.samples.size(); ++i) header.keep.push_back((int)i);
        return;
      }
      pending_ = line;  // a data line before any #CHROM line: headerless VCF
      has_pending_ = true;
      return;
    }
  }

  // the next data lines (views into `store`); false at the end of the file
  bool next_lines(TextBuf &store, std::vector<BlockLineReader::View> &lines, size_t max_lines, size_t target) {
    bool more = in_.next_block(store, lines, max_lines, target);
    if (has_pending_) {
      has_pending_ = false;
      pending_store_.assign(pending_.begin(), pending_.end());
      lines.insert(lines.begin(), BlockLineReader::View{pending_store_.data(), pending_store_.data() + pending_store_.size()});
      return true;
    }
    return more;
  }

 private:
  BlockLineReader in_;
  std::string pending_;
  std::vector<char> pending_store_;
  bool has_pending_ = false;
};

namespace detail {
struct Field {
  const char *b, *e;
  size_t size() const { return (size_t)(e - b); }
  std::string str() const { return std::string(b, e); }
  bool is(const char *s) const { return size() == strlen(s) && memcmp(b, s, size()) == 0; }
};
inline std::string upper(const char *b, const char *e) {
  std::string s(b, e);
  for (auto &ch : s) ch = (char)toupper((unsigned char)ch);
  return s;
}
inline float missing_float() {  // bcf_float_missing: a NaN
  return std::nanf("");
}
// strtod for the plain decimals VCF INFO fields hold ("0.000312", "1.5e-05", "1"): at most 19 significant digits that fit
// 2^53 and a decimal exponent within +-22 -- both the digits and the power of ten are then exact doubles and ONE IEEE
// multiplication or division gives the correctly rounded value, i.e. what strtod returns (Clinger's fast path).
// Anything else (more digits, larger exponents, inf/nan, hex, trailing text) is left to strtod itself.
inline bool fast_decimal(const char *b, const char *e, double *out) {
  static const double P10[23] = {1e0,  1e1,  1e2,  1e3,  1e4,  1e5,  1e6,  1e7,  1e8,  1e9,  1e10, 1e11,
                                 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22};
  const char *p = b;
  bool neg = false;
  if (p < e && (*p == '-' || *p == '+')) neg = *p++ == '-';
  uint64_t m = 0;
  int digits = 0, exp10 = 0;
  bool any = false;
  while (p < e && *p >= '0' && *p <= '9') {
    if (m || *p != '0') {
      if (++digits > 19) return false;
      m = m * 10 + (uint64_t)(*p - '0');
    }
    any = true;
    ++p;
  }
  if (p < e && *p == '.') {
    ++p;
    while (p < e && *p >= '0' && *p <= '9') {
      if (m || *p != '0') {
        if (++digits > 19) return false;
        m = m * 10 + (uint64_t)(*p - '0');
      }
      --exp10;
      any = true;
      ++p;
    }
  }
  if (!any) return false;
  if (p < e && (*p == 'e' || *p == 'E')) {
    ++p;
    bool eneg = false;
    if (p < e && (*p == '-' || *p == '+')) eneg = *p++ == '-';
    if (p >= e || *p < '0' || *p > '9') return false;
    int x = 0;
    while (p < e && *p >= '0' && *p <= '9') {
      x = x * 10 + (*p++ - '0');
      if (x > 9999) return false;
    }
    exp10 += eneg ? -x : x;
  }
  if (p != e || m > (1ull << 53) || exp10 < -22 || exp10 > 22) return false;
  double v = (double)m;
  v = exp10 < 0 ? v / P10[-exp10] : v * P10[exp10];
  *out = neg ? -v : v;
  return true;
}
// one float token the way htslib reads it: strtod, narrowed; "." or nothing = missing
inline float float_token(const char *q, const char *t) {
  double d;
  if (t == q || (t - q == 1 && *q == '.')) return missing_float();
  if (fast_decimal(q, t, &d)) return (float)d;
  return (float)strtod(std::string(q, t).c_str(), nullptr);
}

// the float values of INFO key `key`: returns how many there are (up to `cap` of them are stored), or -1 when the key
// is absent
inline int info_floats(const Field &info, const std::string &key, float *out, int cap) {
  const char *p = info.b;
  while (p < info.e) {
    const char *e = (const char *)memchr(p, ';', (size_t)(info.e - p));
    if (!e) e = info.e;
    if ((size_t)(e - p) > key.size() && memcmp(p, key.data(), key.size()) == 0 && p[key.size()] == '=') {
      const char *q = p + key.size() + 1;
      int n = 0;
      while (q <= e) {
        const char *t = (const char *)memchr(q, ',', (size_t)(e - q));
        if (!t) t = e;
        const float f = float_token(q, t);
        if (n < cap) out[n] = f;
        ++n;
        q = t + 1;
      }
      return n;
    }
    p = e + 1;
  }
  return -1;
}

// ---- extract_genotypes for the layout panels come in: FORMAT is "GT" alone and every column has the same width --
// "a|b" / "a/b" with one-symbol alleles (3 bytes + tab) or one symbol alone (haploid panels, 1 byte + tab).
// Columns then sit at a fixed stride, the run of the mill ("0|0", "0/0", "0") is recognised 16 bytes at a time, and only
// the columns that differ are decoded -- those of the kept samples (-s), that is: `kept_of_col` maps a column to its
// place among the `n_keep` kept ones.  The result is the sparse genotype list parse_record() would build (same
// decisions, variant.hpp:158-211, including the one-allele rows whose second read lands on the NEXT kept sample's
// first entry).  Returns false -- nothing written -- for any other layout: the caller then takes the general path.
inline int gt_symbol(char c) {  // allele index of a one-symbol GT entry; '.' (missing) counts as the reference allele
  if (c >= '0' && c <= '9') return c - '0';
  return c == '.' ? 0 : -1;
}
inline bool fast_gt_columns(const char *s, const char *end, size_t n_cols, const int32_t *kept_of_col, const int *keep,
                            size_t n_keep, Variant &v) {
  if (n_cols == 0 || n_keep == 0 || !s) return false;
  const size_t len = (size_t)(end - s);
  static thread_local std::vector<uint32_t> exc_tl;  // columns that are not the run-of-the-mill one
  std::vector<uint32_t> &exc = exc_tl;
  exc.clear();
  v.gts.clear();
  size_t ref_phased = 0, ref_unphased = 0;
  if (len == 4 * n_cols - 1) {  // ---- "a|b" columns ----
    if (s[1] != '|' && s[1] != '/') return false;
    const char sep = s[1];
    const int guess = sep == '|';  // phasing of the reference-reference columns, to be confirmed by the counts
    const char def4[4] = {'0', sep, '0', '\t'};
    uint32_t def;
    memcpy(&def, def4, 4);
    size_t i = 0;
    const size_t whole = n_cols - 1;  // (the last column has no tab behind it)
#if defined(__SSE2__)
    const __m128i d16 = _mm_set1_epi32((int)def);
    for (; i + 4 <= whole; i += 4) {
      const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + 4 * i));
      const int eq = _mm_movemask_ps(_mm_castsi128_ps(_mm_cmpeq_epi32(c, d16)));
      if (eq == 0xF) continue;
      for (int j = 0; j < 4; ++j)
        if (!((eq >> j) & 1)) exc.push_back((uint32_t)(i + (size_t)j));
    }
#endif
    for (; i < whole; ++i) {
      uint32_t w;
      memcpy(&w, s + 4 * i, 4);
      if (w != def) exc.push_back((uint32_t)i);
    }
    exc.push_back((uint32_t)(n_cols - 1));
    size_t kept_exc = 0;
    for (uint32_t e : exc) {
      const char *q = s + 4 * (size_t)e;
      const int a1 = gt_symbol(q[0]), a2 = gt_symbol(q[2]);
      if (a1 < 0 || a2 < 0 || (q[1] != '|' && q[1] != '/') || (e + 1 < n_cols && q[3] != '\t')) return false;
      const int32_t ki = kept_of_col[e];
      if (ki < 0) continue;  // (a dropped sample: its column only had to be well-formed)
      ++kept_exc;
      const uint16_t h1 = v.text_id_of(a1), h2 = v.text_id_of(a2);
      const uint8_t ph = q[1] == '|';
      if ((h1 | h2) == 0) {
        (ph ? ref_phased : ref_unphased)++;
        if (ph == guess) continue;
      }
      v.gts.push_back(GtEntry{(uint32_t)ki, h1, h2, ph});
    }
    (guess ? ref_phased : ref_unphased) += n_keep - kept_exc;
    if ((ref_phased >= ref_unphased ? 1 : 0) != guess) return false;  // (mixed files: the general path sorts it out)
    v.default_phased = (uint8_t)guess;
  } else if (len == 2 * n_cols - 1) {  // ---- one-symbol columns: kept sample i reads {own symbol, the NEXT kept
    //                                      sample's symbol}, unphased; the last one {own, own}, phased (parse_record) ----
    const char def2[2] = {'0', '\t'};
    uint16_t def;
    memcpy(&def, def2, 2);
    size_t i = 0;
    const size_t whole = n_cols - 1;
#if defined(__SSE2__)
    const __m128i d16 = _mm_set1_epi16((short)def);
    for (; i + 8 <= whole; i += 8) {
      const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + 2 * i));
      const int eq = _mm_movemask_epi8(_mm_cmpeq_epi16(c, d16));
      if (eq == 0xFFFF) continue;
      for (int j = 0; j < 8; ++j)
        if (((eq >> (2 * j)) & 3) != 3) exc.push_back((uint32_t)(i + (size_t)j));
    }
#endif
    for (; i < whole; ++i) {
      uint16_t w;
      memcpy(&w, s + 2 * i, 2);
      if (w != def) exc.push_back((uint32_t)i);
    }
    exc.push_back((uint32_t)(n_cols - 1));
    // a kept column that differs makes its own sample and the kept one before it differ; the last kept sample is
    // always looked at
    size_t n_touched = 0;
    int64_t last_done = -1;
    auto visit = [&](int64_t t) {  // kept index t, ascending over the calls
      if (t < 0 || t <= last_done) return true;
      last_done = t;
      ++n_touched;
      const int a1 = gt_symbol(s[2 * (size_t)keep[t]]);
      const bool last = (size_t)t + 1 == n_keep;
      const int a2 = last ? a1 : gt_symbol(s[2 * (size_t)keep[t + 1]]);
      if (a1 < 0 || a2 < 0) return false;
      const uint16_t h1 = v.text_id_of(a1), h2 = v.text_id_of(a2);
      const uint8_t ph = last ? 1 : 0;
      if ((h1 | h2) == 0) {
        (ph ? ref_phased : ref_unphased)++;
        if (!ph) return true;
      }
      v.gts.push_back(GtEntry{(uint32_t)t, h1, h2, ph});
      return true;
    };
    for (uint32_t e : exc) {
      const char *q = s + 2 * (size_t)e;
      if (gt_symbol(q[0]) < 0 || (e + 1 < n_cols && q[1] != '\t')) return false;
      const int32_t ki = kept_of_col[e];
      if (ki < 0) continue;
      if (!visit((int64_t)ki - 1) || !visit((int64_t)ki)) return false;
    }
    if (!visit((int64_t)n_keep - 1)) return false;
    ref_unphased += n_keep - n_touched;
    if (ref_phased >= ref_unphased) return false;  // (a panel of one or two samples: the general path)
    v.default_phased = 0;
  } else {
    return false;
  }
  v.n_samples_ = (uint32_t)n_keep;
  return true;
}
}  // namespace detail

// Variant(hdr, rec, freq_key, uniform), variant.hpp:66-103, from one VCF data line.
inline Variant parse_record(const char *line_begin, const char *line_end, const VcfHeader &header,
                            const std::string &freq_key, bool uniform, bool freq_key_declared) {
  using detail::Field;
  Field c[9];
  int nf = 0;
  const char *p = line_begin, *end = line_end;
  const char *samples_begin = nullptr;
  while (nf < 9) {
    const char *t = (const char *)memchr(p, '\t', (size_t)(end - p));
    c[nf++] = Field{p, t ? t : end};
    if (!t) break;
    p = t + 1;
    if (nf == 9) samples_begin = p;
  }
  if (nf < 8)
    throw std::runtime_error("malformed VCF record: " + std::string(line_begin, std::min<size_t>(60, (size_t)(line_end - line_begin))));
  Variant v;
  v.seq_name = c[0].str();
  {  // POS: decimal digits (strtoll semantics: optional sign, stops at the first non-digit)
    const char *q = c[1].b;
    bool neg = false;
    if (q < c[1].e && (*q == '-' || *q == '+')) neg = *q++ == '-';
    long long pos = 0;
    while (q < c[1].e && *q >= '0' && *q <= '9') pos = pos * 10 + (*q++ - '0');
    v.ref_pos = (int)((neg ? -pos : pos) - 1);
  }
  v.idx = c[2].str();
  v.ref_sub = detail::upper(c[3].b, c[3].e);
  if (!c[4].is(".")) {
    const char *a = c[4].b;
    while (a <= c[4].e) {
      const char *t = (const char *)memchr(a, ',', (size_t)(c[4].e - a));
      if (!t) t = c[4].e;
      if (!(t > a && a[0] == '<')) v.alts.push_back(detail::upper(a, t));  // symbolic alleles dropped (variant.hpp:82)
      a = t + 1;
    }
  }
  v.quality = c[5].is(".") ? detail::missing_float() : (c[5].b == c[5].e ? 0.0f : detail::float_token(c[5].b, c[5].e));
  v.set_sizes();
  if (!v.has_alts) return v;
  // ---- extract_frequencies (variant.hpp:126-156) ----
  if (!uniform) {
    const size_t na = v.alts.size();
    v.frequencies.assign(na + 1, 0.0f);  // (values the record does not list stay 0)
    const int n_af = freq_key_declared ? detail::info_floats(c[7], freq_key, v.frequencies.data() + 1, (int)na) : -1;
    if (n_af < 0)
      throw std::runtime_error("INFO key " + freq_key + " missing at " + v.seq_name + ":" + std::to_string(v.ref_pos + 1) +
                               " (the reference dereferences NULL here; use -u or -f)");
    double sum = 0.0;
    for (float f : v.frequencies) sum += f;
    v.frequencies[0] = (float)(1.0 - sum);
    if (v.frequencies[0] < 0) v.frequencies[0] = 0.0f;
  } else {
    float u = (float)(1.0 / (double)(v.alts.size() + 1));
    v.frequencies.assign(v.alts.size() + 1, u);
  }
  if (v.frequencies[0] == 1.0) v.is_present = false;
  if (!v.is_present) return v;
  // ---- extract_genotypes (variant.hpp:158-211) ----
  int gt_field = -1;
  if (nf > 8) {
    int idx = 0;
    const char *f = c[8].b;
    while (f <= c[8].e) {
      const char *t = (const char *)memchr(f, ':', (size_t)(c[8].e - f));
      if (!t) t = c[8].e;
      if (t - f == 2 && f[0] == 'G' && f[1] == 'T') {
        gt_field = idx;
        break;
      }
      ++idx;
      f = t + 1;
    }
  }
  if (gt_field < 0 || header.keep.empty()) {
    v.has_alts = false;  // "The record doesn't contain GT information" (variant.hpp:170-175)
    return v;
  }
  // raw codes per kept sample, htslib style: ((allele + 1) << 1) | phased; `first`/`second`/ploidy per sample
  const size_t ns = header.keep.size();
  if (count_rows()) sample_rows().fetch_add(1, std::memory_order_relaxed);
  if (gt_field == 0 && c[8].size() == 2 && header.kept_of_col.size() == header.samples.size() && !general_decode_only() &&
      detail::fast_gt_columns(samples_begin, end, header.samples.size(), header.kept_of_col.data(), header.keep.data(), ns, v)) {
    if (count_rows()) fast_gt_rows().fetch_add(1, std::memory_order_relaxed);
    return v;
  }
  v.gts.clear();
  static thread_local std::vector<int32_t> g0_tl, g1_tl;  // scratch, one set per decoding thread
  static thread_local std::vector<uint8_t> ploidy_tl;
  g0_tl.assign(ns, 0);
  g1_tl.assign(ns, 0);
  ploidy_tl.assign(ns, 1);
  int32_t *const g0 = g0_tl.data(), *const g1 = g1_tl.data();
  uint8_t *const ploidy = ploidy_tl.data();
  const int *const keep = header.keep.data();
  size_t max_ploidy = 1;
  {
    size_t ki = 0;  // next kept sample to fill
    int col = 0;
    const char *s = samples_begin;
    while (s && s <= end && ki < ns) {
      // (sample columns are a few bytes long: plain loops beat memchr here)
      if (gt_field == 0 && end - s >= 4 && (s[3] == '\t' || s[3] == ':') && s[0] >= '0' && s[0] <= '9' && s[2] >= '0' &&
          s[2] <= '9' && (s[1] == '|' || s[1] == '/')) {  // "a|b" / "a/b" with one-digit alleles, GT first
        if (col == keep[ki]) {
          g0[ki] = ((s[0] - '0') + 1) << 1;
          g1[ki] = (((s[2] - '0') + 1) << 1) | (s[1] == '|');
          ploidy[ki] = 2;
          max_ploidy = std::max<size_t>(max_ploidy, 2);
          ++ki;
        }
        s += 3;
        while (s < end && *s != '\t') ++s;
        ++col;
        ++s;
        continue;
      }
      const char *t = s;
      while (t < end && *t != '\t') ++t;
      if (col == keep[ki]) {
        const char *q = s;
        for (int f = 0; f < gt_field && q; ++f) {
          q = (const char *)memchr(q, ':', (size_t)(t - q));
          if (q) ++q;
        }
        size_t n = 0;
        if (q) {
          const char *e = (const char *)memchr(q, ':', (size_t)(t - q));
          if (!e) e = t;
          int ph = 0;
          while (q < e) {
            int32_t code;
            if (*q == '.') {
              code = 0 | ph;
              ++q;
            } else {
              int a = 0;
              while (q < e && *q >= '0' && *q <= '9') a = a * 10 + (*q++ - '0');
              code = ((a + 1) << 1) | ph;
            }
            if (n == 0) g0[ki] = code;
            if (n == 1) g1[ki] = code;
            ++n;
            if (q < e) {
              ph = *q == '|';
              ++q;
            }
          }
        }
        if (n == 0) n = 1;  // an empty field counts as one missing allele
        ploidy[ki] = (uint8_t)std::min<size_t>(n, 255);
        max_ploidy = std::max(max_ploidy, n);
        ++ki;
      }
      ++col;
      s = t + 1;
    }
  }
  const int32_t VECTOR_END = INT32_MIN + 1;
  // genotypes as allele text ids, kept sparse (signatures.hpp): first the phasing flag most all-reference samples
  // carry, then one entry per sample that differs from {0, 0, that flag}
  static thread_local std::vector<uint16_t> h1_tl, h2_tl;
  static thread_local std::vector<uint8_t> ph_tl;
  h1_tl.resize(ns);
  h2_tl.resize(ns);
  ph_tl.resize(ns);
  // (plain pointers: every use of a function-local thread_local goes through its TLS wrapper)
  uint16_t *const h1s = h1_tl.data(), *const h2s = h2_tl.data();
  uint8_t *const phs = ph_tl.data();
  size_t ref_phased = 0, ref_unphased = 0;
  for (size_t i = 0; i < ns; ++i) {
    // the reference reads curr_gt[0] and curr_gt[1] of a row of max_ploidy entries; with ploidy 1 everywhere the
    // second read lands on the NEXT sample's first entry (variant.hpp:184) -- reproduced; the last sample sees
    // the end marker
    int32_t a = g0[i], b;
    if (max_ploidy >= 2)
      b = ploidy[i] >= 2 ? g1[i] : VECTOR_END;
    else
      b = i + 1 < ns ? g0[i + 1] : VECTOR_END;
    int a1, a2;
    bool ph;
    if (b == VECTOR_END) {
      a1 = a2 = (a >> 1) - 1;
      ph = true;
    } else {
      a1 = (a >> 1) - 1;
      a2 = (b >> 1) - 1;
      ph = (b & 1) != 0;
    }
    if (a1 < 0) a1 = 0;
    if (a2 < 0) a2 = 0;
    h1s[i] = v.text_id_of(std::min(a1, 65535));
    h2s[i] = v.text_id_of(std::min(a2, 65535));
    phs[i] = ph ? 1 : 0;
    if ((h1s[i] | h2s[i]) == 0) (ph ? ref_phased : ref_unphased)++;
  }
  v.n_samples_ = (uint32_t)ns;
  v.default_phased = ref_phased >= ref_unphased ? 1 : 0;
  v.gts.reserve(ns - std::max(ref_phased, ref_unphased));
  for (size_t i = 0; i < ns; ++i)
    if ((h1s[i] | h2s[i]) != 0 || phs[i] != v.default_phased)
      v.gts.push_back(GtEntry{(uint32_t)i, h1s[i], h2s[i], phs[i]});
  return v;
}

}  // namespace mh
