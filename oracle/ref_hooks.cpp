// TEST INFRASTRUCTURE ONLY. extern "C" hooks over the reference's OWN classes,
// compiled from the headers where they lie under /root/reference (never copied
// into this repo) against the stand-in library headers in oracle/shim/.
// Output: oracle/_ref/libmalva_ref.so (git-ignored).  Tests use it to pin the
// C restatement in oracle/malva_oracle.c and, through that, the CUDA path.
//
// Hooks map 1:1 onto reference entry points:
//   ref_xxh3            -> XXH3_64bits                      xxhash.h:5037
//   ref_bf_*            -> BF::{add_key,test_key,switch_mode,increment,get_count}
//                                                         bloom_filter.hpp:81-125
//   ref_kmap_*          -> KMAP::{add_key,test_key,increment,get_count}  kmap.hpp:99-131
//   ref_scan_kmer       -> loop body of call_main            main.cpp:490-499
//   ref_reference_pass  -> loop of index_main                main.cpp:383-401
//   ref_genotype        -> VB::genotype + VB::output_variants var_block.hpp:224-396
//   ref_extract_kmers   -> VB::extract_kmers                 var_block.hpp:95-219
#include <cmath>
#include <cstring>
#include <sstream>
#include <string>
#include <vector>

#include "htslib/hts_log.h"
#include "htslib/vcf.h"
#include "kmc_file.h"

#include "bloom_filter.hpp"
#include "kmap.hpp"
#include "var_block.hpp"

extern "C" {

uint64_t ref_xxh3(const char *p, size_t n) { return XXH3_64bits(p, n); }

// ---- BF -------------------------------------------------------------------
void *ref_bf_new(uint64_t size_bits) { return new BF((size_t)size_bits); }
void ref_bf_free(void *b) { delete (BF *)b; }
void ref_bf_add_key(void *b, const char *kmer) { ((BF *)b)->add_key(kmer); }
int ref_bf_test_key(void *b, const char *kmer) { return ((BF *)b)->test_key(kmer) ? 1 : 0; }
void ref_bf_switch_mode(void *b) { ((BF *)b)->switch_mode(); }
int ref_bf_increment(void *b, const char *kmer, uint32_t c) { return ((BF *)b)->increment(kmer, c) ? 1 : 0; }
uint32_t ref_bf_get_count(void *b, const char *kmer) { return ((BF *)b)->get_count(kmer); }

// ---- KMAP -----------------------------------------------------------------
void *ref_kmap_new() { return new KMAP(); }
void ref_kmap_free(void *m) { delete (KMAP *)m; }
void ref_kmap_add_key(void *m, const char *kmer) { ((KMAP *)m)->add_key(kmer); }
int ref_kmap_test_key(void *m, const char *kmer) { return ((KMAP *)m)->test_key(kmer) ? 1 : 0; }
void ref_kmap_increment(void *m, const char *kmer, int c) { ((KMAP *)m)->increment(kmer, c); }
int ref_kmap_get_count(void *m, const char *kmer) { return ((KMAP *)m)->get_count(kmer); }
uint64_t ref_kmap_size(void *m) { return ((KMAP *)m)->kmers.size(); }

// ---- sample scan, one KMC record (main.cpp:490-499) -------------------------
void ref_scan_kmer(void *bf, void *context_bf, void *ref_bf, const char *context_in, uint32_t counter,
                   int k, int ref_k) {
  // stack arrays, as main.cpp:487-488 has them (char context[ref_k + 1]; char kmer[k + 1];)
  char context[130], kmer[130];
  memcpy(context, context_in, (size_t)ref_k);
  context[ref_k] = '\0';
  std::transform(context, context + ref_k, context, ::toupper);
  strncpy(kmer, context + ((ref_k - k) / 2), k);
  kmer[k] = '\0';
  ((KMAP *)ref_bf)->increment(kmer, counter);
  if (!((BF *)context_bf)->test_key(context)) {
    ((BF *)bf)->increment(kmer, counter);
  }
}

// ---- batch variants over packed k-mers (A=0 C=1 G=2 T=3, first base most significant), used by
// bench.py's CPU baseline: the same reference classes, fed like the KMC listing loop feeds them ----
static void unpack_kmer(uint64_t lo, uint64_t hi, int k, char *out) {
  static const char SYM[4] = {'A', 'C', 'G', 'T'};
  for (int j = 0; j < k; ++j) {
    int sh = 2 * (k - 1 - j);
    uint64_t code = sh >= 64 ? (hi >> (sh - 64)) : (lo >> sh);
    out[j] = SYM[code & 3];
  }
  out[k] = '\0';
}
void ref_add_packed(void *bf, void *ref_bf, const uint64_t *lohi, const uint8_t *is_ref, uint64_t n, int k) {
  char kmer[130];
  for (uint64_t i = 0; i < n; ++i) {  // add_kmers_to_bf, main.cpp:133-140
    unpack_kmer(lohi[2 * i], lohi[2 * i + 1], k, kmer);
    if (is_ref[i])
      ((KMAP *)ref_bf)->add_key(kmer);
    else
      ((BF *)bf)->add_key(kmer);
  }
}
void ref_scan_packed(void *bf, void *context_bf, void *ref_bf, const uint64_t *lohi, const uint32_t *counts,
                     uint64_t n, int k, int ref_k) {
  char context[130];
  for (uint64_t i = 0; i < n; ++i) {
    unpack_kmer(lohi[2 * i], lohi[2 * i + 1], ref_k, context);  // kmer_obj.to_string(context), main.cpp:490
    ref_scan_kmer(bf, context_bf, ref_bf, context, counts[i], k, ref_k);
  }
}

// BF::get_count / KMAP::get_count over packed k-mers (bench.py's exact check of the device counters)
void ref_get_counts_packed(void *bf, void *ref_bf, const uint64_t *lohi, const uint8_t *is_ref, uint64_t n, int k,
                           int32_t *out) {
  char kmer[130];
  for (uint64_t i = 0; i < n; ++i) {
    unpack_kmer(lohi[2 * i], lohi[2 * i + 1], k, kmer);
    out[i] = is_ref[i] ? (int32_t)((KMAP *)ref_bf)->get_count(kmer) : (int32_t)((BF *)bf)->get_count(kmer);
  }
}

// set_coverages + VB::genotype over a batch (main.cpp:151-184, 565-566; var_block.hpp:224-330): the CPU
// counterpart of mg_genotype on the reference's own classes.  CSR as in mg_packed_batch (u32 offsets, packed
// k-mers, ref allele = slot 0).  Returns a checksum of the best genotypes so that nothing is optimised away.
uint64_t ref_genotype_batch(void *bf_, void *ref_bf_, uint64_t n_variants, const uint32_t *var_allele_off,
                            const uint32_t *allele_sig_off, const uint32_t *sig_kmer_off, const uint64_t *lohi,
                            const float *freq, int k, float error_rate, int max_cov, int haploid, uint32_t *cov_out,
                            int32_t *best_out, int32_t *gq_out) {
  BF &bf = *(BF *)bf_;
  KMAP &ref_bf = *(KMAP *)ref_bf_;
  uint64_t sum = 0;
  char kmer[130];
  for (uint64_t v = 0; v < n_variants; ++v) {
    const uint32_t a0 = var_allele_off[v], a1 = var_allele_off[v + 1];
    Variant var;
    var.seq_name = "1";
    var.ref_pos = 0;
    var.idx = ".";
    var.ref_sub = "A";
    for (uint32_t i = a0 + 1; i < a1; ++i) var.alts.push_back("C");
    var.quality = 0;
    var.filter = "PASS";
    var.info = ".";
    var.coverages.assign(a1 - a0, 0);
    var.frequencies.assign(freq + a0, freq + a1);
    VB vb(k, error_rate);
    vb.add_variant(var);
    for (uint32_t a = a0; a < a1; ++a) {  // set_coverages, main.cpp:157-182
      uint allele_cov = 0;
      for (uint32_t s = allele_sig_off[a]; s < allele_sig_off[a + 1]; ++s) {
        uint curr_cov = 0;
        int n = 0;
        for (uint32_t q = sig_kmer_off[s]; q < sig_kmer_off[s + 1]; ++q) {
          unpack_kmer(lohi[2 * (uint64_t)q], lohi[2 * (uint64_t)q + 1] & 0x3FFFFFFFFFFFFFFFULL, k, kmer);
          uint w = a == a0 ? (uint)ref_bf.get_count(kmer) : (uint)bf.get_count(kmer);
          if (w > 0) {
            curr_cov = (curr_cov * n + w) / (n + 1);
            ++n;
          }
        }
        if (curr_cov > allele_cov) allele_cov = curr_cov;
      }
      vb.set_variant_coverage(0, (int)(a - a0), allele_cov);
      if (cov_out) cov_out[a] = allele_cov;
    }
    vb.genotype(max_cov, haploid != 0);
    Variant r = vb.get_variant(0);
    // arg-max of VB::output_variants (var_block.hpp:367-394)
    double total = 0.0;
    for (const auto &g : r.computed_gts) total += g.second;
    double best = 0.0;
    int bi = 0, i = 0;
    for (const auto &g : r.computed_gts) {
      double q = g.second / total;
      if (q > best) {
        best = q;
        bi = i;
      }
      ++i;
    }
    if (best_out) best_out[v] = bi;
    if (gq_out) gq_out[v] = (int)round(best * 100);
    sum += (uint64_t)bi + (uint64_t)r.computed_gts.size();
  }
  return sum;
}

// ---- reference rolling pass over one contig (main.cpp:385-400) ---------------
void ref_reference_pass(void *bf_, void *context_bf_, const char *seq, int k_, int ref_k_) {
  BF &bf = *(BF *)bf_;
  BF &context_bf = *(BF *)context_bf_;
  uint k = (uint)k_, ref_k = (uint)ref_k_;
  std::string reference(seq);
  std::string ref_ksub(reference, (ref_k - k) / 2, k);
  std::string context(reference, 0, ref_k);
  if (bf.test_key(ref_ksub.c_str())) context_bf.add_key(context.c_str());
  for (uint p = ref_k; p < reference.size(); ++p) {
    char c1 = reference[p];
    context.erase(0, 1);
    context += c1;
    char c2 = reference[p - (ref_k - k) / 2];
    ref_ksub.erase(0, 1);
    ref_ksub += c2;
    if (bf.test_key(ref_ksub.c_str())) context_bf.add_key(context.c_str());
  }
}

// ---- genotype one variant through VB::genotype + VB::output_variants ---------
// cov/freq have n_alleles entries.  Writes the probabilities (un-normalised, in
// emission order) to probs (capacity cap) and the printed VCF line (verbose) to
// line_out.  Returns the number of computed_gts entries.
int ref_genotype(const uint32_t *cov, const float *freq, int n_alleles, float error_rate, int max_cov,
                 int haploid, double *probs, int cap, char *line_out, int line_cap) {
  Variant v;
  v.seq_name = "1";
  v.ref_pos = 0;
  v.idx = ".";
  v.ref_sub = "A";
  for (int i = 1; i < n_alleles; ++i) v.alts.push_back("C");
  uint32_t q = 0x7F800001u;
  memcpy(&v.quality, &q, 4);
  v.filter = "PASS";
  v.info = ".";
  v.coverages.assign(cov, cov + n_alleles);
  v.frequencies.assign(freq, freq + n_alleles);
  VB vb(35, error_rate);
  vb.add_variant(v);
  vb.genotype(max_cov, haploid != 0);
  Variant r = vb.get_variant(0);
  int n = (int)r.computed_gts.size();
  for (int i = 0; i < n && i < cap; ++i) probs[i] = r.computed_gts[i].second;
  if (line_out && line_cap > 0) {
    std::ostringstream oss;
    std::streambuf *old = std::cout.rdbuf(oss.rdbuf());
    vb.output_variants(haploid != 0, true);
    std::cout.rdbuf(old);
    std::string s = oss.str();
    strncpy(line_out, s.c_str(), (size_t)line_cap - 1);
    line_out[line_cap - 1] = '\0';
  }
  return n;
}

// ---- signature enumeration of one var_block ---------------------------------
// Block description (text, one variant per line, tab separated):
//   ref_pos \t REF \t ALT1,ALT2 \t is_present(0/1) \t a|b a/b a|b ...   (one GT per sample)
// Output (text): one line per signature k-mer list:
//   variant_index \t allele_index \t kmer1,kmer2,...
// Lines are sorted so the unordered_set iteration order does not leak out.
int ref_extract_kmers(const char *block, const char *reference, int k, int haploid, char *out,
                      int out_cap) {
  VB vb(k, 0.001f);
  std::istringstream in(block);
  std::string line;
  while (std::getline(in, line)) {
    if (line.empty()) continue;
    std::vector<std::string> c;
    size_t s = 0;
    while (true) {
      size_t t = line.find('\t', s);
      c.push_back(line.substr(s, t == std::string::npos ? std::string::npos : t - s));
      if (t == std::string::npos) break;
      s = t + 1;
    }
    Variant v;
    v.seq_name = "1";
    v.ref_pos = atoi(c[0].c_str());
    v.idx = ".";
    v.ref_sub = c[1];
    v.ref_size = (int)v.ref_sub.size();
    {
      size_t p = 0;
      while (p <= c[2].size()) {
        size_t t = c[2].find(',', p);
        if (t == std::string::npos) t = c[2].size();
        if (t > p) v.alts.push_back(c[2].substr(p, t - p));
        p = t + 1;
      }
    }
    v.coverages.resize(v.alts.size() + 1, 0);
    v.set_sizes();
    v.is_present = c[3] == "1";
    if (c.size() > 4) {
      std::istringstream gs(c[4]);
      std::string g;
      while (gs >> g) {
        size_t sep = g.find_first_of("|/");
        Geno ge;
        bool ph;
        if (sep == std::string::npos) {
          ge = {atoi(g.c_str()), atoi(g.c_str())};
          ph = true;
        } else {
          ge = {atoi(g.substr(0, sep).c_str()), atoi(g.substr(sep + 1).c_str())};
          ph = g[sep] == '|';
        }
        v.genotypes.push_back(ge);
        v.phasing.push_back(ph);
      }
    }
    vb.add_variant(v);
  }
  VK_GROUP kmers = vb.extract_kmers(std::string(reference), haploid != 0);
  std::vector<std::string> lines;
  for (const auto &var : kmers)
    for (const auto &al : var.second)
      for (const auto &Ks : al.second) {
        std::string l = std::to_string(var.first) + "\t" + std::to_string(al.first) + "\t";
        for (size_t i = 0; i < Ks.size(); ++i) {
          if (i) l += ",";
          l += Ks[i];
        }
        lines.push_back(l);
      }
  std::sort(lines.begin(), lines.end());
  std::string res;
  for (auto &l : lines) res += l + "\n";
  if ((int)res.size() + 1 > out_cap) return -(int)res.size() - 1;
  memcpy(out, res.c_str(), res.size() + 1);
  return (int)res.size();
}

}  // extern "C"
