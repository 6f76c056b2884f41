/* TEST INFRASTRUCTURE ONLY -- CPU restatement of MALVA's genotyping hot path.
 *
 * This is the parity oracle for the CUDA path in malva_b200/csrc.  Only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
 * may load it; the product never routes through it.
 *
 * Pinned against (tests/test_oracle.py): the XXH3 known answers of SURVEY 8c,
 * python-xxhash, the reference's own classes via oracle/_ref/libmalva_ref.so,
 * and the golden VCF example/haploid.malva.vcf (through oracle/_ref).
 *
 * Every function cites the reference file:line it follows (paths relative to
 * the upstream repository root).
 */
#ifndef MALVA_ORACLE_H
#define MALVA_ORACLE_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* xxhash.h:5037-5040 (XXH3_64bits, seed 0, default secret), lengths 0..240 */
uint64_t mo_xxh3_64(const void *data, size_t len);

/* bloom_filter.hpp:58-65 / kmap.hpp:86-97.  out receives k bytes + NUL; the
 * result may contain embedded NULs (complement of a non-ACGTN byte). */
void mo_canonical(const char *kmer, int k, char *out);

/* ---- BF (bloom_filter.hpp:52-157) ---- */
typedef struct mo_bf mo_bf;
mo_bf *mo_bf_new(uint64_t size_bits);
void mo_bf_free(mo_bf *b);
void mo_bf_add_key(mo_bf *b, const char *kmer);                        /* :81-85   */
int mo_bf_test_key(const mo_bf *b, const char *kmer);                  /* :87-91   */
void mo_bf_switch_mode(mo_bf *b);                                      /* :93-98   */
int mo_bf_increment(mo_bf *b, const char *kmer, uint32_t counter);     /* :100-113 */
uint16_t mo_bf_get_count(const mo_bf *b, const char *kmer);            /* :115-125 */
uint64_t mo_bf_size(const mo_bf *b);
uint64_t mo_bf_popcount(const mo_bf *b);
const uint64_t *mo_bf_words(const mo_bf *b);   /* bit i = (words[i>>6] >> (i&63)) & 1 */
const uint16_t *mo_bf_counts(const mo_bf *b);  /* rank-indexed, valid after switch_mode */
/* up to max_out k-mers (k bytes + NUL each, into out), variants first .. first+n_trials-1 of seed (which must start
 * and end with 'A'), whose index in a filter of `size` bits is >= lo; returns how many it found */
uint64_t mo_find_kmers_at(const char *seed, int k, uint64_t size, uint64_t lo, uint64_t first, uint64_t n_trials,
                          char *out, uint64_t max_out);

/* ---- KMAP (kmap.hpp:46-132) ---- */
typedef struct mo_kmap mo_kmap;
mo_kmap *mo_kmap_new(void);
void mo_kmap_free(mo_kmap *m);
void mo_kmap_add_key(mo_kmap *m, const char *kmer);                    /* :108-112 */
int mo_kmap_test_key(const mo_kmap *m, const char *kmer);              /* :99-106  */
void mo_kmap_increment(mo_kmap *m, const char *kmer, int counter);     /* :114-122 */
int mo_kmap_get_count(const mo_kmap *m, const char *kmer);             /* :124-131 */
uint64_t mo_kmap_size(const mo_kmap *m);

/* ---- loops of main.cpp ---- */
/* main.cpp:487-500 over n records; contexts = n x ref_k ASCII bytes, no NULs */
void mo_scan_ascii(mo_bf *bf, const mo_bf *context_bf, mo_kmap *ref_bf, const char *contexts,
                   const uint32_t *counters, uint64_t n, int k, int ref_k);
/* same, from packed 128-bit words (lo,hi pairs; A=0 C=1 G=2 T=3, first base most significant) */
void mo_scan_packed(mo_bf *bf, const mo_bf *context_bf, mo_kmap *ref_bf, const uint64_t *lohi,
                    const uint32_t *counters, uint64_t n, int k, int ref_k);
/* main.cpp:385-400 for one contig (seq already upper-cased, length len) */
void mo_reference_pass(const mo_bf *bf, mo_bf *context_bf, const char *seq, uint64_t len, int k, int ref_k);
/* main.cpp:122-144: signature k-mers given as an ASCII pool + offsets */
void mo_add_signatures(mo_bf *bf, mo_kmap *ref_bf, const char *pool, const uint64_t *kmer_off,
                       const uint8_t *is_ref, uint64_t n);

/* main.cpp:151-184 on a CSR signature group.
 *   allele_sig_off[n_alleles+1] : signatures of each allele slot
 *   sig_kmer_off[n_sigs+1]      : k-mers of each signature (enumeration order)
 *   kmer_off[n_kmers+1]         : byte range of each k-mer in pool
 *   allele_is_ref[n_alleles]    : 1 -> look up ref_bf (KMAP), 0 -> bf (BF)
 * writes cov[n_alleles]. */
void mo_coverages(const mo_bf *bf, const mo_kmap *ref_bf, const char *pool, const uint64_t *kmer_off,
                  const uint64_t *sig_kmer_off, const uint64_t *allele_sig_off, const uint8_t *allele_is_ref,
                  uint64_t n_alleles, uint32_t *cov);

/* var_block.hpp:224-330 for one variant.  Writes un-normalised probabilities in
 * emission order to probs (needs n*(n+1)/2 slots) and returns the number of
 * computed_gts entries; *status = 0 normal, 1 max-coverage veto, 2 no coverage. */
int mo_genotype(const uint32_t *cov, const float *freq, int n_alleles, float error_rate, int max_cov,
                int haploid, double *probs, int *status);
/* var_block.hpp:367-394: total, normalise, first strict maximum, GQ */
void mo_call(const double *probs, int n_gts, int *best_idx, int *gq);
/* mo_genotype + mo_call over a batch (CSR: alleles of variant v are var_allele_off[v] .. var_allele_off[v+1]).
 * The likelihoods of variant v go to lik[lik_off[v] ..], which must hold max(n, n(n+1)/2) slots (n for haploid).
 * A variant with no allele writes no likelihood and reports n_gts 0, status 2, best 0, gq 0 (the GPU's contract,
 * include/malva_gpu.h). */
void mo_genotype_batch(const uint32_t *cov, const float *freq, const uint64_t *var_allele_off, uint64_t n_variants,
                       float error_rate, int max_cov, int haploid, double *lik, const uint64_t *lik_off,
                       int32_t *n_gts, int32_t *status, int32_t *best, int32_t *gq);
/* glibc 2.39 logf restated (verified exhaustively against libm in tests) */
float mo_logf(float x);

#ifdef __cplusplus
}
#endif
#endif
