/* malva_gpu.h -- C ABI of the B200-native MALVA genotyping hot path.
 *
 * The reference (AlgoLab/malva) has no FFI layer: its hot path is the public
 * surface of the header-only classes BF (bloom_filter.hpp:76-146) and KMAP
 * (kmap.hpp:46-131), the four loops of main.cpp that drive them, and
 * VB::genotype / VB::output_variants (var_block.hpp:224-396).  This header is
 * the boundary cut at exactly those call sites, turned into batch calls: the
 * caller owns host buffers, the library owns device memory, every call returns
 * 0 or a negative error code (text via mg_last_error()).  Calls on one context
 * are not thread-safe.  No torch types, no C++ types.
 *
 * k-mer word format of the sample stream: A=0 C=1 G=2 T=3, first base in the
 * most significant position, right-aligned in 128 bits, stored as two
 * little-endian u64 {lo, hi}.  k <= 63, ref_k <= 64.
 *
 * Signature k-mers (index side and genotyping side) are passed as the
 * reference passes them -- ASCII strings -- batched as a byte pool plus n+1
 * offsets; they may be shorter than k or contain non-ACGT symbols and are then
 * hashed exactly as BF::_get_hash would hash them.
 */
#ifndef MALVA_GPU_H
#define MALVA_GPU_H
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MG_OK 0
#define MG_ERR_ARG (-1)     /* bad argument / unsupported parameter        */
#define MG_ERR_CUDA (-2)    /* CUDA runtime failure (no CPU fallback)      */
#define MG_ERR_STATE (-3)   /* call out of order (e.g. scan before finalize) */
#define MG_ERR_NOMEM (-4)
#define MG_ERR_IO (-5)

typedef struct mg_ctx mg_ctx;

const char *mg_last_error(void);
int mg_version(void);
/* number of CUDA devices visible; <0 on failure (used to fail loudly) */
int mg_device_count(void);

/* initialises CUDA on `device` (driver + primary context, 0.5-5 s on a cold box); optional -- meant to be called from
 * a background thread while the host reads its input files */
int mg_warmup(int device);

/* BF bf(size); KMAP ref_bf; BF context_bf(size)      main.cpp:300-302, 451-453 */
int mg_create(mg_ctx **out, int device, int k, int ref_k, uint64_t bf_bits);
void mg_destroy(mg_ctx *ctx);

/* ------------------------------ index side ------------------------------ */
/* add_kmers_to_bf                                        main.cpp:122-144
 * is_ref[i] != 0 -> ref_bf.add_key(kmer i) ; else bf.add_key(kmer i)        */
int mg_add_signatures(mg_ctx *ctx, const char *pool, const uint64_t *kmer_off, const uint8_t *is_ref,
                      uint64_t n);
/* same inserts for signature k-mers the host already packed (exactly k symbols of ACGT each;
 * {lo,hi} words as in the sample stream): 16 B instead of k bytes over PCIe  */
int mg_add_signatures_packed(mg_ctx *ctx, const uint64_t *lohi, const uint8_t *is_ref, uint64_t n);
/* bf.switch_mode()                                       main.cpp:378      */
int mg_finalize_alt(mg_ctx *ctx);
/* reference rolling pass over one (upper-cased) contig   main.cpp:385-400  */
int mg_scan_reference(mg_ctx *ctx, const char *seq, uint64_t len);
/* context_bf.switch_mode()                               main.cpp:404      */
int mg_finalize_context(mg_ctx *ctx);

/* ------------------------------- call side ------------------------------ */
/* sample k-mer scan                                      main.cpp:487-500
 * lohi = n x {lo,hi} u64 pairs, counts = n x u32, HOST memory (pinned memory
 * from mg_host_alloc makes the copies asynchronous and double-buffered).
 * Returns after the work is enqueued; mg_sync() completes it.               */
int mg_scan_sample_kmers(mg_ctx *ctx, const uint64_t *lohi, const uint32_t *counts, uint64_t n);
/* same with DEVICE-resident inputs (GPU-side producers, kernel-only timing)  */
int mg_scan_sample_kmers_device(mg_ctx *ctx, const void *d_lohi, const void *d_counts, uint64_t n);
/* KMC database ingestion without a host-side decode (replaces CKMCFile::ReadNextKmer + CKmerAPI::to_string,
 * main.cpp:482-490).  mg_kmc_open takes the parameters and the prefix LUT of <db>.kmc_pre (lut[j] = number of
 * records before prefix index j; n_lut a multiple of 4^lut_prefix_len); mg_scan_kmc_records takes raw records of
 * <db>.kmc_suf (HOST memory, the bytes after the 4-byte "KMCS" marker): n whole records starting at global
 * record index first_record.  Records whose count is outside [min_count, max_count] are skipped like the KMC API
 * does.  10 bytes per 43-mer over PCIe instead of 20.                                                        */
int mg_kmc_open(mg_ctx *ctx, const uint64_t *lut, uint64_t n_lut, uint32_t lut_prefix_len, uint32_t kmer_len,
                uint32_t counter_size, uint32_t min_count, uint64_t max_count);
int mg_scan_kmc_records(mg_ctx *ctx, const uint8_t *records, uint64_t first_record, uint64_t n);
int mg_sync(mg_ctx *ctx);

/* set_coverages + VB::genotype + arg-max/GQ of VB::output_variants
 *                         main.cpp:151-184, var_block.hpp:224-330, 367-394  */
typedef struct {
  uint64_t n_variants;
  const uint64_t *var_allele_off; /* [n_variants+1]; allele slot j of a variant is allele index j (0 = REF) */
  const uint64_t *allele_sig_off; /* [n_alleles+1]  signatures of each allele slot          */
  const uint64_t *sig_kmer_off;   /* [n_sigs+1]     k-mers of each signature, enumeration order */
  const uint64_t *kmer_off;       /* [n_kmers+1]    byte range of each k-mer in pool        */
  const char *pool;
  const float *freq;              /* [n_alleles]    a-priori allele frequencies (Variant::frequencies) */
} mg_variant_batch;

/* A variant with no allele slot (var_allele_off[v+1] == var_allele_off[v]) has no genotype: it reserves no
 * likelihood slot, none is written for it, and it reports n_gts 0, status 2, best_gt 0, gq 0. */
typedef struct {
  uint32_t *cov;           /* [n_alleles]   Variant::coverages                               */
  int32_t *n_gts;          /* [n_variants]  number of computed_gts entries                   */
  int32_t *status;         /* [n_variants]  0 normal, 1 max-coverage veto, 2 no coverage     */
  int32_t *best_gt;        /* [n_variants]  index (emission order) of the printed GT; 0 if status != 0 */
  int32_t *gq;             /* [n_variants]  printed GQ                                        */
  const uint64_t *lik_off; /* [n_variants+1] slots reserved per variant (>= n or n(n+1)/2)     */
  double *lik;             /* un-normalised probabilities, emission order (may be NULL)      */
} mg_genotype_out;

/* The reference-shaped form: the library packs the batch on the host into the mg_packed_batch form below and runs
 * mg_genotype_packed on it; out->lik == NULL: likelihoods are not returned.  Allele slots, signatures and k-mers
 * of one batch must each number less than 2^32 (MG_ERR_ARG otherwise). */
int mg_genotype(mg_ctx *ctx, const mg_variant_batch *in, const mg_genotype_out *out, float error_rate,
                int max_coverage, int haploid);

/* The same step for signature k-mers the host already packed -- what the C++ host (csrc/host/) sends: 16 B per
 * k-mer instead of k ASCII bytes + an 8-byte offset, u32 offsets, no likelihood traffic unless asked for.
 * kmers[i] = {lo, hi} word of a signature k-mer that is exactly k symbols of ACGT (format of the sample stream);
 *   hi bit 62 set: the k-mer belongs to allele slot 0 and is looked up in ref_bf (KMAP::get_count), else in bf;
 *   hi bit 63 set: IRREGULAR k-mer (shorter than k at a contig end, or holding N / IUPAC symbols,
 *                  var_block.hpp:178-193): its text is irr_pool[irr_off[j] .. irr_off[j+1]) where irr_kmer[j] == i,
 *                  and it is hashed byte-exactly like BF::_get_hash would (bloom_filter.hpp:58-74).
 * out->lik == NULL (and then out->lik_off may be NULL): likelihoods are not returned.                          */
typedef struct {
  uint64_t n_variants;
  const uint32_t *var_allele_off; /* [n_variants+1]                                                          */
  const uint32_t *allele_sig_off; /* [n_alleles+1]                                                           */
  const uint32_t *sig_kmer_off;   /* [n_sigs+1]                                                              */
  const uint64_t *kmers;          /* [n_kmers] x {lo, hi}                                                    */
  const float *freq;              /* [n_alleles]                                                             */
  uint64_t n_irregular;
  const uint64_t *irr_off;        /* [n_irregular+1] byte ranges in irr_pool                                 */
  const char *irr_pool;
  const uint32_t *irr_kmer;       /* [n_irregular] index in kmers[] of each irregular k-mer                  */
} mg_packed_batch;
int mg_genotype_packed(mg_ctx *ctx, const mg_packed_batch *in, const mg_genotype_out *out, float error_rate,
                       int max_coverage, int haploid);
typedef struct {
  uint64_t n_variants, n_alleles, n_sigs, n_kmers;
  uint64_t irr_pool_bytes;
  uint64_t lik_slots; /* sum over variants of max(n, haploid ? n : n(n+1)/2): likelihood slots of the batch */
} mg_packed_dims;
/* every array of in/out DEVICE-resident (enqueued on the context's stream; mg_sync completes it) */
int mg_genotype_packed_device(mg_ctx *ctx, const mg_packed_batch *in, const mg_genotype_out *out,
                              const mg_packed_dims *dims, float error_rate, int max_coverage, int haploid);

/* The two halves of the step on their own, for replicas that sum LOOK-UP RESULTS instead of counters: get_count is
 * linear in the counters (bf: the u16 wrap of a sum of u32 parts; ref_bf: 32-bit wrap-around), so N replicas that each
 * scanned a share of the sample stream look the batch up in their own partial counters (mg_lookup_packed_device:
 * KMAP::get_count / BF::get_count per signature k-mer, bf counters UNMASKED), sum the weight vectors -- 4 bytes per
 * signature k-mer, e.g. one ncclReduce per batch -- and the destination genotypes from the sum
 * (mg_genotype_weights_device: applies BF::get_count's uint16_t to the bf weights in place, then set_coverages +
 * VB::genotype).  No counter array travels.  All pointers DEVICE pointers; enqueued on the context's stream. */
int mg_lookup_packed_device(mg_ctx *ctx, const mg_packed_batch *in, const mg_packed_dims *dims, uint32_t *d_weights);
int mg_genotype_weights_device(mg_ctx *ctx, const mg_packed_batch *in, const mg_genotype_out *out,
                               const mg_packed_dims *dims, uint32_t *d_weights, float error_rate, int max_coverage,
                               int haploid);
/* puts the caller's CUDA stream (a cudaStream_t, e.g. the one its collectives are ordered on) in the place of the
 * context's own first stream: library work then orders with the caller's kernels without host synchronisation.
 * NULL (also the handle of the legacy default stream, which therefore cannot be chosen) restores the private stream. */
int mg_set_stream(mg_ctx *ctx, void *cuda_stream);

/* -------------------- k-mer counting (the step before the path) ---------- */
/* What the wrapper script obtains from `kmc -k<ref_k> -ci2 -cs255` (MALVA:107) and malva-geno lists through the KMC
 * API (main.cpp:482-490): canonical k-mers of the reads, windows with a non-ACGT symbol skipped, k-mers seen fewer
 * than min_count times (or more than max_count) dropped, counts saturated at counter_max, ascending order.
 * mg_count_add takes read bytes in HOST memory, records separated by any non-ACGT byte (e.g. '\n'); a k-mer never
 * spans two calls.  For inputs whose distinct k-mers exceed device memory, run several passes over the reads with
 * mg_count_set_partition (only canonical k-mers whose top part_bits bits lie in [part_lo, part_hi) are counted;
 * passes in ascending prefix order yield the listing order) and mg_count_reset between them. */
typedef struct mg_counter mg_counter;
int mg_count_create(mg_counter **out, int device, int k);
void mg_count_destroy(mg_counter *c);
int mg_count_set_partition(mg_counter *c, int part_bits, uint32_t part_lo, uint32_t part_hi);
int mg_count_reset(mg_counter *c);
int mg_count_add(mg_counter *c, const char *bases, uint64_t n);
/* Counting restricted to what ctx's index can use: from then on mg_count_add inserts only the ref_k-mers whose
 * central k-mer (taken as the sample scan takes it from a record) sets a bit of ctx's bf or is a key of its ref_bf.
 * Every other ref_k-mer changes no counter in mg_scan_counted, and every occurrence of a ref_k-mer gets the same
 * answer, so restricted counting + mg_scan_counted leaves exactly the counters of unrestricted counting; the table
 * only holds the ref_k-mers that matter.  A partition still applies on top.  Needs c and ctx on one device,
 * c's k == ctx's ref_k (MG_ERR_ARG), ctx past mg_finalize_alt and an empty counter -- fresh or just reset
 * (MG_ERR_STATE).  The counter keeps the pointer and reads ctx's index at every mg_count_add: ctx must outlive the
 * restricted adds.  ctx == NULL lifts the restriction (also on an empty counter only). */
int mg_count_restrict(mg_counter *c, mg_ctx *ctx);
/* Counting inputs larger than the table can hold, with one read of the input.
 * mg_count_set_limit caps the table at max_slots slots (0, the default: only device memory limits it; a non-zero cap
 * is at least 65536).  A growth past the cap fails as one that does not fit the device does: MG_ERR_NOMEM, the table
 * left as it was.  The environment variable MG_COUNT_MAX_SLOTS sets the same cap at mg_count_create.
 * mg_count_add_keep counts as mg_count_add does and also returns the 2-bit copy of what it counted: every maximal run
 * of A/C/G/T bytes at least k long, 2 bits a base (A0 C1 G2 T3), 4 to a byte, first base in the high bits, each run
 * from a byte boundary, appended to packed (*n_bytes) with its length in run_len (*n_runs).  Capacities of
 * n / 2 + 1 bytes and n / (k + 1) + 2 runs always suffice (MG_ERR_ARG when they do not).  When the table
 * meets its limit (or device memory) the counter is OVERFLOWED: counting stops, packing goes on for this and later
 * calls, mg_count_stats reports it and mg_count_finish refuses it (MG_ERR_STATE) until mg_count_reset.
 * mg_count_add_packed counts such a copy from host memory (the caller's runs, concatenated), staged through pinned
 * buffers; the partition and the limit apply: it fails with MG_ERR_NOMEM once the table nears its limit, for the
 * caller to reset and count a narrower prefix range.  Both refuse a restricted counter (MG_ERR_STATE). */
int mg_count_set_limit(mg_counter *c, uint64_t max_slots);
int mg_count_add_keep(mg_counter *c, const char *bases, uint64_t n, uint8_t *packed, uint64_t packed_cap,
                      uint32_t *run_len, uint64_t len_cap, uint64_t *n_bytes, uint64_t *n_runs);
int mg_count_add_packed(mg_counter *c, const uint8_t *packed, uint64_t n_bytes, const uint32_t *run_len,
                        uint64_t n_runs);
int mg_count_finish(mg_counter *c, uint32_t min_count, uint32_t counter_max, uint64_t max_count, uint64_t *n_kmers);
int mg_count_download(mg_counter *c, uint64_t *lohi, uint32_t *counts, uint64_t cap);
/* {distinct k-mers in the table, k-mer instances counted, table capacity, kernels launched[, device time of the
 * counting kernels in microseconds[, valid windows examined[, overflowed (0/1)[, device time of the host-to-device
 * copies of mg_count_add_packed in microseconds[, device time of packing in microseconds]]]]]}; n >= 4.  Windows are
 * counted before the partition and index tests of a restricted counter; an unrestricted counter reports its
 * instances there (without a partition it inserts every valid window). */
int mg_count_stats(mg_counter *c, uint64_t *stats, int n);
/* the counted k-mers straight into the sample scan (same device): no database file, no host round trip */
int mg_scan_counted(mg_ctx *ctx, mg_counter *c);

/* ------------------------- batch queries (BF / KMAP) --------------------- */
/* which: 0 = bf, 1 = context_bf, 2 = ref_bf (KMAP).  BF::test_key / KMAP::test_key */
int mg_test_keys(mg_ctx *ctx, int which, const char *pool, const uint64_t *kmer_off, uint64_t n, uint8_t *out);
/* BF::get_count (is_ref==0, u16 semantics) / KMAP::get_count (is_ref!=0, int semantics) */
int mg_get_counts(mg_ctx *ctx, const char *pool, const uint64_t *kmer_off, const uint8_t *is_ref, uint64_t n,
                  int32_t *out);

/* ------------------------------ state access ----------------------------- */
int mg_bf_popcount(mg_ctx *ctx, int which, uint64_t *ones);
/* bit i = (words[i>>6] >> (i&63)) & 1 ; n_words = ceil(bf_bits/64)          */
int mg_bf_download_bits(mg_ctx *ctx, int which, uint64_t *words, uint64_t n_words);
/* rank-indexed u16 counters of bf (valid after mg_finalize_alt)             */
int mg_bf_download_counts(mg_ctx *ctx, uint16_t *counts, uint64_t n);
/* number of ref_bf keys (packed + irregular)                                */
int mg_kmap_size(mg_ctx *ctx, uint64_t *n);

/* {probe lines, set bits of bf, packed ref keys, keys in the overflow table, overflow capacity,
 * irregular (non-ACGT / short) ref keys}; n >= 6 */
int mg_index_stats(mg_ctx *ctx, uint64_t *stats, int n);

/* The live counters sit inside the probe lines (one HBM line per k-mer).  For a sum-reduce across replicas
 * (NCCL between processes) they are gathered into DENSE u32 arrays -- mg_counters_gather -- whose device pointers
 * and lengths mg_counter_buffers returns: [0] one per set bit of bf (rank order), [1] one per ref key held by the
 * probe lines (line order), [2] overflow table.  After the reduce the destination rank calls mg_counters_scatter
 * to write the sums back into its probe lines. */
int mg_counters_gather(mg_ctx *ctx);
int mg_counter_buffers(mg_ctx *ctx, void **d_ptr /*[3]*/, uint64_t *n /*[3]*/);
int mg_counters_scatter(mg_ctx *ctx);

/* Replicas inside one process: ctx[0..n-1] hold the same index (on any devices) and each scanned a share of the
 * sample stream; adds the counters of ctx[1..n-1] into ctx[0] (gather on every device, one N-way sum kernel that
 * reads the peers' dense arrays in place over NVLink, scatter on ctx[0]).  After it ctx[0] answers mg_genotype /
 * mg_get_counts for the whole stream. */
int mg_reduce_counts(mg_ctx **ctx, int n);

/* A new context on `device` holding exactly src's index and live counters: both filters, the ref keys, the rank
 * directory, the overflow table, every counter, the irregular ref keys and the finalize state.  Device-to-device
 * copies (cudaMemcpyPeerAsync; the same device works too) instead of a second load: the index image is canonical.
 * Waits for src's enqueued work first and returns after the copies completed.  Not copied: a sample set, the KMC
 * parameters of mg_kmc_open, a caller stream of mg_set_stream.  The two contexts are independent afterwards (either
 * may be destroyed first).  src must be past mg_finalize_alt (MG_ERR_STATE); a device that is not visible fails
 * like mg_create. */
int mg_replicate(mg_ctx **out, mg_ctx *src, int device);

/* Sample sets: several samples genotyped against one index, each from its own counters.  Every counter a signature
 * k-mer can read has a ROW fixed by the index: rows [0, bf_ones) are the set bits of bf in rank order, the next
 * (ref keys - overflow keys) rows the ref keys held by the probe lines in line order, the last (overflow capacity)
 * rows the slots of the overflow table (mg_index_stats).  A set keeps one u32 COLUMN per sample over those rows,
 * row-major (the counts of one row for all samples are adjacent): 4 bytes x rows of device memory per sample.
 *   mg_samples_begin   allocates a set of n_samples (1..MG_SAMPLE_SET_MAX) zeroed columns; a column never taken
 *                      reads as zero.  Calling it again replaces the set; needs mg_finalize_alt.
 *   mg_samples_take    waits for the scans enqueued so far, then copies every live counter into column s (the
 *                      inline alt counters, bf_counts, the key counts, the overflow counts) and ZEROES the live
 *                      counters: column s holds exactly what the live counters held at the call, and the live
 *                      counters are zero after it, so the next sample scans into a clean index.  Nothing else in the
 *                      index changes.  mg_get_counts, mg_genotype_packed and mg_counters_* keep reading the live
 *                      counters (a gathered dense image is zeroed with them).
 *   mg_genotype_samples_packed   mg_genotype_packed (HOST buffers) for every sample of the set at once: out[s] gets
 *                      exactly what mg_genotype_packed returns on a context whose live counters equal column s.  One
 *                      look-up for the set, then coverage and likelihoods per sample; n_samples must equal the size
 *                      of the set (MG_ERR_ARG), and a set must exist (MG_ERR_STATE).  out[s].lik are all NULL or all
 *                      set; the likelihood slots are those of out[0].lik_off for every sample.
 *                      mg_genotype_kernel_ms reports its look-up, the coverage of all samples and their likelihoods.
 *   mg_samples_end     frees the set (mg_destroy does too). */
#define MG_SAMPLE_SET_MAX 32
int mg_samples_begin(mg_ctx *ctx, int n_samples);
/* the largest set that fits: MG_SAMPLE_SET_MAX at most, and columns in at most 3/4 of the free device memory (the
 * current set counted as free); 0 when not even one column fits */
int mg_samples_capacity(mg_ctx *ctx, int *n);
int mg_samples_take(mg_ctx *ctx, int s);
int mg_genotype_samples_packed(mg_ctx *ctx, const mg_packed_batch *in, const mg_genotype_out *out, int n_samples,
                               float error_rate, int max_coverage, int haploid);
int mg_samples_end(mg_ctx *ctx);

/* index image for the index file (BF::operator>> / KMAP::operator>>, main.cpp:406-412; loading :455-461).
 * Filters travel as sorted lists of set-bit indices (the reference writes the raw 2 x bf_bits/8 bytes), ref_bf
 * as its packed canonical keys.  Call with out == NULL to get the count first.  Import the bits of bf (which=0)
 * and the keys (mg_add_signatures_packed, is_ref=1) BEFORE mg_finalize_alt, the bits of context_bf after it. */
int mg_export_set_bits(mg_ctx *ctx, int which, uint64_t *out, uint64_t cap, uint64_t *n);
int mg_import_set_bits(mg_ctx *ctx, int which, const uint64_t *idx, uint64_t n);
int mg_export_ref_keys(mg_ctx *ctx, uint64_t *lohi, uint64_t cap, uint64_t *n);

/* ------------------------------ measurement ------------------------------ */
/* CUDA-event timing on the library's own streams (64 event slots): record marks a point that follows
 * all work enqueued so far; elapsed waits for event b.  The device-side counterpart of the reference's
 * pelapsed() phase timers (main.cpp:93-115). */
int mg_event_record(mg_ctx *ctx, int idx);
int mg_event_elapsed_ms(mg_ctx *ctx, int a, int b, float *ms);
/* blocks until everything enqueued before mg_event_record(ctx, idx) has completed (e.g. before a pinned
 * buffer handed to mg_scan_kmc_records / mg_scan_sample_kmers is refilled) */
int mg_event_sync(mg_ctx *ctx, int idx);
/* device time of the last mg_genotype call: {signature look-ups, coverage, likelihood} kernels, ms */
int mg_genotype_kernel_ms(mg_ctx *ctx, float *ms3);
/* device time of the rolling-pass kernel of the last mg_scan_reference call (contigs >= ref_k), ms */
int mg_refpass_kernel_ms(mg_ctx *ctx, float *ms);
/* kernels launched by this context so far */
int mg_launch_count(mg_ctx *ctx, uint64_t *n);
/* measured ceilings over `bytes` of HBM, GB/s of useful bytes, best of reps: mode 0 / 2 / 3 = independent
 * random reads of 1 / 2 / 4 separate sectors of an aligned 32 / 64 / 128-byte unit; mode 4 / 5 / 6 = random
 * aligned 128 / 64 / 32-byte units fetched by 8 / 4 / 2 lanes in one coalesced request (mode 4 is the sample
 * scan's pattern); mode 1 = streaming reads */
int mg_diag_bandwidth(int device, int mode, uint64_t bytes, int reps, double *gbs);

/* pinned host memory for the sample stream */
int mg_host_alloc(void **p, size_t bytes);
int mg_host_free(void *p);

/* ----------------------- host-side self tests (no GPU) ------------------- */
/* The device helpers are __host__ __device__; these run them on the CPU so the
 * CPU-only test-suite can pin the exact code the kernels execute.            */
uint64_t mg_selftest_hash_packed(uint64_t lo, uint64_t hi, int k, uint64_t *canon_lo, uint64_t *canon_hi);
uint64_t mg_selftest_hash_packed_k35(uint64_t lo, uint64_t hi);
uint64_t mg_selftest_hash_packed_k43(uint64_t lo, uint64_t hi);
uint64_t mg_selftest_hash_ascii(const char *s, int len);
float mg_selftest_logf(float x);
int mg_selftest_genotype(const uint32_t *cov, const float *freq, int n_alleles, float error_rate, int max_cov,
                         int haploid, double *lik, int *status, int *best_gt, int *gq);

#ifdef __cplusplus
}
#endif
#endif /* MALVA_GPU_H */
