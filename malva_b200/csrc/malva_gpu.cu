// libmalva_gpu.so -- the C ABI of include/malva_gpu.h over the hand-written sm_100a kernels of
// kernels.cuh.  Device data layout: index.cuh (128-byte probe lines = filter bits + ref-key slots with their
// counts + rank + alt counters, overflow table, context filter).
// There is no CPU fallback anywhere: every entry point fails with MG_ERR_CUDA when no device is usable.
#include <cuda_runtime.h>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <cmath>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <cstring>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/malva_gpu.h"
#include "count.cuh"
#include "kernels.cuh"

using mg::DevView;
using mg::u128;

// ---------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static int set_err(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (call);                                                                      \
    if (e__ != cudaSuccess)                                                                        \
      return set_err(MG_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e__)); \
  } while (0)

extern "C" const char *mg_last_error(void) { return g_err; }
extern "C" int mg_version(void) { return 200; }
extern "C" int mg_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    set_err(MG_ERR_CUDA, "cudaGetDeviceCount -> %s", cudaGetErrorString(e));
    return MG_ERR_CUDA;
  }
  return n;
}

// CUDA start-up (driver initialisation + primary context) costs 0.5-5 s on a cold box: a host program calls this
// from a background thread first thing, so that it overlaps with reading its input files.
extern "C" int mg_warmup(int device) {
  CU(cudaSetDevice(device));
  CU(cudaFree(nullptr));
  return MG_OK;
}

// ---------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------
// k-mers (KMC records) per staging chunk of the host-buffer scans; tests/test_gpu_scale.py sizes its inputs to cross
// these chunks on both streams and fails if this changes
constexpr uint64_t STAGE_KMERS = 1ull << 22;

struct mg_ctx {
  int device = 0, k = 0, ref_k = 0, sms = 0;
  uint64_t bf_bits = 0, n_lines = 0, n_ctx_words = 0;
  uint4 *lines = nullptr;          // n_lines x 128 B
  uint32_t *ctx_words = nullptr;   // context_bf bits
  uint32_t *occ = nullptr;         // occupancy pre-filter (index.cuh), one bit per 2^occ_shift bf indices
  uint64_t n_occ_words = 0;
  int occ_shift = 0;
  uint32_t *bf_counts = nullptr;   // one per set bit of bf (dense image; live for set bits 3.. of a line)
  uint32_t *key_counts = nullptr;  // n_lines x 5, wide layout (k >= 48) only
  uint32_t *key_rank = nullptr;    // keys held by the lines before line L (built by the first mg_counters_gather)
  uint32_t *key_dense = nullptr;   // dense image of the in-line key counts (n_keys - ovf_n entries)
  u128 *ovf_keys = nullptr;
  uint32_t *ovf_counts = nullptr;
  int ovf_log2 = 0;
  uint64_t ovf_n = 0;  // keys in the overflow table
  uint64_t bf_ones = 0;
  uint64_t n_keys = 0;  // distinct packed ref keys (lines + overflow)
  void *add_arena = nullptr;  // device staging of mg_add_signatures* batches (grow-only)
  uint64_t add_arena_bytes = 0;
  uint8_t *ref_pinned[2] = {nullptr, nullptr};  // pinned + device chunk buffers of mg_scan_reference
  uint8_t *ref_dev[2] = {nullptr, nullptr};
  cudaEvent_t ref_ev[2] = {nullptr, nullptr}, ref_kev[2] = {nullptr, nullptr};
  std::vector<cudaEvent_t> rp_events;  // start/stop around the rolling-pass kernel of every chunk of the last contig
  size_t rp_chunks = 0;
  bool alt_final = false, ctx_final = false;
  unsigned long long *d_scalars = nullptr;  // [0] new keys [1] irregular [2] popcount [3] error [4] spilled
  std::unordered_map<std::string, int> irregular_ref;  // ref keys that are not k symbols of ACGT (always count 0)
  cudaStream_t stream[2] = {nullptr, nullptr};
  cudaStream_t own_stream0 = nullptr;  // the context's own first stream while mg_set_stream has put the caller's there
  void *d_stage_k[2] = {nullptr, nullptr};
  uint32_t *d_stage_c[2] = {nullptr, nullptr};
  int next_stage = 0;
  uint64_t stage_unit = 0;  // bytes per k-mer the staging buffers were sized for
  uint4 *hit_buf[2] = {nullptr, nullptr};  // deferred filter hits of the scan, one set per stream (grow-only)
  uint32_t *hit_counts[2] = {nullptr, nullptr};
  uint64_t hit_entries[2] = {0, 0}, hit_warps[2] = {0, 0};
  bool defer_hits = true;
  int scan_ctas_per_sm = 64;  // grid cap of the scan kernel, in 256-thread CTAs per SM (measured optimum 32..128, profiles/)
  uint64_t *kmc_lut = nullptr;  // device copy of the KMC prefix LUT (+ guard)
  uint32_t kmc_n_lut = 0, kmc_min = 0;
  uint64_t kmc_max = 0;
  int kmc_prefix_len = 0, kmc_suf_bytes = 0, kmc_counter_size = 0;
  uint64_t launches = 0;  // kernels launched by this context (bench.py's gpu_launches)
  cudaEvent_t tj = nullptr;
  cudaEvent_t ge[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // look-up [0,1], coverage [4,2], genotype [2,3]
  void *geno_scratch = nullptr;  // per-k-mer weights + ref flags of mg_genotype
  uint64_t geno_scratch_bytes = 0;
  void *geno_arena = nullptr;  // device image of the last mg_genotype batch (grow-only)
  double *log_table = nullptr;  // the host libm's log((double)i), i < mg::LOG_TABLE_N (geno.cuh log_int)
  uint64_t geno_arena_bytes = 0;
  cudaEvent_t evs[64] = {};

  DevView view() const {
    DevView v;
    v.lines = lines;
    v.n_lines = n_lines;
    v.ctx_words = ctx_words;
    v.bf_counts = bf_counts;
    v.key_counts = key_counts;
    v.ovf_keys = ovf_keys;
    v.ovf_counts = ovf_counts;
    v.ovf_mask = (1ull << ovf_log2) - 1;
    v.ovf_shift = 64 - ovf_log2;
    v.key_hi_mask = mg::key_hi_mask_for(k);
    v.ovf_flag_hi = mg::ovf_flag_for(k);
    v.inline_counts = k <= mg::INLINE_MAX_K ? 1 : 0;
    v.bf_bits = bf_bits;
    v.bf_mask = (bf_bits & (bf_bits - 1)) == 0 ? bf_bits - 1 : 0;
    v.k = k;
    v.ref_k = ref_k;
    v.occ = occ;
    v.occ_shift = occ_shift;
    return v;
  }
};

static int grid_for(uint64_t n, int threads) { return (int)((n + (uint64_t)threads - 1) / (uint64_t)threads); }

static int ovf_alloc(mg_ctx *c, int log2cap, u128 **keys, uint32_t **counts) {
  uint64_t cap = 1ull << log2cap;
  CU(cudaMalloc(keys, cap * sizeof(u128)));
  CU(cudaMalloc(counts, cap * sizeof(uint32_t)));
  c->launches++;
  mg::k_fill_keys<<<grid_for(cap, 256), 256, 0, c->stream[0]>>>(*keys, cap, mg::key_hi_mask_for(c->k));
  CU(cudaGetLastError());
  CU(cudaMemsetAsync(*counts, 0, cap * sizeof(uint32_t), c->stream[0]));
  return MG_OK;
}

// make room for `extra` more overflow keys at load <= 0.5
static int ovf_reserve(mg_ctx *c, uint64_t extra) {
  uint64_t need = (c->ovf_n + extra) * 2;
  if (need <= (1ull << c->ovf_log2)) return MG_OK;
  int nl = c->ovf_log2;
  while ((1ull << nl) < need) ++nl;
  u128 *nk = nullptr;
  uint32_t *nc = nullptr;
  int rc = ovf_alloc(c, nl, &nk, &nc);
  if (rc) return rc;
  u128 *ok = c->ovf_keys;
  uint32_t *oc = c->ovf_counts;
  uint64_t ocap = 1ull << c->ovf_log2;
  c->ovf_keys = nk;
  c->ovf_counts = nc;
  c->ovf_log2 = nl;
  if (c->ovf_n) {
    c->launches++;
    mg::k_rehash<<<grid_for(ocap, 256), 256, 0, c->stream[0]>>>(ok, ocap, c->view(), nk);
    CU(cudaGetLastError());
  }
  CU(cudaStreamSynchronize(c->stream[0]));
  CU(cudaFree(ok));
  CU(cudaFree(oc));
  return MG_OK;
}

static int ctx_init(mg_ctx *c);
extern "C" int mg_create(mg_ctx **out, int device, int k, int ref_k, uint64_t bf_bits) {
  if (!out) return set_err(MG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (k < 1 || ref_k < k || ref_k > 64 || k > 63)
    return set_err(MG_ERR_ARG, "unsupported k=%d ref_k=%d (need 1 <= k <= 63, k <= ref_k <= 64)", k, ref_k);
  if (bf_bits == 0) return set_err(MG_ERR_ARG, "bf_bits must be > 0 (the reference divides by it)");
  if (bf_bits >= (1ull << 40)) return set_err(MG_ERR_ARG, "bf_bits must be < 2^40");
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return set_err(MG_ERR_CUDA, "device %d not available (%d visible)", device, ndev);
  CU(cudaSetDevice(device));
  mg_ctx *c = new mg_ctx();
  c->device = device;
  c->k = k;
  c->ref_k = ref_k;
  c->bf_bits = bf_bits;
  int rc = ctx_init(c);
  if (rc) {  // (e.g. out of device memory for a large -b): nothing is left behind
    char msg[sizeof(g_err)];
    memcpy(msg, g_err, sizeof(msg));
    mg_destroy(c);
    memcpy(g_err, msg, sizeof(msg));
    return rc;
  }
  *out = c;
  return MG_OK;
}

static int ctx_init(mg_ctx *c) {
  const int device = c->device;
  const uint64_t bf_bits = c->bf_bits;
  c->n_lines = (bf_bits + 255) / 256;
  c->n_ctx_words = c->n_lines * 8;
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  c->sms = prop.multiProcessorCount;
  if (const char *e = getenv("MG_SCAN_CTAS_PER_SM")) c->scan_ctas_per_sm = atoi(e) > 0 ? atoi(e) : 64;
  if (const char *e = getenv("MG_SCAN_DEFER_HITS")) c->defer_hits = atoi(e) != 0;
  for (int i = 0; i < 2; ++i) CU(cudaStreamCreateWithFlags(&c->stream[i], cudaStreamNonBlocking));
  CU(cudaMalloc(&c->lines, c->n_lines * 128));
  CU(cudaMalloc(&c->ctx_words, c->n_ctx_words * 4));
  c->launches++;
  mg::k_init_lines<<<grid_for(c->n_lines * mg::LINE_U4, 256), 256, 0, c->stream[0]>>>(c->lines, c->n_lines,
                                                                                      mg::key_hi_mask_for(c->k));
  CU(cudaGetLastError());
  CU(cudaMemsetAsync(c->ctx_words, 0, c->n_ctx_words * 4, c->stream[0]));
  if (c->k > mg::INLINE_MAX_K) {  // wide keys leave no room for the count inside the slot
    CU(cudaMalloc(&c->key_counts, c->n_lines * mg::LINE_KEYS * 4));
    CU(cudaMemsetAsync(c->key_counts, 0, c->n_lines * mg::LINE_KEYS * 4, c->stream[0]));
  }
  // occupancy pre-filter: at most 2^MG_OCC_LOG2_BITS bits (default 2^29 = 64 MB: half of the 126 MB L2, the measured optimum)
  {
    int cap_log2 = 29;
    if (const char *e = getenv("MG_OCC_LOG2_BITS")) cap_log2 = atoi(e);
    if (cap_log2 > 0) {
      if (cap_log2 < 10) cap_log2 = 10;
      if (cap_log2 > 34) cap_log2 = 34;
      while (((bf_bits - 1) >> c->occ_shift) + 1 > (1ull << cap_log2)) ++c->occ_shift;
      c->n_occ_words = ((((bf_bits - 1) >> c->occ_shift) + 1) + 31) / 32;
      c->n_occ_words = (c->n_occ_words + 3) & ~3ull;  // whole 16-byte pieces (the scan copies them with cp.async)
      CU(cudaMalloc(&c->occ, c->n_occ_words * 4));
      CU(cudaMemsetAsync(c->occ, 0, c->n_occ_words * 4, c->stream[0]));
    }
  }
  {  // log_binomial's logs of small integers from the reference's libm: GT of exact ties comes from their last bits
    std::vector<double> tab(mg::LOG_TABLE_N, 0.0);
    for (int i = 1; i < mg::LOG_TABLE_N; ++i) tab[i] = log((double)i);
    CU(cudaMalloc(&c->log_table, tab.size() * sizeof(double)));
    CU(cudaMemcpy(c->log_table, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
  }
  CU(cudaMalloc(&c->d_scalars, 8 * sizeof(unsigned long long)));
  CU(cudaMemsetAsync(c->d_scalars, 0, 8 * sizeof(unsigned long long), c->stream[0]));
  c->ovf_log2 = 10;
  int rc = ovf_alloc(c, c->ovf_log2, &c->ovf_keys, &c->ovf_counts);
  if (rc) return rc;
  CU(cudaStreamSynchronize(c->stream[0]));
  return MG_OK;
}

extern "C" void mg_destroy(mg_ctx *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  cudaFree(c->lines);
  cudaFree(c->ctx_words);
  cudaFree(c->occ);
  cudaFree(c->bf_counts);
  cudaFree(c->key_counts);
  cudaFree(c->key_rank);
  cudaFree(c->key_dense);
  cudaFree(c->add_arena);
  for (int i = 0; i < 2; ++i) {
    if (c->ref_pinned[i]) cudaFreeHost(c->ref_pinned[i]);
    cudaFree(c->ref_dev[i]);
    if (c->ref_ev[i]) cudaEventDestroy(c->ref_ev[i]);
    if (c->ref_kev[i]) cudaEventDestroy(c->ref_kev[i]);
  }
  for (auto e : c->rp_events) cudaEventDestroy(e);
  cudaFree(c->ovf_keys);
  cudaFree(c->ovf_counts);
  cudaFree(c->d_scalars);
  cudaFree(c->geno_scratch);
  cudaFree(c->geno_arena);
  cudaFree(c->log_table);
  cudaFree(c->kmc_lut);
  for (int i = 0; i < 2; ++i) {
    cudaFree(c->hit_buf[i]);
    cudaFree(c->hit_counts[i]);
    cudaFree(c->d_stage_k[i]);
    cudaFree(c->d_stage_c[i]);
  }
  if (c->own_stream0) c->stream[0] = c->own_stream0;
  for (int i = 0; i < 2; ++i)
    if (c->stream[i]) cudaStreamDestroy(c->stream[i]);
  if (c->tj) cudaEventDestroy(c->tj);
  for (int i = 0; i < 5; ++i)
    if (c->ge[i]) cudaEventDestroy(c->ge[i]);
  for (int i = 0; i < 64; ++i)
    if (c->evs[i]) cudaEventDestroy(c->evs[i]);
  delete c;
}

static int check_too_long(mg_ctx *c) {
  unsigned long long flag = 0;
  CU(cudaMemcpy(&flag, c->d_scalars + 3, 8, cudaMemcpyDeviceToHost));
  if (flag) {
    CU(cudaMemset(c->d_scalars + 3, 0, 8));
    return set_err(MG_ERR_ARG, "signature k-mer longer than 128 bytes");
  }
  return MG_OK;
}

// upload an ASCII pool + offsets (+ optional flags)
struct DevBatch {
  uint8_t *pool = nullptr;
  uint64_t *off = nullptr;
  uint8_t *flags = nullptr;
  ~DevBatch() {
    cudaFree(pool);
    cudaFree(off);
    cudaFree(flags);
  }
};
static int upload_batch(mg_ctx *c, DevBatch &b, const char *pool, const uint64_t *off, const uint8_t *flags,
                        uint64_t n) {
  uint64_t bytes = off[n];
  CU(cudaMalloc(&b.pool, bytes ? bytes : 1));
  CU(cudaMalloc(&b.off, (n + 1) * 8));
  CU(cudaMemcpyAsync(b.pool, pool, bytes, cudaMemcpyHostToDevice, c->stream[0]));
  CU(cudaMemcpyAsync(b.off, off, (n + 1) * 8, cudaMemcpyHostToDevice, c->stream[0]));
  if (flags) {
    CU(cudaMalloc(&b.flags, n ? n : 1));
    CU(cudaMemcpyAsync(b.flags, flags, n, cudaMemcpyHostToDevice, c->stream[0]));
  }
  return MG_OK;
}

struct DevFree {
  void *p = nullptr;
  ~DevFree() { cudaFree(p); }
};

// device staging of an insert batch: one grow-only arena per context instead of five cudaMalloc/cudaFree pairs per
// call (each of which synchronises the device)
static int add_arena(mg_ctx *c, uint64_t bytes, uint8_t **out) {
  if (c->add_arena_bytes < bytes) {
    CU(cudaStreamSynchronize(c->stream[0]));
    cudaFree(c->add_arena);
    c->add_arena = nullptr;
    c->add_arena_bytes = 0;
    CU(cudaMalloc(&c->add_arena, bytes + bytes / 4 + 4096));
    c->add_arena_bytes = bytes + bytes / 4 + 4096;
  }
  *out = reinterpret_cast<uint8_t *>(c->add_arena);
  return MG_OK;
}
static uint64_t al256(uint64_t x) { return (x + 255) & ~255ull; }

// after an insert kernel: account for new keys, run the overflow pass for spilled keys
static int finish_inserts(mg_ctx *c, const uint32_t *d_spill, const uint8_t *d_pool, const uint64_t *d_off,
                          const uint4 *d_packed, unsigned long long *n_irregular) {
  unsigned long long sc[5];
  CU(cudaMemcpyAsync(sc, c->d_scalars, sizeof(sc), cudaMemcpyDeviceToHost, c->stream[0]));
  CU(cudaStreamSynchronize(c->stream[0]));
  c->n_keys += sc[0];
  if (n_irregular) *n_irregular = sc[1];
  if (sc[4]) {
    int rc = ovf_reserve(c, sc[4]);
    if (rc) return rc;
    CU(cudaMemsetAsync(c->d_scalars, 0, 8, c->stream[0]));
    c->launches++;
    mg::k_add_spill<<<grid_for(sc[4], 128), 128, 0, c->stream[0]>>>(d_spill, sc[4], d_pool, d_off, d_packed, c->view(),
                                                                    c->ovf_keys, c->d_scalars);
    CU(cudaGetLastError());
    unsigned long long added = 0;
    CU(cudaMemcpyAsync(&added, c->d_scalars, 8, cudaMemcpyDeviceToHost, c->stream[0]));
    CU(cudaStreamSynchronize(c->stream[0]));
    c->n_keys += added;
    c->ovf_n += added;
  }
  return MG_OK;
}

extern "C" int mg_add_signatures(mg_ctx *c, const char *pool, const uint64_t *off, const uint8_t *is_ref,
                                 uint64_t n) {
  if (!c || !off || !is_ref || (!pool && n && off[n])) return set_err(MG_ERR_ARG, "NULL argument");
  if (c->alt_final) return set_err(MG_ERR_STATE, "mg_add_signatures after mg_finalize_alt");
  if (n == 0) return MG_OK;
  if (n > 0xFFFFFFFFull) return set_err(MG_ERR_ARG, "batch too large (max 2^32-1 k-mers per call)");
  CU(cudaSetDevice(c->device));
  const uint64_t bytes = off[n];
  const uint64_t o_pool = 0, o_off = al256(bytes + 16), o_flags = o_off + al256((n + 1) * 8), o_irr = o_flags + al256(n),
                 o_spill = o_irr + al256(n * 4), total = o_spill + al256(n * 4);
  uint8_t *d = nullptr;
  int rc = add_arena(c, total, &d);
  if (rc) return rc;
  cudaStream_t st = c->stream[0];
  if (bytes) CU(cudaMemcpyAsync(d + o_pool, pool, bytes, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_off, off, (n + 1) * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_flags, is_ref, n, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(c->d_scalars, 0, 8 * sizeof(unsigned long long), st));
  c->launches++;
  mg::k_add_signatures<<<grid_for(n, 128), 128, 0, st>>>(d + o_pool, (const uint64_t *)(d + o_off), d + o_flags, n, c->view(),
                                                         c->occ, c->d_scalars, (uint32_t *)(d + o_irr),
                                                         (uint32_t *)(d + o_spill));
  CU(cudaGetLastError());
  unsigned long long n_irr = 0;
  rc = finish_inserts(c, (const uint32_t *)(d + o_spill), d + o_pool, (const uint64_t *)(d + o_off), nullptr, &n_irr);
  if (rc) return rc;
  if (n_irr) {  // ref keys that are not k x ACGT: keep them host-side (kmap.hpp:86-112 semantics)
    std::vector<uint32_t> idx(n_irr);
    CU(cudaMemcpy(idx.data(), d + o_irr, n_irr * 4, cudaMemcpyDeviceToHost));
    for (uint32_t i : idx) {
      int len = (int)(off[i + 1] - off[i]);
      uint64_t w[18];
      int cut = mg::canonical_ascii(reinterpret_cast<const uint8_t *>(pool) + off[i], len, w);
      c->irregular_ref[std::string(reinterpret_cast<const char *>(w), (size_t)cut)] = 0;
    }
  }
  return check_too_long(c);
}

extern "C" int mg_add_signatures_packed(mg_ctx *c, const uint64_t *lohi, const uint8_t *is_ref, uint64_t n) {
  if (!c || ((!lohi || !is_ref) && n)) return set_err(MG_ERR_ARG, "NULL argument");
  if (c->alt_final) return set_err(MG_ERR_STATE, "mg_add_signatures_packed after mg_finalize_alt");
  if (n == 0) return MG_OK;
  if (n > 0xFFFFFFFFull) return set_err(MG_ERR_ARG, "batch too large (max 2^32-1 k-mers per call)");
  CU(cudaSetDevice(c->device));
  const uint64_t o_k = 0, o_f = al256(n * 16), o_spill = o_f + al256(n), total = o_spill + al256(n * 4);
  uint8_t *d = nullptr;
  int rc = add_arena(c, total, &d);
  if (rc) return rc;
  cudaStream_t st = c->stream[0];
  CU(cudaMemcpyAsync(d + o_k, lohi, n * 16, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_f, is_ref, n, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(c->d_scalars, 0, 8 * sizeof(unsigned long long), st));
  c->launches++;
  mg::k_add_packed<<<grid_for(n, 256), 256, 0, st>>>((const uint4 *)(d + o_k), d + o_f, n, c->view(), c->occ, c->d_scalars,
                                                     (uint32_t *)(d + o_spill));
  CU(cudaGetLastError());
  return finish_inserts(c, (const uint32_t *)(d + o_spill), nullptr, nullptr, (const uint4 *)(d + o_k), nullptr);
}

static int count_ones(mg_ctx *c, const uint32_t *words, uint64_t n_units, int stride, uint32_t *unit_count,
                      unsigned long long *ones) {
  CU(cudaMemsetAsync(c->d_scalars + 2, 0, 8, c->stream[0]));
  c->launches++;
  mg::k_line_popc<<<grid_for(n_units, 256), 256, 0, c->stream[0]>>>(words, n_units, stride, unit_count, c->d_scalars + 2);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(ones, c->d_scalars + 2, 8, cudaMemcpyDeviceToHost, c->stream[0]));
  CU(cudaStreamSynchronize(c->stream[0]));
  return MG_OK;
}

// exclusive prefix sum of per-line u32 values (n_lines + 1 entries in, n_lines + 1 out)
static int line_scan(mg_ctx *c, uint32_t *d_in, uint32_t *d_out) {
  DevFree tmp;
  size_t tmp_bytes = 0;
  CU(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, d_in, d_out, (int64_t)(c->n_lines + 1), c->stream[0]));
  CU(cudaMalloc(&tmp.p, tmp_bytes ? tmp_bytes : 1));
  CU(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, d_in, d_out, (int64_t)(c->n_lines + 1), c->stream[0]));
  c->launches++;
  CU(cudaStreamSynchronize(c->stream[0]));
  return MG_OK;
}

// The canonical index image (index.cuh): key slots sorted within every line; for the (rare) lines that took more
// than five keys, the five smallest stay in the line and the rest go to the overflow table, which is rebuilt with
// the keys placed in ascending (home slot, key) order.  The handful of crowded lines is fixed up on the host.
static int canonicalize_keys(mg_ctx *c) {
  c->launches++;
  mg::k_sort_line_keys<<<grid_for(c->n_lines, 256), 256, 0, c->stream[0]>>>(c->view());
  CU(cudaGetLastError());
  const uint64_t cap = 1ull << c->ovf_log2;
  const uint64_t hi_mask = mg::key_hi_mask_for(c->k), flag = mg::ovf_flag_for(c->k);
  const u128 empty = {~0ull, hi_mask};
  auto is_empty = [&](const u128 &k) { return k.lo == ~0ull && k.hi == hi_mask; };
  std::vector<u128> ovk;
  if (c->ovf_n) {
    std::vector<u128> raw(cap);
    CU(cudaMemcpyAsync(raw.data(), c->ovf_keys, cap * sizeof(u128), cudaMemcpyDeviceToHost, c->stream[0]));
    CU(cudaStreamSynchronize(c->stream[0]));
    for (auto &k : raw) {
      k.hi &= hi_mask;
      if (!is_empty(k)) ovk.push_back(k);
    }
  }
  auto less = [](const u128 &a, const u128 &b) { return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo); };
  if (!ovk.empty()) {
    // line of every overflow key (same hash, same modulo as the device)
    const uint64_t mask = (c->bf_bits & (c->bf_bits - 1)) == 0 ? c->bf_bits - 1 : 0;
    std::vector<std::pair<uint64_t, u128>> by_line;
    for (const auto &k : ovk) {
      u128 canon;
      uint64_t h = mg::canon_hash_rt(k, c->k, &canon);
      by_line.push_back({(mask ? (h & mask) : (h % c->bf_bits)) >> 8, k});
    }
    std::sort(by_line.begin(), by_line.end(), [&](const auto &a, const auto &b) {
      return a.first < b.first || (a.first == b.first && less(a.second, b.second));
    });
    std::vector<uint64_t> ids;
    for (const auto &e : by_line)
      if (ids.empty() || ids.back() != e.first) ids.push_back(e.first);
    DevFree d_ids, d_keys;
    CU(cudaMalloc(&d_ids.p, ids.size() * 8));
    CU(cudaMalloc(&d_keys.p, ids.size() * mg::LINE_KEYS * 16));
    CU(cudaMemcpyAsync(d_ids.p, ids.data(), ids.size() * 8, cudaMemcpyHostToDevice, c->stream[0]));
    c->launches++;
    mg::k_gather_line_keys<<<grid_for(ids.size() * mg::LINE_KEYS, 256), 256, 0, c->stream[0]>>>(
        c->lines, (const uint64_t *)d_ids.p, ids.size(), (uint4 *)d_keys.p);
    CU(cudaGetLastError());
    std::vector<u128> slots(ids.size() * mg::LINE_KEYS);
    CU(cudaMemcpyAsync(slots.data(), d_keys.p, slots.size() * 16, cudaMemcpyDeviceToHost, c->stream[0]));
    CU(cudaStreamSynchronize(c->stream[0]));
    ovk.clear();
    size_t e = 0;
    for (size_t i = 0; i < ids.size(); ++i) {
      std::vector<u128> all;
      for (int s = 0; s < mg::LINE_KEYS; ++s) {
        u128 k = slots[i * mg::LINE_KEYS + s];
        k.hi &= hi_mask;
        if (!is_empty(k)) all.push_back(k);
      }
      for (; e < by_line.size() && by_line[e].first == ids[i]; ++e) all.push_back(by_line[e].second);
      std::sort(all.begin(), all.end(), less);
      for (size_t s = 0; s < (size_t)mg::LINE_KEYS; ++s) slots[i * mg::LINE_KEYS + s] = s < all.size() ? all[s] : empty;
      slots[i * mg::LINE_KEYS + mg::LINE_KEYS - 1].hi |= flag;  // the overflow flag stays
      if (all.size() > (size_t)mg::LINE_KEYS) ovk.insert(ovk.end(), all.begin() + mg::LINE_KEYS, all.end());
    }
    CU(cudaMemcpyAsync(d_keys.p, slots.data(), slots.size() * 16, cudaMemcpyHostToDevice, c->stream[0]));
    c->launches++;
    mg::k_scatter_line_keys<<<grid_for(ids.size() * mg::LINE_KEYS, 256), 256, 0, c->stream[0]>>>(
        c->lines, (const uint64_t *)d_ids.p, ids.size(), (const uint4 *)d_keys.p);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream[0]));
  }
  // the overflow table in canonical form: capacity from the key count alone, keys placed by linear probing in
  // ascending (home slot, key) order -- the same image whatever the order of the inserts was
  int nl = 10;
  while ((1ull << nl) < 2 * ovk.size()) ++nl;
  const uint64_t ncap = 1ull << nl;
  std::vector<u128> table(ncap, empty);
  {
    std::vector<std::pair<uint64_t, u128>> by_home;
    by_home.reserve(ovk.size());
    for (const auto &k : ovk) by_home.push_back({mg::ovf_home(k, 64 - nl), k});
    std::sort(by_home.begin(), by_home.end(), [&](const auto &a, const auto &b) {
      return a.first < b.first || (a.first == b.first && less(a.second, b.second));
    });
    for (const auto &e : by_home) {
      uint64_t slot = e.first;
      while (!is_empty(table[slot])) slot = (slot + 1) & (ncap - 1);
      table[slot] = e.second;
    }
  }
  u128 *nk = nullptr;
  uint32_t *nc = nullptr;
  CU(cudaMalloc(&nk, ncap * sizeof(u128)));
  CU(cudaMalloc(&nc, ncap * sizeof(uint32_t)));
  CU(cudaMemcpyAsync(nk, table.data(), ncap * sizeof(u128), cudaMemcpyHostToDevice, c->stream[0]));
  CU(cudaMemsetAsync(nc, 0, ncap * sizeof(uint32_t), c->stream[0]));
  CU(cudaStreamSynchronize(c->stream[0]));
  CU(cudaFree(c->ovf_keys));
  CU(cudaFree(c->ovf_counts));
  c->ovf_keys = nk;
  c->ovf_counts = nc;
  c->ovf_log2 = nl;
  c->ovf_n = ovk.size();
  return MG_OK;
}

// Keep the occupancy pre-filter resident in L2 while the probe lines stream through it: a persisting
// access-policy window on both of the context's streams (MG_L2_PERSIST=0 disables it).
static int pin_occ_in_l2(mg_ctx *c) {
  if (!c->occ) return MG_OK;
  if (const char *e = getenv("MG_L2_PERSIST"))
    if (atoi(e) == 0) return MG_OK;
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, c->device));
  size_t bytes = c->n_occ_words * 4;
  if (prop.persistingL2CacheMaxSize <= 0 || prop.accessPolicyMaxWindowSize <= 0) return MG_OK;
  size_t carve = bytes < (size_t)prop.persistingL2CacheMaxSize ? bytes : (size_t)prop.persistingL2CacheMaxSize;
  CU(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve));
  cudaStreamAttrValue attr = {};
  attr.accessPolicyWindow.base_ptr = c->occ;
  attr.accessPolicyWindow.num_bytes = bytes < (size_t)prop.accessPolicyMaxWindowSize ? bytes : (size_t)prop.accessPolicyMaxWindowSize;
  attr.accessPolicyWindow.hitRatio = bytes <= carve ? 1.0f : (float)((double)carve / (double)bytes);
  attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
  attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
  for (int i = 0; i < 2; ++i) CU(cudaStreamSetAttribute(c->stream[i], cudaStreamAttributeAccessPolicyWindow, &attr));
  return MG_OK;
}

extern "C" int mg_finalize_alt(mg_ctx *c) {
  if (!c) return set_err(MG_ERR_ARG, "NULL ctx");
  if (c->alt_final) return MG_OK;
  CU(cudaSetDevice(c->device));
  {
    // switch_mode: ones per line -> exclusive scan -> the rank of every line goes into word 28 of the line itself
    DevFree cnt, rank;
    CU(cudaMalloc(&cnt.p, (c->n_lines + 1) * 4));
    CU(cudaMalloc(&rank.p, (c->n_lines + 1) * 4));
    CU(cudaMemsetAsync((uint32_t *)cnt.p + c->n_lines, 0, 4, c->stream[0]));
    unsigned long long ones = 0;
    int rc = count_ones(c, reinterpret_cast<const uint32_t *>(c->lines), c->n_lines, 32, (uint32_t *)cnt.p, &ones);
    if (rc) return rc;
    if (ones > 0xFFFFFFFFull) return set_err(MG_ERR_ARG, "bf has %llu set bits; the rank directory is 32-bit", ones);
    rc = line_scan(c, (uint32_t *)cnt.p, (uint32_t *)rank.p);
    if (rc) return rc;
    c->launches++;
    mg::k_write_rank<<<grid_for(c->n_lines, 256), 256, 0, c->stream[0]>>>(c->view(), (const uint32_t *)rank.p);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream[0]));
    c->bf_ones = ones;
  }
  CU(cudaMalloc(&c->bf_counts, (c->bf_ones ? c->bf_ones : 1) * 4));
  CU(cudaMemset(c->bf_counts, 0, (c->bf_ones ? c->bf_ones : 1) * 4));
  int rc = canonicalize_keys(c);
  if (rc) return rc;
  c->alt_final = true;
  return pin_occ_in_l2(c);
}

// ---- dense counter image (index.cuh): gather before a reduce / download, scatter after a reduce ----
static int counters_xfer(mg_ctx *c, bool scatter) {
  const uint64_t n_line_keys = c->n_keys - c->ovf_n;
  if (!c->key_rank) {  // keys held by the lines before each line: built once, on first use
    DevFree cnt;
    CU(cudaMalloc(&cnt.p, (c->n_lines + 1) * 4));
    CU(cudaMalloc(&c->key_rank, (c->n_lines + 1) * 4));
    CU(cudaMemsetAsync((uint32_t *)cnt.p + c->n_lines, 0, 4, c->stream[0]));
    c->launches++;
    mg::k_line_keycount<<<grid_for(c->n_lines, 256), 256, 0, c->stream[0]>>>(c->view(), (uint32_t *)cnt.p);
    CU(cudaGetLastError());
    int rc = line_scan(c, (uint32_t *)cnt.p, c->key_rank);
    if (rc) return rc;
    CU(cudaMalloc(&c->key_dense, (n_line_keys ? n_line_keys : 1) * 4));
    CU(cudaMemsetAsync(c->key_dense, 0, (n_line_keys ? n_line_keys : 1) * 4, c->stream[0]));
  }
  c->launches++;
  const int grid = grid_for(c->n_lines * 8, 256);
  if (scatter)
    mg::k_counters_xfer<true><<<grid, 256, 0, c->stream[0]>>>(c->view(), c->key_rank, c->key_dense);
  else
    mg::k_counters_xfer<false><<<grid, 256, 0, c->stream[0]>>>(c->view(), c->key_rank, c->key_dense);
  CU(cudaGetLastError());
  return MG_OK;
}
extern "C" int mg_counters_gather(mg_ctx *c) {
  if (!c) return set_err(MG_ERR_ARG, "NULL ctx");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "no counters before mg_finalize_alt");
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  rc = counters_xfer(c, false);
  if (rc) return rc;
  CU(cudaStreamSynchronize(c->stream[0]));
  return MG_OK;
}
extern "C" int mg_counters_scatter(mg_ctx *c) {
  if (!c) return set_err(MG_ERR_ARG, "NULL ctx");
  if (!c->key_rank) return set_err(MG_ERR_STATE, "mg_counters_scatter before mg_counters_gather");
  CU(cudaSetDevice(c->device));
  int rc = counters_xfer(c, true);
  if (rc) return rc;
  CU(cudaStreamSynchronize(c->stream[0]));
  return MG_OK;
}

template <int K, int REFK>
static cudaError_t launch_refpass(mg_ctx *c, const uint8_t *d_chunk, uint64_t chunk_base, uint64_t p_begin, uint64_t p_end) {
  int grid = (int)((p_end - p_begin + mg::RP_TILE - 1) / mg::RP_TILE);
  size_t smem = mg::RP_TILE + 64 + 16;
  c->launches++;
  mg::k_refpass<K, REFK><<<grid, mg::RP_THREADS, smem, c->stream[0]>>>(d_chunk, chunk_base, p_begin, p_end, c->view(),
                                                                        c->ctx_words);
  return cudaGetLastError();
}

// The contig goes to the device in chunks, each carrying the ref_k-1 bytes before its first window end (halo):
// the H2D copy of chunk i+1 (stream 1) overlaps the kernel of chunk i (stream 0).  A caller buffer in pinned memory
// (mg_host_alloc) is copied from directly; pageable memory goes through two pinned staging buffers, filled by
// several host threads (one thread moves ~8 GB/s, the link takes ~50).
// (tests/test_gpu_scale.py plants input at the seams of this size and fails if it changes)
constexpr uint64_t REF_CHUNK = 32ull << 20;  // window end positions per chunk (a multiple of RP_TILE)

static void parallel_memcpy(void *dst, const void *src, size_t n) {
  unsigned t = std::thread::hardware_concurrency();
  t = t > 8 ? 8 : (t < 1 ? 1 : t);
  if (n < (4u << 20) || t == 1) {
    memcpy(dst, src, n);
    return;
  }
  const size_t part = ((n + t - 1) / t + 4095) & ~(size_t)4095;
  std::vector<std::thread> pool;
  for (unsigned i = 1; i < t; ++i) {
    const size_t o = (size_t)i * part;
    if (o >= n) break;
    pool.emplace_back([=] { memcpy((char *)dst + o, (const char *)src + o, std::min(part, n - o)); });
  }
  memcpy(dst, src, std::min(part, n));
  for (auto &th : pool) th.join();
}

extern "C" int mg_scan_reference(mg_ctx *c, const char *seq, uint64_t len) {
  if (!c || (!seq && len)) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "mg_scan_reference before mg_finalize_alt");
  if (c->ctx_final) return set_err(MG_ERR_STATE, "mg_scan_reference after mg_finalize_context");
  CU(cudaSetDevice(c->device));
  int d = (c->ref_k - c->k) / 2;
  cudaStream_t st = c->stream[0], cp = c->stream[1];
  if (len < (uint64_t)c->ref_k) {
    // the reference's substr(d, k) throws when d > size(); a shorter contig is hashed once, truncated
    if ((uint64_t)d > len || len == 0)
      return set_err(MG_ERR_ARG, "contig shorter than (ref_k-k)/2: the reference aborts here");
    DevFree ds;
    CU(cudaMalloc(&ds.p, len));
    CU(cudaMemcpyAsync(ds.p, seq, len, cudaMemcpyHostToDevice, st));
    c->launches++;
    mg::k_refpass_short<<<1, 32, 0, st>>>((const uint8_t *)ds.p, len, c->view(), c->ctx_words);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
    return MG_OK;
  }
  bool pinned_src = false;
  {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, seq) == cudaSuccess)
      pinned_src = at.type == cudaMemoryTypeHost;
    else
      cudaGetLastError();
  }
  const uint64_t halo = (uint64_t)(c->ref_k - 1), buf_bytes = REF_CHUNK + halo + 64;
  for (int i = 0; i < 2; ++i) {
    if (!c->ref_dev[i]) {
      CU(cudaMalloc((void **)&c->ref_dev[i], buf_bytes));
      CU(cudaEventCreateWithFlags(&c->ref_ev[i], cudaEventDisableTiming));
      CU(cudaEventCreateWithFlags(&c->ref_kev[i], cudaEventDisableTiming));
    }
    if (!pinned_src && !c->ref_pinned[i]) CU(cudaHostAlloc((void **)&c->ref_pinned[i], buf_bytes, cudaHostAllocDefault));
  }
  // window end positions p in [ref_k-1, len); chunk j covers [ref_k-1 + j*REF_CHUNK, +REF_CHUNK) and needs the
  // contig bytes [j*REF_CHUNK, (j+1)*REF_CHUNK + halo)
  int slot = 0;
  size_t n_chunks = 0;
  for (uint64_t b0 = 0; b0 + halo < len; b0 += REF_CHUNK, slot ^= 1, ++n_chunks) {
    const uint64_t nbytes = std::min<uint64_t>(REF_CHUNK + halo, len - b0);
    const char *src = seq + b0;
    if (!pinned_src) {
      CU(cudaEventSynchronize(c->ref_ev[slot]));  // the H2D copy that last read this staging buffer is done
      parallel_memcpy(c->ref_pinned[slot], seq + b0, nbytes);
      src = reinterpret_cast<const char *>(c->ref_pinned[slot]);
    }
    CU(cudaStreamWaitEvent(cp, c->ref_kev[slot], 0));  // the kernel that last read this device buffer is done
    CU(cudaMemcpyAsync(c->ref_dev[slot], src, nbytes, cudaMemcpyHostToDevice, cp));
    CU(cudaEventRecord(c->ref_ev[slot], cp));
    CU(cudaStreamWaitEvent(st, c->ref_ev[slot], 0));
    while (c->rp_events.size() < 2 * (n_chunks + 1)) {
      cudaEvent_t e;
      CU(cudaEventCreate(&e));
      c->rp_events.push_back(e);
    }
    CU(cudaEventRecord(c->rp_events[2 * n_chunks], st));
    const uint64_t p_begin = b0 + halo, p_end = b0 + nbytes;
    cudaError_t e;
    if (c->k == 35 && c->ref_k == 43)
      e = launch_refpass<35, 43>(c, c->ref_dev[slot], b0, p_begin, p_end);
    else
      e = launch_refpass<0, 0>(c, c->ref_dev[slot], b0, p_begin, p_end);
    if (e != cudaSuccess) return set_err(MG_ERR_CUDA, "k_refpass launch -> %s", cudaGetErrorString(e));
    CU(cudaEventRecord(c->rp_events[2 * n_chunks + 1], st));
    CU(cudaEventRecord(c->ref_kev[slot], st));
  }
  c->rp_chunks = n_chunks;
  CU(cudaStreamSynchronize(st));
  CU(cudaStreamSynchronize(cp));
  return MG_OK;
}

extern "C" int mg_finalize_context(mg_ctx *c) {
  if (!c) return set_err(MG_ERR_ARG, "NULL ctx");
  c->ctx_final = true;  // context_bf is only ever test_key()'d after this point: no rank/counters needed
  return MG_OK;
}

template <int K, int REFK, int MODE, int THREADS, bool RING, bool ASYNC, int ILP = 1, int LD = 0>
static cudaError_t launch_scan(mg_ctx *c, const mg::ScanSrc &src_in, uint64_t n, cudaStream_t st) {
  constexpr int WARPS = THREADS / 32;
  uint64_t want = (n + THREADS * ILP - 1) / (THREADS * ILP);  // one warp per 32 (64) k-mers
  int per_sm = c->scan_ctas_per_sm;
  if (const char *ev = getenv("MG_SCAN_CTAS_PER_SM")) per_sm = atoi(ev) > 0 ? atoi(ev) : per_sm;  // (sweeps: read per launch)
  uint64_t cap = (uint64_t)c->sms * (uint64_t)per_sm * (256 / THREADS);
  int grid = (int)(want < cap ? want : cap);
  if (grid < 1) grid = 1;
  mg::ScanSrc src = src_in;
  const int si = st == c->stream[1] ? 1 : 0;
  const uint64_t n_warps = (uint64_t)grid * WARPS;
  if (c->defer_hits) {
    // a segment per warp of the grid, sized for one k-mer in 32 hitting the filter (expected: < 1 in 100; whatever
    // exceeds a segment is finished in line by the scan itself)
    const uint64_t per_warp = ((n + n_warps * 32 - 1) / (n_warps * 32)) * 32;
    const uint64_t seg = per_warp / 32 > 8 ? per_warp / 32 : 8;
    if (c->hit_entries[si] < n_warps * seg) {
      cudaFree(c->hit_buf[si]);
      c->hit_buf[si] = nullptr;
      c->hit_entries[si] = 0;
      cudaError_t e = cudaMalloc(&c->hit_buf[si], n_warps * seg * 32);
      if (e != cudaSuccess) return e;
      c->hit_entries[si] = n_warps * seg;
    }
    if (c->hit_warps[si] < n_warps) {
      cudaFree(c->hit_counts[si]);
      c->hit_counts[si] = nullptr;
      c->hit_warps[si] = 0;
      cudaError_t e = cudaMalloc(&c->hit_counts[si], n_warps * 4);
      if (e != cudaSuccess) return e;
      c->hit_warps[si] = n_warps;
    }
    src.hit_buf = c->hit_buf[si];
    src.hit_counts = c->hit_counts[si];
    src.seg_cap = (uint32_t)seg;
  }
  constexpr int SMEM = mg::scan_smem(THREADS, ASYNC, ILP, mg::scan_occs(LD, ASYNC, ILP));
  if (SMEM > 48 * 1024) {  // more than 48 KB of dynamic shared memory needs the opt-in (per device; cheap enough to repeat)
    cudaError_t e = cudaFuncSetAttribute(mg::k_scan<K, REFK, MODE, THREADS, RING, ASYNC, ILP, LD>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
    if (e != cudaSuccess) return e;
  }
  if (LD == 2 && !getenv("MG_SCAN_CARVEOUT")) {  // nothing of this build's traffic needs L1: all of it to shared memory
    cudaError_t e = cudaFuncSetAttribute(mg::k_scan<K, REFK, MODE, THREADS, RING, ASYNC, ILP, LD>,
                                         cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e != cudaSuccess) return e;
  }
  if (const char *ev = getenv("MG_SCAN_CARVEOUT")) {  // (sweeps) shared-memory share of the unified L1, percent
    cudaError_t e = cudaFuncSetAttribute(mg::k_scan<K, REFK, MODE, THREADS, RING, ASYNC, ILP, LD>,
                                         cudaFuncAttributePreferredSharedMemoryCarveout, atoi(ev));
    if (e != cudaSuccess) return e;
    int nb = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, mg::k_scan<K, REFK, MODE, THREADS, RING, ASYNC, ILP, LD>, THREADS, SMEM);
    static int said = -1;
    if (said != atoi(ev) * 1000 + THREADS) {
      said = atoi(ev) * 1000 + THREADS;
      fprintf(stderr, "[k_scan] carveout %d %%: %d CTAs of %d threads per SM, %d B of shared memory each\n", atoi(ev), nb, THREADS, SMEM);
    }
  }
  c->launches++;
  mg::k_scan<K, REFK, MODE, THREADS, RING, ASYNC, ILP, LD><<<grid, THREADS, SMEM, st>>>(src, n, c->view());
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || !src.hit_buf) return e;
  const uint64_t threads = n_warps * src.seg_cap;
  c->launches++;
  mg::k_scan_hits<REFK><<<grid_for(threads, 256), 256, 0, st>>>(src.hit_buf, src.hit_counts, (uint32_t)n_warps, src.seg_cap,
                                                               c->view());
  return cudaGetLastError();
}

template <int MODE>
static int scan_src(mg_ctx *c, const mg::ScanSrc &src, uint64_t n, cudaStream_t st) {
  cudaError_t e;
  if (c->k == 35 && c->ref_k == 43) {
    // MG_SCAN_VARIANT (tuning sweeps, profiles/sweep_k1_r2.py): the schemes tried for the packed-input scan.
    // Default = 0: two k-mers per lane, asynchronous probe rounds, 256-thread CTAs, pre-filter pieces through
    // cp.async (profiles/round2_k1.md).
    int variant = 0;
    if (MODE == 0)
      if (const char *ev = getenv("MG_SCAN_VARIANT")) variant = atoi(ev);
    if (MODE == 0 && variant == 1)
      e = launch_scan<35, 43, 0, 256, true, false>(c, src, n, st);     // one k-mer per lane, synchronous rounds
    else if (MODE == 0 && variant == 2)
      e = launch_scan<35, 43, 0, 256, false, false>(c, src, n, st);    // probe after every batch (the round-1 scheme)
    else if (MODE == 0 && variant == 3)
      e = launch_scan<35, 43, 0, 256, true, true>(c, src, n, st);      // one k-mer per lane, asynchronous rounds
    else if (MODE == 0 && variant == 4)
      e = launch_scan<35, 43, 0, 256, true, false, 2>(c, src, n, st);  // two k-mers per lane, synchronous rounds
    else if (MODE == 0 && variant == 5)
      e = launch_scan<35, 43, 0, 128, true, false, 2>(c, src, n, st);
    else if (MODE == 0 && variant == 6)
      e = launch_scan<35, 43, 0, 128, true, true, 2>(c, src, n, st);   // two k-mers per lane, asynchronous rounds, 128
    else if (MODE == 0 && variant == 7)
      e = launch_scan<35, 43, 0, 256, true, true, 2>(c, src, n, st);     // the default, all loads through L1
    else if (MODE == 0 && variant == 8)
      e = launch_scan<35, 43, 0, 256, true, true, 2, 1>(c, src, n, st);  // the default, loads that do not allocate in L1
    else if (MODE == 0 && variant == 9)
      e = launch_scan<35, 43, 0, 128, true, true, 2, 2>(c, src, n, st);  // the default with 128-thread CTAs
    else if (MODE == 0 && variant == 10)
      e = launch_scan<35, 43, 0, 256, true, false, 1, 2>(c, src, n, st);  // one k-mer per lane, 4 CTAs (32 warps) per SM
    else if (MODE == 0 && variant == 11)
      e = launch_scan<35, 43, 0, 256, true, false, 2, 2>(c, src, n, st);  // two per lane, synchronous, 4 CTAs per SM
    else if (MODE == 0 && variant == 12)
      e = launch_scan<35, 43, 0, 128, true, true, 3, 2>(c, src, n, st);   // three k-mers per lane, 5 CTAs of 128
    else if (MODE == 0 && variant == 13)
      e = launch_scan<35, 43, 0, 128, true, true, 4, 2>(c, src, n, st);   // four k-mers per lane, 4 CTAs of 128
    else if (MODE == 0 && variant == 14)
      e = launch_scan<35, 43, 0, 256, true, true, 3, 2>(c, src, n, st);   // three k-mers per lane, 2 CTAs of 256
    else if (MODE == 0)
      e = launch_scan<35, 43, 0, 256, true, true, 2, 2>(c, src, n, st);
    else
      e = launch_scan<35, 43, MODE, 256, true, false, 1, 2>(c, src, n, st);
  } else {
    if (MODE == 0)
      e = launch_scan<0, 0, 0, 256, true, true, 2, 2>(c, src, n, st);
    else
      e = launch_scan<0, 0, MODE, 256, true, false, 1, 2>(c, src, n, st);
  }
  if (e != cudaSuccess) return set_err(MG_ERR_CUDA, "k_scan launch -> %s", cudaGetErrorString(e));
  return MG_OK;
}

static int scan_device(mg_ctx *c, const void *d_lohi, const void *d_counts, uint64_t n, cudaStream_t st) {
  const uint64_t MAX_LAUNCH = 1ull << 30;  // the kernel indexes k-mers with 32 bits
  for (uint64_t o = 0; o < n; o += MAX_LAUNCH) {
    mg::ScanSrc src = {};
    src.kmers = reinterpret_cast<const uint4 *>(d_lohi) + o;
    src.counts = reinterpret_cast<const uint32_t *>(d_counts) + o;
    int rc = scan_src<0>(c, src, n - o < MAX_LAUNCH ? n - o : MAX_LAUNCH, st);
    if (rc) return rc;
  }
  return MG_OK;
}

extern "C" int mg_scan_sample_kmers_device(mg_ctx *c, const void *d_lohi, const void *d_counts, uint64_t n) {
  if (!c || ((!d_lohi || !d_counts) && n)) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "scan before mg_finalize_alt (BF::increment is a no-op in write mode)");
  if (n == 0) return MG_OK;
  CU(cudaSetDevice(c->device));
  return scan_device(c, d_lohi, d_counts, n, c->stream[0]);
}

// the two device staging buffers of the host-buffer scans, sized for `unit` bytes per k-mer (a packed word, or a
// KMC record of any suffix + counter length)
static int stage_reserve(mg_ctx *c, uint64_t unit) {
  if (unit < 16) unit = 16;
  if (c->stage_unit >= unit) return MG_OK;
  int rc = mg_sync(c);
  if (rc) return rc;
  for (int i = 0; i < 2; ++i) {
    cudaFree(c->d_stage_k[i]);
    c->d_stage_k[i] = nullptr;
    if (!c->d_stage_c[i]) CU(cudaMalloc(&c->d_stage_c[i], STAGE_KMERS * 4));
    CU(cudaMalloc(&c->d_stage_k[i], STAGE_KMERS * unit + 64));
  }
  c->stage_unit = unit;
  return MG_OK;
}

extern "C" int mg_scan_sample_kmers(mg_ctx *c, const uint64_t *lohi, const uint32_t *counts, uint64_t n) {
  if (!c || ((!lohi || !counts) && n)) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "scan before mg_finalize_alt (BF::increment is a no-op in write mode)");
  CU(cudaSetDevice(c->device));
  int rc0 = stage_reserve(c, 16);
  if (rc0) return rc0;
  // chunks alternate between two (stream, device buffer) pairs: the H2D copy of chunk i+1 overlaps the
  // kernel of chunk i.
  for (uint64_t o = 0; o < n; o += STAGE_KMERS) {
    uint64_t m = n - o < STAGE_KMERS ? n - o : STAGE_KMERS;
    int s = c->next_stage;
    c->next_stage ^= 1;
    CU(cudaMemcpyAsync(c->d_stage_k[s], lohi + 2 * o, m * 16, cudaMemcpyHostToDevice, c->stream[s]));
    CU(cudaMemcpyAsync(c->d_stage_c[s], counts + o, m * 4, cudaMemcpyHostToDevice, c->stream[s]));
    int rc = scan_device(c, c->d_stage_k[s], c->d_stage_c[s], m, c->stream[s]);
    if (rc) return rc;
  }
  return MG_OK;
}

// ---- KMC database ingestion without a host-side decode (call sites main.cpp:482-490) ----
extern "C" int mg_kmc_open(mg_ctx *c, const uint64_t *lut, uint64_t n_lut, uint32_t lut_prefix_len, uint32_t kmer_len,
                           uint32_t counter_size, uint32_t min_count, uint64_t max_count) {
  if (!c || !lut || n_lut == 0) return set_err(MG_ERR_ARG, "NULL argument");
  if ((int)kmer_len != c->ref_k)
    return set_err(MG_ERR_ARG, "KMC database holds %u-mers but ref_k is %d (the reference would overrun its buffer)",
                   kmer_len, c->ref_k);
  if (lut_prefix_len > 15 || lut_prefix_len >= kmer_len || (kmer_len - lut_prefix_len) % 4 != 0 || counter_size > 8)
    return set_err(MG_ERR_ARG, "unsupported KMC layout (prefix %u, counter %u bytes)", lut_prefix_len, counter_size);
  if (n_lut % (1ull << (2 * lut_prefix_len)) != 0 || n_lut > 0x7FFFFFFFull)
    return set_err(MG_ERR_ARG, "LUT size %llu is not a multiple of 4^%u", (unsigned long long)n_lut, lut_prefix_len);
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  cudaFree(c->kmc_lut);
  c->kmc_lut = nullptr;
  CU(cudaMalloc(&c->kmc_lut, (n_lut + 1) * 8));
  CU(cudaMemcpy(c->kmc_lut, lut, n_lut * 8, cudaMemcpyHostToDevice));
  CU(cudaMemset(c->kmc_lut + n_lut, 0xFF, 8));
  c->kmc_n_lut = (uint32_t)n_lut;
  c->kmc_prefix_len = (int)lut_prefix_len;
  c->kmc_suf_bytes = (int)((kmer_len - lut_prefix_len) / 4);
  c->kmc_counter_size = (int)counter_size;
  c->kmc_min = min_count;
  c->kmc_max = max_count;
  return MG_OK;
}

extern "C" int mg_scan_kmc_records(mg_ctx *c, const uint8_t *records, uint64_t first_record, uint64_t n) {
  if (!c || (!records && n)) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->kmc_lut) return set_err(MG_ERR_STATE, "mg_scan_kmc_records before mg_kmc_open");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "scan before mg_finalize_alt (BF::increment is a no-op in write mode)");
  CU(cudaSetDevice(c->device));
  const uint64_t rec = (uint64_t)(c->kmc_suf_bytes + c->kmc_counter_size);
  int rc0 = stage_reserve(c, rec);
  if (rc0) return rc0;
  for (uint64_t o = 0; o < n; o += STAGE_KMERS) {
    uint64_t m = n - o < STAGE_KMERS ? n - o : STAGE_KMERS;
    int s = c->next_stage;
    c->next_stage ^= 1;
    CU(cudaMemcpyAsync(c->d_stage_k[s], records + o * rec, m * rec, cudaMemcpyHostToDevice, c->stream[s]));
    mg::ScanSrc src = {};
    src.recs = reinterpret_cast<const uint8_t *>(c->d_stage_k[s]);
    src.lut = c->kmc_lut;
    src.first_rec = first_record + o;
    src.n_lut = c->kmc_n_lut;
    src.prefix_mask = (uint32_t)((1ull << (2 * c->kmc_prefix_len)) - 1);
    src.prefix_len = c->kmc_prefix_len;
    src.suf_bytes = c->kmc_suf_bytes;
    src.counter_size = c->kmc_counter_size;
    src.min_count = c->kmc_min;
    src.max_count = c->kmc_max;
    int rc = scan_src<1>(c, src, m, c->stream[s]);
    if (rc) return rc;
  }
  return MG_OK;
}

extern "C" int mg_sync(mg_ctx *c) {
  if (!c) return set_err(MG_ERR_ARG, "NULL ctx");
  CU(cudaSetDevice(c->device));
  CU(cudaStreamSynchronize(c->stream[0]));
  CU(cudaStreamSynchronize(c->stream[1]));
  return MG_OK;
}

static int lookup_common(mg_ctx *c, const char *pool, const uint64_t *off, const uint8_t *is_ref, uint64_t n,
                         int mode, int which, int32_t *out_host) {
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  DevBatch b;
  rc = upload_batch(c, b, pool, off, is_ref, n);
  if (rc) return rc;
  DevFree d_out;
  CU(cudaMalloc(&d_out.p, (n ? n : 1) * 4));
  c->launches++;
  mg::k_lookup<<<grid_for(n, 128), 128, 0, c->stream[0]>>>(b.pool, b.off, b.flags, n, c->view(), mode, which,
                                                           (int32_t *)d_out.p, c->d_scalars, nullptr, nullptr, nullptr);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out_host, d_out.p, n * 4, cudaMemcpyDeviceToHost, c->stream[0]));
  CU(cudaStreamSynchronize(c->stream[0]));
  return check_too_long(c);
}

extern "C" int mg_test_keys(mg_ctx *c, int which, const char *pool, const uint64_t *off, uint64_t n, uint8_t *out) {
  if (!c || !off || !out || which < 0 || which > 2) return set_err(MG_ERR_ARG, "bad argument");
  if (n == 0) return MG_OK;
  std::vector<int32_t> tmp(n);
  int rc = lookup_common(c, pool, off, nullptr, n, 1, which, tmp.data());
  if (rc) return rc;
  for (uint64_t i = 0; i < n; ++i) {
    if (tmp[i] < 0) {  // irregular KMAP key: host-side set
      int len = (int)(off[i + 1] - off[i]);
      uint64_t w[18];
      int cut = mg::canonical_ascii(reinterpret_cast<const uint8_t *>(pool) + off[i], len, w);
      out[i] = c->irregular_ref.count(std::string(reinterpret_cast<const char *>(w), (size_t)cut)) ? 1 : 0;
    } else {
      out[i] = (uint8_t)tmp[i];
    }
  }
  return MG_OK;
}

extern "C" int mg_get_counts(mg_ctx *c, const char *pool, const uint64_t *off, const uint8_t *is_ref, uint64_t n,
                             int32_t *out) {
  if (!c || !off || !is_ref || !out) return set_err(MG_ERR_ARG, "NULL argument");
  if (n == 0) return MG_OK;
  return lookup_common(c, pool, off, is_ref, n, 0, 0, out);
}

// library-owned scratch of the genotyping calls: per-k-mer weights (+ flags), and the likelihood slots nobody reads
static int geno_scratch(mg_ctx *c, uint64_t need) {
  if (c->geno_scratch_bytes < need) {
    CU(cudaStreamSynchronize(c->stream[0]));
    cudaFree(c->geno_scratch);
    c->geno_scratch = nullptr;
    c->geno_scratch_bytes = 0;
    CU(cudaMalloc(&c->geno_scratch, need + need / 4));
    c->geno_scratch_bytes = need + need / 4;
  }
  return MG_OK;
}
// everything enqueued on the second stream (host-path scans) precedes what stream 0 does next
static int join_streams(mg_ctx *c) {
  if (!c->tj) CU(cudaEventCreateWithFlags(&c->tj, cudaEventDisableTiming));
  CU(cudaEventRecord(c->tj, c->stream[1]));
  CU(cudaStreamWaitEvent(c->stream[0], c->tj, 0));
  return MG_OK;
}

// all pointers of in/out are DEVICE pointers here; scratch (k-mer flags + weights) is library-owned
static int genotype_on_device(mg_ctx *c, const mg_variant_batch *in, const mg_genotype_out *out,
                              const mg_batch_dims *dm, float error_rate, int max_coverage, int haploid) {
  cudaStream_t st = c->stream[0];
  uint64_t nv = dm->n_variants, na = dm->n_alleles, nk = dm->n_kmers;
  int rc = geno_scratch(c, (nk ? nk : 1) * 6);  // i32 weight + ref flag + deferred flag per k-mer
  if (rc) return rc;
  rc = join_streams(c);
  if (rc) return rc;
  int32_t *d_w = reinterpret_cast<int32_t *>(c->geno_scratch);
  uint8_t *d_flags = reinterpret_cast<uint8_t *>(c->geno_scratch) + (nk ? nk : 1) * 4;
  for (int i = 0; i < 5; ++i)
    if (!c->ge[i]) CU(cudaEventCreate(&c->ge[i]));
  CU(cudaEventRecord(c->ge[0], st));
  if (nk) {
    CU(cudaMemsetAsync(d_flags, 0, nk, st));
    c->launches++;
    mg::k_mark_ref<<<grid_for(nv, 256), 256, 0, st>>>(in->var_allele_off, in->allele_sig_off, in->sig_kmer_off, nv,
                                                      d_flags);
    CU(cudaGetLastError());
    const uint8_t *d_pool = reinterpret_cast<const uint8_t *>(in->pool);
    if (c->k == 35 && dm->pool_bytes && (reinterpret_cast<uintptr_t>(d_pool) & 3) == 0) {
      // fast path for well-formed 35-mers; whatever it defers (odd lengths, non-ACGT, pool tail) goes through
      // the generic kernel, which is skipped when nothing was deferred
      uint8_t *d_slow = d_flags + nk;
      CU(cudaMemsetAsync(d_slow, 0, nk, st));
      c->launches++;
      mg::k_lookup_fast<35><<<grid_for(nk, 128), 128, 0, st>>>(d_pool, dm->pool_bytes, in->kmer_off, d_flags, nk,
                                                               c->view(), d_w, d_slow);
      CU(cudaGetLastError());
      c->launches++;
      mg::k_lookup<<<grid_for(nk, 128), 128, 0, st>>>(d_pool, in->kmer_off, d_flags, nk, c->view(), 0, 0, d_w,
                                                      c->d_scalars, d_slow, nullptr, nullptr);
      CU(cudaGetLastError());
    } else {
      c->launches++;
      mg::k_lookup<<<grid_for(nk, 128), 128, 0, st>>>(d_pool, in->kmer_off, d_flags, nk, c->view(), 0, 0, d_w,
                                                      c->d_scalars, nullptr, nullptr, nullptr);
      CU(cudaGetLastError());
    }
  }
  CU(cudaEventRecord(c->ge[1], st));
  CU(cudaEventRecord(c->ge[4], st));
  c->launches++;
  mg::k_coverage<uint64_t><<<grid_for(na, 128), 128, 0, st>>>(d_w, in->sig_kmer_off, in->allele_sig_off, na, out->cov);
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->ge[2], st));
  c->launches++;
  mg::k_genotype<uint64_t><<<grid_for(nv, 128), 128, 0, st>>>(out->cov, in->freq, in->var_allele_off, out->lik_off, nullptr,
                                                              nv, error_rate, max_coverage, haploid, c->log_table,
                                                              out->lik, out->n_gts,
                                                              out->status, out->best_gt, out->gq);
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->ge[3], st));
  return MG_OK;
}

extern "C" int mg_genotype_device(mg_ctx *c, const mg_variant_batch *in, const mg_genotype_out *out,
                                  const mg_batch_dims *dims, float error_rate, int max_coverage, int haploid) {
  if (!c || !in || !out || !dims) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "mg_genotype_device before mg_finalize_alt");
  if (dims->n_variants == 0) return MG_OK;
  if (!in->var_allele_off || !in->allele_sig_off || !in->sig_kmer_off || !in->kmer_off || !in->freq || !out->cov ||
      !out->n_gts || !out->status || !out->best_gt || !out->gq || !out->lik_off || !out->lik)
    return set_err(MG_ERR_ARG, "NULL array in batch");
  CU(cudaSetDevice(c->device));
  return genotype_on_device(c, in, out, dims, error_rate, max_coverage, haploid);
}

extern "C" int mg_genotype(mg_ctx *c, const mg_variant_batch *in, const mg_genotype_out *out, float error_rate,
                           int max_coverage, int haploid) {
  if (!c || !in || !out) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "mg_genotype before mg_finalize_alt");
  uint64_t nv = in->n_variants;
  if (nv == 0) return MG_OK;
  if (!in->var_allele_off || !in->allele_sig_off || !in->sig_kmer_off || !in->kmer_off || !in->freq || !out->cov ||
      !out->n_gts || !out->status || !out->best_gt || !out->gq || !out->lik_off)
    return set_err(MG_ERR_ARG, "NULL array in batch");
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  mg_batch_dims dm;
  dm.n_variants = nv;
  dm.n_alleles = in->var_allele_off[nv];
  dm.n_sigs = in->allele_sig_off[dm.n_alleles];
  dm.n_kmers = in->sig_kmer_off[dm.n_sigs];
  dm.pool_bytes = in->kmer_off[dm.n_kmers];
  uint64_t na = dm.n_alleles, ns = dm.n_sigs, nk = dm.n_kmers, nl = out->lik_off[nv];
  uint64_t pool_bytes = in->kmer_off[nk];
  cudaStream_t st = c->stream[0];
  // one device arena for the whole batch
  auto al = [](uint64_t x) { return (x + 255) & ~255ull; };
  uint64_t o_vao = 0, o_aso = o_vao + al((nv + 1) * 8), o_sko = o_aso + al((na + 1) * 8),
           o_ko = o_sko + al((ns + 1) * 8), o_lo = o_ko + al((nk + 1) * 8), o_freq = o_lo + al((nv + 1) * 8),
           o_pool = o_freq + al(na * 4), o_cov = o_pool + al(pool_bytes), o_i32 = o_cov + al(na * 4),
           o_lik = o_i32 + al(nv * 16), total = o_lik + al(nl * 8) + 256;
  if (c->geno_arena_bytes < total) {  // grow-only device arena, reused across calls
    cudaFree(c->geno_arena);
    c->geno_arena = nullptr;
    c->geno_arena_bytes = 0;
    CU(cudaMalloc(&c->geno_arena, total + total / 4));
    c->geno_arena_bytes = total + total / 4;
  }
  uint8_t *d = (uint8_t *)c->geno_arena;
  CU(cudaMemcpyAsync(d + o_vao, in->var_allele_off, (nv + 1) * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_aso, in->allele_sig_off, (na + 1) * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_sko, in->sig_kmer_off, (ns + 1) * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_ko, in->kmer_off, (nk + 1) * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_lo, out->lik_off, (nv + 1) * 8, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_freq, in->freq, na * 4, cudaMemcpyHostToDevice, st));
  if (pool_bytes) CU(cudaMemcpyAsync(d + o_pool, in->pool, pool_bytes, cudaMemcpyHostToDevice, st));
  mg_variant_batch din;
  din.n_variants = nv;
  din.var_allele_off = reinterpret_cast<uint64_t *>(d + o_vao);
  din.allele_sig_off = reinterpret_cast<uint64_t *>(d + o_aso);
  din.sig_kmer_off = reinterpret_cast<uint64_t *>(d + o_sko);
  din.kmer_off = reinterpret_cast<uint64_t *>(d + o_ko);
  din.pool = reinterpret_cast<const char *>(d + o_pool);
  din.freq = reinterpret_cast<float *>(d + o_freq);
  mg_genotype_out dout;
  int32_t *i32 = reinterpret_cast<int32_t *>(d + o_i32);
  dout.cov = reinterpret_cast<uint32_t *>(d + o_cov);
  dout.n_gts = i32;
  dout.status = i32 + nv;
  dout.best_gt = i32 + 2 * nv;
  dout.gq = i32 + 3 * nv;
  dout.lik_off = reinterpret_cast<uint64_t *>(d + o_lo);
  dout.lik = reinterpret_cast<double *>(d + o_lik);
  rc = genotype_on_device(c, &din, &dout, &dm, error_rate, max_coverage, haploid);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out->cov, dout.cov, na * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out->n_gts, dout.n_gts, nv * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out->status, dout.status, nv * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out->best_gt, dout.best_gt, nv * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out->gq, dout.gq, nv * 4, cudaMemcpyDeviceToHost, st));
  if (out->lik && nl) CU(cudaMemcpyAsync(out->lik, dout.lik, nl * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return check_too_long(c);
}

// ---- the same step for PACKED signature k-mers (2-bit words, u32 offsets): what the C++ host sends ----
// all pointers of in/out are DEVICE pointers
// K4 alone: the count of every signature k-mer of the batch into d_w (raw: bf counters unmasked)
static int lookup_packed_on_device(mg_ctx *c, const mg_packed_batch *in, const mg_packed_dims *dm, int32_t *d_w, bool raw) {
  cudaStream_t st = c->stream[0];
  const uint64_t nk = dm->n_kmers;
  if (!nk) return MG_OK;
  c->launches++;
  {
    const uint64_t want = (nk + mg::LOOKUP_THREADS - 1) / mg::LOOKUP_THREADS, cap = (uint64_t)c->sms * 32;
    const int grid = (int)(want < cap ? want : cap);
    const uint4 *km = (const uint4 *)in->kmers;
    if (c->k == 35 && !raw)
      mg::k_lookup_packed<35, false><<<grid, mg::LOOKUP_THREADS, mg::LOOKUP_SMEM, st>>>(km, nk, c->view(), d_w);
    else if (c->k == 35)
      mg::k_lookup_packed<35, true><<<grid, mg::LOOKUP_THREADS, mg::LOOKUP_SMEM, st>>>(km, nk, c->view(), d_w);
    else if (!raw)
      mg::k_lookup_packed<0, false><<<grid, mg::LOOKUP_THREADS, mg::LOOKUP_SMEM, st>>>(km, nk, c->view(), d_w);
    else
      mg::k_lookup_packed<0, true><<<grid, mg::LOOKUP_THREADS, mg::LOOKUP_SMEM, st>>>(km, nk, c->view(), d_w);
  }
  CU(cudaGetLastError());
  if (in->n_irregular) {  // not k symbols of ACGT: the byte-exact path, written to their places in the weight array
    c->launches++;
    mg::k_lookup<<<grid_for(in->n_irregular, 128), 128, 0, st>>>(
        (const uint8_t *)in->irr_pool, in->irr_off, nullptr, in->n_irregular, c->view(), 0, 0, d_w, c->d_scalars, nullptr,
        in->irr_kmer, (const uint4 *)in->kmers, raw);
    CU(cudaGetLastError());
  }
  return MG_OK;
}
// set_coverages + VB::genotype from the weights in d_w; out->lik == NULL: the likelihoods stay in library scratch
static int genotype_from_weights(mg_ctx *c, const mg_packed_batch *in, const mg_genotype_out *out, const mg_packed_dims *dm,
                                 const int32_t *d_w, double *d_lik, float error_rate, int max_coverage, int haploid) {
  cudaStream_t st = c->stream[0];
  const uint64_t nv = dm->n_variants, na = dm->n_alleles;
  const bool own_lik = out->lik == nullptr;
  c->launches++;
  mg::k_coverage<uint32_t><<<grid_for(na, 128), 128, 0, st>>>(d_w, in->sig_kmer_off, in->allele_sig_off, na, out->cov);
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->ge[2], st));
  if (own_lik) CU(cudaMemsetAsync(c->d_scalars + 5, 0, 8, st));
  c->launches++;
  mg::k_genotype<uint32_t><<<grid_for(nv, 128), 128, 0, st>>>(out->cov, in->freq, in->var_allele_off,
                                                              own_lik ? nullptr : out->lik_off, c->d_scalars + 5, nv,
                                                              error_rate, max_coverage, haploid, c->log_table, d_lik,
                                                              out->n_gts,
                                                              out->status, out->best_gt, out->gq);
  CU(cudaGetLastError());
  CU(cudaEventRecord(c->ge[3], st));
  return MG_OK;
}
static int genotype_packed_on_device(mg_ctx *c, const mg_packed_batch *in, const mg_genotype_out *out,
                                     const mg_packed_dims *dm, float error_rate, int max_coverage, int haploid) {
  cudaStream_t st = c->stream[0];
  const uint64_t nk = dm->n_kmers;
  const bool own_lik = out->lik == nullptr;
  const uint64_t w_bytes = ((nk ? nk : 1) * 4 + 255) & ~255ull;
  int rc = geno_scratch(c, w_bytes + (own_lik ? dm->lik_slots * 8 + 256 : 0));
  if (rc) return rc;
  rc = join_streams(c);
  if (rc) return rc;
  int32_t *d_w = reinterpret_cast<int32_t *>(c->geno_scratch);
  double *d_lik = own_lik ? reinterpret_cast<double *>(reinterpret_cast<uint8_t *>(c->geno_scratch) + w_bytes) : out->lik;
  for (int i = 0; i < 5; ++i)
    if (!c->ge[i]) CU(cudaEventCreate(&c->ge[i]));
  CU(cudaEventRecord(c->ge[0], st));
  rc = lookup_packed_on_device(c, in, dm, d_w, false);
  if (rc) return rc;
  CU(cudaEventRecord(c->ge[1], st));
  CU(cudaEventRecord(c->ge[4], st));
  return genotype_from_weights(c, in, out, dm, d_w, d_lik, error_rate, max_coverage, haploid);
}

// ---- the two halves on their own: replicas sum the LOOK-UP RESULTS of a batch instead of their counters ----
// get_count is linear in the counters (bf: the u16 wrap of a sum is the wrap of the sum of the parts; ref_bf: 32-bit
// wrap-around), so N replicas that each scanned a share of the sample stream can each look the batch up in their own
// partial counters, sum the weight vectors (4 bytes per signature k-mer: NCCL, a few tens of MB per batch) and
// genotype from the sum -- no counter array ever travels, and no layout has to agree between the replicas.
extern "C" int mg_lookup_packed_device(mg_ctx *c, const mg_packed_batch *in, const mg_packed_dims *dims, uint32_t *d_weights) {
  if (!c || !in || !dims || (!d_weights && dims->n_kmers)) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "mg_lookup_packed_device before mg_finalize_alt");
  if ((!in->kmers && dims->n_kmers) || (in->n_irregular && (!in->irr_off || !in->irr_pool || !in->irr_kmer)))
    return set_err(MG_ERR_ARG, "NULL array in batch");
  CU(cudaSetDevice(c->device));
  int rc = join_streams(c);
  if (rc) return rc;
  for (int i = 0; i < 5; ++i)
    if (!c->ge[i]) CU(cudaEventCreate(&c->ge[i]));
  CU(cudaEventRecord(c->ge[0], c->stream[0]));
  rc = lookup_packed_on_device(c, in, dims, reinterpret_cast<int32_t *>(d_weights), true);
  if (rc) return rc;
  CU(cudaEventRecord(c->ge[1], c->stream[0]));
  return MG_OK;
}
extern "C" int mg_genotype_weights_device(mg_ctx *c, const mg_packed_batch *in, const mg_genotype_out *out,
                                          const mg_packed_dims *dims, uint32_t *d_weights, float error_rate,
                                          int max_coverage, int haploid) {
  if (!c || !in || !out || !dims || (!d_weights && dims->n_kmers)) return set_err(MG_ERR_ARG, "NULL argument");
  if (dims->n_variants == 0) return MG_OK;
  if (!in->var_allele_off || !in->allele_sig_off || !in->sig_kmer_off || (!in->kmers && dims->n_kmers) || !in->freq ||
      !out->cov || !out->n_gts || !out->status || !out->best_gt || !out->gq || (out->lik && !out->lik_off))
    return set_err(MG_ERR_ARG, "NULL array in batch");
  CU(cudaSetDevice(c->device));
  const bool own_lik = out->lik == nullptr;
  int rc = geno_scratch(c, own_lik ? dims->lik_slots * 8 + 256 : 256);
  if (rc) return rc;
  for (int i = 0; i < 5; ++i)
    if (!c->ge[i]) CU(cudaEventCreate(&c->ge[i]));
  CU(cudaEventRecord(c->ge[4], c->stream[0]));
  if (dims->n_kmers) {  // BF::get_count returns uint16_t: the wrap-around of the summed bf counters
    c->launches++;
    mg::k_mask_alt<<<grid_for(dims->n_kmers, 256), 256, 0, c->stream[0]>>>((const uint4 *)in->kmers, dims->n_kmers,
                                                                            reinterpret_cast<int32_t *>(d_weights));
    CU(cudaGetLastError());
  }
  return genotype_from_weights(c, in, out, dims, reinterpret_cast<const int32_t *>(d_weights),
                               own_lik ? reinterpret_cast<double *>(c->geno_scratch) : out->lik, error_rate, max_coverage,
                               haploid);
}

// The caller's stream (e.g. torch's current stream) in the place of the context's own first stream: library work
// then orders with the caller's kernels and collectives without host synchronisation.  NULL restores the private one.
extern "C" int mg_set_stream(mg_ctx *c, void *cuda_stream) {
  if (!c) return set_err(MG_ERR_ARG, "NULL ctx");
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  if (!c->own_stream0) c->own_stream0 = c->stream[0];
  c->stream[0] = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : c->own_stream0;
  return c->alt_final ? pin_occ_in_l2(c) : MG_OK;  // (the L2 access-policy window is a stream attribute)
}

static uint64_t lik_slots_of(const uint32_t *var_allele_off, uint64_t nv, int haploid) {
  uint64_t t = 0;
  for (uint64_t i = 0; i < nv; ++i) {
    const uint64_t n = var_allele_off[i + 1] - var_allele_off[i];
    t += std::max<uint64_t>(n, haploid ? n : n * (n + 1) / 2);
  }
  return t;
}

extern "C" int mg_genotype_packed_device(mg_ctx *c, const mg_packed_batch *in, const mg_genotype_out *out,
                                         const mg_packed_dims *dims, float error_rate, int max_coverage, int haploid) {
  if (!c || !in || !out || !dims) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "mg_genotype_packed_device before mg_finalize_alt");
  if (dims->n_variants == 0) return MG_OK;
  if (!in->var_allele_off || !in->allele_sig_off || !in->sig_kmer_off || (!in->kmers && dims->n_kmers) || !in->freq ||
      !out->cov || !out->n_gts || !out->status || !out->best_gt || !out->gq || (out->lik && !out->lik_off) ||
      (in->n_irregular && (!in->irr_off || !in->irr_pool || !in->irr_kmer)))
    return set_err(MG_ERR_ARG, "NULL array in batch");
  CU(cudaSetDevice(c->device));
  return genotype_packed_on_device(c, in, out, dims, error_rate, max_coverage, haploid);
}

extern "C" int mg_genotype_packed(mg_ctx *c, const mg_packed_batch *in, const mg_genotype_out *out, float error_rate,
                                  int max_coverage, int haploid) {
  if (!c || !in || !out) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "mg_genotype_packed before mg_finalize_alt");
  const uint64_t nv = in->n_variants;
  if (nv == 0) return MG_OK;
  if (!in->var_allele_off || !in->allele_sig_off || !in->sig_kmer_off || !in->freq || !out->cov || !out->n_gts ||
      !out->status || !out->best_gt || !out->gq || (out->lik && !out->lik_off) ||
      (in->n_irregular && (!in->irr_off || !in->irr_pool || !in->irr_kmer)))
    return set_err(MG_ERR_ARG, "NULL array in batch");
  CU(cudaSetDevice(c->device));
  mg_packed_dims dm;
  dm.n_variants = nv;
  dm.n_alleles = in->var_allele_off[nv];
  dm.n_sigs = in->allele_sig_off[dm.n_alleles];
  dm.n_kmers = in->sig_kmer_off[dm.n_sigs];
  dm.irr_pool_bytes = in->n_irregular ? in->irr_off[in->n_irregular] : 0;
  dm.lik_slots = out->lik ? out->lik_off[nv] : lik_slots_of(in->var_allele_off, nv, haploid);
  if (dm.n_kmers && !in->kmers) return set_err(MG_ERR_ARG, "NULL array in batch");
  const uint64_t na = dm.n_alleles, ns = dm.n_sigs, nk = dm.n_kmers, ni = in->n_irregular, nl = out->lik ? dm.lik_slots : 0;
  cudaStream_t st = c->stream[0];
  auto al = [](uint64_t x) { return (x + 255) & ~255ull; };
  const uint64_t o_vao = 0, o_aso = o_vao + al((nv + 1) * 4), o_sko = o_aso + al((na + 1) * 4),
                 o_km = o_sko + al((ns + 1) * 4), o_freq = o_km + al(nk * 16), o_io = o_freq + al(na * 4),
                 o_ip = o_io + al((ni + 1) * 8), o_ik = o_ip + al(dm.irr_pool_bytes), o_lo = o_ik + al(ni * 4),
                 o_cov = o_lo + al(nl ? (nv + 1) * 8 : 0), o_i32 = o_cov + al(na * 4), o_lik = o_i32 + al(nv * 16),
                 total = o_lik + al(nl * 8) + 256;
  if (c->geno_arena_bytes < total) {  // grow-only device arena, reused across calls
    CU(cudaStreamSynchronize(st));
    cudaFree(c->geno_arena);
    c->geno_arena = nullptr;
    c->geno_arena_bytes = 0;
    CU(cudaMalloc(&c->geno_arena, total + total / 4));
    c->geno_arena_bytes = total + total / 4;
  }
  uint8_t *d = (uint8_t *)c->geno_arena;
  CU(cudaMemcpyAsync(d + o_vao, in->var_allele_off, (nv + 1) * 4, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_aso, in->allele_sig_off, (na + 1) * 4, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_sko, in->sig_kmer_off, (ns + 1) * 4, cudaMemcpyHostToDevice, st));
  if (nk) CU(cudaMemcpyAsync(d + o_km, in->kmers, nk * 16, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d + o_freq, in->freq, na * 4, cudaMemcpyHostToDevice, st));
  if (ni) {
    CU(cudaMemcpyAsync(d + o_io, in->irr_off, (ni + 1) * 8, cudaMemcpyHostToDevice, st));
    if (dm.irr_pool_bytes) CU(cudaMemcpyAsync(d + o_ip, in->irr_pool, dm.irr_pool_bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d + o_ik, in->irr_kmer, ni * 4, cudaMemcpyHostToDevice, st));
  }
  if (nl) CU(cudaMemcpyAsync(d + o_lo, out->lik_off, (nv + 1) * 8, cudaMemcpyHostToDevice, st));
  mg_packed_batch din = {};
  din.n_variants = nv;
  din.var_allele_off = reinterpret_cast<uint32_t *>(d + o_vao);
  din.allele_sig_off = reinterpret_cast<uint32_t *>(d + o_aso);
  din.sig_kmer_off = reinterpret_cast<uint32_t *>(d + o_sko);
  din.kmers = reinterpret_cast<uint64_t *>(d + o_km);
  din.freq = reinterpret_cast<float *>(d + o_freq);
  din.n_irregular = ni;
  din.irr_off = reinterpret_cast<uint64_t *>(d + o_io);
  din.irr_pool = reinterpret_cast<const char *>(d + o_ip);
  din.irr_kmer = reinterpret_cast<uint32_t *>(d + o_ik);
  mg_genotype_out dout;
  int32_t *i32 = reinterpret_cast<int32_t *>(d + o_i32);
  dout.cov = reinterpret_cast<uint32_t *>(d + o_cov);
  dout.n_gts = i32;
  dout.status = i32 + nv;
  dout.best_gt = i32 + 2 * nv;
  dout.gq = i32 + 3 * nv;
  dout.lik_off = nl ? reinterpret_cast<uint64_t *>(d + o_lo) : nullptr;
  dout.lik = nl ? reinterpret_cast<double *>(d + o_lik) : nullptr;
  int rc = genotype_packed_on_device(c, &din, &dout, &dm, error_rate, max_coverage, haploid);
  if (rc) return rc;
  CU(cudaMemcpyAsync(out->cov, dout.cov, na * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out->n_gts, dout.n_gts, nv * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out->status, dout.status, nv * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out->best_gt, dout.best_gt, nv * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(out->gq, dout.gq, nv * 4, cudaMemcpyDeviceToHost, st));
  if (nl) CU(cudaMemcpyAsync(out->lik, dout.lik, nl * 8, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return check_too_long(c);
}

extern "C" int mg_bf_popcount(mg_ctx *c, int which, uint64_t *ones) {
  if (!c || !ones || which < 0 || which > 1) return set_err(MG_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  unsigned long long v = 0;
  if (which == 0)
    rc = count_ones(c, reinterpret_cast<const uint32_t *>(c->lines), c->n_lines, 32, nullptr, &v);
  else
    rc = count_ones(c, c->ctx_words, c->n_lines, 8, nullptr, &v);
  if (rc) return rc;
  *ones = v;
  return MG_OK;
}

extern "C" int mg_bf_download_bits(mg_ctx *c, int which, uint64_t *words, uint64_t n_words) {
  if (!c || !words || which < 0 || which > 1) return set_err(MG_ERR_ARG, "bad argument");
  if (n_words * 2 > c->n_ctx_words) return set_err(MG_ERR_ARG, "n_words exceeds the filter");
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  if (which == 1) {
    CU(cudaMemcpy(words, c->ctx_words, n_words * 8, cudaMemcpyDeviceToHost));
    return MG_OK;
  }
  DevFree tmp;  // gather the 32 filter bytes of every probe line into a plain bit array
  CU(cudaMalloc(&tmp.p, c->n_lines * 32));
  c->launches++;
  mg::k_extract_bits<<<grid_for(c->n_lines * 2, 256), 256, 0, c->stream[0]>>>(c->lines, c->n_lines, (uint4 *)tmp.p);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(words, tmp.p, n_words * 8, cudaMemcpyDeviceToHost, c->stream[0]));
  CU(cudaStreamSynchronize(c->stream[0]));
  return MG_OK;
}

extern "C" int mg_bf_download_counts(mg_ctx *c, uint16_t *counts, uint64_t n) {
  if (!c || (!counts && n)) return set_err(MG_ERR_ARG, "bad argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "no counters before mg_finalize_alt");
  if (n > c->bf_ones) return set_err(MG_ERR_ARG, "n exceeds popcount");
  CU(cudaSetDevice(c->device));
  int rc = mg_counters_gather(c);  // the counters of the first three set bits of a line live inside the line
  if (rc) return rc;
  std::vector<uint32_t> tmp(n ? n : 1);
  CU(cudaMemcpy(tmp.data(), c->bf_counts, n * 4, cudaMemcpyDeviceToHost));
  for (uint64_t i = 0; i < n; ++i) counts[i] = (uint16_t)tmp[i];  // uint16 wrap-around of int_vector<16>
  return MG_OK;
}

extern "C" int mg_kmap_size(mg_ctx *c, uint64_t *n) {
  if (!c || !n) return set_err(MG_ERR_ARG, "bad argument");
  *n = c->n_keys + c->irregular_ref.size();
  return MG_OK;
}

extern "C" int mg_index_stats(mg_ctx *c, uint64_t *stats, int n) {
  if (!c || !stats || n < 6) return set_err(MG_ERR_ARG, "bad argument");
  stats[0] = c->n_lines;
  stats[1] = c->bf_ones;
  stats[2] = c->n_keys;
  stats[3] = c->ovf_n;
  stats[4] = 1ull << c->ovf_log2;
  stats[5] = c->irregular_ref.size();
  return MG_OK;
}

extern "C" int mg_counter_buffers(mg_ctx *c, void **d_ptr, uint64_t *n) {
  if (!c || !d_ptr || !n) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->alt_final) return set_err(MG_ERR_STATE, "no counters before mg_finalize_alt");
  if (!c->key_rank) return set_err(MG_ERR_STATE, "mg_counter_buffers before mg_counters_gather");
  d_ptr[0] = c->bf_counts;
  n[0] = c->bf_ones;
  d_ptr[1] = c->key_dense;
  n[1] = c->n_keys - c->ovf_n;
  d_ptr[2] = c->ovf_counts;
  n[2] = 1ull << c->ovf_log2;
  return MG_OK;
}

// Replicate-and-reduce inside one process (SURVEY 8e-1): ctx[0..n-1] hold the same index (any devices, the same
// device included), each scanned its share of the sample stream.  Every context gathers its counters into the dense
// image; one kernel per array on ctx[0]'s device then reads the peers' arrays in place over NVLink (peer access) and
// adds them N-way into its own -- no staging copies; ctx[0] scatters the sums back into its probe lines.  Exact
// because the index image is canonical (identical layouts) and the updates are modular adds.
extern "C" int mg_reduce_counts(mg_ctx **ctx, int n) {
  if (!ctx || n < 1) return set_err(MG_ERR_ARG, "bad argument");
  if (n > 16) return set_err(MG_ERR_ARG, "at most 16 contexts");
  for (int i = 0; i < n; ++i) {
    if (!ctx[i]) return set_err(MG_ERR_ARG, "NULL context");
    if (!ctx[i]->alt_final) return set_err(MG_ERR_STATE, "mg_reduce_counts before mg_finalize_alt");
    if (ctx[i]->bf_bits != ctx[0]->bf_bits || ctx[i]->bf_ones != ctx[0]->bf_ones || ctx[i]->n_keys != ctx[0]->n_keys ||
        ctx[i]->ovf_n != ctx[0]->ovf_n || ctx[i]->ovf_log2 != ctx[0]->ovf_log2 || ctx[i]->k != ctx[0]->k)
      return set_err(MG_ERR_ARG, "context %d does not hold the same index as context 0", i);
    for (int j = 0; j < i; ++j)
      if (ctx[j] == ctx[i]) return set_err(MG_ERR_ARG, "context %d listed twice", i);
  }
  if (n == 1) return mg_sync(ctx[0]);
  for (int i = 0; i < n; ++i) {  // (asynchronous on every device: the gathers run side by side)
    CU(cudaSetDevice(ctx[i]->device));
    int rc = mg_sync(ctx[i]);
    if (rc) return rc;
    rc = counters_xfer(ctx[i], false);
    if (rc) return rc;
  }
  for (int i = 0; i < n; ++i) {
    CU(cudaSetDevice(ctx[i]->device));
    CU(cudaStreamSynchronize(ctx[i]->stream[0]));
  }
  mg_ctx *c0 = ctx[0];
  CU(cudaSetDevice(c0->device));
  for (int i = 1; i < n; ++i)
    if (ctx[i]->device != c0->device) {
      int can = 0;
      CU(cudaDeviceCanAccessPeer(&can, c0->device, ctx[i]->device));
      if (!can) return set_err(MG_ERR_CUDA, "device %d cannot read device %d's memory", c0->device, ctx[i]->device);
      cudaError_t e = cudaDeviceEnablePeerAccess(ctx[i]->device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
        return set_err(MG_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d) -> %s", ctx[i]->device, cudaGetErrorString(e));
      cudaGetLastError();
    }
  uint32_t *dst[3] = {c0->bf_counts, c0->key_dense, c0->ovf_counts};
  const uint64_t len[3] = {c0->bf_ones, c0->n_keys - c0->ovf_n, 1ull << c0->ovf_log2};
  for (int a = 0; a < 3; ++a) {
    if (!len[a]) continue;
    mg::PeerPtrs pp;
    pp.n = n - 1;
    for (int i = 1; i < n; ++i) pp.p[i - 1] = a == 0 ? ctx[i]->bf_counts : a == 1 ? ctx[i]->key_dense : ctx[i]->ovf_counts;
    const uint64_t want = (len[a] / 4 + 255) / 256 + 1;
    const int grid = (int)std::min<uint64_t>(want, (uint64_t)c0->sms * 16);
    c0->launches++;
    mg::k_sum_peers<<<grid, 256, 0, c0->stream[0]>>>(dst[a], pp, len[a]);
    CU(cudaGetLastError());
  }
  int rc = counters_xfer(c0, true);
  if (rc) return rc;
  CU(cudaStreamSynchronize(c0->stream[0]));
  return MG_OK;
}

// ---- index image export / import ----
extern "C" int mg_export_set_bits(mg_ctx *c, int which, uint64_t *out, uint64_t cap, uint64_t *n) {
  if (!c || !n || which < 0 || which > 1 || (!out && cap)) return set_err(MG_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  const uint32_t *words = which ? c->ctx_words : reinterpret_cast<const uint32_t *>(c->lines);
  const int stride = which ? 8 : 32;
  DevFree cnt, offs, tmp, idx;
  CU(cudaMalloc(&cnt.p, (c->n_lines + 1) * 4));
  CU(cudaMalloc(&offs.p, (c->n_lines + 1) * 4));
  CU(cudaMemsetAsync((uint32_t *)cnt.p + c->n_lines, 0, 4, c->stream[0]));
  unsigned long long ones = 0;
  rc = count_ones(c, words, c->n_lines, stride, (uint32_t *)cnt.p, &ones);
  if (rc) return rc;
  *n = ones;
  if (!out || cap < ones) return ones && out ? set_err(MG_ERR_ARG, "output buffer too small (%llu needed)", ones) : MG_OK;
  if (ones == 0) return MG_OK;
  if (ones > 0xFFFFFFFFull) return set_err(MG_ERR_ARG, "more than 2^32 set bits");
  size_t tb = 0;
  CU(cub::DeviceScan::ExclusiveSum(nullptr, tb, (uint32_t *)cnt.p, (uint32_t *)offs.p, (int64_t)(c->n_lines + 1), c->stream[0]));
  CU(cudaMalloc(&tmp.p, tb ? tb : 1));
  CU(cub::DeviceScan::ExclusiveSum(tmp.p, tb, (uint32_t *)cnt.p, (uint32_t *)offs.p, (int64_t)(c->n_lines + 1), c->stream[0]));
  CU(cudaMalloc(&idx.p, ones * 8));
  c->launches += 2;
  mg::k_emit_bits<<<grid_for(c->n_lines, 256), 256, 0, c->stream[0]>>>(words, c->n_lines, stride, (uint32_t *)offs.p,
                                                                       c->bf_bits, (uint64_t *)idx.p);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(out, idx.p, ones * 8, cudaMemcpyDeviceToHost, c->stream[0]));
  CU(cudaStreamSynchronize(c->stream[0]));
  return MG_OK;
}

extern "C" int mg_import_set_bits(mg_ctx *c, int which, const uint64_t *idx, uint64_t n) {
  if (!c || which < 0 || which > 1 || (!idx && n)) return set_err(MG_ERR_ARG, "bad argument");
  if (which == 0 && c->alt_final) return set_err(MG_ERR_STATE, "bf is already finalized");
  if (n == 0) return MG_OK;
  CU(cudaSetDevice(c->device));
  DevFree d;
  CU(cudaMalloc(&d.p, n * 8));
  CU(cudaMemcpyAsync(d.p, idx, n * 8, cudaMemcpyHostToDevice, c->stream[0]));
  c->launches++;
  mg::k_set_bits<<<grid_for(n, 256), 256, 0, c->stream[0]>>>(
      (const uint64_t *)d.p, n, c->bf_bits, which ? c->ctx_words : reinterpret_cast<uint32_t *>(c->lines), which == 0,
      c->view(), c->occ);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(c->stream[0]));
  return MG_OK;
}

extern "C" int mg_export_ref_keys(mg_ctx *c, uint64_t *lohi, uint64_t cap, uint64_t *n) {
  if (!c || !n || (!lohi && cap)) return set_err(MG_ERR_ARG, "bad argument");
  *n = c->n_keys;
  if (!lohi) return MG_OK;
  if (cap < c->n_keys) return set_err(MG_ERR_ARG, "output buffer too small (%llu needed)", (unsigned long long)c->n_keys);
  if (c->n_keys == 0) return MG_OK;
  CU(cudaSetDevice(c->device));
  int rc = mg_sync(c);
  if (rc) return rc;
  DevFree d;
  CU(cudaMalloc(&d.p, c->n_keys * 16));
  CU(cudaMemsetAsync(c->d_scalars, 0, 8, c->stream[0]));
  uint64_t ovf_cap = 1ull << c->ovf_log2, total = c->n_lines * mg::LINE_KEYS + ovf_cap;
  c->launches++;
  mg::k_emit_keys<<<grid_for(total, 256), 256, 0, c->stream[0]>>>(c->view(), ovf_cap, c->d_scalars, (u128 *)d.p, c->n_keys);
  CU(cudaGetLastError());
  unsigned long long got = 0;
  CU(cudaMemcpyAsync(&got, c->d_scalars, 8, cudaMemcpyDeviceToHost, c->stream[0]));
  CU(cudaMemcpyAsync(lohi, d.p, c->n_keys * 16, cudaMemcpyDeviceToHost, c->stream[0]));
  CU(cudaStreamSynchronize(c->stream[0]));
  if (got != c->n_keys) return set_err(MG_ERR_STATE, "key count mismatch: %llu in the table, %llu recorded", got, (unsigned long long)c->n_keys);
  return MG_OK;
}

// ---------------------------------------------------------------------------
// K6: canonical k-mer counting (the `kmc` step of the pipeline, MALVA:107) -- count.cuh
// ---------------------------------------------------------------------------
struct mg_counter {
  int device = 0, k = 0, log2cap = 0, part_bits = 0;
  uint32_t part_lo = 0, part_hi = 0;
  cudaStream_t st = nullptr;
  mg::CountSlot *table = nullptr;
  unsigned long long *d_scalars = nullptr;  // [0] distinct keys in the table [1] instances counted [2] emit cursor
  uint8_t *d_seq = nullptr;
  uint64_t seq_cap = 0, n_out = 0, launches = 0;
  u128 *out_keys = nullptr;
  uint32_t *out_counts = nullptr;
  bool finished = false;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  double kernel_ms = 0;  // device time of the counting kernels so far
};
constexpr uint64_t COUNT_CHUNK = 1ull << 26;  // read bytes per kernel launch

static int counter_alloc_table(mg_counter *c, int log2cap, mg::CountSlot **t) {
  uint64_t cap = 1ull << log2cap;
  CU(cudaMalloc(t, cap * sizeof(mg::CountSlot)));
  c->launches++;
  mg::k_count_clear<<<grid_for(cap, 256), 256, 0, c->st>>>(*t, cap);
  CU(cudaGetLastError());
  return MG_OK;
}

extern "C" void mg_count_destroy(mg_counter *c);
extern "C" int mg_count_create(mg_counter **out, int device, int k) {
  if (!out) return set_err(MG_ERR_ARG, "out is NULL");
  *out = nullptr;
  if (k < 1 || k > 63) return set_err(MG_ERR_ARG, "unsupported k=%d (need 1 <= k <= 63)", k);
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return set_err(MG_ERR_CUDA, "device %d not available (%d visible)", device, ndev);
  CU(cudaSetDevice(device));
  mg_counter *c = new mg_counter();
  c->device = device;
  c->k = k;
  auto init = [&]() -> int {
    CU(cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking));
    CU(cudaMalloc(&c->d_scalars, 4 * sizeof(unsigned long long)));
    CU(cudaMemsetAsync(c->d_scalars, 0, 4 * sizeof(unsigned long long), c->st));
    c->log2cap = 16;
    int rc = counter_alloc_table(c, c->log2cap, &c->table);
    if (rc) return rc;
    CU(cudaStreamSynchronize(c->st));
    return MG_OK;
  };
  int rc = init();
  if (rc) {
    char msg[sizeof(g_err)];
    memcpy(msg, g_err, sizeof(msg));
    mg_count_destroy(c);
    memcpy(g_err, msg, sizeof(msg));
    return rc;
  }
  *out = c;
  return MG_OK;
}

extern "C" void mg_count_destroy(mg_counter *c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  cudaFree(c->table);
  cudaFree(c->d_scalars);
  cudaFree(c->d_seq);
  cudaFree(c->out_keys);
  cudaFree(c->out_counts);
  for (int i = 0; i < 2; ++i)
    if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  if (c->st) cudaStreamDestroy(c->st);
  delete c;
}

extern "C" int mg_count_set_partition(mg_counter *c, int part_bits, uint32_t part_lo, uint32_t part_hi) {
  if (!c || part_bits < 0 || part_bits > 30 || part_bits > 2 * c->k) return set_err(MG_ERR_ARG, "bad partition");
  c->part_bits = part_bits;
  c->part_lo = part_lo;
  c->part_hi = part_hi;
  return MG_OK;
}

// empty table, same capacity: the next prefix-partitioned pass
extern "C" int mg_count_reset(mg_counter *c) {
  if (!c) return set_err(MG_ERR_ARG, "NULL counter");
  CU(cudaSetDevice(c->device));
  uint64_t cap = 1ull << c->log2cap;
  c->launches++;
  mg::k_count_clear<<<grid_for(cap, 256), 256, 0, c->st>>>(c->table, cap);
  CU(cudaGetLastError());
  CU(cudaMemsetAsync(c->d_scalars, 0, 4 * sizeof(unsigned long long), c->st));
  CU(cudaStreamSynchronize(c->st));
  c->finished = false;
  return MG_OK;
}

static int counter_reserve(mg_counter *c, uint64_t more) {
  unsigned long long nd = 0;
  CU(cudaMemcpyAsync(&nd, c->d_scalars, 8, cudaMemcpyDeviceToHost, c->st));
  CU(cudaStreamSynchronize(c->st));
  uint64_t need = (nd + more) * 2;
  if (need <= (1ull << c->log2cap)) return MG_OK;
  int nl = c->log2cap;
  while ((1ull << nl) < need) ++nl;
  mg::CountSlot *nt = nullptr;
  int rc = counter_alloc_table(c, nl, &nt);
  if (rc) return rc;
  CU(cudaMemsetAsync(c->d_scalars, 0, 8, c->st));
  uint64_t ocap = 1ull << c->log2cap;
  c->launches++;
  mg::k_count_rehash<<<grid_for(ocap, 256), 256, 0, c->st>>>(c->table, ocap, nt, (1ull << nl) - 1, c->d_scalars);
  CU(cudaGetLastError());
  CU(cudaStreamSynchronize(c->st));
  CU(cudaFree(c->table));
  c->table = nt;
  c->log2cap = nl;
  return MG_OK;
}

extern "C" int mg_count_add(mg_counter *c, const char *bases, uint64_t n) {
  if (!c || (!bases && n)) return set_err(MG_ERR_ARG, "NULL argument");
  if (c->finished) return set_err(MG_ERR_STATE, "mg_count_add after mg_count_finish (call mg_count_reset)");
  CU(cudaSetDevice(c->device));
  const uint64_t halo = (uint64_t)(c->k - 1);
  if (n <= halo) return MG_OK;
  if (!c->d_seq) {
    uint64_t cap = COUNT_CHUNK;
    if (const char *e = getenv("MG_COUNT_CHUNK"))  // (tests shrink it to exercise the sub-chunk seams)
      if (strtoull(e, nullptr, 10) > 2 * halo + 1) cap = strtoull(e, nullptr, 10);
    CU(cudaMalloc(&c->d_seq, cap + 64));
    c->seq_cap = cap;
  }
  // sub-chunks overlap by k-1 bytes: a launch counts the windows that END inside its own part
  for (uint64_t start = 0; start + halo < n;) {
    const uint64_t len = n - start < c->seq_cap ? n - start : c->seq_cap;
    int rc = counter_reserve(c, len);
    if (rc) return rc;
    CU(cudaMemcpyAsync(c->d_seq, bases + start, len, cudaMemcpyHostToDevice, c->st));
    const uint64_t n_pos = len - halo;
    const int grid = (int)((n_pos + mg::CNT_TILE - 1) / mg::CNT_TILE);
    const size_t smem = mg::CNT_TILE + 64;
    const uint64_t mask = (1ull << c->log2cap) - 1;
    c->launches++;
    for (int i = 0; i < 2; ++i)
      if (!c->ev[i]) CU(cudaEventCreate(&c->ev[i]));
    CU(cudaEventRecord(c->ev[0], c->st));
    if (c->k == 43)
      mg::k_count_kmers<43><<<grid, mg::CNT_THREADS, smem, c->st>>>(c->d_seq, len, c->k, c->table, mask, c->part_bits,
                                                                    c->part_lo, c->part_hi, c->d_scalars, c->d_scalars + 1);
    else
      mg::k_count_kmers<0><<<grid, mg::CNT_THREADS, smem, c->st>>>(c->d_seq, len, c->k, c->table, mask, c->part_bits,
                                                                   c->part_lo, c->part_hi, c->d_scalars, c->d_scalars + 1);
    CU(cudaGetLastError());
    CU(cudaEventRecord(c->ev[1], c->st));
    CU(cudaStreamSynchronize(c->st));  // d_seq is reused by the next sub-chunk
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]));
    c->kernel_ms += ms;
    if (start + len >= n) break;
    start += len - halo;  // the next part re-sends the last k-1 bytes as its halo
  }
  return MG_OK;
}

extern "C" int mg_count_finish(mg_counter *c, uint32_t min_count, uint32_t counter_max, uint64_t max_count,
                               uint64_t *n_kmers) {
  if (!c) return set_err(MG_ERR_ARG, "NULL counter");
  CU(cudaSetDevice(c->device));
  cudaFree(c->out_keys);
  cudaFree(c->out_counts);
  c->out_keys = nullptr;
  c->out_counts = nullptr;
  c->n_out = 0;
  const uint64_t cap = 1ull << c->log2cap;
  unsigned long long n = 0;
  CU(cudaMemsetAsync(c->d_scalars + 2, 0, 8, c->st));
  c->launches++;
  mg::k_count_emit<<<grid_for(cap, 256), 256, 0, c->st>>>(c->table, cap, min_count, counter_max, max_count,
                                                          c->d_scalars + 2, nullptr, nullptr);
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(&n, c->d_scalars + 2, 8, cudaMemcpyDeviceToHost, c->st));
  CU(cudaStreamSynchronize(c->st));
  if (n) {
    DevFree k0, v0, tmp;
    CU(cudaMalloc(&k0.p, n * 16));
    CU(cudaMalloc(&v0.p, n * 4));
    CU(cudaMalloc(&c->out_keys, n * 16));
    CU(cudaMalloc(&c->out_counts, n * 4));
    CU(cudaMemsetAsync(c->d_scalars + 2, 0, 8, c->st));
    c->launches++;
    mg::k_count_emit<<<grid_for(cap, 256), 256, 0, c->st>>>(c->table, cap, min_count, counter_max, max_count,
                                                            c->d_scalars + 2, (u128 *)k0.p, (uint32_t *)v0.p);
    CU(cudaGetLastError());
    // KMC lists k-mers in ascending order (prefix bins, sorted suffixes): sort the kept entries by key
    size_t tb = 0;
    CU(cub::DeviceRadixSort::SortPairs(nullptr, tb, (u128 *)k0.p, c->out_keys, (uint32_t *)v0.p, c->out_counts, (int64_t)n,
                                       mg::KmerDecomposer{}, 0, 2 * c->k, c->st));
    CU(cudaMalloc(&tmp.p, tb ? tb : 1));
    CU(cub::DeviceRadixSort::SortPairs(tmp.p, tb, (u128 *)k0.p, c->out_keys, (uint32_t *)v0.p, c->out_counts, (int64_t)n,
                                       mg::KmerDecomposer{}, 0, 2 * c->k, c->st));
    c->launches++;
    CU(cudaStreamSynchronize(c->st));
  }
  c->n_out = n;
  c->finished = true;
  if (n_kmers) *n_kmers = n;
  return MG_OK;
}

extern "C" int mg_count_download(mg_counter *c, uint64_t *lohi, uint32_t *counts, uint64_t cap) {
  if (!c || ((!lohi || !counts) && cap)) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->finished) return set_err(MG_ERR_STATE, "mg_count_download before mg_count_finish");
  if (cap < c->n_out) return set_err(MG_ERR_ARG, "output buffers too small (%llu needed)", (unsigned long long)c->n_out);
  if (!c->n_out) return MG_OK;
  CU(cudaSetDevice(c->device));
  CU(cudaMemcpy(lohi, c->out_keys, c->n_out * 16, cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(counts, c->out_counts, c->n_out * 4, cudaMemcpyDeviceToHost));
  return MG_OK;
}

extern "C" int mg_count_stats(mg_counter *c, uint64_t *stats, int n) {
  if (!c || !stats || n < 4) return set_err(MG_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  unsigned long long sc[2];
  CU(cudaMemcpy(sc, c->d_scalars, 16, cudaMemcpyDeviceToHost));
  stats[0] = sc[0];
  stats[1] = sc[1];
  stats[2] = 1ull << c->log2cap;
  stats[3] = c->launches;
  if (n >= 5) stats[4] = (uint64_t)(c->kernel_ms * 1e3);
  return MG_OK;
}

// the counted k-mers go straight into the sample scan: no KMC database, no host round trip
extern "C" int mg_scan_counted(mg_ctx *ctx, mg_counter *c) {
  if (!ctx || !c) return set_err(MG_ERR_ARG, "NULL argument");
  if (!c->finished) return set_err(MG_ERR_STATE, "mg_scan_counted before mg_count_finish");
  if (c->device != ctx->device) return set_err(MG_ERR_ARG, "counter and context live on different devices");
  if (c->k != ctx->ref_k) return set_err(MG_ERR_ARG, "counter holds %d-mers but ref_k is %d", c->k, ctx->ref_k);
  if (!ctx->alt_final) return set_err(MG_ERR_STATE, "scan before mg_finalize_alt (BF::increment is a no-op in write mode)");
  if (!c->n_out) return MG_OK;
  CU(cudaSetDevice(ctx->device));
  return scan_device(ctx, c->out_keys, c->out_counts, c->n_out, ctx->stream[0]);
}

// ---- timing on the library's own streams (torch.cuda.Event cannot see them) ----
extern "C" int mg_event_record(mg_ctx *c, int idx) {
  if (!c || idx < 0 || idx >= 64) return set_err(MG_ERR_ARG, "bad event index");
  CU(cudaSetDevice(c->device));
  if (!c->tj) CU(cudaEventCreateWithFlags(&c->tj, cudaEventDisableTiming));
  if (!c->evs[idx]) CU(cudaEventCreate(&c->evs[idx]));
  // the event follows everything enqueued so far on both streams, and precedes what comes next
  CU(cudaEventRecord(c->tj, c->stream[1]));
  CU(cudaStreamWaitEvent(c->stream[0], c->tj, 0));
  CU(cudaEventRecord(c->evs[idx], c->stream[0]));
  CU(cudaStreamWaitEvent(c->stream[1], c->evs[idx], 0));
  return MG_OK;
}
extern "C" int mg_event_elapsed_ms(mg_ctx *c, int a, int b, float *ms) {
  if (!c || !ms || a < 0 || b < 0 || a >= 64 || b >= 64 || !c->evs[a] || !c->evs[b])
    return set_err(MG_ERR_ARG, "bad event index");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(c->evs[b]));
  CU(cudaEventElapsedTime(ms, c->evs[a], c->evs[b]));
  return MG_OK;
}
extern "C" int mg_event_sync(mg_ctx *c, int idx) {
  if (!c || idx < 0 || idx >= 64 || !c->evs[idx]) return set_err(MG_ERR_ARG, "bad event index");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(c->evs[idx]));
  return MG_OK;
}
extern "C" int mg_genotype_kernel_ms(mg_ctx *c, float *ms3) {
  if (!c || !ms3 || !c->ge[3]) return set_err(MG_ERR_ARG, "no mg_genotype call to report");
  CU(cudaSetDevice(c->device));
  CU(cudaEventSynchronize(c->ge[3]));
  ms3[0] = 0;  // (mg_genotype_weights_device alone: no look-up of this context to report)
  if (cudaEventQuery(c->ge[1]) == cudaSuccess && cudaEventElapsedTime(&ms3[0], c->ge[0], c->ge[1]) != cudaSuccess) {
    cudaGetLastError();
    ms3[0] = 0;
  }
  CU(cudaEventElapsedTime(&ms3[1], c->ge[4], c->ge[2]));
  CU(cudaEventElapsedTime(&ms3[2], c->ge[2], c->ge[3]));
  return MG_OK;
}
extern "C" int mg_refpass_kernel_ms(mg_ctx *c, float *ms) {
  if (!c || !ms || !c->rp_chunks) return set_err(MG_ERR_ARG, "no mg_scan_reference call to report");
  CU(cudaSetDevice(c->device));
  float total = 0;
  for (size_t j = 0; j < c->rp_chunks; ++j) {  // the rolling-pass kernels of every chunk of the last contig
    float t = 0;
    CU(cudaEventSynchronize(c->rp_events[2 * j + 1]));
    CU(cudaEventElapsedTime(&t, c->rp_events[2 * j], c->rp_events[2 * j + 1]));
    total += t;
  }
  *ms = total;
  return MG_OK;
}
extern "C" int mg_launch_count(mg_ctx *c, uint64_t *n) {
  if (!c || !n) return set_err(MG_ERR_ARG, "bad argument");
  *n = c->launches;
  return MG_OK;
}

// measured ceilings on `device`, GB/s of useful bytes, best of `reps`:
//   mode 0 / 2 / 3 : independent random reads of 1 / 2 / 4 separate sectors of an aligned 32 / 64 / 128-byte unit
//   mode 4 / 5 / 6 : random aligned 128 / 64 / 32-byte units, each fetched by 8 / 4 / 2 lanes in one coalesced
//                    request (mode 4 is k_scan's pattern)
//   mode 1         : streaming 16-byte reads
extern "C" int mg_diag_bandwidth(int device, int mode, uint64_t bytes, int reps, double *gbs) {
  if (!gbs || bytes < (1ull << 20) || reps < 1 || mode < 0 || mode > 6) return set_err(MG_ERR_ARG, "bad argument");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  DevFree buf, sink;
  CU(cudaMalloc(&buf.p, bytes));
  CU(cudaMalloc(&sink.p, 4));
  CU(cudaMemset(buf.p, 0, bytes));
  cudaEvent_t a, b;
  CU(cudaEventCreate(&a));
  CU(cudaEventCreate(&b));
  const int grid = prop.multiProcessorCount * 8;
  const uint64_t per_thread = 256;
  double best = 0.0;
  for (int r = 0; r < reps + 1; ++r) {
    CU(cudaEventRecord(a));
    const int gran = mode == 0 ? 1 : mode == 2 ? 2 : 4;
    double useful;
    if (mode == 1) {
      mg::k_diag_stream<<<grid, 256>>>((const uint4 *)buf.p, bytes / 16, (uint32_t *)sink.p);
      useful = (double)bytes;
    } else if (mode >= 4) {  // 4: 128 B by 8 lanes, 5: 64 B by 4 lanes, 6: 32 B by 2 lanes
      const int ll = mode == 4 ? 3 : mode == 5 ? 2 : 1;
      mg::k_diag_lines<<<grid * 4, 256>>>((const uint4 *)buf.p, bytes / (16ull << ll), ll, per_thread,
                                          (uint32_t *)sink.p);
      useful = (double)grid * 4 * 256 * (double)per_thread * 16.0;
    } else {
      mg::k_diag_random<<<grid * 4, 256>>>((const uint32_t *)buf.p, bytes / (32 * (uint64_t)gran), gran, per_thread,
                                           (uint32_t *)sink.p);
      useful = (double)grid * 4 * 256 * (double)per_thread * 32.0 * gran;
    }
    CU(cudaGetLastError());
    CU(cudaEventRecord(b));
    CU(cudaEventSynchronize(b));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, a, b));
    double g = useful / (ms * 1e-3) / 1e9;
    if (r > 0 && g > best) best = g;  // first repetition is the warm-up
  }
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  *gbs = best;
  return MG_OK;
}

extern "C" int mg_host_alloc(void **p, size_t bytes) {
  if (!p) return set_err(MG_ERR_ARG, "NULL argument");
  CU(cudaHostAlloc(p, bytes, cudaHostAllocDefault));
  return MG_OK;
}
extern "C" int mg_host_free(void *p) {
  CU(cudaFreeHost(p));
  return MG_OK;
}

// ---------------------------------------------------------------------------
// host-side self tests of the __host__ __device__ helpers (CPU-only test-suite)
// ---------------------------------------------------------------------------
extern "C" uint64_t mg_selftest_hash_packed(uint64_t lo, uint64_t hi, int k, uint64_t *canon_lo, uint64_t *canon_hi) {
  u128 x = {lo, hi}, c;
  uint64_t h = mg::canon_hash_rt(x, k, &c);
  if (canon_lo) *canon_lo = c.lo;
  if (canon_hi) *canon_hi = c.hi;
  return h;
}
extern "C" uint64_t mg_selftest_hash_packed_k35(uint64_t lo, uint64_t hi) {
  u128 x = {lo, hi}, c;
  return mg::canon_hash<35>(x, &c);
}
extern "C" uint64_t mg_selftest_hash_packed_k43(uint64_t lo, uint64_t hi) {
  u128 x = {lo, hi}, c;
  return mg::canon_hash<43>(x, &c);
}
extern "C" uint64_t mg_selftest_hash_ascii(const char *s, int len) {
  return mg::hash_ascii(reinterpret_cast<const uint8_t *>(s), len);
}
extern "C" int mg_selftest_pack35(const char *s35, uint64_t *lo, uint64_t *hi) {
  uint32_t t[9] = {0};
  memcpy(t, s35, 35);
  u128 x;
  uint32_t bad = mg::pack_words<35>(t, &x);
  if (lo) *lo = x.lo;
  if (hi) *hi = x.hi;
  return bad ? 0 : 1;
}
extern "C" float mg_selftest_logf(float x) { return mg::glibc_logf(x); }
extern "C" int mg_selftest_genotype(const uint32_t *cov, const float *freq, int n_alleles, float error_rate,
                                    int max_cov, int haploid, double *lik, int *status, int *best_gt, int *gq) {
  return mg::genotype_one(cov, freq, n_alleles, error_rate, max_cov, haploid != 0, nullptr, lik, status, best_gt, gq);
}
