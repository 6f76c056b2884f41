// Hand-written sm_100a kernels of the MALVA hot path (see index.cuh for the data layout).
//   K3  k_add_signatures / k_add_packed / k_add_spill / k_line_popc    index-time inserts + switch_mode
//   K2  k_refpass / k_refpass_short                                    reference rolling pass
//   K1  k_scan / k_scan_hits                                           sample k-mer scan
//   K4  k_lookup_packed / k_lookup_irr / k_lookup / k_coverage         coverage read-back (one sample, or a sample set)
//   K5  k_genotype                                                     likelihoods + posterior arg-max
//       k_counters_xfer / k_sum_peers                                  dense counter image for the multi-GPU reduce
//       k_samples_take_*                                               sample sets: several samples on one index
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

#include "geno.cuh"
#include "index.cuh"
#include "xxh3.cuh"

namespace mg {

__device__ __forceinline__ u128 u128_of(uint4 q) {
  u128 r;
  r.lo = (uint64_t)q.x | ((uint64_t)q.y << 32);
  r.hi = (uint64_t)q.z | ((uint64_t)q.w << 32);
  return r;
}
__device__ __forceinline__ uint4 uint4_of(u128 x) {
  return make_uint4((uint32_t)x.lo, (uint32_t)(x.lo >> 32), (uint32_t)x.hi, (uint32_t)(x.hi >> 32));
}

// scalars: [0] new keys, [1] irregular ref keys, [2] popcount, [3] error flag, [4] spilled keys, [5] scratch cursor
// ---------------------------------------------------------------------------
// K3a: index-time inserts (add_kmers_to_bf, main.cpp:122-144)
// ---------------------------------------------------------------------------
__device__ __forceinline__ void insert_ref_key(const DevView &v, uint32_t *occ_rw, uint64_t h, u128 canon, uint64_t i,
                                               unsigned long long *scalars, uint32_t *spill_idx) {
  const uint64_t idx = bf_index(v, h);
  occ_set(v, occ_rw, idx);
  const uint64_t line = idx >> 8;
  int r = line_insert(v, line, canon);
  if (r == 1) {
    atomicAdd(&scalars[0], 1ull);
  } else if (r < 0) {  // line full: flag it and leave the key for the overflow pass
    line_set_overflow(v, line);
    unsigned long long p = atomicAdd(&scalars[4], 1ull);
    spill_idx[p] = (uint32_t)i;
  }
}
__device__ __forceinline__ void set_bf_bit(const DevView &v, uint32_t *occ_rw, uint64_t h) {
  uint64_t idx = bf_index(v, h);
  occ_set(v, occ_rw, idx);
  atomicOr(line_words(v, idx >> 8) + ((idx & 255) >> 5), 1u << (idx & 31));
}

__global__ void __launch_bounds__(128) k_add_signatures(const uint8_t *__restrict__ pool,
                                                       const uint64_t *__restrict__ off,
                                                       const uint8_t *__restrict__ is_ref, uint64_t n, DevView v,
                                                       uint32_t *occ_rw, unsigned long long *scalars,
                                                       uint32_t *irregular_idx, uint32_t *spill_idx) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t b = off[i], e = off[i + 1];
  int len = (int)(e - b);
  if (len > 128) {
    atomicExch(&scalars[3], 1ull);
    return;
  }
  uint8_t s[128];
  for (int j = 0; j < len; ++j) s[j] = pool[b + j];
  u128 x, canon;
  bool regular = pack_ascii(s, len, v.k, &x);
  if (is_ref[i]) {  // ref_bf.add_key
    if (!regular) {  // not k symbols of ACGT: can never match a sample k-mer; kept on the host
      unsigned long long p = atomicAdd(&scalars[1], 1ull);
      irregular_idx[p] = (uint32_t)i;
      return;
    }
    uint64_t h = canon_hash_rt(x, v.k, &canon);
    insert_ref_key(v, occ_rw, h, canon, i, scalars, spill_idx);
  } else {  // bf.add_key
    uint64_t h = regular ? canon_hash_rt(x, v.k, &canon) : hash_ascii(s, len);
    set_bf_bit(v, occ_rw, h);
  }
}

// same inserts for signature k-mers that arrive already packed (exactly k symbols of ACGT)
__global__ void __launch_bounds__(256) k_add_packed(const uint4 *__restrict__ kmers, const uint8_t *__restrict__ is_ref,
                                                   uint64_t n, DevView v, uint32_t *occ_rw,
                                                   unsigned long long *scalars, uint32_t *spill_idx) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u128 x = mask128(u128_of(kmers[i]), 2 * v.k), canon;
  uint64_t h = canon_hash_rt(x, v.k, &canon);
  if (is_ref[i])
    insert_ref_key(v, occ_rw, h, canon, i, scalars, spill_idx);
  else
    set_bf_bit(v, occ_rw, h);
}

// second pass over the keys whose line was full: insert into the overflow table.
// Keys come either from an ASCII pool (off != nullptr) or from a packed array.
__global__ void __launch_bounds__(128) k_add_spill(const uint32_t *__restrict__ spill_idx, uint64_t n_spill,
                                                  const uint8_t *__restrict__ pool, const uint64_t *__restrict__ off,
                                                  const uint4 *__restrict__ packed, DevView v, u128 *ovf_keys_rw,
                                                  unsigned long long *scalars) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_spill) return;
  uint64_t i = spill_idx[j];
  u128 x, canon;
  if (off) {
    uint64_t b = off[i];
    int len = (int)(off[i + 1] - b);
    uint8_t s[64];
    for (int t = 0; t < len && t < 64; ++t) s[t] = pool[b + t];
    pack_ascii(s, len, v.k, &x);
  } else {
    x = mask128(u128_of(packed[i]), 2 * v.k);
  }
  canon_hash_rt(x, v.k, &canon);
  if (ovf_insert(v, ovf_keys_rw, canon) == 1) atomicAdd(&scalars[0], 1ull);
}

__global__ void k_fill_keys(u128 *keys, uint64_t n, uint64_t hi_mask) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    keys[i].lo = ~0ull;
    keys[i].hi = hi_mask;
  }
}
// a fresh probe-line array: filter bits 0, key slots empty, rank and counters 0
__global__ void k_init_lines(uint4 *lines, uint64_t n_lines, uint64_t hi_mask) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one uint4 per thread
  if (i >= n_lines * LINE_U4) return;
  const int q = (int)(i & 7);
  lines[i] = (q < 2 || q == 7) ? make_uint4(0, 0, 0, 0) : make_uint4(~0u, ~0u, (uint32_t)hi_mask, (uint32_t)(hi_mask >> 32));
}

// re-insert every key of an old overflow table into a larger one (index-build time: counts are all zero)
__global__ void k_rehash(const u128 *old_keys, uint64_t old_cap, DevView v, u128 *ovf_keys_rw) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= old_cap) return;
  u128 key = old_keys[i];
  key.hi &= v.key_hi_mask;
  if (key_empty(v, key)) return;
  ovf_insert(v, ovf_keys_rw, key);
}

// ---------------------------------------------------------------------------
// K3c: canonical index image (run by mg_finalize_alt, before any count exists): the key slots of every line in
// ascending order, empty slots last.  Which slot a key took during the build depended on the order (and the races)
// of the inserts; after this pass it depends on the key set only.
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_sort_line_keys(DevView v) {
  uint64_t line = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= v.n_lines) return;
  uint4 *p = v.lines + line * LINE_U4 + 2;
  u128 q[LINE_KEYS];
#pragma unroll
  for (int s = 0; s < LINE_KEYS; ++s) q[s] = u128_of(p[s]);
  const uint64_t flag = q[LINE_KEYS - 1].hi & v.ovf_flag_hi;
#pragma unroll
  for (int s = 0; s < LINE_KEYS; ++s) q[s].hi &= v.key_hi_mask;
  if (key_empty(v, q[1])) return;  // zero or one key: already canonical (slots fill from the front)
#pragma unroll
  for (int a = 1; a < LINE_KEYS; ++a) {  // insertion sort on (hi, lo); an empty slot is the largest value
#pragma unroll
    for (int b = a; b > 0; --b) {
      if (less128(q[b], q[b - 1])) {
        u128 t = q[b - 1];
        q[b - 1] = q[b];
        q[b] = t;
      }
    }
  }
  q[LINE_KEYS - 1].hi |= flag;
#pragma unroll
  for (int s = 0; s < LINE_KEYS; ++s) p[s] = uint4_of(q[s]);
}
// the five key slots of the listed lines, to / from a dense array (overflow canonicalisation on the host)
__global__ void k_gather_line_keys(const uint4 *lines, const uint64_t *ids, uint64_t n, uint4 *out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * LINE_KEYS) return;
  out[i] = lines[ids[i / LINE_KEYS] * LINE_U4 + 2 + (i % LINE_KEYS)];
}
__global__ void k_scatter_line_keys(uint4 *lines, const uint64_t *ids, uint64_t n, const uint4 *in) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * LINE_KEYS) return;
  lines[ids[i / LINE_KEYS] * LINE_U4 + 2 + (i % LINE_KEYS)] = in[i];
}

// ---------------------------------------------------------------------------
// K3b: switch_mode (bloom_filter.hpp:93-98): ones per probe line (then an exclusive scan -> rank, written into
// word 28 of every line); also used on a plain bit array (stride_u32 = 8) for context_bf statistics
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_line_popc(const uint32_t *__restrict__ words, uint64_t n_units, int stride_u32,
                                                  uint32_t *__restrict__ unit_count, unsigned long long *total) {
  uint64_t b = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t c = 0;
  if (b < n_units) {
    const uint4 *p = reinterpret_cast<const uint4 *>(words + b * (uint64_t)stride_u32);
    uint4 q0 = p[0], q1 = p[1];
    c = __popc(q0.x) + __popc(q0.y) + __popc(q0.z) + __popc(q0.w) + __popc(q1.x) + __popc(q1.y) + __popc(q1.z) +
        __popc(q1.w);
    if (unit_count) unit_count[b] = c;
  }
  __shared__ uint32_t red[8];
  uint32_t s = c;
  for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 8) {
    s = red[threadIdx.x];
    for (int o = 4; o > 0; o >>= 1) s += __shfl_down_sync(0xffu, s, o);
    if (threadIdx.x == 0 && s) atomicAdd(total, (unsigned long long)s);
  }
}
__global__ void __launch_bounds__(256) k_write_rank(DevView v, const uint32_t *__restrict__ rank) {
  uint64_t line = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= v.n_lines) return;
  v.lines[line * LINE_U4 + 7] = make_uint4(rank[line], 0u, 0u, 0u);
}
// keys held by the five slots of every line (empty slots come last once the image is canonical)
__global__ void __launch_bounds__(256) k_line_keycount(DevView v, uint32_t *__restrict__ cnt) {
  uint64_t line = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (line >= v.n_lines) return;
  const uint4 *p = v.lines + line * LINE_U4 + 2;
  uint32_t c = 0;
#pragma unroll
  for (int s = 0; s < LINE_KEYS; ++s) c += key_empty(v, key_of(v, p[s])) ? 0u : 1u;
  cnt[line] = c;
}
// the 256 filter bits of every probe line, gathered into a plain bit array (state download)
__global__ void k_extract_bits(const uint4 *__restrict__ lines, uint64_t n_lines, uint4 *__restrict__ out) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;  // one uint4 (128 bits) per thread
  if (i >= n_lines * 2) return;
  out[i] = lines[(i >> 1) * LINE_U4 + (i & 1)];
}

// ---------------------------------------------------------------------------
// Dense counter image (the multi-GPU reduce, the counter download): the counters that live inside the probe lines
// copied to / from dense arrays -- bf_counts[rank + j] for the inline alt counters (j < 3), key_dense[key_rank[L] + s]
// for the key counts.  Eight lanes per line, one uint4 each: the line array is read once, fully coalesced.
// ---------------------------------------------------------------------------
template <bool SCATTER>
__global__ void __launch_bounds__(256) k_counters_xfer(DevView v, const uint32_t *__restrict__ key_rank,
                                                      uint32_t *__restrict__ key_dense) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t line = t >> 3;
  const int sub = (int)(t & 7);
  const bool ok = line < v.n_lines;
  const uint4 q = ok ? v.lines[line * LINE_U4 + (uint64_t)sub] : make_uint4(0, 0, 0, 0);
  const uint32_t pc = sub < 2 ? (uint32_t)(__popc(q.x) + __popc(q.y) + __popc(q.z) + __popc(q.w)) : 0u;
  const int g0 = (int)(threadIdx.x & 24);
  const uint32_t n_alt = __shfl_sync(0xffffffffu, pc, g0) + __shfl_sync(0xffffffffu, pc, g0 + 1);
  if (!ok) return;
  uint32_t *w = line_words(v, line);
  if (sub == 7) {
    const uint32_t c[3] = {q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < LINE_INLINE_ALT; ++j)
      if ((uint32_t)j < n_alt) {
        if (SCATTER)
          w[LINE_W_RANK + 1 + j] = v.bf_counts[(uint64_t)q.x + (uint64_t)j];
        else
          v.bf_counts[(uint64_t)q.x + (uint64_t)j] = c[j];
      }
  } else if (sub >= 2) {
    const int s = sub - 2;
    if (key_empty(v, key_of(v, q))) return;
    const uint64_t d = (uint64_t)key_rank[line] + (uint64_t)s;
    uint32_t *cp = v.inline_counts ? w + 8 + 4 * s + 3 : v.key_counts + line * LINE_KEYS + (uint64_t)s;
    if (SCATTER)
      *cp = key_dense[d];
    else
      key_dense[d] = v.inline_counts ? q.w : *cp;
  }
}
// dst[i] += sum over peers of src[p][i] (u32, wrap-around): the counter reduce of replicated contexts inside one
// process; the peers' arrays are read in place over NVLink (peer access), no staging copy
struct PeerPtrs {
  const uint32_t *p[15];
  int n;
};
__global__ void __launch_bounds__(256) k_sum_peers(uint32_t *__restrict__ dst, PeerPtrs peers, uint64_t n) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * 4;
  for (uint64_t i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; i < n; i += stride) {
    if (i + 3 < n) {
      uint4 a = *reinterpret_cast<const uint4 *>(dst + i);
      for (int p = 0; p < peers.n; ++p) {
        const uint4 b = *reinterpret_cast<const uint4 *>(peers.p[p] + i);
        a.x += b.x, a.y += b.y, a.z += b.z, a.w += b.w;
      }
      *reinterpret_cast<uint4 *>(dst + i) = a;
    } else {
      for (uint64_t j = i; j < n; ++j)
        for (int p = 0; p < peers.n; ++p) dst[j] += peers.p[p][j];
    }
  }
}

// ---------------------------------------------------------------------------
// K2: reference rolling pass (main.cpp:385-400)
// Each CTA stages a tile of the contig in shared memory (with a ref_k-1 halo, 16-byte loads); each thread rolls
// RP_RUN consecutive windows through 2-bit registers.  Windows that contain a non-ACGT symbol take the
// byte-exact ASCII path (the RCN table maps IUPAC symbols to NUL, bloom_filter.hpp:36-50).
// The contig arrives in chunks (double-buffered H2D copies, malva_gpu.cu): `chunk` holds the bytes
// [chunk_base, ...) of the contig, the launch covers the window end positions [p_begin, p_end).
// ---------------------------------------------------------------------------
constexpr int RP_THREADS = 256;
constexpr int RP_RUN = 16;
constexpr int RP_TILE = RP_THREADS * RP_RUN;

__device__ __forceinline__ uint32_t base_code(uint8_t c) {  // 0..3, or 4 for anything else
  return c == 'A' ? 0u : c == 'C' ? 1u : c == 'G' ? 2u : c == 'T' ? 3u : 4u;
}

template <int K, int REFK>
__global__ void __launch_bounds__(RP_THREADS) k_refpass(const uint8_t *__restrict__ chunk, uint64_t chunk_base,
                                                        uint64_t p_begin, uint64_t p_end, DevView v,
                                                        uint32_t *ctx_words_rw) {
  extern __shared__ uint4 rp_sm4[];
  uint8_t *sm = reinterpret_cast<uint8_t *>(rp_sm4);
  const int k = K > 0 ? K : v.k, ref_k = REFK > 0 ? REFK : v.ref_k;
  const int d = (ref_k - k) / 2;
  const bool odd = ((ref_k - k) & 1) != 0;
  // window end positions handled by this CTA: [p0, p1)
  uint64_t p0 = p_begin + (uint64_t)blockIdx.x * RP_TILE;
  uint64_t p1 = p0 + RP_TILE < p_end ? p0 + RP_TILE : p_end;
  uint64_t base = p0 - (uint64_t)(ref_k - 1);  // first contig byte staged
  const uint8_t *src = chunk + (base - chunk_base);
  int nbytes = (int)(p1 - base);
  if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
    const int n16 = nbytes >> 4;
    for (int i = threadIdx.x; i < n16; i += RP_THREADS) rp_sm4[i] = __ldg(reinterpret_cast<const uint4 *>(src) + i);
    for (int i = (n16 << 4) + threadIdx.x; i < nbytes; i += RP_THREADS) sm[i] = src[i];
  } else {
    for (int i = threadIdx.x; i < nbytes; i += RP_THREADS) sm[i] = src[i];
  }
  __syncthreads();
  uint64_t q0 = p0 + (uint64_t)threadIdx.x * RP_RUN;
  if (q0 >= p1) return;
  uint64_t q1 = q0 + RP_RUN < p1 ? q0 + RP_RUN : p1;
  // prime the rolling state with the ref_k-1 bases before q0
  u128 x = {0, 0};
  uint64_t bad = 0;  // bit j set <=> base (p - j) is not ACGT
  const u128 m = mask128(u128{~0ull, ~0ull}, 2 * ref_k);
  int o = (int)(q0 - base) - (ref_k - 1);
  for (int j = 0; j < ref_k - 1; ++j) {
    uint32_t c = base_code(sm[o + j]);
    x.hi = (x.hi << 2) | (x.lo >> 62);
    x.lo = (x.lo << 2) | (c & 3u);
    bad = (bad << 1) | (c >> 2);
  }
  const uint64_t m43 = ref_k >= 64 ? ~0ull : ((1ull << ref_k) - 1);
  const uint64_t mk = k >= 64 ? ~0ull : ((1ull << k) - 1);
  for (uint64_t p = q0; p < q1; ++p) {
    int sp = (int)(p - base);
    uint32_t c = base_code(sm[sp]);
    x.hi = (x.hi << 2) | (x.lo >> 62);
    x.lo = (x.lo << 2) | (c & 3u);
    x.hi &= m.hi;
    x.lo &= m.lo;
    bad = (bad << 1) | (c >> 2);
    // k-mer window of the reference at this step.  With t = p-(ref_k-1) slides done:
    //   (ref_k-k) even        : ref[p-d-k+1 .. p-d]
    //   odd, t == 0 (primed)  : ref[d .. d+k-1]                 (ends at p-d-1)
    //   odd, 1 <= t < k       : ref[d+t .. d+k-1] ++ ref[k+d+1 .. k+d+t]   (main.cpp:395-397 skips ref[d+k])
    //   odd, t >= k           : ref[p-d-k+1 .. p-d]
    // (t < k only happens in the first chunk of a contig: chunk_base == 0 there, the quirk reads index `chunk`)
    uint64_t t = p - (uint64_t)(ref_k - 1);
    bool quirk = odd && t >= 1 && t < (uint64_t)k;
    int shift = d + ((odd && t == 0) ? 1 : 0);
    uint64_t h35;
    if (!quirk && ((bad >> shift) & mk) == 0) {
      u128 x35 = mask128(shr128(x, 2 * shift), 2 * k), canon;
      h35 = canon_hash_k<K>(x35, k, &canon);
    } else {
      uint8_t s[64];
      if (!quirk) {
        for (int j = 0; j < k; ++j) s[j] = sm[sp - shift - k + 1 + j];
      } else {
        int n_old = k - (int)t;
        for (int j = 0; j < n_old; ++j) s[j] = chunk[(uint64_t)d + t + (uint64_t)j];
        for (int j = 0; j < (int)t; ++j) s[n_old + j] = chunk[(uint64_t)(k + d + 1) + (uint64_t)j];
      }
      h35 = hash_ascii(s, k);
    }
    const uint64_t i35 = bf_index(v, h35);
    if (!occ_test(v, i35) || !bf_test(v, i35)) continue;
    uint64_t h43;
    if ((bad & m43) == 0) {
      u128 canon;
      h43 = canon_hash_k<REFK>(x, ref_k, &canon);
    } else {
      uint8_t s[64];
      for (int j = 0; j < ref_k; ++j) s[j] = sm[sp - ref_k + 1 + j];
      h43 = hash_ascii(s, ref_k);
    }
    uint64_t cidx = bf_index(v, h43);
    atomicOr(ctx_words_rw + (cidx >> 5), 1u << (cidx & 31));
  }
}

// contig shorter than ref_k: the reference hashes the (shorter) substr() results once
__global__ void k_refpass_short(const uint8_t *seq, uint64_t len, DevView v, uint32_t *ctx_words_rw) {
  if (threadIdx.x || blockIdx.x) return;
  int d = (v.ref_k - v.k) / 2;
  int kl = (int)len - d < v.k ? (int)len - d : v.k;
  uint64_t h = hash_ascii(seq + d, kl);
  if (!bf_test(v, bf_index(v, h))) return;
  uint64_t hc = hash_ascii(seq, (int)len);
  uint64_t cidx = bf_index(v, hc);
  atomicOr(ctx_words_rw + (cidx >> 5), 1u << (cidx & 31));
}

// ---------------------------------------------------------------------------
// K1: sample k-mer scan (main.cpp:487-500)
//   ref_bf.increment(kmer, c);  if (!context_bf.test_key(context)) bf.increment(kmer, c);
//
// A warp owns 32 k-mers per iteration (packed input: 64, two per lane): lane i hashes k-mer i (coalesced loads,
// canonical form, XXH3) and tests the L2-resident occupancy pre-filter (its 16-byte piece arrives in shared memory by
// cp.async).  Only about a third of the k-mers of a whole-genome workload need their probe line at all, so probing
// lane by lane would leave two thirds of the lanes idle through the whole probe sequence (the kernel is bound by
// instruction issue, profiles/round1_k1_v5.md).  The k-mers that need a line are therefore COMPACTED: they go into a
// ring in shared memory ({canonical k-mer | line, index, count, bit}; 64-128 entries), and whenever the ring holds 32
// entries the warp runs one FULL probe round:
//   * the 32 probe lines are copied into the warp's 4 KB tile with cp.async (LDGSTS, no register staging): eight
//     unrolled rounds, in each the four 8-lane groups move one line each, lane j of a group moving uint4 j -- a line
//     costs exactly one fully coalesced 128-byte request and all 32 are in flight together.  The tile is XOR-swizzled
//     (uint4 j of row L sits at column j ^ (L & 7)) so that every lane then reads ITS row with conflict-free 16-byte
//     shared loads;
//   * the lane tests its filter bit and compares the five key slots;
//   * a key hit adds the count into the slot itself (the line was fetched a moment ago: the RED lands in L2);
//   * a filter hit needs a second XXH3 (the 43-mer, for the context filter): the scan only records it --
//     {context k-mer, address of the bit's counter, count} -- and k_scan_hits works all of them off afterwards.
// (A bulk copy -- cp.async.bulk + mbarrier, one per line -- was considered for the line gather and rejected: UBLKCP
// takes its addresses from uniform registers, so 32 different lines cost 32 serialised issues per round against the
// 8 LDGSTS of this scheme; profiles/round2_k1.md.)
// ---------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t smem_addr, const void *gptr) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_addr), "l"(gptr) : "memory");
}

// canon_hash<K> (xxh3.cuh) with the 2-bit -> ASCII expansion done by a 256-entry shared-memory table (4 bases per
// look-up) instead of shift/mask/PRMT sequences: the scan kernel is bound by the ALU pipe (LOP3/SHF/PRMT issue at
// half rate), shared-memory loads go through the otherwise idle LSU pipe.  tab[v] = expand4(v).
template <int K>
__device__ __forceinline__ uint64_t canon_hash_lut(u128 x, u128 *canon, const uint32_t *tab) {
  u128 rc = revcomp(x, K);
  bool fwd = less128(x, rc);
  u128 c = fwd ? x : rc, other = fwd ? rc : x;
  u128 r;
  r.lo = ~other.lo;
  r.hi = ~other.hi;
  r = mask128(r, 2 * K);  // LSB-first image of the canonical k-mer
  constexpr int NW = (K + 7) / 8;
  uint64_t w[NW + 1];
  const uint32_t rw[4] = {(uint32_t)r.lo, (uint32_t)(r.lo >> 32), (uint32_t)r.hi, (uint32_t)(r.hi >> 32)};
#pragma unroll
  for (int j = 0; j < NW; ++j) {  // ASCII bytes 8j .. 8j+7 = bases held by bytes 2j and 2j+1 of r
    const uint32_t word = rw[j >> 1];
    uint32_t lo = tab[__byte_perm(word, 0u, (j & 1) ? 0x4442u : 0x4440u)], hi = 0;
    if (8 * j + 4 < K) hi = tab[__byte_perm(word, 0u, (j & 1) ? 0x4443u : 0x4441u)];
    w[j] = (uint64_t)lo | ((uint64_t)hi << 32);
  }
  w[NW] = 0;
  *canon = c;
  return xxh3_64_words(w, K);
}
__device__ __forceinline__ u128 canon_only(u128 x, int k) {
  u128 rc = revcomp(x, k);
  return less128(x, rc) ? x : rc;
}

// The shape of the scan for input MODE (see k_scan), in 256-thread CTAs.
//   ilp:      k-mers per lane and batch: 2 for packed k-mers, 1 for KMC records
//   q:        ring entries per warp: the round in flight (32; MODE 0 only) + the entries that pile up until the next
//             turn (fewer than 32 + 32 * ilp)
//   warp_u4:  shared memory per warp in uint4: the 4 KB tile, the ring keys, the ring meta and a 16-byte landing slot
//             per k-mer of a batch for the pre-filter pieces
//   smem:     bytes per CTA: the warps + the 1 KB expansion table and a deferred-hit counter per warp
//   min_ctas: CTAs per SM that fit the shared memory (227 KB usable, 1 KB reserved per CTA), capped at 1024 threads
//             (64 registers each) -- 768 threads (85 registers) for the two chains of MODE 0
constexpr int SCAN_THREADS = 256;
struct ScanShape {
  int ilp, q, warp_u4, smem, min_ctas;
};
__host__ __device__ constexpr ScanShape scan_shape(int mode) {
  const int ilp = mode == 0 ? 2 : 1, q = mode == 0 ? 128 : 64, warp_u4 = 256 + 2 * q + 32 * ilp;
  const int warps = SCAN_THREADS / 32, smem = warps * warp_u4 * 16 + 256 * 4 + warps * 4;
  const int by_smem = (227 * 1024) / (smem + 1024), by_threads = (mode == 0 ? 768 : 1024) / SCAN_THREADS;
  return {ilp, q, warp_u4, smem, by_smem < by_threads ? by_smem : by_threads};
}

// Where the sample k-mers come from.  MODE 0: packed {lo,hi} words + u32 counts.  MODE 1: raw records of a
// KMC database suffix file (.kmc_suf): (ref_k - p)/4 suffix bytes (2-bit codes, first base most significant)
// + counter_size little-endian count bytes; the p-symbol prefix of record g is the LUT bucket that contains g
// (lut[j] = records before prefix j; listing order = record order).  Decoding them here halves the PCIe
// bytes per k-mer (10 B instead of 20 B for k = 43) and removes the host-side CKmerAPI::to_string pass.
struct ScanSrc {
  const uint4 *kmers;
  const uint32_t *counts;
  const uint8_t *recs;  // 16-byte aligned, padded by 16 bytes
  const uint64_t *lut;  // n_lut entries + a guard of ~0
  uint64_t first_rec;   // global index of recs[0]
  uint32_t n_lut, prefix_mask;
  int prefix_len, suf_bytes, counter_size;
  uint32_t min_count;
  uint64_t max_count;
  // Deferred filter hits: {context k-mer, counter address, count}, 32 bytes each, in the warp's own segment of
  // hit_buf; k_scan_hits finishes them.  A full segment falls back to the in-line path.  hit_buf == nullptr:
  // always in line.
  uint4 *hit_buf;
  uint32_t *hit_counts;  // per warp of the scan grid
  uint32_t seg_cap;      // entries per warp segment
};

__device__ __forceinline__ uint32_t lut_bucket(const uint64_t *lut, uint32_t n_lut, uint64_t g) {
  uint32_t lo = 0, hi = n_lut;  // largest j with lut[j] <= g (lut[0] == 0, lut[n_lut] == ~0)
  while (hi - lo > 1) {
    uint32_t mid = (lo + hi) >> 1;
    if (__ldg(lut + mid) <= g)
      lo = mid;
    else
      hi = mid;
  }
  return lo;
}

// K, REFK: the (k, ref_k) the hashes are specialised for; 0 takes them from the view at run time.  The per-warp state
// is private, the CTA only shares the expansion table.
// MODE 0 (packed k-mers) runs ASYNCHRONOUS rounds: the k-mers of batch i+1 are loaded into registers while batch i
// is hashed, and the gather of a round is only STARTED when the ring holds 32 entries: the warp goes on hashing and
// finishes the round (wait, compare, count) at the next turn, a batch or more later.  Every lane hashes two k-mers
// per batch, written as straight-line code over both so that the two dependent chains (canonical form -> table
// look-ups -> four 128-bit products) interleave: with ~30 resident warps per SM a single chain left the issue slots
// half empty (~11 cycles between two instructions of a warp, ncu).  Both k-mers of every lane go into the ring in one
// go: one ballot / prefix / turn check per batch instead of one per k-mer.
// MODE 1 (KMC records) stages the records of a batch in the tile, one per lane, and runs SYNCHRONOUS rounds: the tile
// is busy with the records until the batch is hashed, so a round starts and finishes before the next batch.
// MODE 0 reads the counts and short context k-mers with ld.global.nc.L1::no_allocate.  Both modes copy the 16-byte
// piece of the pre-filter that holds a k-mer's bit to a shared-memory slot with cp.async.cg (LDGSTS.BYPASS: nothing
// of it passes through L1) and read it from there.  Why: the 32 random pre-filter words of a warp each hold an L1 line
// while in flight; with shared memory carved out for three CTAs the remaining L1 (28-60 KB) capped the loads in flight
// per SM, and the kernel ran 25 % slower at the 228 KB carve-out than at 196 KB (profiles/round2_k1_final.md).  Through
// cp.async the kernel no longer cares, takes the whole carve-out, and has room for a ring deep enough for MODE 0's
// whole batch.
// The schemes measured against this one are in profiles/round2_k1*.md: probing after every batch, one, three or four
// k-mers per lane, synchronous rounds for packed input, 128-thread CTAs, loads through L1, and parking a hashed batch
// in shared memory until its pre-filter word arrives (the extra shared-memory traffic cost more than the hidden L2
// latency).
template <int K, int REFK, int MODE>
__global__ void __launch_bounds__(SCAN_THREADS, scan_shape(MODE).min_ctas) k_scan(ScanSrc src, uint64_t n, DevView v) {
  extern __shared__ uint4 scan_sm[];
  constexpr ScanShape S = scan_shape(MODE);
  constexpr int SCAN_WARPS = SCAN_THREADS / 32, SCAN_Q = S.q, SCAN_WARP_U4 = S.warp_u4;
  const int k = K > 0 ? K : v.k, ref_k = REFK > 0 ? REFK : v.ref_k;
  const int tail = ref_k - k - (ref_k - k) / 2;  // bases of the context after the k-mer (main.cpp:493)
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, sub = lane & 7, grp = lane >> 3;
  uint4 *tile = scan_sm + wid * SCAN_WARP_U4;  // 32 rows x 8 uint4
  uint4 *qkey = tile + 256, *qmeta = qkey + SCAN_Q;
  // this lane's pre-filter landing slots (one per k-mer of a batch, 32 apart)
  const uint4 *oslot = qmeta + SCAN_Q + lane;
  const uint32_t oslot_addr = (uint32_t)__cvta_generic_to_shared(oslot);
  const uint32_t tile_addr = (uint32_t)__cvta_generic_to_shared(tile);
  uint32_t *tab = reinterpret_cast<uint32_t *>(scan_sm + SCAN_WARPS * SCAN_WARP_U4);
  uint32_t *hitc = tab + 256 + wid;  // this warp's deferred-hit counter
  if (lane == 0) *hitc = 0;
  if constexpr (K > 0) {
    for (int t = threadIdx.x; t < 256; t += SCAN_THREADS) tab[t] = expand4((uint32_t)t);
    __syncthreads();
  } else {
    __syncwarp();
  }
  const bool inl = K > 0 ? (K <= INLINE_MAX_K) : (v.inline_counts != 0);
  const uint32_t mz = inl ? 0x7FFFFFFFu : 0xFFFFFFFFu, mw = inl ? 0u : 0x3FFFFFFFu;  // key bits of slot words 2, 3
  auto wrap = [](uint32_t x) { return x >= (uint32_t)SCAN_Q ? x - (uint32_t)SCAN_Q : x; };  // ring positions < 2 * SCAN_Q
  const uint32_t warp_id = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  // 32-bit indices: the host never launches more than 2^30 k-mers at once
  const uint32_t n32 = (uint32_t)n;
  const uint32_t step = ((gridDim.x * blockDim.x) >> 5) * 32;
  // destination of this lane's 16-byte piece within rows grp (even rounds) and grp + 4 (odd rounds) of a round
  const uint32_t d_even = tile_addr + (uint32_t)(grp * 128 + ((sub ^ grp) * 16));
  const uint32_t d_odd = tile_addr + (uint32_t)(grp * 128 + ((sub ^ (grp + 4)) * 16));
  const char *line_src = reinterpret_cast<const char *>(v.lines) + sub * 16;
  // ring state (warp-uniform): fl_n entries from fl_pos on are the round in flight (MODE 0), the pd_n entries after
  // them wait for the next round; fl_pos stays a multiple of 32 (only the very last round is partial)
  uint32_t fl_pos = 0, fl_n = 0, pd_n = 0;
  bool more = true;
  // START a round over the first min(pd_n, 32) pending entries: their 32 probe lines into the tile
  auto start_round = [&]() {
    const uint32_t n_new = pd_n < 32 ? pd_n : 32;
    fl_pos = wrap(fl_pos + fl_n);
    __syncwarp();  // the ring entries are visible; the previous round's reads of the tile are done
    const uint32_t *qline = reinterpret_cast<const uint32_t *>(qmeta + fl_pos + grp);  // .x of entry fl_pos + grp + 4r
    uint32_t lid[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) lid[r] = qline[r * 16];  // (stale entries past n_new are read but never used)
    if (n_new == 32) {
#pragma unroll
      for (int r = 0; r < 8; ++r)
        cp_async16(((r & 1) ? d_odd : d_even) + (uint32_t)(r * 512), line_src + ((uint64_t)lid[r] << 7));
    } else {
#pragma unroll
      for (int r = 0; r < 8; ++r)
        if ((uint32_t)(4 * r + grp) < n_new)
          cp_async16(((r & 1) ? d_odd : d_even) + (uint32_t)(r * 512), line_src + ((uint64_t)lid[r] << 7));
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");
    fl_n = n_new;
    pd_n -= n_new;
  };
  // COMPLETE the round in flight: every lane < fl_n owns row `lane` of the tile
  auto complete_round = [&]() {
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncwarp();
    if ((uint32_t)lane < fl_n) {
      const uint4 kq = qkey[fl_pos + lane], mq = qmeta[fl_pos + lane];
      const uint32_t line = mq.x, cnt = mq.z, bit = mq.w;
      u128 canon, x43;
      if constexpr (MODE == 0) {
        canon = u128_of(kq);
      } else {
        x43 = u128_of(kq);
        canon = canon_only(mask128(shr128(x43, 2 * tail), 2 * k), k);
      }
      const uint4 *mine = tile + lane * 8;
      const int sw = lane & 7;
      const uint32_t fw = reinterpret_cast<const uint32_t *>(mine + ((bit >> 7) ^ sw))[(bit >> 5) & 3];
      const bool bf_hit = (fw >> (bit & 31u)) & 1u;
      const uint32_t c0 = (uint32_t)canon.lo, c1 = (uint32_t)(canon.lo >> 32), c2 = (uint32_t)canon.hi,
                     c3 = (uint32_t)(canon.hi >> 32);
      int slot = -1;
      uint32_t flag_w = 0;
#pragma unroll
      for (int s = 0; s < LINE_KEYS; ++s) {
        const uint4 p = mine[(2 + s) ^ sw];
        if (((p.x ^ c0) | (p.y ^ c1) | ((p.z ^ c2) & mz) | ((p.w ^ c3) & mw)) == 0) slot = s;
        if (s == LINE_KEYS - 1) flag_w = inl ? p.z : p.w;
      }
      // ---- ref_bf.increment ----
      if (slot >= 0) {
        uint32_t *cp = inl ? line_words(v, line) + 8 + 4 * slot + 3 : v.key_counts + (uint64_t)line * LINE_KEYS + (uint32_t)slot;
        atomicAdd(cp, cnt);
      } else if (flag_w >> 31) {  // line overflowed at index time: the key may live in the overflow table
        const int64_t os = ovf_find(v, canon);
        if (os >= 0) atomicAdd(v.ovf_counts + os, cnt);
      }
      // ---- bf.increment unless the context filter vetoes it ----
      if (bf_hit) {
        // counter of the bit: number j of the set bit inside the line, rank of the line
        const uint32_t ws = bit >> 5, below = (1u << (bit & 31u)) - 1u;
        const uint4 b0 = mine[0 ^ sw], b1 = mine[1 ^ sw];
        const uint32_t wx[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
        int j = 0;
#pragma unroll
        for (uint32_t x = 0; x < 8; ++x) j += __popc(wx[x] & (x < ws ? 0xFFFFFFFFu : (x == ws ? below : 0u)));
        const uint32_t rank = reinterpret_cast<const uint32_t *>(mine + (7 ^ sw))[0];
        uint32_t *ap = j < LINE_INLINE_ALT ? line_words(v, line) + LINE_W_RANK + 1 + j
                                           : v.bf_counts + (uint64_t)rank + (uint64_t)j;
        if constexpr (MODE == 0) x43 = u128_of(__ldg(src.kmers + mq.y));
        const uint32_t pos = src.hit_buf ? atomicAdd(hitc, 1u) : 0xFFFFFFFFu;
        if (pos < src.seg_cap) {  // recorded; k_scan_hits finishes it
          uint4 *e = src.hit_buf + ((uint64_t)warp_id * src.seg_cap + pos) * 2;
          const uint64_t a64 = reinterpret_cast<uint64_t>(ap);
          e[0] = uint4_of(x43);
          e[1] = make_uint4((uint32_t)a64, (uint32_t)(a64 >> 32), cnt, 0u);
        } else {
          u128 c43;
          uint64_t h43;
          if constexpr (REFK > 0)
            h43 = canon_hash_lut<REFK>(x43, &c43, tab);
          else
            h43 = canon_hash_rt(x43, ref_k, &c43);
          if (!ctx_test(v, bf_index(v, h43))) atomicAdd(ap, cnt);
        }
      }
    }
    fl_pos = wrap(fl_pos + fl_n);
    fl_n = 0;
  };
  if constexpr (MODE == 0) {  // asynchronous rounds, two k-mers per lane
    // A context k-mer of up to 48 bases never uses the top word of its 16 bytes: it is not loaded at all.  (Loaded
    // and unused, its register gets recycled as a temporary while the 16-byte load is still in flight, and that
    // write-after-write wait exposes the whole load latency -- ncu, profiles/round2_k1.md.)
    constexpr bool SHORT_CTX = REFK > 0 && REFK <= 48;
    auto load_kmer = [&](uint32_t i) {
      if constexpr (SHORT_CTX) {
        const uint2 lo = ldg_na(reinterpret_cast<const uint2 *>(src.kmers + i));
        return make_uint4(lo.x, lo.y, ldg_na(reinterpret_cast<const uint32_t *>(src.kmers + i) + 2), 0u);
      } else {
        return __ldg(src.kmers + i);
      }
    };
    constexpr int ILP = S.ilp;
    constexpr uint32_t W = 32u * ILP;  // k-mers per warp and iteration
    uint32_t base = warp_id * W;
    uint4 q_cur[ILP];
    uint32_t c_cur[ILP];
#pragma unroll
    for (int u = 0; u < ILP; ++u) {
      const uint32_t i = base + 32u * u + lane;
      q_cur[u] = i < n32 ? load_kmer(i) : make_uint4(0, 0, 0, 0);
      c_cur[u] = i < n32 ? ldg_na(src.counts + i) : 0u;
    }
    for (;; base += step * ILP) {
      more = more && base < n32;
      if (more) {
        // the next batch's k-mers are requested before this one is hashed and used one iteration later
        u128 x43[ILP], canon[ILP];
        uint32_t cnt[ILP], idx_hi[ILP], bit[ILP];
        bool need[ILP];
#pragma unroll
        for (int u = 0; u < ILP; ++u) {
          x43[u] = u128_of(q_cur[u]);
          cnt[u] = c_cur[u];
        }
        const uint32_t nb = base + step * ILP;
        if (nb < n32) {
#pragma unroll
          for (int u = 0; u < ILP; ++u) {
            const uint32_t i = nb + 32u * u + lane;
            q_cur[u] = i < n32 ? load_kmer(i) : make_uint4(0, 0, 0, 0);
            c_cur[u] = i < n32 ? ldg_na(src.counts + i) : 0u;
          }
          if (lane < 5 * ILP && nb + step * ILP < n32) {  // and the batch after that into L2 (k-mers, then counts)
            const char *pf = lane < 4 * ILP
                                 ? reinterpret_cast<const char *>(src.kmers + nb + step * ILP) + lane * 128
                                 : reinterpret_cast<const char *>(src.counts + nb + step * ILP) + (lane - 4 * ILP) * 128;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(pf));
          }
        }
        uint64_t idx[ILP];
#pragma unroll
        for (int u = 0; u < ILP; ++u) {  // (straight-line code over the independent chains: they interleave)
          const u128 x35 = mask128(shr128(x43[u], 2 * tail), 2 * k);
          uint64_t h;
          if constexpr (K > 0)
            h = canon_hash_lut<K>(x35, &canon[u], tab);
          else
            h = canon_hash_rt(x35, k, &canon[u]);
          idx[u] = bf_index(v, h);
        }
        // occupancy pre-filter (L2): most probe lines hold nothing for a given k-mer; those are never fetched
        uint32_t ob[ILP];  // bit inside the 16-byte piece
        if (v.occ) {
#pragma unroll
          for (int u = 0; u < ILP; ++u) {
            const uint64_t o = idx[u] >> v.occ_shift;
            ob[u] = (uint32_t)o & 127u;
            cp_async16(oslot_addr + (uint32_t)(u * 512), reinterpret_cast<const char *>(v.occ) + ((o >> 7) << 4));
          }
          asm volatile("cp.async.commit_group;\n" ::: "memory");
          asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        }
#pragma unroll
        for (int u = 0; u < ILP; ++u) {
          bool hit = true;
          if (v.occ) hit = (reinterpret_cast<const uint32_t *>(oslot + u * 32)[ob[u] >> 5] >> (ob[u] & 31u)) & 1u;
          need[u] = base + 32u * u + lane < n32 && hit;
          idx_hi[u] = (uint32_t)(idx[u] >> 8);  // n_lines < 2^32 (bf_bits < 2^40)
          bit[u] = (uint32_t)(idx[u] & 255);
        }
        // all k-mers of the lane go into the ring in one go
        const uint32_t lt = (1u << lane) - 1u, at = fl_pos + fl_n + pd_n;
        uint32_t m[ILP], off = 0;
#pragma unroll
        for (int u = 0; u < ILP; ++u) m[u] = __ballot_sync(0xffffffffu, need[u]);
#pragma unroll
        for (int u = 0; u < ILP; ++u) {
          if (need[u]) {
            const uint32_t e = wrap(at + off + (uint32_t)__popc(m[u] & lt));
            qkey[e] = uint4_of(canon[u]);
            qmeta[e] = make_uint4(idx_hi[u], base + 32u * u + lane, cnt[u], bit[u]);
          }
          off += (uint32_t)__popc(m[u]);
        }
        pd_n += off;
        // a full ring turns: the round in flight is finished (started a batch or more ago: its lines have landed),
        // the next one started (again when the batches passed the pre-filter almost whole)
#pragma unroll 1
        while (pd_n >= 32) {
          if (fl_n) complete_round();
          start_round();
        }
      } else {  // the tail: nothing more to hash
        if (fl_n) complete_round();
        if (pd_n) start_round();
        if (pd_n == 0 && fl_n == 0) break;
      }
    }
  } else {  // synchronous rounds, one KMC record per lane
    for (uint32_t base = warp_id * 32;; base += step) {
      more = more && base < n32;
      if (more) {
        const uint32_t i = base + lane;
        bool live = i < n32;
        u128 x43, canon;
        // stage the warp's 32 records (contiguous bytes) in its shared-memory tile, then decode one per lane
        const int rec = src.suf_bytes + src.counter_size;
        const uint64_t byte0 = (uint64_t)base * (uint64_t)rec, start = byte0 & ~3ull;
        const int n_words = (int)((byte0 - start) + 32u * (uint32_t)rec + 3u) >> 2;
        __syncwarp();  // the previous probe round's reads of the tile are done
        uint32_t *stage = reinterpret_cast<uint32_t *>(tile);
        for (int w = lane; w < n_words; w += 32) stage[w] = __ldg(reinterpret_cast<const uint32_t *>(src.recs + start) + w);
        __syncwarp();
        const uint8_t *rb = reinterpret_cast<const uint8_t *>(stage) + (byte0 - start) + (uint32_t)lane * (uint32_t)rec;
        u128 suf = {0, 0};
        for (int j = 0; j < src.suf_bytes; ++j) {
          suf.hi = (suf.hi << 8) | (suf.lo >> 56);
          suf.lo = (suf.lo << 8) | rb[j];
        }
        uint64_t c64 = src.counter_size ? 0 : 1;
        for (int j = 0; j < src.counter_size; ++j) c64 |= (uint64_t)rb[src.suf_bytes + j] << (8 * j);
        __syncwarp();  // the tile is reused for the probe lines below
        // prefix of each record: one LUT search per warp in the common case (a prefix bucket spans many records)
        const uint64_t g = src.first_rec + i;
        const uint64_t g_first = src.first_rec + base;
        const uint64_t g_last = src.first_rec + (base + 31 < n32 ? base + 31 : n32 - 1);
        uint32_t pj = lut_bucket(src.lut, src.n_lut, g_first);
        if (__ldg(src.lut + pj + 1) <= g_last) pj = lut_bucket(src.lut, src.n_lut, live ? g : g_first);
        u128 pre = {(uint64_t)(pj & src.prefix_mask), 0};
        const int sh = 8 * src.suf_bytes;  // the suffix holds 4 * suf_bytes symbols
        if (sh >= 64) {
          pre.hi = pre.lo << (sh - 64);
          pre.lo = 0;
        } else {
          pre.hi = sh ? (pre.lo >> (64 - sh)) : 0;
          pre.lo <<= sh;
        }
        x43.lo = pre.lo | suf.lo;
        x43.hi = pre.hi | suf.hi;
        // CKMCFile::ReadNextKmer skips records whose count is outside [min_count, max_count]
        if (c64 < src.min_count || c64 > src.max_count) live = false;
        const uint32_t cnt = (uint32_t)c64;
        u128 x35 = mask128(shr128(x43, 2 * tail), 2 * k);
        uint64_t h;
        if constexpr (K > 0)
          h = canon_hash_lut<K>(x35, &canon, tab);
        else
          h = canon_hash_rt(x35, k, &canon);
        const uint64_t idx = bf_index(v, h);
        // occupancy pre-filter (L2): most probe lines hold nothing for a given k-mer; those are never fetched
        bool need = live;
        if (v.occ) {
          const uint64_t o = idx >> v.occ_shift;
          cp_async16(oslot_addr, reinterpret_cast<const char *>(v.occ) + ((o >> 7) << 4));
          asm volatile("cp.async.commit_group;\n" ::: "memory");
          asm volatile("cp.async.wait_group 0;\n" ::: "memory");
          need = live && ((reinterpret_cast<const uint32_t *>(oslot)[((uint32_t)o & 127u) >> 5] >> ((uint32_t)o & 31u)) & 1u);
        }
        const uint32_t need_mask = __ballot_sync(0xffffffffu, need);
        if (need) {
          const uint32_t e = (fl_pos + fl_n + pd_n + (uint32_t)__popc(need_mask & ((1u << lane) - 1u))) & (SCAN_Q - 1);
          qkey[e] = uint4_of(x43);  // (complete_round derives the canonical k-mer from the record's context k-mer)
          qmeta[e] = make_uint4((uint32_t)(idx >> 8), i, cnt, (uint32_t)(idx & 255));  // n_lines < 2^32 (bf_bits < 2^40)
        }
        pd_n += (uint32_t)__popc(need_mask);
      }
      if (pd_n >= 32 || (!more && pd_n)) {
        start_round();
        complete_round();
      }
      if (!more && pd_n == 0) break;
    }
  }
  if (src.hit_buf) {
    __syncwarp();
    if (lane == 0) src.hit_counts[warp_id] = *hitc < src.seg_cap ? *hitc : src.seg_cap;
  }
}

// second half of the scan for the recorded filter hits: 43-mer hash -> context filter -> counter
template <int REFK>
__global__ void __launch_bounds__(256) k_scan_hits(const uint4 *__restrict__ hit_buf, const uint32_t *__restrict__ hit_counts,
                                                  uint32_t n_warps, uint32_t seg_cap, DevView v) {
  __shared__ uint32_t tab[256];
  tab[threadIdx.x] = expand4(threadIdx.x);
  __syncthreads();
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t w = (uint32_t)(t / seg_cap), slot = (uint32_t)(t % seg_cap);
  if (w >= n_warps || slot >= __ldg(hit_counts + w)) return;
  const uint4 a = __ldg(hit_buf + t * 2), b = __ldg(hit_buf + t * 2 + 1);
  u128 x43 = u128_of(a), c43;
  uint32_t *ap = reinterpret_cast<uint32_t *>((uint64_t)b.x | ((uint64_t)b.y << 32));
  uint64_t h43;
  if constexpr (REFK > 0)
    h43 = canon_hash_lut<REFK>(x43, &c43, tab);
  else
    h43 = canon_hash_rt(x43, v.ref_k, &c43);
  if (!ctx_test(v, bf_index(v, h43))) atomicAdd(ap, b.z);
}

// ---------------------------------------------------------------------------
// Sample sets (include/malva_gpu.h, mg_samples_*): the counters of up to 32 samples side by side.  Every counter a
// signature k-mer can read has a ROW that depends on the index only:
//   [0, bf_ones)                    a set bit of bf: its rank + j                     (BF::get_count)
//   [key_base, key_base + keys)     a ref key held by a probe line: key_rank[L] + slot (KMAP::get_count)
//   [ovf_base, ovf_base + ovf cap)  a slot of the overflow table
// and a sample is a column of u32 counts over those rows.  The set is row-major, mat[row * g + s]: the g counts of
// a row share one 128-byte line, so a signature k-mer costs one probe line and one count line for all samples.
// ---------------------------------------------------------------------------
constexpr uint32_t NO_ROW = 0xFFFFFFFFu;
constexpr int SAMPLE_SET_MAX = 32;
struct SampleView {
  uint32_t *mat;
  const uint32_t *key_rank;  // keys held by the lines before line L
  uint64_t key_base, ovf_base;
  int g;
};
__device__ __forceinline__ uint32_t *sample_cell(const SampleView &sv, uint64_t row, int col) {
  return sv.mat + row * (uint64_t)sv.g + (uint64_t)col;
}

// mg_samples_take, dense part: src[i] (bf_counts, ovf_counts) -> row row0 + i of column col; src is zeroed
__global__ void __launch_bounds__(256) k_samples_take_dense(uint32_t *__restrict__ src, uint64_t n, uint64_t row0,
                                                           SampleView sv, int col) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const uint32_t c = src[i];
    *sample_cell(sv, row0 + i, col) = c;
    if (c) src[i] = 0;
  }
}
// mg_samples_take, the counters inside the probe lines (k_counters_xfer's walk: eight lanes per line, one uint4
// each): the inline counters of set bits 0..2 and the key counts go to column col and are zeroed in place.  Runs
// after k_samples_take_dense of bf_counts, whose entries for set bits 0..2 of a line are not live counters.
__global__ void __launch_bounds__(256) k_samples_take_lines(DevView v, SampleView sv, int col) {
  const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint64_t line = t >> 3;
  const int sub = (int)(t & 7);
  const bool ok = line < v.n_lines;
  const uint4 q = ok ? v.lines[line * LINE_U4 + (uint64_t)sub] : make_uint4(0, 0, 0, 0);
  const uint32_t pc = sub < 2 ? (uint32_t)(__popc(q.x) + __popc(q.y) + __popc(q.z) + __popc(q.w)) : 0u;
  const int g0 = (int)(threadIdx.x & 24);
  const uint32_t n_alt = __shfl_sync(0xffffffffu, pc, g0) + __shfl_sync(0xffffffffu, pc, g0 + 1);
  if (!ok) return;
  uint32_t *w = line_words(v, line);
  if (sub == 7) {
    const uint32_t c[3] = {q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < LINE_INLINE_ALT; ++j)
      if ((uint32_t)j < n_alt) *sample_cell(sv, (uint64_t)q.x + (uint64_t)j, col) = c[j];
    if (q.y | q.z | q.w) v.lines[line * LINE_U4 + 7] = make_uint4(q.x, 0u, 0u, 0u);
  } else if (sub >= 2) {
    const int s = sub - 2;
    if (key_empty(v, key_of(v, q))) return;
    const uint64_t row = sv.key_base + (uint64_t)sv.key_rank[line] + (uint64_t)s;
    uint32_t *cp = v.inline_counts ? w + 8 + 4 * s + 3 : v.key_counts + line * LINE_KEYS + (uint64_t)s;
    const uint32_t c = v.inline_counts ? q.w : *cp;
    *sample_cell(sv, row, col) = c;
    if (c) *cp = 0;
  }
}

// ---------------------------------------------------------------------------
// K4: signature look-ups (BF::get_count / KMAP::get_count) + coverage.  One probe line per look-up: the count of a
// ref key is in its slot, the counter of an alt bit in words 29..31 of the line (index.cuh).  Every look-up decodes
// the line with line_alt / line_key (index.cuh) and ends in one of the four readers below: a count, or a ROW of a
// sample set.
// ---------------------------------------------------------------------------
// BF::get_count (u16; RAW: the u32 accumulator, for replicas that sum their look-ups first)
template <bool RAW, class At>
__device__ __forceinline__ int32_t alt_count(const DevView &v, At at, uint32_t bit) {
  if (!v.bf_counts) return 0;  // write mode: no counters yet (bloom_filter.hpp:115-125)
  int j;
  uint4 m;
  if (!line_alt(at, bit, &j, &m)) return 0;
  const uint32_t c = j == 0 ? m.y : (j == 1 ? m.z : (j == 2 ? m.w : __ldg(v.bf_counts + (uint64_t)m.x + (uint64_t)j)));
  return RAW ? (int32_t)c : (int32_t)(c & 0xFFFFu);
}
template <class At>
__device__ __forceinline__ uint32_t alt_row(At at, uint32_t bit) {
  int j;
  uint4 m;
  return line_alt(at, bit, &j, &m) ? m.x + (uint32_t)j : NO_ROW;
}
// KMAP::get_count of ref key `canon`, whose bf index lies in probe line `line`
template <int K, class At>
__device__ __forceinline__ int32_t key_count(const DevView &v, At at, uint64_t line, u128 canon) {
  uint32_t w3;
  bool ovf;
  const int slot = line_key<K>(v, at, canon, &w3, &ovf);
  if (slot >= 0) return inline_keys<K>(v) ? (int32_t)w3 : (int32_t)__ldg(v.key_counts + line * LINE_KEYS + (uint32_t)slot);
  if (!ovf) return 0;
  const int64_t os = ovf_find(v, canon);
  return os < 0 ? 0 : (int32_t)__ldg(v.ovf_counts + os);
}
template <int K, class At>
__device__ __forceinline__ uint32_t key_row(const DevView &v, const SampleView &sv, At at, uint64_t line, u128 canon) {
  uint32_t w3;
  bool ovf;
  const int slot = line_key<K>(v, at, canon, &w3, &ovf);
  if (slot >= 0) return (uint32_t)(sv.key_base + __ldg(sv.key_rank + line) + (uint32_t)slot);
  if (!ovf) return NO_ROW;
  const int64_t os = ovf_find(v, canon);
  return os < 0 ? NO_ROW : (uint32_t)(sv.ovf_base + (uint64_t)os);
}
// the weight of sample s at counter row `row` (NO_ROW, or s past the set: 0): KMAP::get_count's int for a ref key,
// BF::get_count's uint16_t otherwise
__device__ __forceinline__ int32_t sample_weight(const SampleView &sv, uint32_t row, int s, bool ref) {
  const uint32_t c = row != NO_ROW && s < sv.g ? __ldg(sv.mat + (uint64_t)row * (uint64_t)sv.g + (uint64_t)s) : 0u;
  return (int32_t)(ref ? c : (c & 0xFFFFu));
}

// k-mer i of an ASCII pool (any length, any symbols), resolved byte-exactly as the reference does: a ref key (KMAP)
// must be exactly k symbols of ACGT; the Bloom filters hash the canonical ASCII bytes of whatever length was given
// (BF::_get_hash).  Returns 1 with *idx = the bf index (and *canon = the canonical key of a ref key), -1 for a ref key
// that is not k x ACGT (never in the device map: the host keeps those), 0 for a k-mer longer than 128 bytes (flagged
// in scalars[3]).
__device__ __forceinline__ int ascii_kmer(const uint8_t *__restrict__ pool, const uint64_t *__restrict__ off, uint64_t i,
                                          bool ref, const DevView &v, unsigned long long *scalars, uint64_t *idx,
                                          u128 *canon) {
  const uint64_t b = off[i];
  const int len = (int)(off[i + 1] - b);
  if (len > 128) {
    atomicExch(&scalars[3], 1ull);
    return 0;
  }
  uint8_t s[128];
  for (int j = 0; j < len; ++j) s[j] = pool[b + j];
  u128 x;
  uint64_t h;
  if (ref) {
    if (!pack_ascii(s, len, v.k, &x)) return -1;
    h = canon_hash_rt(x, v.k, canon);
  } else {
    const bool regular = len >= 1 && len <= 64 && pack_ascii(s, len, len, &x);
    h = regular ? canon_hash_rt(x, len, canon) : hash_ascii(s, len);
  }
  *idx = bf_index(v, h);
  return 1;
}

// The ASCII look-ups of mg_get_counts and mg_test_keys:
// mode 0: get_count  (is_ref selects KMAP/BF, out = int32 count)
// mode 1: test_key on filter/table `which` (0 bf, 1 context_bf, 2 ref_bf; out = 0/1, -1 = irregular KMAP key)
__global__ void __launch_bounds__(128) k_lookup(const uint8_t *__restrict__ pool, const uint64_t *__restrict__ off,
                                               const uint8_t *__restrict__ is_ref, uint64_t n, DevView v, int mode,
                                               int which, int32_t *__restrict__ out, unsigned long long *scalars) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const bool use_table = mode == 0 ? (is_ref && is_ref[i] != 0) : (which == 2);
  uint64_t idx = 0;
  u128 canon;
  const int r = ascii_kmer(pool, off, i, use_table, v, scalars, &idx, &canon);
  if (r <= 0) {
    out[i] = (mode == 1 && r < 0) ? -1 : 0;  // irregular keys are resolved on the host (always count 0)
    return;
  }
  const uint64_t line = idx >> 8;
  const auto at = line_at(v, line);
  if (use_table && mode == 0) {
    out[i] = key_count<0>(v, at, line, canon);
  } else if (use_table) {
    uint32_t w3;
    bool ovf;
    out[i] = line_key<0>(v, at, canon, &w3, &ovf) >= 0 || (ovf && ovf_find(v, canon) >= 0);
  } else if (mode == 1) {
    out[i] = which == 1 ? ctx_test(v, idx) : bf_test(v, idx);
  } else {
    out[i] = alt_count<false>(v, at, (uint32_t)(idx & 255));
  }
}

// What a look-up of a packed batch writes per k-mer: BF::get_count / KMAP::get_count (COUNT); the same with the bf
// counters as the u32 accumulators they are (RAW: partial results of replicas are summed first, the u16 wrap of
// int_vector<16> is applied to the sum: k_mask_alt); or the weights of every sample of the sample set, sample-major,
// out[s * n + i] (SAMPLES).
enum LookupOut { OUT_COUNT, OUT_RAW, OUT_SAMPLES };

// Packed signature k-mers (exactly k symbols of ACGT, the form the host enumerator emits): {lo, hi} words;
// hi bit 62 = k-mer of allele slot 0 (looked up in ref_bf), hi bit 63 = irregular (not k x ACGT: resolved by
// k_lookup_irr from the side pool).  16 bytes in, 4 bytes out, one probe line per k-mer.
// A warp takes 32 k-mers at a time: every lane hashes one, then the 32 probe lines are gathered into the warp's
// 4 KB shared-memory tile exactly like a round of the sample scan (eight LDGSTS rounds, four whole lines each, the
// line of row L announced by a shuffle), and every lane reads its own row.  One thread fetching its line by itself
// -- five 16-byte loads for a ref key, three for an alt bit -- cost five (three) L1 tag look-ups per line and ran at
// 45 % of the device's random-line rate with the load queues full (ncu, profiles/round2_k4.md).
// SAMPLES: every lane resolves the ROW of its k-mer instead, then the warp reads the 32 rows one after the other with
// the lanes on the samples (one coalesced line per k-mer), transposes them through shared memory and writes 128 bytes
// per store.
constexpr int LOOKUP_THREADS = 256;
constexpr int LOOKUP_SMEM = (LOOKUP_THREADS / 32) * 4096;
__host__ __device__ constexpr int lookup_smem(int out) {  // + the 32 x 33 transposition buffer of every warp
  return LOOKUP_SMEM + (out == OUT_SAMPLES ? (LOOKUP_THREADS / 32) * 32 * 33 * 4 : 0);
}

template <int K, int OUT>
__global__ void __launch_bounds__(LOOKUP_THREADS) k_lookup_packed(const uint4 *__restrict__ kmers, uint64_t n, DevView v,
                                                                 int32_t *__restrict__ out, SampleView sv) {
  extern __shared__ uint4 lk_sm[];
  const int lane = threadIdx.x & 31, sub = lane & 7, grp = lane >> 3;
  uint4 *tile = lk_sm + (threadIdx.x >> 5) * 256;
  const uint32_t tile_addr = (uint32_t)__cvta_generic_to_shared(tile);
  const uint32_t d_even = tile_addr + (uint32_t)(grp * 128 + ((sub ^ grp) * 16));
  const uint32_t d_odd = tile_addr + (uint32_t)(grp * 128 + ((sub ^ (grp + 4)) * 16));
  const char *line_src = reinterpret_cast<const char *>(v.lines) + sub * 16;
  const int k = K > 0 ? K : v.k;
  const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  for (uint64_t base = warp0 * 32; base < n; base += n_warps * 32) {
    const uint64_t i = base + (uint64_t)lane;
    const uint4 q = i < n ? __ldg(kmers + i) : make_uint4(0, 0, 0, 0x80000000u);
    const bool active = !(q.w >> 31);  // (past the end, or irregular: nothing to fetch)
    const bool is_ref = (q.w >> 30) & 1u;
    u128 canon;
    const uint64_t h = canon_hash_k<K>(mask128(u128_of(q), 2 * k), k, &canon);
    const uint64_t idx = bf_index(v, h);
    const uint32_t line = (uint32_t)(idx >> 8), bit = (uint32_t)(idx & 255);
    const uint32_t act = __ballot_sync(0xffffffffu, active);
    __syncwarp();  // the previous batch's reads of the tile (and of the transposition buffer) are done
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const uint32_t lid = __shfl_sync(0xffffffffu, line, 4 * r + grp);
      if ((act >> (4 * r + grp)) & 1u)
        cp_async16(((r & 1) ? d_odd : d_even) + (uint32_t)(r * 512), line_src + ((uint64_t)lid << 7));
    }
    asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;\n" ::: "memory");
    __syncwarp();
    const uint4 *mine = tile + lane * 8;
    const int sw = lane & 7;
    const auto at = [mine, sw](int u) { return mine[u ^ sw]; };
    if constexpr (OUT != OUT_SAMPLES) {
      if (!active) continue;
      out[i] = is_ref ? key_count<K>(v, at, line, canon) : alt_count<OUT == OUT_RAW>(v, at, bit);
    } else {
      const uint32_t row = !active ? NO_ROW : (is_ref ? key_row<K>(v, sv, at, line, canon) : alt_row(at, bit));
      const uint32_t refs = __ballot_sync(0xffffffffu, is_ref);
      uint32_t *tr = reinterpret_cast<uint32_t *>(lk_sm + (LOOKUP_THREADS / 32) * 256) + (threadIdx.x >> 5) * 32 * 33;
#pragma unroll 8
      for (int r = 0; r < 32; ++r)  // the counts of the 32 rows, lanes = samples
        tr[r * 33 + lane] = (uint32_t)sample_weight(sv, __shfl_sync(0xffffffffu, row, r), lane, (refs >> r) & 1u);
      __syncwarp();
      if (i < n)
        for (int s = 0; s < sv.g; ++s) out[(uint64_t)s * n + i] = (int32_t)tr[lane * 33 + s];
    }
  }
}

// The irregular k-mers of a packed batch: k-mer j of the side pool is k-mer irr_kmer[j] of the batch (whose bit 62
// says ref or alt), resolved byte-exactly; written where k_lookup_packed, with the same OUT, writes that k-mer.  An
// irregular alt k-mer can hit a set bit of bf; an irregular ref key is never in the device map and counts 0.
template <int OUT>
__global__ void __launch_bounds__(128) k_lookup_irr(const uint8_t *__restrict__ pool, const uint64_t *__restrict__ off,
                                                   const uint32_t *__restrict__ irr_kmer, uint64_t n_irr,
                                                   const uint4 *__restrict__ kmers, uint64_t n, DevView v,
                                                   int32_t *__restrict__ out, SampleView sv, unsigned long long *scalars) {
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_irr) return;
  const uint64_t i = irr_kmer[j];
  const bool ref = ((kmers[i].w >> 30) & 1u) != 0;
  uint64_t idx = 0;
  u128 canon;
  const bool found = ascii_kmer(pool, off, j, ref, v, scalars, &idx, &canon) > 0;
  const uint64_t line = idx >> 8;
  const uint32_t bit = (uint32_t)(idx & 255);
  const auto at = line_at(v, line);
  if constexpr (OUT != OUT_SAMPLES) {
    out[i] = !found ? 0 : (ref ? key_count<0>(v, at, line, canon) : alt_count<OUT == OUT_RAW>(v, at, bit));
  } else {
    const uint32_t row = !found ? NO_ROW : (ref ? key_row<0>(v, sv, at, line, canon) : alt_row(at, bit));
    for (int s = 0; s < sv.g; ++s) out[(uint64_t)s * n + i] = sample_weight(sv, row, s, ref);
  }
}

// BF::get_count's uint16_t of summed raw bf counters (the k-mers that are not flagged as ref-allele k-mers)
__global__ void __launch_bounds__(256) k_mask_alt(const uint4 *__restrict__ kmers, uint64_t n, int32_t *__restrict__ w) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (!((__ldg(reinterpret_cast<const uint32_t *>(kmers + i) + 3) >> 30) & 1u)) w[i] &= 0xFFFF;
}

// set_coverages (main.cpp:157-182): per allele slot, max over signatures of the order-dependent integer
// running mean of the non-zero k-mer weights
__global__ void __launch_bounds__(128) k_coverage(const int32_t *__restrict__ w, const uint32_t *__restrict__ sig_kmer_off,
                                                 const uint32_t *__restrict__ allele_sig_off, uint64_t n_alleles,
                                                 uint32_t *__restrict__ cov) {
  uint64_t a = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= n_alleles) return;
  uint32_t allele_cov = 0;
  for (uint64_t s = allele_sig_off[a]; s < allele_sig_off[a + 1]; ++s) {
    uint32_t curr = 0;
    int n = 0;
    for (uint64_t q = sig_kmer_off[s]; q < sig_kmer_off[s + 1]; ++q) {
      int32_t wi = w[q];
      if (wi > 0) {
        curr = (curr * (uint32_t)n + (uint32_t)wi) / (uint32_t)(n + 1);
        ++n;
      }
    }
    if (curr > allele_cov) allele_cov = curr;
  }
  cov[a] = allele_cov;
}

// ---------------------------------------------------------------------------
// K5: genotype likelihoods + posterior arg-max (var_block.hpp:224-330, 367-394)
// ---------------------------------------------------------------------------
// log_table: glibc's log of small integers (geno.cuh log_int); NULL on the host self-test path
MG_HD int genotype_one(const uint32_t *cov, const float *freq, int n, float err, int max_cov, bool haploid,
                       const double *log_table, double *lik, int *status, int *best_gt, int *gq) {
  if (n == 0) {  // a variant without alleles has no genotype and no likelihood slot (include/malva_gpu.h)
    *status = 2;
    *best_gt = 0;
    *gq = 0;
    return 0;
  }
  int ng = 0;
  for (int i = 0; i < n; ++i)
    if ((int)cov[i] > max_cov) lik[ng++] = 0.0;  // one {best,0} per offending allele
  if (ng) {
    *status = 1;
    *best_gt = 0;
    *gq = 0;
    return ng;
  }
  if (n == 1) {
    lik[0] = 1.0;
    *status = 0;
    *best_gt = 0;
    *gq = 100;
    return 1;
  }
  uint32_t tot = 0;
  for (int i = 0; i < n; ++i) tot += cov[i];
  if (tot == 0) {
    lik[0] = 0.0;
    *status = 2;
    *best_gt = 0;
    *gq = 0;
    return 1;
  }
  GenoConsts c = geno_consts(err, n);
  double total = 0.0;
  for (int g1 = 0; g1 < n; ++g1) {
    for (int g2 = g1; g2 < n; ++g2) {
      if (haploid && g2 != g1) break;
      double p = (g1 == g2) ? geno_hom(cov[g1], tot, freq[g1], c, log_table)
                            : geno_het(cov[g1], cov[g2], tot, freq[g1], freq[g2], n, c, log_table);
      lik[ng++] = p;
      total = f64_add(total, p);
    }
  }
  double best = 0.0;
  int bi = 0;
  for (int i = 0; i < ng; ++i) {
    double q = lik[i] / total;
    if (q > best) {
      best = q;
      bi = i;
    }
  }
  *status = 0;
  *best_gt = bi;
  *gq = (int)round(f64_mul(best, 100.0));
  return ng;
}

// lik_off != nullptr: the likelihoods of variant vi go to lik[lik_off[vi] ..] (the caller reads them back);
// lik_off == nullptr: nobody reads them, the slots are bump-allocated from `cursor` (scratch)
__global__ void __launch_bounds__(128) k_genotype(const uint32_t *__restrict__ cov, const float *__restrict__ freq,
                                                 const uint32_t *__restrict__ var_allele_off,
                                                 const uint64_t *__restrict__ lik_off, unsigned long long *cursor,
                                                 uint64_t n_variants, float err, int max_cov, int haploid,
                                                 const double *__restrict__ log_table,
                                                 double *__restrict__ lik, int32_t *__restrict__ n_gts,
                                                 int32_t *__restrict__ status, int32_t *__restrict__ best_gt,
                                                 int32_t *__restrict__ gq) {
  uint64_t vi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = vi < n_variants;
  uint64_t a0 = live ? (uint64_t)var_allele_off[vi] : 0;
  int n = live ? (int)(var_allele_off[vi + 1] - a0) : 0;
  uint64_t lo;
  if (lik_off) {
    lo = live ? lik_off[vi] : 0;
  } else {
    // one atomic per warp: an inclusive scan of the lanes' slot counts, the last lane reserves the total
    const uint32_t g = (uint32_t)(haploid ? n : n * (n + 1) / 2);
    const uint32_t slots = live ? (g > (uint32_t)n ? g : (uint32_t)n) : 0u;
    const int lane = threadIdx.x & 31;
    uint32_t incl = slots;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    unsigned long long base = 0;
    if (lane == 31) base = atomicAdd(cursor, (unsigned long long)incl);
    base = __shfl_sync(0xffffffffu, base, 31);
    lo = base + (incl - slots);
  }
  if (!live) return;
  int st, bg, q;
  int ng = genotype_one(cov + a0, freq + a0, n, err, max_cov, haploid != 0, log_table, lik + lo, &st, &bg, &q);
  n_gts[vi] = ng;
  status[vi] = st;
  best_gt[vi] = bg;
  gq[vi] = q;
}

// ---------------------------------------------------------------------------
// index image export / import (the index file of `malva-geno index`, main.cpp:406-412, 455-461):
// filters travel as sorted lists of set-bit indices, ref_bf as a list of packed keys
// ---------------------------------------------------------------------------
// one thread per 256-bit unit; offs = exclusive scan of the per-unit popcounts
__global__ void __launch_bounds__(256) k_emit_bits(const uint32_t *__restrict__ words, uint64_t n_units, int stride_u32,
                                                  const uint32_t *__restrict__ offs, uint64_t n_bits,
                                                  uint64_t *__restrict__ out) {
  uint64_t u = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (u >= n_units) return;
  uint64_t o = offs[u];
  for (int w = 0; w < 8; ++w) {
    uint32_t x = words[u * (uint64_t)stride_u32 + (uint64_t)w];
    while (x) {
      int b = __ffs(x) - 1;
      x &= x - 1;
      uint64_t idx = u * 256 + (uint64_t)w * 32 + (uint64_t)b;
      if (idx < n_bits) out[o++] = idx;
    }
  }
}
__global__ void __launch_bounds__(256) k_set_bits(const uint64_t *__restrict__ idx, uint64_t n, uint64_t n_bits,
                                                 uint32_t *words_rw, int as_lines, DevView v, uint32_t *occ_rw) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint64_t b = idx[i];
  if (b >= n_bits) return;
  if (as_lines) occ_set(v, occ_rw, b);
  uint32_t *w = as_lines ? words_rw + (b >> 8) * 32 + ((b & 255) >> 5) : words_rw + (b >> 5);
  atomicOr(w, 1u << (b & 31));
}
// every non-empty key slot of the probe lines (n_slots = 5 * n_lines) or of the overflow table
__global__ void __launch_bounds__(256) k_emit_keys(DevView v, uint64_t ovf_cap, unsigned long long *counter,
                                                  u128 *__restrict__ out, uint64_t cap) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t n_slots = v.n_lines * LINE_KEYS;
  u128 key;
  if (i < n_slots) {
    key = key_of(v, v.lines[(i / LINE_KEYS) * LINE_U4 + 2 + (i % LINE_KEYS)]);
  } else if (i < n_slots + ovf_cap) {
    key = v.ovf_keys[i - n_slots];
    key.hi &= v.key_hi_mask;
  } else {
    return;
  }
  if (key_empty(v, key)) return;
  unsigned long long o = atomicAdd(counter, 1ull);
  if (o < cap) out[o] = key;
}

// ---------------------------------------------------------------------------
// roofline diagnostics: measured ceilings on this device (bench.py records them)
//   k_diag_random  : independent random reads, `gran` separate 4-byte loads inside one aligned
//                    gran*32-byte unit (1, 2 or 4 sectors)
//   k_diag_lines   : random 128-byte lines, each fetched by 8 lanes x 16 B in ONE coalesced request
//                    (the access pattern of k_scan)
//   k_diag_stream  : streaming 16-byte reads
// ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_diag_random(const uint32_t *__restrict__ buf, uint64_t n_units, int gran,
                                                    uint64_t per_thread, uint32_t *sink) {
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t s = (t + 1) * GOLD;
  uint32_t acc = 0;
#pragma unroll 4
  for (uint64_t i = 0; i < per_thread; ++i) {
    s ^= s >> 29;
    s *= 0xBF58476D1CE4E5B9ULL;
    s ^= s >> 32;
    uint64_t unit = mulhi64(s, n_units);  // uniform in [0, n_units)
    const uint32_t *p = buf + unit * 8 * (uint64_t)gran;
    acc += __ldg(p);
    if (gran >= 2) acc += __ldg(p + 8);
    if (gran >= 4) acc += __ldg(p + 16) + __ldg(p + 24);
    s += GOLD;
  }
  if (acc == 0x12345678u) *sink = acc;
}
__global__ void __launch_bounds__(256) k_diag_lines(const uint4 *__restrict__ buf, uint64_t n_units, int lanes_log2,
                                                   uint64_t per_group, uint32_t *sink) {
  // groups of 2^lanes_log2 lanes (8 / 4 / 2) read one random aligned unit of 128 / 64 / 32 bytes per instruction
  uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t s = ((t >> lanes_log2) + 1) * GOLD;  // one random stream per lane group
  const int sub = threadIdx.x & ((1 << lanes_log2) - 1);
  uint32_t acc = 0;
#pragma unroll 8
  for (uint64_t i = 0; i < per_group; ++i) {
    s ^= s >> 29;
    s *= 0xBF58476D1CE4E5B9ULL;
    s ^= s >> 32;
    uint64_t unit = mulhi64(s, n_units);
    uint4 q = __ldg(buf + (unit << lanes_log2) + sub);
    acc += q.x ^ q.y ^ q.z ^ q.w;
    s += GOLD;
  }
  if (acc == 0x12345678u) *sink = acc;
}
__global__ void __launch_bounds__(256) k_diag_stream(const uint4 *__restrict__ buf, uint64_t n16, uint32_t *sink) {
  uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  uint32_t acc = 0;
  for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += stride) {
    uint4 q = __ldg(buf + i);
    acc += q.x ^ q.y ^ q.z ^ q.w;
  }
  if (acc == 0x12345678u) *sink = acc;
}

}  // namespace mg
