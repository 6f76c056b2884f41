// Device-resident index layout of one malva-geno run, and the per-thread accessors over it.
//
// Measured on B200 (profiles/round1_k1_v1.md): every random read that misses L2 moves a whole 128-byte
// line from HBM, whatever the size of the load, and the device sustains ~4.3e10 such lines per second.  Both
// the sample scan (K1) and the signature look-ups (K4) are bound by the NUMBER of random lines they touch,
// so everything one k-mer needs -- the alt-allele Bloom filter `bf` (bloom_filter.hpp), the exact ref-allele
// map `ref_bf` (kmap.hpp) AND their counters -- sits in ONE 128-byte PROBE LINE addressed by the hash the
// reference computes (XXH3_64bits(canonical k-mer) % bf_bits):
//
//   line L  (L = bf bit index >> 8)              128 bytes = 32 u32 words = 8 x uint4
//     w[0..7]    bits 256L .. 256L+255 of bf      (bit i of bf = bit (i & 31) of word ((i & 255) >> 5))
//     w[8..27]   five key slots {w0,w1,w2,w3}: canonical packed k-mers of the ref-allele signatures whose hash
//                maps to a bf index inside this line, in ascending order, empty slots last
//                  inline layout (k <= 47, 2k <= 94 bits): key in w0..w2 (bit 31 of w2 is never a key bit),
//                      w3 = the key's u32 count (the KMAP value, kmap.hpp:114-122)
//                  wide layout (k >= 48): key in w0..w3 (126 bits), count in key_counts[5L + s]
//                bit 31 of w2 (inline) / w3 (wide) of slot 4 = OVERFLOW: more than five keys hashed here, the
//                largest ones live in the overflow table (ovf_keys / ovf_counts)
//     w[28]      rank: ones of bf before line L   (== sdsl rank_support_v<1>, bloom_filter.hpp:96,108)
//     w[29..31]  u32 counters of the first three set bits of the line; set bit number j of the line (j = ones
//                below it inside the line) counts in w[29+j] if j < 3, else in bf_counts[rank + j]
//
// so a sample k-mer, and a signature k-mer whose count is read back, costs one HBM line; a hit updates the line
// it has just fetched.  bf keeps the reference's exact bit semantics (same hash, same `% size`, same bit) and
// its counters stay keyed by bit index (colliding k-mers share a counter, bloom_filter.hpp:100-125); only where
// things are stored differs.  Counters are u32 accumulators; bf's are read back & 0xFFFF (int_vector<16>).
//
//   bf_counts[r]   u32 per set bit of bf, rank-indexed: the live counter of the bits with j >= 3, and -- after
//                  mg_counters_gather -- of all of them (the dense image the multi-GPU reduce and the download use)
//   ctx_words      context_bf as a plain u32 bit array (consulted only on bf hits)
//   occ            occupancy pre-filter: one bit per 2^occ_shift bf indices (<= 64 MB, kept resident in L2);
//                  the scan and the reference pass consult it first and skip empty probe lines
//   ovf_keys/ovf_counts   open-addressing table (linear probing, load <= 0.5) of the keys beyond the five
//                  smallest of a crowded line.  While the index is built it is filled by 128-bit CAS inserts;
//                  mg_finalize_alt rebuilds it in CANONICAL form: keys placed in ascending (home slot, key) order,
//                  so that -- like the sorted slots of the lines -- its image depends on the key SET only, not on
//                  the order or the races of the inserts: replicas built independently are identical and their
//                  counters add up element by element.
#pragma once
#include <cstdint>

#include "xxh3.cuh"

namespace mg {

constexpr int LINE_U4 = 8;
constexpr int LINE_KEYS = 5;
constexpr int LINE_INLINE_ALT = 3;                        // inline counters of set bits 0..2 of a line
constexpr int LINE_W_RANK = 28;                           // word index of the rank; counters follow
constexpr uint64_t KEY_HI_MASK_WIDE = 0x3FFFFFFFFFFFFFFFULL;  // k <= 63: a key uses at most 126 bits
constexpr uint64_t KEY_HI_MASK_INLINE = 0x000000007FFFFFFFULL;  // k <= 47: at most 94 bits; w3 is the count
constexpr uint64_t GOLD = 0x9E3779B97F4A7C15ULL;
constexpr int INLINE_MAX_K = 47;

struct DevView {  // everything the kernels need, passed by value
  uint4 *lines;
  uint64_t n_lines;
  const uint32_t *ctx_words;
  uint32_t *bf_counts;
  uint32_t *key_counts;  // wide layout only
  const u128 *ovf_keys;
  uint32_t *ovf_counts;
  uint64_t ovf_mask;  // capacity-1
  int ovf_shift;      // 64 - log2(capacity)
  uint64_t bf_bits;
  uint64_t bf_mask;  // bf_bits-1 when bf_bits is a power of two, else 0
  int k, ref_k;
  uint64_t key_hi_mask;  // key bits of a slot's high u64
  uint64_t ovf_flag_hi;  // OVERFLOW flag in the high u64 of slot 4
  int inline_counts;     // 1: the count of a key is w3 of its slot
  // occupancy pre-filter (L2-resident): bit (idx >> occ_shift) is set iff some bf bit or some ref key has its
  // bf index in [idx >> occ_shift << occ_shift, +2^occ_shift).  A clear bit means the probe line holds nothing
  // for this k-mer and the HBM access is skipped altogether.  nullptr = no pre-filter.
  const uint32_t *occ;
  int occ_shift;
};

MG_HD uint64_t key_hi_mask_for(int k) { return k <= INLINE_MAX_K ? KEY_HI_MASK_INLINE : KEY_HI_MASK_WIDE; }
MG_HD uint64_t ovf_flag_for(int k) { return k <= INLINE_MAX_K ? (1ULL << 31) : (1ULL << 63); }
// home slot of a key in the overflow table: any fixed function of the KEY does (the table is private to this
// layout; XXH3 is only needed for the bf index), so look-ups need not carry the hash along
MG_HD uint64_t ovf_home(u128 key, int shift) { return ((key.lo ^ (key.hi * 0xC2B2AE3D27D4EB4FULL)) * GOLD) >> shift; }

#if defined(__CUDACC__)

__device__ __forceinline__ uint64_t bf_index(const DevView &v, uint64_t h) {
  return v.bf_mask ? (h & v.bf_mask) : (h % v.bf_bits);
}
// read-only loads that do not allocate a line in L1 (data with no reuse inside an SM)
__device__ __forceinline__ uint32_t ldg_na(const uint32_t *p) {
  uint32_t r;
  asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ uint2 ldg_na(const uint2 *p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}
__device__ __forceinline__ bool occ_test(const DevView &v, uint64_t idx) {
  if (!v.occ) return true;
  uint64_t o = idx >> v.occ_shift;
  const uint32_t w = __ldg(v.occ + (o >> 5));
  return (w >> (o & 31)) & 1u;
}
__device__ __forceinline__ void occ_set(const DevView &v, uint32_t *occ_rw, uint64_t idx) {
  if (!occ_rw) return;
  uint64_t o = idx >> v.occ_shift;
  uint32_t m = 1u << (o & 31);
  if (!(occ_rw[o >> 5] & m)) atomicOr(occ_rw + (o >> 5), m);
}
__device__ __forceinline__ bool ctx_test(const DevView &v, uint64_t idx) {
  return (__ldg(v.ctx_words + (idx >> 5)) >> (idx & 31)) & 1u;
}
__device__ __forceinline__ uint32_t *line_words(const DevView &v, uint64_t line) {
  return reinterpret_cast<uint32_t *>(v.lines) + line * 32;
}
// (the filter bits and the keys are immutable once the index is built: read-only path)
__device__ __forceinline__ uint32_t line_word(const DevView &v, uint64_t line, int w) {  // w in 0..31
  return __ldg(line_words(v, line) + w);
}
__device__ __forceinline__ bool bf_test(const DevView &v, uint64_t idx) {
  return (line_word(v, idx >> 8, (int)((idx & 255) >> 5)) >> (idx & 31)) & 1u;
}
__device__ __forceinline__ u128 key_of(const DevView &v, uint4 q) {
  u128 r;
  r.lo = (uint64_t)q.x | ((uint64_t)q.y << 32);
  r.hi = ((uint64_t)q.z | ((uint64_t)q.w << 32)) & v.key_hi_mask;
  return r;
}
__device__ __forceinline__ bool key_eq(u128 a, u128 b) { return a.lo == b.lo && a.hi == b.hi; }
__device__ __forceinline__ bool key_empty(const DevView &v, u128 a) { return a.lo == ~0ull && a.hi == v.key_hi_mask; }

// 128-bit compare-and-swap (PTX ISA 8.3+, sm_90+): returns the previous value
__device__ __forceinline__ u128 cas128(u128 *addr, u128 cmp, u128 val) {
  u128 old;
  asm volatile(
      "{\n\t"
      ".reg .b128 c, s, r;\n\t"
      "mov.b128 c, {%2, %3};\n\t"
      "mov.b128 s, {%4, %5};\n\t"
      "atom.global.cas.b128 r, [%6], c, s;\n\t"
      "mov.b128 {%0, %1}, r;\n\t"
      "}"
      : "=l"(old.lo), "=l"(old.hi)
      : "l"(cmp.lo), "l"(cmp.hi), "l"(val.lo), "l"(val.hi), "l"(addr)
      : "memory");
  return old;
}

// slot of `canon` in the overflow table, or -1.  (Keys of the overflow table carry no flag bits; in the inline
// layout their high u64 is < 2^31, so the same mask applies.)
__device__ __forceinline__ int64_t ovf_find(const DevView &v, u128 canon) {
  uint64_t slot = ovf_home(canon, v.ovf_shift);
  while (true) {
    u128 key = key_of(v, __ldg(reinterpret_cast<const uint4 *>(v.ovf_keys + slot)));
    if (key_eq(key, canon)) return (int64_t)slot;
    if (key_empty(v, key)) return -1;
    slot = (slot + 1) & v.ovf_mask;
  }
}

// ---- What a probe line says about one k-mer: the decoder of every signature look-up.  `at(u)` returns uint4 u
// (0..7) of the line: a row of a look-up's swizzled shared-memory tile, or the line in global memory (line_at). ----
__device__ __forceinline__ auto line_at(const DevView &v, uint64_t line) {
  const uint4 *p = v.lines + line * LINE_U4;
  return [p](int u) { return __ldg(p + u); };
}
// Alt bit `bit` (0..255 inside the line): whether it is set.  *j = set bits below it in the line, *m = uint4 7 (the
// rank and the counters of set bits 0..2).
template <class At>
__device__ __forceinline__ bool line_alt(At at, uint32_t bit, int *j, uint4 *m) {
  const uint32_t ws = bit >> 5, below = (1u << (bit & 31u)) - 1u;
  const uint4 b0 = at(0), b1 = at(1);
  *m = at(7);
  const uint32_t wx[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
  uint32_t hit_w = 0;
  int n = 0;
#pragma unroll
  for (uint32_t x = 0; x < 8; ++x) {
    hit_w = x == ws ? wx[x] : hit_w;
    n += __popc(wx[x] & (x < ws ? 0xFFFFFFFFu : (x == ws ? below : 0u)));
  }
  *j = n;
  return (hit_w >> (bit & 31u)) & 1u;
}
// the inline key layout, for a look-up specialised for k = K (0: k of the view)
template <int K>
__device__ __forceinline__ bool inline_keys(const DevView &v) {
  return K > 0 ? (K <= INLINE_MAX_K) : (v.inline_counts != 0);
}
// Ref key `canon`: the slot that holds it, or -1.  *w3 = word 3 of that slot (the count in the inline layout), *ovf =
// the line's OVERFLOW flag.  One masked compare serves both layouts: mz / mw are key_of's key_hi_mask, constants when
// K > 0.
template <int K, class At>
__device__ __forceinline__ int line_key(const DevView &v, At at, u128 canon, uint32_t *w3, bool *ovf) {
  const bool inl = inline_keys<K>(v);
  const uint32_t mz = inl ? 0x7FFFFFFFu : 0xFFFFFFFFu, mw = inl ? 0u : 0x3FFFFFFFu;
  const uint32_t c0 = (uint32_t)canon.lo, c1 = (uint32_t)(canon.lo >> 32), c2 = (uint32_t)canon.hi,
                 c3 = (uint32_t)(canon.hi >> 32);
  int slot = -1;
  uint32_t cnt_w = 0, flag_w = 0;
#pragma unroll
  for (int s = 0; s < LINE_KEYS; ++s) {
    const uint4 p = at(2 + s);
    if (((p.x ^ c0) | (p.y ^ c1) | ((p.z ^ c2) & mz) | ((p.w ^ c3) & mw)) == 0) {
      slot = s;
      cnt_w = p.w;
    }
    if (s == LINE_KEYS - 1) flag_w = inl ? p.z : p.w;
  }
  *w3 = cnt_w;
  *ovf = (flag_w >> 31) != 0;
  return slot;
}

// insert into the five slots of a line; returns 1 = newly inserted, 0 = already present, -1 = line full
// (the caller then sets the overflow flag and spills the key to the overflow table).  Index-build time only:
// every count is still zero, so a slot is {key, 0} as a whole.
__device__ __forceinline__ int line_insert(const DevView &v, uint64_t line, u128 canon) {
  u128 *slots = reinterpret_cast<u128 *>(v.lines + line * LINE_U4 + 2);
  const u128 empty = {~0ull, v.key_hi_mask};
  for (int s = 0; s < LINE_KEYS; ++s) {
    u128 old = cas128(slots + s, empty, canon);
    old.hi &= v.key_hi_mask;
    if (key_empty(v, old)) return 1;
    if (key_eq(old, canon)) return 0;
  }
  return -1;
}
__device__ __forceinline__ void line_set_overflow(const DevView &v, uint64_t line) {
  uint32_t *w = line_words(v, line) + 8 + 4 * (LINE_KEYS - 1) + (v.inline_counts ? 2 : 3);
  atomicOr(w, 0x80000000u);
}
// insert into the open-addressing overflow table (build time); returns 1 = new, 0 = present
__device__ __forceinline__ int ovf_insert(const DevView &v, u128 *ovf_keys_rw, u128 canon) {
  const u128 empty = {~0ull, v.key_hi_mask};
  uint64_t slot = ovf_home(canon, v.ovf_shift);
  while (true) {
    u128 old = cas128(ovf_keys_rw + slot, empty, canon);
    old.hi &= v.key_hi_mask;
    if (key_empty(v, old)) return 1;
    if (key_eq(old, canon)) return 0;
    slot = (slot + 1) & v.ovf_mask;
  }
}

#endif  // __CUDACC__

}  // namespace mg
