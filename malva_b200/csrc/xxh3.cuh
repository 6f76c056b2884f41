// Bit-identical XXH3_64bits (seed 0, default secret) for k-mer sized inputs, and
// the 2-bit k-mer codec that feeds it.  Written for sm_100a; every helper is
// also __host__ so the CPU-only tests can exercise the very same code through
// the mg_selftest_* exports.
//
// Reference behaviour restated here:
//   XXH3_64bits                xxhash.h:5037-5040 -> XXH3_len_0to16_64b :3877-3886,
//                              XXH3_len_17to128_64b :3946-3980, XXH3_mix16B :3913-3943,
//                              XXH3_avalanche :3764-3770, secret :3548-3561
//   canonical k-mer            bloom_filter.hpp:58-65 (lexicographic min, ties -> revcomp)
//   hash input                 the ASCII bytes of the canonical string (bloom_filter.hpp:67-74)
#pragma once
#include <cstdint>

#if defined(__CUDACC__)
#define MG_HD __host__ __device__ __forceinline__
#else
#define MG_HD inline
#endif

namespace mg {

struct u128 {
  uint64_t lo, hi;
};

// first 128 bytes of XXH3_kSecret as little-endian u64 words
#define MG_SEC(i)                                                                                    \
  ((i) == 0 ? 0xBE4BA423396CFEB8ULL : (i) == 1 ? 0x1CAD21F72C81017CULL : (i) == 2 ? 0xDB979083E96DD4DEULL \
   : (i) == 3 ? 0x1F67B3B7A4A44072ULL : (i) == 4 ? 0x78E5C0CC4EE679CBULL : (i) == 5 ? 0x2172FFCC7DD05A82ULL \
   : (i) == 6 ? 0x8E2443F7744608B8ULL : (i) == 7 ? 0x4C263A81E69035E0ULL : (i) == 8 ? 0xCB00C391BB52283CULL \
   : (i) == 9 ? 0xA32E531B8B65D088ULL : (i) == 10 ? 0x4EF90DA297486471ULL : (i) == 11 ? 0xD8ACDEA946EF1938ULL \
   : (i) == 12 ? 0x3F349CE33F76FAA8ULL : (i) == 13 ? 0x1D4F0BC7C7BBDCF9ULL : (i) == 14 ? 0x3159B4CD4BE0518AULL \
                                                                            : 0x647378D9C97E9FC8ULL)

constexpr uint64_t PRIME64_1 = 0x9E3779B185EBCA87ULL;
constexpr uint64_t PRIME64_2 = 0xC2B2AE3D27D4EB4FULL;
constexpr uint64_t PRIME64_3 = 0x165667B19E3779F9ULL;

MG_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}
MG_HD uint64_t brev64(uint64_t v) {
#if defined(__CUDA_ARCH__)
  return __brevll(v);
#else
  v = ((v >> 1) & 0x5555555555555555ULL) | ((v & 0x5555555555555555ULL) << 1);
  v = ((v >> 2) & 0x3333333333333333ULL) | ((v & 0x3333333333333333ULL) << 2);
  v = ((v >> 4) & 0x0F0F0F0F0F0F0F0FULL) | ((v & 0x0F0F0F0F0F0F0F0FULL) << 4);
  return __builtin_bswap64(v);
#endif
}
MG_HD uint64_t bswap64(uint64_t v) {
#if defined(__CUDA_ARCH__)
  uint32_t lo = (uint32_t)v, hi = (uint32_t)(v >> 32);
  return ((uint64_t)__byte_perm(lo, 0, 0x0123) << 32) | (uint64_t)__byte_perm(hi, 0, 0x0123);
#else
  return __builtin_bswap64(v);
#endif
}
MG_HD uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }

// low ^ high half of the 128-bit product (XXH3_mul128_fold64, xxhash.h:3708-3762); one 128-bit multiply lets
// the compiler share the four 32x32 partial products between the two halves
MG_HD uint64_t mul128_fold64(uint64_t a, uint64_t b) {
  unsigned __int128 p = (unsigned __int128)a * b;
  return (uint64_t)p ^ (uint64_t)(p >> 64);
}
MG_HD uint64_t xxh3_avalanche(uint64_t h) {
  h ^= h >> 37;
  h *= 0x165667919E3779F9ULL;
  h ^= h >> 32;
  return h;
}
MG_HD uint64_t xxh64_avalanche(uint64_t h) {
  h ^= h >> 33;
  h *= PRIME64_2;
  h ^= h >> 29;
  h *= PRIME64_3;
  h ^= h >> 32;
  return h;
}
MG_HD uint64_t xxh3_rrmxmx(uint64_t h, uint64_t len) {
  h ^= rotl64(h, 49) ^ rotl64(h, 24);
  h *= 0x9FB21C651E98DF25ULL;
  h ^= (h >> 35) + len;
  h *= 0x9FB21C651E98DF25ULL;
  return h ^ (h >> 28);
}

// Little-endian u64 starting at byte `off` of a message held as LE u64 words.
// The word after the last one touched must be addressable (callers pad by one).
MG_HD uint64_t rd64_at(const uint64_t *w, int off) {
  int j = off >> 3, s = (off & 7) * 8;
  return s == 0 ? w[j] : ((w[j] >> s) | (w[j + 1] << (64 - s)));
}
MG_HD uint32_t rd32_at(const uint64_t *w, int off) { return (uint32_t)rd64_at(w, off); }

MG_HD uint64_t mix16(const uint64_t *w, int off, int si) {
  return mul128_fold64(rd64_at(w, off) ^ MG_SEC(si), rd64_at(w, off + 8) ^ MG_SEC(si + 1));
}

// XXH3_64bits over `len` (<=128) message bytes stored in w[0..(len+7)/8] (+1 pad word).
MG_HD uint64_t xxh3_64_words(const uint64_t *w, int len) {
  if (len > 16) {
    uint64_t acc = (uint64_t)len * PRIME64_1;
    if (len > 32) {
      if (len > 64) {
        if (len > 96) {
          acc += mix16(w, 48, 12);
          acc += mix16(w, len - 64, 14);
        }
        acc += mix16(w, 32, 8);
        acc += mix16(w, len - 48, 10);
      }
      acc += mix16(w, 16, 4);
      acc += mix16(w, len - 32, 6);
    }
    acc += mix16(w, 0, 0);
    acc += mix16(w, len - 16, 2);
    return xxh3_avalanche(acc);
  }
  if (len > 8) {
    uint64_t lo = rd64_at(w, 0) ^ (MG_SEC(3) ^ MG_SEC(4));
    uint64_t hi = rd64_at(w, len - 8) ^ (MG_SEC(5) ^ MG_SEC(6));
    return xxh3_avalanche((uint64_t)len + bswap64(lo) + hi + mul128_fold64(lo, hi));
  }
  if (len >= 4) {
    uint32_t i1 = rd32_at(w, 0), i2 = rd32_at(w, len - 4);
    uint64_t in64 = (uint64_t)i2 + ((uint64_t)i1 << 32);
    return xxh3_rrmxmx(in64 ^ (MG_SEC(1) ^ MG_SEC(2)), (uint64_t)len);
  }
  if (len > 0) {
    uint32_t c1 = (uint32_t)(w[0] & 0xFF);
    uint32_t c2 = (uint32_t)((w[0] >> (8 * (len >> 1))) & 0xFF);
    uint32_t c3 = (uint32_t)((w[0] >> (8 * (len - 1))) & 0xFF);
    uint32_t comb = (c1 << 16) | (c2 << 24) | c3 | ((uint32_t)len << 8);
    uint64_t bitflip = (uint64_t)((uint32_t)MG_SEC(0) ^ (uint32_t)(MG_SEC(0) >> 32));
    return xxh64_avalanche((uint64_t)comb ^ bitflip);
  }
  return xxh64_avalanche(MG_SEC(7) ^ MG_SEC(8));
}

// ---------------------------------------------------------------------------
// 2-bit k-mer codec.  Word layout "MSB-first": base i of a k-mer sits at bits
// [2(k-1-i), 2(k-1-i)+1] of a right-aligned 128-bit integer (A=0 C=1 G=2 T=3),
// so integer order equals lexicographic order of the ASCII strings.
// ---------------------------------------------------------------------------
MG_HD bool less128(u128 a, u128 b) { return a.hi < b.hi || (a.hi == b.hi && a.lo < b.lo); }

MG_HD u128 shr128(u128 x, int s) {  // 0 <= s < 128
  u128 r;
  if (s == 0) return x;
  if (s >= 64) {
    r.lo = x.hi >> (s - 64);
    r.hi = 0;
  } else {
    r.lo = (x.lo >> s) | (x.hi << (64 - s));
    r.hi = x.hi >> s;
  }
  return r;
}
MG_HD u128 mask128(u128 x, int bits) {  // keep the low `bits` bits, 0 < bits <= 128
  if (bits >= 128) return x;
  if (bits >= 64) {
    x.hi &= (bits == 64) ? 0ULL : ((1ULL << (bits - 64)) - 1);
  } else {
    x.hi = 0;
    x.lo &= (1ULL << bits) - 1;
  }
  return x;
}
// reverse the order of the 32 two-bit groups of a u64
MG_HD uint64_t rev_groups64(uint64_t v) {
  uint64_t r = brev64(v);
  return ((r >> 1) & 0x5555555555555555ULL) | ((r & 0x5555555555555555ULL) << 1);
}
// "LSB-first" image of a k-mer: base i at bits [2i, 2i+1]
MG_HD u128 lsb_first(u128 x, int k) {
  u128 r;
  r.lo = rev_groups64(x.hi);
  r.hi = rev_groups64(x.lo);
  return shr128(r, 128 - 2 * k);
}
MG_HD u128 revcomp(u128 x, int k) {
  u128 c;
  c.lo = ~x.lo;
  c.hi = ~x.hi;
  return lsb_first(c, k);  // complement, then reverse the base order
}

// 4 bases (8 bits, base 0 in the low 2 bits) -> 4 ASCII bytes, base 0 in the low byte
MG_HD uint32_t expand4(uint32_t v) {
  uint32_t t = (v | (v << 4)) & 0x0F0Fu;
  t = (t | (t << 2)) & 0x3333u;
#if defined(__CUDA_ARCH__)
  return __byte_perm(0x54474341u, 0u, t);  // "ACGT" as a 4-entry byte table
#else
  const uint32_t tab = 0x54474341u;
  uint32_t r = 0;
  for (int i = 0; i < 4; ++i) r |= ((tab >> (8 * ((t >> (4 * i)) & 3))) & 0xFFu) << (8 * i);
  return r;
#endif
}

MG_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
#if defined(__CUDA_ARCH__)
  return __byte_perm(a, b, sel);
#else
  const uint64_t pool = (uint64_t)a | ((uint64_t)b << 32);
  uint32_t r = 0;
  for (int i = 0; i < 4; ++i) r |= (uint32_t)((pool >> (8 * ((sel >> (4 * i)) & 7))) & 0xFFu) << (8 * i);
  return r;
#endif
}
// 8 bases = one 16-bit half of `word` (HALF 0: bits 0..15, HALF 1: bits 16..31; base 0 in the low 2 bits)
// -> 8 ASCII bytes.  The two bytes are first moved to byte lanes 0 and 2 (one PRMT), the 2-bit codes are then
// spread to nibbles in two shift-or-mask steps, and each nibble indexes the byte table "ACGT" (PRMT).
template <int HALF>
MG_HD uint64_t expand8(uint32_t word) {
  uint32_t t = prmt(word, 0u, HALF ? 0x4342u : 0x4140u);  // {b0, 0, b1, 0}
  t = (t | (t << 4)) & 0x0F0F0F0Fu;
  t = (t | (t << 2)) & 0x33333333u;
  const uint32_t lo = prmt(0x54474341u, 0u, t), hi = prmt(0x54474341u, 0u, t >> 16);
  return (uint64_t)lo | ((uint64_t)hi << 32);
}

// ASCII bytes of a k-mer (given in LSB-first layout) as LE u64 words; bytes
// past k are unspecified but never read by xxh3_64_words(w, K).
template <int K>
MG_HD void ascii_words(u128 r, uint64_t *w) {
  constexpr int NW = (K + 7) / 8;
#pragma unroll
  for (int j = 0; j < NW; ++j) {
    const uint32_t word = (j < 4) ? (uint32_t)(r.lo >> (32 * (j >> 1))) : (uint32_t)(r.hi >> (32 * ((j - 4) >> 1)));
    w[j] = (j & 1) ? expand8<1>(word) : expand8<0>(word);
  }
  w[NW] = 0;
}

// canonical form + hash of a packed K-mer: returns XXH3_64bits(canonical ASCII)
// and the canonical packed word (the exact-table key).
template <int K>
MG_HD uint64_t canon_hash(u128 x, u128 *canon) {
  u128 rc = revcomp(x, K);
  bool fwd = less128(x, rc);  // strcmp(kmer, rc) < 0 keeps kmer, else rc (bloom_filter.hpp:63)
  u128 c = fwd ? x : rc;
  u128 other = fwd ? rc : x;
  // LSB-first image of c == complement of the other strand (see lsb_first/revcomp)
  u128 r;
  r.lo = ~other.lo;
  r.hi = ~other.hi;
  r = mask128(r, 2 * K);
  uint64_t w[(K + 7) / 8 + 1];
  ascii_words<K>(r, w);
  *canon = c;
  return xxh3_64_words(w, K);
}

// runtime-k variant (any 1 <= k <= 64); slower, used when (k, ref_k) is not a
// compiled specialisation.
MG_HD uint64_t canon_hash_rt(u128 x, int k, u128 *canon) {
  u128 rc = revcomp(x, k);
  bool fwd = less128(x, rc);
  u128 c = fwd ? x : rc;
  u128 other = fwd ? rc : x;
  u128 r;
  r.lo = ~other.lo;
  r.hi = ~other.hi;
  r = mask128(r, 2 * k);
  uint64_t w[10];
  for (int j = 0; j < 8; ++j) {
    uint32_t bits16 = (j < 4) ? (uint32_t)(r.lo >> (16 * j)) : (uint32_t)(r.hi >> (16 * (j - 4)));
    w[j] = (uint64_t)expand4(bits16 & 0xFFu) | ((uint64_t)expand4((bits16 >> 8) & 0xFFu) << 32);
  }
  w[8] = w[9] = 0;
  *canon = c;
  return xxh3_64_words(w, k);
}

// canon_hash<K> for a build specialised for k = K, canon_hash_rt for K = 0
template <int K>
MG_HD uint64_t canon_hash_k(u128 x, int k, u128 *canon) {
  if constexpr (K > 0) {
    return canon_hash<K>(x, canon);
  } else {
    return canon_hash_rt(x, k, canon);
  }
}

// ---------------------------------------------------------------------------
// ASCII k-mers (signature side): arbitrary bytes, length <= 128.
// ---------------------------------------------------------------------------
MG_HD uint8_t rcn(uint8_t c) {  // the RCN table of bloom_filter.hpp:36-50 (only non-zero entries)
  switch (c) {
    case 'A': return 'T';
    case 'C': return 'G';
    case 'G': return 'C';
    case 'T': return 'A';
    case 'N': return 'N';
    case 'a': return 'T';
    case 'c': return 'G';
    case 'g': return 'G';  // sic (index 103 of the table)
    case 't': return 'A';
    case 'n': return 'N';
    default: return 0;
  }
}

// Canonical bytes of an ASCII k-mer into w[] (LE words, zero padded, len<=128).
// Returns the length a std::string built from the canonical C string would have
// (kmap.hpp:95 cuts at the first NUL).
MG_HD int canonical_ascii(const uint8_t *s, int len, uint64_t *w /*[18]*/) {
  // strcmp(kmer, rc) < 0 ?  kmer holds no NUL inside len; rc may.
  int cmp = 0;
  for (int i = 0; i < len && cmp == 0; ++i) {
    int a = s[i], b = rcn(s[len - 1 - i]);
    cmp = a - b;
  }
  for (int j = 0; j < 18; ++j) w[j] = 0;
  int cut = len;
  bool seen_nul = false;
  for (int i = 0; i < len; ++i) {
    uint8_t c = (cmp < 0) ? s[i] : rcn(s[len - 1 - i]);
    if (c == 0 && !seen_nul) {
      cut = i;
      seen_nul = true;
    }
    w[i >> 3] |= (uint64_t)c << (8 * (i & 7));
  }
  return cut;
}

MG_HD uint64_t hash_ascii(const uint8_t *s, int len) {
  uint64_t w[18];
  canonical_ascii(s, len, w);
  return xxh3_64_words(w, len);
}

// Pack an ASCII k-mer if it is exactly k symbols of ACGT; false otherwise.
MG_HD bool pack_ascii(const uint8_t *s, int len, int k, u128 *out) {
  if (len != k) return false;
  u128 x;
  x.lo = 0;
  x.hi = 0;
  for (int i = 0; i < len; ++i) {
    uint32_t c;
    switch (s[i]) {
      case 'A': c = 0; break;
      case 'C': c = 1; break;
      case 'G': c = 2; break;
      case 'T': c = 3; break;
      default: return false;
    }
    x.hi = (x.hi << 2) | (x.lo >> 62);
    x.lo = (x.lo << 2) | c;
  }
  *out = x;
  return true;
}

}  // namespace mg
