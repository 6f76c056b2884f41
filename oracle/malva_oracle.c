/* TEST INFRASTRUCTURE ONLY -- see malva_oracle.h.  Plain C restatement of the
 * reference's hot-path arithmetic; not a product code path. */
#include "malva_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

/* ------------------------------------------------------------------------ */
/* XXH3_64bits, seed 0, default secret (xxhash.h:3548-3561, 3764-3980)        */
/* ------------------------------------------------------------------------ */
static const uint8_t kSecret[192] = {
    0xb8, 0xfe, 0x6c, 0x39, 0x23, 0xa4, 0x4b, 0xbe, 0x7c, 0x01, 0x81, 0x2c, 0xf7, 0x21, 0xad, 0x1c,
    0xde, 0xd4, 0x6d, 0xe9, 0x83, 0x90, 0x97, 0xdb, 0x72, 0x40, 0xa4, 0xa4, 0xb7, 0xb3, 0x67, 0x1f,
    0xcb, 0x79, 0xe6, 0x4e, 0xcc, 0xc0, 0xe5, 0x78, 0x82, 0x5a, 0xd0, 0x7d, 0xcc, 0xff, 0x72, 0x21,
    0xb8, 0x08, 0x46, 0x74, 0xf7, 0x43, 0x24, 0x8e, 0xe0, 0x35, 0x90, 0xe6, 0x81, 0x3a, 0x26, 0x4c,
    0x3c, 0x28, 0x52, 0xbb, 0x91, 0xc3, 0x00, 0xcb, 0x88, 0xd0, 0x65, 0x8b, 0x1b, 0x53, 0x2e, 0xa3,
    0x71, 0x64, 0x48, 0x97, 0xa2, 0x0d, 0xf9, 0x4e, 0x38, 0x19, 0xef, 0x46, 0xa9, 0xde, 0xac, 0xd8,
    0xa8, 0xfa, 0x76, 0x3f, 0xe3, 0x9c, 0x34, 0x3f, 0xf9, 0xdc, 0xbb, 0xc7, 0xc7, 0x0b, 0x4f, 0x1d,
    0x8a, 0x51, 0xe0, 0x4b, 0xcd, 0xb4, 0x59, 0x31, 0xc8, 0x9f, 0x7e, 0xc9, 0xd9, 0x78, 0x73, 0x64,
    0xea, 0xc5, 0xac, 0x83, 0x34, 0xd3, 0xeb, 0xc3, 0xc5, 0x81, 0xa0, 0xff, 0xfa, 0x13, 0x63, 0xeb,
    0x17, 0x0d, 0xdd, 0x51, 0xb7, 0xf0, 0xda, 0x49, 0xd3, 0x16, 0x55, 0x26, 0x29, 0xd4, 0x68, 0x9e,
    0x2b, 0x16, 0xbe, 0x58, 0x7d, 0x47, 0xa1, 0xfc, 0x8f, 0xf8, 0xb8, 0xd1, 0x7a, 0xd0, 0x31, 0xce,
    0x45, 0xcb, 0x3a, 0x8f, 0x95, 0x16, 0x04, 0x28, 0xaf, 0xd7, 0xfb, 0xca, 0xbb, 0x4b, 0x40, 0x7e,
};

#define P32_1 0x9E3779B1U
#define P32_2 0x85EBCA77U
#define P32_3 0xC2B2AE3DU
#define P64_1 0x9E3779B185EBCA87ULL
#define P64_2 0xC2B2AE3D27D4EB4FULL
#define P64_3 0x165667B19E3779F9ULL
#define P64_4 0x85EBCA77C2B2AE63ULL
#define P64_5 0x27D4EB2F165667C5ULL

static uint32_t rd32(const uint8_t *p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}
static uint64_t rd64(const uint8_t *p) { return (uint64_t)rd32(p) | ((uint64_t)rd32(p + 4) << 32); }
static uint64_t rotl64(uint64_t x, int r) { return (x << r) | (x >> (64 - r)); }
static uint64_t swap64(uint64_t x) { return __builtin_bswap64(x); }

static uint64_t mul128_fold64(uint64_t a, uint64_t b) {
  __uint128_t p = (__uint128_t)a * b;
  return (uint64_t)p ^ (uint64_t)(p >> 64);
}
static uint64_t xxh3_avalanche(uint64_t h) { /* xxhash.h:3764-3770 */
  h ^= h >> 37;
  h *= 0x165667919E3779F9ULL;
  h ^= h >> 32;
  return h;
}
static uint64_t xxh64_avalanche(uint64_t h) {
  h ^= h >> 33;
  h *= P64_2;
  h ^= h >> 29;
  h *= P64_3;
  h ^= h >> 32;
  return h;
}
static uint64_t rrmxmx(uint64_t h, uint64_t len) { /* xxhash.h:3777-3786 */
  h ^= rotl64(h, 49) ^ rotl64(h, 24);
  h *= 0x9FB21C651E98DF25ULL;
  h ^= (h >> 35) + len;
  h *= 0x9FB21C651E98DF25ULL;
  return h ^ (h >> 28);
}
static uint64_t mix16(const uint8_t *in, const uint8_t *sec) { /* xxhash.h:3913-3943 */
  return mul128_fold64(rd64(in) ^ rd64(sec), rd64(in + 8) ^ rd64(sec + 8));
}

uint64_t mo_xxh3_64(const void *data, size_t len) {
  const uint8_t *in = (const uint8_t *)data;
  const uint8_t *s = kSecret;
  if (len <= 16) { /* xxhash.h:3877-3886 */
    if (len > 8) {
      uint64_t lo = rd64(in) ^ (rd64(s + 24) ^ rd64(s + 32));
      uint64_t hi = rd64(in + len - 8) ^ (rd64(s + 40) ^ rd64(s + 48));
      return xxh3_avalanche(len + swap64(lo) + hi + mul128_fold64(lo, hi));
    }
    if (len >= 4) {
      uint32_t i1 = rd32(in), i2 = rd32(in + len - 4);
      uint64_t bitflip = rd64(s + 8) ^ rd64(s + 16);
      uint64_t in64 = (uint64_t)i2 + ((uint64_t)i1 << 32);
      return rrmxmx(in64 ^ bitflip, len);
    }
    if (len) {
      uint8_t c1 = in[0], c2 = in[len >> 1], c3 = in[len - 1];
      uint32_t comb = ((uint32_t)c1 << 16) | ((uint32_t)c2 << 24) | (uint32_t)c3 | ((uint32_t)len << 8);
      uint64_t bitflip = (uint64_t)(rd32(s) ^ rd32(s + 4));
      return xxh64_avalanche((uint64_t)comb ^ bitflip);
    }
    return xxh64_avalanche(rd64(s + 56) ^ rd64(s + 64));
  }
  if (len <= 128) { /* xxhash.h:3946-3980 */
    uint64_t acc = (uint64_t)len * P64_1;
    if (len > 32) {
      if (len > 64) {
        if (len > 96) {
          acc += mix16(in + 48, s + 96);
          acc += mix16(in + len - 64, s + 112);
        }
        acc += mix16(in + 32, s + 64);
        acc += mix16(in + len - 48, s + 80);
      }
      acc += mix16(in + 16, s + 32);
      acc += mix16(in + len - 32, s + 48);
    }
    acc += mix16(in, s);
    acc += mix16(in + len - 16, s + 16);
    return xxh3_avalanche(acc);
  }
  if (len <= 240) { /* xxhash.h:3985-4050 */
    uint64_t acc = (uint64_t)len * P64_1;
    size_t rounds = len / 16, i;
    for (i = 0; i < 8; ++i) acc += mix16(in + 16 * i, s + 16 * i);
    acc = xxh3_avalanche(acc);
    for (i = 8; i < rounds; ++i) acc += mix16(in + 16 * i, s + 16 * (i - 8) + 3);
    acc += mix16(in + len - 16, s + 136 - 17);
    return xxh3_avalanche(acc);
  }
  abort(); /* the long-input path is unreachable for k-mers */
}

/* ------------------------------------------------------------------------ */
/* canonical form (bloom_filter.hpp:36-65)                                    */
/* ------------------------------------------------------------------------ */
static char rcn(unsigned char c) {
  switch (c) { /* the RCN table: only these entries are non-zero */
    case 'A': return 'T';
    case 'C': return 'G';
    case 'G': return 'C';
    case 'T': return 'A';
    case 'N': return 'N';
    case 'a': return 'T';
    case 'c': return 'G';
    case 'g': return 'G'; /* sic: table typo at index 103 */
    case 't': return 'A';
    case 'n': return 'N';
    default: return 0;
  }
}

void mo_canonical(const char *kmer, int k, char *out) {
  int i;
  for (i = 0; i < k; ++i) out[i] = rcn((unsigned char)kmer[k - 1 - i]);
  out[k] = '\0';
  if (strcmp(kmer, out) < 0) memmove(out, kmer, (size_t)k);
}

static uint64_t kmer_hash(const char *kmer) { /* bloom_filter.hpp:67-74 */
  size_t k = strlen(kmer);
  char buf[512];
  if (k >= sizeof(buf)) abort();
  mo_canonical(kmer, (int)k, buf);
  return mo_xxh3_64(buf, k);
}

/* ------------------------------------------------------------------------ */
/* BF                                                                         */
/* ------------------------------------------------------------------------ */
struct mo_bf {
  int mode;
  uint64_t size;
  uint64_t nwords;
  uint64_t *w;
  uint64_t *blk; /* ones before each 512-bit block */
  uint64_t ones;
  uint16_t *counts;
};

mo_bf *mo_bf_new(uint64_t size_bits) {
  mo_bf *b = (mo_bf *)calloc(1, sizeof(*b));
  b->size = size_bits;
  b->nwords = (size_bits + 63) / 64;
  b->w = (uint64_t *)calloc(b->nwords ? b->nwords : 1, 8);
  return b;
}
void mo_bf_free(mo_bf *b) {
  if (!b) return;
  free(b->w);
  free(b->blk);
  free(b->counts);
  free(b);
}
static int bf_bit(const mo_bf *b, uint64_t i) { return (int)((b->w[i >> 6] >> (i & 63)) & 1ULL); }
static uint64_t bf_rank(const mo_bf *b, uint64_t i) {
  uint64_t wi = i >> 6, r = b->blk[wi >> 3], x;
  for (x = wi & ~7ULL; x < wi; ++x) r += (uint64_t)__builtin_popcountll(b->w[x]);
  if (i & 63) r += (uint64_t)__builtin_popcountll(b->w[wi] & ((1ULL << (i & 63)) - 1));
  return r;
}
void mo_bf_add_key(mo_bf *b, const char *kmer) {
  uint64_t i = kmer_hash(kmer) % b->size;
  b->w[i >> 6] |= 1ULL << (i & 63);
}
int mo_bf_test_key(const mo_bf *b, const char *kmer) { return bf_bit(b, kmer_hash(kmer) % b->size); }
uint64_t mo_find_kmers_at(const char *seed, int k, uint64_t size, uint64_t lo, uint64_t first, uint64_t n_trials,
                          char *out, uint64_t max_out) {
  /* k-mers whose filter index kmer_hash % size is >= lo: trial t is the seed with t written in base 4 into its
   * symbols 1..31; k(+NUL)-byte results go to out.  The seed starts and ends with 'A', so every trial is its own
   * canonical form (its reverse complement starts with 'T') and is hashed as it is. */
  char s[512];
  uint64_t t, found = 0;
  int j, w = k - 2 < 31 ? k - 2 : 31;
  if (k < 3 || k >= (int)sizeof(s) || seed[0] != 'A' || seed[k - 1] != 'A') return 0;
  memcpy(s, seed, (size_t)k);
  s[k] = '\0';
  for (t = first; t < first + n_trials && found < max_out; ++t) {
    for (j = 0; j < w; ++j) s[1 + j] = "ACGT"[(t >> (2 * j)) & 3];
    if (mo_xxh3_64(s, (size_t)k) % size >= lo) memcpy(out + (k + 1) * found++, s, (size_t)k + 1);
  }
  return found;
}
void mo_bf_switch_mode(mo_bf *b) {
  uint64_t nb = b->nwords / 8 + 2, acc = 0, wi;
  b->mode = 1;
  free(b->blk);
  free(b->counts);
  b->blk = (uint64_t *)calloc(nb, 8);
  for (wi = 0; wi < b->nwords; ++wi) {
    if ((wi & 7) == 0) b->blk[wi >> 3] = acc;
    acc += (uint64_t)__builtin_popcountll(b->w[wi]);
  }
  for (wi = (b->nwords + 7) / 8; wi < nb; ++wi) b->blk[wi] = acc;
  b->ones = acc;
  b->counts = (uint16_t *)calloc(acc ? acc : 1, 2);
}
int mo_bf_increment(mo_bf *b, const char *kmer, uint32_t counter) {
  uint64_t i;
  if (!b->mode) return 0;
  i = kmer_hash(kmer) % b->size;
  if (bf_bit(b, i)) {
    uint64_t ci = bf_rank(b, i);
    uint32_t nv = (uint32_t)b->counts[ci] + counter;
    b->counts[ci] = (uint16_t)nv; /* int_vector<16>: truncating store */
  }
  return 1;
}
uint16_t mo_bf_get_count(const mo_bf *b, const char *kmer) {
  if (b->mode) {
    uint64_t i = kmer_hash(kmer) % b->size;
    if (bf_bit(b, i)) return b->counts[bf_rank(b, i)];
  }
  return 0;
}
uint64_t mo_bf_size(const mo_bf *b) { return b->size; }
uint64_t mo_bf_popcount(const mo_bf *b) {
  uint64_t acc = 0, wi;
  for (wi = 0; wi < b->nwords; ++wi) acc += (uint64_t)__builtin_popcountll(b->w[wi]);
  return acc;
}
const uint64_t *mo_bf_words(const mo_bf *b) { return b->w; }
const uint16_t *mo_bf_counts(const mo_bf *b) { return b->counts; }

/* ------------------------------------------------------------------------ */
/* KMAP: exact map keyed by the canonical string cut at its first NUL          */
/* ------------------------------------------------------------------------ */
typedef struct kentry {
  char *key;
  uint32_t len;
  int val;
  struct kentry *next;
} kentry;
struct mo_kmap {
  kentry **bucket;
  uint64_t nb, n;
};
mo_kmap *mo_kmap_new(void) {
  mo_kmap *m = (mo_kmap *)calloc(1, sizeof(*m));
  m->nb = 1024;
  m->bucket = (kentry **)calloc(m->nb, sizeof(kentry *));
  return m;
}
void mo_kmap_free(mo_kmap *m) {
  uint64_t i;
  if (!m) return;
  for (i = 0; i < m->nb; ++i) {
    kentry *e = m->bucket[i];
    while (e) {
      kentry *nx = e->next;
      free(e->key);
      free(e);
      e = nx;
    }
  }
  free(m->bucket);
  free(m);
}
static size_t kmap_key(const char *kmer, char *buf, size_t cap) { /* kmap.hpp:86-97 */
  size_t k = strlen(kmer);
  if (k >= cap) abort();
  mo_canonical(kmer, (int)k, buf);
  return strlen(buf); /* std::string(ckmer) stops at the first NUL */
}
static kentry *kmap_find(const mo_kmap *m, const char *key, size_t len) {
  kentry *e = m->bucket[mo_xxh3_64(key, len) % m->nb];
  for (; e; e = e->next)
    if (e->len == len && memcmp(e->key, key, len) == 0) return e;
  return NULL;
}
static void kmap_grow(mo_kmap *m) {
  uint64_t nnb = m->nb * 4, i;
  kentry **nbk = (kentry **)calloc(nnb, sizeof(kentry *));
  for (i = 0; i < m->nb; ++i) {
    kentry *e = m->bucket[i];
    while (e) {
      kentry *nx = e->next;
      uint64_t h = mo_xxh3_64(e->key, e->len) % nnb;
      e->next = nbk[h];
      nbk[h] = e;
      e = nx;
    }
  }
  free(m->bucket);
  m->bucket = nbk;
  m->nb = nnb;
}
void mo_kmap_add_key(mo_kmap *m, const char *kmer) {
  char buf[512];
  size_t len = kmap_key(kmer, buf, sizeof(buf));
  kentry *e = kmap_find(m, buf, len);
  if (e) {
    e->val = 0; /* kmers[ckmer] = 0 re-sets an existing key */
    return;
  }
  if (m->n >= m->nb) kmap_grow(m);
  e = (kentry *)calloc(1, sizeof(*e));
  e->key = (char *)malloc(len + 1);
  memcpy(e->key, buf, len);
  e->key[len] = 0;
  e->len = (uint32_t)len;
  {
    uint64_t h = mo_xxh3_64(buf, len) % m->nb;
    e->next = m->bucket[h];
    m->bucket[h] = e;
  }
  m->n++;
}
int mo_kmap_test_key(const mo_kmap *m, const char *kmer) {
  char buf[512];
  size_t len = kmap_key(kmer, buf, sizeof(buf));
  return kmap_find(m, buf, len) != NULL;
}
void mo_kmap_increment(mo_kmap *m, const char *kmer, int counter) {
  char buf[512];
  size_t len = kmap_key(kmer, buf, sizeof(buf));
  kentry *e = kmap_find(m, buf, len);
  if (e) e->val = (int)((uint32_t)e->val + (uint32_t)counter);
}
int mo_kmap_get_count(const mo_kmap *m, const char *kmer) {
  char buf[512];
  size_t len = kmap_key(kmer, buf, sizeof(buf));
  kentry *e = kmap_find(m, buf, len);
  return e ? e->val : 0;
}
uint64_t mo_kmap_size(const mo_kmap *m) { return m->n; }

/* ------------------------------------------------------------------------ */
/* loops                                                                      */
/* ------------------------------------------------------------------------ */
void mo_scan_ascii(mo_bf *bf, const mo_bf *context_bf, mo_kmap *ref_bf, const char *contexts,
                   const uint32_t *counters, uint64_t n, int k, int ref_k) {
  char context[512], kmer[512];
  uint64_t i;
  int j;
  for (i = 0; i < n; ++i) { /* main.cpp:488-500 */
    for (j = 0; j < ref_k; ++j) {
      char c = contexts[i * (uint64_t)ref_k + (uint64_t)j];
      context[j] = (c >= 'a' && c <= 'z') ? (char)(c - 32) : c;
    }
    context[ref_k] = 0;
    memcpy(kmer, context + (ref_k - k) / 2, (size_t)k);
    kmer[k] = 0;
    mo_kmap_increment(ref_bf, kmer, (int)counters[i]);
    if (!mo_bf_test_key(context_bf, context)) mo_bf_increment(bf, kmer, counters[i]);
  }
}

void mo_scan_packed(mo_bf *bf, const mo_bf *context_bf, mo_kmap *ref_bf, const uint64_t *lohi,
                    const uint32_t *counters, uint64_t n, int k, int ref_k) {
  static const char SYM[4] = {'A', 'C', 'G', 'T'};
  char context[129];
  uint64_t i;
  int j;
  for (i = 0; i < n; ++i) {
    uint64_t lo = lohi[2 * i], hi = lohi[2 * i + 1];
    for (j = 0; j < ref_k; ++j) {
      int sh = 2 * (ref_k - 1 - j);
      uint64_t code = sh >= 64 ? (hi >> (sh - 64)) : (lo >> sh);
      context[j] = SYM[code & 3];
    }
    mo_scan_ascii(bf, context_bf, ref_bf, context, counters + i, 1, k, ref_k);
  }
}

void mo_reference_pass(const mo_bf *bf, mo_bf *context_bf, const char *seq, uint64_t len, int k, int ref_k) {
  /* main.cpp:385-400.  Window ending at p: context = seq[p-ref_k+1 .. p]; the
   * k-mer window of the first step starts at d=(ref_k-k)/2, and every slide
   * appends seq[p-d], i.e. it ends at p-d. */
  char context[512], ksub[512];
  uint64_t d = (uint64_t)(ref_k - k) / 2, p, cl, kl;
  /* string ref_ksub(reference, d, k); string context(reference, 0, ref_k);  -- substr() clamps to the
   * end of the string, and throws when d > size() (callers never pass that) */
  if (d > len) return;
  kl = len - d < (uint64_t)k ? len - d : (uint64_t)k;
  cl = len < (uint64_t)ref_k ? len : (uint64_t)ref_k;
  memcpy(ksub, seq + d, kl);
  ksub[kl] = 0;
  memcpy(context, seq, cl);
  context[cl] = 0;
  if (mo_bf_test_key(bf, ksub)) mo_bf_add_key(context_bf, context);
  for (p = (uint64_t)ref_k; p < len; ++p) {
    /* erase(0,1) then append: the windows slide literally as in the reference, so for an odd
     * (ref_k - k) the k-mer window is non-contiguous during its first k-1 slides */
    memmove(context, context + 1, cl - 1);
    context[cl - 1] = seq[p];
    memmove(ksub, ksub + 1, kl - 1);
    ksub[kl - 1] = seq[p - d];
    if (mo_bf_test_key(bf, ksub)) mo_bf_add_key(context_bf, context);
  }
}

void mo_add_signatures(mo_bf *bf, mo_kmap *ref_bf, const char *pool, const uint64_t *kmer_off,
                       const uint8_t *is_ref, uint64_t n) {
  char buf[512];
  uint64_t i;
  for (i = 0; i < n; ++i) { /* main.cpp:133-140 */
    uint64_t l = kmer_off[i + 1] - kmer_off[i];
    if (l >= sizeof(buf)) abort();
    memcpy(buf, pool + kmer_off[i], l);
    buf[l] = 0;
    if (is_ref[i])
      mo_kmap_add_key(ref_bf, buf);
    else
      mo_bf_add_key(bf, buf);
  }
}

void mo_coverages(const mo_bf *bf, const mo_kmap *ref_bf, const char *pool, const uint64_t *kmer_off,
                  const uint64_t *sig_kmer_off, const uint64_t *allele_sig_off, const uint8_t *allele_is_ref,
                  uint64_t n_alleles, uint32_t *cov) {
  char buf[512];
  uint64_t a, s, q;
  for (a = 0; a < n_alleles; ++a) { /* main.cpp:157-182 */
    unsigned allele_cov = 0;
    for (s = allele_sig_off[a]; s < allele_sig_off[a + 1]; ++s) {
      unsigned curr_cov = 0;
      int n = 0;
      for (q = sig_kmer_off[s]; q < sig_kmer_off[s + 1]; ++q) {
        uint64_t l = kmer_off[q + 1] - kmer_off[q];
        int w;
        if (l >= sizeof(buf)) abort();
        memcpy(buf, pool + kmer_off[q], l);
        buf[l] = 0;
        w = allele_is_ref[a] ? mo_kmap_get_count(ref_bf, buf) : (int)mo_bf_get_count(bf, buf);
        if (w > 0) {
          curr_cov = (curr_cov * (unsigned)n + (unsigned)w) / (unsigned)(n + 1);
          ++n;
        }
      }
      if (curr_cov > allele_cov) allele_cov = curr_cov;
    }
    cov[a] = allele_cov;
  }
}

/* ------------------------------------------------------------------------ */
/* genotype likelihoods (var_block.hpp:224-330, 792-797), types as in SURVEY 8a */
/* ------------------------------------------------------------------------ */
float mo_logf(float x) { /* glibc 2.39 sysdeps/ieee754/flt-32/e_logf.c, N=16 table */
  static const struct {
    double invc, logc;
  } T[16] = {
      {0x1.661ec79f8f3bep+0, -0x1.57bf7808caadep-2}, {0x1.571ed4aaf883dp+0, -0x1.2bef0a7c06ddbp-2},
      {0x1.49539f0f010bp+0, -0x1.01eae7f513a67p-2},  {0x1.3c995b0b80385p+0, -0x1.b31d8a68224e9p-3},
      {0x1.30d190c8864a5p+0, -0x1.6574f0ac07758p-3}, {0x1.25e227b0b8eap+0, -0x1.1aa2bc79c81p-3},
      {0x1.1bb4a4a1a343fp+0, -0x1.a4e76ce8c0e5ep-4}, {0x1.12358f08ae5bap+0, -0x1.1973c5a611cccp-4},
      {0x1.0953f419900a7p+0, -0x1.252f438e10c1ep-5}, {0x1p+0, 0x0p+0},
      {0x1.e608cfd9a47acp-1, 0x1.aa5aa5df25984p-5},  {0x1.ca4b31f026aap-1, 0x1.c5e53aa362eb4p-4},
      {0x1.b2036576afce6p-1, 0x1.526e57720db08p-3},  {0x1.9c2d163a1aa2dp-1, 0x1.bc2860d22477p-3},
      {0x1.886e6037841edp-1, 0x1.1058bc8a07ee1p-2},  {0x1.767dcf5534862p-1, 0x1.4043057b6ee09p-2},
  };
  static const double Ln2 = 0x1.62e42fefa39efp-1;
  static const double A[3] = {-0x1.00ea348b88334p-2, 0x1.5575b0be00b6ap-2, -0x1.ffffef20a4123p-2};
  uint32_t ix, tmp, iz;
  int i, k;
  double z, r, y0, r2, y;
  float zf;
  memcpy(&ix, &x, 4);
  if (ix == 0x3f800000) return 0.0f;
  if (ix - 0x00800000u >= 0x7f800000u - 0x00800000u) {
    if (ix * 2 == 0) return -INFINITY;
    if (ix == 0x7f800000) return x;
    if ((ix & 0x80000000u) || ix * 2 >= 0xff000000u) return NAN;
    x *= 0x1p23f;
    memcpy(&ix, &x, 4);
    ix -= 23u << 23;
  }
  tmp = ix - 0x3f330000u;
  i = (int)((tmp >> 19) % 16);
  k = (int32_t)tmp >> 23;
  iz = ix - (tmp & 0xff800000u);
  memcpy(&zf, &iz, 4);
  z = (double)zf;
  r = z * T[i].invc - 1;
  y0 = T[i].logc + (double)k * Ln2;
  r2 = r * r;
  y = A[1] * r + A[2];
  y = A[0] * r2 + y;
  y = y * r2 + (y0 + r);
  return (float)y;
}

static double log_binomial(int n, int k) { /* var_block.hpp:792-797 */
  if (n == 0 || n == k || k == 0) return 0;
  return n * log((double)n) - k * log((double)k) - (n - k) * log((double)(n - k));
}

int mo_genotype(const uint32_t *cov, const float *freq, int n_alleles, float error_rate, int max_cov,
                int haploid, double *probs, int *status) {
  int i, ng = 0, vetoes = 0;
  unsigned total_sum = 0;
  size_t n = (size_t)n_alleles;
  for (i = 0; i < n_alleles; ++i) /* var_block.hpp:237-246: one {best,0} per offending allele */
    if ((int)cov[i] > max_cov) probs[vetoes++] = 0.0;
  if (vetoes) {
    *status = 1;
    return vetoes;
  }
  if (n_alleles == 1) { /* var_block.hpp:252-257 */
    probs[0] = 1.0;
    *status = 0;
    return 1;
  }
  for (i = 0; i < n_alleles; ++i) total_sum += cov[i];
  if (total_sum == 0) { /* var_block.hpp:260-266 */
    probs[0] = 0.0;
    *status = 2;
    return 1;
  }
  *status = 0;
  {
    unsigned g1, g2;
    for (g1 = 0; g1 < (unsigned)n_alleles; ++g1) {
      for (g2 = g1; g2 < (unsigned)n_alleles; ++g2) {
        double log_prior, log_posterior, log_prob, prob = 0;
        if (haploid && g2 != g1) break;
        if (g1 == g2) { /* var_block.hpp:275-278 / 298-303 */
          unsigned truth = cov[g1], error = total_sum - truth;
          log_prior = 2 * logf(freq[g1]);
          log_posterior = log_binomial((int)(truth + error), (int)truth) + truth * logf(1 - error_rate) +
                          error * logf(error_rate / (n - 1));
        } else { /* var_block.hpp:307-317 */
          unsigned t1 = cov[g1], t2 = cov[g2], error = total_sum - t1 - t2;
          log_prior = logf(2 * freq[g1] * freq[g2]);
          log_posterior = log_binomial((int)(t1 + t2 + error), (int)(t1 + t2)) +
                          log_binomial((int)(t1 + t2), (int)t1) + t1 * logf((1 - error_rate) / 2) +
                          t2 * logf((1 - error_rate) / 2);
          if (n > 2) log_posterior += error * logf(error_rate / (n - 2));
        }
        log_prob = log_prior + log_posterior;
        if (!isinf(log_prob)) prob = exp(log_prob);
        probs[ng++] = prob;
      }
    }
  }
  return ng;
}

void mo_call(const double *probs, int n_gts, int *best_idx, int *gq) { /* var_block.hpp:367-394 */
  double total = 0.0, best = 0.0;
  int i, bi = 0;
  for (i = 0; i < n_gts; ++i) total += probs[i];
  for (i = 0; i < n_gts; ++i) {
    double q = probs[i] / total;
    if (q > best) {
      bi = i;
      best = q;
    }
  }
  *best_idx = bi;
  *gq = (int)round(best * 100);
}

void mo_genotype_batch(const uint32_t *cov, const float *freq, const uint64_t *var_allele_off, uint64_t n_variants,
                       float error_rate, int max_cov, int haploid, double *lik, const uint64_t *lik_off,
                       int32_t *n_gts, int32_t *status, int32_t *best, int32_t *gq) {
  uint64_t v;
  for (v = 0; v < n_variants; ++v) {
    const uint64_t a0 = var_allele_off[v];
    const int n = (int)(var_allele_off[v + 1] - a0);
    int st = 2, bi = 0, q = 0, ng = 0;
    if (n > 0) { /* a variant without alleles reserves no slot: nothing is written for it */
      ng = mo_genotype(cov + a0, freq + a0, n, error_rate, max_cov, haploid, lik + lik_off[v], &st);
      mo_call(lik + lik_off[v], ng, &bi, &q);
    }
    n_gts[v] = ng;
    status[v] = st;
    best[v] = bi;
    gq[v] = q;
  }
}
