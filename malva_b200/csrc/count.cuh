// K6: canonical k-mer counting on the device -- the step BEFORE the MALVA hot path (SURVEY 8f-4): what the wrapper
// script obtains from `kmc -k43 -ci2 -cs255` (MALVA:107) and malva-geno then lists with the KMC API
// (main.cpp:482-490).  Semantics restated from what the reference's shipped golden pins (SURVEY 8c): canonical
// k-mers (the lexicographic minimum of a k-mer and its reverse complement), windows that contain a non-ACGT symbol
// are skipped, k-mers seen fewer than `min_count` times are dropped, counts saturate at `counter_max`.
//
//   k_count_kmers   each CTA stages a tile of the read bytes (+ k-1 halo) in shared memory; each thread rolls
//                   CNT_RUN consecutive windows through two 128-bit registers (forward strand shifting left, reverse
//                   complement shifting right) and a run length of valid symbols, and inserts the canonical word of
//                   every valid window into an open-addressing table of 32-byte slots {key 16 B, count 4 B}: one
//                   16-byte read of the home slot, a 128-bit CAS only when the slot is empty, one atomicAdd.
//                   Restricted builds (mg_count_restrict) insert only the windows the index can use (index_hit).
//   k_pack_*        the 2-bit copy of the runs of >= k bases (mg_count_add_keep): a stream compaction per sub-chunk
//   k_count_packed  the same windows counted from that copy (mg_count_add_packed); both counting kernels hand each
//                   window to count_window
//   k_count_rehash  table growth (load factor <= 0.5)
//   k_count_emit    kept entries (count >= min_count, saturated) appended to dense arrays; a radix sort by key then
//                   gives KMC's listing order.
#pragma once
#include <cuda_runtime.h>

#include <cstdint>
#include <cub/block/block_scan.cuh>

#include "index.cuh"
#include "xxh3.cuh"

namespace mg {

struct CountSlot {
  u128 key;  // canonical packed k-mer; {~0, ~0} = empty
  uint32_t count;
  uint32_t pad[3];
};
static_assert(sizeof(CountSlot) == 32, "one sector per slot");

constexpr int CNT_THREADS = 256;
constexpr int CNT_RUN = 16;
constexpr int CNT_TILE = CNT_THREADS * CNT_RUN;

__device__ __forceinline__ uint64_t count_hash(u128 x) {
  uint64_t h = (x.lo ^ (x.hi * 0x9E3779B97F4A7C15ULL)) * 0xBF58476D1CE4E5B9ULL;
  h ^= h >> 31;
  h *= 0x94D049BB133111EBULL;
  return h ^ (h >> 29);
}

__device__ __forceinline__ void count_insert(CountSlot *table, uint64_t mask, u128 key, uint32_t add,
                                             unsigned long long *n_distinct) {
  uint64_t slot = count_hash(key) & mask;
  const u128 empty = {~0ull, ~0ull};
  while (true) {
    u128 *kp = &table[slot].key;
    uint4 q = __ldcv(reinterpret_cast<const uint4 *>(kp));
    u128 cur = {(uint64_t)q.x | ((uint64_t)q.y << 32), (uint64_t)q.z | ((uint64_t)q.w << 32)};
    // (a half that reads as all-ones may be one side of a 128-bit store in flight: let the CAS return the truth)
    if (cur.lo == ~0ull || cur.hi == ~0ull) {
      cur = cas128(kp, empty, key);
      if (cur.lo == ~0ull && cur.hi == ~0ull) {
        atomicAdd(n_distinct, 1ull);
        cur = key;
      }
    }
    if (cur.lo == key.lo && cur.hi == key.hi) {
      atomicAdd(&table[slot].count, add);
      return;
    }
    slot = (slot + 1) & mask;
  }
}

// Restricted counting (mg_count_restrict): whether the sample scan can do anything with the canonical ref_k-mer
// `canon` -- its central kc-mer, taken as k_scan takes it from a KMC record, sets a bit of bf or is a ref key of
// ref_bf.  Decided from the filter bits and the keys of the probe line only (immutable after mg_finalize_alt), so
// every occurrence of a ref_k-mer gets the same answer.  KC: kc specialised (K = 0: v.k).
template <int KC>
__device__ __forceinline__ bool index_hit(const DevView &v, u128 canon, int ref_k) {
  const int kc = KC > 0 ? KC : v.k;
  const int tail = ref_k - kc - (ref_k - kc) / 2;  // (as k_scan: bases of the context after the k-mer)
  u128 c;
  const uint64_t idx = bf_index(v, canon_hash_k<KC>(mask128(shr128(canon, 2 * tail), 2 * kc), kc, &c));
  if (!occ_test(v, idx)) return false;  // (L2: the probe line holds nothing for this k-mer)
  const auto at = line_at(v, idx >> 8);
  int j;
  uint4 m;
  if (line_alt(at, (uint32_t)(idx & 255), &j, &m)) return true;
  uint32_t w3;
  bool ovf;
  if (line_key<KC>(v, at, c, &w3, &ovf) >= 0) return true;
  return ovf && ovf_find(v, c) >= 0;
}

// One valid window of either counting kernel, from its forward and reverse-complement words: the canonical form, the
// prefix-partition test, the index test of a restricted build (KC >= 0), the insert; ++*mine when inserted.
template <int KC>
__device__ __forceinline__ void count_window(const u128 &f, const u128 &r, int k, int part_bits, uint32_t part_lo, uint32_t part_hi,
                                             const DevView &v, CountSlot *table, uint64_t mask,
                                             unsigned long long *n_distinct, uint32_t &mine) {
  u128 canon = less128(r, f) ? r : f;  // (ties: the two strands are the same word)
  if (part_bits) {
    uint32_t part = (uint32_t)(shr128(canon, 2 * k - part_bits).lo);
    if (part < part_lo || part >= part_hi) return;
  }
  if constexpr (KC >= 0)
    if (!index_hit<KC>(v, canon, k)) return;
  count_insert(table, mask, canon, 1u, n_distinct);
  ++mine;
}

// seq: read bytes, records separated by any non-ACGT byte (the host puts '\n' between reads).  Window end
// positions [k-1, len).  Only canonical k-mers whose top `part_bits` bits fall in [part_lo, part_hi) are counted
// (prefix-partitioned passes for inputs whose distinct k-mers do not fit the table at once; part_bits = 0: all).
// KC < 0: every k-mer.  KC >= 0 (restricted, k = v.ref_k): only the k-mers index_hit<KC> keeps; *n_windows then
// counts the valid windows, before the partition and index tests.
template <int K, int KC>
__global__ void __launch_bounds__(CNT_THREADS) k_count_kmers(const uint8_t *__restrict__ seq, uint64_t len, int k_rt,
                                                            CountSlot *table, uint64_t mask, int part_bits,
                                                            uint32_t part_lo, uint32_t part_hi,
                                                            unsigned long long *n_distinct,
                                                            unsigned long long *n_instances, DevView v,
                                                            unsigned long long *n_windows) {
  extern __shared__ uint8_t cnt_sm[];
  const int k = K > 0 ? K : k_rt;
  uint64_t p0 = (uint64_t)(k - 1) + (uint64_t)blockIdx.x * CNT_TILE;
  uint64_t p1 = p0 + CNT_TILE < len ? p0 + CNT_TILE : len;
  uint64_t base = p0 - (uint64_t)(k - 1);
  int nbytes = (int)(p1 - base);
  for (int i = threadIdx.x; i < nbytes; i += CNT_THREADS) cnt_sm[i] = seq[base + i];
  __syncthreads();
  uint64_t q0 = p0 + (uint64_t)threadIdx.x * CNT_RUN;
  if (q0 >= p1) return;
  uint64_t q1 = q0 + CNT_RUN < p1 ? q0 + CNT_RUN : p1;
  u128 f = {0, 0}, r = {0, 0};
  int run = 0;  // valid symbols ending at the current position (saturating at k)
  const u128 m = mask128(u128{~0ull, ~0ull}, 2 * k);
  const int top = 2 * (k - 1);  // bit position of the first base
  auto push = [&](uint8_t ch) {
    uint32_t c = ch == 'A' ? 0u : ch == 'C' ? 1u : ch == 'G' ? 2u : ch == 'T' ? 3u : 4u;
    if (c > 3u) {
      run = 0;
      f.lo = f.hi = r.lo = r.hi = 0;
      return;
    }
    f.hi = (f.hi << 2) | (f.lo >> 62);
    f.lo = (f.lo << 2) | c;
    f.hi &= m.hi;
    f.lo &= m.lo;
    r.lo = (r.lo >> 2) | (r.hi << 62);
    r.hi >>= 2;
    uint64_t cc = 3u - c;
    if (top >= 64)
      r.hi |= cc << (top - 64);
    else
      r.lo |= cc << (top & 63);
    if (run < k) ++run;
  };
  int o = (int)(q0 - base) - (k - 1);
  for (int j = 0; j < k - 1; ++j) push(cnt_sm[o + j]);
  uint32_t mine = 0, seen = 0;
  for (uint64_t p = q0; p < q1; ++p) {
    push(cnt_sm[(int)(p - base)]);
    if (run < k) continue;
    if constexpr (KC >= 0) ++seen;
    count_window<KC>(f, r, k, part_bits, part_lo, part_hi, v, table, mask, n_distinct, mine);
  }
  if (mine) atomicAdd(n_instances, (unsigned long long)mine);
  if constexpr (KC >= 0)
    if (seen) atomicAdd(n_windows, (unsigned long long)seen);
}

// ---- the device-packed copy of the reads (mg_count_add_keep) and counting from it (mg_count_add_packed) ----
// A run is a maximal stretch of A/C/G/T bytes of one mg_count_add_keep call, kept when it is at least k long (the
// window rule of k_count_kmers: shorter runs hold no window).  Runs are stored 2 bits a base (A0 C1 G2 T3), 4 to a
// byte, first base in the high bits, each run from a byte boundary; a length entry per run.
//
// Per device sub-chunk, over its own bytes [own, len) (a later sub-chunk's first k-1 bytes are the halo it shares
// with the previous one): a piece is a maximal ACGT stretch there.  A piece that starts at `own` while the previous
// sub-chunk ended inside a run (`carry` bases of it so far) continues that run: its bases go on at 2-bit phase
// carry % 4, its first byte re-written from `carry_byte`.  A piece that reaches the end of the sub-chunk while more
// follow (`more`) is kept whatever its length; the host drops it later if the run ends shorter than k.
constexpr int PACK_THREADS = 256;
constexpr int PACK_RUN = 16;
constexpr int PACK_TILE = PACK_THREADS * PACK_RUN;

__device__ __forceinline__ bool is_acgt(uint8_t ch) { return ch == 'A' || ch == 'C' || ch == 'G' || ch == 'T'; }

// WRITE = false: the number of piece starts of each tile into tile_n.  WRITE = true (tile_n = their exclusive
// prefix): the start and the end position of piece i into starts[i], ends[i].
template <bool WRITE>
__global__ void __launch_bounds__(PACK_THREADS) k_pack_pieces(const uint8_t *__restrict__ seq, uint32_t own, uint32_t len,
                                                             uint32_t *tile_n, uint32_t *starts, uint32_t *ends) {
  using Scan = cub::BlockScan<uint32_t, PACK_THREADS>;
  __shared__ typename Scan::TempStorage tmp;
  const uint64_t p0 = (uint64_t)own + (uint64_t)blockIdx.x * PACK_TILE + (uint64_t)threadIdx.x * PACK_RUN;
  const uint64_t p1 = p0 + PACK_RUN < len ? p0 + PACK_RUN : len;
  auto start_at = [&](uint64_t p) { return is_acgt(seq[p]) && (p == own || !is_acgt(seq[p - 1])); };
  uint32_t n = 0;
  for (uint64_t p = p0; p < p1; ++p) n += start_at(p);
  uint32_t before, total;
  Scan(tmp).ExclusiveSum(n, before, total);
  if (!WRITE) {
    if (threadIdx.x == 0) tile_n[blockIdx.x] = total;
    return;
  }
  uint32_t rank = tile_n[blockIdx.x] + before;  // starts at positions < p
  for (uint64_t p = p0; p < p1; ++p) {
    if (!is_acgt(seq[p])) continue;
    if (start_at(p)) starts[rank++] = (uint32_t)p;
    if (p + 1 == len || !is_acgt(seq[p + 1])) ends[rank - 1] = (uint32_t)p;
  }
}

struct PackPiece {
  uint32_t start, len, phase;
  uint64_t total;  // bases of the run so far (the carried ones included)
  bool kept;
};
__device__ __forceinline__ PackPiece pack_piece(const uint32_t *starts, const uint32_t *ends, uint32_t i, uint32_t own,
                                                uint32_t len, uint32_t carry, bool more, int k) {
  PackPiece q;
  q.start = starts[i];
  q.len = ends[i] - q.start + 1;
  const bool cont = i == 0 && carry && q.start == own;
  q.phase = cont ? carry & 3u : 0u;
  q.total = (uint64_t)q.len + (cont ? carry : 0u);
  q.kept = q.total >= (uint64_t)k || (more && ends[i] + 1 == len);
  return q;
}

// per piece: (output bytes << 32) | kept, for an exclusive scan that gives output byte offsets and run ranks;
// val[n] = 0 so that the scan's last entry holds the totals.  flags: bit 0 piece 0 continues the carried run, bit 1
// it is kept.
__global__ void k_pack_plan(const uint32_t *starts, const uint32_t *ends, uint32_t n, uint32_t own, uint32_t len,
                            uint32_t carry, int more, int k, unsigned long long *val, unsigned long long *flags) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) {
    val[n] = 0;
    return;
  }
  const PackPiece q = pack_piece(starts, ends, i, own, len, carry, more, k);
  val[i] = q.kept ? ((unsigned long long)((q.phase + q.len + 3) / 4) << 32) | 1ull : 0ull;
  if (i == 0) *flags = (carry && q.start == own ? 1ull : 0ull) | (q.kept ? 2ull : 0ull);
}

// one thread per output byte: its piece by binary search over the scanned offsets, 4 bases (or the carried byte's
// bases before the phase of a continued run); the thread of a piece's first byte writes the run's length.
__global__ void k_pack_write(const uint8_t *__restrict__ seq, const uint32_t *starts, const uint32_t *ends, uint32_t n,
                             const unsigned long long *off, uint32_t own, uint32_t len, uint32_t carry,
                             uint8_t carry_byte, int more, int k, uint8_t *out, uint32_t *run_len) {
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= (off[n] >> 32)) return;
  uint32_t lo = 0, hi = n;  // the last piece i with off_bytes[i] <= j (a kept one: a dropped piece has no bytes)
  while (hi - lo > 1) {
    uint32_t mid = (lo + hi) / 2;
    if ((off[mid] >> 32) <= j) lo = mid;
    else hi = mid;
  }
  const PackPiece q = pack_piece(starts, ends, lo, own, len, carry, more, k);
  const uint64_t bj = j - (off[lo] >> 32);
  uint32_t b = 0;
  for (int s = 0; s < 4; ++s) {
    const int64_t x = (int64_t)(4 * bj + s) - (int64_t)q.phase;  // base of the piece in this slot
    uint32_t c = 0;
    if (x < 0) c = (carry_byte >> (6 - 2 * s)) & 3u;
    else if (x < (int64_t)q.len) {
      const uint8_t ch = seq[q.start + x];
      c = ch == 'A' ? 0u : ch == 'C' ? 1u : ch == 'G' ? 2u : 3u;
    }
    b |= c << (6 - 2 * s);
  }
  out[j] = (uint8_t)b;
  if (bj == 0) run_len[off[lo] & 0xffffffffull] = (uint32_t)q.total;
}

// Counting from the packed copy: a staged chunk of runs, run i from byte run_off[i], run_len[i] bases; the chunk's
// base positions are tiled as k_count_kmers tiles the read bytes, and a thread finds the run of its first position by
// a binary search inside the range of runs its tile spans.  Run 0 may be the later part of a run split over two
// chunks: its first skip0 windows were counted with the earlier part.
template <int K>
__global__ void __launch_bounds__(CNT_THREADS) k_count_packed(const uint8_t *__restrict__ packed,
                                                             const uint32_t *__restrict__ run_off,
                                                             const uint32_t *__restrict__ run_len, uint32_t n_runs,
                                                             uint64_t n_pos, uint32_t skip0, int k_rt, CountSlot *table,
                                                             uint64_t mask, int part_bits, uint32_t part_lo,
                                                             uint32_t part_hi, unsigned long long *n_distinct,
                                                             unsigned long long *n_instances) {
  __shared__ uint32_t span[2];
  const int k = K > 0 ? K : k_rt;
  const uint64_t t0 = (uint64_t)blockIdx.x * CNT_TILE, t1 = t0 + CNT_TILE < n_pos ? t0 + CNT_TILE : n_pos;
  auto find = [&](uint64_t pos, uint32_t lo, uint32_t hi) {  // the last run in [lo, hi] starting at or before pos
    while (lo < hi) {
      uint32_t mid = (lo + hi + 1) / 2;
      if (4ull * run_off[mid] <= pos) lo = mid;
      else hi = mid - 1;
    }
    return lo;
  };
  if (threadIdx.x < 2) span[threadIdx.x] = find(threadIdx.x ? t1 - 1 : t0, 0, n_runs - 1);
  __syncthreads();
  const uint64_t q0 = t0 + (uint64_t)threadIdx.x * CNT_RUN;
  if (q0 >= t1) return;
  const uint64_t q1 = q0 + CNT_RUN < t1 ? q0 + CNT_RUN : t1;
  const u128 m = mask128(u128{~0ull, ~0ull}, 2 * k);
  const int top = 2 * (k - 1);
  const DevView none{};
  u128 f = {0, 0}, r = {0, 0};
  auto push = [&](uint64_t j) {
    const uint32_t c = (packed[j >> 2] >> (6 - 2 * (int)(j & 3))) & 3u;
    f.hi = ((f.hi << 2) | (f.lo >> 62)) & m.hi;
    f.lo = ((f.lo << 2) | c) & m.lo;
    r.lo = (r.lo >> 2) | (r.hi << 62);
    r.hi >>= 2;
    const uint64_t cc = 3u - c;
    if (top >= 64)
      r.hi |= cc << (top - 64);
    else
      r.lo |= cc << (top & 63);
  };
  uint32_t mine = 0;
  for (uint32_t i = find(q0, span[0], span[1]); i < n_runs; ++i) {
    const uint64_t rs = 4ull * run_off[i];
    if (rs >= q1) break;
    const uint64_t re = rs + run_len[i];
    const uint64_t first = rs + (uint64_t)(k - 1) + (i == 0 ? skip0 : 0u);  // first window end counted
    const uint64_t a = q0 > first ? q0 : first, b = re < q1 ? re : q1;
    if (a >= b) continue;
    f = r = u128{0, 0};
    for (uint64_t j = a - (uint64_t)(k - 1); j < a; ++j) push(j);
    for (uint64_t p = a; p < b; ++p) {
      push(p);
      count_window<-1>(f, r, k, part_bits, part_lo, part_hi, none, table, mask, n_distinct, mine);
    }
  }
  if (mine) atomicAdd(n_instances, (unsigned long long)mine);
}

__global__ void k_count_clear(CountSlot *table, uint64_t cap) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= cap) return;
  uint4 *p = reinterpret_cast<uint4 *>(table + i);
  p[0] = make_uint4(~0u, ~0u, ~0u, ~0u);
  p[1] = make_uint4(0, 0, 0, 0);
}

__global__ void k_count_rehash(const CountSlot *old_table, uint64_t old_cap, CountSlot *table, uint64_t mask,
                               unsigned long long *n_distinct) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= old_cap) return;
  CountSlot s = old_table[i];
  if (s.key.lo == ~0ull && s.key.hi == ~0ull) return;
  count_insert(table, mask, s.key, s.count, n_distinct);
}

// pass 0 (keys == nullptr): count the kept entries; pass 1: append them
__global__ void k_count_emit(const CountSlot *table, uint64_t cap, uint32_t min_count, uint32_t counter_max,
                             uint64_t max_count, unsigned long long *n_out, u128 *keys, uint32_t *counts) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool keep = false;
  CountSlot s;
  if (i < cap) {
    s = table[i];
    keep = !(s.key.lo == ~0ull && s.key.hi == ~0ull) && s.count >= min_count && (uint64_t)s.count <= max_count;
  }
  // warp-aggregated append
  unsigned ballot = __ballot_sync(0xffffffffu, keep);
  if (!ballot) return;
  int lane = threadIdx.x & 31, leader = __ffs(ballot) - 1;
  unsigned long long basepos = 0;
  if (lane == leader) basepos = atomicAdd(n_out, (unsigned long long)__popc(ballot));
  basepos = __shfl_sync(0xffffffffu, basepos, leader);
  if (keep && keys) {
    unsigned long long o = basepos + __popc(ballot & ((1u << lane) - 1u));
    keys[o] = s.key;
    counts[o] = s.count > counter_max ? counter_max : s.count;
  }
}

// 128-bit keys for cub::DeviceRadixSort: most significant word first
struct KmerDecomposer {
  __host__ __device__ ::cuda::std::tuple<uint64_t &, uint64_t &> operator()(u128 &key) const { return {key.hi, key.lo}; }
};

}  // namespace mg
