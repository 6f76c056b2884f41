"""Shared helpers for the parity tests: seeded synthetic inputs and an oracle-side
model (oracle/liboracle.so) of one malva-geno run that mirrors MalvaGpu call for call."""
from __future__ import annotations

import ctypes as C
import hashlib
import json
import os
import random
from typing import List, Sequence

import numpy as np

from malva_b200 import kmc
from malva_b200.api import SignatureBatch, make_pool

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)
u8p = C.POINTER(C.c_uint8)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)


GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def check_digest(name: str, key: str, digest: str, live: bool, what: str = "") -> None:
    """Results that are compared with the reference's own code (oracle/_ref) where it is built are also pinned by
    their SHA-256, stored under `key` in tests/golden/<name>.json: checked here when the live comparison cannot run
    (live False).  MALVA_RECORD_DIGESTS=1 stores the digest instead."""
    path = os.path.join(GOLDEN, name + ".json")
    digests = json.load(open(path)) if os.path.exists(path) else {}
    if os.environ.get("MALVA_RECORD_DIGESTS"):
        digests[key] = digest
        with open(path, "w") as fh:
            json.dump(digests, fh, indent=0, sort_keys=True)
    elif not live:
        assert key in digests, f"no stored digest for {key} in {path}"
        assert digest == digests[key], f"{key}: results differ from the stored ones {what}"


class NoRef:
    """Stands in for oracle/_ref where it is not built: every hook does nothing and returns None."""

    def __getattr__(self, name):
        return lambda *a: None


class Agree:
    """oracle value == the reference's value, live where oracle/_ref is built (ref_lib not None); the oracle's values
    are hashed in order either way and done() checks the digest with check_digest (file oracle_vs_reference)."""

    def __init__(self, key: str, ref_lib):
        self.key, self.live = key, ref_lib is not None
        self.L = ref_lib if self.live else NoRef()
        self.h, self.n = hashlib.sha256(), 0

    def record(self, *values) -> None:
        for v in values:
            self.h.update(v.tobytes() if isinstance(v, np.ndarray) else repr(v).encode())
        self.n += 1

    def eq(self, mine, theirs, msg=None) -> None:
        if self.live:
            assert mine == theirs, msg
        self.record(mine)

    def done(self) -> None:
        check_digest("oracle_vs_reference", self.key, self.h.hexdigest(), self.live, f"({self.n} checks)")


def rand_seq(rng: random.Random, n: int, alpha: str = "ACGT") -> str:
    return "".join(rng.choice(alpha) for _ in range(n))


def make_genome(rng: random.Random, n: int, n_runs: bool = True) -> str:
    g = list(rand_seq(rng, n))
    if n_runs and n > 400:
        a = n // 3
        g[a:a + 60] = "N" * 60            # an N run (windows hash through the NUL rule)
        b = 2 * n // 3
        for off, ch in zip((0, 7, 19, 20), "WMRN"):  # isolated IUPAC symbols
            g[b + off] = ch
        g[5] = "n"                        # lower-case survives only if the caller forgets toupper
    return "".join(g).upper()


class OracleRun:
    """bf / context_bf / ref_bf of the CPU oracle, driven like MalvaGpu."""

    def __init__(self, L, k: int, ref_k: int, bf_bits: int):
        self.L, self.k, self.ref_k, self.bf_bits = L, k, ref_k, bf_bits
        self.bf = L.mo_bf_new(bf_bits)
        self.ctx = L.mo_bf_new(bf_bits)
        self.kmap = L.mo_kmap_new()

    def close(self):
        self.L.mo_bf_free(self.bf)
        self.L.mo_bf_free(self.ctx)
        self.L.mo_kmap_free(self.kmap)

    def add_signatures(self, kmers: Sequence, is_ref: Sequence[int]):
        pool, off = make_pool(kmers)
        fl = np.asarray(is_ref, dtype=np.uint8)
        self.L.mo_add_signatures(self.bf, self.kmap, pool, off.ctypes.data_as(u64p), fl.ctypes.data_as(u8p), len(fl))

    def finalize_alt(self):
        self.L.mo_bf_switch_mode(self.bf)

    def scan_reference(self, seq: str):
        s = seq.encode() if isinstance(seq, str) else seq
        self.L.mo_reference_pass(self.bf, self.ctx, s, len(s), self.k, self.ref_k)

    def finalize_context(self):
        self.L.mo_bf_switch_mode(self.ctx)

    def scan_sample_kmers(self, packed: np.ndarray, counts: np.ndarray):
        counts = np.ascontiguousarray(counts, dtype=np.uint32)
        self.L.mo_scan_packed(self.bf, self.ctx, self.kmap, packed.ctypes.data_as(u64p), counts.ctypes.data_as(u32p),
                              len(packed), self.k, self.ref_k)

    def bits(self, which: int) -> np.ndarray:
        b = self.ctx if which == 1 else self.bf
        n = (self.bf_bits + 63) // 64
        return np.ctypeslib.as_array(self.L.mo_bf_words(b), shape=(n,)).copy()

    def bf_counts(self) -> np.ndarray:
        n = self.L.mo_bf_popcount(self.bf)
        if n == 0:
            return np.zeros(0, np.uint16)
        return np.ctypeslib.as_array(self.L.mo_bf_counts(self.bf), shape=(n,)).copy()

    def kmap_size(self) -> int:
        return self.L.mo_kmap_size(self.kmap)

    def get_counts(self, kmers, is_ref) -> np.ndarray:
        out = []
        for s, r in zip(kmers, is_ref):
            s = s if isinstance(s, bytes) else s.encode()
            out.append(self.L.mo_kmap_get_count(self.kmap, s) if r else self.L.mo_bf_get_count(self.bf, s))
        return np.array(out, dtype=np.int32)

    def test_keys(self, which: int, kmers) -> np.ndarray:
        out = []
        for s in kmers:
            s = s if isinstance(s, bytes) else s.encode()
            if which == 2:
                out.append(self.L.mo_kmap_test_key(self.kmap, s))
            else:
                out.append(self.L.mo_bf_test_key(self.ctx if which == 1 else self.bf, s))
        return np.array(out, dtype=np.uint8)

    def genotype(self, batch: SignatureBatch, error_rate: float, max_cov: int, haploid: bool):
        """Returns (cov, [per-variant dict(probs, status, best, gq)])."""
        L = self.L
        na = int(batch.var_allele_off[-1])
        is_ref = np.zeros(max(na, 1), dtype=np.uint8)
        for v in range(batch.n_variants):
            if batch.var_allele_off[v + 1] > batch.var_allele_off[v]:
                is_ref[int(batch.var_allele_off[v])] = 1
        cov = np.zeros(max(na, 1), dtype=np.uint32)
        L.mo_coverages(self.bf, self.kmap, batch.pool, batch.kmer_off.ctypes.data_as(u64p),
                       batch.sig_kmer_off.ctypes.data_as(u64p), batch.allele_sig_off.ctypes.data_as(u64p),
                       is_ref.ctypes.data_as(u8p), na, cov.ctypes.data_as(u32p))
        res = []
        for v in range(batch.n_variants):
            a0, a1 = int(batch.var_allele_off[v]), int(batch.var_allele_off[v + 1])
            n = a1 - a0
            probs = np.zeros(max(n * (n + 1) // 2, n, 1), dtype=np.float64)
            st, bi, gq = C.c_int(), C.c_int(), C.c_int()
            c = np.ascontiguousarray(cov[a0:a1])
            f = np.ascontiguousarray(batch.freq[a0:a1])
            ng = L.mo_genotype(c.ctypes.data_as(u32p), f.ctypes.data_as(f32p), n, C.c_float(error_rate), max_cov,
                               int(haploid), probs.ctypes.data_as(f64p), C.byref(st))
            L.mo_call(probs.ctypes.data_as(f64p), ng, C.byref(bi), C.byref(gq))
            res.append(dict(probs=probs[:ng].copy(), status=st.value, best=bi.value if st.value == 0 else 0,
                            gq=gq.value))
        return cov[:na], res


class _DevArray:
    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<u4", "data": (ptr, False), "version": 2}


def counter_arrays(g) -> list:
    """the three u32 counter arrays of a context (what a multi-GPU run sum-reduces), gathered, as host arrays:
    bf counters (rank order), key counts of the probe lines (line order), overflow counts"""
    import torch

    g.sync()
    out = []
    for ptr, n in g.counter_buffers(gather=True):
        out.append(torch.as_tensor(_DevArray(ptr, n), device=f"cuda:{g.device}").cpu().numpy().copy() if n
                   else np.zeros(0, np.uint32))
    return out


def synth_signatures(rng: random.Random, genome: str, k: int, n_var: int, irregular: bool = True):
    """Simple per-variant signatures: the reference window (allele 0) and 1-3 mutated windows (alts).
    Returns nested[v][allele][signature] = [k-mers], freqs[v][allele]."""
    nested, freqs = [], []
    L = len(genome)
    for v in range(n_var):
        p = rng.randrange(k, L - 2 * k)
        w = genome[p:p + k]
        n_alt = rng.choice([1, 1, 1, 2, 3])
        alleles: List[List[List[str]]] = [[[w]]]
        if rng.random() < 0.3:  # a second ref signature with two k-mers (long allele style)
            alleles[0].append([genome[p + 1:p + 1 + k], genome[p + 2:p + 2 + k]])
        for a in range(n_alt):
            q = k // 2
            alt = w[:q] + rng.choice([c for c in "ACGT" if c != w[q]]) + w[q + 1:]
            if a == 1:
                alt = w[:q] + rand_seq(rng, 3) + w[q:k - 3]   # insertion-like
            sigs = [[alt]]
            if rng.random() < 0.25:
                sigs.append([alt[1:] + rng.choice("ACGT"), alt[2:] + rand_seq(rng, 2)])
            alleles.append(sigs)
        if v % 7 == 0:  # an alt signature that also occurs in the reference -> context filter veto
            p2 = rng.randrange(k, L - 2 * k)
            if all(c in "ACGT" for c in genome[p2:p2 + k]):
                alleles[1][0] = [genome[p2:p2 + k]]
        if irregular and v % 17 == 0:
            alleles[1][0] = [alleles[1][0][0][:k - 4]]        # shorter than k (contig end)
        if irregular and v % 19 == 0:
            alleles[0][0] = [w[:5] + "N" + w[6:]]             # non-ACGT ref key
        if irregular and v % 23 == 0:
            alleles[-1][0] = [w[:9] + "W" + w[10:]]           # IUPAC alt key -> NUL bytes in the hash input
        if v % 29 == 0:
            alleles.append([])                                # an allele never enumerated keeps coverage 0
        af = np.random.default_rng(rng.randrange(1 << 30)).random(len(alleles) - 1).astype(np.float32)
        af = af * np.float32(0.6 / max(1, len(af)))
        if v % 13 == 0:
            af[0] = 0.0
        f0 = np.float32(1.0 - float(af.astype(np.float64).sum()))
        nested.append(alleles)
        freqs.append([max(f0, np.float32(0))] + af.tolist())
    return nested, freqs


def flatten(nested):
    """(kmers, is_ref) in add_kmers_to_bf order."""
    ks, fl = [], []
    for alleles in nested:
        for a, sigs in enumerate(alleles):
            for sig in sigs:
                for kmer in sig:
                    ks.append(kmer)
                    fl.append(1 if a == 0 else 0)
    return ks, fl


def synth_sample(rng: random.Random, genome: str, nested, k: int, ref_k: int, n: int, big_counts: bool = False):
    """Sample ref_k-mers: windows of the genome, windows carrying alt alleles, errors, random; with duplicates."""
    d = (ref_k - k) // 2
    alts = [sig[0] for alleles in nested for sigs in alleles[1:] for sig in sigs if len(sig[0]) == k and
            all(c in "ACGT" for c in sig[0])]
    out = []
    L = len(genome)
    while len(out) < n:
        r = rng.random()
        if r < 0.45:
            p = rng.randrange(0, L - ref_k)
            w = genome[p:p + ref_k]
        elif r < 0.8 and alts:
            a = rng.choice(alts)
            w = rand_seq(rng, d) + a + rand_seq(rng, ref_k - k - d)
            if rng.random() < 0.5:  # same k-mer inside its true genomic context (context filter veto path)
                idx = genome.find(a[:k // 2])
                if idx >= d and idx + ref_k - d <= L:
                    w = genome[idx - d:idx - d + ref_k]
                    w = w[:d] + a + w[d + k:]
        else:
            w = rand_seq(rng, ref_k)
        if any(c not in "ACGT" for c in w):
            continue
        if rng.random() < 0.5:
            w = w[::-1].translate(str.maketrans("ACGT", "TGCA"))  # either strand
        out.append(w)
        if rng.random() < 0.2:
            out.append(w)  # duplicate record: both sides must accumulate it twice
    out = out[:n]
    packed = kmc.ints_to_packed([kmc.pack_kmer(w) for w in out])
    hi = 70000 if big_counts else 256
    counts = np.array([rng.randrange(2, hi) for _ in out], dtype=np.uint32)
    return out, packed, counts
