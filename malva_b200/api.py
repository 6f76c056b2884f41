"""Host-side mirror of the reference's hot-path interface, over the C ABI.

The reference drives three objects -- ``BF bf``, ``BF context_bf``, ``KMAP ref_bf``
(main.cpp:300-302) -- through per-k-mer methods.  ``MalvaGpu`` owns the device
copies of all three and exposes the same operations as batch calls, with the
reference's names where a 1:1 method exists:

    reference                                      here
    ---------------------------------------------  -----------------------------------
    add_kmers_to_bf(bf, ref_bf, kmers)  main:122   MalvaGpu.add_signatures(kmers, is_ref)
    bf.switch_mode()                    main:378   MalvaGpu.finalize_alt()
    reference rolling loop              main:385   MalvaGpu.scan_reference(seq)
    context_bf.switch_mode()            main:404   MalvaGpu.finalize_context()
    KMC loop: increment / test_key      main:487   MalvaGpu.scan_sample_kmers(packed, counts)
    set_coverages + VB::genotype        main:151   MalvaGpu.genotype(batch, ...)
    (one run per sample)                           MalvaGpu.samples_begin / samples_take / genotype_samples_packed
    BF::test_key / KMAP::test_key                  MalvaGpu.bf.test_key(...) etc. (views)
    BF::get_count / KMAP::get_count                MalvaGpu.bf.get_count(...)

All arithmetic runs in the CUDA kernels of malva_b200/csrc; nothing here
computes a hash, a count or a likelihood on the CPU.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Iterable, List, Sequence

import numpy as np

from . import _lib
from ._lib import MalvaGpuError, check  # noqa: F401
from .kmc import KMER_DTYPE

BF_ALT, BF_CONTEXT, KMAP_REF = 0, 1, 2


def _as_bytes(k) -> bytes:
    return k if isinstance(k, (bytes, bytearray)) else str(k).encode()


def make_pool(kmers: Iterable) -> tuple:
    """list of ASCII k-mers -> (pool bytes, u64 offsets[n+1])."""
    ks = [_as_bytes(k) for k in kmers]
    off = np.zeros(len(ks) + 1, dtype=np.uint64)
    if ks:
        off[1:] = np.cumsum([len(k) for k in ks], dtype=np.uint64)
    return b"".join(ks), off


def _p(a: np.ndarray, typ):
    return a.ctypes.data_as(typ)


@dataclass
class SignatureBatch:
    """CSR image of a list of VK_GROUPs (var_block.hpp:33): variant -> allele -> signature -> k-mers."""
    var_allele_off: np.ndarray
    allele_sig_off: np.ndarray
    sig_kmer_off: np.ndarray
    kmer_off: np.ndarray
    pool: bytes
    freq: np.ndarray

    @property
    def n_variants(self) -> int:
        return len(self.var_allele_off) - 1

    @staticmethod
    def from_nested(variants: Sequence[Sequence[Sequence[Sequence]]], freqs: Sequence[Sequence[float]]) -> "SignatureBatch":
        """variants[v][allele][signature] = list of k-mer strings; freqs[v][allele] = a-priori frequency."""
        vao, aso, sko, kmers, fr = [0], [0], [0], [], []
        for v, alleles in enumerate(variants):
            assert len(freqs[v]) == len(alleles)
            for a, sigs in enumerate(alleles):
                for ks in sigs:
                    kmers.extend(ks)
                    sko.append(len(kmers))
                aso.append(len(sko) - 1)
                fr.append(freqs[v][a])
            vao.append(len(aso) - 1)
        pool, koff = make_pool(kmers)
        return SignatureBatch(np.array(vao, dtype=np.uint64), np.array(aso, dtype=np.uint64),
                              np.array(sko, dtype=np.uint64), koff, pool, np.array(fr, dtype=np.float32))


IRREGULAR_BIT, REF_ALLELE_BIT = 1 << 63, 1 << 62


@dataclass
class PackedSignatureBatch:
    """The batch form the C++ host sends (mg_packed_batch): k-mers that are exactly k symbols of ACGT as 2-bit words,
    the others ("irregular": shorter at a contig end, or holding N / IUPAC symbols) as text in a side pool."""
    var_allele_off: np.ndarray   # u32
    allele_sig_off: np.ndarray   # u32
    sig_kmer_off: np.ndarray     # u32
    kmers: np.ndarray            # KMER_DTYPE; hi bit 62 = ref allele, hi bit 63 = irregular
    freq: np.ndarray
    irr_off: np.ndarray          # u64 [n_irregular + 1]
    irr_pool: bytes
    irr_kmer: np.ndarray         # u32 [n_irregular]

    @property
    def n_variants(self) -> int:
        return len(self.var_allele_off) - 1

    @staticmethod
    def from_batch(b: "SignatureBatch", k: int) -> "PackedSignatureBatch":
        """re-encodes an ASCII SignatureBatch (test helper: the product's packer is csrc/host/signatures.hpp)"""
        from .kmc import ints_to_packed, pack_kmer
        nk = len(b.kmer_off) - 1
        is_ref = np.zeros(nk, bool)
        for v in range(b.n_variants):
            a0 = int(b.var_allele_off[v])
            if int(b.var_allele_off[v + 1]) > a0:
                s0, s1 = int(b.allele_sig_off[a0]), int(b.allele_sig_off[a0 + 1])
                is_ref[int(b.sig_kmer_off[s0]):int(b.sig_kmer_off[s1])] = True
        texts = [b.pool[int(b.kmer_off[i]):int(b.kmer_off[i + 1])] for i in range(nk)]
        regular = np.array([len(t) == k and set(t) <= set(b"ACGT") for t in texts], bool) if nk else np.zeros(0, bool)
        kmers = np.zeros(nk, dtype=KMER_DTYPE)
        if regular.any():
            kmers[regular] = ints_to_packed([pack_kmer(texts[i].decode()) for i in np.nonzero(regular)[0]])
        irr = np.nonzero(~regular)[0]
        hi = kmers["hi"].copy()
        lo = kmers["lo"].copy()
        hi[irr] = IRREGULAR_BIT
        lo[irr] = np.arange(len(irr), dtype=np.uint64)
        hi[is_ref] |= np.uint64(REF_ALLELE_BIT)
        kmers["hi"], kmers["lo"] = hi, lo
        pool, off = make_pool([texts[i] for i in irr])
        return PackedSignatureBatch(b.var_allele_off.astype(np.uint32), b.allele_sig_off.astype(np.uint32),
                                    b.sig_kmer_off.astype(np.uint32), kmers, b.freq, off, pool, irr.astype(np.uint32))


@dataclass
class GenotypeResult:
    cov: np.ndarray       # u32 per allele slot
    n_gts: np.ndarray     # entries of computed_gts per variant
    status: np.ndarray    # 0 normal / 1 max-coverage veto / 2 no coverage
    best_gt: np.ndarray   # emission-order index of the printed GT
    gq: np.ndarray
    lik_off: np.ndarray
    lik: np.ndarray       # un-normalised probabilities


def genotype_names(n_alleles: int, haploid: bool) -> List[str]:
    """Emission order of VB::genotype (var_block.hpp:270, 290-292)."""
    if haploid:
        return [str(g) for g in range(n_alleles)]
    return [f"{a}/{b}" for a in range(n_alleles) for b in range(a, n_alleles)]


class _View:
    """A BF or KMAP seen through its reference method names (batch of any size)."""

    def __init__(self, owner: "MalvaGpu", which: int):
        self._o, self._w = owner, which

    def add_key(self, kmers) -> None:
        if self._w == BF_CONTEXT:
            raise MalvaGpuError("context_bf is only filled by scan_reference (main.cpp:385-400)")
        ks = [kmers] if isinstance(kmers, (bytes, str)) else list(kmers)
        self._o.add_signatures(ks, [1 if self._w == KMAP_REF else 0] * len(ks))

    def test_key(self, kmers):
        single = isinstance(kmers, (bytes, str))
        ks = [kmers] if single else list(kmers)
        r = self._o.test_keys(self._w, ks)
        return bool(r[0]) if single else r

    def get_count(self, kmers):
        if self._w == BF_CONTEXT:
            raise MalvaGpuError("context_bf carries no counters on the device")
        single = isinstance(kmers, (bytes, str))
        ks = [kmers] if single else list(kmers)
        r = self._o.get_counts(ks, [1 if self._w == KMAP_REF else 0] * len(ks))
        return int(r[0]) if single else r


class MalvaGpu:
    """Device-resident bf / context_bf / ref_bf of one malva-geno run (main.cpp:300-302)."""

    def __init__(self, k: int = 35, ref_k: int = 43, bf_bits: int = 1 << 35, device: int = 0):
        self._attach(k, ref_k, bf_bits, device)
        check(self._L.mg_create(C.byref(self._h), device, k, ref_k, bf_bits))

    def _attach(self, k: int, ref_k: int, bf_bits: int, device: int) -> None:
        self._L = _lib.load()
        self._h = C.c_void_p()
        self.k, self.ref_k, self.bf_bits, self.device = k, ref_k, bf_bits, device
        self._n_samples = 0
        self.bf = _View(self, BF_ALT)
        self.context_bf = _View(self, BF_CONTEXT)
        self.ref_bf = _View(self, KMAP_REF)

    def replicate(self, device: int) -> "MalvaGpu":
        """a new context on `device` (this one's included) holding exactly this index and its live counters
        (mg_replicate: device-to-device copies, no reload); needs finalize_alt.  A sample set is not copied."""
        r = MalvaGpu.__new__(MalvaGpu)
        r._attach(self.k, self.ref_k, self.bf_bits, device)
        check(self._L.mg_replicate(C.byref(r._h), self._h, device))
        return r

    def close(self) -> None:
        if self._h:
            self._L.mg_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- index side -------------------------------------------------------
    def add_signatures(self, kmers, is_ref) -> None:
        pool, off = make_pool(kmers)
        flags = np.asarray(is_ref, dtype=np.uint8)
        assert len(flags) == len(off) - 1
        check(self._L.mg_add_signatures(self._h, pool, _p(off, _lib.u64p), _p(flags, _lib.u8p), len(flags)))

    def add_signatures_packed(self, packed: np.ndarray, is_ref) -> None:
        assert packed.dtype == KMER_DTYPE and packed.flags.c_contiguous
        flags = np.ascontiguousarray(is_ref, dtype=np.uint8)
        assert len(flags) == len(packed)
        check(self._L.mg_add_signatures_packed(self._h, packed.ctypes.data, _p(flags, _lib.u8p), len(packed)))

    def finalize_alt(self) -> None:
        check(self._L.mg_finalize_alt(self._h))

    def scan_reference(self, seq) -> None:
        s = _as_bytes(seq)
        check(self._L.mg_scan_reference(self._h, s, len(s)))

    def scan_reference_ptr(self, ptr: int, n: int) -> None:
        """contig bytes at a host address (pinned memory is copied from directly, without staging)"""
        check(self._L.mg_scan_reference(self._h, C.c_void_p(ptr), n))

    def finalize_context(self) -> None:
        check(self._L.mg_finalize_context(self._h))

    # ---- call side --------------------------------------------------------
    def scan_sample_kmers(self, packed: np.ndarray, counts: np.ndarray, sync: bool = True) -> None:
        assert packed.dtype == KMER_DTYPE and packed.flags.c_contiguous
        counts = np.ascontiguousarray(counts, dtype=np.uint32)
        assert len(counts) == len(packed)
        check(self._L.mg_scan_sample_kmers(self._h, packed.ctypes.data, counts.ctypes.data, len(packed)))
        if sync:
            self.sync()

    def scan_sample_kmers_ptr(self, lohi_ptr: int, counts_ptr: int, n: int, device: bool) -> None:
        """Raw-pointer variant: host (pinned) pointers or device pointers."""
        fn = self._L.mg_scan_sample_kmers_device if device else self._L.mg_scan_sample_kmers
        check(fn(self._h, lohi_ptr, counts_ptr, n))

    def kmc_open(self, db: dict) -> None:
        """db = malva_b200.kmc.open_kmc_db(prefix): hand the prefix LUT + header of a KMC database to the device."""
        lut = np.ascontiguousarray(db["lut"], dtype=np.uint64)
        self._kmc_record_bytes = (db["k"] - db["lut_prefix_len"]) // 4 + db["counter_size"]
        check(self._L.mg_kmc_open(self._h, _p(lut, _lib.u64p), len(lut), db["lut_prefix_len"], db["k"],
                                  db["counter_size"], db["min_count"], db["max_count"]))

    def scan_kmc_records(self, records, first_record: int = 0, n: int | None = None, sync: bool = True) -> None:
        """records: uint8 array (or host address) of whole .kmc_suf records, decoded on the device."""
        if isinstance(records, np.ndarray):
            records = np.ascontiguousarray(records, dtype=np.uint8)
            ptr = records.ctypes.data
            if n is None:
                if not getattr(self, "_kmc_record_bytes", 0):
                    raise MalvaGpuError("scan_kmc_records before kmc_open")
                n = len(records) // self._kmc_record_bytes
        else:
            ptr = int(records)
            if n is None:
                raise MalvaGpuError("scan_kmc_records: n is required with a raw address")
        check(self._L.mg_scan_kmc_records(self._h, ptr, first_record, n))
        if sync:
            self.sync()

    def sync(self) -> None:
        check(self._L.mg_sync(self._h))

    def genotype(self, batch: SignatureBatch, error_rate: float = 0.001, max_coverage: int = 200,
                 haploid: bool = False, want_lik: bool = True) -> GenotypeResult:
        nv = batch.n_variants
        na = int(batch.var_allele_off[-1]) if nv else 0
        nall = np.diff(batch.var_allele_off).astype(np.int64)
        slots = nall if haploid else nall * (nall + 1) // 2
        slots = np.maximum(slots, nall)  # the veto path emits up to n entries
        lik_off = np.zeros(nv + 1, dtype=np.uint64)
        lik_off[1:] = np.cumsum(slots, dtype=np.uint64)
        res = GenotypeResult(np.zeros(max(na, 1), np.uint32)[:na], np.zeros(nv, np.int32), np.zeros(nv, np.int32),
                             np.zeros(nv, np.int32), np.zeros(nv, np.int32), lik_off,
                             np.zeros(int(lik_off[-1]), np.float64))
        if nv == 0:
            return res
        vb = _lib.VariantBatch(nv, _p(batch.var_allele_off, _lib.u64p), _p(batch.allele_sig_off, _lib.u64p),
                               _p(batch.sig_kmer_off, _lib.u64p), _p(batch.kmer_off, _lib.u64p),
                               C.cast(C.c_char_p(batch.pool), C.c_void_p),
                               _p(batch.freq, _lib.f32p))
        cov = np.zeros(max(na, 1), np.uint32)
        out = _lib.GenotypeOut(_p(cov, _lib.u32p), _p(res.n_gts, _lib.i32p), _p(res.status, _lib.i32p),
                               _p(res.best_gt, _lib.i32p), _p(res.gq, _lib.i32p), _p(lik_off, _lib.u64p),
                               _p(res.lik, _lib.f64p) if want_lik and len(res.lik) else None)
        check(self._L.mg_genotype(self._h, C.byref(vb), C.byref(out), C.c_float(error_rate), int(max_coverage),
                                  int(bool(haploid))))
        res.cov = cov[:na]
        return res

    # ---- queries ----------------------------------------------------------
    def test_keys(self, which: int, kmers) -> np.ndarray:
        pool, off = make_pool(kmers)
        out = np.zeros(max(len(off) - 1, 1), dtype=np.uint8)
        check(self._L.mg_test_keys(self._h, which, pool, _p(off, _lib.u64p), len(off) - 1, _p(out, _lib.u8p)))
        return out[:len(off) - 1]

    def get_counts(self, kmers, is_ref) -> np.ndarray:
        pool, off = make_pool(kmers)
        flags = np.asarray(is_ref, dtype=np.uint8)
        out = np.zeros(max(len(flags), 1), dtype=np.int32)
        check(self._L.mg_get_counts(self._h, pool, _p(off, _lib.u64p), _p(flags, _lib.u8p), len(flags),
                                    _p(out, _lib.i32p)))
        return out[:len(flags)]

    def popcount(self, which: int) -> int:
        v = C.c_uint64(0)
        check(self._L.mg_bf_popcount(self._h, which, C.byref(v)))
        return v.value

    def bits(self, which: int) -> np.ndarray:
        n = (self.bf_bits + 63) // 64
        w = np.zeros(n, dtype=np.uint64)
        check(self._L.mg_bf_download_bits(self._h, which, _p(w, _lib.u64p), n))
        return w

    def bf_counts(self) -> np.ndarray:
        n = self.popcount(BF_ALT)
        out = np.zeros(max(n, 1), dtype=np.uint16)
        check(self._L.mg_bf_download_counts(self._h, _p(out, _lib.u16p), n))
        return out[:n]

    def kmap_size(self) -> int:
        v = C.c_uint64(0)
        check(self._L.mg_kmap_size(self._h, C.byref(v)))
        return v.value

    # ---- measurement ------------------------------------------------------
    def event_record(self, idx: int) -> None:
        check(self._L.mg_event_record(self._h, idx))

    def event_elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float(0)
        check(self._L.mg_event_elapsed_ms(self._h, a, b, C.byref(ms)))
        return ms.value

    def genotype_packed(self, batch: "PackedSignatureBatch", error_rate: float = 0.001, max_coverage: int = 200,
                        haploid: bool = False, want_lik: bool = True) -> GenotypeResult:
        """mg_genotype_packed: the batch form the C++ host sends (2-bit k-mer words, u32 offsets)."""
        return self._genotype_packed_sets(batch, 1, False, error_rate, max_coverage, haploid, want_lik)[0]

    def genotype_samples_packed(self, batch: "PackedSignatureBatch", error_rate: float = 0.001, max_coverage: int = 200,
                                haploid: bool = False, want_lik: bool = True,
                                n_samples: int | None = None) -> List[GenotypeResult]:
        """mg_genotype_samples_packed: genotype_packed for every sample of the set (samples_begin), one result per
        column; n_samples defaults to the size of the set."""
        n = self._n_samples if n_samples is None else n_samples
        return self._genotype_packed_sets(batch, n, True, error_rate, max_coverage, haploid, want_lik)

    def _genotype_packed_sets(self, batch, n_sets, samples, error_rate, max_coverage, haploid, want_lik):
        nv = batch.n_variants
        na = int(batch.var_allele_off[-1]) if nv else 0
        nall = np.diff(batch.var_allele_off.astype(np.int64))
        slots = np.maximum(nall if haploid else nall * (nall + 1) // 2, nall)
        lik_off = np.zeros(nv + 1, dtype=np.uint64)
        lik_off[1:] = np.cumsum(slots, dtype=np.uint64)
        res = [GenotypeResult(np.zeros(max(na, 1), np.uint32), np.zeros(nv, np.int32), np.zeros(nv, np.int32),
                              np.zeros(nv, np.int32), np.zeros(nv, np.int32), lik_off,
                              np.zeros(int(lik_off[-1]) if want_lik else 0, np.float64)) for _ in range(max(n_sets, 1))]
        if nv == 0 and not samples:
            res[0].cov = res[0].cov[:0]
            return res
        pb = _lib.PackedBatch(nv, _p(batch.var_allele_off, _lib.u32p), _p(batch.allele_sig_off, _lib.u32p),
                              _p(batch.sig_kmer_off, _lib.u32p), batch.kmers.ctypes.data, _p(batch.freq, _lib.f32p),
                              len(batch.irr_kmer), _p(batch.irr_off, _lib.u64p),
                              C.cast(C.c_char_p(batch.irr_pool), C.c_void_p), _p(batch.irr_kmer, _lib.u32p))
        outs = (_lib.GenotypeOut * len(res))()
        for o, r in zip(outs, res):
            o.cov, o.n_gts, o.status = _p(r.cov, _lib.u32p), _p(r.n_gts, _lib.i32p), _p(r.status, _lib.i32p)
            o.best_gt, o.gq = _p(r.best_gt, _lib.i32p), _p(r.gq, _lib.i32p)
            o.lik_off = _p(lik_off, _lib.u64p) if want_lik and len(r.lik) else None
            o.lik = _p(r.lik, _lib.f64p) if want_lik and len(r.lik) else None
        if samples:
            check(self._L.mg_genotype_samples_packed(self._h, C.byref(pb), outs, n_sets, C.c_float(error_rate),
                                                     int(max_coverage), int(bool(haploid))))
        else:
            check(self._L.mg_genotype_packed(self._h, C.byref(pb), outs, C.c_float(error_rate), int(max_coverage),
                                             int(bool(haploid))))
        for r in res:
            r.cov = r.cov[:na]
        return res[:n_sets]

    # ---- sample sets: several samples genotyped against this index (include/malva_gpu.h) ------------------------
    def samples_begin(self, n: int) -> None:
        """a set of n (1..32) zeroed sample columns; replaces the previous set"""
        check(self._L.mg_samples_begin(self._h, int(n)))
        self._n_samples = int(n)

    def samples_take(self, s: int) -> None:
        """the live counters (everything scanned since the last take) into column s; the live counters are zeroed"""
        check(self._L.mg_samples_take(self._h, int(s)))

    def samples_end(self) -> None:
        check(self._L.mg_samples_end(self._h))
        self._n_samples = 0

    def genotype_packed_device(self, ptrs: dict, dims: tuple, error_rate: float, max_coverage: int, haploid: bool) -> None:
        """ptrs: device addresses keyed like mg_packed_batch / mg_genotype_out fields ("lik"/"lik_off" may be 0);
        dims = (nv, na, ns, nk, n_irregular, irr_pool_bytes, lik_slots)."""
        c = lambda name, typ: C.cast(C.c_void_p(ptrs.get(name) or None), typ)
        nv, na, ns, nk, ni, ipb, slots = dims
        pb = _lib.PackedBatch(nv, c("var_allele_off", _lib.u32p), c("allele_sig_off", _lib.u32p),
                              c("sig_kmer_off", _lib.u32p), C.c_void_p(ptrs["kmers"]), c("freq", _lib.f32p), ni,
                              c("irr_off", _lib.u64p), C.c_void_p(ptrs.get("irr_pool") or None), c("irr_kmer", _lib.u32p))
        out = _lib.GenotypeOut(c("cov", _lib.u32p), c("n_gts", _lib.i32p), c("status", _lib.i32p),
                               c("best_gt", _lib.i32p), c("gq", _lib.i32p), c("lik_off", _lib.u64p), c("lik", _lib.f64p))
        dm = _lib.PackedDims(nv, na, ns, nk, ipb, slots)
        check(self._L.mg_genotype_packed_device(self._h, C.byref(pb), C.byref(out), C.byref(dm), C.c_float(error_rate),
                                                int(max_coverage), int(bool(haploid))))

    def _packed_structs(self, ptrs: dict, dims: tuple):
        c = lambda name, typ: C.cast(C.c_void_p(ptrs.get(name) or None), typ)
        nv, na, ns, nk, ni, ipb, slots = dims
        pb = _lib.PackedBatch(nv, c("var_allele_off", _lib.u32p), c("allele_sig_off", _lib.u32p),
                              c("sig_kmer_off", _lib.u32p), C.c_void_p(ptrs["kmers"]), c("freq", _lib.f32p), ni,
                              c("irr_off", _lib.u64p), C.c_void_p(ptrs.get("irr_pool") or None), c("irr_kmer", _lib.u32p))
        out = _lib.GenotypeOut(c("cov", _lib.u32p), c("n_gts", _lib.i32p), c("status", _lib.i32p),
                               c("best_gt", _lib.i32p), c("gq", _lib.i32p), c("lik_off", _lib.u64p), c("lik", _lib.f64p))
        return pb, out, _lib.PackedDims(nv, na, ns, nk, ipb, slots)

    def lookup_packed_device(self, ptrs: dict, dims: tuple, weights_ptr: int) -> None:
        """K4 alone (mg_lookup_packed_device): raw u32 counts of the batch's signature k-mers into a device buffer;
        replicas sum these vectors instead of their counters.  ptrs / dims as in genotype_packed_device."""
        pb, _, dm = self._packed_structs(ptrs, dims)
        check(self._L.mg_lookup_packed_device(self._h, C.byref(pb), C.byref(dm), C.c_void_p(weights_ptr)))

    def genotype_weights_device(self, ptrs: dict, dims: tuple, weights_ptr: int, error_rate: float, max_coverage: int,
                                haploid: bool) -> None:
        """set_coverages + VB::genotype from (summed) weights (mg_genotype_weights_device); masks the bf weights to
        uint16_t in place first."""
        pb, out, dm = self._packed_structs(ptrs, dims)
        check(self._L.mg_genotype_weights_device(self._h, C.byref(pb), C.byref(out), C.byref(dm), C.c_void_p(weights_ptr),
                                                 C.c_float(error_rate), int(max_coverage), int(bool(haploid))))

    def set_stream(self, cuda_stream: int | None) -> None:
        """library work goes to the caller's CUDA stream (a created stream, e.g. torch.cuda.Stream().cuda_stream);
        None or 0 (which is also the handle of the legacy default stream) restores the context's own"""
        check(self._L.mg_set_stream(self._h, C.c_void_p(cuda_stream or None)))

    def genotype_packed_host(self, ptrs: dict, n_variants: int, n_irregular: int, error_rate: float, max_coverage: int,
                             haploid: bool) -> None:
        """mg_genotype_packed on caller-owned HOST buffers given by address (e.g. pinned memory)."""
        c = lambda name, typ: C.cast(C.c_void_p(ptrs.get(name) or None), typ)
        pb = _lib.PackedBatch(n_variants, c("var_allele_off", _lib.u32p), c("allele_sig_off", _lib.u32p),
                              c("sig_kmer_off", _lib.u32p), C.c_void_p(ptrs["kmers"]), c("freq", _lib.f32p),
                              n_irregular, c("irr_off", _lib.u64p), C.c_void_p(ptrs.get("irr_pool") or None),
                              c("irr_kmer", _lib.u32p))
        out = _lib.GenotypeOut(c("cov", _lib.u32p), c("n_gts", _lib.i32p), c("status", _lib.i32p),
                               c("best_gt", _lib.i32p), c("gq", _lib.i32p), c("lik_off", _lib.u64p), c("lik", _lib.f64p))
        check(self._L.mg_genotype_packed(self._h, C.byref(pb), C.byref(out), C.c_float(error_rate), int(max_coverage),
                                         int(bool(haploid))))

    def scan_counted(self, counter: "KmerCounter") -> None:
        """the counted k-mers of a finished KmerCounter straight into the sample scan (no database file)"""
        check(self._L.mg_scan_counted(self._h, counter._h))
        self.sync()

    def genotype_kernel_ms(self):
        ms = (C.c_float * 3)()
        check(self._L.mg_genotype_kernel_ms(self._h, ms))
        return list(ms)

    def refpass_kernel_ms(self) -> float:
        ms = C.c_float(0)
        check(self._L.mg_refpass_kernel_ms(self._h, C.byref(ms)))
        return ms.value

    def launch_count(self) -> int:
        v = C.c_uint64(0)
        check(self._L.mg_launch_count(self._h, C.byref(v)))
        return v.value

    def counters_gather(self) -> None:
        """the counters that live inside the probe lines -> the dense arrays counter_buffers() points at"""
        check(self._L.mg_counters_gather(self._h))

    def counters_scatter(self) -> None:
        """the dense arrays (e.g. after an NCCL sum-reduce into this rank) -> back into the probe lines"""
        check(self._L.mg_counters_scatter(self._h))

    def counter_buffers(self, gather: bool = True):
        """[(device ptr, n_u32)] x 3 -- bf counters (rank order), key counts of the probe lines (line order),
        overflow counts -- for an external NCCL sum-reduce across replicas: gather, reduce, counters_scatter()
        on the destination rank."""
        if gather:
            self.counters_gather()
        p = (C.c_void_p * 3)()
        n = (C.c_uint64 * 3)()
        check(self._L.mg_counter_buffers(self._h, p, n))
        return [(p[i] or 0, int(n[i])) for i in range(3)]

    def index_stats(self) -> dict:
        s = (C.c_uint64 * 6)()
        check(self._L.mg_index_stats(self._h, s, 6))
        return dict(zip(("probe_lines", "bf_ones", "ref_keys", "overflow_keys", "overflow_capacity",
                         "irregular_ref_keys"), [int(x) for x in s]))


def reduce_counts(contexts) -> None:
    """adds the counters of contexts[1:] into contexts[0] (replicas of one index that scanned shares of the stream)"""
    arr = (C.c_void_p * len(contexts))(*[c._h.value for c in contexts])
    check(_lib.load().mg_reduce_counts(arr, len(contexts)))


class KmerCounter:
    """Canonical k-mer counting on the device (``mg_count_*``): the ``kmc -k<k> -ci2 -cs255`` step of the MALVA
    wrapper (MALVA:107).  ``add(reads)`` takes upper-case read bytes, records separated by any non-ACGT byte."""

    def __init__(self, k: int = 43, device: int = 0):
        self._L = _lib.load()
        self._h = C.c_void_p()
        self.k = k
        check(self._L.mg_count_create(C.byref(self._h), device, k))

    def close(self):
        if self._h:
            self._L.mg_count_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_partition(self, part_bits: int, lo: int, hi: int):
        check(self._L.mg_count_set_partition(self._h, part_bits, lo, hi))

    def reset(self):
        check(self._L.mg_count_reset(self._h))

    def restrict(self, g: "MalvaGpu | None") -> None:
        """Count from now on only the ref_k-mers that ``g``'s index can use (``mg_count_restrict``): their central
        k-mer sets a bit of bf or is a ref key.  ``scan_counted`` then gives ``g`` the counters an unrestricted count
        would.  Needs an empty counter (fresh or just reset) and ``g`` past ``finalize_alt``; ``g`` must stay open
        while restricted adds run.  ``None`` lifts the restriction."""
        check(self._L.mg_count_restrict(self._h, g._h if g is not None else None))

    def add(self, reads) -> None:
        b = reads if isinstance(reads, (bytes, bytearray)) else "\n".join(reads).encode()
        check(self._L.mg_count_add(self._h, bytes(b), len(b)))

    def set_limit(self, max_slots: int) -> None:
        """Cap the table at ``max_slots`` slots (0: device memory only; ``mg_count_set_limit``)."""
        check(self._L.mg_count_set_limit(self._h, max_slots))

    def add_keep(self, reads):
        """``add`` that also returns the 2-bit copy of what it counted (``mg_count_add_keep``): (uint8 packed bytes,
        uint32 run lengths) of every maximal A/C/G/T run at least k long.  Past the table limit the counter is
        overflowed (``stats()["overflowed"]``): counting stops, packing goes on."""
        b = bytes(reads if isinstance(reads, (bytes, bytearray)) else "\n".join(reads).encode())
        packed = np.zeros(len(b) // 2 + 1, dtype=np.uint8)
        run_len = np.zeros(len(b) // (self.k + 1) + 2, dtype=np.uint32)
        nb, nr = C.c_uint64(0), C.c_uint64(0)
        check(self._L.mg_count_add_keep(self._h, b, len(b), _p(packed, _lib.u8p), len(packed), _p(run_len, _lib.u32p),
                                        len(run_len), C.byref(nb), C.byref(nr)))
        return packed[:nb.value].copy(), run_len[:nr.value].copy()

    def add_packed(self, packed, run_len) -> None:
        """count a copy from ``add_keep`` (runs of several calls concatenated; ``mg_count_add_packed``)"""
        packed = np.ascontiguousarray(packed, dtype=np.uint8)
        run_len = np.ascontiguousarray(run_len, dtype=np.uint32)
        check(self._L.mg_count_add_packed(self._h, _p(packed, _lib.u8p), len(packed), _p(run_len, _lib.u32p),
                                          len(run_len)))

    def finish(self, min_count: int = 2, counter_max: int = 255, max_count: int = 10 ** 9):
        """-> (packed k-mers in ascending order, u32 counts)"""
        n = C.c_uint64(0)
        check(self._L.mg_count_finish(self._h, min_count, counter_max, max_count, C.byref(n)))
        keys = np.zeros(n.value, dtype=KMER_DTYPE)
        counts = np.zeros(n.value, dtype=np.uint32)
        check(self._L.mg_count_download(self._h, keys.ctypes.data_as(_lib.u64p), _p(counts, _lib.u32p), n.value))
        return keys, counts

    def stats(self) -> dict:
        s = (C.c_uint64 * 9)()
        check(self._L.mg_count_stats(self._h, s, 9))
        return dict(zip(("distinct", "instances", "capacity", "launches", "kernel_us", "windows", "overflowed",
                         "transfer_us", "pack_us"), [int(x) for x in s]))


def diag_bandwidth(device: int, mode: int, nbytes: int, reps: int = 3) -> float:
    """Measured ceiling in GB/s (see mg_diag_bandwidth): 0/2/3 random 32/64/128 B, 4 coalesced random lines, 1 stream."""
    g = C.c_double(0)
    check(_lib.load().mg_diag_bandwidth(device, mode, nbytes, reps, C.byref(g)))
    return g.value
