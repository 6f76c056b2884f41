"""TEST INFRASTRUCTURE ONLY -- ctypes loaders for the parity checkers.

``oracle()``  -> oracle/liboracle.so        (plain-C restatement, malva_oracle.c)
``kmc_shim()`` -> oracle/libkmc_shim.so     (the stand-in CKMCFile, kmc_shim_hooks.cpp)
``ref()``     -> oracle/_ref/libmalva_ref.so (the reference's own classes, hooks in
                                            ref_hooks.cpp; built only where
                                            /root/reference exists, shipped prebuilt)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
reference legs may import this module.  The product (malva_b200/) never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(HERE, "liboracle.so")
KMC_SHIM_SO = os.path.join(HERE, "libkmc_shim.so")
REF_SO = os.path.join(HERE, "_ref", "libmalva_ref.so")
REF_BIN = os.path.join(HERE, "_ref", "malva-geno-ref")

_u64p = C.POINTER(C.c_uint64)
_u32p = C.POINTER(C.c_uint32)
_u8p = C.POINTER(C.c_uint8)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_intp = C.POINTER(C.c_int)


def build(force: bool = False) -> None:
    """Compile liboracle.so, libkmc_shim.so (and _ref/ where the reference's sources are present: Makefile REF)."""
    if force or not os.path.exists(ORACLE_SO) or \
            os.path.getmtime(ORACLE_SO) < os.path.getmtime(os.path.join(HERE, "malva_oracle.c")):
        subprocess.check_call(["make", "-C", HERE, "liboracle.so"], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", HERE, "libkmc_shim.so"], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-C", HERE, "ref"], stdout=subprocess.DEVNULL)


_oracle = None
_ref = None


def oracle() -> C.CDLL:
    global _oracle
    if _oracle is not None:
        return _oracle
    if not os.path.exists(ORACLE_SO):
        build()
    L = C.CDLL(ORACLE_SO)
    L.mo_xxh3_64.restype = C.c_uint64
    L.mo_xxh3_64.argtypes = [C.c_char_p, C.c_size_t]
    L.mo_canonical.argtypes = [C.c_char_p, C.c_int, C.c_char_p]
    L.mo_bf_new.restype = C.c_void_p
    L.mo_bf_new.argtypes = [C.c_uint64]
    L.mo_bf_free.argtypes = [C.c_void_p]
    L.mo_bf_add_key.argtypes = [C.c_void_p, C.c_char_p]
    L.mo_bf_test_key.argtypes = [C.c_void_p, C.c_char_p]
    L.mo_bf_switch_mode.argtypes = [C.c_void_p]
    L.mo_bf_increment.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32]
    L.mo_bf_get_count.restype = C.c_uint16
    L.mo_bf_get_count.argtypes = [C.c_void_p, C.c_char_p]
    L.mo_bf_size.restype = C.c_uint64
    L.mo_bf_size.argtypes = [C.c_void_p]
    L.mo_bf_popcount.restype = C.c_uint64
    L.mo_bf_popcount.argtypes = [C.c_void_p]
    L.mo_bf_words.restype = _u64p
    L.mo_bf_words.argtypes = [C.c_void_p]
    L.mo_bf_counts.restype = C.POINTER(C.c_uint16)
    L.mo_bf_counts.argtypes = [C.c_void_p]
    L.mo_find_kmers_at.restype = C.c_uint64
    L.mo_find_kmers_at.argtypes = [C.c_char_p, C.c_int, C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_char_p,
                                   C.c_uint64]
    L.mo_kmap_new.restype = C.c_void_p
    L.mo_kmap_free.argtypes = [C.c_void_p]
    L.mo_kmap_add_key.argtypes = [C.c_void_p, C.c_char_p]
    L.mo_kmap_test_key.argtypes = [C.c_void_p, C.c_char_p]
    L.mo_kmap_increment.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.mo_kmap_get_count.argtypes = [C.c_void_p, C.c_char_p]
    L.mo_kmap_size.restype = C.c_uint64
    L.mo_kmap_size.argtypes = [C.c_void_p]
    L.mo_scan_ascii.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, _u32p, C.c_uint64, C.c_int, C.c_int]
    L.mo_scan_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, _u64p, _u32p, C.c_uint64, C.c_int, C.c_int]
    L.mo_reference_pass.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_uint64, C.c_int, C.c_int]
    L.mo_add_signatures.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, _u64p, _u8p, C.c_uint64]
    L.mo_coverages.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, _u64p, _u64p, _u64p, _u8p, C.c_uint64, _u32p]
    L.mo_genotype.argtypes = [_u32p, _f32p, C.c_int, C.c_float, C.c_int, C.c_int, _f64p, _intp]
    L.mo_call.argtypes = [_f64p, C.c_int, _intp, _intp]
    _i32p = C.POINTER(C.c_int32)
    L.mo_genotype_batch.argtypes = [_u32p, _f32p, _u64p, C.c_uint64, C.c_float, C.c_int, C.c_int, _f64p, _u64p,
                                    _i32p, _i32p, _i32p, _i32p]
    L.mo_logf.restype = C.c_float
    L.mo_logf.argtypes = [C.c_float]
    _oracle = L
    return L


def kmc_shim() -> C.CDLL:
    L = C.CDLL(KMC_SHIM_SO)
    L.shim_kmc_list.restype = C.c_long
    L.shim_kmc_list.argtypes = [C.c_char_p, _u64p, C.c_char_p, C.c_long]
    return L


def have_ref() -> bool:
    return os.path.exists(REF_SO) and os.path.exists(REF_BIN)


def ref() -> C.CDLL:
    global _ref
    if _ref is not None:
        return _ref
    L = C.CDLL(REF_SO)
    L.ref_xxh3.restype = C.c_uint64
    L.ref_xxh3.argtypes = [C.c_char_p, C.c_size_t]
    L.ref_bf_new.restype = C.c_void_p
    L.ref_bf_new.argtypes = [C.c_uint64]
    L.ref_bf_free.argtypes = [C.c_void_p]
    L.ref_bf_add_key.argtypes = [C.c_void_p, C.c_char_p]
    L.ref_bf_test_key.argtypes = [C.c_void_p, C.c_char_p]
    L.ref_bf_switch_mode.argtypes = [C.c_void_p]
    L.ref_bf_increment.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32]
    L.ref_bf_get_count.restype = C.c_uint32
    L.ref_bf_get_count.argtypes = [C.c_void_p, C.c_char_p]
    L.ref_kmap_new.restype = C.c_void_p
    L.ref_kmap_free.argtypes = [C.c_void_p]
    L.ref_kmap_add_key.argtypes = [C.c_void_p, C.c_char_p]
    L.ref_kmap_test_key.argtypes = [C.c_void_p, C.c_char_p]
    L.ref_kmap_increment.argtypes = [C.c_void_p, C.c_char_p, C.c_int]
    L.ref_kmap_get_count.argtypes = [C.c_void_p, C.c_char_p]
    L.ref_kmap_size.restype = C.c_uint64
    L.ref_kmap_size.argtypes = [C.c_void_p]
    L.ref_scan_kmer.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_uint32, C.c_int, C.c_int]
    L.ref_add_packed.argtypes = [C.c_void_p, C.c_void_p, _u64p, _u8p, C.c_uint64, C.c_int]
    L.ref_scan_packed.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, _u64p, _u32p, C.c_uint64, C.c_int, C.c_int]
    L.ref_reference_pass.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p, C.c_int, C.c_int]
    L.ref_get_counts_packed.argtypes = [C.c_void_p, C.c_void_p, _u64p, _u8p, C.c_uint64, C.c_int, C.POINTER(C.c_int32)]
    L.ref_genotype_batch.restype = C.c_uint64
    L.ref_genotype_batch.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, _u32p, _u32p, _u32p, _u64p, _f32p, C.c_int,
                                     C.c_float, C.c_int, C.c_int, _u32p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    L.ref_genotype.argtypes = [_u32p, _f32p, C.c_int, C.c_float, C.c_int, C.c_int, _f64p, C.c_int,
                               C.c_char_p, C.c_int]
    L.ref_extract_kmers.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_char_p, C.c_int]
    _ref = L
    return L
