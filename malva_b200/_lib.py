"""ctypes binding of libmalva_gpu.so (the C ABI declared in include/malva_gpu.h).

There is no CPU fallback: if the shared library is missing this raises, and if
no CUDA device is usable every compute entry point returns MG_ERR_CUDA, which
``check`` turns into a ``MalvaGpuError``.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmalva_gpu.so")

u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)
u16p = C.POINTER(C.c_uint16)
u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
f32p = C.POINTER(C.c_float)
f64p = C.POINTER(C.c_double)


class MalvaGpuError(RuntimeError):
    pass


class VariantBatch(C.Structure):
    _fields_ = [
        ("n_variants", C.c_uint64),
        ("var_allele_off", u64p),
        ("allele_sig_off", u64p),
        ("sig_kmer_off", u64p),
        ("kmer_off", u64p),
        ("pool", C.c_void_p),
        ("freq", f32p),
    ]


class GenotypeOut(C.Structure):
    _fields_ = [
        ("cov", u32p),
        ("n_gts", i32p),
        ("status", i32p),
        ("best_gt", i32p),
        ("gq", i32p),
        ("lik_off", u64p),
        ("lik", f64p),
    ]


class PackedBatch(C.Structure):
    _fields_ = [
        ("n_variants", C.c_uint64),
        ("var_allele_off", u32p),
        ("allele_sig_off", u32p),
        ("sig_kmer_off", u32p),
        ("kmers", C.c_void_p),
        ("freq", f32p),
        ("n_irregular", C.c_uint64),
        ("irr_off", u64p),
        ("irr_pool", C.c_void_p),
        ("irr_kmer", u32p),
    ]


class PackedDims(C.Structure):
    _fields_ = [("n_variants", C.c_uint64), ("n_alleles", C.c_uint64), ("n_sigs", C.c_uint64),
                ("n_kmers", C.c_uint64), ("irr_pool_bytes", C.c_uint64), ("lik_slots", C.c_uint64)]


# every symbol include/malva_gpu.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "mg_last_error": (C.c_char_p, []),
    "mg_version": (C.c_int, []),
    "mg_device_count": (C.c_int, []),
    "mg_warmup": (C.c_int, [C.c_int]),
    "mg_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int, C.c_uint64]),
    "mg_destroy": (None, [C.c_void_p]),
    "mg_add_signatures": (C.c_int, [C.c_void_p, C.c_char_p, u64p, u8p, C.c_uint64]),
    "mg_add_signatures_packed": (C.c_int, [C.c_void_p, C.c_void_p, u8p, C.c_uint64]),
    "mg_finalize_alt": (C.c_int, [C.c_void_p]),
    "mg_scan_reference": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64]),
    "mg_finalize_context": (C.c_int, [C.c_void_p]),
    "mg_scan_sample_kmers": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "mg_scan_sample_kmers_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    "mg_kmc_open": (C.c_int, [C.c_void_p, u64p, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                              C.c_uint64]),
    "mg_scan_kmc_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64]),
    "mg_sync": (C.c_int, [C.c_void_p]),
    "mg_genotype": (C.c_int, [C.c_void_p, C.POINTER(VariantBatch), C.POINTER(GenotypeOut), C.c_float, C.c_int,
                              C.c_int]),
    "mg_genotype_packed": (C.c_int, [C.c_void_p, C.POINTER(PackedBatch), C.POINTER(GenotypeOut), C.c_float, C.c_int,
                                     C.c_int]),
    "mg_genotype_packed_device": (C.c_int, [C.c_void_p, C.POINTER(PackedBatch), C.POINTER(GenotypeOut),
                                            C.POINTER(PackedDims), C.c_float, C.c_int, C.c_int]),
    "mg_lookup_packed_device": (C.c_int, [C.c_void_p, C.POINTER(PackedBatch), C.POINTER(PackedDims), C.c_void_p]),
    "mg_genotype_weights_device": (C.c_int, [C.c_void_p, C.POINTER(PackedBatch), C.POINTER(GenotypeOut),
                                             C.POINTER(PackedDims), C.c_void_p, C.c_float, C.c_int, C.c_int]),
    "mg_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mg_count_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_int]),
    "mg_count_destroy": (None, [C.c_void_p]),
    "mg_count_set_partition": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_uint32]),
    "mg_count_reset": (C.c_int, [C.c_void_p]),
    "mg_count_add": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint64]),
    "mg_count_restrict": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mg_count_set_limit": (C.c_int, [C.c_void_p, C.c_uint64]),
    "mg_count_add_keep": (C.c_int, [C.c_void_p, C.c_char_p, C.c_uint64, u8p, C.c_uint64, u32p, C.c_uint64, u64p, u64p]),
    "mg_count_add_packed": (C.c_int, [C.c_void_p, u8p, C.c_uint64, u32p, C.c_uint64]),
    "mg_count_finish": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint64, u64p]),
    "mg_count_download": (C.c_int, [C.c_void_p, u64p, u32p, C.c_uint64]),
    "mg_count_stats": (C.c_int, [C.c_void_p, u64p, C.c_int]),
    "mg_scan_counted": (C.c_int, [C.c_void_p, C.c_void_p]),
    "mg_test_keys": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, u64p, C.c_uint64, u8p]),
    "mg_get_counts": (C.c_int, [C.c_void_p, C.c_char_p, u64p, u8p, C.c_uint64, i32p]),
    "mg_bf_popcount": (C.c_int, [C.c_void_p, C.c_int, u64p]),
    "mg_bf_download_bits": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_uint64]),
    "mg_bf_download_counts": (C.c_int, [C.c_void_p, u16p, C.c_uint64]),
    "mg_kmap_size": (C.c_int, [C.c_void_p, u64p]),
    "mg_index_stats": (C.c_int, [C.c_void_p, u64p, C.c_int]),
    "mg_counters_gather": (C.c_int, [C.c_void_p]),
    "mg_counters_scatter": (C.c_int, [C.c_void_p]),
    "mg_counter_buffers": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), u64p]),
    "mg_reduce_counts": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "mg_replicate": (C.c_int, [C.POINTER(C.c_void_p), C.c_void_p, C.c_int]),
    "mg_samples_begin": (C.c_int, [C.c_void_p, C.c_int]),
    "mg_samples_capacity": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "mg_samples_take": (C.c_int, [C.c_void_p, C.c_int]),
    "mg_genotype_samples_packed": (C.c_int, [C.c_void_p, C.POINTER(PackedBatch), C.POINTER(GenotypeOut), C.c_int,
                                             C.c_float, C.c_int, C.c_int]),
    "mg_samples_end": (C.c_int, [C.c_void_p]),
    "mg_export_set_bits": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_uint64, u64p]),
    "mg_import_set_bits": (C.c_int, [C.c_void_p, C.c_int, u64p, C.c_uint64]),
    "mg_export_ref_keys": (C.c_int, [C.c_void_p, u64p, C.c_uint64, u64p]),
    "mg_event_record": (C.c_int, [C.c_void_p, C.c_int]),
    "mg_event_elapsed_ms": (C.c_int, [C.c_void_p, C.c_int, C.c_int, f32p]),
    "mg_event_sync": (C.c_int, [C.c_void_p, C.c_int]),
    "mg_genotype_kernel_ms": (C.c_int, [C.c_void_p, f32p]),
    "mg_refpass_kernel_ms": (C.c_int, [C.c_void_p, f32p]),
    "mg_launch_count": (C.c_int, [C.c_void_p, u64p]),
    "mg_diag_bandwidth": (C.c_int, [C.c_int, C.c_int, C.c_uint64, C.c_int, f64p]),
    "mg_host_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t]),
    "mg_host_free": (C.c_int, [C.c_void_p]),
    "mg_selftest_hash_packed": (C.c_uint64, [C.c_uint64, C.c_uint64, C.c_int, u64p, u64p]),
    "mg_selftest_hash_packed_k35": (C.c_uint64, [C.c_uint64, C.c_uint64]),
    "mg_selftest_hash_packed_k43": (C.c_uint64, [C.c_uint64, C.c_uint64]),
    "mg_selftest_hash_ascii": (C.c_uint64, [C.c_char_p, C.c_int]),
    "mg_selftest_logf": (C.c_float, [C.c_float]),
    "mg_selftest_genotype": (C.c_int, [u32p, f32p, C.c_int, C.c_float, C.c_int, C.c_int, f64p, C.POINTER(C.c_int),
                                       C.POINTER(C.c_int), C.POINTER(C.c_int)]),
}

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MalvaGpuError(
            f"{LIB_PATH} is missing: build it with `python -m malva_b200.build` "
            "(there is no CPU fallback for the MALVA hot path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().mg_last_error()
        raise MalvaGpuError(f"libmalva_gpu error {rc}: {msg.decode() if msg else '?'}")
