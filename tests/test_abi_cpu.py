"""CPU-only checks of the product library: it loads, exports every symbol the
header declares, fails loudly without a GPU, and its __host__ __device__
helpers (the exact code the kernels run) agree with the oracle."""
import ctypes as C
import os
import random
import re

import numpy as np
import pytest

from malva_b200 import _lib, build, kmc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def L():
    build.build()
    return _lib.load()


def test_header_symbols_all_exported(L):
    hdr = open(os.path.join(ROOT, "include", "malva_gpu.h")).read()
    declared = set(re.findall(r"\b(mg_[a-z0-9_]+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(L, name)


def test_fails_loudly_without_gpu(L):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    h = C.c_void_p()
    rc = L.mg_create(C.byref(h), 0, 35, 43, 1 << 20)
    assert rc == -2 and not h.value  # MG_ERR_CUDA, no silent CPU path
    assert L.mg_last_error()


def test_bad_arguments_rejected(L):
    h = C.c_void_p()
    assert L.mg_create(C.byref(h), 0, 35, 65, 1 << 20) == -1
    assert L.mg_create(C.byref(h), 0, 44, 43, 1 << 20) == -1
    assert L.mg_create(C.byref(h), 0, 35, 43, 0) == -1


def rand_str(rng, k, alpha="ACGT"):
    return "".join(rng.choice(alpha) for _ in range(k))


def test_packed_hash_matches_oracle(L, oracle_lib):
    rng = random.Random(5)
    for k in [35, 43, 1, 3, 4, 8, 9, 16, 17, 31, 32, 33, 47, 63, 64]:
        for _ in range(300):
            s = rand_str(rng, k)
            if rng.random() < 0.1:  # palindromes: ties take the reverse complement
                half = rand_str(rng, k // 2)
                rc = half[::-1].translate(str.maketrans("ACGT", "TGCA"))
                s = (half + rc)[:k] if k % 2 == 0 else s
            x = kmc.pack_kmer(s)
            lo, hi = x & (2 ** 64 - 1), x >> 64
            clo, chi = C.c_uint64(), C.c_uint64()
            h = L.mg_selftest_hash_packed(lo, hi, k, C.byref(clo), C.byref(chi))
            buf = C.create_string_buffer(k + 1)
            oracle_lib.mo_canonical(s.encode(), k, buf)
            canon = buf.raw[:k]
            assert h == oracle_lib.mo_xxh3_64(canon, k), (k, s)
            assert kmc.unpack_kmer((chi.value << 64) | clo.value, k).encode() == canon
            if k == 35:
                assert L.mg_selftest_hash_packed_k35(lo, hi) == h
            if k == 43:
                assert L.mg_selftest_hash_packed_k43(lo, hi) == h


def test_ascii_hash_matches_oracle(L, oracle_lib):
    rng = random.Random(6)
    for _ in range(3000):
        n = rng.choice([0, 1, 2, 3, 5, 8, 9, 15, 16, 17, 30, 35, 35, 35, 43, 64, 100, 128])
        s = rand_str(rng, n, rng.choice(["ACGT", "ACGTN", "ACGTNWMKRYacgtn"])).encode()
        buf = C.create_string_buffer(n + 1)
        oracle_lib.mo_canonical(s, n, buf)
        assert L.mg_selftest_hash_ascii(s, n) == oracle_lib.mo_xxh3_64(buf.raw[:n], n), s


def test_device_logf_port_matches_libm(L):
    libm = C.CDLL("libm.so.6")
    libm.logf.restype = C.c_float
    libm.logf.argtypes = [C.c_float]
    rng = np.random.default_rng(7)
    bits = np.concatenate([rng.integers(1, 0x7F800000, size=300000, dtype=np.uint32),
                           np.array([0, 1, 0x007FFFFF, 0x00800000, 0x3F800000, 0x7F7FFFFF, 0x7F800000], np.uint32)])
    for x in bits.view(np.float32).tolist():
        a = np.float32(L.mg_selftest_logf(x)).view(np.uint32)
        b = np.float32(libm.logf(x)).view(np.uint32)
        assert a == b, x


def test_genotype_host_path_matches_oracle(L, oracle_lib):
    rng = np.random.default_rng(8)
    u32p, f32p, f64p = C.POINTER(C.c_uint32), C.POINTER(C.c_float), C.POINTER(C.c_double)
    for it in range(3000):
        n = int(rng.integers(1, 6))
        haploid = int(rng.integers(0, 2))
        err = float(rng.choice([0.001, 0.01]))
        cov = rng.integers(0, 80, size=n).astype(np.uint32)
        if it % 9 == 0:
            cov[:] = 0
        if it % 10 == 0:
            cov[rng.integers(0, n)] = 201
        freq = rng.random(n).astype(np.float32)
        freq /= freq.sum()
        if it % 6 == 0:
            freq[rng.integers(0, n)] = 0
        cap = max(n * (n + 1) // 2, n)
        la, lb = np.zeros(cap), np.zeros(cap)
        st_a, st_b, bg, gq = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        na = L.mg_selftest_genotype(cov.ctypes.data_as(u32p), freq.ctypes.data_as(f32p), n, C.c_float(err), 200,
                                    haploid, la.ctypes.data_as(f64p), C.byref(st_a), C.byref(bg), C.byref(gq))
        nb = oracle_lib.mo_genotype(cov.ctypes.data_as(u32p), freq.ctypes.data_as(f32p), n, C.c_float(err), 200,
                                    haploid, lb.ctypes.data_as(f64p), C.byref(st_b))
        obi, ogq = C.c_int(), C.c_int()
        oracle_lib.mo_call(lb.ctypes.data_as(f64p), nb, C.byref(obi), C.byref(ogq))
        assert na == nb and st_a.value == st_b.value
        # same libm on the host -> bit identical here; the device is held to tests/geno_util.lik_bound
        assert np.array_equal(la[:na].view(np.uint64), lb[:nb].view(np.uint64)), (cov, freq)
        assert (bg.value, gq.value) == (obi.value, ogq.value)


def test_genotype_zero_alleles_writes_nothing(L):
    """a variant without alleles reserves no likelihood slot (include/malva_gpu.h): genotype_one writes none"""
    lik = np.full(4, 7.0)
    st, bg, gq = C.c_int(-1), C.c_int(-1), C.c_int(-1)
    ng = L.mg_selftest_genotype(np.zeros(1, np.uint32).ctypes.data_as(C.POINTER(C.c_uint32)),
                                np.zeros(1, np.float32).ctypes.data_as(C.POINTER(C.c_float)), 0, C.c_float(0.001), 200, 0,
                                lik.ctypes.data_as(C.POINTER(C.c_double)), C.byref(st), C.byref(bg), C.byref(gq))
    assert (ng, st.value, bg.value, gq.value) == (0, 2, 0, 0)
    assert (lik == 7.0).all()


def test_wordwise_packer_of_the_lookup_kernel(L):
    """pack_words<35> (xxh3.cuh, used by k_lookup_fast): packs ACGT 35-mers exactly like kmc.pack_kmer and rejects
    every other byte value at every position."""
    rng = random.Random(5)
    lo, hi = C.c_uint64(0), C.c_uint64(0)
    for _ in range(2000):
        s = "".join(rng.choice("ACGT") for _ in range(35))
        assert L.mg_selftest_pack35(s.encode(), C.byref(lo), C.byref(hi)) == 1
        assert (hi.value << 64) | lo.value == kmc.pack_kmer(s)
    base = "ACGTTGCAACGTACGTTTGACCAGTACGATCGATCGA"[:35]
    for pos in range(35):
        for byte in range(1, 256):
            if chr(byte) in "ACGT":
                continue
            b = bytearray(base.encode())
            b[pos] = byte
            assert L.mg_selftest_pack35(bytes(b) + b"\0", C.byref(lo), C.byref(hi)) == 0, (pos, byte)
