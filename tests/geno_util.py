"""Genotype-likelihood helpers shared by the CPU and GPU genotype tests: the oracle's batch entry
(mo_genotype_batch) over numpy arrays, and the running-error bound of the reference's likelihood formula
(var_block.hpp:272-318) that both the mpmath check and the device check use."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

U53 = 2.0 ** -53
U32 = 1 << 32


def slots(nall: np.ndarray, haploid: bool) -> np.ndarray:
    """likelihood slots a variant of n alleles needs: its genotypes, or n entries on the max-coverage veto path"""
    nall = np.asarray(nall, dtype=np.int64)
    return np.maximum(nall if haploid else nall * (nall + 1) // 2, nall)


def offsets(counts) -> np.ndarray:
    off = np.zeros(len(counts) + 1, dtype=np.uint64)
    off[1:] = np.cumsum(np.asarray(counts, dtype=np.uint64), dtype=np.uint64)
    return off


@dataclass
class Calls:
    lik: np.ndarray
    lik_off: np.ndarray
    n_gts: np.ndarray
    status: np.ndarray
    best: np.ndarray
    gq: np.ndarray


def oracle_batch(L, cov, freq, var_allele_off, err: float, max_cov: int, haploid: bool) -> Calls:
    """mo_genotype + mo_call for every variant of a CSR batch (cov u32 / freq f32 per allele slot)."""
    cov = np.ascontiguousarray(cov, dtype=np.uint32)
    freq = np.ascontiguousarray(freq, dtype=np.float32)
    vao = np.ascontiguousarray(var_allele_off, dtype=np.uint64)
    nv = len(vao) - 1
    lik_off = offsets(slots(np.diff(vao.astype(np.int64)), haploid))
    lik = np.zeros(max(int(lik_off[-1]), 1), dtype=np.float64)
    outs = [np.zeros(max(nv, 1), dtype=np.int32) for _ in range(4)]
    p = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    L.mo_genotype_batch(p(cov, C.c_uint32), p(freq, C.c_float), p(vao, C.c_uint64), nv, C.c_float(err), int(max_cov),
                        int(haploid), p(lik, C.c_double), p(lik_off, C.c_uint64), *(p(o, C.c_int32) for o in outs))
    return Calls(lik[:int(lik_off[-1])], lik_off, *(o[:nv] for o in outs))


def _xlogx(x: np.ndarray) -> np.ndarray:
    x = x.astype(np.float64)
    return np.where(x > 0, x * np.log(np.where(x > 0, x, 1.0)), 0.0)


def _lbin(nn: np.ndarray, kk: np.ndarray):
    """log_binomial(n, k) = n log n - k log k - (n-k) log(n-k) (ints as the reference passes them): the value, the
    sum of |x log x| (each product carries <= 3 u: log <= 1 ulp, the product's rounding) and the sum of |partial
    results| of the two subtractions (each carries <= 1 u)."""
    a, b, c = _xlogx(nn), _xlogx(kk), _xlogx(nn - kk)
    trivial = (nn == 0) | (nn == kk) | (kk == 0)
    val = np.where(trivial, 0.0, a - b - c)
    prods = np.where(trivial, 0.0, a + b + c)
    parts = np.where(trivial, 0.0, np.abs(a - b) + np.abs(val))
    return val, prods, parts


def _i32(x: np.ndarray) -> np.ndarray:
    """the int conversion of a uint32 value (two's complement)"""
    x = x.astype(np.int64) % U32
    return np.where(x >= 1 << 31, x - U32, x)


def lik_bound(cov: np.ndarray, freq: np.ndarray, err: float, haploid: bool) -> np.ndarray:
    """Relative bound on |computed likelihood - exact value of the reference's formula| for the genotypes of rows
    of n alleles each (cov, freq: (m, n)); columns in emission order.

    Exact value: the float-typed terms (logf priors, (float)t * logf(...)) taken as the floats the reference
    computes, log_binomial and exp evaluated exactly.  A running-error bound: u = 2^-53 times (3 |x log x| for
    every product of log_binomial, plus |r| for every rounded sum r in the reference's evaluation order), plus
    2 u for exp (<= 1 ulp).  It holds for glibc's log (< 0.52 ulp) and CUDA's fp64 log (<= 1 ulp) alike; two
    implementations therefore differ by at most twice the bound."""
    cov = np.asarray(cov, dtype=np.int64)
    m, n = cov.shape
    f = np.maximum(np.asarray(freq, dtype=np.float64), 1e-300)
    tot = cov.sum(axis=1) % U32
    e = np.float32(err)
    c1 = abs(np.log(1.0 - float(e)))
    c2 = abs(np.log(float(e) / max(n - 1, 1)))
    c3 = abs(np.log((1.0 - float(e)) / 2))
    c4 = abs(np.log(float(e) / (n - 2))) if n > 2 else 0.0
    out = []
    with np.errstate(divide="ignore", invalid="ignore"):
        for g1 in range(n):
            for g2 in range(g1, n):
                if haploid and g2 != g1:
                    break
                out.append(_genotype_bound(cov, f, tot, g1, g2, n, c1, c2, c3, c4))
    return np.stack(out, axis=1) if out else np.zeros((m, 0))


def _genotype_bound(cov, f, tot, g1, g2, n, c1, c2, c3, c4):
    """lik_bound of genotype g1/g2 (g1 == g2: homozygous / haploid), var_block.hpp:272-318"""
    if g1 == g2:
        t = cov[:, g1]
        er = (tot - t) % U32
        lb, prods, parts = _lbin(_i32(t + er), _i32(t))
        lp = np.abs(2 * np.log(f[:, g1]))
        s1 = lb - t * c1
        s2 = s1 - er * c2
        runs = np.abs(s1) + np.abs(s2) + np.abs(s2 - lp)
    else:
        t1, t2 = cov[:, g1], cov[:, g2]
        er = (tot - t1 - t2) % U32
        lb1, p1, q1 = _lbin(_i32(t1 + t2 + er), _i32(t1 + t2))
        lb2, p2, q2 = _lbin(_i32(t1 + t2), _i32(t1))
        prods, parts = p1 + p2, q1 + q2
        lp = np.abs(np.log(2 * f[:, g1] * f[:, g2]))
        s1 = lb1 + lb2
        s2 = s1 - t1 * c3
        s3 = s2 - t2 * c3
        runs = np.abs(s1) + np.abs(s2) + np.abs(s3)
        if n > 2:
            s3 = s3 - er * c4
            runs = runs + np.abs(s3)
        runs = runs + np.abs(s3 - lp)
    return U53 * (3 * prods + parts + runs) * 1.001 + 2 * U53


def near_tie_family(n: int, hi: int, fillers=(0, 1)):
    """(a, b, a) at every position of n alleles, a, b in [0, hi]; the other alleles all zero or a small filler
    pattern.  With uniform priors 0/1 and 1/2 (shifted with the position) are mathematically tied whenever their
    coverages match, and the reference's arg-max comes from the last bit of log_binomial's fp64 logs."""
    a, b = np.meshgrid(np.arange(hi + 1), np.arange(hi + 1), indexing="ij")
    a, b = a.ravel(), b.ravel()
    rows = []
    for p in range(n - 2):
        for fill in (fillers if n > 3 else fillers[:1]):
            bg = np.array([(j % 3) * fill for j in range(n)], dtype=np.int64)
            blk = np.tile(bg, (len(a), 1))
            blk[:, p], blk[:, p + 1], blk[:, p + 2] = a, b, a
            rows.append(blk)
    return np.concatenate(rows)


def uniform_freq(m: int, n: int) -> np.ndarray:
    return np.full((m, n), np.float32(1.0 / n), dtype=np.float32)  # float(1/n), vcf_io.hpp:884


def near_ties(lik: np.ndarray, lik_off: np.ndarray, n_gts: np.ndarray, status: np.ndarray, max_ulps: float = 2) -> np.ndarray:
    """indices of the variants (status 0) whose two largest likelihoods differ, but by no more than max_ulps ulps of
    the log-posterior: the arg-max of those is decided by the last bits of the fp64 logs"""
    hits = []
    for g in np.unique(n_gts[status == 0]):
        rows = np.nonzero((status == 0) & (n_gts == g))[0]
        if g < 2 or not len(rows):
            continue
        idx = lik_off[rows].astype(np.int64)[:, None] + np.arange(g)[None, :]
        top = np.sort(lik[idx], axis=1)[:, -2:]
        a, b = top[:, 1], top[:, 0]
        with np.errstate(divide="ignore", invalid="ignore"):
            rel = (a - b) / a
            ulp = np.spacing(np.abs(np.log(a)))
        hits.append(rows[(b > 0) & (a != b) & (rel <= max_ulps * ulp * 1.01)])
    return np.concatenate(hits) if hits else np.zeros(0, np.int64)
