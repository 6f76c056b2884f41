"""The genotype arithmetic of the CPU oracle (oracle/malva_oracle.c), which tests/test_gpu_genotype.py holds the
device to: its batch entry equals its per-variant entries, it equals the reference's own VB::genotype on the
near-tie family (live where oracle/_ref is built, else by digest), and its likelihoods lie within the running-error
bound of tests/geno_util.lik_bound of a 50-digit evaluation of the reference's formula."""
import ctypes as C

import numpy as np
import pytest

import geno_util as gu
from parity_util import Agree

u32p, f32p, f64p = C.POINTER(C.c_uint32), C.POINTER(C.c_float), C.POINTER(C.c_double)


def _per_call(L, cov, freq, err, max_cov, haploid):
    n = len(cov)
    cov = np.ascontiguousarray(cov, dtype=np.uint32)
    freq = np.ascontiguousarray(freq, dtype=np.float32)
    probs = np.zeros(max(n * (n + 1) // 2, n, 1), dtype=np.float64)
    st, bi, gq = C.c_int(), C.c_int(), C.c_int()
    ng = L.mo_genotype(cov.ctypes.data_as(u32p), freq.ctypes.data_as(f32p), n, C.c_float(err), max_cov, int(haploid),
                       probs.ctypes.data_as(f64p), C.byref(st))
    L.mo_call(probs.ctypes.data_as(f64p), ng, C.byref(bi), C.byref(gq))
    return probs[:ng], st.value, bi.value, gq.value


def test_oracle_batch_equals_per_call(oracle_lib):
    rng = np.random.default_rng(11)
    for haploid in (False, True):
        for err in (0.001, 0.05):
            nall = rng.integers(1, 9, size=3000)
            nall[::37] = 0                                         # variants without alleles
            vao = gu.offsets(nall)
            na = int(vao[-1])
            cov = rng.integers(0, 120, size=na).astype(np.uint32)
            cov[rng.random(na) < 0.3] = 0
            cov[rng.random(na) < 0.02] = 201                       # the max-coverage veto
            freq = rng.random(na).astype(np.float32)
            freq[rng.random(na) < 0.05] = 0
            r = gu.oracle_batch(oracle_lib, cov, freq, vao, err, 200, haploid)
            for v in range(len(nall)):
                a0, a1 = int(vao[v]), int(vao[v + 1])
                if a1 == a0:
                    assert (r.n_gts[v], r.status[v], r.best[v], r.gq[v]) == (0, 2, 0, 0)
                    continue
                probs, st, bi, gq = _per_call(oracle_lib, cov[a0:a1], freq[a0:a1], err, 200, haploid)
                o = int(r.lik_off[v])
                assert (r.n_gts[v], r.status[v], r.best[v], r.gq[v]) == (len(probs), st, bi, gq), v
                assert np.array_equal(r.lik[o:o + len(probs)].view(np.uint64), probs.view(np.uint64)), v
            assert set(r.status.tolist()) == {0, 1, 2}


def test_near_tie_family_against_reference(oracle_lib, ref_or_none):
    """the family of docs: the oracle decides GT on it exactly like the reference (which is what the device is
    then held to), and the family really contains arg-maxes decided by 1-2 ulps of the log-posterior"""
    agree = Agree("test_near_tie_family_against_reference", ref_or_none)
    for err in (0.001, 0.01, 0.05):
        for n in (3, 4, 5):
            cov = gu.near_tie_family(n, 40)
            freq = gu.uniform_freq(len(cov), n)
            r = gu.oracle_batch(oracle_lib, cov.ravel(), freq.ravel(), gu.offsets([n] * len(cov)), err, 200, False)
            ties = gu.near_ties(r.lik, r.lik_off, r.n_gts, r.status)
            assert len(ties) > 0, (err, n)
            names = [f"{x}/{y}" for x in range(n) for y in range(x, n)]
            for v in range(len(cov)):
                o, g = int(r.lik_off[v]), int(r.n_gts[v])
                gt = "0/0" if r.status[v] != 0 else names[r.best[v]]
                if agree.live:
                    probs = np.zeros(64)
                    line = C.create_string_buffer(4096)
                    c, f = np.ascontiguousarray(cov[v], np.uint32), np.ascontiguousarray(freq[v])
                    ng = agree.L.ref_genotype(c.ctypes.data_as(u32p), f.ctypes.data_as(f32p), n, C.c_float(err), 200,
                                              0, probs.ctypes.data_as(f64p), 64, line, 4096)
                    assert ng == g and np.array_equal(probs[:ng].view(np.uint64), r.lik[o:o + g].view(np.uint64))
                    assert line.value.decode().rstrip("\n").split("\t")[-1] == f"{gt}:{r.gq[v]}", (cov[v], err)
                agree.record(r.lik[o:o + g].view(np.uint64), f"{gt}:{r.gq[v]}")
    agree.done()


# ---- the likelihood bound against a 50-digit evaluation of the reference's formula ----

def _logf(L, x) -> np.float32:
    return np.float32(L.mo_logf(float(np.float32(x))))


def _exact(L, mp, cov, freq, err, haploid, logs):
    """the reference's formula with its float-typed terms as the floats it computes, the rest exact"""
    n = len(cov)
    tot = int(sum(cov))
    e = np.float32(err)
    c1 = _logf(L, np.float32(1) - e)
    c2 = _logf(L, e / np.float32(n - 1))
    c3 = _logf(L, (np.float32(1) - e) / np.float32(2))
    c4 = _logf(L, e / np.float32(n - 2)) if n > 2 else np.float32(0)

    def lg(x):
        if x not in logs:
            logs[x] = mp.log(x)
        return logs[x]

    def lbin(nn, kk):
        if nn == 0 or nn == kk or kk == 0:
            return mp.mpf(0)
        return nn * lg(nn) - kk * lg(kk) - (nn - kk) * lg(nn - kk)

    out = []
    for g1 in range(n):
        for g2 in range(g1, n):
            if haploid and g2 != g1:
                break
            if g1 == g2:
                t = cov[g1]
                lp = np.float32(2) * _logf(L, freq[g1])
                post = lbin(tot, t) + mp.mpf(float(np.float32(t) * c1)) + mp.mpf(float(np.float32(tot - t) * c2))
            else:
                t1, t2 = cov[g1], cov[g2]
                lp = _logf(L, np.float32(2) * freq[g1] * freq[g2])
                post = lbin(tot, t1 + t2) + lbin(t1 + t2, t1) + mp.mpf(float(np.float32(t1) * c3)) + \
                    mp.mpf(float(np.float32(t2) * c3))
                if n > 2:
                    post += mp.mpf(float(np.float32(tot - t1 - t2) * c4))
            out.append(None if np.isinf(lp) else mp.mpf(float(lp)) + post)
    return out


def _bound_vectors(seed: int, count: int):
    """vectors with tot from 1 to 2^30 (log-uniform) that keep some likelihood away from underflow: one dominant
    allele and a few reads on the others, or an even split"""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        n = int(rng.integers(2, 6))
        tot = int(np.exp(rng.uniform(0, np.log(2.0 ** 30))))
        cov = np.zeros(n, dtype=np.int64)
        if rng.random() < 0.8:
            minor = rng.integers(0, 4, size=n)
            cov[:] = minor
            cov[int(rng.integers(0, n))] = max(tot - int(minor.sum()), 0)
        else:
            cut = np.sort(rng.integers(0, tot + 1, size=n - 1))
            cov[:] = np.diff(np.concatenate([[0], cut, [tot]]))
        freq = rng.random(n).astype(np.float32)
        freq /= freq.sum()
        err = float(rng.choice([1e-8, 1e-4, 0.001, 0.01, 0.05]))
        out.append((cov, freq.astype(np.float32), err, bool(rng.integers(0, 2))))
    return out


def test_likelihoods_within_running_error_bound(oracle_lib):
    mp = pytest.importorskip("mpmath").mp
    mp.dps = 50
    logs = {}
    checked = 0
    worst = {}   # decade of tot -> (largest observed relative error, largest bound)
    for cov, freq, err, haploid in _bound_vectors(12, 3000):
        n = len(cov)
        r = gu.oracle_batch(oracle_lib, cov, freq, [0, n], err, 2 ** 31 - 1, haploid)
        got = r.lik[:r.n_gts[0]]
        if r.status[0] != 0:
            continue
        bound = gu.lik_bound(cov[None, :], freq[None, :], err, haploid)[0]
        for i, s in enumerate(_exact(oracle_lib, mp, [int(x) for x in cov], freq, err, haploid, logs)):
            if s is None:
                assert got[i] == 0.0
                continue
            if s < -745:            # below the smallest subnormal: exp gives 0
                assert got[i] == 0.0 or s > -746
                continue
            if s < -700:            # subnormal results: relative error is not meaningful there
                continue
            ex = mp.exp(s)
            rel = float(abs(mp.mpf(float(got[i])) - ex) / ex)
            assert rel <= bound[i], (cov, freq, err, haploid, i, rel, bound[i])
            d = int(np.log10(max(int(cov.sum()), 1)))
            w = worst.get(d, (0.0, 0.0))
            worst[d] = (max(w[0], rel), max(w[1], bound[i]))
            checked += 1
    assert checked > 3000
    assert set(worst) >= set(range(0, 10)), sorted(worst)
    # what DESIGN.md §3 states: the bound stays below 1e-11 for tot < 10^3 and below 1e-9 for tot < 10^4 (the default
    # -c 200 with up to 50 alleles); the observed error passes 1e-9 from tot ~ 10^5 on
    assert max(worst[d][1] for d in range(0, 3)) < 1e-11, worst
    assert max(worst[d][1] for d in range(0, 4)) < 1e-9, worst
    assert max(worst[d][0] for d in range(0, 5)) < 1e-9, worst
    assert min(worst[d][0] for d in range(5, 10)) > 1e-9, worst
