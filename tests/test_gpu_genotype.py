"""K5 (genotype_one / k_genotype) and the coverage kernels in front of it, against the CPU oracle, domain by domain.

Harness: mg_genotype_weights_device with one signature of one k-mer per allele, so that the weight vector IS the
coverage vector.  Every k-mer carries hi bit 62 (the ref-allele flag), so k_mask_alt leaves weights >= 2^16 alone;
only the u16-wrap rows of the coverage domain clear it.  Every batch runs twice, with the likelihoods returned and
with lik == NULL (the kernel's bump-allocated scratch): coverages, n_gts, status, GT and GQ must not differ.

Bar: n_gts, status, best GT and GQ exact; which likelihoods are 0 exact; NaN likelihoods with the oracle's bit
pattern; every other likelihood within twice the running-error bound of geno_util.lik_bound (both sides lie within
it of the exact value of the reference's formula, tests/test_genotype_cpu.py)."""
import itertools

import numpy as np
import pytest

import geno_util as gu

pytestmark = pytest.mark.gpu

ERRS = (0.001, 0.01, 0.05)
REF_BIT = 1 << 62
SENTINEL = np.array([0x7FF4DEADBEEF0001], dtype=np.uint64).view(np.float64)[0]   # a NaN nothing computes
GUARD = 8


@pytest.fixture(scope="module")
def ctx():
    from malva_b200 import MalvaGpu

    g = MalvaGpu(k=35, ref_k=43, bf_bits=1 << 16)
    yield g
    g.close()


def run_device(g, weights, sig_kmer_off, allele_sig_off, var_allele_off, freq, err, max_cov, haploid, want_lik,
               ref_bit=None):
    """mg_genotype_weights_device on one batch; returns (cov, Calls).  weights: u32 per k-mer (counts >= 2^31 arrive
    as negative int32, as from a sum of look-up results)."""
    import torch

    dev = torch.device("cuda", 0)
    nk = len(weights)
    vao = np.asarray(var_allele_off, dtype=np.int64)
    nv, na, ns = len(vao) - 1, int(vao[-1]), len(sig_kmer_off) - 1
    lik_off = gu.offsets(gu.slots(np.diff(vao), haploid))
    hi = np.full(nk, REF_BIT, dtype=np.int64) if ref_bit is None else np.where(ref_bit, REF_BIT, 0).astype(np.int64)
    kmers = np.stack([np.arange(nk, dtype=np.int64), hi], axis=1)
    i32 = lambda a: torch.from_numpy(np.ascontiguousarray(np.asarray(a, dtype=np.int64).astype(np.int32))).to(dev)
    t = {"var_allele_off": i32(vao), "allele_sig_off": i32(allele_sig_off), "sig_kmer_off": i32(sig_kmer_off),
         "kmers": torch.from_numpy(kmers).to(dev), "freq": torch.from_numpy(np.ascontiguousarray(freq, np.float32)).to(dev),
         "cov": torch.zeros(max(na, 1), dtype=torch.int32, device=dev)}
    for name in ("n_gts", "status", "best_gt", "gq"):
        t[name] = torch.full((nv,), -7, dtype=torch.int32, device=dev)
    if want_lik:   # GUARD slots past the last reserved one: nothing may write there
        t["lik_off"] = torch.from_numpy(lik_off.view(np.int64)).to(dev)
        t["lik"] = torch.empty((int(lik_off[-1]) + GUARD,), dtype=torch.float64, device=dev)
        t["lik"].view(torch.int64).fill_(int(np.float64(SENTINEL).view(np.int64)))
    w = torch.from_numpy(np.ascontiguousarray(np.asarray(weights, dtype=np.int64) % gu.U32).astype(np.uint32)
                         .view(np.int32)).to(dev)
    ptrs = {n: x.data_ptr() for n, x in t.items()}
    dims = (nv, na, ns, nk, 0, 0, int(lik_off[-1]))
    torch.cuda.synchronize()
    g.genotype_weights_device(ptrs, dims, w.data_ptr(), err, max_cov, haploid)
    g.sync()
    h = {n: x.cpu().numpy() for n, x in t.items()}
    lik = np.zeros(0)
    if want_lik:
        lik = h["lik"]
        assert np.array_equal(lik[int(lik_off[-1]):].view(np.uint64), np.full(GUARD, np.float64(SENTINEL)).view(np.uint64)), \
            "a write past the batch's likelihood slots"
        lik = lik[:int(lik_off[-1])]
    return h["cov"][:na].view(np.uint32), gu.Calls(lik, lik_off, h["n_gts"], h["status"], h["best_gt"], h["gq"])


def _first_bad(mask, cov_of, what):
    bad = np.nonzero(mask)[0]
    if len(bad):
        v = int(bad[0])
        raise AssertionError(f"{what}: {len(bad)} variants differ, e.g. variant {v} cov {cov_of(v)}")


def compare(L, label, cov, freq, vao, err, max_cov, haploid, dev_pair, checked):
    """device (with and without likelihoods) against the oracle on the coverage vector the device computed"""
    (cov_d, d), (cov_s, s) = dev_pair
    vao = np.asarray(vao, dtype=np.int64)
    o = gu.oracle_batch(L, cov, freq, vao, err, max_cov, haploid)
    cov_of = lambda v: cov[vao[v]:vao[v + 1]].tolist()
    tag = f"{label} err={err} haploid={haploid} max_cov={max_cov}"
    assert np.array_equal(cov_d, cov_s), f"{tag}: coverages differ between the lik and lik == NULL runs"
    for name, a, b in (("n_gts", d.n_gts, s.n_gts), ("status", d.status, s.status), ("GT", d.best, s.best),
                       ("GQ", d.gq, s.gq)):
        _first_bad(a != b, cov_of, f"{tag}: {name} with lik == NULL")
    _first_bad(d.n_gts != o.n_gts, cov_of, f"{tag}: n_gts")
    _first_bad(d.status != o.status, cov_of, f"{tag}: status")
    sub = np.array([0 < o.lik[a:a + g].max(initial=0) < 2.0 ** -1022 if g else False
                    for a, g in zip(o.lik_off[:-1].astype(np.int64), o.n_gts)]) if (d.best != o.best).any() else None
    _first_bad(d.best != o.best, cov_of, f"{tag}: GT" + ("" if sub is None else
               f" ({int((sub & (d.best != o.best)).sum())} of them with every likelihood below DBL_MIN)"))
    _first_bad(d.gq != o.gq, cov_of, f"{tag}: GQ")
    # likelihoods: constants of the veto / no-coverage / one-allele paths bit-exact, NaN bit-exact, the rest bounded
    nall = np.diff(vao)
    bad = np.zeros(len(nall), bool)
    const = np.nonzero((o.n_gts > 0) & ((o.status != 0) | (nall == 1)))[0]
    if len(const):
        ng = o.n_gts[const].astype(np.int64)
        starts = np.concatenate([[0], np.cumsum(ng)[:-1]])
        idx = np.repeat(o.lik_off[const].astype(np.int64), ng) + np.arange(int(ng.sum())) - np.repeat(starts, ng)
        diff = (d.lik[idx].view(np.uint64) != o.lik[idx].view(np.uint64)).astype(np.int64)
        bad[const] |= np.add.reduceat(diff, starts) > 0
    for n in np.unique(nall[nall > 1]):
        r = np.nonzero((nall == n) & (o.status == 0))[0]
        if not len(r):
            continue
        ng = int(o.n_gts[r[0]])
        idx = o.lik_off[r].astype(np.int64)[:, None] + np.arange(ng)[None, :]
        got, exp = d.lik[idx], o.lik[idx]
        c = np.stack([cov[vao[r] + j] for j in range(n)], axis=1).astype(np.int64)
        f = np.stack([freq[vao[r] + j] for j in range(n)], axis=1)
        nan = np.isnan(got) | np.isnan(exp)
        with np.errstate(invalid="ignore", over="ignore"):
            bound = 2 * gu.lik_bound(c, f, err, haploid) * np.abs(exp) + 2.0 ** -1070
            ok = np.where(nan, got.view(np.uint64) == exp.view(np.uint64),
                          (got == exp) | (((got == 0) == (exp == 0)) & (np.abs(got - exp) <= bound)))
        bad[r] |= ~ok.all(axis=1)
        checked["nan"] += int(nan.any(axis=1).sum())
    _first_bad(bad, cov_of, f"{tag}: likelihoods")
    checked["vectors"] += len(nall)
    return o


def run_and_compare(g, L, label, cov, freq, vao, err, max_cov, haploid, checked):
    """the one-k-mer-per-allele harness: weights = coverages"""
    na = int(vao[-1])
    ident = np.arange(na + 1)
    pair = [run_device(g, cov, ident, ident, vao, freq, err, max_cov, haploid, want) for want in (True, False)]
    assert np.array_equal(pair[0][0], np.asarray(cov, dtype=np.int64) % gu.U32), f"{label}: coverages"
    return compare(L, label, np.asarray(cov, np.uint32), freq, vao, err, max_cov, haploid, pair, checked)


def prior_sets(n: int, m: int, rng, which=("uniform", "af", "ref0", "one")):
    """(m, n) float32 priors per set: uniform float(1/n); random AFs with f0 = 1 - sum; f0 = 0; f = 1, 0, ..."""
    out = []
    for w in which:
        if w == "uniform":
            f = np.full((m, n), np.float32(1.0 / n), np.float32)
        elif w == "af":
            af = rng.random((m, n - 1)).astype(np.float32) * np.float32(0.6 / max(n - 1, 1))
            f = np.concatenate([(1.0 - af.astype(np.float64).sum(axis=1, keepdims=True)).astype(np.float32), af], axis=1)
        elif w == "ref0":
            f = np.full((m, n), np.float32(1.0 / max(n - 1, 1)), np.float32)
            f[:, 0] = 0
        else:
            f = np.zeros((m, n), np.float32)
            f[:, 0] = 1
        out.append(f)
    return out


def grid_domain(g, L, label, rows, rng, priors=("uniform", "af", "ref0", "one"), errs=ERRS, max_cov=200):
    """rows (m, n) of one allele count under every prior set, haploid and diploid, every error rate"""
    m, n = rows.shape
    fs = prior_sets(n, m, rng, priors)
    cov = np.tile(rows, (len(fs), 1))
    freq = np.concatenate(fs)
    vao = np.arange(len(cov) + 1, dtype=np.int64) * n
    checked = {"vectors": 0, "nan": 0}
    outs = {}
    for haploid in (False, True):
        for err in errs:
            outs[(haploid, err)] = run_and_compare(g, L, label, cov.ravel(), freq.ravel(), vao, err, max_cov, haploid,
                                                   checked)
    print(f"{label}: {checked['vectors']} vectors checked")
    return outs, checked


def test_d1_two_alleles_across_the_veto(ctx, oracle_lib):
    """n = 2, every coverage vector in [0, 260]^2: crosses the max-coverage veto at 200/201"""
    a, b = np.meshgrid(np.arange(261), np.arange(261), indexing="ij")
    _, checked = grid_domain(ctx, oracle_lib, "D1", np.stack([a.ravel(), b.ravel()], axis=1), np.random.default_rng(1))
    assert checked["vectors"] == 261 * 261 * 4 * 6


def test_d2_three_alleles_dense(ctx, oracle_lib):
    """n = 3, every coverage vector in [0, 64]^3"""
    rows = np.array(list(itertools.product(range(65), repeat=3)), dtype=np.int64)
    _, checked = grid_domain(ctx, oracle_lib, "D2", rows, np.random.default_rng(2), priors=("uniform", "af", "one"))
    assert checked["vectors"] == 65 ** 3 * 3 * 6


def test_d3_uniform_prior_near_ties(ctx, oracle_lib):
    """(a, b, a) at every position of n = 3..8 alleles among zeros and small fillers, a, b in [0, 200], uniform
    priors: GT there is decided by the last bits of log_binomial's fp64 logs (DESIGN §3)"""
    rng = np.random.default_rng(3)
    ties = {err: 0 for err in ERRS}
    total = 0
    for n in range(3, 9):
        outs, checked = grid_domain(ctx, oracle_lib, f"D3 n={n}", gu.near_tie_family(n, 200), rng, priors=("uniform",))
        total += checked["vectors"]
        for err in ERRS:
            o = outs[(False, err)]
            ties[err] += len(gu.near_ties(o.lik, o.lik_off, o.n_gts, o.status))
    print(f"D3: {total} vectors checked, oracle arg-maxes decided by <= 2 ulps: {ties}")
    assert all(v > 0 for v in ties.values()), ties


def test_d4_many_alleles_mixed_in_each_warp(ctx, oracle_lib):
    """n in {8, 16, 32, 64} drawn per variant (every warp mixes them): n(n+1)/2 slots, and the warp-scan bump
    allocator of the lik == NULL run"""
    rng = np.random.default_rng(4)
    nall = rng.choice([8, 16, 32, 64], size=6000)
    vao = gu.offsets(nall).astype(np.int64)
    na = int(vao[-1])
    cov = np.where(rng.random(na) < 0.15, rng.integers(1, 120, size=na), 0)
    cov[rng.random(na) < 0.002] = 201
    freq = np.zeros(na, np.float32)
    kinds = rng.integers(0, 4, size=len(nall))
    for v, n in enumerate(nall):
        freq[vao[v]:vao[v + 1]] = prior_sets(int(n), 1, rng, (("uniform", "af", "ref0", "one")[kinds[v]],))[0][0]
    checked = {"vectors": 0, "nan": 0}
    for haploid in (False, True):
        for err in ERRS:
            o = run_and_compare(ctx, oracle_lib, "D4", cov, freq, vao, err, 200, haploid, checked)
            assert set(o.status.tolist()) == {0, 1, 2}
    print(f"D4: {checked['vectors']} vectors checked")


def test_d5_extremes(ctx, oracle_lib):
    """max_cov 0 / 10^9 / 2^31-1; coverages of 2^20, 2^30, 2^31-1 (tot wraps; (int)(t + er) goes negative and
    log_binomial returns NaN); priors of 1e-40 (subnormal), 1e-20 pairs (subnormal product), 1e-30 (product 0);
    error rates 1e-8 and 0.5"""
    rng = np.random.default_rng(5)
    V = [0, 1, 5, 100, 200, 201, 1 << 20, 1 << 30, 10 ** 9, (1 << 31) - 1]
    checked = {"vectors": 0, "nan": 0}
    for n in (2, 3, 4):
        rows = np.array(list(itertools.product(V, repeat=n)), dtype=np.int64)
        if n == 4:
            rows = rows[rng.choice(len(rows), 2500, replace=False)]
        m = len(rows)
        fs = prior_sets(n, m, rng, ("uniform", "one"))
        for p in (1e-40, 1e-20, 1e-30):
            f = np.full((m, n), np.float32(p), np.float32)
            f[::2, 0] = np.float32(0.5)
            fs.append(f)
        cov = np.tile(rows, (len(fs), 1)).ravel()
        freq = np.concatenate(fs).ravel()
        vao = np.arange(m * len(fs) + 1, dtype=np.int64) * n
        for max_cov in (0, 200, 10 ** 9, (1 << 31) - 1):
            for haploid in (False, True):
                for err in ERRS + (1e-8, 0.5):
                    run_and_compare(ctx, oracle_lib, f"D5 n={n}", cov, freq, vao, err, max_cov, haploid, checked)
    print(f"D5: {checked['vectors']} vectors checked, {checked['nan']} with NaN likelihoods")
    assert checked["nan"] > 0, "no vector made tot pass 2^31"


def _py_coverages(w_u32, ref_bit, sig_kmer_off, allele_sig_off):
    """set_coverages (main.cpp:157-182) in Python integers: BF::get_count's uint16_t on alt k-mers, weights <= 0
    (as int) skipped, the running mean in unsigned 32-bit arithmetic"""
    w = np.where(ref_bit, w_u32, w_u32 & 0xFFFF).astype(np.int64)
    w = np.where(w >= 1 << 31, w - gu.U32, w).tolist()
    so, ao = sig_kmer_off.tolist(), allele_sig_off.tolist()
    out = []
    for a in range(len(ao) - 1):
        best = 0
        for s in range(ao[a], ao[a + 1]):
            curr, n = 0, 0
            for q in range(so[s], so[s + 1]):
                if w[q] > 0:
                    curr = ((curr * n + w[q]) % gu.U32) // (n + 1)
                    n += 1
            best = max(best, curr)
        out.append(best)
    return np.array(out, dtype=np.int64)


def test_d6_coverage_kernels(ctx, oracle_lib):
    """k_coverage + k_mask_alt: signatures of 1-300 k-mers, weights <= 0 skipped (incl. counts >= 2^31, negative as
    int32), u32 overflow of the running mean, alt weights 65535 / 65536 / 65537 wrapped to u16, alleles without a
    signature"""
    rng = np.random.default_rng(6)
    nall = rng.integers(1, 5, size=1500)
    vao = gu.offsets(nall).astype(np.int64)
    na = int(vao[-1])
    n_sig = rng.choice([0, 1, 1, 2, 3], size=na)
    aso = gu.offsets(n_sig).astype(np.int64)
    sig_len = rng.choice([1, 2, 3, 7, 40, 150, 300], size=int(aso[-1]))
    sko = gu.offsets(sig_len).astype(np.int64)
    nk = int(sko[-1])
    kind = rng.integers(0, 8, size=nk)
    w = np.select([kind == 0, kind == 1, kind == 2, kind == 3, kind == 4],
                  [0, rng.integers(1 << 31, 1 << 32, size=nk), rng.integers(1 << 30, 1 << 31, size=nk),
                   rng.choice([65535, 65536, 65537, 131071], size=nk), (1 << 31) - 1],
                  rng.integers(1, 90, size=nk)).astype(np.int64)
    # ref flag per k-mer: allele slot 0 of each variant, plus every k-mer of variants whose alt weights stay unmasked
    allele_of_sig = np.repeat(np.arange(na), n_sig)
    allele_of_kmer = np.repeat(allele_of_sig, sig_len)
    slot0 = np.zeros(na, bool)
    slot0[vao[:-1][nall > 0]] = True
    wrap_variant = rng.random(len(nall)) < 0.5
    ref_bit = slot0[allele_of_kmer] | ~np.repeat(wrap_variant, nall)[allele_of_kmer]
    exp_cov = _py_coverages(w, ref_bit, sko, aso)
    assert (exp_cov > (1 << 16)).any() and ((exp_cov > 0) & (exp_cov < 100)).any()
    freq = np.concatenate([prior_sets(int(n), 1, rng, ("af",))[0][0] for n in nall])
    checked = {"vectors": 0, "nan": 0}
    for max_cov in (200, (1 << 31) - 1):
        for haploid in (False, True):
            for err in ERRS:
                pair = [run_device(ctx, w, sko, aso, vao, freq, err, max_cov, haploid, want, ref_bit)
                        for want in (True, False)]
                assert np.array_equal(pair[0][0], exp_cov), "coverages against main.cpp:157-182"
                compare(oracle_lib, "D6", exp_cov.astype(np.uint32), freq, vao, err, max_cov, haploid, pair, checked)
    print(f"D6: {nk} k-mers in {int(aso[-1])} signatures, {checked['vectors']} vectors checked")


def test_d7_zero_allele_variants(ctx, oracle_lib):
    """a variant without alleles reserves no likelihood slot: it writes none and reports n_gts 0, status 2, GT 0,
    GQ 0 (include/malva_gpu.h); the variants next to it in the same warp are unaffected"""
    rng = np.random.default_rng(7)
    nall = rng.integers(1, 6, size=512)
    nall[rng.random(512) < 0.3] = 0
    nall[0], nall[1], nall[-1] = 0, 3, 0      # before a normal variant, and last (just before the guard slots)
    vao = gu.offsets(nall).astype(np.int64)
    na = int(vao[-1])
    cov = rng.integers(1, 60, size=na)        # every real variant has coverage: non-zero likelihoods everywhere
    freq = rng.random(na).astype(np.float32)
    checked = {"vectors": 0, "nan": 0}
    for haploid in (False, True):
        for err in ERRS:
            o = run_and_compare(ctx, oracle_lib, "D7", cov, freq, vao, err, 200, haploid, checked)
            z = nall == 0
            assert (o.n_gts[z] == 0).all() and (o.status[z] == 2).all() and (o.best[z] == 0).all()
            assert (o.gq[z] == 0).all()
    print(f"D7: {checked['vectors']} vectors checked")
