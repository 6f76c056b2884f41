"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU
oracle on the same seeded inputs.  Bar: bit-exact bits, counters, coverages,
GT and GQ; likelihoods within 1e-9 relative (north_star)."""
import random

import numpy as np
import pytest

from malva_b200 import MalvaGpu, MalvaGpuError, SignatureBatch, kmc
from malva_b200.api import PackedSignatureBatch, reduce_counts
import parity_util as util

pytestmark = pytest.mark.gpu

LIK_RTOL = 1e-9


def _run_pair(oracle_lib, k, ref_k, bf_bits, seed, n_var=300, glen=20000, n_sample=6000, big_counts=False):
    rng = random.Random(seed)
    genome = util.make_genome(rng, glen)
    nested, freqs = util.synth_signatures(rng, genome, k, n_var)
    ks, fl = util.flatten(nested)
    g = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits)
    o = util.OracleRun(oracle_lib, k, ref_k, bf_bits)
    # index side, in three batches (exercises table growth + rehash)
    cuts = [0, len(ks) // 3, 2 * len(ks) // 3, len(ks)]
    for a, b in zip(cuts[:-1], cuts[1:]):
        g.add_signatures(ks[a:b], fl[a:b])
        o.add_signatures(ks[a:b], fl[a:b])
    g.finalize_alt()
    o.finalize_alt()
    g.scan_reference(genome)
    o.scan_reference(genome)
    g.finalize_context()
    o.finalize_context()
    words, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, n_sample, big_counts)
    g.scan_sample_kmers(packed, counts)
    o.scan_sample_kmers(packed, counts)
    return g, o, genome, nested, freqs, ks, fl, words


@pytest.mark.parametrize("k,ref_k,bf_bits", [
    (35, 43, 1 << 22),          # default k / ref_k, power-of-two filter (mask path)
    (35, 43, 3 * (1 << 20) + 7),  # non power of two (modulo path), dense -> many bit collisions
    (31, 39, 1 << 22),          # runtime-k kernels, 17..32-byte XXH3 branch
    (36, 43, 1 << 21),          # odd ref_k - k: the reference's non-contiguous window quirk
    (15, 21, 1 << 20),          # <=16-byte XXH3 branch
    (43, 43, 1 << 21),          # k == ref_k
    (63, 64, 1 << 21),          # widest supported words
])
def test_index_scan_state_bit_exact(oracle_lib, k, ref_k, bf_bits):
    g, o, genome, nested, freqs, ks, fl, words = _run_pair(oracle_lib, k, ref_k, bf_bits, seed=100 + k)
    try:
        assert np.array_equal(g.bits(0), o.bits(0)), "bf bits"
        assert np.array_equal(g.bits(1), o.bits(1)), "context_bf bits"
        assert g.popcount(0) == int(np.unpackbits(o.bits(0).view(np.uint8)).sum())
        assert g.popcount(1) > 0, "reference pass never hit: test input too weak"
        assert g.kmap_size() == o.kmap_size()
        gc, oc = g.bf_counts(), o.bf_counts()
        assert np.array_equal(gc, oc), "rank-indexed bf counters"
        assert oc.sum() > 0
        # every signature k-mer, plus unrelated keys, through get_count / test_key
        rng = random.Random(7)
        extra = [util.rand_seq(rng, k) for _ in range(200)] + [util.rand_seq(rng, k - 2, "ACGTN") for _ in range(50)]
        q = ks + extra
        for flag in (0, 1):
            fl_q = [flag] * len(q)
            assert np.array_equal(g.get_counts(q, fl_q), o.get_counts(q, fl_q)), f"get_count is_ref={flag}"
        for which in (0, 1, 2):
            assert np.array_equal(g.test_keys(which, q), o.test_keys(which, q)), f"test_key which={which}"
        ctx_q = [genome[p:p + ref_k] for p in range(0, len(genome) - ref_k, 37)]
        assert np.array_equal(g.test_keys(1, ctx_q), o.test_keys(1, ctx_q))
        ref_counts = o.get_counts(ks, [1] * len(ks))
        assert (ref_counts > 0).sum() > 20
    finally:
        g.close()
        o.close()


def test_scan_dense_filter_big_counts_bit_exact(oracle_lib):
    """the (35, 43) packed-input scan leaves exactly the oracle's counters on a dense non-power-of-two filter with
    counts past 2^16"""
    g, o, genome, nested, freqs, ks, fl, words = _run_pair(oracle_lib, 35, 43, 3 * (1 << 18) + 5, seed=4242, n_var=400,
                                                           n_sample=9000, big_counts=True)
    try:
        assert np.array_equal(g.bf_counts(), o.bf_counts()), "rank-indexed bf counters"
        for flag in (0, 1):
            fl_q = [flag] * len(ks)
            assert np.array_equal(g.get_counts(ks, fl_q), o.get_counts(ks, fl_q)), f"get_count is_ref={flag}"
        assert int(o.bf_counts().astype(np.int64).sum()) > 0 and (o.get_counts(ks, [1] * len(ks)) > 0).sum() > 20
    finally:
        g.close()
        o.close()


@pytest.mark.parametrize("occ_log2,defer", [(0, 1), (10, 1), (10, 0), (16, 0), (29, 0)])
@pytest.mark.parametrize("k,ref_k", [(35, 43), (31, 39)])
def test_prefilter_granularity_and_hit_path(oracle_lib, monkeypatch, occ_log2, defer, k, ref_k):
    """the small filters of this file get one pre-filter bit per filter bit; the whole-genome shape has one per 64.
    MG_OCC_LOG2_BITS caps the pre-filter (0 = none at all; 10 and 16 = one bit per 4096 / 64 filter bits here) and
    MG_SCAN_DEFER_HITS picks whether filter hits are finished in line or by k_scan_hits: same counters either way"""
    monkeypatch.setenv("MG_OCC_LOG2_BITS", str(occ_log2))     # (both read when the context is created)
    monkeypatch.setenv("MG_SCAN_DEFER_HITS", str(defer))
    g, o, genome, nested, freqs, ks, fl, words = _run_pair(oracle_lib, k, ref_k, 1 << 22, seed=900 + occ_log2 + defer,
                                                           n_var=400, n_sample=9000, big_counts=True)
    try:
        assert np.array_equal(g.bits(1), o.bits(1)), "context_bf bits (the reference pass goes through the pre-filter too)"
        assert np.array_equal(g.bf_counts(), o.bf_counts()), "rank-indexed bf counters"
        for flag in (0, 1):
            fl_q = [flag] * len(ks)
            assert np.array_equal(g.get_counts(ks, fl_q), o.get_counts(ks, fl_q)), f"get_count is_ref={flag}"
        assert int(o.bf_counts().astype(np.int64).sum()) > 0
    finally:
        g.close()
        o.close()


def test_u16_wraparound_and_int_counts(oracle_lib):
    # counts up to 70000 per record: bf counters wrap mod 2^16, ref_bf counts do not
    g, o, genome, nested, freqs, ks, fl, words = _run_pair(oracle_lib, 35, 43, 1 << 18, seed=5, n_sample=20000,
                                                          big_counts=True)
    try:
        assert np.array_equal(g.bf_counts(), o.bf_counts())
        a, b = g.get_counts(ks, [1] * len(ks)), o.get_counts(ks, [1] * len(ks))
        assert np.array_equal(a, b)
        assert b.max() > 65535
    finally:
        g.close()
        o.close()


@pytest.mark.parametrize("glen", [10, 20, 42, 43, 44, 4095 + 43, 4096 + 43, 4097 + 43, 9000])
def test_reference_pass_edges(oracle_lib, glen):
    # contigs shorter than ref_k, exactly ref_k, around the CTA tile size
    k, ref_k, bits = 35, 43, 1 << 16
    rng = random.Random(glen)
    genome = util.rand_seq(rng, glen)
    g, o = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bits), util.OracleRun(oracle_lib, k, ref_k, bits)
    try:
        d = (ref_k - k) // 2
        alts = [genome[p:p + k] for p in range(d, max(d + 1, glen - k), 5)] if glen >= k + d else [genome[d:]]
        alts += [util.rand_seq(rng, k) for _ in range(20)]
        for x in (g, o):
            x.add_signatures(alts, [0] * len(alts))
            x.finalize_alt()
            x.scan_reference(genome)
            x.finalize_context()
        assert np.array_equal(g.bits(1), o.bits(1))
        if glen >= ref_k:
            assert g.popcount(1) > 0
    finally:
        g.close()
        o.close()


def test_empty_and_ragged_inputs(oracle_lib):
    g = MalvaGpu(k=35, ref_k=43, bf_bits=1 << 16)
    try:
        g.add_signatures([], [])
        g.finalize_alt()
        with pytest.raises(MalvaGpuError):  # the reference's substr(d, k) throws on a contig shorter than d
            g.scan_reference("")
        g.scan_reference("ACGT")  # shorter than ref_k: one truncated probe, no hit
        g.finalize_context()
        g.scan_sample_kmers(np.zeros(0, dtype=kmc.KMER_DTYPE), np.zeros(0, dtype=np.uint32))
        assert g.popcount(0) == 0 and g.popcount(1) == 0 and g.kmap_size() == 0
        assert len(g.bf_counts()) == 0
        b = SignatureBatch.from_nested([[[], []]], [[0.9, 0.1]])  # a variant whose alleles have no signatures
        r = g.genotype(b, 0.001, 200, False)
        assert r.cov.tolist() == [0, 0] and r.status.tolist() == [2] and r.gq.tolist() == [0]
        assert g.get_counts(["A" * 35, ""], [0, 1]).tolist() == [0, 0]
    finally:
        g.close()


@pytest.mark.parametrize("haploid", [False, True])
@pytest.mark.parametrize("err", [0.001, 0.05])
@pytest.mark.parametrize("k,ref_k", [(35, 43), (31, 39), (63, 64)])  # k_lookup_packed<35>, <0>, wide keys (k >= 48)
def test_coverage_and_genotype(oracle_lib, k, ref_k, haploid, err):
    g, o, genome, nested, freqs, ks, fl, words = _run_pair(oracle_lib, k, ref_k, 1 << 22, seed=42, n_var=600,
                                                          n_sample=20000)
    try:
        batch = SignatureBatch.from_nested(nested, freqs)
        max_cov = 120  # low enough that some alleles trip the veto
        r = g.genotype(batch, err, max_cov, haploid)
        cov, exp = o.genotype(batch, err, max_cov, haploid)
        assert np.array_equal(r.cov, cov), "COVS"
        assert (cov > 0).sum() > 100
        seen = set()
        for v, e in enumerate(exp):
            assert r.status[v] == e["status"], v
            assert r.n_gts[v] == len(e["probs"]), v
            assert r.best_gt[v] == e["best"], (v, r.lik[int(r.lik_off[v]):int(r.lik_off[v]) + r.n_gts[v]], e)
            assert r.gq[v] == e["gq"], v
            got = r.lik[int(r.lik_off[v]):int(r.lik_off[v]) + r.n_gts[v]]
            assert np.allclose(got, e["probs"], rtol=LIK_RTOL, atol=0.0), (v, got, e["probs"])
            assert np.array_equal(got == 0, e["probs"] == 0)
            seen.add(e["status"])
        assert seen == {0, 1, 2}, seen
        # mg_genotype packs the batch on the host: the Python packer of the same batch gives identical bits out
        pb = PackedSignatureBatch.from_batch(batch, k)
        assert len(pb.irr_kmer) > 0, "the synthetic signatures should include irregular k-mers"
        rp = g.genotype_packed(pb, err, max_cov, haploid)
        for name in ("cov", "status", "n_gts", "best_gt", "gq"):
            assert np.array_equal(getattr(rp, name), getattr(r, name)), name
        for v in range(batch.n_variants):
            a, b = int(r.lik_off[v]), int(rp.lik_off[v])
            assert np.array_equal(r.lik[a:a + r.n_gts[v]].view(np.uint64), rp.lik[b:b + rp.n_gts[v]].view(np.uint64)), v
        rq = g.genotype_packed(pb, err, max_cov, haploid, want_lik=False)   # likelihoods stay on the device
        for name in ("cov", "status", "n_gts", "best_gt", "gq"):
            assert np.array_equal(getattr(rq, name), getattr(r, name)), name
    finally:
        g.close()
        o.close()


def test_scan_large_batch_properties(oracle_lib):
    """Full-size style properties that need no oracle: linearity (scanning a batch twice doubles every
    counter mod 2^16 / 2^32) and order independence (a permuted batch gives identical state)."""
    k, ref_k, bits = 35, 43, 1 << 26
    rng = random.Random(9)
    genome = util.make_genome(rng, 50000)
    nested, freqs = util.synth_signatures(rng, genome, k, 1500)
    ks, fl = util.flatten(nested)
    words, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 200000)
    states = []
    for variant in ("once", "twice", "permuted"):
        g = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bits)
        g.add_signatures(ks, fl)
        g.finalize_alt()
        g.scan_reference(genome)
        g.finalize_context()
        if variant == "permuted":
            perm = np.random.default_rng(1).permutation(len(packed))
            g.scan_sample_kmers(packed[perm].copy(), counts[perm].copy())
        else:
            g.scan_sample_kmers(packed, counts)
            if variant == "twice":
                g.scan_sample_kmers(packed, counts)
        states.append((g.bf_counts().astype(np.uint32), g.get_counts(ks, [1] * len(ks)).astype(np.int64)))
        g.close()
    once, twice, perm = states
    assert np.array_equal(once[0], perm[0]) and np.array_equal(once[1], perm[1])
    assert np.array_equal((once[0] * 2) & 0xFFFF, twice[0])
    assert np.array_equal(once[1] * 2, twice[1])
    assert once[0].sum() > 0 and once[1].sum() > 0


@pytest.mark.parametrize("version,p,k,ref_k,csz,minc,maxc", [
    (0x200, 7, 35, 43, 1, 3, 200), (0, 3, 35, 43, 1, 3, 200), (0x200, 3, 31, 39, 1, 3, 200), (0, 5, 36, 41, 1, 3, 200),
    (0x200, 7, 35, 43, 2, 3, 1000),            # -cs1000: two counter bytes
    (0x200, 7, 35, 43, 3, 2, 70000),
    (0x200, 3, 35, 43, 4, 3, (1 << 33) + 7),   # 64-bit max_count (high word of the KMC 3 header)
    (0x200, 3, 60, 63, 2, 3, 60000),           # 15 suffix bytes + 2 counter bytes: records longer than a packed word
    (0, 1, 21, 21, 4, 250, 250),               # a one-value [min, max] window; k == ref_k
])
def test_kmc_records_decoded_on_device(oracle_lib, tmp_path, version, p, k, ref_k, csz, minc, maxc):
    """mg_scan_kmc_records (raw .kmc_suf records + prefix LUT, decoded by the scan kernel) must leave the same
    state as the oracle scanning the KMC listing -- including the [min_count, max_count] record filter -- over the
    header variants of tests/test_kmc_format_cpu.py (counter sizes 1-4, KMC1 / 0x200, LUT prefix lengths)."""
    rng = random.Random(4000 + p + k)
    bits = 1 << 20
    genome = util.make_genome(rng, 20000)
    nested, freqs = util.synth_signatures(rng, genome, k, 300)
    ks, fl = util.flatten(nested)
    words, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 5000, big_counts=csz > 1)
    counts = np.minimum(counts, min(256 ** csz - 1, 70000)).astype(np.uint32)
    counts[::7] = 2          # below min_count: skipped by ReadNextKmer
    counts[::11] = 250       # above max_count = 200 (one-byte cases): skipped too
    counts[::13] = minc      # the edges themselves are kept
    counts[::17] = min(maxc, 256 ** csz - 1)
    if minc == maxc:
        counts[::2] = minc
    counts[::19] = minc - 1  # (below min_count whatever it is)
    prefix = str(tmp_path / "db")
    kmc.write_kmc_db(prefix, packed, counts, ref_k, lut_prefix_len=p, version=version, counter_size=csz, min_count=minc,
                     max_count=maxc)
    listed, lcounts, kk = kmc.read_kmc_db(prefix)
    assert kk == ref_k and 0 < len(listed) < len(packed)
    db = kmc.open_kmc_db(prefix)
    assert db["total"] == len(packed)
    g, o = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bits), util.OracleRun(oracle_lib, k, ref_k, bits)
    try:
        for x in (g, o):
            x.add_signatures(ks, fl)
            x.finalize_alt()
            x.scan_reference(genome)
            x.finalize_context()
        o.scan_sample_kmers(listed, lcounts)
        g.kmc_open(db)
        rec = db["record_bytes"]
        half = (db["total"] // 2 // 32) * 32 + 5   # two calls, the second starting inside a warp tile
        g.scan_kmc_records(db["records"][:half * rec], 0, half)
        g.scan_kmc_records(db["records"][half * rec:], half, db["total"] - half)
        assert np.array_equal(g.bf_counts(), o.bf_counts())
        assert np.array_equal(g.get_counts(ks, [1] * len(ks)), o.get_counts(ks, [1] * len(ks)))
        assert o.bf_counts().sum() > 0
        with pytest.raises(MalvaGpuError):      # a database of the wrong k-mer length is refused
            bad = dict(db)
            bad["k"] = ref_k + 4
            g.kmc_open(bad)
    finally:
        g.close()
        o.close()


@pytest.mark.parametrize("bf_bits", [1 << 13, 1 << 22])
def test_replicas_built_in_any_order_have_one_image_and_their_counters_add_up(oracle_lib, bf_bits):
    """Multi-GPU contract (DESIGN 7): every replica builds the index on its own, scans a share of the stream, and the
    counter arrays are added ELEMENT BY ELEMENT.  That is only exact if the index image does not depend on the order
    (or the races) of the inserts.  2^13 bits = 32 probe lines for ~1,000 ref keys: every line overflows."""
    k, ref_k = 35, 43
    rng = random.Random(99)
    genome = util.make_genome(rng, 30000)
    nested, _ = util.synth_signatures(rng, genome, k, 700)
    ks, fl = util.flatten(nested)
    words, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 30000)
    order = list(range(len(ks)))
    rng.shuffle(order)
    a, b, whole = (MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits) for _ in range(3))
    o = util.OracleRun(oracle_lib, k, ref_k, bf_bits)
    try:
        a.add_signatures(ks, fl)                                   # one batch, file order
        for s in range(0, len(order), 97):                         # shuffled, many small batches
            idx = order[s:s + 97]
            b.add_signatures([ks[i] for i in idx], [fl[i] for i in idx])
        whole.add_signatures(list(reversed(ks)), list(reversed(fl)))
        o.add_signatures(ks, fl)
        for x in (a, b, whole, o):
            x.finalize_alt()
            x.scan_reference(genome)
            x.finalize_context()
        if bf_bits == 1 << 13:
            assert a.index_stats()["overflow_keys"] > 100
        assert a.index_stats() == b.index_stats() == whole.index_stats()
        half = len(packed) // 2
        a.scan_sample_kmers(packed[:half], counts[:half])
        b.scan_sample_kmers(packed[half:], counts[half:])
        whole.scan_sample_kmers(packed, counts)
        o.scan_sample_kmers(packed, counts)
        ca, cb, cw = util.counter_arrays(a), util.counter_arrays(b), util.counter_arrays(whole)
        for i, name in enumerate(("bf counters", "line key counts", "overflow counts")):
            assert len(ca[i]) == len(cb[i]) == len(cw[i]), name
            assert np.array_equal(ca[i] + cb[i], cw[i]), name
        assert cw[1].sum() + cw[2].sum() > 0
        # and the single-replica answers are the reference's
        assert np.array_equal(whole.get_counts(ks, fl), o.get_counts(ks, fl))
        assert np.array_equal(whole.bf_counts(), o.bf_counts())
        # the in-process reduce (gather, N-way sum over peer memory, scatter back into the probe lines)
        reduce_counts([a, b])
        assert np.array_equal(a.get_counts(ks, fl), o.get_counts(ks, fl))
        assert np.array_equal(a.bf_counts(), o.bf_counts())
        # ... and the scan keeps working on the scattered counters
        a.scan_sample_kmers(packed, counts)
        whole.scan_sample_kmers(packed, counts)
        assert np.array_equal(a.get_counts(ks, fl), whole.get_counts(ks, fl))
        assert np.array_equal(a.bf_counts(), whole.bf_counts())
    finally:
        for x in (a, b, whole, o):
            x.close()


def test_replicas_sum_lookup_results_instead_of_counters(oracle_lib):
    """the other multi-GPU scheme (include/malva_gpu.h: mg_lookup_packed_device / mg_genotype_weights_device): every
    replica looks the batch up in its own partial counters (bf counters raw), the weight vectors are summed (what
    bench.py does with ncclReduce), and the genotypes computed from the sum equal a single context's -- incl. the
    uint16 wrap-around of bf counters that only the SUM exceeds.  The library's work is put on torch's stream."""
    import torch

    k, ref_k, bits = 35, 43, 1 << 22
    rng = random.Random(2024)
    genome = util.make_genome(rng, 30000)
    nested, freqs = util.synth_signatures(rng, genome, k, 500)
    ks, fl = util.flatten(nested)
    words, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 30000, big_counts=True)
    a, b, whole = (MalvaGpu(k=k, ref_k=ref_k, bf_bits=bits) for _ in range(3))
    try:
        for x in (a, b, whole):
            x.add_signatures(ks, fl)
            x.finalize_alt()
            x.scan_reference(genome)
            x.finalize_context()
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        for x in (a, b, whole):
            x.set_stream(side.cuda_stream)
        half = len(packed) // 2
        # each half is scanned several times so that bf counters pass 2^16 in the sum but not in either part
        for _ in range(3):
            a.scan_sample_kmers(packed[:half], counts[:half])
            b.scan_sample_kmers(packed[half:], counts[half:])
            whole.scan_sample_kmers(packed, counts)
        batch = SignatureBatch.from_nested(nested, freqs)
        pb = PackedSignatureBatch.from_batch(batch, k)
        exp = whole.genotype_packed(pb, 0.001, 10 ** 9, False)
        dev = torch.device("cuda", 0)
        nv, na = pb.n_variants, int(pb.var_allele_off[-1])
        nk = len(pb.kmers)
        t = {"var_allele_off": torch.from_numpy(pb.var_allele_off.astype(np.int32)).to(dev),
             "allele_sig_off": torch.from_numpy(pb.allele_sig_off.astype(np.int32)).to(dev),
             "sig_kmer_off": torch.from_numpy(pb.sig_kmer_off.astype(np.int32)).to(dev),
             "kmers": torch.from_numpy(pb.kmers.view(np.int64).reshape(-1, 2).copy()).to(dev),
             "freq": torch.from_numpy(pb.freq).to(dev),
             "irr_off": torch.from_numpy(pb.irr_off.astype(np.int64)).to(dev),
             "irr_pool": torch.from_numpy(np.frombuffer(pb.irr_pool, np.uint8).copy()).to(dev),
             "irr_kmer": torch.from_numpy(pb.irr_kmer.astype(np.int32)).to(dev),
             "cov": torch.zeros(na, dtype=torch.int32, device=dev)}
        for nme in ("n_gts", "status", "best_gt", "gq"):
            t[nme] = torch.zeros(nv, dtype=torch.int32, device=dev)
        ptrs = {n: x.data_ptr() for n, x in t.items()}
        nall = np.diff(pb.var_allele_off.astype(np.int64))
        dims = (nv, na, len(pb.sig_kmer_off) - 1, nk, len(pb.irr_kmer), len(pb.irr_pool),
                int(np.maximum(nall * (nall + 1) // 2, nall).sum()))
        wa = torch.zeros(nk, dtype=torch.int32, device=dev)
        wb = torch.zeros(nk, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        with torch.cuda.stream(side):                          # no host synchronisation between the five calls
            a.lookup_packed_device(ptrs, dims, wa.data_ptr())
            b.lookup_packed_device(ptrs, dims, wb.data_ptr())
            total = wa + wb                                    # (stream-ordered with the library's kernels)
            a.genotype_weights_device(ptrs, dims, total.data_ptr(), 0.001, 10 ** 9, False)
        torch.cuda.synchronize()
        assert int((total.to(torch.int64) & 0xFFFFFFFF).max()) > 65535, "the wrap-around is not exercised"
        for x in (a, b, whole):
            x.set_stream(0)
        assert np.array_equal(t["cov"].cpu().numpy().view(np.uint32), exp.cov)
        for nme, e in (("n_gts", exp.n_gts), ("status", exp.status), ("best_gt", exp.best_gt), ("gq", exp.gq)):
            assert np.array_equal(t[nme].cpu().numpy(), e), nme
        assert (exp.cov > 0).sum() > 100
    finally:
        for x in (a, b, whole):
            x.close()


def test_kmc_database_with_several_bins(oracle_lib, tmp_path):
    """the layout real KMC2 files have: one prefix LUT per bin, records sorted within a bin only.  The device finds
    the prefix of a record from its global index through the concatenated LUT."""
    k, ref_k, bits, p = 35, 43, 1 << 20, 3
    rng = random.Random(515)
    genome = util.make_genome(rng, 20000)
    nested, _ = util.synth_signatures(rng, genome, k, 300)
    ks, fl = util.flatten(nested)
    _, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 6000)
    counts = np.minimum(counts, 255).astype(np.uint32)
    # one record per distinct k-mer (a KMC database never lists a k-mer twice)
    vals = kmc.packed_to_ints(packed)
    first = {}
    for i, v in enumerate(vals):
        first.setdefault(v, i)
    keep = sorted(first.values())
    packed, counts = packed[keep], counts[keep]
    prefix = str(tmp_path / "binned")
    kmc.write_kmc_db_binned(prefix, packed, counts, ref_k, bin_of=lambda v: (v * 2654435761 >> 7) % 5, n_bins=5,
                            lut_prefix_len=p)
    listed, lcounts, kk = kmc.read_kmc_db(prefix)
    assert kk == ref_k and len(listed) == len(packed)
    assert sorted(kmc.packed_to_ints(listed)) == sorted(kmc.packed_to_ints(packed))
    assert kmc.packed_to_ints(listed) != sorted(kmc.packed_to_ints(listed)), "bins should break the global order"
    db = kmc.open_kmc_db(prefix)
    assert len(db["lut"]) == 5 * 4 ** p
    g, o = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bits), util.OracleRun(oracle_lib, k, ref_k, bits)
    try:
        for x in (g, o):
            x.add_signatures(ks, fl)
            x.finalize_alt()
            x.scan_reference(genome)
            x.finalize_context()
        o.scan_sample_kmers(listed, lcounts)
        g.kmc_open(db)
        g.scan_kmc_records(db["records"], 0, db["total"])
        assert np.array_equal(g.bf_counts(), o.bf_counts())
        assert np.array_equal(g.get_counts(ks, [1] * len(ks)), o.get_counts(ks, [1] * len(ks)))
        assert o.bf_counts().sum() > 0
    finally:
        g.close()
        o.close()
