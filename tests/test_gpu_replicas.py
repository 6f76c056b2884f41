"""Replicated and reloaded contexts against the CPU oracle, at every probe-line key layout (DESIGN 2, 7).

`malva-geno call --devices` loads the index file onto several contexts (mg_import_set_bits, mg_add_signatures_packed,
mg_finalize_alt), each context scans a share of the sample stream and mg_reduce_counts adds the counters into the
first one; bench.py's replicas sum look-up results instead.  Both rest on the canonical probe-line image and on
k_counters_xfer, which branches on the key layout (the count in w3 of the slot for k <= 47, in key_counts for
k >= 48; the overflow flag in w2 / w3 of slot 4) and on where an alt counter lives (w29..31 for the first three set
bits of a line, bf_counts[rank + j] for the others).  A slip there changes nothing on one context, so every test
here checks the replicated or reloaded result against the oracle, at the layouts where the index code branches and
at filter sizes that reach overflowed keys, dense lines and a partial last line.  Each asserts that its input
reaches the edge it is there for."""
import ctypes as C
import random

import numpy as np
import pytest

from malva_b200 import MalvaGpu, MalvaGpuError, SignatureBatch, kmc
from malva_b200.api import IRREGULAR_BIT, PackedSignatureBatch, check, reduce_counts
import parity_util as util

pytestmark = pytest.mark.gpu

LAYOUTS = [
    (35, 43),   # specialised kernels, inline keys
    (31, 39),   # run-time-k kernels, inline keys
    (47, 55),   # last inline layout: 94-bit keys, overflow flag at w2 bit 31
    (48, 56),   # first wide layout: key in w0..w3, count in key_counts, overflow flag at w3 bit 31
    (63, 64),   # widest keys, odd ref_k - k
]
DENSE, MODULO, SPARSE = 1 << 13, 3 * (1 << 12) + 7, 1 << 22
FILTERS = [pytest.param(DENSE, id="2^13"), pytest.param(MODULO, id="3x2^12+7"), pytest.param(SPARSE, id="2^22")]
BIG_REF = (1 << 31) + 12345   # count of the records that make a ref key's replica parts wrap u32 in the sum
# seeds of the reduce test whose bf has a number of set bits that is not a multiple of 4, with peer counts on the
# last ones (at 2^13 every line holds five keys, so the array of line key counts is a multiple of 4 long); 7100 else
REDUCE_SEEDS = {(35, MODULO): 7101, (47, MODULO): 7103, (48, MODULO): 7102, (63, DENSE): 7101, (63, MODULO): 7103}


def _n_gpus() -> int:
    from malva_b200 import _lib

    return _lib.load().mg_device_count()


def _find_kmers(L, k: int, bf_bits: int, lo: int, n: int = 1, first: int = 0) -> list:
    """n k-mers of k ACGT symbols, each its own canonical form, whose filter index is >= lo (searched in the oracle)"""
    out = C.create_string_buffer((k + 1) * n)
    got = L.mo_find_kmers_at(b"A" * k, k, bf_bits, lo, first, 1 << 28, out, n)
    assert got == n, "k-mer search did not finish"
    return [out.raw[j * (k + 1):j * (k + 1) + k].decode() for j in range(n)]


def _window(rng, genome: str, kmer: str, k: int, ref_k: int, o=None) -> str:
    """a sample ref_k-mer with `kmer` in the place the scan reads; with the oracle o, one whose context is not in
    context_bf (so the bf counter of the k-mer is incremented)"""
    d = (ref_k - k) // 2
    while True:
        w = util.rand_seq(rng, d) + kmer + util.rand_seq(rng, ref_k - k - d)
        if o is None or not o.test_keys(1, [w])[0]:
            return w


def _records(windows, counts):
    return kmc.ints_to_packed([kmc.pack_kmer(w) for w in windows]), np.asarray(counts, dtype=np.uint32)


def _regular(s: str, k: int) -> bool:
    return len(s) == k and set(s) <= set("ACGT")


def _inputs(L, k: int, ref_k: int, bf_bits: int, seed: int, n_var: int = 700):
    """genome and signatures, plus a variant whose ref and alt k-mers sit in the last 7 bits of the filter (the
    partial last probe line of the modulo filter); also returns that ref k-mer"""
    rng = random.Random(seed)
    genome = util.make_genome(rng, 30000)
    nested, freqs = util.synth_signatures(rng, genome, k, n_var)
    top_ref, top_alt = _find_kmers(L, k, bf_bits, bf_bits - 7, n=2)
    nested.append([[[top_ref]], [[top_alt]]])
    freqs.append([0.7, 0.3])
    return rng, genome, nested, freqs, top_ref


def _insert(g, ks, fl, k: int, order, batch: int, packed: bool) -> None:
    """signature k-mers in `order`, `batch` per call; packed: the regular ones through mg_add_signatures_packed, the
    irregular ones (short, N / IUPAC) through the text path"""
    for s in range(0, len(order), batch):
        idx = order[s:s + batch]
        reg = [i for i in idx if packed and _regular(ks[i], k)]
        txt = [i for i in idx if not (packed and _regular(ks[i], k))]
        if reg:
            g.add_signatures_packed(kmc.ints_to_packed([kmc.pack_kmer(ks[i]) for i in reg]), [fl[i] for i in reg])
        if txt:
            g.add_signatures([ks[i] for i in txt], [fl[i] for i in txt])


def _finish_index(x, genome: str) -> None:
    x.finalize_alt()
    x.scan_reference(genome)
    x.finalize_context()


def _line_positions(words: np.ndarray, bf_bits: int):
    """(line, number of set bits below it inside its line) of every set bit of bf, in rank order"""
    pos = np.flatnonzero(np.unpackbits(words.view(np.uint8), bitorder="little"))
    pos = pos[pos < bf_bits]
    line = pos >> 8
    first = np.searchsorted(line, line, side="left")
    return line, np.arange(len(pos)) - first


def _check_filter_edges(g, o, bf_bits: int) -> None:
    """the input reaches the edge its filter size is there for"""
    st = g.index_stats()
    line, j = _line_positions(o.bits(0), bf_bits)
    counts = o.bf_counts()
    if bf_bits == DENSE:
        assert st["overflow_keys"] > 100, st
    if bf_bits == MODULO:
        assert (j >= 3).any() and counts[j >= 3].any(), "no counted bit past the three inline counters of its line"
        assert bf_bits % 256 == 7 and (line == st["probe_lines"] - 1).any(), "the partial last line holds no bit"
    if bf_bits in (DENSE, MODULO):
        assert st["overflow_keys"] > 0
        assert counts[line == st["probe_lines"] - 1].any(), "the last line's counters are never hit"


def _same_genotypes(r, cov, exp) -> None:
    assert np.array_equal(r.cov, cov), "COVS"
    assert r.status.tolist() == [e["status"] for e in exp], "status"
    assert r.n_gts.tolist() == [len(e["probs"]) for e in exp], "n_gts"
    assert r.best_gt.tolist() == [e["best"] for e in exp], "GT"
    assert r.gq.tolist() == [e["gq"] for e in exp], "GQ"
    assert (cov > 0).sum() > 100


def _same_counts(g, o, queries) -> None:
    for flag in (0, 1):
        fl_q = [flag] * len(queries)
        assert np.array_equal(g.get_counts(queries, fl_q), o.get_counts(queries, fl_q)), f"get_count is_ref={flag}"
    assert np.array_equal(g.bf_counts(), o.bf_counts()), "rank-indexed bf counters"


def _queries(rng, ks, k: int) -> list:
    return ks + [util.rand_seq(rng, k) for _ in range(200)] + [util.rand_seq(rng, k - 2, "ACGTN") for _ in range(50)]


def _u32_sum(images) -> list:
    return [np.sum(np.stack([im[a] for im in images]), axis=0, dtype=np.uint32) for a in range(3)]


def _reduce_cases():
    cases = [pytest.param(kr, bits, n, False, id=f"k{kr[0]}-{fid}-R{n}")
             for kr in LAYOUTS for bits, fid in ((DENSE, "2^13"), (MODULO, "3x2^12+7"), (SPARSE, "2^22"))
             for n in (2, 3, 16)]
    # replicas spread over the visible devices: the sum kernel reads the peers' arrays over NVLink
    cases += [pytest.param((35, 43), DENSE, 3, True, id="k35-2^13-R3-devices"),
              pytest.param((48, 56), MODULO, 3, True, id="k48-3x2^12+7-R3-devices")]
    return cases


@pytest.mark.parametrize("layout,bf_bits,n_rep,spread", _reduce_cases())
def test_counter_reduce_matches_oracle(oracle_lib, layout, bf_bits, n_rep, spread):
    """R replicas, each built in its own insert order and batching (text and packed inserts), have one index image;
    each scans a share of one stream, their gathered dense images add up element by element (u32) to the image of
    one context that scanned it all, and after mg_reduce_counts context 0 answers like the oracle that scanned the
    whole stream -- counts, bf counters and genotypes -- including a ref key whose sum wraps u32 though no part does.
    A second round of scans and a second reduce add up the same way."""
    k, ref_k = layout
    devs = [0]
    if spread:
        n = _n_gpus()
        if n < 2:
            pytest.skip("needs more GPUs")
        devs = list(range(n))
    rng, genome, nested, freqs, top_ref = _inputs(oracle_lib, k, ref_k, bf_bits, seed=REDUCE_SEEDS.get((k, bf_bits), 7100))
    ks, fl = util.flatten(nested)
    reps = [MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits, device=devs[i % len(devs)]) for i in range(n_rep)]
    whole = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits)
    o = util.OracleRun(oracle_lib, k, ref_k, bf_bits)
    try:
        for i, g in enumerate(reps):          # every replica its own order and batching
            order = list(range(len(ks)))
            random.Random(i).shuffle(order)
            _insert(g, ks, fl, k, order, (61, 97, 500, len(ks))[i % 4], packed=i % 2 == 1)
        whole.add_signatures(list(reversed(ks)), list(reversed(fl)))
        o.add_signatures(ks, fl)
        for x in reps + [whole, o]:
            _finish_index(x, genome)
        stats = whole.index_stats()
        assert all(g.index_stats() == stats for g in reps), [g.index_stats() for g in reps]
        assert stats["irregular_ref_keys"] > 0, "the text path for irregular ref keys is not exercised"

        # one stream in R contiguous shares; the top line's ref key is sampled too, and two records of a genomic
        # ref key carry counts near 2^31 in shares 0 and 1: each part fits u32, their sum wraps
        _, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 30000)
        d = (ref_k - k) // 2
        wrap_key, p = next((s, genome.find(s) - d) for alleles in nested for s in alleles[0][0]
                           if _regular(s, k) and genome.find(s) >= ref_k
                           and set(genome[genome.find(s) - d:genome.find(s) - d + ref_k]) <= set("ACGT"))
        wrap_rec = _records([genome[p:p + ref_k]], [BIG_REF])
        top_rec = _records([_window(rng, genome, top_ref, k, ref_k) for _ in range(3)], [1000, 2000, 3000])
        cuts = np.linspace(0, len(packed), n_rep + 1).astype(int)
        shares = [(packed[a:b], counts[a:b]) for a, b in zip(cuts[:-1], cuts[1:])]
        for s, rec in ((0, wrap_rec), (1, wrap_rec), (n_rep - 1, top_rec)):
            shares[s] = (np.concatenate([shares[s][0], rec[0]]), np.concatenate([shares[s][1], rec[1]]))
        all_p = np.concatenate([s[0] for s in shares])
        all_c = np.concatenate([s[1] for s in shares])
        for g, (sp, sc) in zip(reps, shares):
            g.scan_sample_kmers(sp, sc)
        whole.scan_sample_kmers(all_p, all_c)
        o.scan_sample_kmers(all_p, all_c)
        _check_filter_edges(whole, o, bf_bits)

        images = [util.counter_arrays(g) for g in reps]
        cw = util.counter_arrays(whole)
        for a, name in enumerate(("bf counters", "line key counts", "overflow counts")):
            assert all(len(im[a]) == len(cw[a]) for im in images), name
            assert np.array_equal(_u32_sum(images)[a], cw[a]), name
        assert len(cw[1]) == stats["ref_keys"] - stats["overflow_keys"]
        tails = [(a, len(cw[a]) % 4) for a in (0, 1) if len(cw[a]) % 4]
        assert tails, "every dense array is a multiple of 4 long: the scalar tail of the sum is not exercised"
        assert any(im[a][-r:].any() for im in images[1:] for a, r in tails), "the tails hold no peer counts"

        parts = [int(g.get_counts([wrap_key], [1])[0]) & 0xFFFFFFFF for g in reps]
        assert sum(parts) >= 1 << 32 and max(parts) < 1 << 32, parts

        with pytest.raises(MalvaGpuError, match="error -1:.*listed twice"):
            reduce_counts(reps[:15] + [reps[1]])
        if n_rep == 16:
            with pytest.raises(MalvaGpuError, match="error -1:.*at most 16"):   # 17 distinct contexts
                reduce_counts(reps + [whole])
        reduce_counts(reps)                    # (the refused calls added nothing)
        q = _queries(rng, ks, k)
        _same_counts(reps[0], o, q)
        assert np.array_equal(reps[0].get_counts([wrap_key], [1]).view(np.uint32), np.array([sum(parts) & 0xFFFFFFFF],
                                                                                             np.uint32))
        assert all(np.array_equal(x, y) for x, y in zip(util.counter_arrays(reps[0]), cw))
        batch = SignatureBatch.from_nested(nested, freqs)
        r = reps[0].genotype_packed(PackedSignatureBatch.from_batch(batch, k), 0.001, 120, False, want_lik=False)
        _same_genotypes(r, *o.genotype(batch, 0.001, 120, False))

        # round two: every replica scans another share, context 0 scans on the scattered sums; the second reduce
        # adds what each context holds at that point
        for i, g in enumerate(reps):
            sp, sc = shares[(i + 1) % n_rep]
            g.scan_sample_kmers(sp, sc)
        before = _u32_sum([util.counter_arrays(g) for g in reps])
        reduce_counts(reps)
        after = util.counter_arrays(reps[0])
        for a in range(3):
            assert np.array_equal(after[a], before[a]), a
    finally:
        for x in reps + [whole, o]:
            x.close()


def _device_batch(pb: PackedSignatureBatch, dev):
    """the packed batch and the genotype outputs as torch tensors on dev: (tensors, device addresses, dims)"""
    import torch

    nv, na = pb.n_variants, int(pb.var_allele_off[-1])
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
    nall = np.diff(pb.var_allele_off.astype(np.int64))
    dims = (nv, na, len(pb.sig_kmer_off) - 1, len(pb.kmers), len(pb.irr_kmer), len(pb.irr_pool),
            int(np.maximum(nall * (nall + 1) // 2, nall).sum()))
    return t, {n: x.data_ptr() for n, x in t.items()}, dims


@pytest.mark.parametrize("bf_bits", [pytest.param(DENSE, id="2^13"), pytest.param(SPARSE, id="2^22")])
@pytest.mark.parametrize("k,ref_k", LAYOUTS)
def test_lookup_sum_at_every_layout(oracle_lib, k, ref_k, bf_bits):
    """the other multi-GPU scheme (include/malva_gpu.h: mg_lookup_packed_device / mg_genotype_weights_device): every
    replica looks the batch up in its own partial counters (bf counters raw), the weight vectors are summed (what
    bench.py does with ncclReduce), and the genotypes computed from the sum equal a single context's and the oracle's
    -- incl. the uint16 wrap-around of a bf counter that only the SUM exceeds, on the bit of an irregular alt k-mer
    (looked up by k_lookup, not k_lookup_packed).  The library's work is put on torch's stream."""
    import torch

    rng = random.Random(2024 + k)
    genome = util.make_genome(rng, 30000)
    nested, freqs = util.synth_signatures(rng, genome, k, 500)
    # an irregular alt k-mer (k - 4 symbols, a contig end) and a regular k-mer of the sample stream on one bf bit,
    # the last one of the filter
    short_alt = _find_kmers(oracle_lib, k - 4, bf_bits, bf_bits - 1)[0]
    hitter = _find_kmers(oracle_lib, k, bf_bits, bf_bits - 1, first=1 << 40)[0]
    p = next(p for p in range(k, len(genome)) if set(genome[p:p + k]) <= set("ACGT"))
    nested.append([[[genome[p:p + k]]], [[short_alt]]])
    freqs.append([0.6, 0.4])
    ks, fl = util.flatten(nested)
    a, b, whole = (MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits) for _ in range(3))
    o = util.OracleRun(oracle_lib, k, ref_k, bf_bits)
    try:
        for x in (a, b, whole, o):
            x.add_signatures(ks, fl)
            _finish_index(x, genome)
        assert np.array_equal(whole.bits(0), o.bits(0)) and int(o.bits(0)[-1]) >> 63 == 1
        # (counts past 2^16 per record where few sample k-mers share a bit with the irregular one)
        _, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 30000, big_counts=bf_bits == SPARSE)
        half = len(packed) // 2
        hit = _records([_window(rng, genome, hitter, k, ref_k, o)], [12000])
        halves = [(np.concatenate([packed[:half], hit[0]]), np.concatenate([counts[:half], hit[1]])),
                  (np.concatenate([packed[half:], hit[0]]), np.concatenate([counts[half:], hit[1]]))]
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        for x in (a, b, whole):
            x.set_stream(side.cuda_stream)
        # each half is scanned several times so that bf counters pass 2^16 in the sum but not in either part
        for _ in range(3):
            for x, (hp, hc) in ((a, halves[0]), (b, halves[1])):
                x.scan_sample_kmers(hp, hc)
            for hp, hc in halves:
                whole.scan_sample_kmers(hp, hc)
                o.scan_sample_kmers(hp, hc)
        batch = SignatureBatch.from_nested(nested, freqs)
        pb = PackedSignatureBatch.from_batch(batch, k)
        ix = len(ks) - 1
        assert ks[ix] == short_alt and int(pb.kmers["hi"][ix]) & IRREGULAR_BIT
        exp = whole.genotype_packed(pb, 0.001, 10 ** 9, False)
        dev = torch.device("cuda", 0)
        t, ptrs, dims = _device_batch(pb, dev)
        wa = torch.zeros(dims[3], dtype=torch.int32, device=dev)
        wb = torch.zeros(dims[3], dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        with torch.cuda.stream(side):                          # no host synchronisation between the five calls
            a.lookup_packed_device(ptrs, dims, wa.data_ptr())
            b.lookup_packed_device(ptrs, dims, wb.data_ptr())
            total = wa + wb                                    # (stream-ordered with the library's kernels)
            raw = total.clone()
            a.genotype_weights_device(ptrs, dims, total.data_ptr(), 0.001, 10 ** 9, False)
        torch.cuda.synchronize()
        for x in (a, b, whole):
            x.set_stream(0)
        pa, pb_, s = (int(w[ix]) & 0xFFFFFFFF for w in (wa, wb, raw))
        assert pa < 1 << 16 and pb_ < 1 << 16 and s >= 1 << 16, ("the irregular k-mer's wrap is not exercised", pa, pb_)
        assert int(total[ix]) == s & 0xFFFF
        assert int((raw.to(torch.int64) & 0xFFFFFFFF).max()) > 65535, "the wrap-around is not exercised"
        got = {nme: t[nme].cpu().numpy() for nme in ("cov", "n_gts", "status", "best_gt", "gq")}
        got["cov"] = got["cov"].view(np.uint32)
        for nme, e in got.items():
            assert np.array_equal(e, getattr(exp, nme)), nme
        _same_genotypes(exp, *o.genotype(batch, 0.001, 10 ** 9, False))
    finally:
        for x in (a, b, whole, o):
            x.close()


def _export_bits(g, which: int) -> np.ndarray:
    n = C.c_uint64(0)
    check(g._L.mg_export_set_bits(g._h, which, None, 0, C.byref(n)))
    out = np.zeros(max(n.value, 1), np.uint64)
    check(g._L.mg_export_set_bits(g._h, which, out.ctypes.data_as(util.u64p), n.value, C.byref(n)))
    return out[:n.value]


def _export_keys(g) -> np.ndarray:
    n = C.c_uint64(0)
    check(g._L.mg_export_ref_keys(g._h, None, 0, C.byref(n)))
    out = np.zeros(max(2 * n.value, 2), np.uint64)
    check(g._L.mg_export_ref_keys(g._h, out.ctypes.data_as(util.u64p), n.value, C.byref(n)))
    return out[:2 * n.value].view(kmc.KMER_DTYPE)


def _import_bits(g, which: int, idx: np.ndarray) -> None:
    idx = np.ascontiguousarray(idx, dtype=np.uint64)
    check(g._L.mg_import_set_bits(g._h, which, idx.ctypes.data_as(util.u64p), len(idx)))


@pytest.mark.parametrize("bf_bits", FILTERS)
@pytest.mark.parametrize("k,ref_k", LAYOUTS)
def test_reloaded_index_equals_the_built_one(oracle_lib, k, ref_k, bf_bits):
    """`malva-geno call` never builds its index from the signatures: it loads the set bits of bf and context_bf and
    the packed ref keys that `index` exported.  A context loaded that way must hold the image of the context that
    built them -- same bits, keys and probe lines, same counters and genotypes after the same scans, and counters that
    add up with the built context's in mg_reduce_counts."""
    rng, genome, nested, freqs, top_ref = _inputs(oracle_lib, k, ref_k, bf_bits, seed=8200 + k + bf_bits % 1013)
    ks, fl = util.flatten(nested)
    a = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits)
    b = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits)
    o = util.OracleRun(oracle_lib, k, ref_k, bf_bits)
    try:
        order = list(range(len(ks)))
        rng.shuffle(order)
        _insert(a, ks, fl, k, order, 83, packed=False)
        o.add_signatures(ks, fl)
        for x in (a, o):
            _finish_index(x, genome)
        bf_idx, ctx_idx, keys = _export_bits(a, 0), _export_bits(a, 1), _export_keys(a)
        want_keys = sorted({kmc.canonical_int(kmc.pack_kmer(s), k) for s, f in zip(ks, fl) if f and _regular(s, k)})
        assert sorted(kmc.packed_to_ints(keys)) == want_keys    # (in the order of a racing emit kernel)
        # the sequence of call_main (csrc/host/malva_geno.cpp)
        _import_bits(b, 0, bf_idx)
        b.add_signatures_packed(keys, np.ones(len(keys), np.uint8))
        b.finalize_alt()
        _import_bits(b, 1, ctx_idx)
        b.finalize_context()
        for which in (0, 1):
            assert np.array_equal(_export_bits(b, which), _export_bits(a, which)), which
            assert np.array_equal(b.bits(which), o.bits(which)) and np.array_equal(a.bits(which), o.bits(which))
        assert sorted(kmc.packed_to_ints(_export_keys(b))) == want_keys, "keys of the reloaded index"
        # the index file carries packed keys only: the irregular ref keys (N / IUPAC, short) stay behind, and they
        # never count (KMAP::get_count of a key no sample k-mer can equal)
        sa, sb = a.index_stats(), b.index_stats()
        assert sa.pop("irregular_ref_keys") > 0 and sb.pop("irregular_ref_keys") == 0
        assert sa == sb
        q = _queries(rng, ks, k)
        ctx_q = [genome[p:p + ref_k] for p in range(0, len(genome) - ref_k, 37)]
        for which, qq in ((0, q), (1, q), (1, ctx_q), (2, [s for s in q if _regular(s, k)])):
            want = o.test_keys(which, qq)
            assert np.array_equal(a.test_keys(which, qq), want) and np.array_equal(b.test_keys(which, qq), want), which

        # a built and a reloaded context share one image: their shares of a stream add up in mg_reduce_counts
        _, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 20000)
        top = _records([_window(rng, genome, top_ref, k, ref_k) for _ in range(2)], [700, 900])
        packed, counts = np.concatenate([packed, top[0]]), np.concatenate([counts, top[1]])
        half = len(packed) // 2 + 3
        a.scan_sample_kmers(packed[:half], counts[:half])
        b.scan_sample_kmers(packed[half:], counts[half:])
        o.scan_sample_kmers(packed, counts)
        _check_filter_edges(a, o, bf_bits)
        ia, ib = util.counter_arrays(a), util.counter_arrays(b)
        reduce_counts([a, b])
        _same_counts(a, o, q)
        assert all(np.array_equal(x, y) for x, y in zip(util.counter_arrays(a), _u32_sum([ia, ib])))
        # the same scans on both: B completes the stream, then both scan it once more
        b.scan_sample_kmers(packed[:half], counts[:half])
        for x in (a, b, o):
            x.scan_sample_kmers(packed, counts)
        ia, ib = util.counter_arrays(a), util.counter_arrays(b)
        assert all(np.array_equal(x, y) for x, y in zip(ia, ib)), "counter images of the built and the reloaded index"
        assert ia[1].any() and ia[0].any()
        for g in (a, b):
            _same_counts(g, o, q)
        batch = SignatureBatch.from_nested(nested, freqs)
        pb = PackedSignatureBatch.from_batch(batch, k)
        ra, rb = (g.genotype_packed(pb, 0.001, 150, False) for g in (a, b))
        for nme in ("cov", "n_gts", "status", "best_gt", "gq"):
            assert np.array_equal(getattr(ra, nme), getattr(rb, nme)), nme
        for v in range(batch.n_variants):       # (the slots past n_gts of a variant are not written)
            sl = slice(int(ra.lik_off[v]), int(ra.lik_off[v]) + int(ra.n_gts[v]))
            assert np.array_equal(ra.lik[sl].view(np.uint64), rb.lik[sl].view(np.uint64)), v
        _same_genotypes(ra, *o.genotype(batch, 0.001, 150, False))
    finally:
        for x in (a, b, o):
            x.close()
