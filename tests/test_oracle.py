"""Pins the CPU oracle (oracle/malva_oracle.c) before anything trusts it.

Anchors: XXH3 known answers (SURVEY 8c), python-xxhash, the reference's own
classes through oracle/_ref/libmalva_ref.so, and glibc's logf.  Where oracle/_ref
is not built, the oracle's side of each comparison with the reference is checked
against its digest in tests/golden/oracle_vs_reference.json (parity_util.Agree).
"""
import ctypes as C
import random

import numpy as np
import pytest

from parity_util import Agree

KATS = [
    (b"ACGT" * 8 + b"ACG", 0x6AE639F026113AEA),
    (b"ACGT" * 10 + b"ACG", 0x1E2873EC7681F59A),
]


@pytest.fixture
def agree(request, ref_or_none):
    return Agree(request.node.name, ref_or_none)


def rand_kmer(rng, k, alphabet="ACGT"):
    return "".join(rng.choice(alphabet) for _ in range(k)).encode()


def test_xxh3_known_answers(oracle_lib):
    for s, h in KATS:
        assert oracle_lib.mo_xxh3_64(s, len(s)) == h


def test_xxh3_against_python_xxhash_all_lengths(oracle_lib):
    xxhash = pytest.importorskip("xxhash")
    rng = random.Random(1)
    for n in range(0, 241):
        for _ in range(4):
            s = bytes(rng.randrange(256) for _ in range(n))
            assert oracle_lib.mo_xxh3_64(s, n) == xxhash.xxh3_64_intdigest(s), n


def test_xxh3_against_reference_build(oracle_lib, agree):
    rng = random.Random(2)
    for n in list(range(0, 130)) + [200, 240]:
        s = bytes(rng.randrange(256) for _ in range(n))
        agree.eq(oracle_lib.mo_xxh3_64(s, n), agree.L.ref_xxh3(s, n))
    agree.done()


def test_logf_restatement_matches_libm(oracle_lib):
    libm = C.CDLL("libm.so.6")
    libm.logf.restype = C.c_float
    libm.logf.argtypes = [C.c_float]
    rng = np.random.default_rng(3)
    bits = np.concatenate([
        rng.integers(1, 0x7F800000, size=200000, dtype=np.uint32),
        np.array([0, 1, 0x00800000, 0x3F800000, 0x3F7FFFFF, 0x3F800001, 0x7F7FFFFF, 0x7F800000], dtype=np.uint32),
    ])
    xs = bits.view(np.float32)
    for x in xs.tolist():
        a = np.float32(oracle_lib.mo_logf(x))
        b = np.float32(libm.logf(x))
        assert a.view(np.uint32) == b.view(np.uint32), x


@pytest.mark.parametrize("k", [35, 43, 16, 31, 64])
def test_bf_matches_reference_class(oracle_lib, agree, k):
    ref_lib = agree.L
    rng = random.Random(10 + k)
    size = 5003 if k != 35 else 4096  # non power of two and power of two
    ob = oracle_lib.mo_bf_new(size)
    rb = ref_lib.ref_bf_new(size)
    alpha = ["ACGT", "ACGTN", "ACGTNWMRacgtn"]
    keys = [rand_kmer(rng, rng.choice([k, k, k, max(1, k - 3)]), rng.choice(alpha)) for _ in range(600)]
    for s in keys[:300]:
        oracle_lib.mo_bf_add_key(ob, s)
        ref_lib.ref_bf_add_key(rb, s)
    for s in keys:
        agree.eq(oracle_lib.mo_bf_test_key(ob, s), ref_lib.ref_bf_test_key(rb, s))
    # increments before switch_mode are no-ops in both
    inc = oracle_lib.mo_bf_increment(ob, keys[0], 5)
    agree.eq(inc, ref_lib.ref_bf_increment(rb, keys[0], 5))
    assert inc == 0
    oracle_lib.mo_bf_switch_mode(ob)
    ref_lib.ref_bf_switch_mode(rb)
    for s in keys:
        c = rng.choice([1, 2, 255, 40000, 70000])
        oracle_lib.mo_bf_increment(ob, s, c)
        ref_lib.ref_bf_increment(rb, s, c)
    for s in keys:
        agree.eq(oracle_lib.mo_bf_get_count(ob, s), ref_lib.ref_bf_get_count(rb, s))
    oracle_lib.mo_bf_free(ob)
    ref_lib.ref_bf_free(rb)
    agree.done()


def test_kmap_matches_reference_class(oracle_lib, agree):
    ref_lib = agree.L
    rng = random.Random(20)
    om = oracle_lib.mo_kmap_new()
    rm = ref_lib.ref_kmap_new()
    keys = [rand_kmer(rng, rng.choice([35, 35, 20]), rng.choice(["ACGT", "ACGTN", "ACGTWK"])) for _ in range(3000)]
    for s in keys[:1500]:
        oracle_lib.mo_kmap_add_key(om, s)
        ref_lib.ref_kmap_add_key(rm, s)
    agree.eq(oracle_lib.mo_kmap_size(om), ref_lib.ref_kmap_size(rm))
    for s in keys:
        c = rng.choice([1, 7, 255, 2 ** 31 - 1])
        oracle_lib.mo_kmap_increment(om, s, c)
        ref_lib.ref_kmap_increment(rm, s, c)
    # re-adding an existing key resets it to 0 in both
    oracle_lib.mo_kmap_add_key(om, keys[0])
    ref_lib.ref_kmap_add_key(rm, keys[0])
    for s in keys:
        agree.eq(oracle_lib.mo_kmap_test_key(om, s), ref_lib.ref_kmap_test_key(rm, s))
        agree.eq(oracle_lib.mo_kmap_get_count(om, s), ref_lib.ref_kmap_get_count(rm, s))
    oracle_lib.mo_kmap_free(om)
    ref_lib.ref_kmap_free(rm)
    agree.done()


def _u32(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint32))


def test_scan_and_reference_pass_match_reference_loops(oracle_lib, agree):
    ref_lib = agree.L
    rng = random.Random(30)
    k, ref_k, size = 35, 43, 1 << 16
    genome = "".join(rng.choice("ACGT") for _ in range(6000))
    genome = genome[:2000] + "NNNNNNNNNNNNWM" + genome[2014:]
    ob, oc, om = oracle_lib.mo_bf_new(size), oracle_lib.mo_bf_new(size), oracle_lib.mo_kmap_new()
    rb, rc, rm = ref_lib.ref_bf_new(size), ref_lib.ref_bf_new(size), ref_lib.ref_kmap_new()
    # alt signatures = mutated windows, ref signatures = true windows
    for _ in range(400):
        p = rng.randrange(0, len(genome) - k)
        w = genome[p:p + k]
        alt = (w[:17] + rng.choice("ACGT") + w[18:]).encode()
        oracle_lib.mo_bf_add_key(ob, alt)
        ref_lib.ref_bf_add_key(rb, alt)
        oracle_lib.mo_kmap_add_key(om, w.encode())
        ref_lib.ref_kmap_add_key(rm, w.encode())
    oracle_lib.mo_bf_switch_mode(ob)
    ref_lib.ref_bf_switch_mode(rb)
    oracle_lib.mo_reference_pass(ob, oc, genome.encode(), len(genome), k, ref_k)
    ref_lib.ref_reference_pass(rb, rc, genome.encode(), k, ref_k)
    oracle_lib.mo_bf_switch_mode(oc)
    ref_lib.ref_bf_switch_mode(rc)
    assert oracle_lib.mo_bf_popcount(oc) > 0
    ctxs = []
    for _ in range(4000):
        p = rng.randrange(0, len(genome) - ref_k)
        w = genome[p:p + ref_k]
        if any(ch not in "ACGT" for ch in w):
            continue
        if rng.random() < 0.3:
            q = rng.randrange(ref_k)
            w = w[:q] + rng.choice("ACGT") + w[q + 1:]
        ctxs.append(w)
    counts = np.array([rng.choice([2, 3, 9, 255]) for _ in ctxs], dtype=np.uint32)
    blob = "".join(ctxs).encode()
    oracle_lib.mo_scan_ascii(ob, oc, om, blob, _u32(counts), len(ctxs), k, ref_k)
    for w, c in zip(ctxs, counts.tolist()):
        ref_lib.ref_scan_kmer(rb, rc, rm, w.encode(), c, k, ref_k)
    nonzero = 0
    for p in range(0, len(genome) - ref_k):
        w43 = genome[p:p + ref_k].encode()
        w35 = genome[p + 4:p + 4 + k].encode()
        agree.eq(oracle_lib.mo_bf_test_key(oc, w43), ref_lib.ref_bf_test_key(rc, w43))
        agree.eq(oracle_lib.mo_bf_get_count(ob, w35), ref_lib.ref_bf_get_count(rb, w35))
        a = oracle_lib.mo_kmap_get_count(om, w35)
        agree.eq(a, ref_lib.ref_kmap_get_count(rm, w35))
        nonzero += a > 0
    assert nonzero > 50
    agree.done()


def test_scan_packed_equals_scan_ascii(oracle_lib):
    from malva_b200 import kmc

    rng = random.Random(31)
    k, ref_k, size = 35, 43, 1 << 14
    ctxs = [rand_kmer(rng, ref_k).decode() for _ in range(500)]
    counts = np.array([rng.randrange(2, 256) for _ in ctxs], dtype=np.uint32)
    res = []
    for mode in ("ascii", "packed"):
        b, c, m = oracle_lib.mo_bf_new(size), oracle_lib.mo_bf_new(size), oracle_lib.mo_kmap_new()
        for w in ctxs[:250]:
            oracle_lib.mo_bf_add_key(b, w[4:39].encode())
            oracle_lib.mo_kmap_add_key(m, w[4:39].encode())
        oracle_lib.mo_bf_switch_mode(b)
        oracle_lib.mo_bf_switch_mode(c)
        if mode == "ascii":
            oracle_lib.mo_scan_ascii(b, c, m, "".join(ctxs).encode(), _u32(counts), len(ctxs), k, ref_k)
        else:
            packed = kmc.ints_to_packed([kmc.pack_kmer(w) for w in ctxs])
            oracle_lib.mo_scan_packed(b, c, m, packed.ctypes.data_as(C.POINTER(C.c_uint64)), _u32(counts),
                                      len(ctxs), k, ref_k)
        res.append([(oracle_lib.mo_bf_get_count(b, w[4:39].encode()),
                     oracle_lib.mo_kmap_get_count(m, w[4:39].encode())) for w in ctxs])
    assert res[0] == res[1]
    assert sum(x[1] for x in res[0]) > 0


def _genotype_oracle(L, cov, freq, err, max_cov, haploid):
    n = len(cov)
    cov = np.asarray(cov, dtype=np.uint32)
    freq = np.asarray(freq, dtype=np.float32)
    probs = np.zeros(max(n * (n + 1) // 2, n), dtype=np.float64)
    status = C.c_int(0)
    ng = L.mo_genotype(_u32(cov), freq.ctypes.data_as(C.POINTER(C.c_float)), n, C.c_float(err), max_cov,
                       int(haploid), probs.ctypes.data_as(C.POINTER(C.c_double)), C.byref(status))
    bi, gq = C.c_int(0), C.c_int(0)
    L.mo_call(probs.ctypes.data_as(C.POINTER(C.c_double)), ng, C.byref(bi), C.byref(gq))
    return probs[:ng].copy(), status.value, bi.value, gq.value


def _genotype_ref(L, cov, freq, err, max_cov, haploid):
    n = len(cov)
    cov = np.asarray(cov, dtype=np.uint32)
    freq = np.asarray(freq, dtype=np.float32)
    probs = np.zeros(64, dtype=np.float64)
    line = C.create_string_buffer(4096)
    ng = L.ref_genotype(_u32(cov), freq.ctypes.data_as(C.POINTER(C.c_float)), n, C.c_float(err), max_cov,
                        int(haploid), probs.ctypes.data_as(C.POINTER(C.c_double)), 64, line, 4096)
    return probs[:ng].copy(), line.value.decode()


def test_genotype_bit_exact_against_reference(oracle_lib, agree):
    rng = np.random.default_rng(40)
    checked = 0
    for it in range(4000):
        n = int(rng.integers(2, 5))
        haploid = bool(rng.integers(0, 2))
        err = float(rng.choice([0.001, 0.01, 0.05]))
        cov = rng.integers(0, 60, size=n)
        if it % 11 == 0:
            cov[:] = 0
        if it % 13 == 0:
            cov[rng.integers(0, n)] = 250  # above max_cov
        if rng.random() < 0.5:
            cov[rng.integers(0, n)] = 0
        af = rng.random(n - 1).astype(np.float32) * np.float32(0.5 / (n - 1))
        if it % 7 == 0:
            af[0] = 0.0
        f0 = np.float32(1.0 - float(np.sum(af.astype(np.float64))))
        freq = np.concatenate([[max(f0, np.float32(0))], af]).astype(np.float32)
        po, status, bi, gq = _genotype_oracle(oracle_lib, cov, freq, err, 200, haploid)
        names = [str(g) for g in range(n)] if haploid else [f"{a}/{b}" for a in range(n) for b in range(a, n)]
        exp_gt = ("0" if haploid else "0/0") if status != 0 else names[bi]
        if agree.live:
            pr, line = _genotype_ref(agree.L, cov, freq, err, 200, haploid)
            assert len(po) == len(pr)
            assert np.array_equal(po.view(np.uint64), pr.view(np.uint64)), (cov, freq, po, pr)
            # GT and GQ as printed by the reference's output_variants
            gtgq = line.rstrip("\n").split("\t")[-1]
            assert gtgq == f"{exp_gt}:{gq}", (line, status, bi, gq)
        agree.record(po.view(np.uint64), f"{exp_gt}:{gq}")
        checked += 1
    assert checked == 4000
    agree.done()


@pytest.mark.parametrize("k,ref_k", [(35, 43), (36, 43), (31, 40), (20, 21), (43, 43), (15, 21)])
@pytest.mark.parametrize("glen", [12, 30, 43, 44, 100, 1500])
def test_reference_pass_matches_reference_loop_all_shapes(oracle_lib, agree, k, ref_k, glen):
    """Odd (ref_k - k) makes the reference's k-mer window non-contiguous for its first k-1 slides
    (main.cpp:395-397); contigs shorter than ref_k hash truncated substr() results."""
    ref_lib = agree.L
    rng = random.Random(1000 * k + ref_k + glen)
    d = (ref_k - k) // 2
    if glen < d:
        pytest.skip("the reference throws std::out_of_range here")
    genome = "".join(rng.choice("ACGT") for _ in range(glen))
    if glen > 200:
        genome = genome[:100] + "NNWN" + genome[104:]
    size = 1 << 12
    ob, oc = oracle_lib.mo_bf_new(size), oracle_lib.mo_bf_new(size)
    rb, rc = ref_lib.ref_bf_new(size), ref_lib.ref_bf_new(size)
    # dense alt filter: about a third of all probes hit, so the context filter gets many bits
    for _ in range(1500):
        s = "".join(rng.choice("ACGT") for _ in range(k)).encode()
        oracle_lib.mo_bf_add_key(ob, s)
        ref_lib.ref_bf_add_key(rb, s)
    oracle_lib.mo_reference_pass(ob, oc, genome.encode(), len(genome), k, ref_k)
    ref_lib.ref_reference_pass(rb, rc, genome.encode(), k, ref_k)
    n = size // 64
    a = np.ctypeslib.as_array(oracle_lib.mo_bf_words(oc), shape=(n,)).copy()
    # compare through test_key on every window the reference could have inserted, plus popcount
    ref_lib.ref_bf_switch_mode(rc)
    oracle_lib.mo_bf_switch_mode(oc)
    probes = set()
    for p in range(0, max(1, glen - ref_k + 1)):
        probes.add(genome[p:p + ref_k])
    probes.add(genome[:ref_k])
    present = []
    for w in sorted(probes):
        hit = oracle_lib.mo_bf_test_key(oc, w.encode())
        agree.eq(hit, ref_lib.ref_bf_test_key(rc, w.encode()), w)
        if hit:
            present.append(w)
    assert int(np.unpackbits(a.view(np.uint8)).sum()) == len(_distinct_bits(present, size, oracle_lib))
    if glen >= 100:
        assert len(present) > 5
    agree.done()


def _distinct_bits(present, size, oracle_lib):
    """bit indices of the probes reported as present (by both filters: checked k-mer by k-mer)."""
    import ctypes as C
    out = set()
    for w in present:
        buf = C.create_string_buffer(len(w) + 1)
        oracle_lib.mo_canonical(w.encode(), len(w), buf)
        out.add(oracle_lib.mo_xxh3_64(buf.raw[:len(w)], len(w)) % size)
    return out
