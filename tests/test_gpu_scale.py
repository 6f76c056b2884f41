"""The device paths that only run at the sizes the CLI uses, against the CPU oracle on the same input, exactly:

A. the reference pass across its 32 MB contig chunks (halo, non-ACGT symbols at a seam, the last chunk holding a
   single window, pinned and pageable sources, several contigs through one context);
B. host-buffer scans across their 2^22-k-mer staging chunks (both streams in flight in one call, the stream join
   before genotyping, KMC record offsets past the first chunk, staging buffers that grow between calls);
C. filters of 2^33 bits and more, on the mask and the 64-bit modulo path of bf_index, with keys planted in the last
   probe line.

The chunk sizes are the production constants (REF_CHUNK and STAGE_KMERS in malva_b200/csrc/malva_gpu.cu): every
test asserts the number of kernel launches its input must cause, so a change of either constant fails here instead
of quietly moving the seams away from what the inputs plant."""
import ctypes as C
import math
import os
import random
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from malva_b200 import MalvaGpu, SignatureBatch, kmc
from malva_b200.api import PackedSignatureBatch, check
import parity_util as util

REF_CHUNK = 32 << 20          # window end positions per k_refpass launch
STAGE_KMERS = 1 << 22         # k-mers (or KMC records) per staging chunk of a host-buffer scan
SCAN_LAUNCHES = 2             # per staging chunk: k_scan + k_scan_hits (deferred filter hits, the default)
ACGT = np.frombuffer(b"ACGT", np.uint8)


def _bases(rng: np.random.Generator, n: int) -> np.ndarray:
    return ACGT[rng.integers(0, 4, n, dtype=np.uint8)]


def _window_kmer(seq: np.ndarray, p: int, k: int, ref_k: int) -> bytes:
    """the k-mer the reference tests for the window ending at p (main.cpp:385-400; the odd ref_k-k quirk of the
    first k slides of a contig included, as oracle/malva_oracle.c restates it)"""
    d, h = (ref_k - k) // 2, ref_k - 1
    t = p - h
    if (ref_k - k) % 2 and t == 0:
        return seq[d:d + k].tobytes()
    if (ref_k - k) % 2 and 1 <= t < k:
        return seq[d + t:d + k].tobytes() + seq[k + d + 1:k + d + 1 + t].tobytes()
    return seq[p - d - k + 1:p - d + 1].tobytes()


def _ref_chunks(n: int, ref_k: int) -> int:
    return 1 if n < ref_k else math.ceil((n - (ref_k - 1)) / REF_CHUNK)


# ---------------------------------------------------------------------------------------------------------------
# A. reference pass across chunk seams
# ---------------------------------------------------------------------------------------------------------------
def _seam_contig(rng: np.random.Generator, n: int, k: int, ref_k: int, pattern0: int):
    """a random contig of n bases with something planted at every chunk seam s = j*REF_CHUNK + ref_k-1 (the first
    window of chunk j), the pattern cycling with the seam: 0 nothing; 1 an N in the halo (the last ref_k-1 bytes of
    chunk j-1), inside the context of the windows s-2 .. s+1 but not in their k-mers; 2 IUPAC symbols inside the
    k-mers of the windows s-1, s and s+k..; 3 an N run across the seam.  Returns (seq, seams, alt k-mers): the
    k-mers of the windows s-2 .. s+k-1 (the first k windows of the later chunk: the odd-length quirk must not apply
    there), of the first k+2 windows of the contig, and of 2,000 random windows."""
    h, d = ref_k - 1, (ref_k - k) // 2
    seq = _bases(rng, n)
    seams = [j * REF_CHUNK + h for j in range(1, _ref_chunks(n, ref_k))]
    for j, s in enumerate(seams):
        pat = (pattern0 + j) % 4
        if pat == 1:
            seq[s - h + 1] = ord("N")
        elif pat == 2:
            seq[s - d] = ord("W")
            seq[s - d - k] = ord("M")
            seq[s + 1] = ord("R")
        elif pat == 3:
            seq[s - 20:s + 20] = ord("N")
    ps = [p for s in seams for p in range(s - 2, min(s + k, n))]
    ps += list(range(h, min(h + k + 2, n)))
    ps += rng.integers(h, n, 2000).tolist()
    return seq, seams, [_window_kmer(seq, p, k, ref_k) for p in ps]


def _scan_contigs(oracle_lib, k, ref_k, contigs, pinned_too=False):
    """every contig through a pageable-source context (and a pinned-source one), the oracle in step: context_bf
    compared after each contig, plus test_key on the seam windows"""
    bits = 1 << 22
    alts = [a for _, _, al in contigs for a in al]
    o = util.OracleRun(oracle_lib, k, ref_k, bits)
    gs = [MalvaGpu(k=k, ref_k=ref_k, bf_bits=bits) for _ in range(2 if pinned_too else 1)]
    L = gs[0]._L
    pin = C.c_void_p()
    try:
        if pinned_too:
            assert L.mg_host_alloc(C.byref(pin), max(len(s) for s, _, _ in contigs)) == 0
        for x in [o] + gs:
            x.add_signatures(alts, [0] * len(alts))
            x.finalize_alt()
        for seq, seams, _ in contigs:
            raw = seq.tobytes()
            o.scan_reference(raw)
            want = o.bits(1)
            h = ref_k - 1
            wins = [raw[p - h:p + 1] for s in seams for p in range(s - 2, min(s + 3, len(raw)))]
            ow = o.test_keys(1, wins)
            assert ow.all(), "a planted seam window does not set its context bit: the planting is wrong"
            for i, g in enumerate(gs):
                n0 = g.launch_count()
                if i == 0:
                    g.scan_reference(raw)
                else:
                    C.memmove(pin, raw, len(raw))
                    g.scan_reference_ptr(pin.value, len(raw))
                assert g.launch_count() - n0 == _ref_chunks(len(raw), ref_k), \
                    "k_refpass launches per contig changed: REF_CHUNK moved, update the contig lengths of this file"
                got = g.bits(1)
                if not np.array_equal(got, want):
                    w = int(np.flatnonzero(got != want)[0])
                    raise AssertionError(f"context_bf differs ({'pinned' if i else 'pageable'} source, contig of "
                                         f"{len(raw)} bases, seams {seams}): first in word {w}")
                assert np.array_equal(g.test_keys(1, wins), ow)
        assert int(np.unpackbits(want.view(np.uint8)).sum()) > 1000
    finally:
        for x in [o] + gs:
            x.close()
        if pin.value:
            L.mg_host_free(pin)


@pytest.mark.gpu
@pytest.mark.slow
def test_reference_pass_chunk_seams_35_43(oracle_lib):
    """the specialised kernel over contigs of one chunk (C+h), one chunk and a single window (C+h+1), three chunks
    whose last holds one window (2C+h+1), and an odd length above 2C, with a contig shorter than ref_k
    (k_refpass_short) between the last two; pageable and pinned sources give the oracle's bits"""
    k, ref_k = 35, 43
    h = ref_k - 1
    rng = np.random.default_rng(35)
    lengths = [REF_CHUNK + h, REF_CHUNK + h + 1, 2 * REF_CHUNK + h + 1, 20, 2 * REF_CHUNK + 123457]
    contigs = []
    for i, n in enumerate(lengths):
        if n < ref_k:
            contigs.append((_bases(rng, n), [], []))
        else:
            contigs.append(_seam_contig(rng, n, k, ref_k, pattern0=i))
    assert sum(len(s) for _, s, _ in contigs) == 5
    _scan_contigs(oracle_lib, k, ref_k, contigs, pinned_too=True)


@pytest.mark.gpu
@pytest.mark.slow
@pytest.mark.parametrize("k,ref_k,n", [
    (36, 43, 2 * REF_CHUNK + 42 + 1),   # runtime-length kernel; odd ref_k-k: the quirk of the first chunk only
    (31, 39, 2 * REF_CHUNK + 9999),
])
def test_reference_pass_chunk_seams_runtime_k(oracle_lib, k, ref_k, n):
    rng = np.random.default_rng(k * 100 + ref_k)
    contig = _seam_contig(rng, n, k, ref_k, pattern0=k)
    assert len(contig[1]) == 2
    _scan_contigs(oracle_lib, k, ref_k, [contig])


# ---------------------------------------------------------------------------------------------------------------
# B. host-buffer scans across staging chunks
# ---------------------------------------------------------------------------------------------------------------
N_SAMPLE = 2 * STAGE_KMERS + (STAGE_KMERS // 2) + 37      # three chunks and a ragged tail


@pytest.fixture(scope="module")
def sample_run(oracle_lib):
    """10.5 M sample k-mers drawn from a pool of 10^5 synth_sample k-mers (filter hits, key hits, context vetoes),
    counts up to 70,000; the oracle's state after scanning them"""
    k, ref_k, bits = 35, 43, 1 << 22
    rng = random.Random(2718)
    genome = util.make_genome(rng, 60000)
    nested, freqs = util.synth_signatures(rng, genome, k, 1500)
    ks, fl = util.flatten(nested)
    words, pool, _ = util.synth_sample(rng, genome, nested, k, ref_k, 100000)
    npr = np.random.default_rng(31)
    idx = npr.integers(0, len(pool), N_SAMPLE)
    packed = pool[idx]
    counts = npr.integers(2, 256, N_SAMPLE, dtype=np.uint32)
    big = npr.random(N_SAMPLE) < 0.01
    counts[big] = npr.integers(30000, 70001, int(big.sum()), dtype=np.uint32)
    o = util.OracleRun(oracle_lib, k, ref_k, bits)
    o.add_signatures(ks, fl)
    o.finalize_alt()
    o.scan_reference(genome)
    o.finalize_context()
    o.scan_sample_kmers(packed, counts)
    # the input does what it claims: some filter counter passes 2^16 (a pool k-mer whose middle k-mer hits bf, whose
    # context is not vetoed, drawn for more than 65535 in all), and some ref key count does too
    tot = np.bincount(idx, weights=counts.astype(np.float64), minlength=len(pool))
    heavy = [words[i] for i in np.flatnonzero(tot > 65535)]
    d = (ref_k - k) // 2
    hit = o.test_keys(0, [w[d:d + k] for w in heavy]) & (1 - o.test_keys(1, heavy))
    assert hit.sum() > 0, "no bf counter wraps past 2^16"
    ref_counts = o.get_counts(ks, [1] * len(ks))
    assert ref_counts.max() > 65535 and (ref_counts > 0).sum() > 100
    assert o.bf_counts().astype(np.int64).sum() > 0
    yield dict(k=k, ref_k=ref_k, bits=bits, genome=genome, nested=nested, freqs=freqs, ks=ks, fl=fl, packed=packed,
               counts=counts, o=o)
    o.close()


def _indexed(r):
    g = MalvaGpu(k=r["k"], ref_k=r["ref_k"], bf_bits=r["bits"])
    g.add_signatures(r["ks"], r["fl"])
    g.finalize_alt()
    g.scan_reference(r["genome"])
    g.finalize_context()
    return g


def _same_counts(g, o, ks):
    assert np.array_equal(g.bf_counts(), o.bf_counts()), "rank-indexed bf counters"
    for flag in (0, 1):
        fq = [flag] * len(ks)
        assert np.array_equal(g.get_counts(ks, fq), o.get_counts(ks, fq)), f"get_count is_ref={flag}"
    assert g.kmap_size() == o.kmap_size()


@pytest.mark.gpu
@pytest.mark.slow
@pytest.mark.parametrize("source", ["pageable", "pinned", "split"])
def test_sample_scan_across_staging_chunks(sample_run, source):
    """pageable: one call, three chunks and a tail on alternating streams; pinned: the same from mg_host_alloc
    memory; split: calls of 2^20+1, 2^22-1 and 2^22+1 k-mers (the stream a call starts on flips between calls),
    then the rest from device memory -- the counters of all three equal the oracle's after the whole input"""
    import torch

    r = sample_run
    packed, counts = r["packed"], r["counts"]
    g = _indexed(r)
    L = g._L
    pk, pc = C.c_void_p(), C.c_void_p()
    try:
        n0 = g.launch_count()
        if source == "pageable":
            g.scan_sample_kmers(packed, counts)
            assert g.launch_count() - n0 == 3 * SCAN_LAUNCHES, "three staging chunks, on alternating streams"
        elif source == "pinned":
            assert L.mg_host_alloc(C.byref(pk), packed.nbytes) == 0 and L.mg_host_alloc(C.byref(pc), counts.nbytes) == 0
            C.memmove(pk, packed.ctypes.data, packed.nbytes)
            C.memmove(pc, counts.ctypes.data, counts.nbytes)
            g.scan_sample_kmers_ptr(pk.value, pc.value, len(packed), device=False)
            g.sync()
            assert g.launch_count() - n0 == 3 * SCAN_LAUNCHES
        else:
            o = 0
            for m, chunks in ((STAGE_KMERS // 4 + 1, 1), (STAGE_KMERS - 1, 1), (STAGE_KMERS + 1, 2)):
                n0 = g.launch_count()
                g.scan_sample_kmers(packed[o:o + m], counts[o:o + m])
                assert g.launch_count() - n0 == chunks * SCAN_LAUNCHES
                o += m
            assert 0 < len(packed) - o < STAGE_KMERS
            tk = torch.from_numpy(packed[o:].view(np.uint8).copy()).cuda()
            tc = torch.from_numpy(counts[o:].view(np.int32).copy()).cuda()
            torch.cuda.synchronize()
            g.scan_sample_kmers_ptr(tk.data_ptr(), tc.data_ptr(), len(packed) - o, device=True)
            g.sync()
            del tk, tc
        _same_counts(g, r["o"], r["ks"])
    finally:
        g.close()
        for p in (pk, pc):
            if p.value:
                L.mg_host_free(p)


@pytest.mark.gpu
@pytest.mark.slow
def test_scan_on_both_streams_then_genotype_without_a_sync(sample_run):
    """the library on the caller's stream: a multi-chunk host scan (chunks on that stream and on the context's
    second one), then genotype_packed with no synchronisation in between -- it must wait for both streams"""
    import torch

    r = sample_run
    g = _indexed(r)
    side = torch.cuda.Stream()
    try:
        batch = SignatureBatch.from_nested(r["nested"], r["freqs"])
        pb = PackedSignatureBatch.from_batch(batch, r["k"])
        torch.cuda.synchronize()
        g.set_stream(side.cuda_stream)
        n0 = g.launch_count()
        g.scan_sample_kmers(r["packed"], r["counts"], sync=False)
        assert g.launch_count() - n0 == 3 * SCAN_LAUNCHES
        res = g.genotype_packed(pb, 0.001, 10 ** 9, False, want_lik=False)
        g.set_stream(0)
        torch.cuda.synchronize()
        cov, exp = r["o"].genotype(batch, 0.001, 10 ** 9, False)
        assert np.array_equal(res.cov, cov), "COVS"
        assert (cov > 0).sum() > 100
        assert res.status.tolist() == [e["status"] for e in exp]
        assert res.best_gt.tolist() == [e["best"] for e in exp]
        assert res.gq.tolist() == [e["gq"] for e in exp]
    finally:
        g.set_stream(0)
        g.close()


def kmc_image(packed: np.ndarray, counts: np.ndarray, k: int, p: int, csz: int):
    """what kmc.write_kmc_db writes, with numpy: (LUT of 4^p + 1 entries with its guard, the .kmc_suf records
    without the markers, the sort order).  Records sorted by value, suffix 2-bit big-endian, counter little-endian."""
    order = np.lexsort((packed["lo"], packed["hi"]))
    lo, hi = packed["lo"][order], packed["hi"][order]
    s2 = 2 * (k - p)
    if s2 >= 64:
        prefix = hi >> np.uint64(s2 - 64)
    else:
        prefix = (hi << np.uint64(64 - s2)) | (lo >> np.uint64(s2))
    sb = (k - p) // 4
    rec = np.empty((len(order), sb + csz), np.uint8)
    for i in range(sb):
        sh = 8 * (sb - 1 - i)
        rec[:, i] = ((lo >> np.uint64(sh)) if sh < 64 else (hi >> np.uint64(sh - 64))) & np.uint64(0xFF)
    rec[:, sb:] = counts[order].astype("<u8").view(np.uint8).reshape(-1, 8)[:, :csz]
    lut = np.zeros(4 ** p + 1, np.uint64)
    lut[1:] = np.cumsum(np.bincount(prefix.astype(np.int64), minlength=4 ** p))
    return lut, rec.reshape(-1), order


def _random_kmers(rng: np.random.Generator, n: int, k: int) -> np.ndarray:
    out = np.zeros(n, dtype=kmc.KMER_DTYPE)
    out["lo"] = rng.integers(0, 1 << 64, n, dtype=np.uint64, endpoint=False) if k >= 32 else \
        rng.integers(0, 1 << (2 * k), n, dtype=np.uint64)
    if k > 32:
        out["hi"] = rng.integers(0, 1 << (2 * (k - 32)), n, dtype=np.uint64)
    return out


@pytest.mark.parametrize("k,p,csz", [(43, 7, 1), (63, 3, 2), (21, 1, 4)])
def test_numpy_kmc_image_matches_write_kmc_db(tmp_path, k, p, csz):
    """kmc_image (the writer of the KMC scale test) is byte for byte kmc.write_kmc_db"""
    rng = np.random.default_rng(k)
    packed = np.unique(_random_kmers(rng, 3000, k))
    counts = rng.integers(1, 256 ** csz if csz < 4 else 1 << 32, len(packed), dtype=np.uint64).astype(np.uint32)
    prefix = str(tmp_path / "db")
    kmc.write_kmc_db(prefix, packed, counts, k, lut_prefix_len=p, counter_size=csz, min_count=1,
                     max_count=256 ** csz - 1)
    lut, rec, order = kmc_image(packed, counts, k, p, csz)
    suf = open(prefix + ".kmc_suf", "rb").read()
    assert suf == b"KMCS" + rec.tobytes() + b"KMCS"
    pre = open(prefix + ".kmc_pre", "rb").read()
    assert np.array_equal(np.frombuffer(pre, "<u8", count=4 ** p + 1, offset=4), lut)
    listed, lcounts, _ = kmc.read_kmc_db(prefix)
    assert np.array_equal(listed, packed[order]) and np.array_equal(lcounts, counts[order])
    assert len(np.unique(lut)) > 1


@pytest.mark.gpu
@pytest.mark.slow
@pytest.mark.parametrize("k,ref_k,p,csz", [
    (35, 43, 7, 1),      # 10-byte records
    (60, 63, 3, 2),      # 17-byte records: the staging buffers of a 16-byte packed scan grow on the same context
])
def test_kmc_records_across_staging_chunks(oracle_lib, k, ref_k, p, csz):
    """6.3 M KMC records (10^5 of them synth_sample k-mers, the rest random) scanned in two calls, the second
    starting at a record inside the first staging chunk that is not a multiple of 32 and covering two chunks:
    the device finds every record's prefix from first_record + its offset"""
    rng = random.Random(1000 + k)
    bits = 1 << 22
    genome = util.make_genome(rng, 40000)
    nested, _ = util.synth_signatures(rng, genome, k, 800)
    ks, fl = util.flatten(nested)
    _, pool, pool_counts = util.synth_sample(rng, genome, nested, k, ref_k, 40000)
    npr = np.random.default_rng(k)
    total = STAGE_KMERS + STAGE_KMERS // 2 + 12345
    packed = np.unique(np.concatenate([pool, _random_kmers(npr, total, ref_k)]))[:total]
    assert len(packed) == total
    top = 256 ** csz - 1
    counts = npr.integers(2, min(top, 5000) + 1, total, dtype=np.uint32)
    counts[::97] = 1                                   # below min_count: skipped
    lut, rec, order = kmc_image(packed, counts, ref_k, p, csz)
    keep = (counts[order] >= 2)
    listed, lcounts = packed[order][keep], counts[order][keep]
    db = dict(k=ref_k, lut=lut[:-1], lut_prefix_len=p, counter_size=csz, min_count=2, max_count=top)
    rb = (ref_k - p) // 4 + csz
    g, o = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bits), util.OracleRun(oracle_lib, k, ref_k, bits)
    try:
        for x in (g, o):
            x.add_signatures(ks, fl)
            x.finalize_alt()
            x.scan_reference(genome)
            x.finalize_context()
        if rb > 16:                                    # a packed scan first: 16-byte staging units
            g.scan_sample_kmers(pool, pool_counts)
            o.scan_sample_kmers(pool, pool_counts)
        o.scan_sample_kmers(listed, lcounts)
        g.kmc_open(db)
        first = STAGE_KMERS // 2 + 5
        assert first % 32 and total - first > STAGE_KMERS
        n0 = g.launch_count()
        g.scan_kmc_records(rec[:first * rb], 0, first)
        n1 = g.launch_count()
        g.scan_kmc_records(rec[first * rb:], first, total - first)
        assert (n1 - n0, g.launch_count() - n1) == (SCAN_LAUNCHES, 2 * SCAN_LAUNCHES)
        _same_counts(g, o, ks)
        assert o.bf_counts().astype(np.int64).sum() > 0 and (o.get_counts(ks, [1] * len(ks)) > 0).sum() > 20
    finally:
        g.close()
        o.close()


# ---------------------------------------------------------------------------------------------------------------
# C. filters past 2^32 bits
# ---------------------------------------------------------------------------------------------------------------
def _top_kmers(L, k: int, bf_bits: int, want: int = 3) -> list:
    """k-mers whose filter index lies in the top 256 of bf_bits (the last probe line where bf_bits is a multiple
    of 256): ~bf_bits/256 trials each, searched in the oracle on several threads"""
    threads = max(1, min(16, os.cpu_count() or 1))
    per = 1 << 24
    seed = b"A" * k
    found, base = [], 0
    while len(found) < want:
        assert base < 1 << 40, "hash search did not finish"

        def run(i, b=base):
            out = C.create_string_buffer((k + 1) * want)
            n = L.mo_find_kmers_at(seed, k, bf_bits, bf_bits - 256, b + i * per, per, out, want)
            return [out.raw[j * (k + 1):j * (k + 1) + k].decode() for j in range(n)]

        with ThreadPoolExecutor(threads) as ex:
            for got in ex.map(run, range(threads)):
                found += got
        base += threads * per
    return found


def _set_bits_device(g, which: int) -> np.ndarray:
    n = C.c_uint64(0)
    check(g._L.mg_export_set_bits(g._h, which, None, 0, C.byref(n)))
    out = np.zeros(max(n.value, 1), np.uint64)
    check(g._L.mg_export_set_bits(g._h, which, out.ctypes.data_as(util.u64p), n.value, C.byref(n)))
    return out[:n.value]


def _set_bits_oracle(o: util.OracleRun, which: int) -> np.ndarray:
    """set-bit indices from the oracle's words in place (no copy of a multi-GB bitmap)"""
    b = o.ctx if which == 1 else o.bf
    words = np.ctypeslib.as_array(o.L.mo_bf_words(b), shape=((o.bf_bits + 63) // 64,))
    nz = np.flatnonzero(words)
    rows, cols = np.nonzero(np.unpackbits(words[nz].view(np.uint8), bitorder="little").reshape(-1, 64))
    return nz[rows].astype(np.uint64) * np.uint64(64) + cols.astype(np.uint64)


@pytest.mark.gpu
@pytest.mark.slow
@pytest.mark.parametrize("bf_bits", [1 << 33, 3 << 33, (3 << 33) + 1], ids=["2^33", "3x2^33", "3x2^33+1"])
@pytest.mark.parametrize("k,ref_k", [(35, 43), (63, 64)])
def test_filter_past_2_32_bits(oracle_lib, k, ref_k, bf_bits):
    """-b 1 (mask path), -b 3 and an odd modulus (the 64-bit % path): the whole run -- index, reference pass, sample
    scan, genotypes -- equals the oracle's, with signatures in the last probe line of the filter"""
    rng = random.Random(bf_bits % 1000 + k)
    genome = util.make_genome(rng, 30000)
    nested, freqs = util.synth_signatures(rng, genome, k, 1000)
    top = _top_kmers(oracle_lib, k, bf_bits)
    for t in top:                                      # each its own variant, sampled like the other alt k-mers
        pos = rng.randrange(k, len(genome) - 2 * k)
        nested.append([[[genome[pos:pos + k]]], [[t]]])
        freqs.append([0.6, 0.4])
    ks, fl = util.flatten(nested)
    words, packed, counts = util.synth_sample(rng, genome, nested, k, ref_k, 30000, big_counts=True)
    g = MalvaGpu(k=k, ref_k=ref_k, bf_bits=bf_bits)
    o = util.OracleRun(oracle_lib, k, ref_k, bf_bits)
    try:
        for x in (g, o):
            x.add_signatures(ks, fl)
            x.finalize_alt()
            x.scan_reference(genome)
            x.finalize_context()
            x.scan_sample_kmers(packed, counts)
        for which, least in ((0, 1000), (1, 50)):
            got, want = _set_bits_device(g, which), _set_bits_oracle(o, which)
            assert np.array_equal(got, want), f"set bits of {'context_bf' if which else 'bf'}"
            assert len(want) > least and (want >= 1 << 32).sum() * 3 >= len(want), "bits below 2^32 only"
            if which == 0:
                assert want.max() >= bf_bits - 256, "no signature in the last probe line"
        assert (o.get_counts(top, [0] * len(top)) > 0).any(), "no sample k-mer reaches the last probe line"
        assert g.kmap_size() == o.kmap_size()
        assert np.array_equal(g.bf_counts(), o.bf_counts())
        extra = [util.rand_seq(rng, k) for _ in range(200)]
        q = ks + extra
        for flag in (0, 1):
            assert np.array_equal(g.get_counts(q, [flag] * len(q)), o.get_counts(q, [flag] * len(q)))
        for which in (0, 1, 2):
            assert np.array_equal(g.test_keys(which, q), o.test_keys(which, q)), f"test_key which={which}"
        ctx_q = [genome[p:p + ref_k] for p in range(0, len(genome) - ref_k, 53)]
        assert np.array_equal(g.test_keys(1, ctx_q), o.test_keys(1, ctx_q))
        batch = SignatureBatch.from_nested(nested, freqs)
        res = g.genotype_packed(PackedSignatureBatch.from_batch(batch, k), 0.001, 120, False, want_lik=False)
        cov, exp = o.genotype(batch, 0.001, 120, False)
        assert np.array_equal(res.cov, cov), "COVS"
        assert (cov > 0).sum() > 100
        assert res.status.tolist() == [e["status"] for e in exp]
        assert res.best_gt.tolist() == [e["best"] for e in exp]
        assert res.gq.tolist() == [e["gq"] for e in exp]
    finally:
        g.close()
        o.close()
