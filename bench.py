#!/usr/bin/env python
"""bench.py -- throughput of the MALVA genotyping hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload wg|wg3|small]
                    [--dump-outputs DIR]

Metric (BASELINE.json): sample k-mers/sec through the Bloom-filter + signature count (headline `value`),
with variants genotyped/sec reported beside it.  One "step" = one pass of the call-side hot path over one
batch of synthetic input: scan B sample 43-mers (K1) and genotype the proportional share V of variants
(K4 + K5), against index structures of whole-genome size (BASELINE config 3: 4 GiB filters, ~1e8 alt bits,
~1e8 ref keys).  `value` uses inputs resident in HBM; `e2e` goes through the host-buffer C-ABI calls with
the H2D / D2H copies inside the timed region.

Before anything is timed the run CHECKS ITSELF at the bench shape (2^35-bit filters): (a) after the first scan of
the full 1e8 + 1e8-key index, the counts of 1e5 random ref keys and 1e5 random alt keys are compared with an
independent recount of the batch (from how the batch was built, not through any hash); (b) a second context of
the same filter size holding the CPU sample's keys scans the CPU sample, and every key's count, every coverage,
GT and GQ is compared EXACTLY with the reference's own BF / KMAP / VB::genotype (oracle/_ref) fed the same input.
`"verified": true` in the line means both held; a mismatch exits non-zero.

N > 1 (torchrun, one process per GPU): replicate-and-reduce (SURVEY 8e): every rank holds the full index and scans
its own share of the sample stream; at genotyping time every rank looks the step's signature k-mers up in its own
partial counters and the LOOK-UP RESULTS (4 bytes per signature k-mer) are sum-reduced to rank 0 with NCCL, inside
the timed region and overlapped with the next scan; rank 0 genotypes from the sums (exact: get_count is linear in
the counters).  Weak scaling: B k-mers per rank per step.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K, REF_K = 35, 43
SEED = 20261018 + 3  # SURVEY 8d: seed = 20261018 + cfg
ERR, MAX_COV = 0.001, 200

WORKLOADS = {
    # BASELINE.json configs[3]: synthetic whole-genome index structures on one GPU (4 GiB filters)
    "wg": dict(bf_bits=1 << 35, n_alt=100_000_000, n_ref=100_000_000, ref_bases=250_000_000, batch=1 << 27,
               variants=2_850_000, name="synthetic whole-genome 30x (cfg[3]): 2^35-bit filters, 1e8 alt + 1e8 ref "
                                        "signature k-mers; step = 2^27 sample 43-mers + 2.85e6 variants"),
    # the upper end of SURVEY's 1-3e8 signatures per kind (sensitivity line, profiles/)
    "wg3": dict(bf_bits=1 << 35, n_alt=300_000_000, n_ref=300_000_000, ref_bases=250_000_000, batch=1 << 27,
                variants=2_850_000, name="synthetic whole-genome 30x, dense end: 2^35-bit filters, 3e8 alt + 3e8 ref "
                                         "signature k-mers; step = 2^27 sample 43-mers + 2.85e6 variants"),
    # the whole-genome load factors on probe lines that fit L2 (64 MB; run with MG_OCC_LOG2_BITS=21): the scan with
    # its random DRAM traffic taken away = the arithmetic floor of K1 (profiles/round2_k1.md; not a bench line)
    "l2": dict(bf_bits=1 << 27, n_alt=390_625, n_ref=390_625, ref_bases=1_000_000, batch=1 << 27, variants=90_000,
               name="whole-genome load factors, L2-resident probe lines (not a bench line)"),
    # small twin for quick checks (not a bench line)
    "small": dict(bf_bits=1 << 30, n_alt=2_000_000, n_ref=2_000_000, ref_bases=5_000_000, batch=1 << 22,
                  variants=90_000, name="small twin (not a bench line)"),
}
HIT_REF, HIT_ALT = 0.03, 0.007  # SURVEY 8a: expected per-k-mer hit rates of ref_bf / bf
ALGO_BYTES_PER_KMER = 84         # SURVEY 8d: 20 B streamed + 2 random 32 B sectors
ALGO_BYTES_PER_REF_BASE = 33     # SURVEY 8d: 1 B streamed + one random 32 B sector
ALGO_BYTES_PER_SIG_KMER = 36     # SURVEY 8d: 4 B index + one random 32 B sector


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def config_of(wl, world):
    """identical in both arms (the driver compares them)"""
    return {"workload": wl["name"], "k": K, "ref_k": REF_K, "bf_bits": wl["bf_bits"],
            "kmers_per_step_per_gpu": wl["batch"], "variants_per_step_per_gpu": wl["variants"],
            "hit_rates": {"ref_bf": HIT_REF, "bf": HIT_ALT},
            "l2_policy": "inputs larger than L2: 2.7 GB streamed per step, two batches alternate, probes "
                         "spread over 17 GB of probe lines",
            "parallelism": f"replicate-and-reduce x{world}" if world > 1 else "1 GPU"}


# ------------------------------------------------------------------------------------------------
# synthetic data (torch is used for device memory and random numbers only)
# ------------------------------------------------------------------------------------------------
def rand_kmers(torch, n, k, gen, dev):
    """n random k-mers as int64 [n, 2] = (lo, hi) two's-complement images of the u64 words."""
    lo = (torch.randint(0, 1 << 32, (n,), dtype=torch.int64, generator=gen, device=dev) << 32) | \
        torch.randint(0, 1 << 32, (n,), dtype=torch.int64, generator=gen, device=dev)
    bits_hi = 2 * k - 64
    if bits_hi > 0:
        hi = torch.randint(0, 1 << bits_hi, (n,), dtype=torch.int64, generator=gen, device=dev)
    else:
        hi = torch.zeros(n, dtype=torch.int64, device=dev)
        lo = lo & ((1 << (2 * k)) - 1)
    return torch.stack([lo, hi], dim=1).contiguous()


def embed(torch, sig, gen, dev):
    """35-mer words -> 43-mer words with 4 random flanking bases on each side."""
    n = sig.shape[0]
    lo, hi = sig[:, 0], sig[:, 1]
    fl = torch.randint(0, 256, (n, 2), dtype=torch.int64, generator=gen, device=dev)
    nlo = (lo << 8) | fl[:, 1]
    nhi = (hi << 8) | ((lo >> 56) & 0xFF) | (fl[:, 0] << 14)
    return torch.stack([nlo, nhi], dim=1)


def make_sample_batch(torch, n, alt, ref, gen, dev, keep_plan=False):
    x = rand_kmers(torch, n, REF_K, gen, dev)
    n_ref, n_alt = int(n * HIT_REF), int(n * HIT_ALT)
    pos = torch.randperm(n, generator=gen, device=dev)[: n_ref + n_alt]
    ri = torch.randint(0, ref.shape[0], (n_ref,), generator=gen, device=dev)
    ai = torch.randint(0, alt.shape[0], (n_alt,), generator=gen, device=dev)
    x[pos[:n_ref]] = embed(torch, ref[ri], gen, dev)
    x[pos[n_ref:]] = embed(torch, alt[ai], gen, dev)
    counts = torch.randint(2, 256, (n,), dtype=torch.int32, generator=gen, device=dev)
    plan = (pos, ri, ai) if keep_plan else None
    return x.contiguous(), counts, plan


def make_kmc_records(torch, x, counts, p=7):
    """A batch of 43-mer words -> (sorted raw .kmc_suf records uint8 [n*10], prefix LUT int64 [4^p]) as KMC lays them out."""
    lo, hi = x[:, 0], x[:, 1]
    o1 = torch.argsort(lo ^ (-(1 << 63)), stable=True)          # unsigned order of the low word
    o2 = torch.argsort(hi[o1], stable=True)
    order = o1[o2]
    lo, hi, c = lo[order], hi[order], counts[order]
    suf_syms = REF_K - p                                         # 36 symbols = 72 bits = 9 bytes
    prefix = hi >> (2 * suf_syms - 64)
    lut = torch.zeros(4 ** p, dtype=torch.int64, device=x.device)
    lut[1:] = torch.cumsum(torch.bincount(prefix, minlength=4 ** p), 0)[:-1]
    rec = torch.empty((x.shape[0], 10), dtype=torch.uint8, device=x.device)
    rec[:, 0] = (hi & 0xFF).to(torch.uint8)
    for j in range(8):
        rec[:, 1 + j] = ((lo >> (56 - 8 * j)) & 0xFF).to(torch.uint8)
    rec[:, 9] = (c & 0xFF).to(torch.uint8)
    return rec.reshape(-1), lut


def kmers_to_ascii(torch, sig, k):
    """[n,2] int64 words -> uint8 [n,k] ASCII."""
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device=sig.device)
    cols = []
    for j in range(k):
        sh = 2 * (k - 1 - j)
        code = ((sig[:, 1] >> (sh - 64)) if sh >= 64 else (sig[:, 0] >> sh)) & 3
        cols.append(lut[code])
    return torch.stack(cols, dim=1).contiguous()


def variant_csr(nv, seed):
    """CSR skeleton of nv variants: 97% biallelic, 3% with 2-3 ALTs; one signature per allele, 1 k-mer (85%) or 2-3."""
    g = np.random.default_rng(seed)
    n_all = np.where(g.random(nv) < 0.97, 2, g.integers(3, 5, nv)).astype(np.int64)
    vao = np.zeros(nv + 1, np.uint32)
    vao[1:] = np.cumsum(n_all)
    na = int(vao[-1])
    aso = np.arange(na + 1, dtype=np.uint32)              # one signature per allele slot
    n_k = np.where(g.random(na) < 0.85, 1, g.integers(2, 4, na)).astype(np.int64)
    sko = np.zeros(na + 1, np.uint32)
    sko[1:] = np.cumsum(n_k)
    nk = int(sko[-1])
    is_ref_allele = np.zeros(na, bool)
    is_ref_allele[vao[:-1].astype(np.int64)] = True
    kmer_is_ref = np.repeat(is_ref_allele, n_k)
    af = (g.random(na) * 0.3).astype(np.float32)
    freq = af.copy()
    starts = vao[:-1].astype(np.int64)
    sums = np.add.reduceat(af.astype(np.float64), starts) - af[starts]
    freq[starts] = np.maximum(1.0 - sums, 0).astype(np.float32)
    lik_slots = int((n_all * (n_all + 1) // 2).sum())
    return dict(vao=vao, aso=aso, sko=sko, freq=freq, kmer_is_ref=kmer_is_ref, dims=(nv, na, na, nk), lik_slots=lik_slots,
                miss=g.random(nk) < 0.3)        # k-mers the sample does not support


def make_variant_batch(torch, nv, alt, ref, gen, dev):
    """the packed batch form the C++ host sends (mg_packed_batch): {lo, hi} words, hi bit 62 = ref-allele k-mer"""
    vb = variant_csr(nv, SEED + 7)
    nk = vb["dims"][3]
    t_is_ref = torch.from_numpy(vb["kmer_is_ref"]).to(dev)
    ri = torch.randint(0, ref.shape[0], (nk,), generator=gen, device=dev)
    ai = torch.randint(0, alt.shape[0], (nk,), generator=gen, device=dev)
    words = torch.where(t_is_ref[:, None], ref[ri], alt[ai])
    miss = torch.from_numpy(vb["miss"]).to(dev)
    words = torch.where(miss[:, None], rand_kmers(torch, nk, K, gen, dev), words)
    words[:, 1] |= t_is_ref.to(torch.int64) << 62
    vb["kmers"] = words.contiguous()
    return vb


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi SM clock + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.idx), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for l in self.proc.stdout:
            self.lines.append((time.time(), l.strip()))

    def mark(self):
        """start of the timed region: earlier samples are dropped"""
        self.t_mark = time.time()

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        t_mark = getattr(self, "t_mark", 0.0)
        for ts, l in self.lines:
            if ts < t_mark:
                continue
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "samples": len(sm), "reasons": sorted(reasons)}


class DevArray:
    """A library-owned device buffer seen as a torch tensor (for the NCCL reduce)."""

    def __init__(self, ptr, n, typestr="<i4"):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


def measured_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(p["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (driver-measured copy bandwidth)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


def profile_json(name):
    try:
        return json.load(open(os.path.join(ROOT, "profiles", name)))
    except Exception:
        return {}


DUMP_MAX_VARIANTS = 1 << 19   # ~40 MB of float64 with their alleles: under 64 MB at every workload


def dump_outputs(out_dir, d, vao):
    """What the last timed step returned to its caller (per-allele coverage, per-variant n_gts / status / GT / GQ) as
    float64 .npy files, so that two builds can be compared output for output.  Above DUMP_MAX_VARIANTS variants a
    fixed, seeded sample of them is written (with all their alleles); variant_index / allele_index name the rows."""
    nv = len(vao) - 1
    if nv > DUMP_MAX_VARIANTS:
        vi = np.sort(np.random.default_rng(SEED + 1000).choice(nv, DUMP_MAX_VARIANTS, replace=False))
    else:
        vi = np.arange(nv)
    lo = vao[vi].astype(np.int64)
    n = vao[vi + 1].astype(np.int64) - lo
    ai = np.arange(int(n.sum())) - np.repeat(np.cumsum(n) - n, n) + np.repeat(lo, n)
    out = {"variant_index": vi, "allele_index": ai, "cov": d["cov"].cpu().numpy()[ai]}
    for name in ("n_gts", "status", "best_gt", "gq"):
        out[name] = d[name].cpu().numpy()[vi]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))
    log(f"outputs of the last timed step ({len(vi)} of {nv} variants, {len(ai)} alleles) written to {out_dir}")


def bind_to_gpu_numa(local_rank):
    """Pin this process to the CPUs of the NUMA node its GPU hangs off, BEFORE any pinned buffer is allocated: the
    buffers are then node-local and eight ranks' H2D streams do not all cross the socket interconnect."""
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)],
                           capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if not q:
            return {"bound": False, "why": "no bus id"}
        bus = q[-12:] if len(q) >= 12 else q           # 00000000:1B:00.0 -> 0000:1b:00.0
        base = f"/sys/bus/pci/devices/{bus}"
        node = int(open(base + "/numa_node").read().strip())
        cpus = open(base + "/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            if "-" in part:
                a, b = part.split("-")
                ids.update(range(int(a), int(b) + 1))
            elif part:
                ids.add(int(part))
        avail = os.sched_getaffinity(0)
        ids &= avail
        if node < 0 or not ids or ids == avail:
            return {"bound": False, "numa_node": node, "why": "single node or no locality information"}
        os.sched_setaffinity(0, ids)
        return {"bound": True, "numa_node": node, "cpus": len(ids)}
    except Exception as e:  # noqa: BLE001
        return {"bound": False, "why": str(e)[:80]}


# ------------------------------------------------------------------------------------------------
# CPU side: the reference's own BF + KMAP + VB classes (oracle/_ref), or the C restatement when absent.
# Used as the checker of the self-test, as `cpu_baseline*` and as the `--impl reference` arm.
# ------------------------------------------------------------------------------------------------
u64p, u32p, u8p, i32p, f32p = (C.POINTER(t) for t in (C.c_uint64, C.c_uint32, C.c_uint8, C.c_int32, C.c_float))


def cpu_inputs(n_sig, n_s):
    """Bounded CPU-side sample of the workload: n_sig alt + n_sig ref signature k-mers, n_s sample k-mers built
    like the device batches (same hit rates)."""
    g = np.random.default_rng(SEED)

    def rk(n, k):
        lo = g.integers(0, 1 << 63, n, dtype=np.uint64) * 2 + g.integers(0, 2, n, dtype=np.uint64)
        hi = g.integers(0, 1 << (2 * k - 64), n, dtype=np.uint64)
        return np.stack([lo, hi], axis=1)

    alt, ref = rk(n_sig, K), rk(n_sig, K)
    smp = rk(n_s, REF_K)

    def emb(sig):
        fl = g.integers(0, 256, (len(sig), 2), dtype=np.uint64)
        lo = (sig[:, 0] << np.uint64(8)) | fl[:, 1]
        hi = (sig[:, 1] << np.uint64(8)) | (sig[:, 0] >> np.uint64(56)) | (fl[:, 0] << np.uint64(14))
        return np.stack([lo, hi], axis=1)

    n_r, n_a = int(n_s * HIT_REF), int(n_s * HIT_ALT)
    pos = g.permutation(n_s)[: n_r + n_a]
    smp[pos[:n_r]] = emb(ref[g.integers(0, n_sig, n_r)])
    smp[pos[n_r:]] = emb(alt[g.integers(0, n_sig, n_a)])
    counts = g.integers(2, 256, n_s).astype(np.uint32)
    # a variant batch over the same keys (packed form)
    nv = 200_000
    vb = variant_csr(nv, SEED + 11)
    nk = vb["dims"][3]
    words = np.where(vb["kmer_is_ref"][:, None], ref[g.integers(0, n_sig, nk)], alt[g.integers(0, n_sig, nk)])
    words = np.where(vb["miss"][:, None], rk(nk, K), words)
    words[:, 1] |= vb["kmer_is_ref"].astype(np.uint64) << np.uint64(62)
    vb["kmers"] = np.ascontiguousarray(words)
    return alt, ref, smp, counts, vb


class CpuReference:
    """bf / context_bf / ref_bf as the reference's own objects (kind "reference") or the C restatement ("port")"""

    def __init__(self, bf_bits, alt_np, ref_np):
        from oracle import pyoracle
        self.have_ref = pyoracle.have_ref()
        flags = np.concatenate([np.zeros(len(alt_np), np.uint8), np.ones(len(ref_np), np.uint8)])
        keys = np.ascontiguousarray(np.concatenate([alt_np, ref_np]))
        self.keys, self.flags = keys, flags
        if self.have_ref:
            L, self.kind = pyoracle.ref(), "reference"
            self.L = L
            self.bf, self.ctx, self.km = L.ref_bf_new(bf_bits), L.ref_bf_new(bf_bits), L.ref_kmap_new()
            L.ref_add_packed(self.bf, self.km, keys.ctypes.data_as(u64p), flags.ctypes.data_as(u8p), len(flags), K)
            L.ref_bf_switch_mode(self.bf)
            L.ref_bf_switch_mode(self.ctx)
        else:
            L, self.kind = pyoracle.oracle(), "port"
            self.L = L
            self.bf, self.ctx, self.km = L.mo_bf_new(bf_bits), L.mo_bf_new(bf_bits), L.mo_kmap_new()
            from malva_b200.kmc import packed_to_strings, KMER_DTYPE
            for arr, is_ref in ((alt_np, 0), (ref_np, 1)):
                for s in packed_to_strings(arr.view(KMER_DTYPE).reshape(-1), K):
                    (L.mo_kmap_add_key(self.km, s.encode()) if is_ref else L.mo_bf_add_key(self.bf, s.encode()))
            L.mo_bf_switch_mode(self.bf)
            L.mo_bf_switch_mode(self.ctx)

    def scan(self, a, c):
        """main.cpp:487-500 over packed k-mers; returns seconds"""
        a, c = np.ascontiguousarray(a), np.ascontiguousarray(c)
        fn = self.L.ref_scan_packed if self.have_ref else self.L.mo_scan_packed
        t0 = time.perf_counter()
        fn(self.bf, self.ctx, self.km, a.ctypes.data_as(u64p), c.ctypes.data_as(u32p), len(c), K, REF_K)
        return time.perf_counter() - t0

    def get_counts(self):
        """BF::get_count / KMAP::get_count of every key (reference build only)"""
        out = np.zeros(len(self.flags), np.int32)
        self.L.ref_get_counts_packed(self.bf, self.km, self.keys.ctypes.data_as(u64p), self.flags.ctypes.data_as(u8p),
                                     len(self.flags), K, out.ctypes.data_as(i32p))
        return out

    def genotype(self, vb, n):
        """set_coverages + VB::genotype + arg-max over the first n variants; returns (seconds, cov, best, gq)"""
        na = int(vb["vao"][n])
        cov, best, gq = np.zeros(na, np.uint32), np.zeros(n, np.int32), np.zeros(n, np.int32)
        t0 = time.perf_counter()
        self.L.ref_genotype_batch(self.bf, self.km, n, vb["vao"].ctypes.data_as(u32p), vb["aso"].ctypes.data_as(u32p),
                                  vb["sko"].ctypes.data_as(u32p), vb["kmers"].ctypes.data_as(u64p),
                                  vb["freq"].ctypes.data_as(f32p), K, C.c_float(ERR), MAX_COV, 0,
                                  cov.ctypes.data_as(u32p), best.ctypes.data_as(i32p), gq.ctypes.data_as(i32p))
        return time.perf_counter() - t0, cov, best, gq

    def reference_pass(self, n_bases):
        """main.cpp:382-402 over n_bases random bases; returns seconds"""
        seq = np.random.default_rng(SEED + 5).integers(0, 4, n_bases).astype(np.uint8)
        s = bytes(np.array([65, 67, 71, 84], np.uint8)[seq])
        t0 = time.perf_counter()
        if self.have_ref:
            self.L.ref_reference_pass(self.bf, self.ctx, s, K, REF_K)
        else:
            self.L.mo_reference_pass(self.bf, self.ctx, s, len(s), K, REF_K)
        return time.perf_counter() - t0

    def close(self):
        if self.have_ref:
            self.L.ref_bf_free(self.bf), self.L.ref_bf_free(self.ctx), self.L.ref_kmap_free(self.km)
        else:
            self.L.mo_bf_free(self.bf), self.L.mo_bf_free(self.ctx), self.L.mo_kmap_free(self.km)


def cpu_legs(wl, n_sig, n_scan, gpu_device=None):
    """The CPU baselines (k-mers/s, variants/s, reference bases/s on one host core) over a bounded sample, and -- when
    gpu_device is given -- the exact check of a GPU context of the same filter size against them."""
    alt, ref, smp, counts, vb = cpu_inputs(n_sig, n_scan)
    t0 = time.perf_counter()
    cpu = CpuReference(wl["bf_bits"], alt, ref)
    t_build = time.perf_counter() - t0
    t_scan = cpu.scan(smp, counts)
    n_geno = 50_000
    out = {"kind": cpu.kind, "cores": 1, "host_cores_available": os.cpu_count(),
           "kmers_per_sec": n_scan / t_scan, "n_scan": n_scan, "n_sig": n_sig, "build_s": t_build}
    check = None
    if cpu.have_ref:
        t_geno, r_cov, r_best, r_gq = cpu.genotype(vb, n_geno)
        out["variants_per_sec"] = n_geno / t_geno
        out["n_genotyped"] = n_geno
        n_bases = 1_000_000
        out["ref_bases_per_sec"] = n_bases / cpu.reference_pass(n_bases)
        if gpu_device is not None:
            from malva_b200 import MalvaGpu
            from malva_b200.api import PackedSignatureBatch
            from malva_b200.kmc import KMER_DTYPE, packed_to_strings
            expected = cpu.get_counts()
            g = MalvaGpu(k=K, ref_k=REF_K, bf_bits=wl["bf_bits"], device=gpu_device)
            try:
                g.add_signatures_packed(cpu.keys.reshape(-1).view(KMER_DTYPE), cpu.flags)
                g.finalize_alt()
                g.finalize_context()
                g.scan_sample_kmers(np.ascontiguousarray(smp).reshape(-1).view(KMER_DTYPE), counts)
                # every key's count through the reference-facing string interface, in chunks
                got = np.zeros(len(cpu.flags), np.int32)
                step = 500_000
                for o in range(0, len(got), step):
                    ks = packed_to_strings(cpu.keys[o:o + step].reshape(-1).view(KMER_DTYPE), K)
                    got[o:o + step] = g.get_counts(ks, cpu.flags[o:o + step])
                nk = int(vb["sko"][int(vb["aso"][int(vb["vao"][n_geno])])])
                pb = PackedSignatureBatch(vb["vao"][:n_geno + 1], vb["aso"][:int(vb["vao"][n_geno]) + 1],
                                          vb["sko"][:int(vb["aso"][int(vb["vao"][n_geno])]) + 1],
                                          vb["kmers"][:nk].reshape(-1).view(KMER_DTYPE), vb["freq"], np.zeros(1, np.uint64),
                                          b"", np.zeros(0, np.uint32))
                r = g.genotype_packed(pb, ERR, MAX_COV, False, want_lik=False)
                check = {"keys_checked": int(len(got)), "key_counts_equal": bool(np.array_equal(got, expected)),
                         "nonzero_counts": int((expected != 0).sum()),
                         "variants_checked": n_geno, "cov_equal": bool(np.array_equal(r.cov, r_cov)),
                         "gt_equal": bool(np.array_equal(r.best_gt, r_best)), "gq_equal": bool(np.array_equal(r.gq, r_gq)),
                         "covered_alleles": int((r_cov > 0).sum())}
            finally:
                g.close()
    cpu.close()
    return out, check


def run_reference_arm(args, wl, rank, world):
    if rank != 0:
        return
    n_sig = 20_000_000 if args.workload != "small" else 1_000_000
    per_step = 400_000
    n_scan = per_step * (args.steps + args.warmup)
    alt, ref, smp, counts, vb = cpu_inputs(n_sig, min(n_scan, 4_000_000))
    reps = -(-n_scan // len(counts))
    smp, counts = np.tile(smp, (reps, 1)), np.tile(counts, reps)
    t0 = time.perf_counter()
    cpu = CpuReference(wl["bf_bits"], alt, ref)
    t_build = time.perf_counter() - t0
    t_total = 0.0
    for s in range(args.warmup + args.steps):
        t = cpu.scan(smp[s * per_step:(s + 1) * per_step], counts[s * per_step:(s + 1) * per_step])
        if s >= args.warmup:
            t_total += t
    ms = t_total / args.steps * 1e3
    rate = per_step / (ms * 1e-3)
    extra = {}
    if cpu.have_ref:
        t_geno, _, _, _ = cpu.genotype(vb, 50_000)
        extra["variants_per_sec"] = 50_000 / t_geno
        extra["ref_bases_per_sec"] = 1_000_000 / cpu.reference_pass(1_000_000)
    cpu.close()
    sample = (f"{per_step} sample 43-mers per step (a bounded sample of the {wl['batch']} of the workload) against "
              f"2^{int(np.log2(wl['bf_bits']))}-bit filters holding {n_sig} alt bits + {n_sig} ref keys (the workload has "
              f"{wl['n_alt']} + {wl['n_ref']}: the reference's unordered_map<string,int> needs ~100 B per key; fewer keys "
              "flatter the CPU); the reference's own BF/KMAP classes, single-threaded like the reference (no threads in "
              f"malva-geno, KMC run with -t1); index build {t_build:.0f} s untimed")
    line = {"impl": "reference", "metric": "sample_kmers_per_sec", "value": rate, "unit": "k-mers/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": config_of(wl, world),
            "cpu_baseline": {"value": rate, "unit": "k-mers/s", "cores": 1, "kind": cpu.kind, "sample": sample,
                             "host_cores_available": os.cpu_count(), **extra},
            "e2e": {"value": rate, "unit": "k-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args, wl, rank, local_rank, world):
    numa = bind_to_gpu_numa(local_rank) if not args.no_numa else {"bound": False, "why": "--no-numa"}
    import torch
    import torch.distributed as dist

    from malva_b200 import MalvaGpu
    from malva_b200.api import diag_bandwidth
    from malva_b200.kmc import KMER_DTYPE

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the MALVA hot path has no CPU fallback")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED)           # identical index on every rank (replicate-and-reduce)
    t_setup = time.time()
    g = MalvaGpu(k=K, ref_k=REF_K, bf_bits=wl["bf_bits"], device=local_rank)
    alt = rand_kmers(torch, wl["n_alt"], K, gen, dev)
    ref = rand_kmers(torch, wl["n_ref"], K, gen, dev)
    chunk = 1 << 24
    for arr, flag in ((alt, 0), (ref, 1)):
        for o in range(0, arr.shape[0], chunk):
            h = arr[o:o + chunk].cpu().numpy().view(np.uint64).reshape(-1).view(KMER_DTYPE)
            g.add_signatures_packed(h, np.full(len(h), flag, np.uint8))
    g.finalize_alt()
    # reference rolling pass (K2) over a synthetic contig that carries some alt signatures
    rb = torch.randint(0, 4, (wl["ref_bases"],), dtype=torch.uint8, generator=gen, device=dev)
    lut = torch.tensor([65, 67, 71, 84], dtype=torch.uint8, device=dev)
    ref_seq = lut[rb.long()] if wl["ref_bases"] <= 50_000_000 else torch.cat(
        [lut[rb[i:i + 50_000_000].long()] for i in range(0, wl["ref_bases"], 50_000_000)])
    del rb
    n_plant = min(200_000, wl["ref_bases"] // 1000)
    plant = kmers_to_ascii(torch, alt[:n_plant], K)
    # one plant per stride, jittered: the planted windows never overlap, so the scatter below is deterministic
    # and every rank builds the same context filter
    stride = (wl["ref_bases"] - 200) // n_plant
    ppos = 100 + torch.arange(n_plant, device=dev) * stride + \
        torch.randint(0, max(1, stride - K), (n_plant,), generator=gen, device=dev)
    ref_seq[(ppos[:, None] + torch.arange(K, device=dev)[None, :]).reshape(-1)] = plant.reshape(-1)
    ref_pinned = ref_seq.cpu().pin_memory()
    ref_bytes = ref_pinned.numpy().tobytes()   # the same contig in pageable memory
    del ref_seq
    g.scan_reference(ref_bytes)    # cold call (allocations, first touch)
    g.event_record(0)
    g.scan_reference(ref_bytes)    # idempotent (bits are only ever set): the warm calls are the ones timed
    g.event_record(1)
    g.scan_reference_ptr(ref_pinned.data_ptr(), wl["ref_bases"])
    g.event_record(6)
    refpass_pageable_ms = g.event_elapsed_ms(0, 1)   # pageable contig: threaded staging copies + chunked H2D + kernels
    refpass_pinned_ms = g.event_elapsed_ms(1, 6)     # pinned contig: chunked H2D overlapped with the kernels
    refpass_kernel_ms = g.refpass_kernel_ms()        # the rolling-pass kernels alone (sum over chunks)
    del ref_bytes, ref_pinned
    g.finalize_context()
    pop_alt, pop_ctx, n_keys = g.popcount(0), g.popcount(1), g.kmap_size()
    stats = g.index_stats()
    # sample batches, device resident (2 batches rotate so that no step re-reads the previous step's lines)
    # every rank scans its own share of the stream (--verify: the same share, so that the reduced counters must be
    # exactly world x one rank's)
    gen.manual_seed(SEED + 100 + (0 if args.verify else rank))
    B = wl["batch"]
    b0 = make_sample_batch(torch, B, alt, ref, gen, dev, keep_plan=True)
    batches = [b0[:2], make_sample_batch(torch, B, alt, ref, gen, dev)[:2]]
    vb = make_variant_batch(torch, wl["variants"], alt, ref, gen, dev)
    nv, na, ns, nk = vb["dims"]
    d = {k2: torch.from_numpy(vb[k1]).to(dev) for k1, k2 in (("vao", "var_allele_off"), ("aso", "allele_sig_off"),
                                                              ("sko", "sig_kmer_off"), ("freq", "freq"))}
    d["kmers"] = vb["kmers"]
    d["cov"] = torch.zeros(na, dtype=torch.int32, device=dev)
    for nme in ("n_gts", "status", "best_gt", "gq"):
        d[nme] = torch.zeros(nv, dtype=torch.int32, device=dev)
    ptrs = {k2: t.data_ptr() for k2, t in d.items()}
    pdims = (nv, na, ns, nk, 0, 0, vb["lik_slots"])
    torch.cuda.synchronize()
    log(f"[rank {rank}] setup {time.time() - t_setup:.1f}s: bf ones {pop_alt}, context ones {pop_ctx}, ref keys {n_keys} "
        f"({stats['overflow_keys']} in the overflow table), "
        f"K2 reference pass {wl['ref_bases'] / refpass_kernel_ms / 1e6:.1f} Gbases/s (kernels), "
        f"{wl['ref_bases'] / refpass_pinned_ms / 1e6:.1f} from pinned, {wl['ref_bases'] / refpass_pageable_ms / 1e6:.1f} "
        f"from pageable memory; numa {numa}")

    # ---- self-check (a): first scan of the full index against an independent recount of the batch ----
    verify = {}
    if not args.no_verify:
        kk, cc = batches[0]
        g.scan_sample_kmers_ptr(kk.data_ptr(), cc.data_ptr(), B, device=True)
        g.sync()
        pos, ri, ai = b0[2]
        n_r = ri.shape[0]
        exp_ref = torch.zeros(ref.shape[0], dtype=torch.int64, device=dev).index_add_(0, ri, cc[pos[:n_r]].long())
        exp_alt = torch.zeros(alt.shape[0], dtype=torch.int64, device=dev).index_add_(0, ai, cc[pos[n_r:]].long())
        sub = torch.randint(0, min(ref.shape[0], alt.shape[0]), (100_000,), generator=gen, device=dev)
        # (half of the subset are keys the batch did hit)
        sub[:50_000] = ri[torch.randint(0, n_r, (50_000,), generator=gen, device=dev)]
        ks_ref = [bytes(r) for r in kmers_to_ascii(torch, ref[sub], K).cpu().numpy()]
        got_ref = torch.from_numpy(g.get_counts(ks_ref, np.ones(len(ks_ref), np.uint8)).astype(np.int64)).to(dev)
        sub_a = sub.clone()
        sub_a[:50_000] = ai[torch.randint(0, ai.shape[0], (50_000,), generator=gen, device=dev)]
        ks_alt = [bytes(r) for r in kmers_to_ascii(torch, alt[sub_a], K).cpu().numpy()]
        got_alt = torch.from_numpy(g.get_counts(ks_alt, np.zeros(len(ks_alt), np.uint8)).astype(np.int64)).to(dev)
        # ref_bf is an exact map: equality.  bf counters are per BIT (colliding keys and false-positive sample
        # k-mers share them, bloom_filter.hpp:100-125): above the recount for the ~0.4 % of bits the filter's own
        # collision rate predicts; and a sample k-mer whose 43-mer hits a set bit of context_bf is not counted
        # (main.cpp:495-499; 9e5 set bits in 2^35: a few dozen k-mers per batch), so a handful may lie below
        ref_ok = bool(torch.equal(got_ref, exp_ref[sub]))
        ea = exp_alt[sub_a] & 0xFFFF
        alt_eq_frac = float((got_alt == ea).double().mean())
        alt_below = float((got_alt < ea).double().mean()) if int(exp_alt.max()) < 65536 else 0.0
        verify["recount_full_index"] = {"ref_keys_checked": 100_000, "ref_counts_equal": ref_ok,
                                        "ref_nonzero": int((exp_ref[sub] != 0).sum()),
                                        "alt_keys_checked": 100_000, "alt_counts_equal_fraction": alt_eq_frac,
                                        "alt_counts_below_recount_fraction": alt_below,
                                        "alt_nonzero": int((ea != 0).sum())}
        del exp_ref, exp_alt, got_ref, got_alt
        log(f"[rank {rank}] self-check (a) {verify['recount_full_index']}")
        if not (ref_ok and alt_below < 1e-3 and alt_eq_frac > 0.97):
            print(json.dumps({"verified": False, **verify}), flush=True)
            raise SystemExit(3)
    del alt, ref

    counters = []

    def reduce_counters():
        """the other exact scheme (malva-geno call --devices, --verify): gather the counters (every rank) -> ncclReduce
        of the dense arrays -> scatter into rank 0's probe lines"""
        nonlocal counters
        bufs = g.counter_buffers(gather=True)
        if not counters:
            counters = [torch.as_tensor(DevArray(p, n), device=dev) for p, n in bufs if n]
        for t in counters:
            dist.reduce(t, dst=0)
        torch.cuda.synchronize()
        if rank == 0:
            g.counters_scatter()

    def barrier():
        g.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    # N > 1: the library works on torch's stream, so that its kernels and the NCCL reduces order without host syncs
    w_bufs = [torch.zeros(max(nk, 1), dtype=torch.int32, device=dev) for _ in range(2)] if world > 1 else None
    if world > 1:
        torch.cuda.synchronize()
        side = torch.cuda.Stream(device=dev)           # (torch's default stream is handle 0 = "restore" for mg_set_stream)
        torch.cuda.set_stream(side)
        g.set_stream(side.cuda_stream)

    def finish(p):
        """the reduce of a step's look-up results has landed: rank 0 genotypes from the sums"""
        p[0].wait()                                    # (the stream waits, not the host)
        if rank == 0:
            g.genotype_weights_device(ptrs, pdims, p[1].data_ptr(), ERR, MAX_COV, False)

    def run_steps(n_steps, timed):
        pending = None
        for i in range(n_steps):
            if timed:
                g.event_record(10 + 2 * (i % 8))
            kk, cc = batches[i & 1]
            g.scan_sample_kmers_ptr(kk.data_ptr(), cc.data_ptr(), B, device=True)
            if timed:
                g.event_record(11 + 2 * (i % 8))
            if world == 1:
                g.genotype_packed_device(ptrs, pdims, ERR, MAX_COV, False)
                continue
            w = w_bufs[i & 1]
            g.lookup_packed_device(ptrs, pdims, w.data_ptr())
            work = dist.reduce(w, dst=0, async_op=True)    # overlaps the next step's scan
            if pending:
                finish(pending)
            pending = (work, w)
        if pending:
            finish(pending)

    sampler = ClockSampler(local_rank)
    sampler.start()
    run_steps(args.warmup, False)
    barrier()
    launches0 = g.launch_count()
    sampler.mark()
    g.event_record(2)
    run_steps(args.steps, True)
    g.event_record(3)
    region_ms = g.event_elapsed_ms(2, 3)
    clocks = sampler.stop()
    launches = g.launch_count() - launches0
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, d, vb["vao"])
    scan_ms = [g.event_elapsed_ms(10 + 2 * j, 11 + 2 * j) for j in range(min(8, args.steps))]
    geno_ms = g.genotype_kernel_ms() if rank == 0 else None
    tm = torch.tensor([region_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    region_ms = float(tm.item())
    verified_reduce = reduce_ms = None
    if world > 1 and args.verify:
        # identical replicas (canonical index image) that scanned identical batches:
        #  (1) the summed look-up results of a step are exactly world x one rank's
        w_own = torch.zeros(max(nk, 1), dtype=torch.int32, device=dev)
        g.lookup_packed_device(ptrs, pdims, w_own.data_ptr())
        w_sum = w_own.clone()
        dist.reduce(w_sum, dst=0)
        ok_w = bool(torch.equal(w_sum, w_own * world)) and int(w_own.abs().sum().item()) != 0
        #  (2) the counter arrays themselves (gather -> ncclReduce -> scatter) are world x one rank's, element by element
        before = [t.clone() for t in [torch.as_tensor(DevArray(p, n), device=dev)
                                      for p, n in g.counter_buffers(gather=True) if n]]
        torch.cuda.synchronize()
        t_red0 = time.perf_counter()
        reduce_counters()
        reduce_ms = (time.perf_counter() - t_red0) * 1e3
        if rank == 0:
            after = [torch.as_tensor(DevArray(p, n), device=dev) for p, n in g.counter_buffers(gather=True) if n]
            ok_c = all(bool(torch.equal(t, b * world)) for t, b in zip(after, before)) and \
                any(int(b.sum().item()) != 0 for b in before)
            verified_reduce = ok_w and ok_c
            log(f"[verify] summed look-up results == {world} x rank 0's: {ok_w}; reduced counters == {world} x rank 0's: {ok_c}")
    ms_per_step = region_ms / args.steps
    value = world * B / (ms_per_step * 1e-3)

    # ---- host-side inputs of the e2e leg, all in pinned memory (allocated after the NUMA binding) ----
    #  (a) the batch as raw KMC suffix records (+ prefix LUT): what malva-geno call reads from <db>.kmc_suf
    #  (b) the same batch as packed {lo,hi} words + u32 counts (the host-decoded form)
    #  (c) the variant batch in the packed form the C++ host sends; outputs land in pinned buffers too
    e2e = None
    h2d_ceiling = None
    if not args.no_e2e:
        pin = lambda t: t.cpu().pin_memory()
        kmc_rec, kmc_lut = make_kmc_records(torch, batches[0][0], batches[0][1])
        h_rec = pin(kmc_rec)
        kmc_db = dict(lut=kmc_lut.cpu().numpy().astype(np.uint64), lut_prefix_len=7, k=REF_K, counter_size=1, min_count=2,
                      max_count=255)
        del kmc_rec
        hk, hc = pin(batches[0][0]), pin(batches[0][1])
        h_in = {k2: pin(torch.from_numpy(vb[k1])) for k1, k2 in (("vao", "var_allele_off"), ("aso", "allele_sig_off"),
                                                                 ("sko", "sig_kmer_off"), ("freq", "freq"))}
        h_in["kmers"] = pin(vb["kmers"])
        h_out = {"cov": torch.zeros(na, dtype=torch.int32).pin_memory()}
        for nme in ("n_gts", "status", "best_gt", "gq"):
            h_out[nme] = torch.zeros(nv, dtype=torch.int32).pin_memory()
        h_ptrs = {k2: t.data_ptr() for k2, t in {**h_in, **h_out}.items()}
        csr_bytes = sum(t.numel() * t.element_size() for t in h_in.values())

        # the box's own ceiling: every rank copies 1 GiB of pinned memory to its GPU at the same time
        src = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
        dst = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
        dst.copy_(src, non_blocking=True)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(4):
            dst.copy_(src, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        mine = 4 * (1 << 30) / (e0.elapsed_time(e1) * 1e-3) / 1e9
        t = torch.tensor([mine, -mine], dtype=torch.float64, device=dev)
        tsum = t.clone()
        if world > 1:
            dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        h2d_ceiling = {"aggregate_GBps": float(tsum[0]), "slowest_rank_GBps": float(-t[1]), "fastest_rank_GBps": float(t[0]),
                       "how": "1 GiB pinned -> device x4 per rank, all ranks at once, CUDA events"}
        del src, dst

        def e2e_leg(scan):
            steps = args.steps
            scan()
            g.genotype_packed_host(h_ptrs, nv, 0, ERR, MAX_COV, False)
            if world > 1:
                g.sync()
                reduce_counters()                                        # (first call builds the key ranks: not timed)
            barrier()
            t0 = time.perf_counter()
            g.event_record(4)
            for _ in range(steps):
                scan()                                                   # asynchronous, chunked, double-buffered H2D + K1
                g.genotype_packed_host(h_ptrs, nv, 0, ERR, MAX_COV, False)  # H2D batch, K4+K5, D2H results; returns when landed
            if world > 1:
                g.sync()
                reduce_counters()                                        # the counters of all ranks on rank 0
            g.event_record(5)
            ms = max(g.event_elapsed_ms(4, 5), (time.perf_counter() - t0) * 1e3) / steps
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())

        g.kmc_open(kmc_db)
        e2e_ms = e2e_leg(lambda: g.scan_kmc_records(h_rec.data_ptr(), 0, B, sync=False))
        e2e_packed_ms = e2e_leg(lambda: g.scan_sample_kmers_ptr(hk.data_ptr(), hc.data_ptr(), B, device=False))
        d2h = 4 * na + 16 * nv
        h2d = B * 10 + csr_bytes
        e2e = {"value": world * B / (e2e_ms * 1e-3), "unit": "k-mers/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "variants_per_sec": world * nv / (e2e_ms * 1e-3),
               "h2d_GBps_per_gpu": h2d / (e2e_ms * 1e-3) / 1e9,
               "note": "per step: mg_scan_kmc_records(pinned raw .kmc_suf records, 10 B per 43-mer, decoded on the device) + "
                       "mg_genotype_packed(pinned host batch, 16 B per signature k-mer) -> pinned host results"
                       + ("; the NCCL counter reduce (gather, ncclReduce, scatter) is inside the timed region" if world > 1 else ""),
               "packed128": {"value": world * B / (e2e_packed_ms * 1e-3), "ms_per_step": e2e_packed_ms,
                             "h2d_bytes_per_step": B * 20 + csr_bytes,
                             "note": "same step with host-decoded {lo,hi} words + u32 counts (20 B per 43-mer) through "
                                     "mg_scan_sample_kmers"}}

    # ---- self-check (b) + CPU baselines (rank 0, N = 1 only): the reference's own classes on a bounded sample ----
    cpu = None
    if world == 1 and not args.no_cpu:
        cpu, check = cpu_legs(wl, 2_000_000, 4_000_000, gpu_device=None if args.no_verify else local_rank)
        if check is not None:
            verify["reference_at_bench_shape"] = check
            log(f"[rank {rank}] self-check (b) {check}")
            if not (check["key_counts_equal"] and check["cov_equal"] and check["gt_equal"] and check["gq_equal"]):
                print(json.dumps({"verified": False, **verify}), flush=True)
                raise SystemExit(3)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- rooflines, measured live with CUDA events on the kernels' stream ----
    peak, peak_src = measured_peaks()
    k1_ms = float(np.mean(scan_ms))
    achieved = B * ALGO_BYTES_PER_KMER / (k1_ms * 1e-3) / 1e9
    rand_gbs = stream_gbs = line_gbs = None
    if not args.no_diag:
        try:
            rand_gbs = diag_bandwidth(local_rank, 0, 16 << 30, 3)
            line_gbs = diag_bandwidth(local_rank, 4, 16 << 30, 3)
            stream_gbs = diag_bandwidth(local_rank, 1, 16 << 30, 3)
        except Exception as e:  # noqa: BLE001
            log("diag_bandwidth failed:", e)
    traffic = profile_json("k1_traffic.json").get("dram_bytes_per_launch")
    k4_bytes = nk * ALGO_BYTES_PER_SIG_KMER + na * 8 + nv * 8 + vb["lik_slots"] * 8
    k4_ms = float(sum(geno_ms))
    k2_bytes = wl["ref_bases"] * ALGO_BYTES_PER_REF_BASE
    n_chunks = -(-wl["ref_bases"] // (32 << 20))
    line = {
        "metric": "sample_kmers_per_sec", "value": value, "unit": "k-mers/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config_of(wl, world),
        "variants_per_sec": world * nv / (k4_ms * 1e-3),
        "variants_per_sec_note": "K4+K5 kernels (signature look-ups, coverage, likelihood), device-resident packed batch",
        "kernel_ms": {"k1_scan": k1_ms, "k4_lookup": geno_ms[0], "k4_coverage": geno_ms[1], "k5_genotype": geno_ms[2],
                      "k2_reference_pass": refpass_kernel_ms, "k2_reference_pass_incl_h2d_pinned": refpass_pinned_ms,
                      "k2_reference_pass_incl_h2d_pageable": refpass_pageable_ms},
        "ref_bases_per_sec": wl["ref_bases"] / (refpass_kernel_ms * 1e-3),
        "ref_bases_per_sec_incl_h2d": wl["ref_bases"] / (refpass_pinned_ms * 1e-3),
        "ref_bases_per_sec_incl_h2d_pageable": wl["ref_bases"] / (refpass_pageable_ms * 1e-3),
        "index": {"bf_ones": pop_alt, "context_ones": pop_ctx, "ref_keys": n_keys, "overflow_keys": stats["overflow_keys"]},
        "e2e": e2e,
        "h2d_ceiling_GBps_at_N": h2d_ceiling,
        "numa_binding": numa,
        "gpu_launches": launches,
        **({"multi_gpu": "every rank scans its own share of the sample stream into its replica's counters and looks the "
                         "variant batch up in them (K4, raw); the 4-byte look-up results are summed onto rank 0 (ncclReduce, "
                         f"{4 * nk} B per step, overlapped with the next step's scan) which computes coverage + "
                         "likelihoods from the sums (get_count is linear in the counters)"} if world > 1 else {}),
        **({"verify_reduce_exact": verified_reduce} if verified_reduce is not None else {}),
        **({"counter_reduce_ms": reduce_ms} if reduce_ms is not None else {}),
        **({"verified": True, "verify": verify} if verify else {}),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": "k_scan<35,43>", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                     "algorithmic_bytes_per_kmer": ALGO_BYTES_PER_KMER,
                     "measured_random_32B_sector_GBps": rand_gbs, "measured_random_128B_line_GBps": line_gbs,
                     "measured_stream_read_GBps": stream_gbs,
                     "frac_of_random_sector_ceiling": (achieved / rand_gbs) if rand_gbs else None,
                     "lines_per_sec_vs_ceiling": (B / (k1_ms * 1e-3)) / (line_gbs * 1e9 / 128) if line_gbs else None},
        "roofline_k4k5": {"bound": "hbm", "kernel": "k_lookup_packed<35> + k_coverage + k_genotype",
                          "achieved": k4_bytes / (k4_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                          "frac": k4_bytes / (k4_ms * 1e-3) / 1e9 / peak,
                          "algorithmic_bytes": k4_bytes,
                          "algorithmic_bytes_note": "36 B per signature k-mer + 8 B per allele in + 8 B per variant and per "
                                                    "genotype slot out (SURVEY 8d)",
                          "traffic": profile_json("k4_traffic.json").get("dram_bytes_per_launch"),
                          "lines_per_sec_vs_ceiling": (nk / (geno_ms[0] * 1e-3)) / (line_gbs * 1e9 / 128) if line_gbs else None},
        "roofline_k2": {"bound": "hbm", "kernel": "k_refpass<35,43>", "achieved": k2_bytes / (refpass_kernel_ms * 1e-3) / 1e9,
                        "peak": peak, "unit": "GB/s", "frac": k2_bytes / (refpass_kernel_ms * 1e-3) / 1e9 / peak,
                        "algorithmic_bytes": k2_bytes, "launches": n_chunks,
                        "algorithmic_bytes_note": "33 B per reference base over the whole contig (one launch per 32 Mi-base "
                                                  "chunk; `traffic` is the DRAM traffic of one full-chunk launch = 1.107e9 "
                                                  "algorithmic bytes)",
                        "traffic": profile_json("k2_traffic.json").get("dram_bytes_per_launch")},
    }
    if cpu:
        line["cpu_baseline"] = {
            "value": cpu["kmers_per_sec"], "unit": "k-mers/s", "cores": 1, "kind": cpu["kind"],
            "sample": f"{cpu['n_scan']} sample 43-mers against 2^{int(np.log2(wl['bf_bits']))}-bit filters with {cpu['n_sig']} alt "
                      f"bits + {cpu['n_sig']} ref keys (full workload: {wl['n_alt']} + {wl['n_ref']}), the reference's own BF/KMAP "
                      "classes, 1 thread (malva-geno is single-threaded)",
            "host_cores_available": cpu["host_cores_available"]}
        if "variants_per_sec" in cpu:
            line["cpu_baseline_variants"] = {
                "value": cpu["variants_per_sec"], "unit": "variants/s", "cores": 1, "kind": cpu["kind"],
                "sample": f"{cpu['n_genotyped']} variants of the same shape: set_coverages (BF/KMAP::get_count per signature "
                          "k-mer, main.cpp:151-184) + VB::genotype + arg-max (var_block.hpp:224-394); signature enumeration "
                          "and VCF parsing not included"}
            line["cpu_baseline_ref_bases"] = {
                "value": cpu["ref_bases_per_sec"], "unit": "bases/s", "cores": 1, "kind": cpu["kind"],
                "sample": "1e6 random bases through the reference's rolling loop (main.cpp:382-402)"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="wg", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs and self-check (b)")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer end-to-end leg (profiling runs)")
    ap.add_argument("--no-diag", action="store_true", help="skip the bandwidth microbenchmarks (profiling runs)")
    ap.add_argument("--no-verify", action="store_true", help="skip the self-checks (profiling runs)")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the process to the GPU's NUMA node")
    ap.add_argument("--verify", action="store_true",
                    help="N > 1: every rank scans the same batches; checks that the NCCL-reduced counters are exactly "
                         "N x one rank's (replicas are identical, the reduce is exact)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (coverages, GT, GQ; a seeded sample of the variants "
                         "at large workloads) as DIR/<name>.npy, float64")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times the sample scan alone, which returns nothing to its caller")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, wl, rank, world)
    else:
        run_ours(args, wl, rank, local_rank, world)


if __name__ == "__main__":
    main()
