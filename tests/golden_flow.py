"""The malva-geno index+call flow over tests/golden/haploid, parameterised by the backend that holds
bf / context_bf / ref_bf: the CPU oracle (OracleRun) or the GPU (MalvaGpu).  Returns VCF body lines.

Signatures come from the reference's own VB::extract_kmers (oracle/_ref hook) where it is built, else from
`malva-geno signatures`, which tests/test_host_cpu.py holds equal to it on this example."""
import os
import subprocess

import vcf_blocks
from malva_b200 import SignatureBatch, genotype_names, kmc
from malva_b200 import build as mbuild
from parity_util import flatten

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "haploid")


def gold_lines(name):
    return [l for l in open(os.path.join(GOLD, name)).read().split("\n") if l and l[0] != "#"]


def cli_extractor(fa, vcf, flags, index_mode):
    """`malva-geno signatures` -> extract(b, blk) giving nested[v][allele] = [signatures] of the b-th var_block,
    the shape of vcf_blocks.ref_extract"""
    cmd = [mbuild.CLI, "signatures"] + (["--index-blocks"] if index_mode else []) + flags + [fa, vcf]
    sigs = {}
    for l in subprocess.run(cmd, capture_output=True, text=True, check=True).stdout.split("\n"):
        if l and not l.startswith("#"):
            b, _, _, vi, allele, kmers = l.split("\t")
            sigs.setdefault((int(b), int(vi), int(allele)), []).append(kmers.split(","))

    def extract(b, blk):
        return [[sorted(sigs.get((b, vi, a), [])) for a in range(len(v.alts) + 1)] for vi, v in enumerate(blk)]
    return extract


def run_haploid_example(backend, ref_lib, genotype):
    """backend: add_signatures/finalize_alt/scan_reference/finalize_context/scan_sample_kmers.
    genotype(batch) -> (cov, list of (status, best, gq, lik array)) per variant.  ref_lib: oracle/_ref or None."""
    k, ref_k, haploid = 35, 43, True
    fa_path, vcf_path = os.path.join(GOLD, "haploid.fa"), os.path.join(GOLD, "haploid.vcf.gz")
    fa = open(fa_path).read().split("\n")
    refs = {fa[0][1:].split()[0]: "".join(fa[1:]).upper()}
    _, recs = vcf_blocks.read_vcf(vcf_path, "AF")
    if ref_lib is not None:
        extract_index = extract_call = \
            lambda b, blk, contig: vcf_blocks.ref_extract(ref_lib, blk, refs[contig], k, haploid)
    else:
        by_cli = [cli_extractor(fa_path, vcf_path, ["-1", "-k", str(k)], m) for m in (True, False)]
        extract_index, extract_call = (lambda b, blk, contig, f=f: f(b, blk) for f in by_cli)
    used = []
    for b, (contig, blk) in enumerate(vcf_blocks.blocks(recs, k, index_mode=True)):
        if contig not in used:
            used.append(contig)
        ks, fl = flatten(extract_index(b, blk, contig))
        backend.add_signatures(ks, fl)
    backend.finalize_alt()
    for contig in used:
        backend.scan_reference(refs[contig])
    backend.finalize_context()
    packed, counts, kk = kmc.read_kmc_db(os.path.join(GOLD, "haploid"))
    assert kk == ref_k and len(packed) == 4503
    backend.scan_sample_kmers(packed, counts)
    lines = []
    for b, (contig, blk) in enumerate(vcf_blocks.blocks(recs, k, index_mode=False)):
        nested = extract_call(b, blk, contig)
        batch = SignatureBatch.from_nested(nested, [v.freqs for v in blk])
        cov, res = genotype(batch)
        for i, v in enumerate(blk):
            a0, a1 = int(batch.var_allele_off[i]), int(batch.var_allele_off[i + 1])
            names = genotype_names(a1 - a0, haploid)
            status, best, gq, lik = res[i]
            total = lik.sum()
            if status == 0:
                gts = ",".join(f"{n}:{(p / total):.6f}" if total > 0 else f"{n}:-nan" for n, p in zip(names, lik))
                gt = names[best]
            else:
                gts = ",".join("0:-nan" for _ in lik)
                gt = "0"
            covs = ",".join(str(int(c)) for c in cov[a0:a1])
            lines.append("\t".join([v.chrom, str(v.pos0 + 1), v.vid, v.ref, ",".join(v.alts), v.qual, "PASS",
                                    f"COVS={covs};GTS={gts}", "GT:GQ", f"{gt}:{gq}"]))
    return lines
