"""Cost of sex-chromosome ploidy (genotype-cohort.py --ploidy-file / --sample-sex) in the cohort's genotype + VCF step.

C2's catalogue (25 k SVs, synth) on the device, loaded random counters for S samples, and a catalogue of R records
(C2's VCF body repeated) for the text.  The step is what genotype_cohort_vcf does per block: the genotype kernel, the
site statistics and the formatter, with all tags (nine without ploidy, ten with it; the text is made and dropped, not
written).  With ploidy, half the samples are M, half F, and the rules are GRCh38's non-PAR chrX and chrY for M (1) and
chrY for F (0); the record classes are computed once, outside the timed step, as genotype_cohort_vcf does.  Timed
alternating without and with ploidy (median of 5 each), then one torch.profiler pass of each that splits out the genotype
kernel.  The card's name, power limit and max SM clock are printed with the numbers.

    python profiles/cohort_ploidy_timing.py --out DIR
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "svjedi-graph_b200")
sys.path[:0] = [ROOT, PKG]

RULES = "chrX 2781 155701382 M 1\nchrY 1 57227415 M 1\nchrY 1 57227415 F 0\n"


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    return r.stdout.strip().splitlines()[0]


def one_case(tables, vcf_text, n_rec, n_samples, out_dir):
    import numpy as np

    from svjg import capi, cohort, genotype
    rng = np.random.default_rng(3)
    body = [ln for ln in vcf_text.splitlines(True) if not ln.startswith("#")]
    head = "".join(ln for ln in vcf_text.splitlines(True) if ln.startswith("#"))
    reps = -(-n_rec // len(body))
    v = genotype.NativeVcf.from_input((head + "".join(body) * reps).encode())
    n = n_rec
    co = cohort.Cohort(tables, n_samples)
    for s in range(n_samples):
        c = rng.integers(0, 40, (tables.num_sv, 2)).astype(np.uint32)
        c[rng.random(tables.num_sv) < 0.3, 0] = 0
        c[rng.random(tables.num_sv) < 0.3, 1] = 0
        co.load_counts(s, c)
    idx = rng.integers(0, tables.num_sv, n).astype(np.uint32)
    ty = rng.integers(0, 4, n).astype(np.uint8)
    names = [f"s{k}" for k in range(n_samples)]
    rules = cohort.PloidyRules(RULES, "".join(f"{nm} {'MF'[k % 2]}\n" for k, nm in enumerate(names)), names)
    t0 = time.perf_counter()
    rclass, table = rules.record_classes(v)
    classes_s = time.perf_counter() - t0
    capi.check(capi.lib.svjg_cohort_set_ploidy(co._h, table.shape[0], table.shape[1], table.ctypes.data,
                                               rules.sex_index.ctypes.data))
    step = max(1, cohort.BLOCK_BYTES // (cohort.CELL_BYTES * n_samples))
    blocks = {False: cohort._Block(min(step, n) * n_samples, min(step, n)),
              True: cohort._Block(min(step, n) * n_samples, min(step, n), ploidy=True)}
    joined = "\t".join(names).encode()
    masks = {False: cohort.info_tags_mask(cohort.INFO_TAGS), True: cohort.info_tags_mask(cohort.PLOIDY_INFO_TAGS)}

    def one_pass(ploidy):
        blk = blocks[ploidy]
        n_gt = np.zeros(n_samples, np.uint64)
        out_bytes = 0
        fmt = capi.lib.svjg_vcf_format_cohort_ploidy if ploidy else capi.lib.svjg_vcf_format_cohort_tags
        for lo in range(0, n, step):
            hi = min(n, lo + step)
            gt, fl, ad, pl = cohort._genotype_block(co, idx[lo:hi], ty[lo:hi], 3, genotype.ERR, blk,
                                                    rclass[lo:hi] if ploidy else None)
            site = [a.ctypes.data for a in cohort._site_stats(co, hi - lo, blk, ploidy)]
            buf, n_out = C.c_void_p(), C.c_uint64()
            capi.check(fmt(v._h, lo, hi, n_samples, joined, len(joined), gt.ctypes.data, fl.ctypes.data, ad.ctypes.data,
                           pl.ctypes.data, masks[ploidy], *site, C.byref(buf), C.byref(n_out), n_gt.ctypes.data))
            out_bytes += n_out.value
            capi.lib.svjg_buffer_free(buf)
        return out_bytes

    sizes = {p: one_pass(p) for p in (False, True)}                          # warm-up
    times = {False: [], True: []}
    for _ in range(5):
        for p in (False, True):
            t0 = time.perf_counter()
            one_pass(p)
            times[p].append(time.perf_counter() - t0)
    import torch
    from torch.profiler import ProfilerActivity, profile
    kern_ms = {}
    for p in (False, True):
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            one_pass(p)
        us = 0.0
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA and "genotype_cohort_kernel" in ev.name:
                us += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        kern_ms[p] = us / 1e3
        prof.export_chrome_trace(os.path.join(out_dir, f"cohort_ploidy_{n_rec}x{n_samples}_{int(p)}.pt.trace.json"))
    med = {p: sorted(t)[2] for p, t in times.items()}
    return {"records": n, "samples": n_samples, "block_records": step, "classes": int(table.shape[0]),
            "haploid_or_zero_records": int((table[rclass] != 2).any(axis=1).sum()), "record_classes_s": classes_s,
            "wall_s_diploid": sorted(times[False]), "wall_s_ploidy": sorted(times[True]),
            "median_diploid_s": med[False], "median_ploidy_s": med[True], "added_fraction": med[True] / med[False] - 1,
            "text_bytes_diploid": sizes[False], "text_bytes_ploidy": sizes[True],
            "profiled_genotype_kernel_ms_diploid": kern_ms[False], "profiled_genotype_kernel_ms_ploidy": kern_ms[True]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cases", default="1000000x64")
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    from svjg import alnfilter, graphgen, synth
    result = {"card": card()}
    chrom_len = synth.human_like_chroms(1.0)
    rows = synth.catalogue("delins", 25_000, chrom_len, 1002, ins_max=5000)     # C2's catalogue (synth.WORKLOADS)
    g = graphgen.build_graph(chrom_len, rows)
    import io
    buf = io.StringIO()
    g.write_gfa(buf)
    tables = alnfilter.Tables.from_memory(g.edges_json(), buf.getvalue()).to_device(0)
    vcf_text = synth.vcf_text(rows)
    result["cases"] = []
    for case in args.cases.split(","):
        r, s = (int(x) for x in case.split("x"))
        result["cases"].append(one_case(tables, vcf_text, r, s, args.out))
        print(json.dumps(result["cases"][-1]), flush=True)
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    with open(os.path.join(args.out, "cohort_ploidy_timing.json"), "w") as fh:
        fh.write(text + "\n")


if __name__ == "__main__":
    main()
