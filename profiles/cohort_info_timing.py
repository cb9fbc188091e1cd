"""Cost of the population INFO tags (genotype-cohort.py --info-tags) in the cohort's genotype + VCF step.

C2's catalogue (25 k SVs, synth) on the device, loaded random counters for S samples, and a catalogue of R records
(C2's VCF body repeated) for the text.  The step is what genotype_cohort_vcf does per block: svjg_cohort_genotype,
then, with the tags, svjg_cohort_site_stats, then svjg_vcf_format_cohort_tags (the text is made and dropped, not
written).  Timed alternating without and with all tags (median of 5 each), then one torch.profiler pass with the tags
that splits the stats kernel, the genotype kernel and the copies.  Cases: 1 M records x 64 samples and
100 k records x 4 096 samples (the longest exact tests).  The card's name, power limit and max SM clock are printed
with the numbers.

    python profiles/cohort_info_timing.py --out DIR
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
        c[rng.random(tables.num_sv) < 0.3, 0] = 0                          # some hom-alt and het cells
        c[rng.random(tables.num_sv) < 0.3, 1] = 0
        co.load_counts(s, c)
    idx = rng.integers(0, tables.num_sv, n).astype(np.uint32)
    ty = rng.integers(0, 4, n).astype(np.uint8)
    step = max(1, cohort.BLOCK_BYTES // (cohort.CELL_BYTES * n_samples))
    blk = cohort._Block(min(step, n) * n_samples, min(step, n))
    names = "\t".join(f"s{k}" for k in range(n_samples)).encode()
    all_mask = cohort.info_tags_mask(cohort.INFO_TAGS)

    def one_pass(mask):
        n_gt = np.zeros(n_samples, np.uint64)
        out_bytes = 0
        for lo in range(0, n, step):
            hi = min(n, lo + step)
            gt, fl, ad, pl = cohort._genotype_block(co, idx[lo:hi], ty[lo:hi], 3, genotype.ERR, blk)
            site = [None] * 3
            if mask:
                site = [a.ctypes.data for a in cohort._site_stats(co, hi - lo, blk)]
            buf, n_out = C.c_void_p(), C.c_uint64()
            capi.check(capi.lib.svjg_vcf_format_cohort_tags(v._h, lo, hi, n_samples, names, len(names), gt.ctypes.data,
                                                            fl.ctypes.data, ad.ctypes.data, pl.ctypes.data, mask, *site,
                                                            C.byref(buf), C.byref(n_out), n_gt.ctypes.data))
            out_bytes += n_out.value
            capi.lib.svjg_buffer_free(buf)
        return out_bytes

    sizes = {0: one_pass(0), all_mask: one_pass(all_mask)}                 # warm-up
    times = {0: [], all_mask: []}
    for _ in range(5):
        for mask in (0, all_mask):
            t0 = time.perf_counter()
            one_pass(mask)
            times[mask].append(time.perf_counter() - t0)
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        one_pass(all_mask)
    kern = {"cohort_site_stats_kernel": 0.0, "genotype_cohort_kernel": 0.0}
    copy_d2h = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        for k in kern:
            if k in ev.name:
                kern[k] += us
        if "DtoH" in ev.name or "Device -> Pageable" in ev.name or "Device -> Pinned" in ev.name:
            copy_d2h += us
    prof.export_chrome_trace(os.path.join(out_dir, f"cohort_info_{n_rec}x{n_samples}.pt.trace.json"))
    med = {m: sorted(t)[2] for m, t in times.items()}
    return {"records": n, "samples": n_samples, "block_records": step,
            "wall_s_no_tags": sorted(times[0]), "wall_s_all_tags": sorted(times[all_mask]),
            "median_no_tags_s": med[0], "median_all_tags_s": med[all_mask],
            "added_fraction": med[all_mask] / med[0] - 1,
            "text_bytes_no_tags": sizes[0], "text_bytes_all_tags": sizes[all_mask],
            "d2h_bytes_cells": n * n_samples * cohort.CELL_BYTES, "d2h_bytes_added": n * 32,
            "profiled_site_stats_kernel_ms": kern["cohort_site_stats_kernel"] / 1e3,
            "profiled_genotype_kernel_ms": kern["genotype_cohort_kernel"] / 1e3,
            "profiled_d2h_ms": copy_d2h / 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cases", default="1000000x64,100000x4096")
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
    with open(os.path.join(args.out, "cohort_info_timing.json"), "w") as fh:
        fh.write(text + "\n")


if __name__ == "__main__":
    main()
