"""Cost of genotype posteriors (genotype-cohort.py --posteriors) in the cohort's genotype + VCF step.

C2's catalogue (25 k SVs, synth) on the device, loaded random counters for S samples, and a catalogue of R records
(C2's VCF body repeated) for the text.  The step is what genotype_cohort_vcf does per block: the genotype kernel, the
site statistics (all nine tags) and the formatter, and with posteriors the posterior kernel (svjg_cohort_posteriors,
with the block's NEED_K cells patched in) between them; the text is made and dropped, not written.  The block size
follows genotype_cohort_vcf: 256 MiB of cell arrays, 34 B per cell without posteriors and 59 B with them.  Timed
alternating without and with posteriors (median of --runs each), then one torch.profiler pass with posteriors that
splits out the posterior kernel, and a histogram of EM steps per record.  The card's name, power limit and max SM
clock are printed with the numbers.

    python profiles/cohort_posterior_timing.py --out DIR [--cases 1000000x64,100000x4096]
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


def one_case(tables, vcf_text, n_rec, n_samples, runs, out_dir):
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
    steps = {p: max(1, cohort.BLOCK_BYTES // ((cohort.CELL_BYTES + (cohort.POST_CELL_BYTES if p else 0)) * n_samples))
             for p in (False, True)}
    blocks = {p: cohort._Block(min(steps[p], n) * n_samples, min(steps[p], n), post_records=min(steps[p], n) if p else 0)
              for p in (False, True)}
    joined = "\t".join(names).encode()
    mask = cohort.info_tags_mask(cohort.INFO_TAGS)
    iters = np.zeros(n, np.uint8)

    def one_pass(post):
        blk, step = blocks[post], steps[post]
        n_gt = np.zeros(n_samples, np.uint64)
        out_bytes = 0
        for lo in range(0, n, step):
            hi = min(n, lo + step)
            gt, fl, ad, pl = cohort._genotype_block(co, idx[lo:hi], ty[lo:hi], 3, genotype.ERR, blk)
            site = [a.ctypes.data for a in cohort._site_stats(co, hi - lo, blk)]
            buf, n_out = C.c_void_p(), C.c_uint64()
            if post:
                pa = [a.ctypes.data for a in cohort._posteriors(co, hi - lo, blk, iters[lo:hi])]
                capi.check(capi.lib.svjg_vcf_format_cohort_post(
                    v._h, lo, hi, n_samples, joined, len(joined), gt.ctypes.data, fl.ctypes.data, ad.ctypes.data,
                    pl.ctypes.data, 0, mask, *site, *pa, C.byref(buf), C.byref(n_out), n_gt.ctypes.data))
            else:
                capi.check(capi.lib.svjg_vcf_format_cohort_tags(
                    v._h, lo, hi, n_samples, joined, len(joined), gt.ctypes.data, fl.ctypes.data, ad.ctypes.data,
                    pl.ctypes.data, mask, *site, C.byref(buf), C.byref(n_out), n_gt.ctypes.data))
            out_bytes += n_out.value
            capi.lib.svjg_buffer_free(buf)
        return out_bytes

    sizes = {p: one_pass(p) for p in (False, True)}                          # warm-up
    times = {False: [], True: []}
    for _ in range(runs):
        for p in (False, True):
            t0 = time.perf_counter()
            one_pass(p)
            times[p].append(time.perf_counter() - t0)
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        one_pass(True)
    kern_us = {"cohort_posterior_kernel": 0.0, "genotype_cohort_kernel": 0.0, "cohort_patch_kernel": 0.0}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            for k in kern_us:
                if k in ev.name:
                    kern_us[k] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
    prof.export_chrome_trace(os.path.join(out_dir, f"cohort_posterior_{n_rec}x{n_samples}.pt.trace.json"))
    med = {p: sorted(t)[len(t) // 2] for p, t in times.items()}
    hist = np.bincount(iters, minlength=capi.POST_MAX_ITERS + 1)
    return {"records": n, "samples": n_samples, "block_records_plain": steps[False], "block_records_post": steps[True],
            "wall_s_plain": sorted(times[False]), "wall_s_posteriors": sorted(times[True]),
            "median_plain_s": med[False], "median_posteriors_s": med[True], "added_fraction": med[True] / med[False] - 1,
            "text_bytes_plain": sizes[False], "text_bytes_posteriors": sizes[True],
            "d2h_bytes_posteriors": n * n_samples * cohort.POST_CELL_BYTES + n * 8,
            "profiled_kernel_ms": {k: us / 1e3 for k, us in kern_us.items()},
            "em_steps_histogram": {str(k): int(c) for k, c in enumerate(hist) if c},
            "em_steps_mean": float(iters.mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cases", default="1000000x64,100000x4096")
    ap.add_argument("--runs", type=int, default=5)
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
        result["cases"].append(one_case(tables, vcf_text, r, s, args.runs, args.out))
        print(json.dumps(result["cases"][-1]), flush=True)
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    with open(os.path.join(args.out, "cohort_posterior_timing.json"), "w") as fh:
        fh.write(text + "\n")


if __name__ == "__main__":
    main()
