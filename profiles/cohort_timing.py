"""Cohort genotyping on one GPU, against today's route of two command lines per sample.

C2's catalogue (25 k SVs, synth) and S samples with distinct genotype draws (simulate_gaf with S seeds on the same
graph).  Timed, alternating, on one box:
  (A) per sample: filter-alignments.py, then predict-genotype.py (2 S processes);
  (B) one genotype-cohort.py over all samples.
Before any time is printed, every column of (B) is checked against the SAMPLE column of (A).  Then the genotype
step alone: svjg_cohort_genotype over --kernel-records records x --kernel-samples samples of loaded random counts,
in the blocks genotype_cohort_vcf uses, with a torch.profiler pass that splits kernel and copy times.
The card's name, power limit and max SM clock are printed with the numbers.

    python profiles/cohort_timing.py --out DIR [--samples 8] [--records 750000] [--rounds 2]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "svjedi-graph_b200")
sys.path[:0] = [ROOT, PKG]


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, check=True)
    return r.stdout.strip().splitlines()[0]


def run(script, *args):
    t0 = time.perf_counter()
    r = subprocess.run([sys.executable, os.path.join(PKG, script), *args], capture_output=True, text=True)
    dt = time.perf_counter() - t0
    if r.returncode:
        raise SystemExit(f"{script} failed: {r.stderr}")
    return dt, r.stdout


def check_columns(single, cohort_text, names):
    """Column k of the cohort VCF is the SAMPLE column of sample k's single-sample VCF, every other byte the same."""
    a = [t.split("\n") for t in single]
    b = cohort_text.split("\n")
    assert all(len(x) == len(b) for x in a), "line counts differ"
    for j, line in enumerate(b):
        first = a[0][j]
        if first.startswith("#CHROM"):
            assert line == first[:-len("SAMPLE")] + "\t".join(names), j
        elif "\t" not in first or line == first:
            assert line == first and all(x[j] == first for x in a), j
        else:
            assert line == first.rsplit("\t", 1)[0] + "".join("\t" + x[j].rsplit("\t", 1)[1] for x in a), j


def kernel_alone(tables, n_rec, n_samples, out_dir):
    import numpy as np
    from svjg import cohort, genotype
    rng = np.random.default_rng(3)
    co = cohort.Cohort(tables, n_samples)
    for s in range(n_samples):
        co.load_counts(s, rng.integers(0, 100, (tables.num_sv, 2)).astype(np.uint32))
    idx = rng.integers(0, tables.num_sv, n_rec).astype(np.uint32)
    ty = rng.integers(0, 4, n_rec).astype(np.uint8)
    step = max(1, cohort.BLOCK_BYTES // (cohort.CELL_BYTES * n_samples))
    blk = cohort._Block(step * n_samples)

    def one_pass():
        for lo in range(0, n_rec, step):
            cohort._genotype_block(co, idx[lo:lo + step], ty[lo:lo + step], 3, genotype.ERR, blk)
    one_pass()                                                        # warm-up: module load, LUT, block buffers
    times = []
    for _ in range(5):
        t0 = time.perf_counter()
        one_pass()                                                    # every block call ends in a stream synchronise
        times.append(time.perf_counter() - t0)
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        one_pass()
    kern = copy_d2h = copy_h2d = 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        if "genotype_cohort_kernel" in ev.name:
            kern += us
        elif "DtoH" in ev.name or "Device -> Pageable" in ev.name or "Device -> Pinned" in ev.name:
            copy_d2h += us
        elif "HtoD" in ev.name or "-> Device" in ev.name:
            copy_h2d += us
    prof.export_chrome_trace(os.path.join(out_dir, "cohort_genotype.pt.trace.json"))
    cells = n_rec * n_samples
    return {"records": n_rec, "samples": n_samples, "cells": cells, "block_records": step,
            "bytes_per_cell_d2h": cohort.CELL_BYTES, "wall_s": sorted(times), "wall_s_median": sorted(times)[2],
            "profiled_kernel_ms": kern / 1e3, "profiled_d2h_ms": copy_d2h / 1e3, "profiled_h2d_ms": copy_h2d / 1e3,
            "d2h_GBps": cells * cohort.CELL_BYTES / (copy_d2h / 1e6) / 1e9 if copy_d2h else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--samples", type=int, default=8)
    ap.add_argument("--records", type=int, default=750_000)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--kernel-records", type=int, default=1_000_000)
    ap.add_argument("--kernel-samples", type=int, default=64)
    args = ap.parse_args()
    os.makedirs(args.out, exist_ok=True)
    from svjg import alnfilter, graphgen, synth
    result = {"card": card()}
    t0 = time.perf_counter()
    chrom_len = synth.human_like_chroms(1.0)
    rows = synth.catalogue("delins", 25_000, chrom_len, 1002, ins_max=5000)     # C2's catalogue (synth.WORKLOADS)
    g = graphgen.build_graph(chrom_len, rows)
    with tempfile.TemporaryDirectory() as tmp:
        prefix = os.path.join(tmp, "c2")
        edges = g.edges_json()
        open(prefix + "_svs_edges.json", "w").write(edges)
        with open(prefix + ".gfa", "w") as fh:
            g.write_gfa(fh)
        open(prefix + ".vcf", "w").write(synth.vcf_text(rows))
        gafs = []
        for s in range(args.samples):
            gafs.append(os.path.join(tmp, f"sample{s}.gaf"))
            with open(gafs[-1], "w") as fh:
                fh.write(synth.simulate_gaf_parallel(g, args.records, 2000 + s, mean_len=31_000))
            os.symlink(prefix + "_svs_edges.json", os.path.join(tmp, f"p{s}_svs_edges.json"))
        result["input_gib"] = sum(os.path.getsize(p) for p in gafs) / 2**30
        result["setup_s"] = time.perf_counter() - t0
        names = [f"sample{s}" for s in range(args.samples)]
        a_times, b_times, single = [], [], None
        for _ in range(args.rounds):
            t_a = 0.0
            single = []
            for s, gaf in enumerate(gafs):
                p = os.path.join(tmp, f"p{s}")
                dt1, _ = run("filter-alignments.py", "-a", gaf, "-g", prefix + ".gfa", "-p", p)
                dt2, _ = run("predict-genotype.py", "-d", p + "_informative_aln.json", "-v", prefix + ".vcf",
                             "-o", p + "_genotype.vcf")
                t_a += dt1 + dt2
                single.append(open(p + "_genotype.vcf").read())
                os.unlink(p + "_informative_aln.json")
            a_times.append(t_a)
            dt, stdout = run("genotype-cohort.py", "-p", prefix, "-g", prefix + ".gfa", "-v", prefix + ".vcf", "-a", *gafs,
                             "-o", prefix + "_cohort.vcf", "--names", ",".join(names))
            b_times.append(dt)
            check_columns(single, open(prefix + "_cohort.vcf").read(), names)
        result.update({"samples": args.samples, "records_per_sample": args.records, "route_A_s": a_times,
                       "route_B_s": b_times, "columns_checked": True,
                       "A_per_sample_s": min(a_times) / args.samples, "B_per_sample_s": min(b_times) / args.samples,
                       "B_stdout": stdout.splitlines()})
        tables = alnfilter.Tables.from_memory(edges, open(prefix + ".gfa").read()).to_device(0)
        result["genotype_alone"] = kernel_alone(tables, args.kernel_records, args.kernel_samples, args.out)
    text = json.dumps(result, indent=1)
    print(text)
    with open(os.path.join(args.out, "cohort_timing.json"), "w") as fh:
        fh.write(text + "\n")


if __name__ == "__main__":
    main()
