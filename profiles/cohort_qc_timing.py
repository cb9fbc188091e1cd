"""Cost of the sample QC table and the relatedness table (genotype-cohort.py --sample-qc / --relatedness).

1. The genotype + VCF text step with and without both switches, alternating (median of --runs each): C2's catalogue
   (25 k SVs, synth) on the device, random counters loaded for S samples, and a catalogue of R records (C2's VCF body
   repeated).  The step is genotype_cohort_vcf (genotype kernel, site statistics of all nine tags, text made and
   dropped); with the switches also the pack kernel per block, the pair kernel, the copies back and both tables'
   text.
2. The pair kernel alone at S in --pair-samples over min(1 M, --pair-cells / S) records of bit planes (all ./.: the
   kernel's time does not depend on the bits), timed by torch.profiler (device time of cohort_pair_kernel), with the
   work 5 popcounts x S (S - 1) / 2 x words reported as POPC per second.

The card's name, power limit and max SM clock are printed with the numbers.

    python profiles/cohort_qc_timing.py --out DIR [--cases 1000000x64,100000x4096] [--pair-samples 1024,4096,16384]
"""
import argparse
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


class _Sink:
    def write(self, b):
        return len(b)


def one_case(tables, vcf_text, n_rec, n_samples, runs):
    import numpy as np

    from svjg import cohort, genotype
    rng = np.random.default_rng(3)
    body = [ln for ln in vcf_text.splitlines(True) if not ln.startswith("#")]
    head = "".join(ln for ln in vcf_text.splitlines(True) if ln.startswith("#"))
    reps = -(-n_rec // len(body))
    lines = body * reps
    v = genotype.NativeVcf.from_input((head + "".join(lines[:n_rec])).encode())
    co = cohort.Cohort(tables, n_samples)
    for s in range(n_samples):
        c = rng.integers(0, 40, (tables.num_sv, 2)).astype(np.uint32)
        c[rng.random(tables.num_sv) < 0.3, 0] = 0
        c[rng.random(tables.num_sv) < 0.3, 1] = 0
        co.load_counts(s, c)
    names = [f"s{k}" for k in range(n_samples)]
    tags = cohort.INFO_TAGS

    def one_pass(qc):
        t0 = time.perf_counter()
        res = cohort.genotype_cohort_vcf(tables, co, v, names, out=_Sink(), info_tags=tags, sample_qc=qc,
                                         relatedness=qc)
        t1 = time.perf_counter()
        if qc:
            cohort.sample_qc_text(names, res[2])
            cohort.write_relatedness(_Sink(), names, res[3])
        return t1 - t0, time.perf_counter() - t1

    one_pass(False)
    one_pass(True)                                                          # warm-up
    times = {False: [], True: []}
    tables_s = []
    for _ in range(runs):
        for qc in (False, True):
            step, text = one_pass(qc)
            times[qc].append(step + text)
            if qc:
                tables_s.append(text)
    co.close()
    med = {p: sorted(t)[len(t) // 2] for p, t in times.items()}
    return {"records": n_rec, "samples": n_samples, "wall_s_plain": sorted(times[False]),
            "wall_s_qc": sorted(times[True]), "median_plain_s": med[False], "median_qc_s": med[True],
            "added_fraction": med[True] / med[False] - 1, "qc_table_text_s": sorted(tables_s)}


def pair_kernel(tables, n_samples, n_rec, runs):
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile

    from svjg import capi, cohort
    co = cohort.Cohort(tables, n_samples)
    words = -(-n_rec // 32)
    capi.check(capi.lib.svjg_cohort_qc_begin(co._h, words, 1))
    _fill_words(co, words)
    pairs = np.zeros((n_samples * (n_samples - 1) // 2, 5), np.uint32)
    walls, kern = [], []
    for k in range(runs + 1):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            t0 = time.perf_counter()
            capi.check(capi.lib.svjg_cohort_relatedness(co._h, pairs.ctypes.data))
            wall = time.perf_counter() - t0
        us = sum(getattr(ev, "device_time_total", 0) or ev.cuda_time_total for ev in prof.events()
                 if ev.device_type == torch.autograd.DeviceType.CUDA and "cohort_pair_kernel" in ev.name)
        if k:                                                                 # the first is the warm-up
            walls.append(wall)
            kern.append(us / 1e6)
    co.close()
    popc = 5 * n_samples * (n_samples - 1) // 2 * words
    ks = sorted(kern)[len(kern) // 2]
    return {"samples": n_samples, "records": 32 * words, "words": words, "pairs": n_samples * (n_samples - 1) // 2,
            "popc": popc, "kernel_s": sorted(kern), "median_kernel_s": ks, "popc_per_s": popc / ks,
            "call_wall_s": sorted(walls), "pair_bytes_copied": pairs.nbytes}


def _fill_words(co, words):
    """Packs `words` words of every sample's planes through the cohort's own path: blocks of whole words of records
    outside the gate (all ./.; the pair kernel's time does not depend on the bits), at most 2^25 cells a block."""
    import numpy as np

    from svjg import capi, cohort, genotype
    per = max(1, (1 << 25) // (32 * co.n_samples))                          # words per block
    idx = np.full(32 * per, capi.NO_SV, np.uint32)
    ty = np.zeros(32 * per, np.uint8)
    blk = cohort._Block(len(idx) * co.n_samples)
    done = 0
    while done < words:
        n = 32 * min(per, words - done)
        cohort._genotype_block(co, idx[:n], ty[:n], 3, genotype.ERR, blk)
        capi.check(capi.lib.svjg_cohort_qc_add(co._h, n))
        done += n // 32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cases", default="1000000x64,100000x4096")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--pair-samples", default="1024,4096,16384")
    ap.add_argument("--pair-cells", type=float, default=1e9,
                    help="records of the pair kernel runs: this many cells over S, at most 1 M")
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
    result["pair_kernel"] = []
    for s in (int(x) for x in args.pair_samples.split(",") if x):
        result["pair_kernel"].append(pair_kernel(tables, s, min(1_000_000, int(args.pair_cells) // s), args.runs))
        print(json.dumps(result["pair_kernel"][-1]), flush=True)
    vcf_text = synth.vcf_text(rows)
    result["cases"] = []
    for case in (c for c in args.cases.split(",") if c):
        r, s = (int(x) for x in case.split("x"))
        result["cases"].append(one_case(tables, vcf_text, r, s, args.runs))
        print(json.dumps(result["cases"][-1]), flush=True)
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    with open(os.path.join(args.out, "cohort_qc_timing.json"), "w") as fh:
        fh.write(text + "\n")


if __name__ == "__main__":
    main()
