"""Cost of the relationship matrix and the PCA (genotype-cohort.py --grm / --pca).

1. The GRM kernels alone at S in --grm-samples over min(1 M, --grm-cells / S) records: random counters loaded for S
   samples of C2's catalogue (25 k SVs, synth), the records genotyped and packed into the bit planes block by block
   through the cohort path, then svjg_cohort_grm timed by torch.profiler (device time of cohort_grm_kernel and
   cohort_grm_prep_kernel).  The work S (S + 1) / 2 x records (every record of a word with a used record costs the
   same) is reported as pair-records per second.  The host numpy.linalg.eigh of the resulting S x S matrix is timed
   once per S (cohort.pca with 10 components).
2. The genotype + VCF text step with and without --grm --pca, alternating (median of --runs each): the same counters
   over a catalogue of R records (C2's VCF body repeated).  The step is genotype_cohort_vcf (genotype kernel, site
   statistics of all nine tags, text made and dropped); with the switches also the pack kernel per block, both GRM
   kernels, the copy back, the PCA and the five files' bytes (made and dropped).

The card's name, power limit and max SM clock are printed with the numbers.

    python profiles/cohort_grm_timing.py --out DIR [--cases 1000000x64,100000x4096] [--grm-samples 1024,4096,16384]
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


def _load_random_counters(tables, co, seed=3):
    import numpy as np
    rng = np.random.default_rng(seed)
    for s in range(co.n_samples):
        c = rng.integers(0, 40, (tables.num_sv, 2)).astype(np.uint32)
        c[rng.random(tables.num_sv) < 0.3, 0] = 0
        c[rng.random(tables.num_sv) < 0.3, 1] = 0
        co.load_counts(s, c)


def one_case(tables, vcf_text, n_rec, n_samples, runs):
    from svjg import cohort, genotype
    body = [ln for ln in vcf_text.splitlines(True) if not ln.startswith("#")]
    head = "".join(ln for ln in vcf_text.splitlines(True) if ln.startswith("#"))
    lines = body * -(-n_rec // len(body))
    v = genotype.NativeVcf.from_input((head + "".join(lines[:n_rec])).encode())
    co = cohort.Cohort(tables, n_samples)
    _load_random_counters(tables, co)
    names = [f"s{k}" for k in range(n_samples)]
    k = min(10, n_samples)

    def one_pass(grm):
        t0 = time.perf_counter()
        res = cohort.genotype_cohort_vcf(tables, co, v, names, out=_Sink(), info_tags=cohort.INFO_TAGS, grm=grm)
        t1 = time.perf_counter()
        if grm:
            G, N = res[4]
            cohort.write_grm(_Sink(), _Sink(), _Sink(), names, G, N)
            vals, vecs = cohort.pca(G, k)
            cohort.write_pca(_Sink(), _Sink(), names, vals, vecs)
        return t1 - t0, time.perf_counter() - t1

    one_pass(False)
    one_pass(True)                                                          # warm-up
    times = {False: [], True: []}
    after = []
    for _ in range(runs):
        for grm in (False, True):
            step, rest = one_pass(grm)
            times[grm].append(step + rest)
            if grm:
                after.append(rest)
    co.close()
    med = {p: sorted(t)[len(t) // 2] for p, t in times.items()}
    return {"records": n_rec, "samples": n_samples, "wall_s_plain": sorted(times[False]),
            "wall_s_grm_pca": sorted(times[True]), "median_plain_s": med[False], "median_grm_pca_s": med[True],
            "added_fraction": med[True] / med[False] - 1, "files_and_pca_s": sorted(after)}


def grm_kernel(tables, n_samples, n_rec, runs):
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile

    from svjg import capi, cohort, genotype
    co = cohort.Cohort(tables, n_samples)
    _load_random_counters(tables, co)
    per = max(32, (1 << 25) // n_samples // 32 * 32)                       # records per block, whole words
    words = sum(-(-min(per, n_rec - lo) // 32) for lo in range(0, n_rec, per))
    capi.check(capi.lib.svjg_cohort_qc_begin(co._h, words, 1))
    idx = (np.arange(n_rec) % tables.num_sv).astype(np.uint32)
    ty = np.zeros(n_rec, np.uint8)
    blk = cohort._Block(per * n_samples)
    for lo in range(0, n_rec, per):
        hi = min(n_rec, lo + per)
        cohort._genotype_block(co, idx[lo:hi], ty[lo:hi], 3, genotype.ERR, blk)
        capi.check(capi.lib.svjg_cohort_qc_add(co._h, hi - lo))
    P = n_samples * (n_samples + 1) // 2
    g = np.zeros(P)
    nn = np.zeros(P, np.uint32)
    walls, kern, prep = [], [], []
    for k in range(runs + 1):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            t0 = time.perf_counter()
            capi.check(capi.lib.svjg_cohort_grm(co._h, 0.01, g.ctypes.data, nn.ctypes.data))
            wall = time.perf_counter() - t0
        dev = {}
        for ev in prof.events():
            if ev.device_type == torch.autograd.DeviceType.CUDA:
                for name in ("cohort_grm_prep_kernel", "cohort_grm_kernel"):
                    if name in ev.name:
                        dev[name] = dev.get(name, 0) + (getattr(ev, "device_time_total", 0) or ev.cuda_time_total)
        if k:                                                                 # the first is the warm-up
            walls.append(wall)
            kern.append(dev.get("cohort_grm_kernel", 0) / 1e6)
            prep.append(dev.get("cohort_grm_prep_kernel", 0) / 1e6)
    co.close()
    G = cohort.grm_square(g, n_samples, np.float64)
    diag_n = cohort.grm_square(nn, n_samples, np.uint32).diagonal()
    t0 = time.perf_counter()
    cohort.pca(G, 10)
    eigh_s = time.perf_counter() - t0
    pair_records = P * 32 * words
    ks = sorted(kern)[len(kern) // 2]
    return {"samples": n_samples, "records": n_rec, "words": words, "pairs": P,
            "used_records_max_n": int(diag_n.max()), "pair_records": pair_records, "kernel_s": sorted(kern),
            "median_kernel_s": ks, "pair_records_per_s": pair_records / ks, "prep_kernel_s": sorted(prep),
            "call_wall_s": sorted(walls), "bytes_copied": g.nbytes + nn.nbytes, "host_pca_eigh_s": eigh_s,
            "host_threads": os.cpu_count()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--cases", default="1000000x64,100000x4096")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--grm-samples", default="1024,4096,16384")
    ap.add_argument("--grm-cells", type=float, default=1e9,
                    help="records of the GRM kernel runs: this many cells over S, at most 1 M")
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
    result["grm_kernel"] = []
    for s in (int(x) for x in args.grm_samples.split(",") if x):
        result["grm_kernel"].append(grm_kernel(tables, s, min(1_000_000, int(args.grm_cells) // s), args.runs))
        print(json.dumps(result["grm_kernel"][-1]), flush=True)
    vcf_text = synth.vcf_text(rows)
    result["cases"] = []
    for case in (c for c in args.cases.split(",") if c):
        r, s = (int(x) for x in case.split("x"))
        result["cases"].append(one_case(tables, vcf_text, r, s, args.runs))
        print(json.dumps(result["cases"][-1]), flush=True)
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    with open(os.path.join(args.out, "cohort_grm_timing.json"), "w") as fh:
        fh.write(text + "\n")


if __name__ == "__main__":
    main()
