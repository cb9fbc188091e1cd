#!/usr/bin/env python3
"""bench.py — throughput of the B200 hot path (GAF filter + allele counts + genotype) on the
BASELINE.json workload, one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C2] [--scale 1.0] [--catalogue full]
    python bench.py --impl reference ...      # CPU arm: the UNMODIFIED reference scripts on the host cores
    torchrun ... bench.py --gpus N [--scaling strong]
    python bench.py --dump-outputs DIR ...    # also write what the last timed step computed as DIR/<name>.npy

A "step" is one pass of the hot path over one batch of synthetic GAF (one file of the named config per
GPU): counters reset -> filter chain (probe, scan, exact kernels) -> counters of all ranks summed (inside
the genotype kernel over NVLink peer memory, or ncclAllReduce) -> genotype kernel.
`value`  alignments/s with the batch resident in HBM (CUDA events, max over ranks).
`e2e`    the same job through the C ABI with HOST buffers: pinned GAF bytes in ->
         `informative_aln.json` bytes + `genotype.vcf` bytes out, in host memory; every copy, the JSON
         text and the VCF text inside the timed region; two batches in flight (the text of batch k is copied
         back while batch k + 1 is uploaded), `one_batch_at_a_time` beside it.  At N > 1: one such job per GPU at once.
`--scaling strong`: ONE batch cut by bytes at line ends over the N ranks (svjg.shard.shard_cuts), the
         hits of all ranks checked against a one-GPU pass over the whole batch before timing.
"""
import argparse
import ctypes as C
import io
import json
import math
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "svjedi-graph_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "gaf_alignments_filtered_assigned_per_sec"
UNIT = "alignments/s"
REF_DIR = os.path.join(ROOT, "baseline", "_ref")          # the three unmodified scripts, copied by __graft_entry__.build()
REF_SCRIPTS = ("filter-alignments.py", "predict-genotype.py")
DUMP_BYTES = 60_000_000   # --dump-outputs: the arrays of all files together; with the .npy headers below 64 MB
DUMP_SEED = 20240601      # rows kept where an output is larger than its share


def at_least_one(text):
    n = int(text)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {n}")
    return n


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=at_least_one, default=100, help="timed steps of the hot path")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="C2", choices=["C2", "C3", "C4", "C5"])
    ap.add_argument("--scale", type=float, default=None, help="shrink SV and record counts (default: full; C5: per-GPU shard)")
    ap.add_argument("--catalogue", default="scaled", choices=["scaled", "full"],
                    help="full: the SV catalogue (and genome) at the config's stated size whatever --scale says; "
                         "C5 then probes its 1 M-SV tables (459 MB, beyond L2) with a --scale shard of the records")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: one batch per GPU (weak), or one batch cut by bytes over the GPUs (strong)")
    ap.add_argument("--e2e-steps", type=int, default=None)
    ap.add_argument("--kernel-only", action="store_true", help="developer mode: print the kernel times and stop")
    ap.add_argument("--cpu-sample", type=int, default=20_000, help="records per host process the CPU arm is timed on")
    ap.add_argument("--scan-blocks", type=int, default=0, help="developer: blocks per SM the scan kernel is sized for (6 or 8)")
    ap.add_argument("--tile-lines", type=int, default=0, help="developer: lines a tile of the scan kernel should hold")
    ap.add_argument("--collective", default="p2p", choices=["p2p", "nccl"],
                    help="N > 1: counters summed inside the genotype kernel over NVLink peer memory (p2p), or ncclAllReduce")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="one GPU: write the counters, hit tuples and genotype arrays of the last timed step to DIR/<name>.npy "
                         "(float64, at most 64 MB in all: a larger array is cut to the same seeded sample of rows every run)")
    return ap.parse_args()


def dump_outputs(out_dir, arrays):
    """Writes each array of ``arrays`` (name -> numpy array, rows first) as ``out_dir/<name>.npy`` in float64, which
    holds every integer the path computes exactly.  Each array gets an equal share of DUMP_BYTES; one with more rows
    than fit keeps a sorted sample drawn with DUMP_SEED, so arrays of equal length keep the same rows and two builds
    that compute the same thing write the same files.  Returns name -> (rows written, rows computed)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays))
    kept = {}
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64)
        n_max = share // (8 * max(1, int(np.prod(a.shape[1:]))))
        if len(a) > n_max:
            rows = np.random.default_rng(DUMP_SEED).choice(len(a), size=n_max, replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
        kept[name] = (len(a), len(arrays[name]))
    return kept


def workload(args, stream):
    """Synthetic batch of the named config.  Tables are identical on every rank; `stream` selects the reads."""
    from svjg import synth
    scale = args.scale
    if scale is None:
        # C5 (1M SVs / 200M records over 8 GPUs) is sized per GPU: 1/8 of the records would be 25 M; 4 M by default
        scale = 1.0 if args.workload != "C5" else 0.02
    t0 = time.time()
    # synthetic inputs are deterministic; keep them for later runs on the same box (untimed either way)
    import pickle
    cscale = 1.0 if args.catalogue == "full" else None
    cache = os.path.join(os.environ.get("SVJG_CACHE", "/tmp"), f"svjg_wl_{args.workload}_{scale:g}_{args.catalogue}_{stream}.pkl")
    if os.path.exists(cache):
        with open(cache, "rb") as fh:
            g, vcf, gaf = pickle.load(fh)
    else:
        g, vcf, gaf = synth.make_workload(args.workload, scale=scale, stream0=stream, catalogue_scale=cscale)
        try:
            with open(cache + f".{os.getpid()}", "wb") as fh:
                pickle.dump((g, vcf, gaf), fh, protocol=pickle.HIGHEST_PROTOCOL)
            os.replace(cache + f".{os.getpid()}", cache)
        except Exception:
            pass
    buf = io.StringIO()
    g.write_gfa(buf)
    return g, vcf, gaf, buf.getvalue(), scale, time.time() - t0


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum of the filter chain per launch, from the ncu --set full
    captures summarised under profiles/ (profiles/ncu_traffic.py writes the table); None where no capture exists."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            return json.load(fh).get(key, {}).get("dram_bytes")
    except Exception:
        return None


class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50", "-i", str(index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        inside = [r for t, r in self.rows if t0 <= t <= t1 + 0.06] or [r for _, r in self.rows[-3:]]
        sm, mx, reasons = [], None, set()
        for r in inside:
            f = [x.strip() for x in r.split(",")]
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except Exception:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU arm: the unmodified reference scripts (baseline/_ref/, copied from /root/reference by build())
# as subprocesses with their own command lines; the oracle port only where they are not there
# --------------------------------------------------------------------------------------------------
GT_SAMPLE = 4000          # SV lines the reference genotyper is timed on where the catalogue is beyond 100 k (cpu_arm)


def reference_available():
    return all(os.path.exists(os.path.join(REF_DIR, s)) for s in REF_SCRIPTS)


def first_lines(text, n):
    pos = 0
    for _ in range(n):
        j = text.find("\n", pos)
        if j < 0:
            return text
        pos = j + 1
    return text[:pos]


class ReferenceRun:
    """One directory with the inputs of filter-alignments.py / predict-genotype.py as files:
    `<tmp>/wl.gfa`, `<tmp>/wl.vcf`, and per shard k `<tmp>/s<k>.gaf` + `<tmp>/s<k>_svs_edges.json` (a link to
    the one table file; the script finds it through its -p prefix, filter-alignments.py:78)."""

    def __init__(self, gaf_text, edges_text, gfa_text, vcf_text, n_procs, per_proc):
        self.dir = tempfile.mkdtemp(prefix="svjg_ref_")
        self.n_procs = n_procs
        with open(os.path.join(self.dir, "wl.gfa"), "w") as fh:
            fh.write(gfa_text)
        with open(os.path.join(self.dir, "wl.vcf"), "w") as fh:
            fh.write(vcf_text)
        with open(os.path.join(self.dir, "edges.json"), "w") as fh:
            fh.write(edges_text)
        sample = first_lines(gaf_text, n_procs * per_proc)
        lines = sample.splitlines(True)
        self.n_sample = len(lines)
        share = (len(lines) + n_procs - 1) // n_procs
        for k in range(n_procs):
            with open(os.path.join(self.dir, f"s{k}.gaf"), "w") as fh:
                fh.writelines(lines[k * share:(k + 1) * share])
            os.symlink("edges.json", os.path.join(self.dir, f"s{k}_svs_edges.json"))
        open(os.path.join(self.dir, "empty.gaf"), "w").close()
        os.symlink("edges.json", os.path.join(self.dir, "empty_svs_edges.json"))

    def _filter(self, tags):
        procs = [subprocess.Popen([sys.executable, os.path.join(REF_DIR, "filter-alignments.py"), "-a", f"{t}.gaf", "-g", "wl.gfa",
                                   "-p", t], cwd=self.dir, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE) for t in tags]
        for p in procs:
            _, err = p.communicate()
            if p.returncode:
                raise SystemExit("reference filter-alignments.py failed: " + err.decode()[-300:])

    def startup_seconds(self):
        """filter-alignments.py on an empty GAF: interpreter start + table load, which do not grow with the records"""
        t0 = time.perf_counter()
        self._filter(["empty"])
        return time.perf_counter() - t0

    def step(self):
        """(seconds of the line-sharded filter processes, seconds of predict-genotype.py on the merged JSON)"""
        t0 = time.perf_counter()
        self._filter([f"s{k}" for k in range(self.n_procs)])
        t1 = time.perf_counter()
        # harness, untimed: per-key lists concatenated in shard order = what one process would have appended (:166)
        merged = {}
        for k in range(self.n_procs):
            with open(os.path.join(self.dir, f"s{k}_informative_aln.json")) as fh:
                for key, (ref, alt) in json.load(fh).items():
                    m = merged.setdefault(key, [[], []])
                    m[0] += ref
                    m[1] += alt
        with open(os.path.join(self.dir, "merged.json"), "w") as fh:
            fh.write(json.dumps(merged, sort_keys=True, indent=4))
        t2 = time.perf_counter()
        r = subprocess.run([sys.executable, os.path.join(REF_DIR, "predict-genotype.py"), "-d", "merged.json", "-v", "wl.vcf",
                            "-o", "out.vcf"], cwd=self.dir, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
        if r.returncode:
            raise SystemExit("reference predict-genotype.py failed: " + r.stderr.decode()[-300:])
        return t1 - t0, time.perf_counter() - t2

    def close(self):
        shutil.rmtree(self.dir, ignore_errors=True)


_PORT = None


def _port_shard(k):
    from oracle import svjg_oracle as O
    d = O.filter_alignments(_PORT[0][k], _PORT[1], _PORT[2])
    O.dumps_informative(d)
    return O.hit_counts(d)


def port_step(lines_by_shard, edges, alt, vcf_lines):
    """The oracle port in forked workers: only when baseline/_ref/ is not there."""
    import multiprocessing as mp
    from oracle import svjg_oracle as O
    global _PORT
    _PORT = (lines_by_shard, edges, alt)
    t0 = time.perf_counter()
    with mp.get_context("fork").Pool(len(lines_by_shard)) as pool:
        parts = pool.map(_port_shard, range(len(lines_by_shard)), chunksize=1)
    counts = {}
    for c in parts:
        for k, (a, b) in c.items():
            x = counts.get(k, (0, 0))
            counts[k] = (x[0] + a, x[1] + b)
    t1 = time.perf_counter()
    O.genotype_vcf(counts, vcf_lines)
    return t1 - t0, time.perf_counter() - t1


def cpu_arm(gaf_text, edges_text, gfa_text, vcf_text, n_rec, n_procs, per_proc, steps, warmup):
    """Times `steps` steps of the CPU implementation on a bounded sample: n_procs processes x per_proc records
    through the filter (+ JSON), then the genotyper over the whole VCF.  Returns the projection to the whole
    batch: the filter grows with the records, its start-up and the genotyper do not."""
    # predict-genotype.py builds the list of the dictionary's keys once per VCF line (:216): hours at a million SVs.
    # Beyond 100 k SVs its leg runs on the first GT_SAMPLE SV lines and is projected by lines (the per-line cost,
    # one pass over the same keys, does not change).
    n_sv_lines = sum(1 for ln in vcf_text.splitlines() if ln and not ln.startswith("#"))
    gt_scale = 1.0
    if n_sv_lines > 100_000:
        kept, n_kept = [], 0
        for ln in vcf_text.splitlines(True):
            if not ln.startswith("#"):
                if n_kept == GT_SAMPLE:
                    break
                n_kept += 1
            kept.append(ln)
        vcf_text = "".join(kept)
        gt_scale = n_sv_lines / GT_SAMPLE
    if reference_available():
        run = ReferenceRun(gaf_text, edges_text, gfa_text, vcf_text, n_procs, per_proc)
        try:
            t0 = run.startup_seconds()
            tf, tg = [], []
            for i in range(warmup + steps):
                a, b = run.step()
                if i >= warmup:
                    tf.append(a)
                    tg.append(b)
            n_sample = run.n_sample
        finally:
            run.close()
        kind = "reference"
        what = "unmodified filter-alignments.py + predict-genotype.py (baseline/_ref) as subprocesses"
    else:
        lines = first_lines(gaf_text, n_procs * per_proc).splitlines(True)
        share = (len(lines) + n_procs - 1) // n_procs
        shards = [lines[k * share:(k + 1) * share] for k in range(n_procs)]
        alt = {}
        for line in gfa_text.splitlines(True):
            if line.startswith("S"):
                c = line.split("\t")
                if "." in c[1].split(":")[-1]:
                    alt[c[1]] = len(line.rstrip().split("\t")[2])
        edges = json.loads(edges_text)
        vcf_lines = vcf_text.splitlines(True)
        t0, tf, tg = 0.0, [], []
        for i in range(warmup + steps):
            a, b = port_step(shards, edges, alt, vcf_lines)
            if i >= warmup:
                tf.append(a)
                tg.append(b)
        n_sample = len(lines)
        kind = "port"
        what = "oracle/svjg_oracle.py in forked workers (baseline/_ref is not there)"
    f = sum(tf) / len(tf)
    gsec = sum(tg) / len(tg) * gt_scale
    if gt_scale != 1.0:
        what += f"; genotyper timed on the first {GT_SAMPLE} of {n_sv_lines} SV lines and projected by lines"
    start = min(t0, f)
    projected = start + (f - start) * n_rec / max(1, n_sample) + gsec
    return {"value": n_rec / projected, "kind": kind, "what": what, "n_sample": n_sample, "filter_s": f, "startup_s": start,
            "genotype_s": gsec, "step_s": f + gsec, "projected_s": projected}


def cpu_baseline_c(gaf_text, edges_text, gfa_text, n_sample=None, check=None):
    """The C restatement of the reference filter (oracle/svjg_oracle.c) on the host cores: filter only
    (no JSON text, no genotypes), one thread and all threads.  An extra line of context beside
    cpu_baseline, never the thing measured.  ``check`` = (sv ids, counters [num_sv, 2], number of hits) of
    the GPU path for the same batch: the whole batch is then compared counter by counter (key "parity")."""
    try:
        from oracle import c_oracle as CO
        CO.ensure_built()
        alt = {}
        for line in gfa_text.splitlines(True):
            if line.startswith("S"):
                c = line.split("\t")
                if "." in c[1].split(":")[-1]:
                    alt[c[1]] = len(line.rstrip().split("\t")[2])
        t = CO.Tables(json.loads(edges_text), alt)
        if n_sample:
            gaf_text = first_lines(gaf_text, n_sample)
        gaf = gaf_text.encode()
        n_rec = gaf.count(b"\n")
        cores = min(32, os.cpu_count() or 1)
        out = {"unit": UNIT, "kind": "port (C)", "records": n_rec, "what": "oracle/svjg_oracle.c, filter + counters + hit tuples only"}
        for label, th in (("one_thread", 1), ("all_threads", cores)):
            t0 = time.perf_counter()
            counts, st = CO.filter_counts(t, gaf, threads=th)
            out[label] = {"value": st["n_records"] / (time.perf_counter() - t0), "threads": th}
        if check is not None:
            ids, got, n_hits = check
            same = list(ids) == list(t.sv_ids) and got.shape == counts.shape and bool((got == counts).all()) \
                and int(n_hits) == st["n_hits"]
            out["parity"] = {"ok": same, "checked": f"all {n_rec} records of rank 0's batch: {counts.shape[0]} x 2 counters and the "
                                                     f"number of hits ({st['n_hits']}) against the C oracle, bit for bit"}
        return out
    except Exception as exc:                      # context only: never fails the bench
        return {"unavailable": f"{type(exc).__name__}: {exc}"[:200]}


def run_reference(args):
    """CPU arm of the driver: rank 0 alone, all host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    g, vcf, gaf, gfa_text, scale, gen_s = workload(args, 0)
    edges_text = g.edges_json()
    n_vcf = sum(1 for l in vcf.splitlines() if l and not l.startswith("#"))
    n_rec = gaf.count("\n")
    cores = max(1, os.cpu_count() or 1)
    per_proc = max(1000, min(args.cpu_sample, n_rec // cores))
    r = cpu_arm(gaf, edges_text, gfa_text, vcf, n_rec, cores, per_proc, args.steps, args.warmup)
    sample = (f"{r['n_sample']} records per step ({cores} processes x {per_proc}) through the filter ({r['filter_s']:.2f} s, of which "
              f"start-up {r['startup_s']:.2f} s) projected to {n_rec} records, plus the genotyper over all {n_vcf} SVs once per step "
              f"({r['genotype_s']:.2f} s, one process: it is quadratic in the SVs); {r['what']}")
    line = {
        "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000 * r["step_s"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic", "impl": "reference",
        "config": {"workload": f"{args.workload} x{scale:g}: {n_rec} GAF records, {n_vcf} VCF SVs ({r['n_sample']} records timed per step)"},
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": cores, "kind": r["kind"], "sample": sample},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "cpu_baseline_c": cpu_baseline_c(first_lines(gaf, r["n_sample"]), edges_text, gfa_text),
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist

    from svjg import alnfilter, capi, genotype, shard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU (there is no CPU fallback); use --impl reference for the CPU arm")
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs writes the outputs of one GPU: run it without torchrun")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    strong = args.scaling == "strong" and world > 1

    if args.scan_blocks:
        capi.check(capi.lib.svjg_filter_tune(capi.TUNE_SCAN_BLOCKS, args.scan_blocks))
    if args.tile_lines:
        capi.check(capi.lib.svjg_filter_tune(capi.TUNE_TILE_LINES, args.tile_lines))
    g, vcf, gaf, gfa_text, scale, gen_s = workload(args, 0 if strong else rank)
    edges_text = g.edges_json()
    tables = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(local)
    gaf_all = gaf.encode()
    whole, cuts = None, None
    if strong:
        # one batch, cut by bytes at line ends: rank r filters [cuts[r], cuts[r+1])
        cuts = shard.shard_cuts(gaf_all, world)
        whole = gaf_all
        gaf_bytes = gaf_all[cuts[rank]:cuts[rank + 1]]
    else:
        gaf_bytes = gaf_all
    n_bytes = len(gaf_bytes)
    n_rec = gaf_bytes.count(b"\n")
    h_gaf = torch.frombuffer(bytearray(gaf_bytes), dtype=torch.uint8).pin_memory()
    h_gaf_np = h_gaf.numpy()
    d_gaf = h_gaf.to(dev)

    # genotype inputs (host string work done once, untimed: it is per-catalogue, not per-read)
    nvcf = genotype.NativeVcf.from_input(vcf.encode())
    sv_idx = nvcf.index_tables(tables)
    sv_ty = nvcf.svtype
    n_sv = int(nvcf.n)
    lo, hi = (n_sv * rank) // world, (n_sv * (rank + 1)) // world      # SV shard of this rank
    n_loc = hi - lo
    d_idx = torch.from_numpy(sv_idx[lo:hi].view(np.int32).copy()).to(dev)
    d_ty = torch.from_numpy(sv_ty[lo:hi].copy()).to(dev)
    lut = torch.from_numpy(genotype.log10comb_lut()).to(dev)
    la, lb, lh = math.log10(1 - genotype.ERR), math.log10(genotype.ERR), math.log10(1 / 2)
    d_pl = torch.empty((max(1, n_loc), 3), dtype=torch.int64, device=dev)
    d_gt = torch.empty(max(1, n_loc), dtype=torch.uint8, device=dev)
    d_ad = torch.empty((max(1, n_loc), 2), dtype=torch.int32, device=dev)
    d_fl = torch.empty(max(1, n_loc), dtype=torch.uint8, device=dev)

    # size the hit buffers from one untimed pass
    filt = alnfilter.DeviceFilter(tables, hit_cap=1024, device=local)
    filt.reset()
    filt.run(d_gaf)                                   # the cursor counts every hit, stored or not
    st = filt.read_stats()
    if st["status"]:
        raise SystemExit(f"synthetic GAF rejected: {st}")
    n_hits = st["n_hits"]
    filt = alnfilter.DeviceFilter(tables, hit_cap=n_hits + 1024, device=local)
    stream = torch.cuda.current_stream(dev)
    sp = C.c_void_p(stream.cuda_stream)
    lib = capi.lib

    def hit_digest(sv2, off, ln, base):
        """order-free digest of a hit list (the kernels append in any order)"""
        with np.errstate(over="ignore"):
            x = (sv2.astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)) ^ ((off.astype(np.uint64) + np.uint64(base)) * np.uint64(0xC2B2AE3D27D4EB4F)) \
                ^ (ln.astype(np.uint64) * np.uint64(0x165667B19E3779F9))
            return (int(np.bitwise_xor.reduce(x)), int(x.sum(dtype=np.uint64))) if x.size else (0, 0)

    strong_check = None
    if strong:
        # the ranks' shards together must be the one-GPU result: counters summed, hit lists united
        filt.reset()
        filt.run(d_gaf)
        mine = filt.result()
        part = torch.from_numpy(mine.counts.view(np.int32).copy()).to(dev)
        dist.all_reduce(part)
        dx, ds = hit_digest(mine.hit_sv2, mine.hit_off, mine.hit_len, cuts[rank])
        dig = torch.tensor([dx & 0x7FFFFFFFFFFFFFFF, dx >> 63, ds & 0x7FFFFFFFFFFFFFFF, ds >> 63, mine.n_hits], dtype=torch.int64, device=dev)
        digs = [torch.zeros_like(dig) for _ in range(world)]
        dist.all_gather(digs, dig)
        if rank == 0:
            d_whole = torch.frombuffer(bytearray(whole), dtype=torch.uint8).to(dev)
            one = alnfilter.DeviceFilter(tables, hit_cap=sum(int(d[4]) for d in digs) + 1024, device=local)
            one.reset()
            one.run(d_whole)
            ref = one.result()
            wx, ws = hit_digest(ref.hit_sv2, ref.hit_off, ref.hit_len, 0)
            gx = gs = 0
            for d in digs:
                gx ^= int(d[0]) | (int(d[1]) << 63)
                gs = (gs + (int(d[2]) | (int(d[3]) << 63))) & 0xFFFFFFFFFFFFFFFF
            same = bool((part.cpu().numpy().view(np.uint32) == ref.counts).all()) and (gx, gs) == (wx, ws) \
                and sum(int(d[4]) for d in digs) == ref.n_hits
            strong_check = {"ok": same, "checked": f"counters and the united hit list of {world} byte-range shards against one GPU over "
                                                   f"the whole batch ({ref.n_hits} hits)"}
            if not same:
                raise SystemExit("strong scaling: the shards' results differ from the one-GPU result")
            del d_whole, one

    xchg = None
    if world > 1 and args.collective == "p2p":
        from svjg.shard import CounterExchange

        def gather_bytes(b):
            out = [None] * world
            dist.all_gather_object(out, b)
            return out
        xchg = CounterExchange(tables.num_sv, rank, world, gather_bytes)
    step_no = [0]
    # N > 1 with the fused exchange: the genotype kernel of step k waits (on the device) for the filter of the slowest
    # rank; it runs on a stream of its own so that this rank's filter of step k + 1 does not wait with it.  The three
    # counter buffers of the exchange region are taken in turn; step k + 3 reuses buffer k % 3 behind this rank's
    # genotype kernel of step k + 1 (include/svjg.h).
    side = torch.cuda.Stream(dev) if xchg else None
    side_p = C.c_void_p(side.cuda_stream) if xchg else None
    filt_done = [torch.cuda.Event() for _ in range(3)]
    geno_done = [torch.cuda.Event() for _ in range(3)]

    def step(ev=None):
        step_no[0] += 1
        k = step_no[0]
        # p2p: this rank's counters live in its exchange region (three buffers, taken in turn)
        counts_ptr = xchg.counts_ptr(k) if xchg else filt.counts.data_ptr()
        if xchg and k > 2:
            stream.wait_event(geno_done[(k - 2) % 3])      # every rank has read buffer k % 3 of step k - 3
        capi.check(lib.svjg_filter_reset(counts_ptr, tables.num_sv, filt.stats.data_ptr(), sp))
        if ev:
            ev[0].record(stream)
        capi.check(lib.svjg_filter_device(tables._h, d_gaf.data_ptr(), n_bytes, 0, 100, counts_ptr,
                                          filt.hit_sv2.data_ptr(), filt.hit_off.data_ptr(), filt.hit_len.data_ptr(),
                                          filt.hit_cap, filt.stats.data_ptr(), sp))
        if ev:
            ev[1].record(stream)
        if world > 1 and not xchg:
            dist.all_reduce(filt.counts)                   # per-SV REF/ALT counters, NCCL sum over NVLink
        if ev:
            ev[2].record(stream)
        if xchg:
            # announces this rank's counters, waits on the device for all ranks, then sums their counters
            # where they lie (NVLink peer reads): all-reduce and genotype step in one kernel
            filt_done[k % 3].record(stream)
            side.wait_event(filt_done[k % 3])
            xchg.genotype(k, d_idx.data_ptr(), d_ty.data_ptr(), n_loc, 3, la, lb, lh, lut.data_ptr(), genotype.LUT_NMAX,
                          d_pl.data_ptr(), d_gt.data_ptr(), d_ad.data_ptr(), d_fl.data_ptr(), side_p)
            geno_done[k % 3].record(side)
            if ev:
                ev[3].record(side)
        else:
            capi.check(lib.svjg_genotype_device(filt.counts.data_ptr(), d_idx.data_ptr(), d_ty.data_ptr(), n_loc, 3, la, lb, lh,
                                                lut.data_ptr(), genotype.LUT_NMAX, None, d_pl.data_ptr(), d_gt.data_ptr(),
                                                d_ad.data_ptr(), d_fl.data_ptr(), sp))
            if ev:
                ev[3].record(stream)

    def sync_all():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    if xchg:
        # untimed self-check of the fused exchange: NCCL all-reduce + plain genotype kernel must give the same
        capi.check(lib.svjg_filter_reset(filt.counts.data_ptr(), tables.num_sv, filt.stats.data_ptr(), sp))
        capi.check(lib.svjg_filter_device(tables._h, d_gaf.data_ptr(), n_bytes, 0, 100, filt.counts.data_ptr(),
                                          filt.hit_sv2.data_ptr(), filt.hit_off.data_ptr(), filt.hit_len.data_ptr(),
                                          filt.hit_cap, filt.stats.data_ptr(), sp))
        dist.all_reduce(filt.counts)
        capi.check(lib.svjg_genotype_device(filt.counts.data_ptr(), d_idx.data_ptr(), d_ty.data_ptr(), n_loc, 3, la, lb, lh,
                                            lut.data_ptr(), genotype.LUT_NMAX, None, d_pl.data_ptr(), d_gt.data_ptr(),
                                            d_ad.data_ptr(), d_fl.data_ptr(), sp))
        want = (d_pl.clone(), d_gt.clone(), d_ad.clone(), d_fl.clone())
        d_pl.zero_(), d_gt.zero_(), d_ad.zero_(), d_fl.zero_()
        step()
        torch.cuda.synchronize(dev)
        got = (d_pl, d_gt, d_ad, d_fl)
        if xchg.timed_out() or not all(torch.equal(a, b) for a, b in zip(want, got)):
            raise SystemExit(f"rank {rank}: fused counter exchange disagrees with NCCL all-reduce + genotype")
    for _ in range(max(3, args.warmup)):
        step()
    sync_all()
    K = args.steps
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local) if rank == 0 else None
    time.sleep(0.15)
    t_wall0 = time.time()
    e0.record(stream)
    for k in range(K):
        step(evs[k])
    if side is not None:
        stream.wait_stream(side)                           # the last genotype kernels belong to the timed steps
    e1.record(stream)
    sync_all()
    t_wall1 = time.time()
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    total_ms = e0.elapsed_time(e1)
    filt_ms = sum(e[0].elapsed_time(e[1]) for e in evs) / K
    comm_ms = sum(e[1].elapsed_time(e[2]) for e in evs) / K
    geno_ms = sum(e[2].elapsed_time(e[3]) for e in evs) / K     # with the fused exchange: until every rank's counters were there
    if world > 1:
        t = torch.tensor([total_ms, filt_ms, geno_ms, comm_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, filt_ms, geno_ms, comm_ms = t.tolist()
        tot = torch.tensor([n_rec, n_bytes, n_hits], dtype=torch.int64, device=dev)
        dist.all_reduce(tot)
        job_rec, job_bytes, job_hits = (int(x) for x in tot)
    else:
        job_rec, job_bytes, job_hits = n_rec, n_bytes, n_hits
    st = filt.read_stats()
    if xchg and xchg.timed_out():
        raise SystemExit(f"rank {rank}: a wait in the fused counter exchange timed out")
    dumped = None
    if args.dump_outputs:
        # the last timed step's results, read before the measurements below launch on the same buffers
        nh = st["n_hits"]
        if st["status"] or nh > filt.hit_cap:
            raise SystemExit(f"--dump-outputs: the last timed step did not complete: {st}")
        sv2 = filt.hit_sv2[:nh].cpu().numpy().view(np.uint32)
        off = filt.hit_off[:nh].cpu().numpy().view(np.uint32)
        ln = filt.hit_len[:nh].cpu().numpy().view(np.uint32)
        order = np.lexsort((ln, sv2, off))               # the kernels append hits in any order: sorted into file order
        dumped = dump_outputs(args.dump_outputs, {
            "counts": filt.counts[:tables.num_sv].cpu().numpy().view(np.uint32),
            "hit_sv2": sv2[order], "hit_off": off[order], "hit_len": ln[order],
            "genotype_gt": d_gt[:n_loc].cpu().numpy(), "genotype_flags": d_fl[:n_loc].cpu().numpy(),
            "genotype_ad2": d_ad[:n_loc].cpu().numpy().view(np.uint32), "genotype_pl": d_pl[:n_loc].cpu().numpy(),
        })

    # the dominant kernel on its own: the library records CUDA events around its scan kernel on this stream
    def timed_scan(n_iter):
        capi.check(lib.svjg_filter_profile(1))
        tot_ms, ms = 0.0, C.c_float()
        for _ in range(n_iter):
            capi.check(lib.svjg_filter_reset(filt.counts.data_ptr(), tables.num_sv, filt.stats.data_ptr(), sp))
            capi.check(lib.svjg_filter_device(tables._h, d_gaf.data_ptr(), n_bytes, 0, 100, filt.counts.data_ptr(),
                                              filt.hit_sv2.data_ptr(), filt.hit_off.data_ptr(), filt.hit_len.data_ptr(),
                                              filt.hit_cap, filt.stats.data_ptr(), sp))
            capi.check(lib.svjg_filter_scan_ms(C.byref(ms)))
            tot_ms += ms.value
        capi.check(lib.svjg_filter_profile(0))
        return tot_ms / n_iter
    timed_scan(2)
    scan_ms = timed_scan(max(3, min(K, 10)))
    if args.kernel_only:
        if rank == 0:
            print(json.dumps({"kernel_ms": {"filter": filt_ms, "allreduce": comm_ms, "genotype": geno_ms}, "scan_ms": scan_ms,
                              "GBps": n_bytes / filt_ms / 1e6, "stats": st, "strong_check": strong_check}))
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- end to end through the C ABI with host buffers: pinned GAF bytes in, JSON bytes + VCF bytes out
    Ke = args.e2e_steps or max(3, min(K, 20))
    host_out = alnfilter.HostBuffers(tables, n_hits + 1024)     # pinned result arrays, allocated once like h_gaf
    out_bytes = [0, 0]

    from concurrent.futures import ThreadPoolExecutor
    side_pool = ThreadPoolExecutor(4)
    # two batches in flight, like a run over several samples: a second handle of the same tables (own workspace and
    # streams) takes every other batch, so the text of batch k is rendered and copied back (D2H) and its genotypes
    # and VCF text are made while batch k + 1 is uploaded (H2D) and filtered.  Every batch still pays all of its
    # copies inside the timed region.
    handles = [tables, tables.clone().to_device(dev.index)]
    host_out2 = alnfilter.HostBuffers(tables, 16)
    counts_of = [host_out.counts, host_out2.counts]
    text_job, vcf_job = [None, None], [None, None]

    def take(b):
        """the results of the batch that used handle b last are in host memory"""
        if text_job[b] is not None:
            js = text_job[b].result()
            text_job[b] = None
            if js is None:
                raise SystemExit("the device JSON renderer declined the synthetic batch")
            out_bytes[0] = len(js)
        if vcf_job[b] is not None:
            out_bytes[1] = vcf_job[b].result()
            vcf_job[b] = None

    def vcf_of(counts):
        # the counters are genotyped and genotype.vcf is written (predict-genotype.py:216-275)
        gt, fl, ad, pl = genotype.genotype_host(counts, sv_idx, sv_ty)
        vt, n_gt = nvcf.format_buffer(gt, fl, ad, pl)
        return vt.nbytes

    def e2e_step(k, overlap):
        b = k & 1 if overlap else 0
        take(b)                             # batch k - 2 is done before its handle and its counters are used again
        # H2D in chunks + kernels; the counters come back first ...
        res = alnfilter.filter_json_begin(handles[b], h_gaf, counts=counts_of[b])
        # ... informative_aln.json is assembled on the device (:160-175) and copied back as text on a thread of its own ...
        text_job[b] = side_pool.submit(alnfilter.filter_json_finish, handles[b])
        # ... beside the genotypes and the VCF text
        vcf_job[b] = side_pool.submit(vcf_of, res.counts)
        if not overlap:
            take(b)
        return res

    def e2e_run(overlap):
        for k in range(2):
            res = e2e_step(k, overlap)
        take(0), take(1)
        sync_all()
        t0 = time.perf_counter()
        for k in range(Ke):
            res = e2e_step(k, overlap)
        take(0), take(1)
        sync_all()
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t[0])
        return sec, res

    e2e_serial_s, res = e2e_run(False)       # one batch at a time: the latency of a batch
    e2e_s, res = e2e_run(True)
    h2d = n_bytes + tables.num_sv * 8 + n_sv * 5
    d2h = tables.num_sv * 8 + 64 + out_bytes[0] + n_sv * (24 + 1 + 8 + 1)        # counters, stats, the JSON text, genotypes

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = load_peaks()
    algo_bytes = n_bytes + 16 * n_hits            # DESIGN.md: line bytes once + 12 B hit tuple + 4 B counter RMW
    achieved = algo_bytes / (filt_ms * 1e-3) / 1e9
    geno_bytes = 42 * n_loc
    if world == 1:
        r = cpu_arm(gaf, edges_text, gfa_text, vcf, n_rec, 1, min(100_000, n_rec), 1, 0)
        cpu_line = {"value": r["value"], "unit": UNIT, "cores": 1, "kind": r["kind"],
                    "sample": f"first {r['n_sample']} records of the batch through the filter ({r['filter_s']:.2f} s, of which start-up "
                              f"{r['startup_s']:.2f} s) projected to {n_rec} records, plus the genotyper over all {n_sv} SVs "
                              f"({r['genotype_s']:.2f} s); {r['what']}, one process like the reference"}
        cpu_c = cpu_baseline_c(gaf, edges_text, gfa_text, check=(tables.sv_ids, res.counts, res.n_hits))
    else:
        cpu_line = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": "timed at N=1 only"}
        cpu_c = None
    key = f"{args.workload}:{args.catalogue}"
    line = {
        "metric": METRIC, "value": job_rec * K / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": K,
        "warmup": max(3, args.warmup), "ms_per_step": total_ms / K, "higher_is_better": True, "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic",
        "config": {
            "workload": f"{args.workload} x{scale:g}{' (catalogue at full size)' if args.catalogue == 'full' else ''} "
                        f"{'cut by bytes over the GPUs' if strong else 'per GPU'}: {n_rec} GAF records ({n_bytes / 1e6:.1f} MB) on rank 0, "
                        f"{n_sv} VCF SVs, {tables.num_links} link keys, {tables.num_sv} sv keys",
            "records_per_gpu": n_rec, "gaf_bytes_per_gpu": n_bytes, "hits_per_gpu": n_hits, "job_records": job_rec, "svs": n_sv,
            "multi_node_records": st["n_multi"], "l2": "input larger than L2 (no flush needed)" if n_bytes > 200e6
            else "input smaller than L2: resident re-reads possible",
            "tables_device_bytes": tables.device_bytes, "gen_seconds": round(gen_s, 1),
        },
        "svs_genotyped_per_sec": n_sv / (geno_ms * 1e-3) if geno_ms > 0 else None,
        "kernel_ms": {"filter": filt_ms, "filter_scan_only": scan_ms, "allreduce": comm_ms, "genotype": geno_ms},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": load_traffic(key), "kernel": "filter chain: probe+scan+exact", "algorithmic_bytes_per_launch": algo_bytes,
                     "peak_source": peak_src,
                     "dominant_kernel": {"name": "scan_kernel", "ms": scan_ms, "share_of_chain": scan_ms / filt_ms,
                                         "achieved": algo_bytes / (scan_ms * 1e-3) / 1e9, "frac": algo_bytes / (scan_ms * 1e-3) / 1e9 / peak,
                                         "algorithmic_bytes_per_launch": algo_bytes},
                     "genotype_kernel": {"achieved": geno_bytes / (geno_ms * 1e-3) / 1e9 if geno_ms > 0 else None,
                                         "bytes_per_launch": geno_bytes}},
        "cpu_baseline": cpu_line,
        "cpu_baseline_c": cpu_c,
        "e2e": {"value": (n_rec * world if not strong else job_rec) * Ke / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h, "steps": Ke, "ms_per_step": 1000 * e2e_s / Ke,
                "json_bytes_per_step": out_bytes[0], "vcf_bytes_per_step": out_bytes[1],
                "one_batch_at_a_time": {"value": (n_rec * world if not strong else job_rec) * Ke / e2e_serial_s, "unit": UNIT,
                                        "ms_per_step": 1000 * e2e_serial_s / Ke},
                "what": "svjg_filter_json_begin (pinned GAF bytes in, counters out) -> [svjg_filter_json_finish: informative_aln.json text "
                        "rendered on the device, copied back] beside [svjg_genotype_host -> genotype.vcf text (svjg_vcf_format)], all in host memory; "
                        "two batches in flight on two handles of the tables (the text of batch k goes back while batch k + 1 comes in); "
                        "one_batch_at_a_time = the same steps strictly one after the other"
                        + ("; one such job per GPU at once" if world > 1 else "")},
        "collective": ("p2p-fused: counters summed inside the genotype kernel over NVLink peer memory" if xchg else
                       ("nccl all_reduce" if world > 1 else "none (one GPU)")),
        "strong_check": strong_check,
        "gpu_launches": 5 * K,   # reset + probe + scan + exact + genotype
        "clocks": clocks,
    }
    if dumped is not None:
        line["dumped_outputs"] = {name: {"rows": n, "of": total} for name, (n, total) in dumped.items()}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
