"""Drop-in command lines of the post-mapping stages: the same flags, files and exit
statuses as the reference's filter-alignments.py (:29-71), predict-genotype.py (:31-48)
and svjedi-graph.py (:28-71); the work is done by libsvjg.so on the GPU.  Where the
reference dies with a traceback (exit status 1) these print one line and exit 1."""
from __future__ import annotations

import argparse
import subprocess
import sys


def _die(msg):
    sys.stderr.write(f"svjg: {msg}\n")
    sys.exit(1)


def leave(status):
    """Ends a front-end process: every output file is closed by now, so the page-locked buffers and the CUDA
    context are not taken down one by one (0.3 s); an exception (SystemExit from _die included) never gets here."""
    import os
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(int(status or 0))


def _start_device():
    """The CUDA context takes about a second to create: do it on a thread while the files are read."""
    import os
    import threading
    # the front-end processes use every kernel of the library and nothing else on the GPU: loading the
    # kernels with the context is 0.5 s faster than on first launch (set before the first CUDA call)
    os.environ.setdefault("CUDA_MODULE_LOADING", "EAGER")
    # the driver brings up every GPU it can see (a good 0.1 s each on an 8-GPU node): show it the ones that are used
    os.environ.setdefault("CUDA_VISIBLE_DEVICES", ",".join(str(d) for d in range(_n_gpus())))
    from . import capi
    box = {}

    def run():
        box["rc"] = capi.lib.svjg_device_init(0)
        box["msg"] = capi.lib.svjg_last_error().decode("utf-8", "replace") if box["rc"] else ""
    th = threading.Thread(target=run, daemon=True)
    th.start()

    def wait():
        th.join()
        if box.get("rc"):
            raise capi.SvjgError(box["rc"], box["msg"])
    return wait


_T0 = [None]


def _lap(what):
    """SVJG_TIMING=1: wall clock of the front-end's stages on stderr (profiling hook, as in csrc/tables.cpp)."""
    import os
    import time
    if "SVJG_TIMING" not in os.environ:
        return
    now = time.perf_counter()
    if _T0[0] is not None:
        sys.stderr.write(f"svjg timing: {what:<28s} {now - _T0[0]:8.3f} s\n")
    _T0[0] = now


def _n_gpus():
    """SVJG_GPUS=N: the filter stage shards its GAF over N GPUs of the node (an extension; the reference has
    one process and no device).  Default 1."""
    import os
    try:
        return max(1, int(os.environ.get("SVJG_GPUS", "1")))
    except ValueError:
        _die("SVJG_GPUS must be a number of GPUs")


def _load_tables(prefix, gfa_file, device_ready=None):
    from . import alnfilter
    t = alnfilter.Tables.load(prefix + "_svs_edges.json", gfa_file)      # host work: JSON + GFA parse, table build
    if device_ready:
        device_ready()
    return t.to_device(0)


def _replicas(tables, n):
    """`tables` on device 0 plus a copy on each of the devices 1 .. n-1 (uploaded on threads)."""
    from concurrent.futures import ThreadPoolExecutor
    if n <= 1:
        return [tables]
    with ThreadPoolExecutor(n - 1) as pool:
        return [tables] + list(pool.map(lambda d: tables.clone().to_device(d), range(1, n)))


def _filter_to_json(tables, gaf_file, out_json, dover_given=False, gaf=None, stream=None, d_over=100, min_identity=None):
    """filter-alignments.py:119-175.  Returns (FilterResult, page-locked GAF bytes).  ``stream``: an open
    pipe to filter while it is being written (alnfilter.filter_stream) instead of a file."""
    from . import alnfilter, capi, gzio
    if dover_given:
        # -O leaves a list in d_over and `int >= list` raises at the first overlap test (:269);
        # count every test the reference would make
        tables.set_flags(capi.FLAG_EXACT_CHECKS)
    if gaf is None and stream is None:
        with open(gaf_file, "rb") as fh:
            head = fh.read(2)
        if gzio.is_gzip(head):                                              # extension: gzip / bgzip input
            gaf = alnfilter.RegisteredBytes(alnfilter.translate_newlines(gzio.read_bytes(gaf_file)))
        else:
            gaf = alnfilter.read_file_pinned(gaf_file)
            if alnfilter.translate_newlines(gaf) is not gaf:               # carriage returns: text-mode line ends
                gaf = alnfilter.RegisteredBytes(alnfilter.translate_newlines(gaf))
    written = None                      # bytes of the JSON file where the device has written it
    n_gpus = _n_gpus()
    if stream is not None:
        res, gaf = alnfilter.filter_stream(tables, stream, d_over=d_over)
    elif n_gpus > 1:
        # one file, N byte ranges cut at line ends, one GPU each; counters summed, hits merged in range order
        # (an extension; SVJG_GPUS=N).  Each range stays on its device, the text is rendered on device 0 with the
        # lines of the other ranges read over NVLink; without peer access: hit lists to the host, host emitter
        replicas = _replicas(tables, n_gpus)
        res = None if min_identity is not None else alnfilter.filter_json_multi_begin(replicas, gaf, d_over=d_over)
        if res is None:
            res = alnfilter.filter_host_multi(replicas, gaf, d_over=d_over)
        elif not (dover_given and res.stats["n_checks"] > 0):
            written = alnfilter.filter_json_write(tables, out_json)
            if written is None:
                res = alnfilter.filter_host_multi(replicas, gaf, d_over=d_over)
    elif min_identity is not None:
        res = alnfilter.filter_host(tables, gaf, d_over=d_over)                # the hit list on the host: it is thinned below
    else:
        # the text of informative_aln.json is assembled on the device and written slice by slice as it comes back;
        # the host emitter takes over where the device renderer declines (non-ASCII bytes in a stored line, a giant list)
        res = alnfilter.filter_json_begin(tables, gaf, d_over=d_over)
        _lap("filter")
        if res is None:                                                        # the file does not fit the device
            res = alnfilter.filter_host(tables, gaf, d_over=d_over)
        elif not (dover_given and res.stats["n_checks"] > 0):                  # (-O: the reference stops before it writes)
            written = alnfilter.filter_json_write(tables, out_json)
            if written is None:
                res = alnfilter.filter_host(tables, gaf, d_over=d_over)
    if min_identity is not None:
        res = alnfilter.apply_min_identity(tables, gaf, res, min_identity)
    if dover_given and res.stats["n_checks"] > 0:
        _die("-O/--dover makes the reference fail at its first breakpoint-overlap test (TypeError); same here")
    if written is None:
        alnfilter.write_informative_json(tables, gaf, res, out_json)
    _lap("JSON file written")
    return res, gaf


def filter_main(argv=None):
    ap = argparse.ArgumentParser(description="---")
    ap.add_argument("-a", "--gaf", metavar="<align_file>", nargs=1, help="align file in gaf format", required=True)
    ap.add_argument("-g", "--gfa", metavar="<graph_file>", nargs=1, help="variant graph in gfa format", required=True)
    ap.add_argument("-i", "--gfainfo", metavar="<gfa_info>", nargs=1, help="gfa info", required=False)
    ap.add_argument("-O", "--dover", metavar="<min_breakpoint_overlap>", nargs=1, required=False, default=100)
    ap.add_argument("-o", "--outputDir", metavar="<outputDirectory>", type=str, required=False)
    ap.add_argument("-p", "--prefix", metavar="<prefix", type=str, required=False)
    # two switches the reference does not have (its -O cannot be used, :269; its identity is parsed and dropped, :193-196)
    ap.add_argument("--min-overlap", metavar="<bases>", type=int, default=None,
                    help="NOT in the reference: aligned bases required on each side of a breakpoint (default 100, "
                         "filter-alignments.py:56); the reference's own -O/--dover stops at its first overlap test and so does ours")
    ap.add_argument("--min-identity", metavar="<fraction>", type=float, default=None,
                    help="NOT in the reference, off by default: drop alignments whose identity (the id:f: tag, else "
                         "matches / alignment length: filter-alignments.py:193-196) is below this")
    args = ap.parse_args(argv)
    if not args.prefix:
        # the reference never assigns svs_edges_dict without -p (UnboundLocalError, :95)
        _die("-p/--prefix is required: <prefix>_svs_edges.json holds the link -> SV table")
    out_json = args.prefix + "_informative_aln.json"
    if args.outputDir:
        out_json = "/".join([args.outputDir, out_json])
    from . import alnfilter, capi, gzio
    try:
        import os
        import stat
        _lap("")
        ready = _start_device()
        pipe = None
        if not stat.S_ISREG(os.stat(args.gaf[0]).st_mode):                 # `minigraph ... | filter-alignments.py -a /dev/stdin`
            pipe = open(args.gaf[0], "rb")
            if gzio.is_gzip(pipe.peek(2)[:2]):                             # compressed: inflate it whole (below)
                raw = gzio.inflate(pipe.read())
                pipe.close()
                pipe = None
        else:
            raw = gzio.read_bytes(args.gaf[0])                             # read (gzip / bgzip: inflate) while the context comes up
        if pipe is not None:
            with pipe:                                                     # filtered segment by segment while the mapper writes
                tables = _load_tables(args.prefix, args.gfa[0], ready)
                _filter_to_json(tables, args.gaf[0], out_json, dover_given=args.dover != 100, stream=pipe,
                                d_over=100 if args.min_overlap is None else args.min_overlap, min_identity=args.min_identity)
            return 0
        _lap("GAF read")
        raw = alnfilter.translate_newlines(raw)                            # text-mode line ends, like the reference
        _lap("line ends")
        tables = _load_tables(args.prefix, args.gfa[0], ready)
        _lap("tables + context")
        gaf = alnfilter.RegisteredBytes(raw)                                # page-lock in place
        _lap("page-lock")
        _filter_to_json(tables, args.gaf[0], out_json, dover_given=args.dover != 100, gaf=gaf,
                        d_over=100 if args.min_overlap is None else args.min_overlap, min_identity=args.min_identity)
    except (alnfilter.InputError, capi.SvjgError, OSError) as exc:
        _die(str(exc))
    return 0


def genotype_main(argv=None):
    ap = argparse.ArgumentParser(description="Structural variations genotyping using long reads")
    ap.add_argument("-d", "--aln", metavar="<alndict>", nargs=1, required=True)
    ap.add_argument("-v", "--vcf", metavar="<vcffile>", help="vcf format", required=True)
    ap.add_argument("-o", "--output", metavar="<output>", nargs=1, help="output file")
    ap.add_argument("-e", "--err", nargs=1, type=float, help="allele error probability")
    ap.add_argument("-ms", "--minsupport", metavar="<minNbAln>", type=int, default=3,
                    help="Minimum number of alignments to genotype a SV (default: 3>=)")
    args = ap.parse_args(argv)
    output = "genotype_results.txt" if args.output is None else args.output[0]
    e = args.err[0] if args.err is not None else 0.00005
    from . import capi, genotype, gzio
    try:
        _lap("")
        ready = _start_device()
        counts = genotype.AlnCounts.load(args.aln[0])
        _lap("informative_aln.json read")
        ready()
        _lap("context")
        lines = gzio.read_bytes(args.vcf)                      # the file's bytes: keys and text are built by the library
        with open(output, "wb") as out:         # the reference opens the output before it reads the VCF (:92)
            _, n = genotype.genotype_vcf_from_json(counts, lines, args.minsupport, e, out=out)
        _lap("genotypes + VCF written")
    except (genotype.VcfError, capi.SvjgError, OSError, ValueError) as exc:
        _die(str(exc))
    print(f"Genotyped svs: {n}")
    return 0


def _sample_name(path):
    import os
    name = os.path.basename(path)
    if name.endswith(".gz"):
        name = name[:-3]
    if name.endswith(".gaf"):
        name = name[:-4]
    return name


def _read_sample(files):
    """The files of one sample as the filter front-end reads them (gzip / bgzip inflated, text-mode line ends),
    each page-locked in place."""
    from . import alnfilter, gzio
    return [alnfilter.RegisteredBytes(alnfilter.translate_newlines(gzio.read_bytes(f))) for f in files]


def cohort_main(argv=None):
    """genotype-cohort.py (an extension; the reference genotypes one sample per run): many samples' GAF files
    against one catalogue, one multi-sample VCF whose column s is what filter-alignments.py + predict-genotype.py
    write for sample s alone.  The tables are loaded and the device started once; the counters of every sample stay
    on the device."""
    ap = argparse.ArgumentParser(description="Genotype one SV catalogue in many samples")
    ap.add_argument("-p", "--prefix", metavar="<prefix>", type=str, required=False,
                    help="<prefix>_svs_edges.json holds the link -> SV table")
    ap.add_argument("-g", "--gfa", metavar="<graph_file>", required=True, help="variant graph in gfa format")
    ap.add_argument("-v", "--vcf", metavar="<vcffile>", required=True, help="the SV catalogue in vcf format")
    ap.add_argument("-a", "--gaf", metavar="<align_file>", nargs="+", required=True,
                    help="one argument per sample; a comma-joined argument is one sample whose files are counted together")
    ap.add_argument("-o", "--output", metavar="<output>", required=True, help="multi-sample VCF")
    ap.add_argument("--names", metavar="<n1,n2,...>", default=None,
                    help="sample names (default: the first file's name without .gz and .gaf)")
    ap.add_argument("-ms", "--minsupport", metavar="<minNbAln>", type=int, default=3,
                    help="Minimum number of alignments to genotype a SV (default: 3>=)")
    ap.add_argument("-e", "--err", type=float, default=0.00005, help="allele error probability")
    ap.add_argument("--min-overlap", metavar="<bases>", type=int, default=None,
                    help="aligned bases required on each side of a breakpoint (default 100)")
    ap.add_argument("--info-tags", metavar="<LIST>", default=None,
                    help="population INFO tags computed over the samples, a comma list of NS, AN, AC, AF, AC_Het, "
                         "AC_Hom, F_MISSING, HWE, ExcHet, or all (written in that order; default: none, the catalogue's "
                         "INFO as it is)")
    args = ap.parse_args(argv)
    import os
    if not args.prefix:
        _die("-p/--prefix is required: <prefix>_svs_edges.json holds the link -> SV table")
    info_tags = ()
    if args.info_tags is not None:
        from .cohort import parse_info_tags
        try:
            info_tags = parse_info_tags(args.info_tags)
        except ValueError as exc:
            _die(f"--info-tags: {exc}")
    if os.environ.get("SVJG_GPUS", "1").strip() != "1":
        _die("genotype-cohort runs on one GPU: SVJG_GPUS must be 1")
    samples = [[f for f in a.split(",")] for a in args.gaf]
    if any(not f for files in samples for f in files):
        _die("empty file name in -a")
    names = args.names.split(",") if args.names is not None else [_sample_name(files[0]) for files in samples]
    if len(names) != len(samples):
        _die(f"{len(names)} names for {len(samples)} samples")
    for nm in names:
        if not nm or any(c in nm for c in "\t\r\n"):
            _die(f"bad sample name {nm!r}: names must be non-empty and hold no tab, CR or LF")
    if len(set(names)) != len(names):
        _die("sample names must be unique")
    d_over = 100 if args.min_overlap is None else args.min_overlap
    out_path = os.path.abspath(args.output)
    from concurrent.futures import ThreadPoolExecutor

    from . import alnfilter, capi, cohort, genotype, gzio
    tmp = None
    try:
        _lap("")
        ready = _start_device()
        vcf = gzio.read_bytes(args.vcf)
        _lap("VCF read")
        tables = _load_tables(args.prefix, args.gfa, ready)
        _lap("tables + context")
        co = cohort.Cohort(tables, len(samples))
        with ThreadPoolExecutor(1) as pool:
            # sample k + 1 is read, inflated, translated and page-locked while sample k is filtered
            nxt = pool.submit(_read_sample, samples[0])
            for k, files in enumerate(samples):
                bufs = nxt.result()
                nxt = pool.submit(_read_sample, samples[k + 1]) if k + 1 < len(samples) else None
                for f, b in zip(files, bufs):
                    try:
                        co.filter(k, b.array, d_over=d_over)
                    except alnfilter.InputError as exc:
                        raise alnfilter.InputError(f"sample {names[k]!r}, file {f}: {exc}") from None
                del bufs
                _lap(f"sample {k} filtered")
        import tempfile
        fd, tmp = tempfile.mkstemp(prefix="." + os.path.basename(out_path) + ".", dir=os.path.dirname(out_path))
        with os.fdopen(fd, "wb") as out:
            _, n_gt = cohort.genotype_cohort_vcf(tables, co, vcf, names, args.minsupport, args.err, out=out,
                                                 info_tags=info_tags)
        os.replace(tmp, out_path)
        tmp = None
        _lap("genotypes + VCF written")
    except (alnfilter.InputError, genotype.VcfError, capi.SvjgError, OSError, ValueError) as exc:
        if tmp is not None:
            os.unlink(tmp)
        _die(str(exc))
    for nm, n in zip(names, n_gt):
        print(f"Genotyped svs in {nm}: {n}")
    return 0


class _MapperOutput:
    """File-like view (read(n) only) of what ends up in <prefix>.gaf: what the file already holds (the
    reference appends, svjedi-graph.py:100-104), then the standard output of one mapper process after the
    other; every byte read from a mapper is also appended to the file.  ``returncode`` is the last
    mapper's, the one the reference looks at (:107)."""

    def __init__(self, commands, gaf_path):
        self._commands = list(commands)
        self._path = gaf_path
        self._old = open(gaf_path, "rb")
        self._out = open(gaf_path, "ab")
        self._proc = None
        self.returncode = None

    def read(self, n):
        if self._old is not None:
            data = self._old.read(n)
            if data:
                return data
            self._old.close()
            self._old = None
        while True:
            if self._proc is None:
                if not self._commands:
                    return b""
                self._proc = subprocess.Popen(self._commands.pop(0), shell=True, stdout=subprocess.PIPE)
            data = self._proc.stdout.read(n)
            if data:
                self._out.write(data)
                return data
            self._proc.stdout.close()
            self.returncode = self._proc.wait()
            self._proc = None

    def drain(self):
        while self.read(1 << 24):
            pass

    def close(self):
        if self._old is not None:
            self._old.close()
        self._out.close()


def pipeline_main(svjg_dir, argv=None):
    """svjedi-graph.py: graph construction and mapping are external tools exactly as in the
    reference (:85-108); filtering and genotyping run fused in this process — the counters
    go from one stage to the next in memory, no JSON is read back — and still write both output files."""
    ap = argparse.ArgumentParser()
    ap.add_argument("-v", "--vcf", type=str, help="SV set in vcf format", required=True)
    ap.add_argument("-r", "--ref", type=str, help="Reference genome in fasta format", required=True)
    ap.add_argument("-q", "--reads", type=str, help="Long reads in fastq format", required=True)
    ap.add_argument("-p", "--prefix", type=str, help="Prefix of generated files", required=True)
    ap.add_argument("-t", "--threads", type=int, help="Number of threads to use for read mapping", default=[1])
    ap.add_argument("-ms", "--minsupport", metavar="<minNbAln>", type=int, default=3,
                    help="Minimum number of alignments to genotype a SV (default: 3>=)")
    args = ap.parse_args(argv)
    import os
    out_gfa, out_gaf = args.prefix + ".gfa", args.prefix + ".gaf"

    print("Constructing variation graph...")
    construct = os.environ.get("SVJG_CONSTRUCT_GRAPH", f"{svjg_dir}/construct-graph.py")
    if subprocess.run(f"python3 {construct} -v {args.vcf} -r {args.ref} -o {out_gfa}", shell=True).returncode == 1:
        sys.exit("Failed to contruct the variation graph.\nExiting SVJedi-graph.")

    if os.environ.get("SVJG_STREAM"):
        return _pipeline_streamed(args, out_gfa, out_gaf)

    print("Mapping reads on graph...")
    subprocess.run(f"touch {out_gaf}", shell=True)
    proc = None
    for fq in args.reads.split(","):
        proc = subprocess.run(f"minigraph -x lr -t{args.threads} {out_gfa} {fq} >> {out_gaf}", shell=True)
    if proc.returncode == 1:
        sys.exit("Failed to map the reads on the graph.\nExiting SVJedi-graph.")

    print("Filtering alignment file...")
    from . import alnfilter, capi, genotype, gzio
    try:
        tables = _load_tables(args.prefix, out_gfa)
        res, _gaf = _filter_to_json(tables, out_gaf, args.prefix + "_informative_aln.json")
    except (alnfilter.InputError, capi.SvjgError, OSError) as exc:
        sys.stderr.write(f"svjg: {exc}\n")
        sys.exit("Failed to filter the alignments.\nExiting SVJedi-graph.")

    print("Genotyping SVs...")
    try:
        lines = gzio.read_bytes(args.vcf)                      # the file's bytes: keys and text are built by the library
        with open(args.prefix + "_genotype.vcf", "wb") as out:
            _, n = genotype.genotype_vcf(tables, res.counts, lines, args.minsupport, out=out)
    except (genotype.VcfError, capi.SvjgError, OSError, ValueError) as exc:
        sys.stderr.write(f"svjg: {exc}\n")
        sys.exit("Failed to predict the genotypes.\nExiting SVJedi-graph.")
    print(f"Genotyped svs: {n}")
    return 0


def _pipeline_streamed(args, out_gfa, out_gaf):
    """SVJG_STREAM=1 (SURVEY.md §8(f) row N3): stages 2-3 overlapped.  The mappers' output is appended to
    <prefix>.gaf as in the reference and filtered segment by segment while they run; the messages, files and
    exit statuses are those of the sequential run (a mapper failure is reported before a filter failure)."""
    from . import alnfilter, capi, genotype, gzio
    print("Mapping reads on graph...")
    subprocess.run(f"touch {out_gaf}", shell=True)
    chain = _MapperOutput([f"minigraph -x lr -t{args.threads} {out_gfa} {fq}" for fq in args.reads.split(",")], out_gaf)
    failure = None
    tables = res = gaf = None
    try:
        try:
            tables = _load_tables(args.prefix, out_gfa)
            res, gaf = alnfilter.filter_stream(tables, chain)
        except (alnfilter.InputError, capi.SvjgError, OSError) as exc:
            failure = exc
            chain.drain()                                    # the reference maps everything before it filters
    finally:
        chain.close()
    if chain.returncode == 1:
        sys.exit("Failed to map the reads on the graph.\nExiting SVJedi-graph.")
    print("Filtering alignment file...")
    try:
        if failure is not None:
            raise failure
        alnfilter.write_informative_json(tables, gaf, res, args.prefix + "_informative_aln.json")
    except (alnfilter.InputError, capi.SvjgError, OSError) as exc:
        sys.stderr.write(f"svjg: {exc}\n")
        sys.exit("Failed to filter the alignments.\nExiting SVJedi-graph.")
    print("Genotyping SVs...")
    try:
        lines = gzio.read_bytes(args.vcf)
        with open(args.prefix + "_genotype.vcf", "wb") as out:
            _, n = genotype.genotype_vcf(tables, res.counts, lines, args.minsupport, out=out)
    except (genotype.VcfError, capi.SvjgError, OSError, ValueError) as exc:
        sys.stderr.write(f"svjg: {exc}\n")
        sys.exit("Failed to predict the genotypes.\nExiting SVJedi-graph.")
    print(f"Genotyped svs: {n}")
    return 0
