"""Cohort genotyping (svjg/cohort.py, genotype-cohort.py): many samples against one catalogue, one multi-sample VCF
whose column s is byte for byte what filter-alignments.py + predict-genotype.py write for sample s alone.
CPU part: the multi-sample text (svjg_vcf_format_cohort) against the single-sample text and a Python statement of
the cell, the oracle composition (oracle_cohort_vcf) on the reference's golden VCFs, and the command line's argument checks.
GPU part (-m gpu): the command line and the module against the oracles, the cohort kernel against
genotype.genotype_host, errors, and a full-size catalogue."""
import ctypes as C
import gzip
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import PKG, alt_len_from_gfa_text, read_golden
from oracle import svjg_oracle as O
from svjg import capi, genotype

GOLDEN_TAGS = ["c1", "s2", "s3", "s4"]


def _golden_vcf(tag):
    return read_golden("c1.vcf" if tag == "c1" else f"{tag}.vcf.gz")


def _golden_counts(tag):
    if tag == "c1":
        return O.hit_counts(json.loads(read_golden("c1_informative_aln.json.gz")))
    return {k: tuple(v) for k, v in json.loads(read_golden(f"{tag}_counts.json.gz")).items()}


def oracle_cohort_vcf(counts_per_sample, names, vcf_lines, min_support=3, e=0.00005):
    """The multi-sample VCF of a cohort composed from the oracle: O.genotype_vcf per sample, the sample columns spliced
    side by side and the column header naming the samples.  Returns (output text, [genotyped count per sample])."""
    outs = [O.genotype_vcf(c, vcf_lines, min_support, e) for c in counts_per_sample]
    kinds = []                                # per output line: "h" header text, "c" column header, "b" body
    for line in vcf_lines:
        if line.startswith("##FORMAT"):
            continue
        if line.startswith("##"):
            kinds.append("h")
        elif line.startswith("#C"):
            kinds += ["h"] * (O.FORMAT_HEADER.count("\n") - 1) + ["c"]
        else:
            kinds.append("b")
    per_sample = [text.split("\n") for text, _n in outs]
    out = []
    for j, kind in enumerate(kinds):
        first = per_sample[0][j]
        if kind == "h":
            out.append(first)
        elif kind == "c":
            out.append(first[:-len("SAMPLE")] + "\t".join(names))
        else:
            out.append(first.rsplit("\t", 1)[0] + "".join("\t" + p[j].rsplit("\t", 1)[1] for p in per_sample))
    return "\n".join(out + per_sample[0][len(kinds):]), [n for _text, n in outs]


def _random_cells(rng, n_cells):
    """gt / flags / ad2 / pl as the genotype kernel could return them: gated and genotyped cells, halves, negative
    and 19-digit PLs."""
    fl = rng.choice([0, capi.GT_GENOTYPED, capi.GT_GENOTYPED | capi.GT_HALVED_0, capi.GT_GENOTYPED | capi.GT_HALVED_1],
                    size=n_cells).astype(np.uint8)
    gt = rng.integers(0, 4, n_cells, dtype=np.uint8)
    ad = rng.integers(0, 3000, (n_cells, 2), dtype=np.uint32)
    ad[rng.random(n_cells) < 0.05] = 0xFFFFFFFF
    pl = rng.integers(-5000, 100000, (n_cells, 3), dtype=np.int64)
    pl[rng.random(n_cells) < 0.02, 0] = np.iinfo(np.int64).min
    pl[rng.random(n_cells) < 0.02, 2] = np.iinfo(np.int64).max
    return gt, fl, ad, pl


def _format_cohort(v, lo, hi, names, gt, fl, ad, pl, n_gt):
    joined = "\t".join(names).encode()
    arrs = [np.ascontiguousarray(a) for a in (gt, fl, ad, pl)]
    buf, n_out = C.c_void_p(), C.c_uint64()
    capi.check(capi.lib.svjg_vcf_format_cohort(v._h, lo, hi, len(names), joined, len(joined),
                                               *(a.ctypes.data for a in arrs), C.byref(buf), C.byref(n_out),
                                               n_gt.ctypes.data))
    try:
        return C.string_at(buf.value, n_out.value).decode("ascii")
    finally:
        capi.lib.svjg_buffer_free(buf)


def _cell_text(gt, f, t1, t2, pl):
    if not f & capi.GT_GENOTYPED:
        return "./.:0:0,0:.,.,."
    h0, h1 = bool(f & capi.GT_HALVED_0), bool(f & capi.GT_HALVED_1)
    return (f"{genotype.GT_TEXT[gt]}:{O._py_num_str(t1 + t2, h0 or h1)}:{O._py_num_str(t1, h0)},"
            f"{O._py_num_str(t2, h1)}:{pl[0]},{pl[1]},{pl[2]}")


def _python_cohort_text(lines, names, gt, fl, ad, pl):
    header, recs = genotype.parse_vcf(lines)
    S = len(names)
    out, hi = [], 0
    col = genotype._FORMAT_LINES[:-len("SAMPLE\n")] + "\t".join(names) + "\n"

    def hdr(text):
        return col if text == genotype._FORMAT_LINES else text
    for i, (head, _code, _key) in enumerate(recs):
        while hi < len(header) and header[hi][0] <= i:
            out.append(hdr(header[hi][1]))
            hi += 1
        cells = [_cell_text(int(gt[i * S + s]), int(fl[i * S + s]), int(ad[i * S + s, 0]), int(ad[i * S + s, 1]),
                            pl[i * S + s].tolist()) for s in range(S)]
        out.append(head + "\tGT:DP:AD:PL" + "".join("\t" + c for c in cells) + "\n")
    out += [hdr(h[1]) for h in header[hi:]]
    return "".join(out)


def _fuzz_vcfs():
    return [c["vcf"] for c in json.loads(read_golden("fuzz_vcf.json.gz"))]


def test_one_sample_named_SAMPLE_is_the_single_sample_text():
    rng = np.random.default_rng(41)
    n_checked = 0
    for text in [_golden_vcf(t) for t in GOLDEN_TAGS] + _fuzz_vcfs():
        try:
            v = genotype.NativeVcf.from_input(text.encode())
        except genotype.VcfError:
            continue
        if v is None:
            continue
        gt, fl, ad, pl = _random_cells(rng, v.n)
        want, want_n = v.format(gt, fl, ad, pl)
        n_gt = np.zeros(1, np.uint64)
        assert _format_cohort(v, 0, v.n, ["SAMPLE"], gt, fl, ad, pl, n_gt) == want
        assert int(n_gt[0]) == want_n
        n_checked += 1
    assert n_checked > 500


@pytest.mark.parametrize("tag", GOLDEN_TAGS)
def test_blocks_do_not_change_the_bytes(tag):
    text = _golden_vcf(tag) + "##trailing=1\n"
    v = genotype.NativeVcf.from_input(text.encode())
    S, names = 7, [f"s{k}" for k in range(7)]
    rng = np.random.default_rng(7)
    gt, fl, ad, pl = _random_cells(rng, v.n * S)
    n_whole = np.zeros(S, np.uint64)
    whole = _format_cohort(v, 0, v.n, names, gt, fl, ad, pl, n_whole)
    assert whole == _python_cohort_text(text.splitlines(True), names, gt, fl, ad, pl)
    assert n_whole.tolist() == [int(((fl[s::S] & capi.GT_GENOTYPED) != 0).sum()) for s in range(S)]
    for trial in range(4):
        cuts = sorted(set([0, v.n] + rng.integers(0, v.n + 1, 1 + trial * 10).tolist() + [1, 2]))
        if trial == 3:
            cuts = list(range(v.n + 1))                            # blocks of one record
        n_gt = np.zeros(S, np.uint64)
        pieces = [_format_cohort(v, lo, hi, names, gt[lo * S:hi * S], fl[lo * S:hi * S], ad[lo * S:hi * S],
                                 pl[lo * S:hi * S], n_gt) for lo, hi in zip(cuts, cuts[1:])]
        assert "".join(pieces) == whole
        assert n_gt.tolist() == n_whole.tolist()


def test_empty_and_header_only_vcfs():
    for text in ["", "##a=1\n", "##a=1\n#CHROM\tPOS\n##b=2\n"]:
        v = genotype.NativeVcf.from_input(text.encode())
        n_gt = np.zeros(2, np.uint64)
        got = _format_cohort(v, 0, 0, ["x", "y"], *(np.zeros(0, t) for t in (np.uint8, np.uint8)),
                             np.zeros((0, 2), np.uint32), np.zeros((0, 3), np.int64), n_gt)
        assert got == _python_cohort_text(text.splitlines(True), ["x", "y"], None, None, None, None)


@pytest.mark.parametrize("tag", GOLDEN_TAGS)
def test_oracle_composition_reproduces_the_golden_vcfs(tag):
    want = read_golden("c1_genotype.vcf" if tag == "c1" else f"{tag}_genotype.vcf.gz")
    n_want = int(read_golden(f"{tag}_stdout.txt").split(":")[1])
    text, n = oracle_cohort_vcf([_golden_counts(tag)], ["SAMPLE"], _golden_vcf(tag).splitlines(True))
    assert text == want and n == [n_want]


def _cohort(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(PKG, "genotype-cohort.py"), *args], capture_output=True,
                          text=True, env=env)


@pytest.mark.parametrize("extra,env,message", [
    (["--names", "a,a"], {}, "unique"),
    (["--names", "a\tb,c"], {}, "tab"),
    (["--names", "a"], {}, "1 names for 2 samples"),
    (["--names", "a,,"], {}, "3 names for 2 samples"),
    (["--names", "a,"], {}, "non-empty"),
    ([], {"SVJG_GPUS": "2"}, "SVJG_GPUS"),
    ("no-prefix", {}, "-p/--prefix is required"),
])
def test_command_line_refuses_bad_arguments_before_the_device(tmp_path, extra, env, message):
    args = ["-g", "x.gfa", "-v", "x.vcf", "-a", "one.gaf", "two.gaf", "-o", str(tmp_path / "out.vcf")]
    if extra == "no-prefix":
        extra = []
    else:
        args = ["-p", str(tmp_path / "x")] + args
    # no CUDA device: a check that came after the device start would fail with another message
    r = _cohort(*args, *extra, env=dict(os.environ, CUDA_VISIBLE_DEVICES="", **env))
    assert r.returncode == 1 and message in r.stderr, r.stderr
    assert not os.listdir(tmp_path)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
def _write_inputs(tmp_path, tag):
    p = str(tmp_path / tag)
    open(p + ".gaf", "w").write(read_golden(f"{tag}.gaf.gz"))
    open(p + ".gfa", "w").write(read_golden(f"{tag}.gfa.gz"))
    open(p + "_svs_edges.json", "w").write(read_golden("c1_svs_edges.json" if tag == "c1" else f"{tag}_svs_edges.json.gz"))
    open(p + ".vcf", "w").write(_golden_vcf(tag))
    return p


@pytest.mark.gpu
@pytest.mark.parametrize("tag", GOLDEN_TAGS)
def test_one_sample_writes_the_golden_vcf(tmp_path, tag):
    p = _write_inputs(tmp_path, tag)
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", p + ".gaf", "-o", p + "_genotype.vcf", "--names", "SAMPLE")
    assert r.returncode == 0, r.stderr
    assert open(p + "_genotype.vcf").read() == read_golden("c1_genotype.vcf" if tag == "c1" else f"{tag}_genotype.vcf.gz")
    assert r.stdout == read_golden(f"{tag}_stdout.txt").replace("Genotyped svs:", "Genotyped svs in SAMPLE:")


def _python_oracle_counts(tag, gaf_text):
    edges = json.loads(read_golden("c1_svs_edges.json" if tag == "c1" else f"{tag}_svs_edges.json.gz"))
    alt = alt_len_from_gfa_text(read_golden(f"{tag}.gfa.gz"))
    return O.hit_counts(O.filter_alignments(O.text_mode_lines(gaf_text), edges, alt))


@pytest.mark.gpu
def test_s2_cohort_of_seven_samples(tmp_path):
    from oracle import c_oracle as CO
    from svjg import alnfilter, cli, cohort
    CO.ensure_built()
    p = _write_inputs(tmp_path, "s2")
    gaf = read_golden("s2.gaf.gz")
    lines = gaf.splitlines(True)
    files = {"whole": gaf, "half1": "".join(lines[:len(lines) // 2]), "half2": "".join(lines[len(lines) // 2:]),
             "x48": gaf * 48, "empty": ""}
    for name, text in files.items():
        open(f"{p}_{name}.gaf", "w").write(text)
    with gzip.open(f"{p}_crlf.gaf.gz", "wb") as fh:
        fh.write(gaf.replace("\n", "\r\n").encode())
    samples = [[f"{p}_whole.gaf"], [f"{p}_half1.gaf"], [f"{p}_half2.gaf"], [f"{p}_x48.gaf"], [f"{p}_empty.gaf"],
               [f"{p}_crlf.gaf.gz"], [f"{p}_half1.gaf", f"{p}_half2.gaf"]]
    texts = [files["whole"], files["half1"], files["half2"], files["x48"], "", gaf, gaf]
    names = [f"n{k}" for k in range(7)]
    vcf = _golden_vcf("s2")
    per_text = {}
    for text in texts:
        if text not in per_text and text != files["x48"]:
            per_text[text] = _python_oracle_counts("s2", text)
    # the oracle counts per line: 48 copies count 48 times what one copy counts
    per_text[files["x48"]] = {k: (48 * a, 48 * b) for k, (a, b) in per_text[gaf].items()}
    want, want_n = oracle_cohort_vcf([per_text[t] for t in texts], names, vcf.splitlines(True))
    # the module
    edges_text, gfa_text = read_golden("s2_svs_edges.json.gz"), read_golden("s2.gfa.gz")
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    co = cohort.Cohort(t, 7)
    for k, fs in enumerate(samples):
        for b in cli._read_sample(fs):
            co.filter(k, b.array)
    ct = CO.Tables(json.loads(edges_text), alt_len_from_gfa_text(gfa_text))
    for k, text in enumerate(texts):
        assert (co.counts(k) == CO.filter_counts(ct, text.encode())[0]).all(), names[k]
    assert (co.counts(6) == co.counts(0)).all() and (co.counts(3) == 48 * co.counts(0)).all()
    assert (co.counts(3) > 256).any()                                   # NEED_K cells
    got, got_n = cohort.genotype_cohort_vcf(t, co, vcf.encode(), names)
    assert got == want and got_n == want_n
    # the command line
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *[",".join(fs) for fs in samples], "-o", p + "_c.vcf",
                "--names", ",".join(names))
    assert r.returncode == 0, r.stderr
    assert open(p + "_c.vcf").read() == want
    assert r.stdout == "".join(f"Genotyped svs in {nm}: {n}\n" for nm, n in zip(names, want_n))
    # default names: the first file's name without .gz and .gaf
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", f"{p}_crlf.gaf.gz", f"{p}_half1.gaf,{p}_half2.gaf",
                "-o", p + "_d.vcf")
    assert r.returncode == 0, r.stderr
    assert "\tFORMAT\ts2_crlf\ts2_half1\n" in open(p + "_d.vcf").read()


def _synthetic(n_sv=2000, seed=5):
    from svjg import graphgen, synth
    chrom_len = synth.human_like_chroms(0.03)
    rows = synth.catalogue("mix", n_sv, chrom_len, seed=seed, ins_max=300, del_max=2000)
    g = graphgen.build_graph(chrom_len, rows)
    buf = io.StringIO()
    g.write_gfa(buf)
    return g, rows, g.edges_json(), buf.getvalue()


@pytest.mark.gpu
def test_forty_samples_against_the_oracle():
    from oracle import c_oracle as CO
    from svjg import alnfilter, cohort, synth
    CO.ensure_built()
    g, rows, edges_text, gfa_text = _synthetic()
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    ct = CO.Tables(json.loads(edges_text), alt_len_from_gfa_text(gfa_text))
    co = cohort.Cohort(t, 40)
    dicts = []
    for s in range(40):
        gaf = synth.simulate_gaf(g, 2500, seed=100 + s, mean_len=6000).encode()
        co.filter(s, gaf)
        want = CO.filter_counts(ct, gaf)[0]
        assert (co.counts(s) == want).all()
        dicts.append(CO.counts_dict(ct, want))
    assert t.num_sv > 1500
    vcf = synth.vcf_text(rows)
    names = [f"sample{s}" for s in range(40)]
    want, want_n = oracle_cohort_vcf(dicts, names, vcf.splitlines(True))
    assert min(want_n) > 100
    for block in (None, 1, 7):
        assert cohort.genotype_cohort_vcf(t, co, vcf.encode(), names, block_records=block) == (want, want_n)


@pytest.mark.gpu
@pytest.mark.parametrize("ms,e", [(0, 5e-5), (3, 5e-5), (0, 0.2), (3, 0.2)])
def test_cohort_kernel_equals_genotype_host(ms, e):
    from svjg import alnfilter, cohort
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    S, n = 37, 5000
    rng = np.random.default_rng(ms * 1000 + int(e * 100))
    co = cohort.Cohort(t, S)
    counts = []
    for s in range(S):
        c = rng.integers(0, 601, (t.num_sv, 2)).astype(np.uint32)
        c[rng.random(t.num_sv) < 0.2] = 0
        c[rng.random((t.num_sv, 2)) < 0.2] = 0
        c[rng.random((t.num_sv, 2)) < 0.5] %= 40
        co.load_counts(s, c)
        assert (co.counts(s) == c).all()
        counts.append(c)
    idx = rng.integers(0, t.num_sv, n).astype(np.uint32)
    idx[rng.random(n) < 0.05] = capi.NO_SV
    ty = rng.choice([0, 1, 2, 3, 255, 0x80, 0x81, 0x82, 0x83], size=n).astype(np.uint8)
    blk = cohort._Block(n * S)
    gt, fl, ad, pl = (a.copy() for a in cohort._genotype_block(co, idx, ty, ms, e, blk))
    assert (fl & capi.GT_NEED_K).sum() == 0
    n_big = 0
    for s in range(S):
        w_gt, w_fl, w_ad, w_pl = genotype.genotype_host(counts[s], idx, ty, ms, e)
        assert (gt[s::S] == w_gt).all() and (fl[s::S] == w_fl).all()
        assert (ad[s::S] == w_ad).all() and (pl[s::S] == w_pl).all()
        n_big += int(((w_ad.astype(np.uint64) + 1) // 2 > 256).any(axis=1).sum())
    assert n_big > 1000 and (fl & capi.GT_GENOTYPED).sum() > 10000


def _five_c1_samples(tmp_path, damaged_at=None):
    p = _write_inputs(tmp_path, "c1")
    gaf = read_golden("c1.gaf.gz")
    lines = gaf.splitlines(True)
    paths = []
    for k in range(5):
        text = "".join(lines[k * 7:])
        if k == damaged_at:
            fx = json.loads(read_golden("fuzz_lines.json.gz"))
            bad = next(c["line"] for c in fx["cases"] if c["rc"] == 1 and "\r" not in c["line"] and len(c["line"]) > 40)
            text = "".join(lines[:len(lines) // 2]) + bad.rstrip("\n") + "\n" + "".join(lines[len(lines) // 2:])
        paths.append(f"{p}_{k}.gaf")
        open(paths[-1], "w").write(text)
    return p, paths


@pytest.mark.gpu
def test_damaged_line_names_sample_file_and_offset(tmp_path):
    import re
    p, paths = _five_c1_samples(tmp_path, damaged_at=2)
    r = subprocess.run([sys.executable, os.path.join(PKG, "filter-alignments.py"), "-a", paths[2], "-g", p + ".gfa",
                        "-p", p, "-o", str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 1
    where = re.search(r"GAF line at byte \d+", r.stderr).group(0)
    out = str(tmp_path / "cohort.vcf")
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *paths, "-o", out)
    assert r.returncode == 1
    assert "'c1_2'" in r.stderr and paths[2] in r.stderr and where + ":" in r.stderr, r.stderr
    assert not [f for f in os.listdir(tmp_path) if "cohort" in f]


@pytest.mark.gpu
def test_error_rate_outside_0_1(tmp_path):
    p, paths = _five_c1_samples(tmp_path)
    out = str(tmp_path / "cohort.vcf")
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *paths, "-o", out, "-e", "1.5")
    assert r.returncode == 1 and "error rate" in r.stderr
    assert not [f for f in os.listdir(tmp_path) if "cohort" in f]
    open(p + "_none.gaf", "w").write("")
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", p + "_none.gaf", p + "_none.gaf", "--names", "a,b",
                "-o", out, "-e", "1.5")
    assert r.returncode == 0, r.stderr
    body = [ln for ln in open(out).read().splitlines() if not ln.startswith("#")]
    assert body and all(ln.endswith("\tGT:DP:AD:PL\t./.:0:0,0:.,.,.\t./.:0:0,0:.,.,.") for ln in body)
    assert r.stdout == "Genotyped svs in a: 0\nGenotyped svs in b: 0\n"


@pytest.mark.gpu
def test_full_size_c2_three_samples():
    from oracle import c_oracle as CO
    from svjg import alnfilter, cohort, synth
    CO.ensure_built()
    g, vcf, gaf0 = synth.make_workload("C2", scale=0.25)
    buf = io.StringIO()
    g.write_gfa(buf)
    edges_text, gfa_text = g.edges_json(), buf.getvalue()
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    ct = CO.Tables(json.loads(edges_text), alt_len_from_gfa_text(gfa_text))
    co = cohort.Cohort(t, 3)
    dicts = []
    for s in range(3):
        gaf = (gaf0 if s == 0 else synth.simulate_gaf(g, len(gaf0.splitlines()) // 2, seed=500 + s, mean_len=31000)).encode()
        co.filter(s, gaf)
        want = CO.filter_counts(ct, gaf)[0]
        assert (co.counts(s) == want).all()
        dicts.append(CO.counts_dict(ct, want))
    names = ["a", "b", "c"]
    got = cohort.genotype_cohort_vcf(t, co, vcf.encode(), names)
    assert got == oracle_cohort_vcf(dicts, names, vcf.splitlines(True))
    assert min(got[1]) > 1000
