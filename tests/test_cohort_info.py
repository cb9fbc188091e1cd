"""Population INFO tags of the cohort VCF (genotype-cohort.py --info-tags; svjg_cohort_site_stats on the device,
svjg_vcf_format_cohort_tags on the host).
The Python statement of the tags is here: `hwe_exchet` (the HWE exact test and the excess-heterozygosity p in the
streaming double-precision form of DESIGN.md §8a) and `add_info_tags` (the text: INFO rewritten from the cells of each
record, ##INFO lines replaced), applied on top of the cohort composition of test_cohort.py.
CPU part: the oracle's p-values against exact rational arithmetic, the formatter against the Python text with
oracle-supplied statistics, the command line's argument checks.
GPU part (-m gpu): the kernel's counts and p-values bit for bit against the oracle, and the command line against the
oracle composition plus the oracle tags."""
import ctypes as C
import os
import random
import re
from fractions import Fraction

import numpy as np
import pytest

from conftest import read_golden
from svjg import capi, cohort, genotype
from test_cohort import (GOLDEN_TAGS, _cohort, _format_cohort, _fuzz_vcfs, _golden_vcf, _python_cohort_text,
                         _python_oracle_counts, _random_cells, _synthetic, _write_inputs, oracle_cohort_vcf)

TAGS = cohort.INFO_TAGS
INFO_HEADER = {
    "NS": '##INFO=<ID=NS,Number=1,Type=Integer,Description="Number of samples with data">\n',
    "AN": '##INFO=<ID=AN,Number=1,Type=Integer,Description="Total number of alleles in called genotypes">\n',
    "AC": '##INFO=<ID=AC,Number=A,Type=Integer,Description="Allele count in genotypes">\n',
    "AF": '##INFO=<ID=AF,Number=A,Type=Float,Description="Allele frequency">\n',
    "AC_Het": '##INFO=<ID=AC_Het,Number=A,Type=Integer,Description="Allele counts in heterozygous genotypes">\n',
    "AC_Hom": '##INFO=<ID=AC_Hom,Number=A,Type=Integer,Description="Allele counts in homozygous genotypes">\n',
    "F_MISSING": '##INFO=<ID=F_MISSING,Number=1,Type=Float,Description="Fraction of missing genotypes">\n',
    "HWE": '##INFO=<ID=HWE,Number=A,Type=Float,Description="HWE test (PMID:15789306); 1=good, 0=bad">\n',
    "ExcHet": '##INFO=<ID=ExcHet,Number=A,Type=Float,Description="Test excess heterozygosity; 1=good, 0=bad">\n',
}
PER_ALT = {"AC", "AF", "AC_Het", "AC_Hom", "HWE", "ExcHet"}


# ---------------------------------------------------------------------------------------------------------------
# the Python statement
# ---------------------------------------------------------------------------------------------------------------
def _walk(r0, h, r2):
    """The terms (k, v) of the walk in order: mid's 1.0, the down walk, the up walk."""
    n = r0 + h + r2
    rare = 2 * min(r0, r2) + h
    mid = rare * (2 * n - rare) // (2 * n)
    if (mid ^ rare) & 1:
        mid += 1
    terms = [(mid, 1.0)]
    k, homr, v = mid, (rare - mid) // 2, 1.0
    homc = n - mid - homr
    while k >= 2:
        v = v * float(k * (k - 1)) / float(4 * (homr + 1) * (homc + 1))
        k, homr, homc = k - 2, homr + 1, homc + 1
        terms.append((k, v))
    k, homr, v = mid, (rare - mid) // 2, 1.0
    homc = n - mid - homr
    while k <= rare - 2:
        v = v * float(4 * homr * homc) / float((k + 2) * (k + 1))
        k, homr, homc = k + 2, homr - 1, homc - 1
        terms.append((k, v))
    return terms


def hwe_exchet(r0, h, r2):
    """(HWE, ExcHet) of one record's genotype counts, every operation one IEEE double rounded to nearest."""
    if 2 * min(r0, r2) + h == 0:
        return 1.0, 1.0
    terms = _walk(r0, h, r2)
    total = 0.0
    v_obs = 0.0
    for k, v in terms:                               # pass 1
        total += v
        if k == h:
            v_obs = v
    acc_hwe = acc_exc = 0.0
    for k, v in terms:                               # pass 2: the same terms in the same order
        if v <= v_obs:
            acc_hwe += v
        if k >= h:
            acc_exc += v
    return min(1.0, acc_hwe / total), min(1.0, acc_exc / total)


def _g6(x):
    return "%.6g" % x


def _tag_values(r0, h, r2, m, multi_alt):
    ns = r0 + h + r2
    hwe, exc = hwe_exchet(r0, h, r2) if ns else (None, None)
    vals = {"NS": str(ns), "AN": str(2 * ns), "AC": str(h + 2 * r2), "AF": _g6((h + 2 * r2) / (2 * ns)) if ns else ".",
            "AC_Het": str(h), "AC_Hom": str(2 * r2), "F_MISSING": _g6(m / (ns + m)),
            "HWE": _g6(hwe) if ns else ".", "ExcHet": _g6(exc) if ns else "."}
    if multi_alt:
        vals.update({t: "." for t in PER_ALT})
    return vals


def _lines(text):
    """The lines of a catalogue as the native parser reads them (text mode: "\\r\\n" and "\\r" end a line)."""
    return re.findall(r"[^\n]*\n|[^\n]+$", text.replace("\r\n", "\n").replace("\r", "\n"))


def add_info_tags(text, vcf_lines, tags):
    """The cohort VCF ``text`` (written without tags for the catalogue ``vcf_lines``) with the INFO tags ``tags``:
    each record's INFO loses its items keyed by a selected tag and gains TAG=value, counted from its sample cells;
    ##INFO lines of a selected ID are dropped and the new ones go in front of the ##FORMAT lines."""
    tags = [t for t in TAGS if t in tags]
    pieces = _lines(text)
    out, j = [], 0
    for line in vcf_lines:
        if line.startswith("##FORMAT"):
            continue
        if line.startswith("##"):
            p = pieces[j]
            j += 1
            if not any(p.startswith(f"##INFO=<ID={t},") or p.startswith(f"##INFO=<ID={t}>") for t in tags):
                out.append(p)
        elif line.startswith("#C"):
            out += [INFO_HEADER[t] for t in tags] + pieces[j:j + 5]
            j += 5
        else:
            cols = pieces[j].rstrip("\n").split("\t")
            j += 1
            gts = [c.split(":")[0] for c in cols[9:]]
            r0, h, r2 = gts.count("0/0"), gts.count("0/1"), gts.count("1/1")
            vals = _tag_values(r0, h, r2, len(gts) - r0 - h - r2, "," in cols[4])
            items = [] if cols[7] in (".", "") else cols[7].split(";")
            kept = [it for it in items if it.split("=", 1)[0] not in tags]
            cols[7] = ";".join(kept + [f"{t}={vals[t]}" for t in tags])
            out.append("\t".join(cols) + "\n")
    assert j == len(pieces)
    return "".join(out)


def _oracle_stats(gt, fl, S):
    """gcount [n][4], hwe [n], exchet [n] of cells as the text shows them (a cell not genotyped is ./.)."""
    g = np.where(fl & capi.GT_GENOTYPED, gt, 3).reshape(-1, S)
    gcount = np.stack([(g == 0).sum(1), (g == 1).sum(1), (g == 2).sum(1), (g == 3).sum(1)], axis=1).astype(np.uint32)
    p = np.array([hwe_exchet(int(a), int(b), int(c)) for a, b, c, _m in gcount], np.float64).reshape(-1, 2)
    return gcount, np.ascontiguousarray(p[:, 0]), np.ascontiguousarray(p[:, 1])


def _format_tags(v, lo, hi, names, gt, fl, ad, pl, mask, gcount, hwe, exc, n_gt=None):
    joined = "\t".join(names).encode()
    arrs = [np.ascontiguousarray(a) for a in (gt, fl, ad, pl, gcount, hwe, exc)]
    n_gt = np.zeros(len(names), np.uint64) if n_gt is None else n_gt
    buf, n_out = C.c_void_p(), C.c_uint64()
    rc = capi.lib.svjg_vcf_format_cohort_tags(v._h, lo, hi, len(names), joined, len(joined),
                                              *(a.ctypes.data for a in arrs[:4]), mask,
                                              *(a.ctypes.data for a in arrs[4:]), C.byref(buf), C.byref(n_out),
                                              n_gt.ctypes.data)
    capi.check(rc)
    try:
        return C.string_at(buf.value, n_out.value).decode("ascii")
    finally:
        capi.lib.svjg_buffer_free(buf)


def _mask(tags):
    return cohort.info_tags_mask(tags)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the exact tests against rational arithmetic
# ---------------------------------------------------------------------------------------------------------------
_FACT = [1]


def _fact(n):
    while len(_FACT) <= n:
        _FACT.append(_FACT[-1] * len(_FACT))
    return _FACT[n]


def _exact(r0, h, r2):
    """The genotype-count distribution in closed form (Levene): P(k) is proportional to N! 2^k / (homr! k! homc!),
    an integer.  Returns the exact HWE p, the one that counts the terms within 1e-9 of P(h) as ties, and ExcHet."""
    n = r0 + h + r2
    rare = 2 * min(r0, r2) + h
    w = {}
    for k in range(rare % 2, rare + 1, 2):
        homr = (rare - k) // 2
        w[k] = _fact(n) * 2 ** k // (_fact(homr) * _fact(k) * _fact(n - k - homr))
    total = sum(w.values())
    obs = w[h]
    strict = Fraction(sum(x for x in w.values() if x <= obs), total)
    loose = Fraction(sum(x for x in w.values() if x * 10 ** 9 <= obs * (10 ** 9 + 1)), total)
    exc = Fraction(sum(x for k, x in w.items() if k >= h), total)
    return strict, loose, exc


def _agrees(x, p):
    return abs(Fraction(x) - p) <= p * Fraction(1, 10 ** 12) or (x < 1e-300 and p < Fraction(1e-300))


def _check_exact(r0, h, r2):
    hwe, exc = hwe_exchet(r0, h, r2)
    strict, loose, p_exc = _exact(r0, h, r2)
    assert _agrees(hwe, min(strict, 1)) or _agrees(hwe, min(loose, 1)), (r0, h, r2, hwe, float(strict))
    assert _agrees(exc, min(p_exc, 1)), (r0, h, r2, exc, float(p_exc))


def test_exact_tests_against_rationals_small_n():
    n_checked = 0
    for n in range(1, 41):
        for r0 in range(n + 1):
            for h in range(n + 1 - r0):
                _check_exact(r0, h, n - r0 - h)
                n_checked += 1
    assert n_checked == sum((n + 1) * (n + 2) // 2 for n in range(1, 41))


def test_exact_tests_against_rationals_large_n():
    rng = random.Random(2005)
    cases = [(0, 2000, 0), (1000, 0, 1000), (1999, 1, 0), (0, 1, 1999), (1, 1998, 1), (500, 1000, 500)]
    for _ in range(30):
        n = rng.randint(41, 2000)
        r0 = rng.randint(0, n)
        h = rng.randint(0, n - r0)
        cases.append((r0, h, n - r0 - h))
    tiny = 0
    for r0, h, r2 in cases:
        _check_exact(r0, h, r2)
        tiny += hwe_exchet(r0, h, r2)[0] < 1e-100
    assert tiny >= 3                                        # the far tails are among the cases


def test_exact_tests_fixed_points():
    assert hwe_exchet(5, 0, 0) == (1.0, 1.0) and hwe_exchet(0, 0, 7) == (1.0, 1.0)
    assert hwe_exchet(0, 0, 0) == (1.0, 1.0)
    hwe, exc = hwe_exchet(0, 40, 0)                         # all het: far from equilibrium, excess of het
    assert hwe < 1e-10 and exc < 1e-10
    hwe, exc = hwe_exchet(20, 0, 20)                        # no het at all
    assert hwe < 1e-10 and exc == 1.0


# ---------------------------------------------------------------------------------------------------------------
# CPU: the formatter
# ---------------------------------------------------------------------------------------------------------------
_CATALOGUE = (
    "##fileformat=VCFv4.2\n"
    '##INFO=<ID=SVTYPE,Number=1,Type=String,Description="Type of structural variant">\n'
    '##INFO=<ID=END,Number=1,Type=Integer,Description="End position">\n'
    '##INFO=<ID=AF,Number=A,Type=Float,Description="Allele frequency of the catalogue">\n'
    '##INFO=<ID=AC>\n'
    '##INFO=<ID=AFX,Number=1,Type=Float,Description="kept">\n'
    '##INFO=<ID=XAF,Number=1,Type=Float,Description="kept">\n'
    '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n'
    "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\told\n"
    "chr1\t1000\tdel1\tN\t<DEL>\t.\tPASS\tSVTYPE=DEL;END=1600;AF=0.25;AC=3;NS=9;AFX=0.1;XAF=2\tGT\t0/1\n"
    "chr1\t2000\tins1\tN\t<INS>\t.\tPASS\tSVTYPE=INS;AF;AC_Het=4;;HWE=0.5\n"
    "chr1\t3000\tdel2\tN\t<DEL>,<INS>\t.\tPASS\tSVTYPE=DEL;END=3900;ExcHet=1\n"
    "chr2\t500\tbnd1\tN\tN[chr3:100[\t.\tPASS\tSVTYPE=BND;F_MISSING=0\n"
    "chr2\t5000\tinv1\tN\t<INV>\t.\tPASS\tEND=7000;SVTYPE=INV\n"
    "chr2\t9000\tdel3\tN\t<DEL>\t.\tPASS\tSVTYPE=DEL;END=9900;AN=4;AC_Hom=2\n"
    '##INFO=<ID=HWE,Number=A,Type=Float,Description="trailing">\n'
    '##INFO=<ID=HWEX,Number=A,Type=Float,Description="trailing, kept">\n'
)


def _cells_with_missing_record(rng, n, S, missing_record):
    gt, fl, ad, pl = _random_cells(rng, n * S)
    fl[missing_record * S:(missing_record + 1) * S] = 0          # NS = 0
    return gt, fl, ad, pl


def test_every_tag_subset_in_canonical_order():
    v = genotype.NativeVcf.from_input(_CATALOGUE.encode())
    S, names = 7, [f"s{k}" for k in range(7)]
    rng = np.random.default_rng(3)
    gt, fl, ad, pl = _cells_with_missing_record(rng, v.n, S, 4)
    stats = _oracle_stats(gt, fl, S)
    lines = _lines(_CATALOGUE)
    base = _python_cohort_text(lines, names, gt, fl, ad, pl)
    assert _format_cohort(v, 0, v.n, names, gt, fl, ad, pl, np.zeros(S, np.uint64)) == base
    for mask in range(1 << len(TAGS)):
        tags = [t for k, t in enumerate(TAGS) if mask >> k & 1]
        shuffled = tags[:]
        random.Random(mask).shuffle(shuffled)
        if tags:
            assert cohort.parse_info_tags(",".join(shuffled)) == tuple(tags)
        assert _mask(shuffled) == mask
        got = _format_tags(v, 0, v.n, names, gt, fl, ad, pl, mask, *stats)
        assert got == add_info_tags(base, lines, tags), tags
    allt = _format_tags(v, 0, v.n, names, gt, fl, ad, pl, _mask(TAGS), *stats)
    body = [ln.split("\t") for ln in allt.splitlines() if not ln.startswith("#")]
    assert body[0][7].startswith("SVTYPE=DEL;END=1600;AFX=0.1;XAF=2;NS=")           # AF, AC, NS dropped
    assert body[1][7].startswith("SVTYPE=INS;;NS=")                                # flag AF dropped, empty item kept
    assert ";AC=.;AF=.;AC_Het=.;AC_Hom=.;F_MISSING=" in body[2][7] and body[2][7].endswith("HWE=.;ExcHet=.")
    assert body[4][7] == "END=7000;SVTYPE=INV;NS=0;AN=0;AC=0;AF=.;AC_Het=0;AC_Hom=0;F_MISSING=1;HWE=.;ExcHet=."
    for kept in ("SVTYPE", "END", "AFX", "XAF", "HWEX"):
        assert f"##INFO=<ID={kept}," in allt
    assert "##INFO=<ID=AC>" not in allt and "catalogue" not in allt and 'Description="trailing"' not in allt
    assert allt.index("##INFO=<ID=NS,") < allt.index("##FORMAT=<ID=GT")


def test_f_missing_in_e_notation_and_counts_that_do_not_add_up():
    text = ("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n"
            "chr1\t100\ta\tN\t<INV>\t.\tPASS\tSVTYPE=INV;END=900\n"
            "chr1\t2000\tb\tN\t<INV>\t.\tPASS\tSVTYPE=INV;END=2900\n"
            "chr1\t4000\tc\tN\t<INV>\t.\tPASS\tSVTYPE=INV;END=4900\n")
    v = genotype.NativeVcf.from_input(text.encode())
    S = 12000
    names = [f"x{k}" for k in range(S)]
    rng = np.random.default_rng(5)
    gt, fl, ad, pl = _random_cells(rng, 3 * S)
    fl[:] |= capi.GT_GENOTYPED
    gt[:] = rng.integers(0, 3, 3 * S)
    gt[7] = 3                                                   # record 0: one missing cell in 12 000
    fl[S + 5] = 0                                               # record 1: one cell not genotyped
    stats = _oracle_stats(gt, fl, S)
    got = _format_tags(v, 0, 3, names, gt, fl, ad, pl, _mask(TAGS), *stats)
    lines = _lines(text)
    assert got == add_info_tags(_python_cohort_text(lines, names, gt, fl, ad, pl), lines, TAGS)
    infos = [ln.split("\t")[7] for ln in got.splitlines() if not ln.startswith("#")]
    assert "F_MISSING=8.33333e-05" in infos[0] and "F_MISSING=8.33333e-05" in infos[1] and "F_MISSING=0;" in infos[2]
    bad = stats[0].copy()
    bad[1, 3] += 1
    with pytest.raises(capi.SvjgError, match="add up"):
        _format_tags(v, 0, 3, names, gt, fl, ad, pl, _mask(["NS"]), bad, stats[1], stats[2])
    with pytest.raises(capi.SvjgError, match="INFO tag bit"):
        _format_tags(v, 0, 3, names, gt, fl, ad, pl, 1 << len(TAGS), *stats)


@pytest.mark.parametrize("tag", GOLDEN_TAGS)
def test_golden_catalogues_blocks_and_mask_zero(tag):
    text = _golden_vcf(tag) + '##INFO=<ID=AF,Number=A,Type=Float,Description="x">\n'
    v = genotype.NativeVcf.from_input(text.encode())
    S, names = 5, [f"s{k}" for k in range(5)]
    rng = np.random.default_rng(11)
    gt, fl, ad, pl = _random_cells(rng, v.n * S)
    stats = _oracle_stats(gt, fl, S)
    lines = _lines(text)
    base = _format_cohort(v, 0, v.n, names, gt, fl, ad, pl, np.zeros(S, np.uint64))
    assert _format_tags(v, 0, v.n, names, gt, fl, ad, pl, 0, *stats) == base
    for tags in (TAGS, ("AF", "HWE"), ("NS", "F_MISSING", "ExcHet")):
        mask = _mask(tags)
        whole = _format_tags(v, 0, v.n, names, gt, fl, ad, pl, mask, *stats)
        assert whole == add_info_tags(base, lines, tags)
        for step in (1, 7):
            n_gt = np.zeros(S, np.uint64)
            pieces = [_format_tags(v, lo, min(v.n, lo + step), names, gt[lo * S:(lo + step) * S],
                                   fl[lo * S:(lo + step) * S], ad[lo * S:(lo + step) * S], pl[lo * S:(lo + step) * S],
                                   mask, *(a[lo:lo + step] for a in stats), n_gt=n_gt)
                      for lo in range(0, v.n, step)]
            assert "".join(pieces) == whole
            assert n_gt.tolist() == [int(((fl[s::S] & capi.GT_GENOTYPED) != 0).sum()) for s in range(S)]


def test_fuzz_catalogues():
    rng = np.random.default_rng(17)
    n_checked = 0
    for k, text in enumerate(_fuzz_vcfs()):
        try:
            v = genotype.NativeVcf.from_input(text.encode())
        except genotype.VcfError:
            continue
        if v is None:
            continue
        S, names = 3, ["a", "b", "c"]
        gt, fl, ad, pl = _random_cells(rng, v.n * S)
        stats = _oracle_stats(gt, fl, S)
        base = _format_cohort(v, 0, v.n, names, gt, fl, ad, pl, np.zeros(S, np.uint64))
        tags = TAGS if k % 2 else [t for t in TAGS if rng.random() < 0.5]
        assert _format_tags(v, 0, v.n, names, gt, fl, ad, pl, 0, *stats) == base
        assert _format_tags(v, 0, v.n, names, gt, fl, ad, pl, _mask(tags), *stats) == \
            add_info_tags(base, _lines(text), tags)
        n_checked += 1
    assert n_checked > 500


@pytest.mark.parametrize("value,message", [
    ("bogus", "unknown INFO tag"),
    ("NS,NS", "twice"),
    ("", "unknown INFO tag ''"),
    ("NS,,AF", "unknown INFO tag ''"),
    ("all,NS", "unknown INFO tag 'all'"),
    ("af", "unknown INFO tag 'af'"),
])
def test_command_line_refuses_bad_info_tags_before_the_device(tmp_path, value, message):
    args = ["-p", str(tmp_path / "x"), "-g", "x.gfa", "-v", "x.vcf", "-a", "one.gaf", "-o", str(tmp_path / "out.vcf"),
            "--info-tags", value]
    # no CUDA device: a check that came after the device start would fail with another message
    r = _cohort(*args, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and "--info-tags" in r.stderr and message in r.stderr, r.stderr
    assert not os.listdir(tmp_path)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
# counters that give 0/0, 0/1, 1/1 and ./. (no hit: outside the gate) for an INV record, whatever -e
_GT_COUNTS = np.array([[20, 0], [10, 10], [0, 20], [0, 0]], np.uint32)


def _kernel_case(t, S, n, seed, special=True):
    """A cohort of S samples whose genotype in record i is drawn from a per-record mix: the counters of
    _GT_COUNTS per sample and SV; then the last records are all-het, all-hom-alt, monomorphic, and nobody's."""
    rng = np.random.default_rng(seed)
    co = cohort.Cohort(t, S)
    mix = rng.dirichlet([0.5, 0.5, 0.5, 0.2], n)
    mix[rng.random(n) < 0.3, 3] = 0
    mix /= mix.sum(1, keepdims=True)
    want_g = np.stack([rng.choice(4, S, p=mix[i]) for i in range(n)])          # [n][S]
    if special and n >= 6:
        want_g[-6:] = [[1], [2], [0], [3], [0], [1]]                             # rows broadcast over the samples
    for s in range(S):
        c = np.zeros((t.num_sv, 2), np.uint32)
        c[:n] = _GT_COUNTS[want_g[:, s]]
        co.load_counts(s, c)
    idx = np.arange(n, dtype=np.uint32)
    ty = np.full(n, 2, np.uint8)                                              # INV: no halving
    if special and n >= 6:
        idx[-2] = capi.NO_SV                                                  # not in the tables
        ty[-1] = 255                                                          # not a genotyped type
    return co, idx, ty, want_g


def _check_kernel(co, idx, ty, S):
    n = len(idx)
    blk = cohort._Block(n * S, n)
    gt, fl, _ad, _pl = cohort._genotype_block(co, idx, ty, 3, genotype.ERR, blk)
    gcount, hwe, exc = (a.copy() for a in cohort._site_stats(co, n, blk))
    w_count, w_hwe, w_exc = _oracle_stats(gt, fl, S)
    assert (gcount == w_count).all()
    assert (hwe.view(np.uint64) == w_hwe.view(np.uint64)).all()
    assert (exc.view(np.uint64) == w_exc.view(np.uint64)).all()
    return gcount, hwe, exc


@pytest.mark.gpu
@pytest.mark.parametrize("S,n", [(40, 500), (3000, 300), (1, 500)])
def test_kernel_equals_the_oracle_bit_for_bit(S, n):
    from svjg import alnfilter
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    assert t.num_sv >= n
    co, idx, ty, want_g = _kernel_case(t, S, n, seed=S)
    gcount, hwe, exc = _check_kernel(co, idx, ty, S)
    # the counters gave the genotypes they were chosen for
    want = np.stack([(want_g == g).sum(1) for g in range(4)], axis=1)
    want[-2:] = [0, 0, 0, S]
    assert (gcount == want).all()
    assert gcount[-6].tolist() == [0, S, 0, 0] and gcount[-5].tolist() == [0, 0, S, 0]
    assert gcount[-4].tolist() == [S, 0, 0, 0] and gcount[-3].tolist() == [0, 0, 0, S]
    assert hwe[-5] == exc[-5] == hwe[-4] == exc[-4] == 1.0
    if S == 3000:
        assert hwe[-6] == exc[-6] == 0.0                                  # all het: the observed term underflows
        assert (hwe[:-6] < 1e-300).any() and (hwe[:-6] > 0.5).any()
    # a call that does not follow the block it reads is refused
    with pytest.raises(capi.SvjgError, match="record count"):
        capi.check(capi.lib.svjg_cohort_site_stats(co._h, n + 1, gcount.ctypes.data, hwe.ctypes.data, exc.ctypes.data))


def _s2_cohort(tmp_path):
    p = _write_inputs(tmp_path, "s2")
    gaf = read_golden("s2.gaf.gz")
    lines = gaf.splitlines(True)
    files = {"whole": gaf, "half1": "".join(lines[:len(lines) // 2]), "half2": "".join(lines[len(lines) // 2:]),
             "x48": gaf * 48, "empty": ""}
    for name, text in files.items():
        open(f"{p}_{name}.gaf", "w").write(text)
    samples = [[f"{p}_whole.gaf"], [f"{p}_half1.gaf"], [f"{p}_half2.gaf"], [f"{p}_x48.gaf"], [f"{p}_empty.gaf"],
               [f"{p}_whole.gaf"], [f"{p}_half1.gaf", f"{p}_half2.gaf"]]
    texts = [gaf, files["half1"], files["half2"], files["x48"], "", gaf, gaf]
    per_text = {}
    for text in texts:
        if text not in per_text and text != files["x48"]:
            per_text[text] = _python_oracle_counts("s2", text)
    per_text[files["x48"]] = {k: (48 * a, 48 * b) for k, (a, b) in per_text[gaf].items()}
    return p, samples, [per_text[x] for x in texts]


@pytest.mark.gpu
def test_s2_cohort_with_info_tags(tmp_path):
    from svjg import alnfilter, cli
    p, samples, counts = _s2_cohort(tmp_path)
    names = [f"n{k}" for k in range(7)]
    vcf = _golden_vcf("s2")
    base, want_n = oracle_cohort_vcf(counts, names, vcf.splitlines(True))
    want = add_info_tags(base, _lines(vcf), TAGS)
    assert want != base and "HWE=" in want
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *[",".join(fs) for fs in samples], "-o", p + "_t.vcf",
                "--names", ",".join(names), "--info-tags", "all")
    assert r.returncode == 0, r.stderr
    assert open(p + "_t.vcf").read() == want
    assert r.stdout == "".join(f"Genotyped svs in {nm}: {n}\n" for nm, n in zip(names, want_n))
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *[",".join(fs) for fs in samples], "-o", p + "_u.vcf",
                "--names", ",".join(names), "--info-tags", "HWE,AF,NS")
    assert r.returncode == 0, r.stderr
    assert open(p + "_u.vcf").read() == add_info_tags(base, _lines(vcf), ("NS", "AF", "HWE"))
    # the module, blocks forced small
    t = alnfilter.Tables.from_memory(read_golden("s2_svs_edges.json.gz"), read_golden("s2.gfa.gz")).to_device(0)
    co = cohort.Cohort(t, 7)
    for k, fs in enumerate(samples):
        for b in cli._read_sample(fs):
            co.filter(k, b.array)
    assert (co.counts(3) > 256).any()                                   # NEED_K cells: patched on the host
    for block in (None, 1, 7):
        assert cohort.genotype_cohort_vcf(t, co, vcf.encode(), names, block_records=block, info_tags=TAGS) == (want, want_n)


@pytest.mark.gpu
def test_need_k_cohort_with_info_tags(tmp_path):
    p, _samples, _counts = _s2_cohort(tmp_path)
    base_counts = _python_oracle_counts("s2", read_golden("s2.gaf.gz"))
    vcf = _golden_vcf("s2")
    names = ["x48", "one"]
    base, _n = oracle_cohort_vcf([{k: (48 * a, 48 * b) for k, (a, b) in base_counts.items()}, base_counts], names,
                                 vcf.splitlines(True))
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", f"{p}_x48.gaf", f"{p}_whole.gaf", "-o", p + "_k.vcf",
                "--names", ",".join(names), "--info-tags", "all")
    assert r.returncode == 0, r.stderr
    assert open(p + "_k.vcf").read() == add_info_tags(base, _lines(vcf), TAGS)


@pytest.mark.gpu
def test_without_the_switch_the_file_is_unchanged(tmp_path):
    p = _write_inputs(tmp_path, "c1")
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", p + ".gaf", "-o", p + "_g.vcf", "--names", "SAMPLE")
    assert r.returncode == 0, r.stderr
    assert open(p + "_g.vcf").read() == read_golden("c1_genotype.vcf")
