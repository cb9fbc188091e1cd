"""Sex-chromosome ploidy of the cohort VCF (genotype-cohort.py --ploidy-file / --sample-sex; PloidyRules in
svjg/cohort.py, svjg_cohort_genotype_ploidy and svjg_cohort_site_stats_ploidy on the device,
svjg_vcf_format_cohort_ploidy on the host).
The Python statement is here:
  * the ploidy of a cell (`ploidy_of`): the rule for the sample's sex whose CHROM is the record's CHROM column and whose
    [FROM, TO] holds its POS column, else the sex's `* * *` default, else 2;
  * a haploid cell (`haploid_call`): genotype_counts' exact Fraction sums L0 and L2 (oracle/svjg_oracle.py) compared,
    "0" if L0 > L2, "1" if L2 > L0, "." on a tie or below -ms, with PL[0] and PL[2] of the diploid cell; a ploidy-0 cell
    is ".:DP:AD:." (".:0:0,0:." outside the gate), a haploid cell outside the gate ".:0:0,0:.,.";
  * the tags (`add_ploidy_tags`): NS = r0 + h + r2 + a0 + a1, AN = 2 (r0 + h + r2) + a0 + a1, AC = h + 2 r2 + a1,
    AF = AC / AN, AC_Het = h, AC_Hom = 2 r2, F_MISSING = m / S, HWE and ExcHet of (r0, h, r2), AC_Hemi = a1;
applied on top of the cohort composition of test_cohort.py.
CPU part: both file parsers, the record classes, the formatter, the command line's checks.  GPU part (-m gpu): the
kernels against the statement cell by cell and bit for bit, and the command line against the oracle composition."""
import ctypes as C
import math
import os
import random
from fractions import Fraction

import numpy as np
import pytest

from conftest import read_golden
from oracle import svjg_oracle as O
from svjg import capi, cohort, genotype
from test_cohort import (GOLDEN_TAGS, _cell_text, _cohort, _fuzz_vcfs, _golden_vcf, _python_oracle_counts,
                         _random_cells, _synthetic, oracle_cohort_vcf)
from test_cohort_info import (_CATALOGUE, INFO_HEADER, PER_ALT, _format_tags, _g6, _lines, _s2_cohort, add_info_tags,
                              hwe_exchet)

TAGS = cohort.PLOIDY_INFO_TAGS
HEADER = dict(INFO_HEADER, AC_Hemi='##INFO=<ID=AC_Hemi,Number=A,Type=Integer,Description="Allele counts in hemizygous '
                                   'genotypes">\n')
PL3 = '##FORMAT=<ID=PL,Number=3,Type=Integer,Description="Phred-scaled likelihood for each genotype">\n'
PLG = PL3.replace("Number=3", "Number=G")
SVTYPE_NAME = {0: "DEL", 1: "INS", 2: "INV", 3: "BND"}


# ---------------------------------------------------------------------------------------------------------------
# the Python statement
# ---------------------------------------------------------------------------------------------------------------
def ploidy_of(rules, defaults, chrom, pos, sex):
    """rules: (chrom, from, to, sex, ploidy) tuples; defaults: sex -> ploidy."""
    for c, lo, hi, x, p in rules:
        if c == chrom and x == sex and lo <= pos <= hi:
            return p
    return defaults.get(sex, 2)


def haploid_call(n0, n1, svtype, min_support=3, e=0.00005):
    """(GT text, PL0, PL2) of a haploid cell that passes the gate: the sums of genotype_counts, L0 and L2 only."""
    t1, t2 = 2 * n0, 2 * n1
    h1 = h2 = False
    if svtype == "DEL" and n0 > 0:
        t1, h1 = n0, True
    elif svtype == "INS" and n1 > 0:
        t2, h2 = n1, True
    c1 = t1 / 2 if h1 else t1 // 2
    c2 = t2 / 2 if h2 else t2 // 2
    a, b = math.log10(1 - e), math.log10(e)
    l0 = Fraction(c1 * a) + Fraction(c2 * b)
    l2 = Fraction(c2 * a) + Fraction(c1 * b)
    gt = "0" if l0 > l2 else "1" if l2 > l0 else "."
    if t1 + t2 < 2 * min_support:
        gt = "."
    pl = O.genotype_counts(n0, n1, svtype, min_support, e)[3]
    return gt, pl[0], pl[2]


def _ploidy_cell_text(g, f, t1, t2, pl):
    if g <= 3:
        return _cell_text(g, f, t1, t2, pl)
    if not f & capi.GT_GENOTYPED:
        return ".:0:0,0:." if g == capi.GT_NO_CALL else ".:0:0,0:.,."
    h0, h1 = bool(f & capi.GT_HALVED_0), bool(f & capi.GT_HALVED_1)
    dp_ad = f"{O._py_num_str(t1 + t2, h0 or h1)}:{O._py_num_str(t1, h0)},{O._py_num_str(t2, h1)}"
    if g == capi.GT_NO_CALL:
        return f".:{dp_ad}:."
    return f"{'01.'[g - capi.GT_HAP_REF]}:{dp_ad}:{pl[0]},{pl[2]}"


def _python_ploidy_text(lines, names, gt, fl, ad, pl):
    """The ploidy formatter's text without tags: the cohort text with the cells above and PL Number=G."""
    header, recs = genotype.parse_vcf(lines)
    S = len(names)
    col = (genotype._FORMAT_LINES[:-len("SAMPLE\n")] + "\t".join(names) + "\n").replace(PL3, PLG)
    out, hi = [], 0

    def hdr(text):
        return col if text == genotype._FORMAT_LINES else text
    for i, (head, _code, _key) in enumerate(recs):
        while hi < len(header) and header[hi][0] <= i:
            out.append(hdr(header[hi][1]))
            hi += 1
        k = range(i * S, i * S + S)
        out.append(head + "\tGT:DP:AD:PL" + "".join(
            "\t" + _ploidy_cell_text(int(gt[c]), int(fl[c]), int(ad[c, 0]), int(ad[c, 1]), pl[c].tolist()) for c in k)
            + "\n")
    out += [hdr(h[1]) for h in header[hi:]]
    return "".join(out)


def _ploidy_tag_values(r0, h, r2, a0, a1, m, multi_alt):
    dip = r0 + h + r2
    ns, an, ac = dip + a0 + a1, 2 * dip + a0 + a1, h + 2 * r2 + a1
    hwe, exc = hwe_exchet(r0, h, r2) if dip else (None, None)
    vals = {"NS": str(ns), "AN": str(an), "AC": str(ac), "AF": _g6(ac / an) if an else ".", "AC_Het": str(h),
            "AC_Hom": str(2 * r2), "F_MISSING": _g6(m / (ns + m)), "HWE": _g6(hwe) if dip else ".",
            "ExcHet": _g6(exc) if dip else ".", "AC_Hemi": str(a1)}
    if multi_alt:
        vals.update({t: "." for t in PER_ALT | {"AC_Hemi"}})
    return vals


def add_ploidy_tags(text, vcf_lines, tags):
    """add_info_tags of test_cohort_info.py with the counts of haploid calls ("0", "1") and AC_Hemi."""
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
            out += [HEADER[t] for t in tags] + pieces[j:j + 5]
            j += 5
        else:
            cols = pieces[j].rstrip("\n").split("\t")
            j += 1
            gts = [c.split(":")[0] for c in cols[9:]]
            n = [gts.count(g) for g in ("0/0", "0/1", "1/1", "0", "1")]
            vals = _ploidy_tag_values(*n, len(gts) - sum(n), "," in cols[4])
            items = [] if cols[7] in (".", "") else cols[7].split(";")
            kept = [it for it in items if it.split("=", 1)[0] not in tags]
            cols[7] = ";".join(kept + [f"{t}={vals[t]}" for t in tags])
            out.append("\t".join(cols) + "\n")
    assert j == len(pieces)
    return "".join(out)


def _stats6(gt, fl, S):
    """gcount [n][6], hwe, exchet of cells as the text shows them."""
    g = np.where(fl & capi.GT_GENOTYPED, gt, 3).reshape(-1, S)
    cols = [(g == c).sum(1) for c in (0, 1, 2, capi.GT_HAP_REF, capi.GT_HAP_ALT)]
    gcount = np.stack(cols + [S - sum(cols)], axis=1).astype(np.uint32)
    p = np.array([hwe_exchet(int(a), int(b), int(c)) for a, b, c in gcount[:, :3]], np.float64).reshape(-1, 2)
    return gcount, np.ascontiguousarray(p[:, 0]), np.ascontiguousarray(p[:, 1])


def _format_ploidy(v, lo, hi, names, gt, fl, ad, pl, mask, gcount, hwe, exc, n_gt=None):
    joined = "\t".join(names).encode()
    arrs = [np.ascontiguousarray(a) for a in (gt, fl, ad, pl, gcount, hwe, exc)]
    n_gt = np.zeros(len(names), np.uint64) if n_gt is None else n_gt
    buf, n_out = C.c_void_p(), C.c_uint64()
    capi.check(capi.lib.svjg_vcf_format_cohort_ploidy(v._h, lo, hi, len(names), joined, len(joined),
                                                      *(a.ctypes.data for a in arrs[:4]), mask,
                                                      *(a.ctypes.data for a in arrs[4:]), C.byref(buf), C.byref(n_out),
                                                      n_gt.ctypes.data))
    try:
        return C.string_at(buf.value, n_out.value).decode("ascii")
    finally:
        capi.lib.svjg_buffer_free(buf)


def _ploidy_cells(rng, n_cells):
    """_random_cells with codes 0-7: genotyped and gated cells of every ploidy."""
    gt, fl, ad, pl = _random_cells(rng, n_cells)
    gt[:] = rng.integers(0, 8, n_cells)
    return gt, fl, ad, pl


def _genotyped(gt, fl, S):
    return [int((((fl[s::S] & capi.GT_GENOTYPED) != 0) & (gt[s::S] != capi.GT_NO_CALL)).sum()) for s in range(S)]


# ---------------------------------------------------------------------------------------------------------------
# CPU: the two files
# ---------------------------------------------------------------------------------------------------------------
_LOCI = ("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\n" + "".join(
    f"{c}\t{p}\t{c}_{p}\tN\t<INV>\t.\tPASS\tSVTYPE=INV;END={p + 500}\n"
    for c, p in [("chrX", 1), ("chrX", 2780), ("chrX", 2781), ("chrX", 155701382), ("chrX", 155701383),
                 ("chrY", 10000), ("chr1", 2781), ("X", 5000)]))


def test_accepted_files_with_comments_defaults_and_window_edges():
    pf = ("# GRCh38-like, written by hand\n\n"
          "chrX 1 2780 M 2\n"
          "chrX\t2781\t155701382\tM\t1   # trailing words are a sixth column: not here\n".split("   #")[0] + "\n"
          "  chrY 1 57227415 M 1\n"
          "chrY 1 57227415 F 0\n"
          "* * * M 2\n"
          "# * * * F 1\n"
          "chrX 2781 155701382 U 1\n")
    sf = "# name sex\nb F\n\nnot_in_cohort M\na M\nc U\n"
    r = cohort.PloidyRules(pf, sf, ["a", "b", "c"])
    assert r.sample_sex == ["M", "F", "U"] and r.sexes == ["F", "M", "U"] and r.sex_index.tolist() == [1, 0, 2]
    v = genotype.NativeVcf.from_input(_LOCI.encode())
    rclass, table = r.record_classes(v)
    got = table[rclass].tolist()                           # [record][F, M, U]
    assert got == [[2, 2, 2], [2, 2, 2], [2, 1, 1], [2, 1, 1], [2, 2, 2], [0, 1, 2], [2, 2, 2], [2, 2, 2]]
    assert len(table) == len({tuple(x) for x in got})


def _refused_ploidy(text, match):
    with pytest.raises(ValueError, match=match):
        cohort.PloidyRules(text, "a M\n", ["a"])


@pytest.mark.parametrize("text,match", [
    ("chrX 1 100 M 1\nchrX 100 200 M 1\n", "overlap"),
    ("chrX 1 100 M 1\nchrX 50 60 M 2\n", "overlap"),
    ("chrX 10 20 M 1\nchrX 10 20 M 1\n", "overlap"),
    ("chrX 101 100 M 1\n", "FROM 101 > TO 100"),
    ("chrX 1.5 100 M 1\n", "decimal integers"),
    ("chrX 1 1e9 M 1\n", "decimal integers"),
    ("chrX -1 100 M 1\n", "decimal integers"),
    ("chrX * 100 M 1\n", "decimal integers"),
    ("chrX 1 100 M 3\n", "must be 0, 1 or 2"),
    ("chrX 1 100 M x\n", "must be 0, 1 or 2"),
    ("chrX 1 100 M -1\n", "must be 0, 1 or 2"),
    ("* * * M 4\n", "must be 0, 1 or 2"),
    ("chrX 1 100 M\n", "4 columns"),
    ("chrX 1 100 M 1 2\n", "6 columns"),
    ("* * * M 1\n# c\n* * * M 1\n", "line 3: a second default"),
])
def test_ploidy_file_refusals(text, match):
    _refused_ploidy(text, match)


def _one_class_per_record(n_rec, n_sex=6):
    """Rules that give record i of a catalogue the ploidy digits of i in base 3, one per sex."""
    sexes = [f"s{k}" for k in range(n_sex)]
    r = cohort.PloidyRules("".join(f"chr1 {1000 * i + 1} {1000 * i + 1} {x} {(i // 3 ** k) % 3}\n"
                                   for i in range(n_rec) for k, x in enumerate(sexes)),
                           "".join(f"n{k} {x}\n" for k, x in enumerate(sexes)), [f"n{k}" for k in range(n_sex)])
    text = "".join(f"chr1\t{1000 * i + 1}\tr{i}\tN\t<INV>\t.\tPASS\tSVTYPE=INV;END={1000 * i + 600}\n" for i in range(n_rec))
    return r.record_classes(genotype.NativeVcf.from_input(text.encode()))


def test_rules_of_other_sexes_do_not_overlap_and_limits():
    cohort.PloidyRules("chrX 1 100 M 1\nchrX 1 100 F 2\nchrY 1 100 M 1\n* * * M 2\n* * * F 2\n", "a M\n", ["a"])
    _refused_ploidy("".join(f"* * * s{k} 1\n" for k in range(64)), "65 sex labels")
    cohort.PloidyRules("".join(f"* * * s{k} 1\n" for k in range(63)), "a M\n", ["a"])
    rclass, table = _one_class_per_record(255)
    assert len(table) == 255 and sorted(rclass.tolist()) == list(range(255))
    with pytest.raises(ValueError, match="256 distinct ploidy vectors: at most 255"):
        _one_class_per_record(256)


@pytest.mark.parametrize("text,match", [
    ("a M\n", "no sex for sample 'b'"),
    ("", "no sex for sample 'a' and 1 more"),
    ("a M\nb F\na M\n", "line 3: sample 'a' is listed twice"),
    ("a M\nb\n", "line 2: 1 columns"),
    ("a M extra\nb F\n", "line 1: 3 columns"),
])
def test_sample_sex_refusals(text, match):
    with pytest.raises(ValueError, match=match):
        cohort.PloidyRules("* * * M 1\n", text, ["a", "b"])


@pytest.mark.parametrize("pos", ["1e3", "-5", "+5", "5_0", " 5", ""])
def test_catalogue_pos_must_be_decimal(pos):
    text = f"chrX\t{pos}\tr\tN\t<INS>\t.\tPASS\tSVTYPE=INS\n"
    v = genotype.NativeVcf.from_input(text.encode())
    r = cohort.PloidyRules("chrX 1 10 M 1\n", "a M\n", ["a"])
    with pytest.raises(genotype.VcfError, match="not a decimal integer"):
        r.record_classes(v)


def _random_rules(rng, chroms, max_pos):
    rules, defaults, lines = [], {}, []
    for x in ("M", "F", "U"):
        if rng.random() < 0.5:
            defaults[x] = rng.randint(0, 2)
            lines.append(f"* * * {x} {defaults[x]}")
        for c in rng.sample(chroms, min(len(chroms), rng.randint(0, 4))):
            cuts = sorted(rng.sample(range(1, max_pos + 2), min(max_pos, rng.randint(1, 6)) * 2))
            for lo, hi in zip(cuts[::2], cuts[1::2]):
                hi = hi - 1 if rng.random() < 0.5 and hi > lo else hi
                p = rng.randint(0, 2)
                rules.append((c, lo, hi, x, p))
                lines.append(f"{c}\t{lo} {hi}  {x} {p}")
    rng.shuffle(lines)
    return rules, defaults, "\n".join(lines) + "\n"


def test_record_classes_against_brute_force():
    rng = random.Random(23)
    cats = [_golden_vcf(t) for t in GOLDEN_TAGS] + _fuzz_vcfs()[::7]
    n_checked = 0
    for text in cats:
        try:
            v = genotype.NativeVcf.from_input(text.encode())
        except genotype.VcfError:
            continue
        if v is None or not v.n:
            continue
        recs = [ln.split("\t") for ln in _lines(text) if not ln.startswith("#")]
        try:
            loci = [(c[0], int(c[1])) for c in recs]
        except ValueError:
            with pytest.raises(genotype.VcfError, match="decimal"):
                v.loci()
            continue
        if not all(c[1].isdigit() and len(c[1]) <= 18 for c in recs):
            with pytest.raises(genotype.VcfError, match="decimal"):
                v.loci()
            continue
        chroms = sorted({c for c, _p in loci}) + ["chrNone"]
        max_pos = max(p for _c, p in loci) + 2
        for _ in range(3):
            rules, defaults, ptext = _random_rules(rng, chroms, max_pos)
            # windows that end or start exactly on some record's POS
            c, p = rng.choice(loci)
            if not any(r[0] == c and r[3] == "M" for r in rules):
                rules.append((c, p, p + rng.randint(0, 3), "M", 1))
                ptext += f"{c} {p} {rules[-1][2]} M 1\n"
            r = cohort.PloidyRules(ptext, "a M\nb F\nc U\n", ["a", "b", "c"])
            rclass, table = r.record_classes(v)
            want = [[ploidy_of(rules, defaults, c, p, x) for x in r.sexes] for c, p in loci]
            assert table[rclass].tolist() == want
            assert len(table) == len({tuple(w) for w in want})
            n_checked += 1
    assert n_checked > 150


# ---------------------------------------------------------------------------------------------------------------
# CPU: the formatter
# ---------------------------------------------------------------------------------------------------------------
def test_every_tag_subset_and_the_number_g_header():
    v = genotype.NativeVcf.from_input(_CATALOGUE.encode())
    S, names = 9, [f"s{k}" for k in range(9)]
    rng = np.random.default_rng(29)
    gt, fl, ad, pl = _ploidy_cells(rng, v.n * S)
    fl[4 * S:5 * S] = 0                                     # a record with no call at all
    gt[5 * S:6 * S] = rng.choice([capi.GT_HAP_REF, capi.GT_HAP_ALT, capi.GT_NO_CALL], S)   # no diploid call
    fl[5 * S:6 * S] |= capi.GT_GENOTYPED
    stats = _stats6(gt, fl, S)
    assert stats[0][5, :3].sum() == 0 and stats[0][5, 3:5].sum() > 0
    lines = _lines(_CATALOGUE)
    base = _python_ploidy_text(lines, names, gt, fl, ad, pl)
    assert PLG in base and PL3 not in base
    n_gt = np.zeros(S, np.uint64)
    assert _format_ploidy(v, 0, v.n, names, gt, fl, ad, pl, 0, *stats, n_gt=n_gt) == base
    assert n_gt.tolist() == _genotyped(gt, fl, S)
    for mask in range(1 << len(TAGS)):
        tags = [t for k, t in enumerate(TAGS) if mask >> k & 1]
        shuffled = tags[:]
        random.Random(mask).shuffle(shuffled)
        if tags:
            assert cohort.parse_info_tags(",".join(shuffled), ploidy=True) == tuple(tags)
        assert cohort.info_tags_mask(shuffled) == mask
        assert _format_ploidy(v, 0, v.n, names, gt, fl, ad, pl, mask, *stats) == add_ploidy_tags(base, lines, tags), tags
    body = [ln.split("\t") for ln in _format_ploidy(v, 0, v.n, names, gt, fl, ad, pl, (1 << 10) - 1, *stats)
            .splitlines() if not ln.startswith("#")]
    assert body[2][7].endswith("HWE=.;ExcHet=.;AC_Hemi=.")                          # multi-ALT: Number=A is "."
    assert ";HWE=.;ExcHet=.;AC_Hemi=" in body[5][7] and "AF=." not in body[5][7]    # haploid calls only
    with pytest.raises(capi.SvjgError, match="INFO tag bit"):
        _format_ploidy(v, 0, v.n, names, gt, fl, ad, pl, 1 << 10, *stats)
    bad = gt.copy()
    bad[3] = 8
    with pytest.raises(capi.SvjgError, match="gt code"):
        _format_ploidy(v, 0, v.n, names, bad, fl, ad, pl, 0, *stats)
    # the formatter without ploidy knows neither the codes nor AC_Hemi
    with pytest.raises(capi.SvjgError, match="INFO tag bit"):
        _format_tags(v, 0, v.n, names, gt, fl, ad, pl, 1 << 9, *(a[:, :4] if a.ndim == 2 else a for a in stats))


def test_haploid_and_no_call_cell_text():
    text = "chrX\t100\tr\tN\t<DEL>\t.\tPASS\tSVTYPE=DEL;END=900\n"
    v = genotype.NativeVcf.from_input(text.encode())
    gt = np.array([4, 5, 6, 7, 4, 6, 7], np.uint8)
    G, H0 = capi.GT_GENOTYPED, capi.GT_HALVED_0
    fl = np.array([G | H0, G, G, G | H0, 0, 0, 0], np.uint8)
    ad = np.array([[7, 4], [0, 12], [2, 2], [9, 6], [0, 0], [0, 0], [0, 0]], np.uint32)
    pl = np.array([[-3, 99, -40], [-90, 5, 7], [1, 2, 3], [0, 0, 0], [0, 0, 0], [0, 0, 0], [0, 0, 0]], np.int64)
    stats = _stats6(gt, fl, 7)
    n_gt = np.zeros(7, np.uint64)
    got = _format_ploidy(v, 0, 1, list("abcdefg"), gt, fl, ad, pl, 0, *stats, n_gt=n_gt)
    assert got.endswith("\tGT:DP:AD:PL\t0:5.5:3.5,2:-3,-40\t1:6:0,6:-90,7\t.:2:1,1:1,3\t.:7.5:4.5,3:.\t.:0:0,0:.,."
                        "\t.:0:0,0:.,.\t.:0:0,0:.\n")
    assert n_gt.tolist() == [1, 1, 1, 0, 0, 0, 0]


@pytest.mark.parametrize("tag", GOLDEN_TAGS)
def test_golden_catalogues_blocks(tag):
    text = _golden_vcf(tag) + '##INFO=<ID=AC_Hemi,Number=A,Type=Integer,Description="x">\n'
    v = genotype.NativeVcf.from_input(text.encode())
    S, names = 5, [f"s{k}" for k in range(5)]
    rng = np.random.default_rng(31)
    gt, fl, ad, pl = _ploidy_cells(rng, v.n * S)
    stats = _stats6(gt, fl, S)
    lines = _lines(text)
    base = _python_ploidy_text(lines, names, gt, fl, ad, pl)
    for tags in ((), TAGS, ("AF", "AC_Hemi"), ("NS", "AN", "F_MISSING", "HWE")):
        mask = cohort.info_tags_mask(tags)
        whole = _format_ploidy(v, 0, v.n, names, gt, fl, ad, pl, mask, *stats)
        assert whole == add_ploidy_tags(base, lines, tags)
        assert ('Description="x"' in whole) == ("AC_Hemi" not in tags)
        for step in (1, 7):
            n_gt = np.zeros(S, np.uint64)
            pieces = [_format_ploidy(v, lo, min(v.n, lo + step), names, *(a[lo * S:(lo + step) * S] for a in (gt, fl, ad, pl)),
                                     mask, *(a[lo:lo + step] for a in stats), n_gt=n_gt) for lo in range(0, v.n, step)]
            assert "".join(pieces) == whole
            assert n_gt.tolist() == _genotyped(gt, fl, S)


def test_fuzz_catalogues():
    rng = np.random.default_rng(37)
    n_checked = 0
    for k, text in enumerate(_fuzz_vcfs()[::3]):
        try:
            v = genotype.NativeVcf.from_input(text.encode())
        except genotype.VcfError:
            continue
        if v is None:
            continue
        S, names = 3, ["a", "b", "c"]
        gt, fl, ad, pl = _ploidy_cells(rng, v.n * S)
        stats = _stats6(gt, fl, S)
        tags = TAGS if k % 2 else [t for t in TAGS if rng.random() < 0.5]
        base = _python_ploidy_text(_lines(text), names, gt, fl, ad, pl)
        assert _format_ploidy(v, 0, v.n, names, gt, fl, ad, pl, cohort.info_tags_mask(tags), *stats) == \
            add_ploidy_tags(base, _lines(text), tags)
        n_checked += 1
    assert n_checked > 150


@pytest.mark.parametrize("tag", GOLDEN_TAGS)
def test_diploid_codes_give_the_existing_bytes_but_the_pl_line(tag):
    text = _golden_vcf(tag)
    v = genotype.NativeVcf.from_input(text.encode())
    S, names = 4, ["w", "x", "y", "z"]
    rng = np.random.default_rng(41)
    gt, fl, ad, pl = _random_cells(rng, v.n * S)
    stats = _stats6(gt, fl, S)
    assert (stats[0][:, 3:5] == 0).all()
    old_stats = (np.ascontiguousarray(stats[0][:, [0, 1, 2, 5]]),) + stats[1:]
    for tags in ((), cohort.INFO_TAGS, ("AF", "ExcHet")):
        mask = cohort.info_tags_mask(tags)
        old = _format_tags(v, 0, v.n, names, gt, fl, ad, pl, mask, *old_stats)
        new = _format_ploidy(v, 0, v.n, names, gt, fl, ad, pl, mask, *stats)
        assert PL3 in old and new == old.replace(PL3, PLG)
        if tags:
            assert old == add_info_tags(_python_ploidy_text(_lines(text), names, gt, fl, ad, pl).replace(PLG, PL3),
                                        _lines(text), tags)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the command line
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("extra,message", [
    (["--ploidy-file", "P"], "given together"),
    (["--sample-sex", "X"], "given together"),
    (["--info-tags", "AC_Hemi"], "--info-tags: AC_Hemi counts haploid calls"),
    (["--info-tags", "NS,AC_Hemi"], "needs --ploidy-file"),
    (["--ploidy-file", "P", "--sample-sex", "X", "--info-tags", "AC_hemi"], "unknown INFO tag 'AC_hemi'"),
    (["--ploidy-file", "missing.txt", "--sample-sex", "X"], "missing.txt"),
    (["--ploidy-file", "P:chrX 1 10 M 1\nchrX 10 20 M 1\n", "--sample-sex", "X"], "overlap"),
    (["--ploidy-file", "P:chrX 20 10 M 1\n", "--sample-sex", "X"], "FROM 20 > TO 10"),
    (["--ploidy-file", "P:chrX 1 10 M 3\n", "--sample-sex", "X"], "0, 1 or 2"),
    (["--ploidy-file", "P", "--sample-sex", "X:one M\n"], "no sex for sample 'two'"),
    (["--ploidy-file", "P", "--sample-sex", "X:one M\ntwo F\none M\n"], "listed twice"),
])
def test_command_line_refuses_before_the_device(tmp_path, extra, message):
    files = tmp_path / "in"
    files.mkdir()
    args = []
    for a in extra:
        if a[:1] in ("P", "X") and a[1:2] in ("", ":"):         # a file to write: "P" / "X" or "P:<its text>"
            body = a[2:] if len(a) > 1 else ("chrX 1 10 M 1\n" if a == "P" else "one M\ntwo F\n")
            path = files / ("p.txt" if a[0] == "P" else "x.txt")
            path.write_text(body)
            a = str(path)
        args.append(a)
    out = tmp_path / "out"
    out.mkdir()
    r = _cohort("-p", str(out / "x"), "-g", "x.gfa", "-v", "x.vcf", "-a", "one.gaf", "two.gaf", "-o", str(out / "o.vcf"),
                *args, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    # no CUDA device: a check that came after the device start would fail with another message
    assert r.returncode == 1 and message in r.stderr, r.stderr
    assert not os.listdir(out)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
def _set_ploidy(co, table, sex):
    table, sex = np.ascontiguousarray(table, np.uint8), np.ascontiguousarray(sex, np.uint8)
    capi.check(capi.lib.svjg_cohort_set_ploidy(co._h, table.shape[0], table.shape[1], table.ctypes.data, sex.ctypes.data))


@pytest.mark.gpu
@pytest.mark.parametrize("ms,e", [(0, 5e-5), (3, 5e-5), (0, 0.2), (3, 0.2)])
def test_ploidy_kernel_against_the_statement(ms, e):
    from svjg import alnfilter
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    S, n = 37, 3000
    rng = np.random.default_rng(ms * 1000 + int(e * 100) + 7)
    co = cohort.Cohort(t, S)
    counts = []
    for s in range(S):
        c = rng.integers(0, 601, (t.num_sv, 2)).astype(np.uint32)
        c[rng.random(t.num_sv) < 0.2] = 0
        c[rng.random((t.num_sv, 2)) < 0.2] = 0
        c[rng.random((t.num_sv, 2)) < 0.5] %= 40
        tie = rng.random(t.num_sv) < 0.1
        c[tie, 1] = c[tie, 0]                                               # L0 == L2 where the SV does not halve
        co.load_counts(s, c)
        counts.append(c)
    idx = rng.integers(0, t.num_sv, n).astype(np.uint32)
    idx[rng.random(n) < 0.05] = capi.NO_SV
    ty = rng.choice([0, 1, 2, 3, 255, 0x80, 0x81, 0x82, 0x83], size=n).astype(np.uint8)
    n_sexes, n_classes = 3, 11
    table = rng.integers(0, 3, (n_classes, n_sexes)).astype(np.uint8)
    table[0] = 2
    table[1] = 1
    table[2] = 0
    sex = rng.integers(0, n_sexes, S).astype(np.uint8)
    rclass = rng.integers(0, n_classes, n).astype(np.uint8)
    _set_ploidy(co, table, sex)
    blk = cohort._Block(n * S)
    gt, fl, ad, pl = (a.copy() for a in cohort._genotype_block(co, idx, ty, ms, e, blk, rclass))
    assert (fl & capi.GT_NEED_K).sum() == 0
    ploidy = table[rclass][:, sex].reshape(-1)                                   # [n * S], record-major
    n_hap = n_hap_k = 0
    for s in range(S):
        w_gt, w_fl, w_ad, w_pl = genotype.genotype_host(counts[s], idx, ty, ms, e)
        p = ploidy[s::S]
        assert (fl[s::S] == w_fl).all() and (ad[s::S] == w_ad).all()
        dip = p == 2
        assert (gt[s::S][dip] == w_gt[dip]).all() and (pl[s::S][dip] == w_pl[dip]).all()
        hap = p == 1
        assert (pl[s::S][hap][:, [0, 2]] == w_pl[hap][:, [0, 2]]).all()
        zero = p == 0
        assert (gt[s::S][zero] == capi.GT_NO_CALL).all()
        assert ((gt[s::S][hap & ((w_fl & capi.GT_GENOTYPED) == 0)]) == capi.GT_HAP_MISSING).all()
        for i in np.nonzero(hap & ((w_fl & capi.GT_GENOTYPED) != 0))[0]:
            n0, n1 = (int(x) for x in counts[s][idx[i]])
            want, pl0, pl2 = haploid_call(n0, n1, SVTYPE_NAME[int(ty[i]) & 0x3F], ms, e)
            assert "01."[gt[i * S + s] - capi.GT_HAP_REF] == want, (i, s, n0, n1)
            assert [str(pl[i * S + s, 0]), str(pl[i * S + s, 2])] == [pl0, pl2]
            n_hap += 1
            n_hap_k += (int(ad[i * S + s, 0]) + 1) // 2 + (int(ad[i * S + s, 1]) + 1) // 2 > 256
    codes = np.bincount(gt, minlength=8)
    assert n_hap > 5000 and n_hap_k > 500 and (codes[4:8] > 100).all(), codes


def _stats_case(t, S, n, seed):
    rng = np.random.default_rng(seed)
    co = cohort.Cohort(t, S)
    counts = np.array([[20, 0], [10, 10], [0, 20], [0, 0], [3, 3]], np.uint32)        # 0/0, 0/1, 1/1, gated, tie
    pick = rng.integers(0, 5, (n, S))
    pick[-3:] = [[1], [4], [3]]
    for s in range(S):
        c = np.zeros((t.num_sv, 2), np.uint32)
        c[:n] = counts[pick[:, s]]
        co.load_counts(s, c)
    table = np.array([[2, 2], [1, 2], [0, 1], [1, 1], [0, 0]], np.uint8)
    rclass = rng.integers(0, 5, n).astype(np.uint8)
    rclass[-2:] = [3, 4]
    sex = (np.arange(S) % 2).astype(np.uint8)
    _set_ploidy(co, table, sex)
    return co, np.arange(n, dtype=np.uint32), np.full(n, 2, np.uint8), rclass


@pytest.mark.gpu
@pytest.mark.parametrize("S,n", [(40, 500), (3000, 300), (1, 500)])
def test_stats_kernel_bit_for_bit(S, n):
    from svjg import alnfilter
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    co, idx, ty, rclass = _stats_case(t, S, n, seed=S + 1)
    blk = cohort._Block(n * S, n, ploidy=True)
    gt, fl, _ad, _pl = cohort._genotype_block(co, idx, ty, 3, genotype.ERR, blk, rclass)
    gcount, hwe, exc = (a.copy() for a in cohort._site_stats(co, n, blk, ploidy=True))
    w = _stats6(gt, fl, S)
    assert (gcount == w[0]).all()
    assert (hwe.view(np.uint64) == w[1].view(np.uint64)).all() and (exc.view(np.uint64) == w[2].view(np.uint64)).all()
    assert (gcount[:, 3:5].sum(1) > 0).any() and (gcount[:, :3].sum(1) > 0).any()
    assert gcount[-2].tolist()[:5] == [0, 0, 0, 0, 0] and gcount[-1].tolist() == [0, 0, 0, 0, 0, S]  # ties, ploidy 0
    with pytest.raises(capi.SvjgError, match="record count"):
        capi.check(capi.lib.svjg_cohort_site_stats_ploidy(co._h, n + 1, gcount.ctypes.data, hwe.ctypes.data,
                                                          exc.ctypes.data))


# chrX: the window starts and ends on records (220705, 1736132) and leaves the first two chrX records outside
S2_PLOIDY = "# test rules\nchrX 220705 1736132 M 1\nchrY 1 60000000 M 1\nchrY 1 60000000 F 0\n"
S2_RULES = [("chrX", 220705, 1736132, "M", 1), ("chrY", 1, 60000000, "M", 1), ("chrY", 1, 60000000, "F", 0)]


def oracle_ploidy_vcf(counts, names, vcf_lines, sexes, rules, defaults, min_support=3, e=0.00005):
    """The cohort composition of the oracle with the ploidy of each cell applied: haploid cells called by
    haploid_call from the same counters, ploidy-0 cells without a call; PL Number=G."""
    text, _n = oracle_cohort_vcf(counts, names, vcf_lines, min_support, e)
    out, ins_seen, n_gt = [], {}, [0] * len(names)
    for line in _lines(text):
        if line.startswith("#"):
            out.append(PLG if line == PL3 else line)
            continue
        cols = line.rstrip("\n").split("\t")
        svtype, key, _len = O.vcf_sv_key(cols[0], cols[1], cols[4], cols[7], ins_seen)
        for s, x in enumerate(sexes):
            cell = cols[9 + s]
            p = ploidy_of(rules, defaults, cols[0], int(cols[1]), x)
            gated = not cell.endswith(":.,.,.")
            n_gt[s] += gated and p != 0
            if p == 2:
                continue
            if not gated:
                cols[9 + s] = ".:0:0,0:." if p == 0 else ".:0:0,0:.,."
            elif p == 0:
                cols[9 + s] = ".:" + ":".join(cell.split(":")[1:3]) + ":."
            else:
                g, pl0, pl2 = haploid_call(*counts[s][key], svtype, min_support, e)
                cols[9 + s] = f"{g}:" + ":".join(cell.split(":")[1:3]) + f":{pl0},{pl2}"
        out.append("\t".join(cols) + "\n")
    return "".join(out), n_gt


@pytest.mark.gpu
def test_s2_cohort_with_ploidy(tmp_path):
    from svjg import alnfilter, cli
    p, samples, counts = _s2_cohort(tmp_path)
    names = [f"n{k}" for k in range(7)]
    sexes = ["F", "M"] * 3 + ["F"]
    open(p + "_ploidy.txt", "w").write(S2_PLOIDY)
    open(p + "_sex.txt", "w").write("".join(f"{nm}\t{x}\n" for nm, x in zip(names, sexes)) + "other F\n")
    vcf = _golden_vcf("s2")
    base, want_n = oracle_ploidy_vcf(counts, names, vcf.splitlines(True), sexes, S2_RULES, {})
    want = add_ploidy_tags(base, _lines(vcf), TAGS)
    body = [ln.split("\t") for ln in base.splitlines() if not ln.startswith("#")]
    hap = [c for ln in body for c in ln[9:] if c[:2] in ("0:", "1:")]
    assert len(hap) > 10 and any(c.startswith("1:") for c in hap)
    assert any(c.startswith(".:") and not c.endswith(",.") and c.count(":") == 3 and c != ".:0:0,0:." for ln in body
               for c in ln[9:])                                                   # ploidy 0 with reads
    assert any(ln[0] == "chrX" and "/" in ln[10].split(":")[0] for ln in body)     # chrX outside the window: diploid
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *[",".join(fs) for fs in samples], "-o", p + "_p.vcf",
                "--names", ",".join(names), "--info-tags", "all", "--ploidy-file", p + "_ploidy.txt",
                "--sample-sex", p + "_sex.txt")
    assert r.returncode == 0, r.stderr
    assert open(p + "_p.vcf").read() == want
    assert r.stdout == "".join(f"Genotyped svs in {nm}: {n}\n" for nm, n in zip(names, want_n))
    # the module, blocks forced small
    t = alnfilter.Tables.from_memory(read_golden("s2_svs_edges.json.gz"), read_golden("s2.gfa.gz")).to_device(0)
    co = cohort.Cohort(t, 7)
    for k, fs in enumerate(samples):
        for b in cli._read_sample(fs):
            co.filter(k, b.array)
    pr = cohort.PloidyRules(S2_PLOIDY, open(p + "_sex.txt").read(), names)
    for block in (None, 1, 7):
        assert cohort.genotype_cohort_vcf(t, co, vcf.encode(), names, block_records=block, info_tags=TAGS,
                                          ploidy=pr) == (want, want_n)


@pytest.mark.gpu
def test_haploid_cells_beyond_the_lut(tmp_path):
    """s2's largest counts are halved DEL / INS alleles: 48 copies stay within the 256-entry log10 C(n, k) table, 72
    copies of chrX:1736132 (INS, 1 and 6 hits) do not.  That record is haploid in the M sample."""
    from svjg import alnfilter
    p = _s2_cohort(tmp_path)[0]
    gaf = read_golden("s2.gaf.gz")
    open(p + "_x72.gaf", "w").write(gaf * 72)
    one = _python_oracle_counts("s2", gaf)
    counts = [{k: (72 * a, 72 * b) for k, (a, b) in one.items()}, one]
    names, sexes = ["x72", "one"], ["M", "F"]
    open(p + "_ploidy.txt", "w").write(S2_PLOIDY)
    open(p + "_sex.txt", "w").write("x72 M\none F\n")
    vcf = _golden_vcf("s2")
    base, want_n = oracle_ploidy_vcf(counts, names, vcf.splitlines(True), sexes, S2_RULES, {})
    r = _cohort("-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", p + "_x72.gaf", p + "_whole.gaf", "-o", p + "_k.vcf",
                "--names", ",".join(names), "--info-tags", "all", "--ploidy-file", p + "_ploidy.txt",
                "--sample-sex", p + "_sex.txt")
    assert r.returncode == 0, r.stderr
    assert open(p + "_k.vcf").read() == add_ploidy_tags(base, _lines(vcf), TAGS)
    # the device flags that cell NEED_K and keeps its haploid code
    t = alnfilter.Tables.from_memory(read_golden("s2_svs_edges.json.gz"), read_golden("s2.gfa.gz")).to_device(0)
    co = cohort.Cohort(t, 2)
    co.filter(0, open(p + "_x72.gaf", "rb").read())
    co.filter(1, gaf.encode())
    pr = cohort.PloidyRules(S2_PLOIDY, "x72 M\none F\n", names)
    v = genotype.NativeVcf.from_input(vcf.encode())
    rclass, table = pr.record_classes(v)
    _set_ploidy(co, table, pr.sex_index)
    n = v.n
    blk = cohort._Block(n * 2)
    idx, ty = np.ascontiguousarray(v.index_tables(t)), np.ascontiguousarray(v.svtype)
    la, lb, lh = math.log10(1 - genotype.ERR), math.log10(genotype.ERR), math.log10(0.5)
    lut = genotype.log10comb_lut()
    capi.check(capi.lib.svjg_cohort_genotype_ploidy(co._h, idx.ctypes.data, ty.ctypes.data, rclass.ctypes.data, n, 3, la,
                                                    lb, lh, lut.ctypes.data, genotype.LUT_NMAX, blk.pl.ctypes.data,
                                                    blk.gt.ctypes.data, blk.ad2.ctypes.data, blk.flags.ctypes.data))
    need = (blk.flags[:2 * n] & capi.GT_NEED_K) != 0
    hap = (blk.gt[:2 * n] >= capi.GT_HAP_REF) & (blk.gt[:2 * n] <= capi.GT_HAP_MISSING)
    assert (need & hap).sum() >= 1 and (need & ~hap).sum() >= 1


@pytest.mark.gpu
def test_diploid_everywhere_is_todays_output_but_the_pl_line(tmp_path):
    p, samples, counts = _s2_cohort(tmp_path)
    names = [f"n{k}" for k in range(7)]
    open(p + "_ploidy.txt", "w").write("chrX 1 100000000 M 2\nchrY 1 100000000 F 2\n* * * M 2\n")
    open(p + "_sex.txt", "w").write("".join(f"{nm} {'MF'[k % 2]}\n" for k, nm in enumerate(names)))
    vcf = _golden_vcf("s2")
    base, want_n = oracle_cohort_vcf(counts, names, vcf.splitlines(True))
    want = add_info_tags(base, _lines(vcf), cohort.INFO_TAGS)
    args = ["-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *[",".join(fs) for fs in samples], "--names", ",".join(names),
            "--info-tags", ",".join(cohort.INFO_TAGS)]
    r = _cohort(*args, "-o", p + "_2.vcf", "--ploidy-file", p + "_ploidy.txt", "--sample-sex", p + "_sex.txt")
    assert r.returncode == 0, r.stderr
    got = open(p + "_2.vcf").read()
    assert PLG in got and got == want.replace(PL3, PLG)
    assert r.stdout == "".join(f"Genotyped svs in {nm}: {n}\n" for nm, n in zip(names, want_n))
