"""Genotype posteriors of the cohort VCF (genotype-cohort.py --posteriors; svjg_cohort_posteriors on the device,
svjg_vcf_format_cohort_post on the host).
The Python statement is here (`posteriors`, `add_posteriors`):
  * a cell contributes when it is SVJG_GT_GENOTYPED and its code is not SVJG_GT_NO_CALL; codes 0-3 are diploid, 4-6
    haploid.  Cells below -ms and ties contribute;
  * weights w_g = T[PL_g - m], T[k] = 10.0 ** (-k / 10) (cohort.phred_weights), 0.0 beyond the table; m is the smallest
    PL of the cell (a haploid cell: of PL0 and PL2, and it has w0 and w2 only);
  * EM per record, A = the sum of the contributing cells' ploidies, from f = 0.5: q = 1 - f, P0 = q*q, P1 = (f*q)*2,
    P2 = f*f; diploid a = w0*P0, b = w1*P1, c = w2*P2, den = (a+b)+c, e = (b + c*2)/den; haploid a = w0*q, c = w2*f,
    den = a+c, e = c/den.  E = the sum of e in warp order: lane l sums the cells s = l (mod 32) in increasing s from
    0.0, then x = x + x[l ^ o] for o = 16, 8, 4, 2, 1.  f_new = E / A; stop when |f_new - f| <= 1e-10 or after 100
    steps; f^ = f_new.  Every step is one IEEE double operation (numpy's float64 here);
  * GP = a/den, b/den, c/den at f^ (haploid a/den, c/den); GQ = max{q <= 99 : err <= T[q]}, err = the sum in index
    order of the other genotypes' terms over den, "." for a missing call (codes 3 and 6);
  * text: FORMAT GT:DP:AD:PL:GP:GQ, "%.6g" values, ":.:." after a non-contributing cell and in every cell of a record
    whose ALT holds a comma; INFO AF_EM=f^ after the tags ("." with A = 0 or a comma in ALT); the ##INFO line of AF_EM
    after those of the tags, the ##FORMAT lines of GP and GQ after PL's; a catalogue's AF_EM items and lines dropped.
CPU part: the statement against independent mathematics, the formatter against the text, the command line.  GPU part
(-m gpu): the kernel bit for bit against the statement, and the command line on the s2 cohort."""
import ctypes as C
import os
from fractions import Fraction

import numpy as np
import pytest

from conftest import read_golden
from svjg import capi, cohort, genotype
from test_cohort import GOLDEN_TAGS, _cohort, _golden_vcf, _python_oracle_counts, _random_cells, _synthetic
from test_cohort_info import _CATALOGUE, _format_tags, _g6, _lines, _s2_cohort
from test_cohort_ploidy import S2_PLOIDY, _format_ploidy, _set_ploidy, _stats6

T = cohort.phred_weights()
GQ_NONE = capi.POST_GQ_NONE
AF_EM_LINE = ('##INFO=<ID=AF_EM,Number=A,Type=Float,Description="ALT allele frequency estimated by EM over the samples\' '
              'genotype likelihoods">\n')
GP_GQ_LINES = ('##FORMAT=<ID=GP,Number=G,Type=Float,Description="Genotype posterior probabilities under a Hardy-Weinberg '
               'prior at the allele frequency AF_EM">\n'
               '##FORMAT=<ID=GQ,Number=1,Type=Integer,Description="Phred-scaled posterior probability that the genotype '
               'call is wrong (floored, at most 99)">\n')


# ---------------------------------------------------------------------------------------------------------------
# the Python statement
# ---------------------------------------------------------------------------------------------------------------
def cell_kinds(gt, fl):
    """0: the cell does not contribute, else its ploidy (1 or 2)."""
    gt, fl = np.asarray(gt), np.asarray(fl)
    contrib = ((fl & capi.GT_GENOTYPED) != 0) & (gt != capi.GT_NO_CALL)
    return np.where(contrib, np.where(gt >= capi.GT_HAP_REF, 1, 2), 0).astype(np.int64)


def cell_weights(pl, kind):
    """w [cells][3]: T[PL_g - m], 0.0 beyond the table; haploid cells use PL0 and PL2 (w1 = 0); others 0."""
    pl = np.asarray(pl, np.int64)
    hap = kind == 1
    m = np.where(hap, np.minimum(pl[:, 0], pl[:, 2]), pl.min(1))
    d = pl - m[:, None]
    w = np.where(d > capi.POST_PLW_N - 1, 0.0, T[np.clip(d, 0, capi.POST_PLW_N - 1)])
    w[hap, 1] = 0.0
    w[kind == 0] = 0.0
    return w


def _terms(kind, w, f):
    """a, b, c, den of every cell at the frequency f of its record ([n][S] arrays)."""
    f = f[:, None]
    q = 1.0 - f
    p0, p1, p2 = q * q, (f * q) * 2.0, f * f
    dip = kind == 2
    a = np.where(dip, w[..., 0] * p0, w[..., 0] * q)
    b = np.where(dip, w[..., 1] * p1, 0.0)
    c = np.where(dip, w[..., 2] * p2, w[..., 2] * f)
    den = np.where(dip, (a + b) + c, a + c)
    return a, b, c, den


def em(kind, w):
    """(f^ [n], iters [n]) of records with cells kind [n][S], w [n][S][3]; f^ NaN and 0 steps when A = 0."""
    n, S = kind.shape
    A = kind.sum(1).astype(np.float64)
    f = np.where(A > 0, 0.5, np.nan)
    it = np.zeros(n, np.int64)
    active = A > 0
    lane = np.arange(32)
    with np.errstate(divide="ignore", invalid="ignore"):
        while active.any():
            r = np.nonzero(active)[0]
            a, b, c, den = _terms(kind[r], w[r], f[r])
            e = np.where(kind[r] == 2, (b + c * 2.0) / den, c / den)
            e = np.where(kind[r] == 0, 0.0, e)
            x = np.zeros((r.size, 32))
            for j in range(0, S, 32):
                cols = e[:, j:j + 32]
                x[:, :cols.shape[1]] = x[:, :cols.shape[1]] + cols
            for o in (16, 8, 4, 2, 1):
                x = x + x[:, lane ^ o]
            f_new = x[:, 0] / A[r]
            it[r] += 1
            done = (np.abs(f_new - f[r]) <= capi.POST_TOL) | (it[r] == capi.POST_MAX_ITERS)
            f[r] = f_new
            active[r[done]] = False
    return f, it


def posteriors(gt, fl, pl, S):
    """The statement on the cells of n records ([n * S] record-major): (af [n], gp [n * S][3], gq [n * S] u8,
    iters [n], err [n * S] (NaN where there is no GQ))."""
    gt = np.asarray(gt, np.int64)
    kind = cell_kinds(gt, fl)
    w = cell_weights(pl, kind)
    n = kind.size // S
    f, it = em(kind.reshape(n, S), w.reshape(n, S, 3))
    a, b, c, den = _terms(kind.reshape(n, S), w.reshape(n, S, 3), np.where(np.isnan(f), 0.5, f))
    a, b, c, den = (x.reshape(-1) for x in (a, b, c, den))
    out = kind == 0
    with np.errstate(divide="ignore", invalid="ignore"):
        gp = np.stack([a / den, np.where(kind == 2, b / den, 0.0), c / den], axis=1)
        gp[out] = 0.0
        other = np.select([gt == 0, gt == 1, gt == 2, gt == capi.GT_HAP_REF, gt == capi.GT_HAP_ALT],
                          [b + c, a + c, a + b, c, a], np.nan)
        err = np.where(out, np.nan, other / den)
    gq = np.where(np.isnan(err), GQ_NONE, (err[:, None] <= T[None, :capi.POST_GQ_MAX + 1]).sum(1) - 1).astype(np.uint8)
    return f, gp, gq, it.astype(np.uint8), err


def _cell_post_text(kind, gp, gq, multi_alt):
    if kind == 0 or multi_alt:
        return ":.:."
    vals = [gp[0], gp[1], gp[2]] if kind == 2 else [gp[0], gp[2]]
    return ":" + ",".join(_g6(x) for x in vals) + ":" + ("." if gq == GQ_NONE else str(int(gq)))


def add_posteriors(text, gt, fl, af, gp, gq, S):
    """The cohort VCF ``text`` (written without posteriors) with them: the statement's text rules."""
    kind = cell_kinds(gt, fl)
    out, j = [], 0
    for line in _lines(text):
        if line.startswith("##INFO=<ID=AF_EM,") or line.startswith("##INFO=<ID=AF_EM>"):
            continue
        if line.startswith("##FORMAT=<ID=GT,"):
            out.append(AF_EM_LINE)
        if line.startswith("#"):
            out.append(line)
            if line.startswith("##FORMAT=<ID=PL,"):
                out.append(GP_GQ_LINES)
            continue
        cols = line.rstrip("\n").split("\t")
        multi_alt = "," in cols[4]
        items = [] if cols[7] in (".", "") else cols[7].split(";")
        kept = [it for it in items if it.split("=", 1)[0] != "AF_EM"]
        val = "." if multi_alt or np.isnan(af[j]) else _g6(af[j])
        cols[7] = ";".join(kept + [f"AF_EM={val}"])
        cols[8] += ":GP:GQ"
        for s in range(S):
            k = j * S + s
            cols[9 + s] += _cell_post_text(kind[k], gp[k], gq[k], multi_alt)
        out.append("\t".join(cols) + "\n")
        j += 1
    return "".join(out)


# ---------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------
def _format_post(v, lo, hi, names, gt, fl, ad, pl, ploidy, mask, stats, af, gp, gq, n_gt=None):
    joined = "\t".join(names).encode()
    arrs = [np.ascontiguousarray(a) for a in (gt, fl, ad, pl)]
    site = [None if a is None else np.ascontiguousarray(a) for a in stats]
    post = [None if a is None else np.ascontiguousarray(a) for a in (af, gp, gq)]
    n_gt = np.zeros(len(names), np.uint64) if n_gt is None else n_gt
    buf, n_out = C.c_void_p(), C.c_uint64()
    ptr = [None if a is None else a.ctypes.data for a in site + post]
    capi.check(capi.lib.svjg_vcf_format_cohort_post(v._h, lo, hi, len(names), joined, len(joined),
                                                    *(a.ctypes.data for a in arrs), int(ploidy), mask, *ptr,
                                                    C.byref(buf), C.byref(n_out), n_gt.ctypes.data))
    try:
        return C.string_at(buf.value, n_out.value).decode("ascii")
    finally:
        capi.lib.svjg_buffer_free(buf)


def _cells(rng, n_cells, ploidy):
    """Cells of every kind with PLs a genotype call can have (0 to 20 000, some equal triples)."""
    gt, fl, ad, pl = _random_cells(rng, n_cells)
    if ploidy:
        gt[:] = rng.integers(0, 8, n_cells)
    fl[rng.random(n_cells) < 0.05] |= capi.GT_NEED_K                     # patched cells: the text does not look
    pl[:] = rng.integers(0, 20000, (n_cells, 3))
    pl[rng.random(n_cells) < 0.3] %= 40
    pl[rng.random(n_cells) < 0.05] = 7
    return gt, fl, ad, pl


def _stats(gt, fl, S, ploidy):
    st = _stats6(gt, fl, S)
    return st if ploidy else (np.ascontiguousarray(st[0][:, [0, 1, 2, 5]]),) + st[1:]


def _base(v, lo, hi, names, cells, ploidy, mask, stats):
    fmt = _format_ploidy if ploidy else _format_tags
    return fmt(v, lo, hi, names, *cells, mask, *stats)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the statement against independent mathematics
# ---------------------------------------------------------------------------------------------------------------
def _random_cohort(rng, S):
    n_cells = S
    gt = rng.integers(0, 8, n_cells).astype(np.uint8)
    fl = np.where(rng.random(n_cells) < 0.9, capi.GT_GENOTYPED, 0).astype(np.uint8)
    style = rng.integers(0, 4)
    if style == 0:
        pl = rng.integers(0, 60, (n_cells, 3))
    elif style == 1:
        pl = rng.integers(0, 5000, (n_cells, 3))
    elif style == 2:                                  # low depth: a few phred units between the genotypes
        pl = rng.integers(0, 12, (n_cells, 3))
    else:
        pl = np.where(rng.random((n_cells, 3)) < 0.5, rng.integers(0, 30, (n_cells, 3)), rng.integers(0, 400, (n_cells, 3)))
    return gt, fl, pl.astype(np.int64)


def _neg_loglik(kind, w, f):
    q = 1.0 - f
    dip = kind == 2
    lik = np.where(dip, w[:, 0] * q * q + w[:, 1] * 2 * f * q + w[:, 2] * f * f, w[:, 0] * q + w[:, 2] * f)
    return -np.log(lik[kind > 0]).sum()


def test_statement_against_the_likelihood_maximiser_gp_sums_and_exact_gq():
    from scipy.optimize import minimize_scalar
    rng = np.random.default_rng(61)
    n_conv = n_gq = 0
    for trial in range(300):
        S = int(rng.integers(1, 201))
        gt, fl, pl = _random_cohort(rng, S)
        af, gp, gq, it, err = posteriors(gt, fl, pl, S)
        kind = cell_kinds(gt, fl)
        w = cell_weights(pl, kind)
        if kind.sum() == 0:
            assert np.isnan(af[0]) and it[0] == 0 and (gq == GQ_NONE).all() and (gp == 0).all()
            continue
        assert 0.0 <= af[0] <= 1.0 and 1 <= it[0] <= capi.POST_MAX_ITERS
        if it[0] < capi.POST_MAX_ITERS:
            opt = minimize_scalar(lambda f: _neg_loglik(kind, w, f), bounds=(0.0, 1.0), method="bounded",
                                  options={"xatol": 1e-12})
            # f^ is the maximiser, or (a flat likelihood) at least as likely as the one found
            assert abs(af[0] - opt.x) <= 1e-6 or _neg_loglik(kind, w, af[0]) <= opt.fun, (trial, af[0], opt.x)
            n_conv += 1
        rows = gp[kind > 0]
        sums = rows.sum(1)
        assert (np.abs(sums - 1.0) <= 4 * np.spacing(1.0)).all()
        for k in np.nonzero(~np.isnan(err))[0]:
            e = float(err[k])
            if any(abs(e - T[q]) <= 1e-12 for q in range(capi.POST_GQ_MAX + 1)):
                continue
            fe = Fraction(e)
            want = capi.POST_GQ_MAX
            if fe > 0:                     # the largest q with err <= 10^(-q/10), i.e. err^10 * 10^q <= 1
                want = 0
                while want < capi.POST_GQ_MAX and fe ** 10 * 10 ** (want + 1) <= 1:
                    want += 1
            assert gq[k] == want, (k, e, gq[k], want)
            n_gq += 1
        assert (gq[(kind > 0) & np.isin(gt, [3, capi.GT_HAP_MISSING])] == GQ_NONE).all()
    assert n_conv > 150 and n_gq > 3000


def test_warp_order_is_the_lane_order_then_the_butterfly():
    """The statement's sum differs from a plain left-to-right sum in the last bits for some cohorts: the order is
    part of the contract."""
    rng = np.random.default_rng(5)
    differ = 0
    for _ in range(200):
        S = 100
        gt, fl, pl = _random_cohort(rng, S)
        kind = cell_kinds(gt, fl)
        w = cell_weights(pl, kind)
        if not kind.sum():
            continue
        f = np.array([0.37])
        a, b, c, den = _terms(kind[None], w[None], f)
        with np.errstate(divide="ignore", invalid="ignore"):
            e = np.where(kind == 2, (b + c * 2.0) / den, c / den)[0]
        e = np.where(kind == 0, 0.0, e)
        plain = 0.0
        for x in e:
            plain += x
        lanes = [0.0] * 32
        for s in range(S):
            lanes[s % 32] += e[s]
        for o in (16, 8, 4, 2, 1):
            lanes = [lanes[l] + lanes[l ^ o] for l in range(32)]
        assert len(set(lanes)) == 1
        differ += lanes[0] != plain
    assert differ > 0


def test_phred_weights():
    assert T.size == capi.POST_PLW_N and T[0] == 1.0 and T[10] == 0.1 and T[-1] == 0.0
    assert (np.diff(T) <= 0).all() and (np.diff(T[:3000]) < 0).all() and T[3000] > 0 and T[3240] == 0.0


# ---------------------------------------------------------------------------------------------------------------
# CPU: the formatter
# ---------------------------------------------------------------------------------------------------------------
AF_EM_CATALOGUE = _CATALOGUE.replace("##INFO=<ID=AFX,", '##INFO=<ID=AF_EM,Number=A,Type=Float,Description="old">\n'
                                     "##INFO=<ID=AFX,")


def _af_em_catalogue():
    lines = _lines(AF_EM_CATALOGUE)
    out, k = [], 0
    for ln in lines:
        if not ln.startswith("#"):
            cols = ln.rstrip("\n").split("\t")
            if k % 2 == 0:
                cols[7] = ("AF_EM=0.5" if cols[7] in (".", "") else "AF_EM=0.5;" + cols[7] + ";AF_EM=x")
            ln = "\t".join(cols) + "\n"
            k += 1
        out.append(ln)
    return "".join(out)


@pytest.mark.parametrize("ploidy", [False, True])
def test_every_cell_kind_tags_and_blocks(ploidy):
    text = _af_em_catalogue()
    assert "AF_EM=0.5;" in text and 'Description="old"' in text
    v = genotype.NativeVcf.from_input(text.encode())
    S, names = 9, [f"s{k}" for k in range(9)]
    rng = np.random.default_rng(71 + ploidy)
    cells = _cells(rng, v.n * S, ploidy)
    gt, fl, ad, pl = cells
    fl[4 * S:5 * S] &= ~np.uint8(capi.GT_GENOTYPED)                    # A = 0: no cell contributes
    af, gp, gq, _it, _err = posteriors(gt, fl, pl, S)
    assert np.isnan(af[4]) and not np.isnan(af).all()
    lines = _lines(text)
    assert any("," in ln.split("\t")[4] for ln in lines if not ln.startswith("#"))       # a multi-ALT record
    tag_sets = [(), cohort.INFO_TAGS, ("AF", "HWE"), ("NS",)] + ([cohort.PLOIDY_INFO_TAGS] if ploidy else [])
    stats = _stats(gt, fl, S, ploidy)
    for tags in tag_sets:
        mask = cohort.info_tags_mask(tags)
        base = _base(v, 0, v.n, names, cells, ploidy, mask, stats)
        want = add_posteriors(base, gt, fl, af, gp, gq, S)
        n_gt = np.zeros(S, np.uint64)
        whole = _format_post(v, 0, v.n, names, *cells, ploidy, mask, stats, af, gp, gq, n_gt=n_gt)
        assert whole == want, tags
        assert 'Description="old"' not in whole and "AF_EM=x" not in whole and "AF_EM=0.5;" not in whole
        for step in (1, 7):
            n_b = np.zeros(S, np.uint64)
            pieces = [_format_post(v, lo, min(v.n, lo + step), names,
                                   *(a[lo * S:(lo + step) * S] for a in cells), ploidy, mask,
                                   [a[lo:lo + step] for a in stats], af[lo:lo + step], gp[lo * S:(lo + step) * S],
                                   gq[lo * S:(lo + step) * S], n_gt=n_b) for lo in range(0, v.n, step)]
            assert "".join(pieces) == whole
            assert (n_b == n_gt).all()
    body = [ln.split("\t") for ln in whole.splitlines() if not ln.startswith("#")]
    assert all(c.endswith(":.:.") for c in body[4][9:])
    multi = [b for b in body if "," in b[4]]
    assert multi and all(c.endswith(":.:.") for b in multi for c in b[9:]) and all("AF_EM=." in b[7] for b in multi)
    kinds = cell_kinds(gt, fl)
    assert set(kinds.tolist()) == ({0, 1, 2} if ploidy else {0, 2})


def test_cell_text_of_each_code_and_the_probability_text():
    text = "chrX\t100\tr\tN\t<DEL>\t.\tPASS\tSVTYPE=DEL;END=900\n"
    v = genotype.NativeVcf.from_input(text.encode())
    G = capi.GT_GENOTYPED
    gt = np.array([0, 1, 2, 3, 4, 5, 6, 7, 0, 4, 7], np.uint8)
    fl = np.array([G, G, G, G, G, G, G, G, 0, 0, 0], np.uint8)
    S = gt.size
    ad = np.full((S, 2), 4, np.uint32)
    pl = np.array([[0, 30, 60]] * S, np.int64)
    edge = 0.9999995
    vals = [0.0, 1.0, 5e-324, 1e-300, 0.5, 1 / 3, np.nextafter(edge, 0), edge, np.nextafter(edge, 2), 0.99999951,
            np.nextafter(0.99999951, 0), 0.9999994999999, 0.12345649999, 2.5e-7, 0.999999, 0.9999996]
    gp = np.array([[vals[(3 * k + j) % len(vals)] for j in range(3)] for k in range(S)], np.float64)
    gq = np.array([0, 7, 99, GQ_NONE, 12, 0, GQ_NONE, GQ_NONE, GQ_NONE, GQ_NONE, GQ_NONE], np.uint8)
    af = np.array([0.25])
    stats = _stats(gt, fl, S, True)
    base = _base(v, 0, 1, [f"c{k}" for k in range(S)], (gt, fl, ad, pl), True, 0, stats)
    got = _format_post(v, 0, 1, [f"c{k}" for k in range(S)], gt, fl, ad, pl, 1, 0, stats, af, gp, gq)
    assert got == add_posteriors(base, gt, fl, af, gp, gq, S)
    cells = got.splitlines()[-1].split("\t")
    assert cells[7] == "SVTYPE=DEL;END=900;AF_EM=0.25" and cells[8] == "GT:DP:AD:PL:GP:GQ"
    assert cells[9] == "0/0:4:2,2:0,30,60:0,1,4.94066e-324:0"
    assert cells[12].endswith(":.") and cells[12].count(":") == 5                          # code 3: GP, GQ "."
    assert cells[13].startswith("0:") and cells[13].split(":")[3].count(",") == 1 and cells[13].split(":")[4].count(",") == 1
    assert cells[16].endswith(":.:.") and cells[17].endswith(":.:.") and cells[19].endswith(":.:.")
    for x in vals:
        row = np.array([[x, x, x]])
        one = _format_post(v, 0, 1, ["a"], gt[:1], fl[:1], ad[:1], pl[:1], 0, 0, (None,) * 3, af, row, gq[:1])
        assert one.splitlines()[-1].split("\t")[9].split(":")[4] == ",".join([_g6(x)] * 3), x


@pytest.mark.parametrize("tag", GOLDEN_TAGS)
def test_null_posteriors_give_todays_bytes_through_every_entry_point(tag):
    text = _golden_vcf(tag)
    v = genotype.NativeVcf.from_input(text.encode())
    S, names = 4, ["w", "x", "y", "z"]
    rng = np.random.default_rng(43)
    for ploidy in (False, True):
        cells = _random_cells(rng, v.n * S)
        if ploidy:
            cells[0][:] = rng.integers(0, 8, v.n * S)
        stats = _stats(cells[0], cells[1], S, ploidy)
        for tags in ((), cohort.INFO_TAGS):
            mask = cohort.info_tags_mask(tags)
            want = _base(v, 0, v.n, names, cells, ploidy, mask, stats)
            assert _format_post(v, 0, v.n, names, *cells, ploidy, mask, stats, None, None, None) == want
    # svjg_vcf_format (one sample named SAMPLE) and svjg_vcf_format_cohort are the same formatter
    gt, fl, ad, pl = _random_cells(rng, v.n)
    buf, n_out, n_gt = C.c_void_p(), C.c_uint64(), C.c_uint64()
    capi.check(capi.lib.svjg_vcf_format(v._h, gt.ctypes.data, fl.ctypes.data, ad.ctypes.data, pl.ctypes.data,
                                        C.byref(buf), C.byref(n_out), C.byref(n_gt)))
    try:
        single = C.string_at(buf.value, n_out.value).decode("ascii")
    finally:
        capi.lib.svjg_buffer_free(buf)
    stats = _stats(gt, fl, 1, False)
    assert _format_post(v, 0, v.n, ["SAMPLE"], gt, fl, ad, pl, 0, 0, stats, None, None, None) == single
    assert single == genotype.format_vcf(*genotype.parse_vcf(_lines(text)), gt, fl, ad, pl)[0]


def test_formatter_refuses_partial_posteriors_and_bad_gq():
    v = genotype.NativeVcf.from_input(_CATALOGUE.encode())
    S = 2
    rng = np.random.default_rng(3)
    cells = _cells(rng, v.n * S, False)
    af, gp, gq, _it, _err = posteriors(cells[0], cells[1], cells[3], S)
    with pytest.raises(capi.SvjgError, match="go together"):
        _format_post(v, 0, v.n, ["a", "b"], *cells, 0, 0, (None,) * 3, af, None, gq)
    bad = gq.copy()
    bad[0] = 100
    with pytest.raises(capi.SvjgError, match="GQ out of range"):
        _format_post(v, 0, v.n, ["a", "b"], *cells, 0, 0, (None,) * 3, af, gp, bad)
    with pytest.raises(capi.SvjgError, match="ploidy must be"):
        _format_post(v, 0, v.n, ["a", "b"], *cells, 2, 0, (None,) * 3, af, gp, gq)


# ---------------------------------------------------------------------------------------------------------------
# CPU: the command line
# ---------------------------------------------------------------------------------------------------------------
def test_help_names_the_switch():
    r = _cohort("--help")
    assert r.returncode == 0 and "--posteriors" in r.stdout and "GQ" in r.stdout


@pytest.mark.parametrize("extra,message", [
    (["--info-tags", "AC_Hemi"], "--info-tags: AC_Hemi counts haploid calls"),
    (["--ploidy-file", "P"], "given together"),
    (["--info-tags", "NS,AF_EM"], "unknown INFO tag 'AF_EM'"),
    (["--names", "a,a"], "unique"),
])
def test_switch_combines_and_adds_no_refusal(tmp_path, extra, message):
    files = tmp_path / "in"
    files.mkdir()
    args = []
    for a in extra:
        if a == "P":
            (files / "p.txt").write_text("chrX 1 10 M 1\n")
            a = str(files / "p.txt")
        args.append(a)
    out = tmp_path / "out"
    out.mkdir()
    r = _cohort("-p", str(out / "x"), "-g", "x.gfa", "-v", "x.vcf", "-a", "one.gaf", "two.gaf", "-o", str(out / "o.vcf"),
                "--posteriors", *args, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and message in r.stderr, r.stderr
    assert not os.listdir(out)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
_KIND_COUNTS = np.array([[12, 0], [6, 6], [0, 12], [1, 1], [0, 0]], np.uint32)    # 0/0, 0/1, 1/1, below -ms, gated


def _kernel_case(t, S, n, rng, ploidy):
    """A cohort of S samples and n records whose cells are genotyped from chosen counts (INV: no halving)."""
    co = cohort.Cohort(t, S)
    pick = rng.integers(0, 5, (n, S))
    pick[0] = 4                                                       # every cell outside the gate
    for s in range(S):
        c = np.zeros((t.num_sv, 2), np.uint32)
        c[:n] = _KIND_COUNTS[pick[:, s]]
        c[1:n:9] = [300, 280]                                         # beyond the log10 C(n, k) table: NEED_K
        co.load_counts(s, c)
    idx = np.arange(n, dtype=np.uint32)
    idx[0] = capi.NO_SV
    ty = np.full(n, 2, np.uint8)
    rclass = None
    if ploidy:
        _set_ploidy(co, np.array([[2, 2], [1, 2], [0, 1], [1, 1]], np.uint8), (np.arange(S) % 2).astype(np.uint8))
        rclass = rng.integers(0, 4, n).astype(np.uint8)
    return co, idx, ty, rclass


def _patch(rng, gt, fl, S):
    """Cells (record-major indices) and PL triples sent through the patch: a third of the genotyped cells with random
    PLs, gaps beyond the table and equal triples, and every cell of one record with a diploid contributing cell set to
    (0, 0, 30) (haploid cells (0, 0, 0): e = f), whose likelihood is flat at f = 0, so that its EM runs to the step
    cap."""
    genotyped = np.nonzero(fl & capi.GT_GENOTYPED)[0]
    cell = rng.choice(genotyped, size=max(1, genotyped.size // 3), replace=False)
    pl = rng.integers(0, 200, (cell.size, 3)).astype(np.int64)
    q = rng.random(cell.size)
    pl[q < 0.2] = rng.integers(0, 30000, (int((q < 0.2).sum()), 3))        # gaps beyond 4095
    pl[(q >= 0.2) & (q < 0.3)] = 17                                        # all equal
    kinds = cell_kinds(gt, fl)
    rows = np.unique(np.nonzero(kinds == 2)[0] // S)
    slow = rows[rows > 0][len(rows) // 2]
    row = np.arange(slow * S, slow * S + S)
    keep = ~np.isin(cell, row)
    cell = np.concatenate([cell[keep], row])
    pl = np.concatenate([pl[keep], np.where((kinds[row] == 1)[:, None], [[0, 0, 0]], [[0, 0, 30]])])
    return cell, pl


def _run_posteriors(co, n, blk, cell, pl):
    S = co.n_samples
    af, iters = np.zeros(n), np.zeros(n, np.uint8)
    gp, gq = np.zeros((n * S, 3)), np.zeros(n * S, np.uint8)
    cell, pl = np.ascontiguousarray(cell, np.uint32), np.ascontiguousarray(pl, np.int64)
    rc = capi.lib.svjg_cohort_posteriors(co._h, n, cell.size, cell.ctypes.data, pl.ctypes.data, T.ctypes.data, T.size,
                                         af.ctypes.data, gp.ctypes.data, gq.ctypes.data, iters.ctypes.data)
    return rc, af, gp, gq, iters


def _same_bits(x, y):
    return x.shape == y.shape and (np.ascontiguousarray(x).view(np.uint64) == np.ascontiguousarray(y).view(np.uint64)).all()


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 31, 32, 33, 64, 129, 3000])
def test_kernel_bit_for_bit(S):
    from svjg import alnfilter
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    n = 40 if S == 3000 else 300
    rng = np.random.default_rng(S)
    for ploidy in (False, True):
        co, idx, ty, rclass = _kernel_case(t, S, n, rng, ploidy)
        blk = cohort._Block(n * S, post_records=n)
        gt, fl, _ad, pl = (a.copy() for a in cohort._genotype_block(co, idx, ty, 3, genotype.ERR, blk, rclass))
        need = blk.need.copy()
        assert need.size > 0
        # without the host's PLs the NEED_K cells cannot be used
        rc, *_ = _run_posteriors(co, n, blk, np.zeros(0, np.uint32), np.zeros((0, 3), np.int64))
        assert rc == capi.E_ARG and "NEED_K" in capi.lib.svjg_last_error().decode()
        cell, ppl = _patch(rng, gt, fl, S)
        cell = np.concatenate([need, cell]).astype(np.uint32)        # the NEED_K cells: the host's PLs first
        ppl = np.concatenate([pl[need], ppl])
        cell, first = np.unique(cell[::-1], return_index=True)       # one patch per cell: the last one
        ppl = ppl[::-1][first]
        rc, af, gp, gq, iters = _run_posteriors(co, n, blk, cell, ppl)
        assert rc == capi.OK, capi.lib.svjg_last_error()
        pl[cell] = ppl
        w_af, w_gp, w_gq, w_it, _err = posteriors(gt, fl, pl, S)
        assert _same_bits(af, w_af) and _same_bits(gp, w_gp)
        assert (gq == w_gq).all() and (iters == w_it).all()
        assert np.isnan(af[0]) and iters[0] == 0 and (gq[:S] == GQ_NONE).all()
        assert (iters == capi.POST_MAX_ITERS).any() and ((iters > 0) & (iters < capi.POST_MAX_ITERS)).any()
        if ploidy:
            kinds = cell_kinds(gt, fl)
            assert (kinds == 1).any() and (gt == capi.GT_NO_CALL).any()


@pytest.mark.gpu
def test_extreme_cohorts():
    """One strong 1/1 cell among 4 095 strong 0/0 cells, and every cell a strong 1/1: f stays in [1/S, 1], den > 0."""
    from svjg import alnfilter
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    S, n = 4096, 3
    co = cohort.Cohort(t, S)
    for s in range(S):
        c = np.zeros((t.num_sv, 2), np.uint32)
        c[:n] = [12, 0]
        co.load_counts(s, c)
    blk = cohort._Block(n * S, post_records=n)
    gt, fl, _ad, pl = (a.copy() for a in cohort._genotype_block(co, np.arange(n, dtype=np.uint32), np.full(n, 2, np.uint8),
                                                                  3, genotype.ERR, blk))
    strong_ref, strong_alt = [0, 9000, 20000], [20000, 9000, 0]
    ppl = np.array([strong_ref] * S + [strong_ref] * (S - 1) + [strong_alt] + [strong_alt] * S, np.int64)
    cell = np.arange(n * S, dtype=np.uint32)
    rc, af, gp, gq, iters = _run_posteriors(co, n, blk, cell, ppl)
    assert rc == capi.OK
    pl[:] = ppl
    w = posteriors(gt, fl, pl, S)
    assert _same_bits(af, w[0]) and _same_bits(gp, w[1]) and (gq == w[2]).all() and (iters == w[3]).all()
    assert af[0] == 0.0 and af[1] == 1 / S and af[2] == 1.0
    assert np.isfinite(gp).all()


def _cells_of_text(text):
    """gt codes, flags and PL triples of the cells of a cohort VCF, as its text shows them (without GP and GQ)."""
    codes = {"0/0": 0, "0/1": 1, "1/1": 2, "./.": 3, "0": 4, "1": 5, ".": 6}
    gt, fl, pl, S = [], [], [], None
    for line in text.splitlines():
        if line.startswith("#"):
            continue
        cols = line.split("\t")
        S = len(cols) - 9
        for c in cols[9:]:
            f = c.split(":")
            pls = f[3].split(",")
            if "." in pls:                      # outside the gate, or ploidy 0: the cell does not contribute
                gt.append(capi.GT_NO_CALL if len(pls) == 1 else 3 if len(pls) == 3 else capi.GT_HAP_MISSING)
                fl.append(0)
                pl.append([0, 0, 0])
            else:
                gt.append(codes[f[0]])
                fl.append(capi.GT_GENOTYPED)
                p = [int(x) for x in pls]
                pl.append(p if len(p) == 3 else [p[0], 0, p[1]])
    return np.array(gt, np.uint8), np.array(fl, np.uint8), np.array(pl, np.int64), S


def _strip_posteriors(text):
    out = []
    for line in _lines(text):
        if line == AF_EM_LINE:
            continue
        if line.startswith("#"):
            out.append(line.replace(GP_GQ_LINES, ""))
            continue
        cols = line.rstrip("\n").split("\t")
        items = cols[7].split(";")
        assert items[-1].startswith("AF_EM=")
        cols[7] = ";".join(items[:-1]) or "."
        assert cols[8].endswith(":GP:GQ")
        cols[8] = cols[8][:-6]
        cols[9:] = [":".join(c.split(":")[:-2]) for c in cols[9:]]
        out.append("\t".join(cols) + "\n")
    return "".join(out).replace(GP_GQ_LINES, "")


def _check_run(plain, post):
    """``post`` is ``plain`` with the statement's posteriors of its cells."""
    gt, fl, pl, S = _cells_of_text(plain)
    af, gp, gq, _it, _err = posteriors(gt, fl, pl, S)
    assert post == add_posteriors(plain, gt, fl, af, gp, gq, S)
    return gt, fl, af


@pytest.mark.gpu
def test_s2_cohort_through_the_command_line(tmp_path):
    p, samples, _counts = _s2_cohort(tmp_path)
    names = [f"n{k}" for k in range(7)]
    sexes = ["F", "M"] * 3 + ["F"]
    open(p + "_ploidy.txt", "w").write(S2_PLOIDY)
    open(p + "_sex.txt", "w").write("".join(f"{nm}\t{x}\n" for nm, x in zip(names, sexes)))
    common = ["-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *[",".join(fs) for fs in samples], "--names",
              ",".join(names)]
    extra = ["--info-tags", "all", "--ploidy-file", p + "_ploidy.txt", "--sample-sex", p + "_sex.txt"]
    for k, more in enumerate(([], extra)):
        r0 = _cohort(*common, *more, "-o", p + f"_{k}a.vcf")
        r1 = _cohort(*common, *more, "-o", p + f"_{k}b.vcf", "--posteriors")
        assert r0.returncode == 0 and r1.returncode == 0, r1.stderr
        assert r0.stdout == r1.stdout
        plain, post = open(p + f"_{k}a.vcf").read(), open(p + f"_{k}b.vcf").read()
        assert _strip_posteriors(post) == plain
        gt, fl, af = _check_run(plain, post)
        kinds = cell_kinds(gt, fl)
        assert (kinds == 2).any() and (not more or (kinds == 1).any()) and not np.isnan(af).all()


@pytest.mark.gpu
def test_need_k_cells_through_the_command_line(tmp_path):
    """72 copies of s2 take cells (diploid, and haploid in the M sample) beyond the log10 C(n, k) table."""
    p = _s2_cohort(tmp_path)[0]
    gaf = read_golden("s2.gaf.gz")
    open(p + "_x72.gaf", "w").write(gaf * 72)
    open(p + "_ploidy.txt", "w").write(S2_PLOIDY)
    open(p + "_sex.txt", "w").write("x72 M\none F\n")
    common = ["-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", p + "_x72.gaf", p + "_whole.gaf", "--names", "x72,one",
              "--ploidy-file", p + "_ploidy.txt", "--sample-sex", p + "_sex.txt"]
    r0 = _cohort(*common, "-o", p + "_a.vcf")
    r1 = _cohort(*common, "-o", p + "_b.vcf", "--posteriors", "--info-tags", "AF,NS")
    r2 = _cohort(*common, "-o", p + "_c.vcf", "--info-tags", "AF,NS")
    assert r0.returncode == 0 and r1.returncode == 0 and r2.returncode == 0, r1.stderr
    plain, post = open(p + "_c.vcf").read(), open(p + "_b.vcf").read()
    assert _strip_posteriors(post) == plain
    _check_run(plain, post)
    # the cells beyond the table in sample x72 take part in the estimate
    one = _python_oracle_counts("s2", gaf)
    assert max(a + b for a, b in one.values()) * 72 > 256
    body = [ln.split("\t") for ln in post.splitlines() if not ln.startswith("#")]
    assert any(c.split(":")[0] in ("0", "1") and c.split(":")[-1] != "." for ln in body for c in ln[9:10])
