"""Sample QC table and pairwise relatedness of a cohort (genotype-cohort.py --sample-qc / --relatedness, DESIGN.md §8a).

The contract, stated here in Python:

* A cell's code is the final device code, the one the VCF prints: 0 = 0/0, 1 = 0/1, 2 = 1/1, 3 = ./., 4 = haploid 0,
  5 = haploid 1, 6 = haploid ., 7 = ploidy 0.  The NEED_K patch never changes it.
* Sample QC (``sample_counts``): per sample, the count of each code over every record (row ALL) and over the records of
  each SVTYPE code (rows DEL, INS, INV, BND: svtype & 0x3F = 0..3; a record of any other type counts in ALL only).
  The table shows HOM_REF HET HOM_ALT HAP_REF HAP_ALT = codes 0 1 2 4 5, MISSING = codes 3 + 6, NO_PLOIDY = code 7,
  CALL_RATE = called / (called + MISSING) with called the sum of the first five, HET_HOM_RATIO = HET / HOM_ALT; each
  ratio one double division, "%.6g", "." over 0.
* Relatedness (``pair_counts_brute``): for each pair i < j (i major) over the records where both cells are diploid and
  called (codes 0-2): NSV, HET1 / HET2 (i / j is 0/1), HETHET (both 0/1), IBS0 (one 0/0, the other 1/1); KINSHIP =
  (HETHET - 2 IBS0) / (HET1 + HET2), one double division of the exact integers, "%.6g", "." when HET1 + HET2 = 0
  (the KING-robust estimator, Manichaikul et al. 2010).
* On the device (``planes``): three bit planes per sample, C = codes 0-2, H = code 1, A = code 2; bit r of word w is
  record 32 w + r of the block that took word w, each block starting a new word, other bits 0.  The pair counts are
  popcounts of those words (``pair_counts_from_planes``), so they do not depend on the blocks.
"""
import io
import math
import os

import numpy as np
import pytest

from conftest import read_golden
from svjg import capi, cohort, genotype
from test_cohort import _cohort, _synthetic
from test_cohort_info import _s2_cohort
from test_cohort_ploidy import S2_PLOIDY, _set_ploidy

RELATEDNESS_HEADER = "#ID1\tID2\tNSV\tHET1\tHET2\tHETHET\tIBS0\tKINSHIP\n"


# ---------------------------------------------------------------------------------------------------------------
# the statement
# ---------------------------------------------------------------------------------------------------------------
def sample_counts(codes, ty):
    """[S][5][8] u32 histogram of the codes [n][S] of records of types ty [n]."""
    n, S = codes.shape
    h = np.zeros((S, 5, 8), np.int64)
    t = np.asarray(ty) & 0x3F
    for r in range(n):
        for s in range(S):
            h[s, 0, codes[r, s]] += 1
            if t[r] <= 3:
                h[s, 1 + t[r], codes[r, s]] += 1
    return h.astype(np.uint32)


def pair_counts_brute(codes):
    """[S (S - 1) / 2][5] = NSV, HET1, HET2, HETHET, IBS0 per pair i < j, i major: a loop over pairs and records."""
    n, S = codes.shape
    out = []
    for i in range(S):
        for j in range(i + 1, S):
            c = [0] * 5
            for r in range(n):
                a, b = int(codes[r, i]), int(codes[r, j])
                if a > 2 or b > 2:
                    continue
                c[0] += 1
                c[1] += a == 1
                c[2] += b == 1
                c[3] += a == 1 and b == 1
                c[4] += {a, b} == {0, 2}
            out.append(c)
    return np.array(out, np.uint32).reshape(-1, 5)


def pair_counts(codes):
    """pair_counts_brute by integer matrix products (for the larger cohorts of the GPU tests)."""
    S = codes.shape[1]
    C = (codes <= 2).astype(np.int64)
    H = (codes == 1).astype(np.int64)
    A = (codes == 2).astype(np.int64)
    R = (codes == 0).astype(np.int64)
    i, j = np.triu_indices(S, 1)
    m = [C.T @ C, H.T @ C, C.T @ H, H.T @ H, A.T @ R + R.T @ A]
    return np.stack([x[i, j] for x in m], axis=1).astype(np.uint32).reshape(-1, 5)


def planes(codes, blocks):
    """[3][S][words] u32 planes C, H, A of the codes [n][S] cut into blocks of the given record counts."""
    n, S = codes.shape
    assert sum(blocks) == n
    out, lo = [], 0
    weight = (np.uint64(1) << np.arange(32, dtype=np.uint64))[None, :, None]
    for m in blocks:
        w = -(-m // 32)
        sub = np.full((32 * w, S), 3, np.uint8)
        sub[:m] = codes[lo:lo + m]
        lo += m
        sub = sub.reshape(w, 32, S)
        out.append(np.stack([((cond.astype(np.uint64) * weight).sum(axis=1)).T
                             for cond in (sub <= 2, sub == 1, sub == 2)]))
    if not out:
        return np.zeros((3, S, 0), np.uint32)
    return np.concatenate(out, axis=2).astype(np.uint32)


def _popc(x):
    return np.unpackbits(np.ascontiguousarray(x, np.uint32).view(np.uint8)).sum()


def pair_counts_from_planes(p):
    """The device's form: per word, popc(Ci&Cj), popc(Hi&Cj), popc(Hj&Ci), popc(Hi&Hj), popc((Ai&Rj)|(Ri&Aj)),
    R = C & ~H & ~A."""
    C, H, A = p
    R = C & ~H & ~A
    S = C.shape[0]
    out = []
    for i in range(S):
        for j in range(i + 1, S):
            out.append([_popc(C[i] & C[j]), _popc(H[i] & C[j]), _popc(H[j] & C[i]), _popc(H[i] & H[j]),
                        _popc((A[i] & R[j]) | (R[i] & A[j]))])
    return np.array(out, np.uint32).reshape(-1, 5)


def _ratio(a, b):
    return "." if b == 0 else f"{a / b:.6g}"


def sample_qc_table(names, h):
    lines = ["#SAMPLE\tSVTYPE\tHOM_REF\tHET\tHOM_ALT\tHAP_REF\tHAP_ALT\tMISSING\tNO_PLOIDY\tCALL_RATE\tHET_HOM_RATIO\n"]
    for nm, hs in zip(names, h):
        for ty, c in zip(("ALL", "DEL", "INS", "INV", "BND"), hs.tolist()):
            called, miss = c[0] + c[1] + c[2] + c[4] + c[5], c[3] + c[6]
            lines.append(f"{nm}\t{ty}\t{c[0]}\t{c[1]}\t{c[2]}\t{c[4]}\t{c[5]}\t{miss}\t{c[7]}\t"
                         f"{_ratio(called, called + miss)}\t{_ratio(c[1], c[2])}\n")
    return "".join(lines)


def kinship(c):
    """None when HET1 + HET2 = 0."""
    den = int(c[1]) + int(c[2])
    return None if den == 0 else (int(c[3]) - 2 * int(c[4])) / den


def relatedness_table(names, pairs, min_kinship=None):
    lines, k = [RELATEDNESS_HEADER], 0
    S = len(names)
    for i in range(S):
        for j in range(i + 1, S):
            c = pairs[k].tolist()
            k += 1
            kin = kinship(c)
            if min_kinship is not None and (kin is None or not kin >= min_kinship):
                continue
            lines.append(f"{names[i]}\t{names[j]}\t{c[0]}\t{c[1]}\t{c[2]}\t{c[3]}\t{c[4]}\t"
                         f"{'.' if kin is None else f'{kin:.6g}'}\n")
    return "".join(lines)


def _random_codes(rng, n, S):
    codes = rng.integers(0, 8, (n, S)).astype(np.uint8)
    codes.reshape(-1)[:8] = np.arange(8)[:min(8, codes.size)]          # every code, when there is room
    return codes


# ---------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2, 3, 40])
@pytest.mark.parametrize("n", [1, 45, 100])
def test_statement_forms_agree(S, n):
    rng = np.random.default_rng(1000 * S + n)
    codes = _random_codes(rng, n, S)
    ty = rng.choice(np.array([0, 1, 2, 3, 0x80, 0x83, 9, 255], np.uint8), n)
    want = pair_counts_brute(codes)
    assert want.shape == (S * (S - 1) // 2, 5)
    assert (pair_counts(codes) == want).all()
    for blocks in ([n], [1] * n, [7] * (n // 7) + ([n % 7] if n % 7 else []), [33] * (n // 33) + ([n % 33] if n % 33 else [])):
        p = planes(codes, blocks)
        assert p.shape == (3, S, sum(-(-m // 32) for m in blocks))
        assert (pair_counts_from_planes(p) == want).all()
    h = sample_counts(codes, ty)
    assert (h[:, 0].sum(axis=1) == n).all()
    assert (h[:, 1:].sum(axis=(1, 2)) == ((ty & 0x3F) <= 3).sum()).all()
    assert (h[:, 1:].sum(axis=1) <= h[:, 0]).all()


def test_kinship_of_identical_and_opposite_samples():
    g = np.array([0, 1, 1, 2, 2, 0, 3, 1], np.uint8)
    codes = np.stack([g, g, np.where(g == 0, 2, np.where(g == 2, 0, g))], axis=1)
    c = pair_counts_brute(codes)
    assert c[0].tolist() == [7, 3, 3, 3, 0] and kinship(c[0]) == 0.5
    assert c[1].tolist() == [7, 3, 3, 3, 4] and kinship(c[1]) == (3 - 8) / 6


def _format(names, pairs, min_kinship=None):
    buf = io.BytesIO()
    cohort.write_relatedness(buf, names, pairs, min_kinship)
    return buf.getvalue().decode()


def _random_pairs(rng, S):
    P = S * (S - 1) // 2
    pairs = rng.integers(0, 50, (P, 5)).astype(np.uint32)
    pairs[rng.random(P) < 0.1, 1:3] = 0                                   # KINSHIP "."
    pairs[rng.random(P) < 0.1, 3] = pairs[rng.random(P) < 0.1, 4] = 0
    if P:
        pairs[0] = [10, 3, 3, 3, 0]                                       # 0.5
        pairs[-1] = [10, 0, 0, 0, 0]                                      # "."
    return pairs


@pytest.mark.parametrize("S", [1, 2, 5, 130, 400])
def test_format_relatedness(S, monkeypatch):
    rng = np.random.default_rng(S)
    names = [f"s{k}" + "x" * (k % 3) for k in range(S)]
    pairs = _random_pairs(rng, S)
    for mk in (None, 0.0, 0.25, 0.5, -1.0, -0.0, 10.0):
        want = relatedness_table(names, pairs, mk)
        assert _format(names, pairs, mk) == want
    if S == 1:
        assert _format(names, pairs) == RELATEDNESS_HEADER
    # several row ranges per table: the pieces joined are the whole
    monkeypatch.setattr(cohort, "RELATEDNESS_PIECE_PAIRS", 7)
    assert _format(names, pairs, 0.1) == relatedness_table(names, pairs, 0.1)
    assert _format(names, pairs) == relatedness_table(names, pairs)


def test_format_relatedness_refusals():
    import ctypes as C
    pairs = np.zeros((3, 5), np.uint32)
    buf, n = C.c_void_p(), C.c_uint64()
    for names, use_min, mk, msg in ((b"a\tb\tc", 1, math.nan, "finite"), (b"a\tb\tc", 1, math.inf, "finite"),
                                    (b"a\tb", 0, 0.0, "names")):
        rc = capi.lib.svjg_format_relatedness(3, names, len(names), pairs.ctypes.data, 0, 3, use_min, mk, C.byref(buf),
                                              C.byref(n))
        assert rc == capi.E_ARG and msg in capi.lib.svjg_last_error().decode()
    rc = capi.lib.svjg_format_relatedness(3, b"a\tb\tc", 5, pairs.ctypes.data, 2, 4, 0, 0.0, C.byref(buf), C.byref(n))
    assert rc == capi.E_ARG
    with pytest.raises(ValueError):
        _format(["a", "b"], pairs)


def test_sample_qc_text():
    rng = np.random.default_rng(4)
    h = rng.integers(0, 30, (6, 5, 8)).astype(np.uint32)
    h[0, 1] = 0                                                            # no DEL: both ratios "."
    h[1, 2, [0, 1, 2, 4, 5]] = 0                                           # nothing called: CALL_RATE 0
    h[2, 3, 2] = 0                                                         # HET_HOM_RATIO "."
    names = [f"n{k}" for k in range(6)]
    text = cohort.sample_qc_text(names, h)
    assert text == sample_qc_table(names, h)
    rows = [ln.split("\t") for ln in text.splitlines()[1:]]
    assert len(rows) == 30 and [r[1] for r in rows[:5]] == ["ALL", "DEL", "INS", "INV", "BND"]
    assert rows[1][9:] == [".", "."] and rows[7][9] == "0" and rows[13][10] == "."


def test_help_names_the_switches():
    r = _cohort("--help")
    assert r.returncode == 0 and "--sample-qc" in r.stdout and "--relatedness" in r.stdout
    assert "--min-kinship" in r.stdout and "16384" in r.stdout


@pytest.mark.parametrize("extra,message", [
    (["--min-kinship", "0.1"], "--min-kinship needs --relatedness"),
    (["--relatedness", "R", "--min-kinship", "nan"], "finite"),
    (["--relatedness", "R", "--min-kinship", "inf"], "finite"),
    (["--relatedness", "R", "--min-kinship=-inf"], "finite"),
    (["--relatedness", "R", "--min-kinship", "x"], "finite"),
    (["--relatedness", "O"], "--relatedness names the same file"),
    (["--sample-qc", "O"], "--sample-qc names the same file"),
    (["--sample-qc", "R", "--relatedness", "R"], "--relatedness names the same file"),
    (["--relatedness", "R", "MANY"], "at most 16384 samples"),
    (["--sample-qc", "Q", "--relatedness", "R", "--ploidy-file", "P"], "given together"),
])
def test_command_line_refusals(tmp_path, extra, message):
    out = tmp_path / "out"
    out.mkdir()
    args = []
    for a in extra:
        if a == "MANY":
            args += ["-a"] + [f"g{k}.gaf" for k in range(16385)]
            continue
        args.append({"R": str(out / "r.tsv"), "Q": str(out / "q.tsv"), "O": str(out / "o.vcf"),
                     "P": str(tmp_path / "p.txt")}.get(a, a))
    (tmp_path / "p.txt").write_text("chrX 1 10 M 1\n")
    r = _cohort("-p", str(out / "x"), "-g", "x.gfa", "-v", "x.vcf", "-a", "one.gaf", "two.gaf", "-o", str(out / "o.vcf"),
                *args, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and message in r.stderr, r.stderr
    assert not os.listdir(out)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
_KIND_COUNTS = np.array([[12, 0], [6, 6], [0, 12], [1, 1], [0, 0]], np.uint32)    # 0/0, 0/1, 1/1, below -ms, gated
_TYPES = np.array([0, 1, 2, 3, 0x81, 9], np.uint8)                                 # DEL INS INV BND, short INS, other


def _qc_case(t, S, n, rng, ploidy):
    co = cohort.Cohort(t, S)
    pick = rng.integers(0, 5, (n, S))
    for s in range(S):
        c = np.zeros((t.num_sv, 2), np.uint32)
        c[:n] = _KIND_COUNTS[pick[:, s]]
        c[1:n:9] = [300, 280]                                         # beyond the log10 C(n, k) table: NEED_K
        co.load_counts(s, c)
    idx = np.arange(n, dtype=np.uint32)
    idx[0] = capi.NO_SV
    ty = rng.choice(_TYPES, n)
    rclass = None
    if ploidy:
        _set_ploidy(co, np.array([[2, 2], [1, 2], [0, 1], [1, 1]], np.uint8), (np.arange(S) % 2).astype(np.uint8))
        rclass = rng.integers(0, 4, n).astype(np.uint8)
    return co, idx, ty, rclass


def _run_blocks(co, idx, ty, rclass, step):
    """The block loop of genotype_cohort_vcf with svjg_cohort_qc_add after each block: (codes [n][S], block sizes)."""
    S, n = co.n_samples, len(idx)
    blocks = [min(step, n - lo) for lo in range(0, n, step)]
    capi.check(capi.lib.svjg_cohort_qc_begin(co._h, sum(-(-m // 32) for m in blocks), 1))
    blk = cohort._Block(min(step, n) * S)
    codes = []
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        gt = cohort._genotype_block(co, idx[lo:hi], ty[lo:hi], 3, genotype.ERR, blk,
                                    None if rclass is None else rclass[lo:hi])[0]
        capi.check(capi.lib.svjg_cohort_qc_add(co._h, hi - lo))
        codes.append(gt.reshape(hi - lo, S).copy())
    return np.concatenate(codes), blocks


def _read_back(co, n_words):
    S = co.n_samples
    h = np.zeros((S, 5, 8), np.uint32)
    capi.check(capi.lib.svjg_cohort_qc_sample_counts(co._h, h.ctypes.data))
    p = np.zeros((3, S, n_words), np.uint32)
    capi.check(capi.lib.svjg_cohort_qc_planes(co._h, p.ctypes.data))
    pairs = np.zeros((S * (S - 1) // 2, 5), np.uint32)
    capi.check(capi.lib.svjg_cohort_relatedness(co._h, pairs.ctypes.data if pairs.size else None))
    return h, p, pairs


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 2, 31, 32, 33, 127, 128, 129, 200, 1000])
def test_kernels_against_the_statement(S):
    from svjg import alnfilter
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    n = 100 if S == 1000 else 150
    rng = np.random.default_rng(S)
    for ploidy in (True, False):
        co, idx, ty, rclass = _qc_case(t, S, n, rng, ploidy)
        want_pairs = None
        for step in ((1, 7, 31, 32, 33, n) if ploidy else (n, 33)):
            codes, blocks = _run_blocks(co, idx, ty, rclass, step)
            if ploidy:
                assert {4, 5, 6, 7} <= set(np.unique(codes).tolist())
            assert {0, 1, 2, 3} <= set(np.unique(codes).tolist())
            h, p, pairs = _read_back(co, sum(-(-m // 32) for m in blocks))
            assert (p == planes(codes, blocks)).all()
            hist_want = np.zeros((S, 5, 8), np.int64)
            t6 = ty & 0x3F
            for code in range(8):
                hit = (codes == code).astype(np.int64)
                hist_want[:, 0, code] = hit.sum(axis=0)
                for k in range(4):
                    hist_want[:, 1 + k, code] = hit[t6 == k].sum(axis=0)
            assert (h == hist_want).all()
            if want_pairs is None:
                want_pairs = pair_counts(codes)
            assert (pairs == want_pairs).all()
        co.close()


@pytest.mark.gpu
def test_api_refusals_and_the_module():
    from svjg import alnfilter
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    S, n = 33, 70
    rng = np.random.default_rng(2)
    co, idx, ty, _rc = _qc_case(t, S, n, rng, False)
    assert capi.lib.svjg_cohort_qc_add(co._h, 0) == capi.E_ARG                   # no qc_begin
    blk = cohort._Block(n * S)
    capi.check(capi.lib.svjg_cohort_qc_begin(co._h, 2, 0))
    cohort._genotype_block(co, idx[:40], ty[:40], 3, genotype.ERR, blk)
    assert capi.lib.svjg_cohort_qc_add(co._h, 39) == capi.E_ARG                  # not the block's size
    capi.check(capi.lib.svjg_cohort_qc_add(co._h, 40))
    assert capi.lib.svjg_cohort_qc_add(co._h, 40) == capi.E_ARG                  # the same block twice
    cohort._genotype_block(co, idx[40:], ty[40:], 3, genotype.ERR, blk)
    assert capi.lib.svjg_cohort_qc_add(co._h, 30) == capi.E_ARG                  # beyond n_words
    pairs = np.zeros((S * (S - 1) // 2, 5), np.uint32)
    assert capi.lib.svjg_cohort_relatedness(co._h, pairs.ctypes.data) == capi.E_ARG   # no want_pairs
    co.close()
    # genotype_cohort_vcf: the same text, and tables that do not depend on the blocks
    from svjg import synth
    v = genotype.NativeVcf.from_input(synth.vcf_text(_rows).encode())
    co = cohort.Cohort(t, S)
    for s in range(S):
        co.load_counts(s, _KIND_COUNTS[rng.integers(0, 5, t.num_sv)])
    names = [f"s{k}" for k in range(S)]
    text, n_gt = cohort.genotype_cohort_vcf(t, co, v, names)
    codes = _vcf_codes(text)
    assert {0, 1, 2, 3} <= set(np.unique(codes).tolist())
    for step in (None, 7, 33):
        res = cohort.genotype_cohort_vcf(t, co, v, names, block_records=step, sample_qc=True, relatedness=True)
        assert res[:2] == (text, n_gt)
        assert (res[2] == sample_counts(codes, v.svtype)).all() and (res[3] == pair_counts(codes)).all()
    res = cohort.genotype_cohort_vcf(t, co, v, names, sample_qc=True)
    assert res[:2] == (text, n_gt) and res[3] is None and (res[2] == sample_counts(codes, v.svtype)).all()
    res = cohort.genotype_cohort_vcf(t, co, v, names, relatedness=True)
    assert res[:2] == (text, n_gt) and res[2] is None and (res[3] == pair_counts(codes)).all()
    co.close()
    with pytest.raises(capi.SvjgError, match="SVJG_QC_MAX_PAIR_SAMPLES"):
        big = cohort.Cohort(t, capi.QC_MAX_PAIR_SAMPLES + 1)
        try:
            capi.check(capi.lib.svjg_cohort_qc_begin(big._h, 1, 1))
        finally:
            big.close()


def _vcf_codes(text):
    """gt codes [n][S] of a written cohort VCF, from its GT fields (a ploidy-0 cell has a one-value PL: '.')."""
    codes = {"0/0": 0, "0/1": 1, "1/1": 2, "./.": 3, "0": 4, "1": 5}
    rows = []
    for line in text.splitlines():
        if line.startswith("#"):
            continue
        row = []
        for c in line.split("\t")[9:]:
            f = c.split(":")
            row.append(codes[f[0]] if f[0] in codes else 7 if f[3] == "." else 6)
        rows.append(row)
    return np.array(rows, np.uint8)


def _catalogue_types(vcf_text):
    return np.array([rec[1] for rec in genotype.parse_vcf(vcf_text.splitlines(True))[1]], np.uint8)


def _parse_qc(path):
    return [ln.split("\t") for ln in open(path).read().splitlines()]


def _check_tables(vcf_path, cat_path, names, qc_path, rel_path, min_kinship=None):
    text = open(vcf_path).read()
    codes = _vcf_codes(text)
    ty = _catalogue_types(open(cat_path).read())
    assert codes.shape == (len(ty), len(names))
    h = sample_counts(codes, ty)
    assert open(qc_path).read() == sample_qc_table(names, h)
    pairs = pair_counts(codes)
    assert open(rel_path).read() == relatedness_table(names, pairs, min_kinship)
    return codes, h, pairs


@pytest.mark.gpu
def test_s2_cohort_through_the_command_line(tmp_path):
    p, samples, _counts = _s2_cohort(tmp_path)
    samples = samples + [samples[3]]                                   # the x48 GAF again, under a second name
    names = [f"n{k}" for k in range(7)] + ["dup"]
    sexes = ["F", "M"] * 3 + ["F", "M"]
    open(p + "_ploidy.txt", "w").write(S2_PLOIDY)
    open(p + "_sex.txt", "w").write("".join(f"{nm}\t{x}\n" for nm, x in zip(names, sexes)))
    common = ["-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", *[",".join(fs) for fs in samples], "--names",
              ",".join(names), "--info-tags", "all", "--ploidy-file", p + "_ploidy.txt", "--sample-sex", p + "_sex.txt",
              "--posteriors"]
    r0 = _cohort(*common, "-o", p + "_a.vcf")
    r1 = _cohort(*common, "-o", p + "_b.vcf", "--sample-qc", p + "_q.tsv", "--relatedness", p + "_r.tsv")
    r2 = _cohort(*common, "-o", p + "_c.vcf", "--relatedness", p + "_r2.tsv", "--min-kinship", "0.3")
    assert r0.returncode == 0 and r1.returncode == 0 and r2.returncode == 0, r1.stderr + r2.stderr
    assert r0.stdout == r1.stdout == r2.stdout
    plain = open(p + "_a.vcf", "rb").read()
    assert open(p + "_b.vcf", "rb").read() == plain and open(p + "_c.vcf", "rb").read() == plain
    codes, h, pairs = _check_tables(p + "_b.vcf", p + ".vcf", names, p + "_q.tsv", p + "_r.tsv")
    assert open(p + "_r2.tsv").read() == relatedness_table(names, pairs, 0.3)
    assert {0, 1, 2, 3, 4, 5, 7} <= set(np.unique(codes).tolist())
    rel = {(r[0], r[1]): r for r in _parse_qc(p + "_r.tsv")[1:]}
    for a, b in (("n3", "dup"), ("n0", "n5")):                         # the same GAF twice
        assert rel[a, b][6] == "0" and rel[a, b][7] == "0.5", rel[a, b]
    qc = {(r[0], r[1]): r for r in _parse_qc(p + "_q.tsv")[1:]}
    assert qc["n4", "ALL"][9] == "0"                                   # the empty sample
    assert all(r[7] == "." for (a, b), r in rel.items() if "n4" in (a, b))
    assert ("n3", "dup") in {(r[0], r[1]) for r in _parse_qc(p + "_r2.tsv")[1:]}
    # the males' haploid calls are in the sample table, and missing from their pairs
    assert sum(int(r[5]) + int(r[6]) for (nm, ty), r in qc.items() if ty == "ALL") > 0
    # a table that cannot be written: none of the three outputs is left behind
    r = _cohort(*common, "-o", p + "_d.vcf", "--sample-qc", p + "_dq.tsv", "--relatedness", p + "_none/r.tsv")
    assert r.returncode == 1 and "No such file" in r.stderr, r.stderr
    assert not [f for f in os.listdir(tmp_path) if "_d" in f and f.endswith((".vcf", ".tsv")) or f.startswith(".")]


@pytest.mark.gpu
def test_need_k_cells_through_the_command_line(tmp_path):
    """72 copies of s2 take cells beyond the log10 C(n, k) table (patched on the host): the tables still match the
    VCF's GT fields."""
    p = _s2_cohort(tmp_path)[0]
    gaf = read_golden("s2.gaf.gz")
    open(p + "_x72.gaf", "w").write(gaf * 72)
    open(p + "_ploidy.txt", "w").write(S2_PLOIDY)
    open(p + "_sex.txt", "w").write("x72 M\none F\nagain F\n")
    common = ["-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", p + "_x72.gaf", p + "_whole.gaf", p + "_x72.gaf",
              "--names", "x72,one,again", "--ploidy-file", p + "_ploidy.txt", "--sample-sex", p + "_sex.txt"]
    for k, more in enumerate(([], ["--posteriors", "--info-tags", "AF,NS"])):
        r0 = _cohort(*common, *more, "-o", p + f"_{k}a.vcf")
        r1 = _cohort(*common, *more, "-o", p + f"_{k}b.vcf", "--sample-qc", p + f"_{k}q.tsv", "--relatedness",
                     p + f"_{k}r.tsv")
        assert r0.returncode == 0 and r1.returncode == 0, r1.stderr
        assert open(p + f"_{k}a.vcf", "rb").read() == open(p + f"_{k}b.vcf", "rb").read()
        _check_tables(p + f"_{k}b.vcf", p + ".vcf", ["x72", "one", "again"], p + f"_{k}q.tsv", p + f"_{k}r.tsv")
