"""Genetic relationship matrix and principal components of a cohort (genotype-cohort.py --grm / --pca, DESIGN.md §8a).

The contract, stated here in Python:

* A cell's code is the final device code, the one the VCF prints (0 = 0/0, 1 = 0/1, 2 = 1/1, 3 = ./., 4-6 haploid,
  7 = ploidy 0).  Only diploid called cells (codes 0-2) carry a dosage g = code; every other cell is missing.
* Per record (``record_table``): AN = 2 x (cells with codes 0-2), AC = (code 1) + 2 x (code 2).  The record is used iff
  0 < AC < AN and double(min(AC, AN - AC)) / double(AN) >= min_maf.  Then p = AC / AN, s = 2.0 * p,
  w = 1.0 / (s * (1.0 - p)), v_g = g - s and u_g = w * v_g, each one double operation rounded to nearest.
* Per pair i <= j (``grm_statement``): N_ij = the used records where both cells are diploid called; acc_ij = +0.0, then
  acc = acc + (u_{g_i} * v_{g_j}) record by record in ascending order, the multiply and the add rounded separately;
  G_ij = acc_ij / N_ij, 0.0 when N_ij = 0; G_ji = G_ij.
* PCA (``cohort.pca``): numpy.linalg.eigh of the full symmetric G; the K largest eigenvalues in descending order and
  their unit eigenvectors, each flipped so that its component of largest absolute value (the first on ties) is > 0.
* Files: PREFIX.grm.bin / PREFIX.grm.N.bin = G / N as little-endian float32, lower triangle row by row with the
  diagonal; PREFIX.grm.id = "NAME\\tNAME" per sample; PREFIX.eigenvec = "#IID\\tPC1 ... PCK" then one "%.6g" line per
  sample; PREFIX.eigenval = one "%.6g" eigenvalue per line.

A missing cell or an unused record enters the device's sum as a +-0 term, which leaves a sum that starts at +0.0
unchanged, so the bits do not depend on the blocks or on the padding bits of the planes.
"""
import io
import os
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest

from svjg import capi, cohort, genotype
from test_cohort import _cohort, _synthetic
from test_cohort_info import _s2_cohort
from test_cohort_ploidy import S2_PLOIDY, _set_ploidy
from test_cohort_qc import _KIND_COUNTS, _TYPES, _run_blocks, _vcf_codes, pair_counts


# ---------------------------------------------------------------------------------------------------------------
# the statement
# ---------------------------------------------------------------------------------------------------------------
def record_table(codes, min_maf):
    """(used [n] bool, u [n][3], v [n][3]) of the codes [n][S]; zeros for the records that are not used."""
    codes = np.asarray(codes)
    called = codes <= 2
    an = 2 * called.sum(axis=1).astype(np.int64)
    ac = (codes == 1).sum(axis=1).astype(np.int64) + 2 * (codes == 2).sum(axis=1).astype(np.int64)
    used = (ac > 0) & (ac < an)
    used[used] = np.minimum(ac[used], an[used] - ac[used]).astype(np.float64) / an[used].astype(np.float64) >= min_maf
    u = np.zeros((len(codes), 3))
    v = np.zeros((len(codes), 3))
    p = ac[used].astype(np.float64) / an[used].astype(np.float64)
    s = 2.0 * p
    w = 1.0 / (s * (1.0 - p))
    v[used] = np.arange(3.0)[None, :] - s[:, None]
    u[used] = w[:, None] * v[used]
    return used, u, v


def grm_statement(codes, min_maf):
    """(G [S][S] float64, N [S][S] uint32) of the codes [n][S]: one record at a time, in order."""
    codes = np.asarray(codes)
    n, S = codes.shape
    used, u, v = record_table(codes, min_maf)
    called = codes <= 2
    g = np.where(called, codes, 0).astype(np.int64)
    acc = np.zeros((S, S))
    for r in np.flatnonzero(used):
        ur = np.where(called[r], u[r][g[r]], 0.0)
        vr = np.where(called[r], v[r][g[r]], 0.0)
        acc += np.multiply.outer(ur, vr)
    cu = (called & used[:, None]).astype(np.int64)
    N = cu.T @ cu
    G = np.zeros((S, S))
    np.divide(acc, N, out=G, where=N > 0)
    iu = np.triu_indices(S)
    G.T[iu] = G[iu]                                               # the pair i <= j is u_i v_j
    return G, N.astype(np.uint32)


def grm_exact(codes, min_maf):
    """G and N by exact rational arithmetic of the formula, and the scale sum |terms| / N of each pair."""
    codes = np.asarray(codes)
    n, S = codes.shape
    used, _u, _v = record_table(codes, min_maf)
    terms = []
    for r in np.flatnonzero(used):
        row = codes[r]
        an = 2 * int((row <= 2).sum())
        ac = int((row == 1).sum()) + 2 * int((row == 2).sum())
        s = Fraction(2 * ac, an)
        w = 1 / (s * (1 - Fraction(ac, an)))
        terms.append((r, [[w * (a - s) * (b - s) for b in range(3)] for a in range(3)]))
    G, N, scale = np.zeros((S, S), object), np.zeros((S, S), np.int64), np.zeros((S, S))
    for i in range(S):
        for j in range(i, S):
            acc, mag, k = Fraction(0), 0.0, 0
            for r, t in terms:
                a, b = int(codes[r, i]), int(codes[r, j])
                if a <= 2 and b <= 2:
                    acc += t[a][b]
                    mag += abs(float(t[a][b]))
                    k += 1
            G[i, j] = G[j, i] = acc / k if k else Fraction(0)
            N[i, j] = N[j, i] = k
            scale[i, j] = scale[j, i] = mag / k if k else 0.0
    return G, N, scale


def packed(M):
    """The packed upper triangle of svjg_cohort_grm (pair i <= j at i (2 S - i + 1) / 2 + j - i)."""
    return M[np.triu_indices(M.shape[0])]


def _random_codes(rng, n, S, p_missing=0.15):
    f = rng.uniform(0.02, 0.98, n)
    codes = rng.binomial(2, f[:, None], (n, S)).astype(np.uint8)
    codes[rng.random((n, S)) < p_missing] = 3
    codes[rng.random((n, S)) < 0.05] = rng.integers(4, 8, 1)[0]
    return codes


# ---------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("min_maf", [0.0, 0.1])
def test_statement_against_exact_arithmetic(min_maf):
    rng = np.random.default_rng(40)
    S, n = 40, 300
    codes = _random_codes(rng, n, S)
    codes[:5] = 0                                                 # monomorphic
    codes[5:8] = 2
    codes[8, :] = 0
    codes[8, 3] = 1                                               # one het: MAF 1 / AN
    codes[:, 7] = 3                                               # an all-missing sample
    used = record_table(codes, min_maf)[0]
    assert not used[:8].any() and used[8] == (min_maf == 0.0) and used.sum() > 200
    G, N = grm_statement(codes, min_maf)
    Gx, Nx, scale = grm_exact(codes, min_maf)
    assert (N == Nx).all() and (G == G.T).all()
    err = np.abs(G - Gx.astype(np.float64))
    assert (err <= 1e-12 * scale).all(), err.max()
    assert (G[7] == 0).all() and (N[7] == 0).all()
    assert np.abs(np.diag(G)[N.diagonal() > 0] - 1).max() < 0.5   # the diagonal is about 1 for unrelated samples


def test_duplicated_sample_gives_identical_rows():
    rng = np.random.default_rng(2)
    base = _random_codes(rng, 200, 12)
    codes = np.concatenate([base[:, :5], base[:, 4:5], base[:, 5:], base[:, 9:10]], axis=1)   # 4 twice, 9 twice
    G, N = grm_statement(codes, 0.01)
    assert (G[4] == G[5]).all() and (N[4] == N[5]).all()         # adjacent: the same roundings
    assert (N[10] == N[13]).all()
    assert np.allclose(G[10], G[13], rtol=1e-12, atol=1e-14)      # apart: u_j v_i and u_i v_j round differently


def _two_populations(rng, n_a, n_b, n):
    fa = rng.uniform(0.05, 0.95, n)
    fb = np.clip(fa + rng.choice([-0.4, 0.4], n), 0.02, 0.98)
    codes = np.concatenate([rng.binomial(2, fa[:, None], (n, n_a)), rng.binomial(2, fb[:, None], (n, n_b))], axis=1)
    codes = codes.astype(np.uint8)
    codes[rng.random(codes.shape) < 0.05] = 3
    return codes


def test_two_populations_split_by_pc1():
    rng = np.random.default_rng(7)
    codes = _two_populations(rng, 15, 25, 400)
    G, _N = grm_statement(codes, 0.01)
    vals, vecs = cohort.pca(G, 3)
    assert vals[0] > vals[1] >= vals[2]
    pc1 = vecs[:, 0]
    assert (np.sign(pc1[:15]) == np.sign(pc1[0])).all() and (np.sign(pc1[15:]) == -np.sign(pc1[0])).all()


def test_pca_sign_rule_and_order():
    x = np.array([1.0, -1.0, 0.5, 0.25])
    x /= np.linalg.norm(x)
    y = np.array([0.0, 0.1, -0.9, 0.2])
    y -= (y @ x) * x
    y /= np.linalg.norm(y)
    for sx, sy in ((1, 1), (-1, -1), (1, -1)):
        G = 3.0 * np.outer(sx * x, sx * x) + 2.0 * np.outer(sy * y, sy * y)
        vals, vecs = cohort.pca(G, 2)
        assert np.allclose(vals, [3.0, 2.0])
        lead = np.argmax(np.abs(vecs), axis=0)
        assert (vecs[lead, [0, 1]] > 0).all()
        assert np.isclose(abs(vecs[:, 0] @ x), 1.0) and np.allclose(vecs[:, 1], -y)   # x: |x0| = |x1| up to rounding
        assert np.allclose(np.linalg.norm(vecs, axis=0), 1.0)
    # an exact tie of |a| and |-a|: the first is made positive (eigh gives (-a, a) here)
    vals, vecs = cohort.pca(np.array([[2.0, -2.0, 0.0], [-2.0, 2.0, 0.0], [0.0, 0.0, 1.0]]), 1)
    assert vals[0] == 4.0 and vecs[0, 0] > 0 and vecs[0, 0] == -vecs[1, 0] and vecs[2, 0] == 0
    with pytest.raises(ValueError):
        cohort.pca(np.eye(3), 4)
    with pytest.raises(ValueError):
        cohort.pca(np.eye(3), 0)


def test_pca_repeats_itself_across_processes():
    """The command line computes the PCA in its own process: numpy's eigh gives the same bits in another one."""
    rng = np.random.default_rng(5)
    G, _N = grm_statement(_two_populations(rng, 30, 50, 300), 0.01)
    code = ("import sys, numpy as np; sys.path.insert(0, sys.argv[1]); from svjg import cohort; "
            "G = np.frombuffer(sys.stdin.buffer.read()).reshape(80, 80); v, e = cohort.pca(G, 10); "
            "sys.stdout.buffer.write(v.tobytes() + e.tobytes())")
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "svjedi-graph_b200")
    r = subprocess.run([sys.executable, "-c", code, pkg], input=G.tobytes(), capture_output=True, check=True)
    vals, vecs = cohort.pca(G, 10)
    assert r.stdout == vals.tobytes() + vecs.tobytes()


def _write(names, G, N):
    b, nb, ids = io.BytesIO(), io.BytesIO(), io.BytesIO()
    cohort.write_grm(b, nb, ids, names, G, N)
    return b.getvalue(), nb.getvalue(), ids.getvalue().decode()


@pytest.mark.parametrize("S", [1, 2, 7, 300])
def test_write_grm(S, monkeypatch):
    rng = np.random.default_rng(S)
    codes = _random_codes(rng, 60, S)
    G, N = grm_statement(codes, 0.0)
    names = [f"s{k}" for k in range(S)]
    b, nb, ids = _write(names, G, N)
    il = np.tril_indices(S)
    assert len(b) == len(nb) == 4 * S * (S + 1) // 2
    assert (np.frombuffer(b, "<f4") == G[il].astype(np.float32)).all()
    assert (np.frombuffer(nb, "<f4") == N[il].astype(np.float32)).all()
    want = [G[i, j] for i in range(min(S, 7)) for j in range(i + 1)]            # GCTA's order: row i, j = 0 .. i
    assert (np.frombuffer(b, "<f4")[:len(want)] == np.array(want, np.float32)).all()
    assert ids == "".join(f"{nm}\t{nm}\n" for nm in names)
    with pytest.raises(ValueError):
        _write(names + ["x"], G, N)


def test_grm_square_is_the_packed_triangle():
    rng = np.random.default_rng(3)
    for S in (1, 2, 9):
        M = rng.random((S, S))
        M = np.triu(M) + np.triu(M, 1).T
        assert (cohort.grm_square(packed(M), S, np.float64) == M).all()


def test_write_pca():
    rng = np.random.default_rng(9)
    G, _N = grm_statement(_two_populations(rng, 6, 5, 200), 0.01)
    vals, vecs = cohort.pca(G, 4)
    names = [f"n{k}" for k in range(11)]
    vo, eo = io.BytesIO(), io.BytesIO()
    cohort.write_pca(vo, eo, names, vals, vecs)
    lines = vo.getvalue().decode().splitlines()
    assert lines[0] == "#IID\tPC1\tPC2\tPC3\tPC4"
    assert [ln.split("\t")[0] for ln in lines[1:]] == names
    assert lines[1] == "n0\t" + "\t".join("%.6g" % x for x in vecs[0])
    got = np.array([[float(x) for x in ln.split("\t")[1:]] for ln in lines[1:]])
    assert np.allclose(got, vecs, rtol=1e-5, atol=1e-6)
    assert eo.getvalue().decode() == "".join("%.6g\n" % x for x in vals)
    with pytest.raises(ValueError):
        cohort.write_pca(vo, eo, names[:-1], vals, vecs)


def test_help_names_the_switches():
    r = _cohort("--help")
    assert r.returncode == 0
    for opt in ("--grm", "--pca", "--pca-components", "--grm-min-maf"):
        assert opt in r.stdout


@pytest.mark.parametrize("extra,message", [
    (["--pca-components", "3"], "--pca-components needs --pca"),
    (["--pca", "P", "--pca-components", "0"], "between 1 and the number of samples (2)"),
    (["--pca", "P", "--pca-components", "3"], "between 1 and the number of samples (2)"),
    (["--pca", "P"], "--pca-components 10: it must be between 1"),
    (["--pca", "P", "--pca-components", "x"], "must be an integer"),
    (["--grm-min-maf", "0.1"], "--grm-min-maf needs --grm or --pca"),
    (["--grm", "G", "--grm-min-maf", "0.6"], "in [0, 0.5]"),
    (["--grm", "G", "--grm-min-maf=-0.1"], "in [0, 0.5]"),
    (["--grm", "G", "--grm-min-maf", "nan"], "in [0, 0.5]"),
    (["--pca", "P", "--pca-components", "2", "--grm-min-maf", "inf"], "in [0, 0.5]"),
    (["--grm", "G", "--grm-min-maf", "x"], "in [0, 0.5]"),
    (["--grm", "OG"], "--grm names the same file"),
    (["--pca", "OP", "--pca-components", "1"], "--pca names the same file"),
    (["--grm", "G", "--relatedness", "GB"], "--grm names the same file"),
    (["--grm", "G", "--sample-qc", "GI"], "--grm names the same file"),
    (["--grm", "G", "MANY"], "--grm takes at most 16384 samples"),
    (["--pca", "P", "MANY"], "--pca takes at most 16384 samples"),
])
def test_command_line_refusals(tmp_path, extra, message):
    out = tmp_path / "out"
    out.mkdir()
    args = []
    for a in extra:
        if a == "MANY":
            args += ["-a"] + [f"g{k}.gaf" for k in range(16385)]
            continue
        args.append({"G": str(out / "g"), "P": str(out / "p"), "GB": str(out / "g.grm.bin"),
                     "GI": str(out / "g.grm.id"), "OG": str(out / "o"), "OP": str(out / "o")}.get(a, a))
    o = out / ("o.grm.N.bin" if "OG" in extra else "o.eigenval" if "OP" in extra else "o.vcf")
    r = _cohort("-p", str(out / "x"), "-g", "x.gfa", "-v", "x.vcf", "-a", "one.gaf", "two.gaf", "-o", str(o),
                *args, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 1 and message in r.stderr, r.stderr
    assert not os.listdir(out)


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
def _grm_case(t, S, n, rng, ploidy):
    """A cohort of S samples over n records: random cell kinds with NEED_K cells, monomorphic records (0/0 and 1/1),
    records of a single het, a sample with no call, and (``ploidy``) haploid and ploidy-0 cells."""
    co = cohort.Cohort(t, S)
    pick = rng.integers(0, 5, (n, S))
    pick[2:5] = 0
    pick[5:7] = 2
    pick[7:9] = 0
    pick[7:9, 0] = 1
    if S > 2:
        pick[:, S // 2] = 3
    for s in range(S):
        c = np.zeros((t.num_sv, 2), np.uint32)
        c[:n] = _KIND_COUNTS[pick[:, s]]
        if s != S // 2 or S <= 2:
            c[1:n:9] = [300, 280]                                     # beyond the log10 C(n, k) table: NEED_K
        co.load_counts(s, c)
    idx = np.arange(n, dtype=np.uint32)
    idx[0] = capi.NO_SV
    ty = rng.choice(_TYPES, n)
    ty[2:9] = 0                                                       # DEL: the hand-made records are genotyped
    rclass = None
    if ploidy:
        _set_ploidy(co, np.array([[2, 2], [1, 2], [0, 1], [1, 1]], np.uint8), (np.arange(S) % 2).astype(np.uint8))
        rclass = rng.integers(0, 4, n).astype(np.uint8)
        rclass[:12] = 0
    return co, idx, ty, rclass


def _device_grm(co, min_maf):
    S = co.n_samples
    g = np.full(S * (S + 1) // 2, np.nan)
    nn = np.full(S * (S + 1) // 2, 0xFFFFFFFF, np.uint32)
    capi.check(capi.lib.svjg_cohort_grm(co._h, min_maf, g.ctypes.data, nn.ctypes.data))
    return g, nn


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 2, 63, 64, 65, 129, 1000])
def test_grm_kernel_against_the_statement(S):
    from svjg import alnfilter
    _g, _rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    n = 100 if S == 1000 else 150
    rng = np.random.default_rng(S)
    for ploidy in (True, False):
        co, idx, ty, rclass = _grm_case(t, S, n, rng, ploidy)
        want = {}
        for step in ((1, 7, 31, 32, 33, n) if ploidy or S <= 65 else (n, 33)):
            codes, _blocks = _run_blocks(co, idx, ty, rclass, step)
            if ploidy:
                assert {4, 5, 6, 7} <= set(np.unique(codes).tolist())
            for min_maf in (0.0, 0.05, 0.5):
                if min_maf not in want:
                    G, N = grm_statement(codes, min_maf)
                    want[min_maf] = (packed(G), packed(N), G)
                    if S > 2:
                        used = record_table(codes, min_maf)[0]
                        assert not used[2:7].any() and (codes[:, S // 2] > 2).all()
                        assert (G[S // 2] == 0).all()
                        if min_maf == 0.05 and S >= 63:
                            assert not used[7:9].any() and record_table(codes, 0.0)[0][7:9].all()
                g, nn = _device_grm(co, min_maf)
                assert (nn == want[min_maf][1]).all(), step
                assert g.tobytes() == want[min_maf][0].tobytes(), (step, min_maf)
            # the planes are only read: the relatedness counts after the matrix are still those of the codes
            pairs = np.zeros((S * (S - 1) // 2, 5), np.uint32)
            capi.check(capi.lib.svjg_cohort_relatedness(co._h, pairs.ctypes.data if pairs.size else None))
            assert (pairs == pair_counts(codes)).all()
            g, nn = _device_grm(co, 0.0)
            assert g.tobytes() == want[0.0][0].tobytes()
        if S > 2:
            vals, vecs = cohort.pca(want[0.0][2], min(3, S))
            assert (np.abs(vecs[S // 2]) < 1e-12).all()               # the sample with no call
        co.close()


@pytest.mark.gpu
def test_grm_api_refusals_and_the_module():
    from svjg import alnfilter, synth
    _g, rows, edges_text, gfa_text = _synthetic(600, seed=9)
    t = alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0)
    S = 40
    rng = np.random.default_rng(4)
    co = cohort.Cohort(t, S)
    g = np.zeros(S * (S + 1) // 2)
    nn = np.zeros(S * (S + 1) // 2, np.uint32)
    assert capi.lib.svjg_cohort_grm(co._h, 0.01, g.ctypes.data, nn.ctypes.data) == capi.E_ARG     # no qc_begin
    capi.check(capi.lib.svjg_cohort_qc_begin(co._h, 4, 0))
    assert capi.lib.svjg_cohort_grm(co._h, 0.01, g.ctypes.data, nn.ctypes.data) == capi.E_ARG     # no want_pairs
    capi.check(capi.lib.svjg_cohort_qc_begin(co._h, 4, 1))
    for bad in (-0.01, 0.51, float("nan"), float("inf")):
        assert capi.lib.svjg_cohort_grm(co._h, bad, g.ctypes.data, nn.ctypes.data) == capi.E_ARG
    assert capi.lib.svjg_cohort_grm(co._h, 0.01, None, nn.ctypes.data) == capi.E_ARG
    assert capi.lib.svjg_cohort_grm(co._h, 0.01, g.ctypes.data, None) == capi.E_ARG
    capi.check(capi.lib.svjg_cohort_grm(co._h, 0.5, g.ctypes.data, nn.ctypes.data))             # nothing packed yet
    assert not g.any() and not nn.any()
    # genotype_cohort_vcf: the same text and tables with the matrix, which follows the VCF's GT fields
    v = genotype.NativeVcf.from_input(synth.vcf_text(rows).encode())
    for s in range(S):
        co.load_counts(s, _KIND_COUNTS[rng.integers(0, 5, t.num_sv)])
    names = [f"s{k}" for k in range(S)]
    text, n_gt = cohort.genotype_cohort_vcf(t, co, v, names)
    codes = _vcf_codes(text)
    ref = cohort.genotype_cohort_vcf(t, co, v, names, sample_qc=True, relatedness=True)
    for step in (None, 7, 33):
        res = cohort.genotype_cohort_vcf(t, co, v, names, block_records=step, sample_qc=True, relatedness=True,
                                         grm=True, grm_min_maf=0.05)
        assert len(res) == 5 and res[:2] == (text, n_gt)
        assert (res[2] == ref[2]).all() and (res[3] == ref[3]).all()
        G, N = grm_statement(codes, 0.05)
        assert res[4][0].dtype == np.float64 and res[4][1].dtype == np.uint32
        assert res[4][0].tobytes() == G.tobytes() and (res[4][1] == N).all()
    res = cohort.genotype_cohort_vcf(t, co, v, names, grm=True)
    assert res[:4] == (text, n_gt, None, None)
    assert res[4][0].tobytes() == grm_statement(codes, cohort.GRM_MIN_MAF)[0].tobytes()
    with pytest.raises(ValueError, match="grm_min_maf"):
        cohort.genotype_cohort_vcf(t, co, v, names, grm=True, grm_min_maf=0.7)
    co.close()


def _read_f4(path):
    return np.fromfile(path, "<f4")


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
    r0 = _cohort(*common, "-o", p + "_a.vcf", "--sample-qc", p + "_qa.tsv", "--relatedness", p + "_ra.tsv")
    r1 = _cohort(*common, "-o", p + "_b.vcf", "--sample-qc", p + "_qb.tsv", "--relatedness", p + "_rb.tsv",
                 "--grm", p + "_g", "--pca", p + "_p", "--pca-components", "5")
    r2 = _cohort(*common, "-o", p + "_c.vcf", "--pca", p + "_p2", "--pca-components", "8", "--grm-min-maf", "0.2")
    assert r0.returncode == 0 and r1.returncode == 0 and r2.returncode == 0, r1.stderr + r2.stderr
    assert r0.stdout == r1.stdout == r2.stdout
    plain = open(p + "_a.vcf", "rb").read()
    assert open(p + "_b.vcf", "rb").read() == plain and open(p + "_c.vcf", "rb").read() == plain
    assert open(p + "_qa.tsv", "rb").read() == open(p + "_qb.tsv", "rb").read()
    assert open(p + "_ra.tsv", "rb").read() == open(p + "_rb.tsv", "rb").read()
    codes = _vcf_codes(plain.decode())
    assert {0, 1, 2, 3, 4, 5, 7} <= set(np.unique(codes).tolist())
    for prefix, min_maf, k in ((p + "_g", 0.01, None), (p + "_p", 0.01, 5), (p + "_p2", 0.2, 8)):
        G, N = grm_statement(codes, min_maf)
        assert record_table(codes, min_maf)[0].any()
        if k is None:
            il = np.tril_indices(len(names))
            assert (_read_f4(prefix + ".grm.bin") == G[il].astype(np.float32)).all()
            assert (_read_f4(prefix + ".grm.N.bin") == N[il].astype(np.float32)).all()
            assert open(prefix + ".grm.id").read() == "".join(f"{nm}\t{nm}\n" for nm in names)
            assert G[3, 7] == G[3, 3] and N[3, 7] == N[3, 3] > 0                   # the same GAF twice
            assert (G[4] == 0).all() and (N[4] == 0).all()                          # the empty sample
            continue
        assert not os.path.exists(prefix + ".grm.bin")
        vals, vecs = cohort.pca(G, k)
        vo, eo = io.BytesIO(), io.BytesIO()
        cohort.write_pca(vo, eo, names, vals, vecs)
        assert open(prefix + ".eigenvec", "rb").read() == vo.getvalue()
        assert open(prefix + ".eigenval", "rb").read() == eo.getvalue()
    # an output that cannot be written: none of the outputs is left behind
    r = _cohort(*common, "-o", p + "_d.vcf", "--grm", p + "_dg", "--pca", p + "_none/p", "--pca-components", "2")
    assert r.returncode == 1 and "No such file" in r.stderr, r.stderr
    assert not [f for f in os.listdir(tmp_path) if "_d" in f and not f.endswith(".gaf") or f.startswith(".")]


@pytest.mark.gpu
def test_need_k_cells_through_the_command_line(tmp_path):
    """72 copies of s2 take cells beyond the log10 C(n, k) table (patched on the host): the matrix still follows the
    VCF's GT fields."""
    from conftest import read_golden
    p = _s2_cohort(tmp_path)[0]
    open(p + "_x72.gaf", "w").write(read_golden("s2.gaf.gz") * 72)
    common = ["-p", p, "-g", p + ".gfa", "-v", p + ".vcf", "-a", p + "_x72.gaf", p + "_whole.gaf", p + "_x72.gaf",
              p + "_half1.gaf", "--names", "x72,one,again,half"]
    r0 = _cohort(*common, "-o", p + "_a.vcf")
    r1 = _cohort(*common, "-o", p + "_b.vcf", "--grm", p + "_g", "--grm-min-maf", "0")
    assert r0.returncode == 0 and r1.returncode == 0, r1.stderr
    plain = open(p + "_a.vcf", "rb").read()
    assert open(p + "_b.vcf", "rb").read() == plain
    G, N = grm_statement(_vcf_codes(plain.decode()), 0.0)
    il = np.tril_indices(4)
    assert (_read_f4(p + "_g.grm.bin") == G[il].astype(np.float32)).all()
    assert (_read_f4(p + "_g.grm.N.bin") == N[il].astype(np.float32)).all()
