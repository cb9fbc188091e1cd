"""The cohort kernels at the shapes real cohorts run them at (DESIGN.md §8a): many plane words and K slabs, the
product's own block steps, every instance of the posterior kernel, the largest sample grid, the pack kernel's capped
grid, the ploidy table at its limits and the exact tests at a large N.

The statements of the contract live in test_cohort_qc, test_cohort_grm, test_cohort_posteriors, test_cohort_ploidy and
test_cohort_info.  They are too slow at these shapes, so this file has fast references of the same semantics, and a
CPU test shows that they equal the statements, bit for bit, on small random codes:

* pair counts: float64 products of the 0/1 planes (every partial sum is an integer below 2^53, so exact whatever the
  order), or boolean sums over the codes for a chosen set of pairs;
* histogram: np.bincount per sample; planes: np.packbits(bitorder="little") per block, each block starting a word;
* relationship matrix on a chosen set of pairs: the products u[r, g_i] * v[r, g_j] and their sum in ascending record
  order, by np.multiply and np.add.accumulate along the records (a sequential scan: no pairwise sums, no BLAS, no
  FMA).  The scan starts at the first term instead of +0.0; adding +0.0 at the end gives the same bits (the two sums
  differ at most by the sign of a zero that no later term touches).

The device cases are marked gpu.  Host memory: the 16 384-sample case holds about 2.7 GB of pair counts, then 1.6 GB
of G and N; the pack kernel's case about 1.1 GB of pinned block arrays.
"""
import functools
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from svjg import capi, cohort, genotype
from test_cohort import _synthetic
from test_cohort_grm import _random_codes as _grm_codes
from test_cohort_grm import grm_statement, record_table
from test_cohort_info import _GT_COUNTS, hwe_exchet
from test_cohort_ploidy import SVTYPE_NAME, _set_ploidy, _stats6, haploid_call
from test_cohort_posteriors import _kernel_case, _patch, _run_posteriors, _same_bits, cell_kinds, posteriors
from test_cohort_qc import _KIND_COUNTS, _TYPES, _vcf_codes, pair_counts_brute, planes, sample_counts
from test_cohort_qc import _random_codes as _qc_codes

TILE = 64                                    # PAIR_T and GRM_T of genotype.cu
_WORKERS = max(1, min(8, os.cpu_count() or 1))


# ---------------------------------------------------------------------------------------------------------------
# fast references
# ---------------------------------------------------------------------------------------------------------------
def _chunked(fn, n_items, per):
    """fn(lo, hi) over [0, n_items) in pieces of ``per``, on a few threads (numpy releases the GIL in its loops)."""
    spans = [(lo, min(n_items, lo + per)) for lo in range(0, n_items, per)]
    with ThreadPoolExecutor(_WORKERS) as ex:
        list(ex.map(lambda s: fn(*s), spans))


def pair_counts_fast(codes):
    """pair_counts_brute of every pair i < j, by float64 matrix products of the 0/1 planes."""
    S = codes.shape[1]
    C, H, A, R = (x.astype(np.float64) for x in (codes <= 2, codes == 1, codes == 2, codes == 0))
    i, j = np.triu_indices(S, 1)
    m = [C.T @ C, H.T @ C, C.T @ H, H.T @ H, A.T @ R + R.T @ A]
    return np.stack([x[i, j] for x in m], axis=1).astype(np.uint32).reshape(-1, 5)


def pair_counts_at(codes, pi, pj):
    """pair_counts_brute of the pairs (pi[k], pj[k]), pi < pj, by boolean sums over the codes."""
    n = codes.shape[0]
    C, H, A, R = codes <= 2, codes == 1, codes == 2, codes == 0
    out = np.zeros((len(pi), 5), np.uint32)

    def work(lo, hi):
        a, b = pi[lo:hi], pj[lo:hi]
        Ci, Cj, Hi, Hj = C[:, a], C[:, b], H[:, a], H[:, b]
        out[lo:hi, 0] = (Ci & Cj).sum(0)
        out[lo:hi, 1] = (Hi & Cj).sum(0)
        out[lo:hi, 2] = (Ci & Hj).sum(0)
        out[lo:hi, 3] = (Hi & Hj).sum(0)
        out[lo:hi, 4] = ((A[:, a] & R[:, b]) | (R[:, a] & A[:, b])).sum(0)

    _chunked(work, len(pi), max(1, (1 << 23) // max(n, 1)))
    return out


def sample_counts_fast(codes, ty):
    """sample_counts by np.bincount: row ALL, then the records of each SVTYPE code 0-3."""
    n, S = codes.shape
    t = np.asarray(ty) & 0x3F
    off = 8 * np.arange(S, dtype=np.int64)
    h = np.zeros((S, 5, 8), np.int64)
    for row, sel in enumerate([slice(None)] + [t == k for k in range(4)]):
        h[:, row] = np.bincount((codes[sel].astype(np.int64) + off).ravel(), minlength=8 * S).reshape(S, 8)
    return h.astype(np.uint32)


def planes_fast(codes, blocks):
    """planes by np.packbits: per block, bit r of word w is record 32 w + r of the block."""
    n, S = codes.shape
    assert sum(blocks) == n
    out, lo = [], 0
    for m in blocks:
        w = -(-m // 32)
        sub = codes[lo:lo + m]
        lo += m
        per = []
        for cond in (sub <= 2, sub == 1, sub == 2):
            bits = np.zeros((S, 32 * w), bool)
            bits[:, :m] = cond.T
            per.append(np.ascontiguousarray(np.packbits(bits, axis=1, bitorder="little")).view("<u4"))
        out.append(np.stack(per))
    if not out:
        return np.zeros((3, S, 0), np.uint32)
    return np.concatenate(out, axis=2).astype(np.uint32)


def grm_at(codes, min_maf, pi, pj):
    """(G [P] float64, N [P] uint32) of grm_statement at the pairs (pi[k], pj[k]), pi <= pj, bit for bit."""
    codes = np.asarray(codes)
    used, u, v = record_table(codes, min_maf)
    rows = np.flatnonzero(used)
    c = codes[rows]
    called = c <= 2
    g = np.where(called, c, 0).astype(np.int64)
    # sample-major [S][records]: a pair's terms are one contiguous row, scanned in record order
    U = np.ascontiguousarray(np.where(called, np.take_along_axis(u[rows], g, axis=1), 0.0).T)
    V = np.ascontiguousarray(np.where(called, np.take_along_axis(v[rows], g, axis=1), 0.0).T)
    called = np.ascontiguousarray(called.T)
    G = np.zeros(len(pi))
    N = np.zeros(len(pi), np.uint32)

    def work(lo, hi):
        a, b = pi[lo:hi], pj[lo:hi]
        nn = N[lo:hi] = (called[a] & called[b]).sum(1)
        if len(rows):
            T = np.multiply(U[a], V[b])
            np.add.accumulate(T, axis=1, out=T)
            G[lo:hi] = np.divide(T[:, -1] + 0.0, nn, out=np.zeros(hi - lo), where=nn > 0)

    _chunked(work, len(pi), max(1, (1 << 22) // max(len(rows), 1)))
    return G, N


def _touching(S, samples):
    """The pairs i <= j with i or j in ``samples``, as (i, j) arrays."""
    x = np.arange(S, dtype=np.int64)
    ii = np.concatenate([np.minimum(k, x) for k in samples]) if len(samples) else np.zeros(0, np.int64)
    jj = np.concatenate([np.maximum(k, x) for k in samples]) if len(samples) else np.zeros(0, np.int64)
    return ii, jj


def pair_set(S, rng, touch=None, n_random=20000, diagonal_tiles=True):
    """Pairs i <= j to check, sorted and unique: every pair when S <= 2 TILE; otherwise every pair of the first and last
    tile rows and columns (or of the samples ``touch``), of every diagonal tile, and about ``n_random`` random pairs."""
    if S <= 2 * TILE:
        i, j = np.triu_indices(S)
        return i.astype(np.int64), j.astype(np.int64)
    if touch is None:
        touch = np.concatenate([np.arange(TILE), np.arange((S - 1) // TILE * TILE, S)])
    parts = [_touching(S, np.asarray(touch, np.int64))]
    if diagonal_tiles:
        for lo in range(0, S, TILE):
            a, b = np.triu_indices(min(TILE, S - lo))
            parts.append((a + lo, b + lo))
    r = rng.integers(0, S, (2, n_random))
    parts.append((r.min(0), r.max(0)))
    key = np.unique(np.concatenate([a * S + b for a, b in parts]))
    return key // S, key % S


def pair_index(S, i, j):
    """Index of pair i < j in svjg_cohort_relatedness's output."""
    i, j, S = (np.asarray(x, np.int64) for x in (i, j, S))
    return i * (2 * S - i - 1) // 2 + (j - i - 1)


def grm_index(S, i, j):
    """Index of pair i <= j in svjg_cohort_grm's packed triangle."""
    i, j, S = (np.asarray(x, np.int64) for x in (i, j, S))
    return i * (2 * S - i + 1) // 2 + (j - i)


def _bits(x):
    return np.ascontiguousarray(x, np.float64).view(np.uint64)


def _words(blocks):
    return sum(-(-m // 32) for m in blocks)


def _blocks(n, step):
    return [min(step, n - lo) for lo in range(0, n, step)]


# ---------------------------------------------------------------------------------------------------------------
# CPU: the fast references are the statements
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2, 40, 65])
@pytest.mark.parametrize("n", [1, 300])
def test_fast_references_equal_the_statements(S, n):
    rng = np.random.default_rng(7000 + 100 * S + n)
    for make in (_qc_codes, _grm_codes):
        codes = make(rng, n, S)
        ty = rng.choice(np.array([0, 1, 2, 3, 0x80, 0x83, 9, 255], np.uint8), n)
        want = pair_counts_brute(codes)
        assert (pair_counts_fast(codes) == want).all()
        i, j = np.triu_indices(S, 1)
        assert (pair_counts_at(codes, i, j) == want).all()
        if S > 2:                                                  # a sampled subset, in another order
            k = rng.permutation(len(i))[:len(i) // 3]
            assert (pair_counts_at(codes, i[k], j[k]) == want[pair_index(S, i[k], j[k])]).all()
        assert (sample_counts_fast(codes, ty) == sample_counts(codes, ty)).all()
        for blocks in ([n], _blocks(n, 7), _blocks(n, 33), _blocks(n, 97), [1] * min(n, 40) + _blocks(n - min(n, 40), 61)):
            assert (planes_fast(codes, blocks) == planes(codes, blocks)).all()
        for min_maf in (0.0, 0.05, 0.5):
            G, N = grm_statement(codes, min_maf)
            i, j = np.triu_indices(S)
            g, nn = grm_at(codes, min_maf, i, j)
            assert (_bits(g) == _bits(G[i, j])).all() and (nn == N[i, j]).all()
            if min_maf == 0.0 and n > 1 and S > 1:
                assert (G[i, j] != 0).any()
            if S > 2:
                k = rng.permutation(len(i))[:len(i) // 4]
                g, nn = grm_at(codes, min_maf, i[k], j[k])
                assert (_bits(g) == _bits(G[i[k], j[k]])).all() and (nn == N[i[k], j[k]]).all()


def test_sums_that_cancel_keep_the_sign_of_the_statement():
    """Terms that are all -0.0, or that cancel exactly: the scan gives +0.0 as the statement does."""
    codes = np.array([[0, 2], [2, 0], [1, 1], [0, 0]], np.uint8)      # u_0 v_2 and u_2 v_0 cancel for pair (0, 1)
    G, N = grm_statement(codes, 0.0)
    g, nn = grm_at(codes, 0.0, np.array([0, 0, 1]), np.array([0, 1, 1]))
    assert (_bits(g) == _bits(G[[0, 0, 1], [0, 1, 1]])).all() and (nn == N[[0, 0, 1], [0, 1, 1]]).all()
    codes = np.array([[3, 0], [0, 1], [1, 0]], np.uint8)
    G, N = grm_statement(codes, 0.0)
    g, nn = grm_at(codes, 0.0, np.array([0, 0, 1]), np.array([0, 1, 1]))
    assert (_bits(g) == _bits(G[[0, 0, 1], [0, 1, 1]])).all() and (nn == N[[0, 0, 1], [0, 1, 1]]).all()


def test_pair_sets_and_indices():
    rng = np.random.default_rng(3)
    for S in (1, 2, 128):
        i, j = pair_set(S, rng)
        assert len(i) == S * (S + 1) // 2
    S = 1000
    i, j = pair_set(S, rng)
    assert (i <= j).all() and len(np.unique(i * S + j)) == len(i)
    first = (i < TILE) | (j >= 960)
    assert first.sum() == sum(S - k for k in range(TILE)) + sum(k + 1 for k in range(960, S)) - TILE * (S - 960)
    assert ((j // TILE == i // TILE) & ~first).sum() == sum(TILE * (TILE + 1) // 2 for _ in range(1, 15))
    assert pair_index(S, 0, 1) == 0 and pair_index(S, S - 2, S - 1) == S * (S - 1) // 2 - 1
    assert grm_index(S, 0, 0) == 0 and grm_index(S, S - 1, S - 1) == S * (S + 1) // 2 - 1
    ii, jj = np.triu_indices(7, 1)
    assert (pair_index(7, ii, jj) == np.arange(len(ii))).all()
    ii, jj = np.triu_indices(7)
    assert (grm_index(7, ii, jj) == np.arange(len(ii))).all()


# ---------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _tables(n_sv):
    from svjg import alnfilter
    _g, rows, edges_text, gfa_text = _synthetic(n_sv, seed=9)
    return alnfilter.Tables.from_memory(edges_text, gfa_text).to_device(0), rows


def _run(co, pick, ty, step):
    """svjg_cohort_qc_begin with want_pairs, then the block loop of genotype_cohort_vcf with svjg_cohort_qc_add after
    each block.  idx cycles over the catalogue, and before each block every sample's counters are drawn afresh from
    ``pick`` ([n][S] rows of _KIND_COUNTS) for the SVs of the block: while a block holds no SV twice, record r gets the
    cells of pick[r] whatever the step.  Returns (codes [n][S], block sizes)."""
    S, n = co.n_samples, len(pick)
    idx = (np.arange(n) % co.num_sv).astype(np.uint32)
    blocks = _blocks(n, step)
    capi.check(capi.lib.svjg_cohort_qc_begin(co._h, _words(blocks), 1))
    blk = cohort._Block(min(step, n) * S)
    codes = np.empty((n, S), np.uint8)
    c = np.zeros((co.num_sv, 2), np.uint32)
    for lo in range(0, n, step):
        hi = min(n, lo + step)
        for s in range(S):
            c[idx[lo:hi]] = _KIND_COUNTS[pick[lo:hi, s]]
            co.load_counts(s, c)
        gt = cohort._genotype_block(co, idx[lo:hi], ty[lo:hi], 3, genotype.ERR, blk)[0]
        capi.check(capi.lib.svjg_cohort_qc_add(co._h, hi - lo))
        codes[lo:hi] = gt.reshape(hi - lo, S)
    return codes, blocks


def _hist_and_planes(co, n_words):
    S = co.n_samples
    h = np.zeros((S, 5, 8), np.uint32)
    capi.check(capi.lib.svjg_cohort_qc_sample_counts(co._h, h.ctypes.data))
    p = np.zeros((3, S, n_words), np.uint32)
    capi.check(capi.lib.svjg_cohort_qc_planes(co._h, p.ctypes.data))
    return h, p


def _device_pairs(co):
    S = co.n_samples
    pairs = np.zeros((S * (S - 1) // 2, 5), np.uint32)
    capi.check(capi.lib.svjg_cohort_relatedness(co._h, pairs.ctypes.data if pairs.size else None))
    return pairs


def _device_grm(co, min_maf):
    S = co.n_samples
    g = np.full(S * (S + 1) // 2, np.nan)
    nn = np.full(S * (S + 1) // 2, 0xFFFFFFFF, np.uint32)
    capi.check(capi.lib.svjg_cohort_grm(co._h, min_maf, g.ctypes.data, nn.ctypes.data))
    return g, nn


class _Refs:
    """References of one codes array, computed once: the runs whose blocks hold no SV twice share their codes."""

    def __init__(self, codes, ty, rng, mafs):
        S = codes.shape[1]
        self.hist = sample_counts_fast(codes, ty)
        self.pairs = pair_counts_fast(codes)
        self.pi, self.pj = pair_set(S, rng)
        self.gp = grm_index(S, self.pi, self.pj)
        self.grm = {m: grm_at(codes, m, self.pi, self.pj) for m in mafs}


def _idle_words(used, blocks):
    """Words (in the device's layout) with no used record that have a used word before and after them."""
    u, lo = [], 0
    for m in blocks:
        b = np.zeros(-(-m // 32) * 32, bool)
        b[:m] = used[lo:lo + m]
        lo += m
        u.append(b.reshape(-1, 32).any(1))
    u = np.concatenate(u)
    hit = np.flatnonzero(u)
    return int((~u[hit[0]:hit[-1]]).sum()) if hit.size else 0


def _scale_pick(rng, n, S):
    """Cell kinds of n records: random, then 200 monomorphic records (0/0, then 1/1: whole words of records that no
    relationship sum uses) and 600 records missing everywhere (a whole block of steps 517 and 33)."""
    pick = rng.integers(0, 5, (n, S))
    pick[3000:3100] = 0
    pick[3100:3200] = 2
    pick[12400:13000] = 4
    ty = rng.choice(_TYPES, n)
    ty[3000:3200] = 0                                                 # DEL: the monomorphic records are genotyped
    return pick, ty


@pytest.mark.gpu
@pytest.mark.parametrize("S", [64, 65, 1000])
def test_qc_relatedness_and_grm_over_many_words_and_slabs(S):
    """About 20 000 records: 626 plane words, 40 K slabs of the pair kernel, y-blocks of the pack kernel that add to one
    sample's histogram, hundreds of relationship words with whole unused words between used ones."""
    t, _rows = _tables(8000)
    n = 20011
    assert t.num_sv > 7895
    rng = np.random.default_rng(S)
    pick, ty = _scale_pick(rng, n, S)
    co = cohort.Cohort(t, S)
    # at S = 1 000 the loads of step 33 (606 blocks x S) and a second relationship reference (step n) cost minutes
    steps = (7895, 4549, 517, 33, n) if S < 1000 else (7895, 4549, 517)
    mafs = (0.0, 0.05, 0.5) if S < 1000 else (0.05, 0.5)
    refs = {}
    for step in steps:
        codes, blocks = _run(co, pick, ty, step)
        key = codes.tobytes()
        if key not in refs:
            refs[key] = _Refs(codes, ty, rng, mafs)
        ref = refs[key]
        if step <= t.num_sv:                                          # the hand-made runs are there
            assert (codes[3000:3100] == 0).all() and (codes[3100:3200] == 2).all() and (codes[12400:13000] == 3).all()
            assert _idle_words(record_table(codes, 0.0)[0], blocks) >= 6
            if step in (517, 33):
                assert any(lo >= 12400 and lo + m <= 13000 for lo, m in zip(np.cumsum([0] + blocks), blocks))
        h, p = _hist_and_planes(co, _words(blocks))
        assert (h == ref.hist).all(), step
        assert (p == planes_fast(codes, blocks)).all(), step
        assert (_device_pairs(co) == ref.pairs).all(), step
        for min_maf in mafs:
            g, nn = _device_grm(co, min_maf)
            G, N = ref.grm[min_maf]
            assert (nn[ref.gp] == N).all(), (step, min_maf)
            assert (_bits(g[ref.gp]) == _bits(G)).all(), (step, min_maf)
            if S <= 2 * TILE:
                assert len(ref.gp) == len(g)
        # the planes are only read: the relatedness counts after the matrix are still those of the codes
        assert (_device_pairs(co) == ref.pairs).all(), step
    assert len(refs) == (2 if n in steps else 1)                      # the shared codes, and those of step n
    co.close()


@pytest.mark.gpu
def test_slab_edges_inside_and_between_blocks():
    """S = 65 with 15, 16, 17, 32 and 33 words in all: the 16-word K slab ends inside a block or between two."""
    t, _rows = _tables(8000)
    S = 65
    rng = np.random.default_rng(65)
    co = cohort.Cohort(t, S)
    seen = set()
    for W in (15, 16, 17, 32, 33):
        for step in (33, 70, 97, 300):
            n = next(m for m in range(1, 40 * W) if _words(_blocks(m, step)) == W)
            pick = rng.integers(0, 5, (n, S))
            ty = rng.choice(_TYPES, n)
            codes, blocks = _run(co, pick, ty, step)
            assert _words(blocks) == W
            seen.add((W, len(blocks) > 1))
            h, p = _hist_and_planes(co, W)
            assert (h == sample_counts_fast(codes, ty)).all(), (W, step)
            assert (p == planes_fast(codes, blocks)).all(), (W, step)
            assert (_device_pairs(co) == pair_counts_fast(codes)).all(), (W, step)
            i, j = np.triu_indices(S)
            for min_maf in (0.0, 0.05):
                g, nn = _device_grm(co, min_maf)
                G, N = grm_at(codes, min_maf, i, j)
                assert (nn == N).all() and (_bits(g) == _bits(G)).all(), (W, step, min_maf)
    assert all((W, True) in seen for W in (15, 16, 17, 32, 33))
    co.close()


@pytest.mark.gpu
def test_largest_sample_grid():
    """S = SVJG_QC_MAX_PAIR_SAMPLES = 16 384 at the product's step 481 (BLOCK_BYTES // (34 S)): 256 tiles per side,
    32 896 CTAs, 134 M pairs, 3 blocks, 48 words, 3 slabs; one sample more is refused."""
    t, rows = _tables(8000)
    S = capi.QC_MAX_PAIR_SAMPLES
    step = cohort.BLOCK_BYTES // (cohort.CELL_BYTES * S)
    assert S == 16384 and step == 481
    n = 3 * step
    rng = np.random.default_rng(16384)
    pick = rng.integers(0, 5, (n, S))
    ty = rng.choice(_TYPES, n)
    co = cohort.Cohort(t, S)
    codes, blocks = _run(co, pick, ty, step)
    assert _words(blocks) == 48
    h, p = _hist_and_planes(co, 48)
    assert (h == sample_counts_fast(codes, ty)).all()
    assert (p == planes_fast(codes, blocks)).all()
    edge = [0, 63, 64, 8191, 16319, 16320, 16383]
    pi, pj = pair_set(S, rng, touch=edge, n_random=100000, diagonal_tiles=False)
    off = pi < pj
    want_pairs = pair_counts_at(codes, pi[off], pj[off])
    pairs = _device_pairs(co)
    assert (pairs[pair_index(S, pi[off], pj[off])] == want_pairs).all()
    assert (pairs[pair_index(S, S - 2, S - 1)] == pair_counts_at(codes, np.array([S - 2]), np.array([S - 1]))).all()
    del pairs
    G, N = grm_at(codes, 0.01, pi, pj)
    assert (G != 0).sum() > len(G) // 2
    g, nn = _device_grm(co, 0.01)
    k = grm_index(S, pi, pj)
    assert (nn[k] == N).all() and (_bits(g[k]) == _bits(G)).all()
    del g, nn
    co.close()
    # one sample more: refused by the C API and by the module, before any work
    from svjg import synth
    big = cohort.Cohort(t, S + 1)
    try:
        assert capi.lib.svjg_cohort_qc_begin(big._h, 1, 1) == capi.E_ARG
        assert "SVJG_QC_MAX_PAIR_SAMPLES" in capi.lib.svjg_last_error().decode()
        capi.check(capi.lib.svjg_cohort_qc_begin(big._h, 1, 0))          # the sample table alone is fine
        vcf = synth.vcf_text(rows).encode()
        names = [f"s{k}" for k in range(S + 1)]
        with pytest.raises(ValueError, match="at most 16384"):
            cohort.genotype_cohort_vcf(t, big, vcf, names, relatedness=True)
        with pytest.raises(ValueError, match="at most 16384"):
            cohort.genotype_cohort_vcf(t, big, vcf, names, grm=True)
    finally:
        big.close()


@pytest.mark.gpu
def test_pack_kernel_beyond_its_grid_cap():
    """S = 2 and one block of 65 535 * 8 * 32 + 40 records: gridDim.y of the pack kernel is capped at 65 535 and its y
    loop runs a second lap, which ends in a partial word."""
    t, _rows = _tables(8000)
    S, n = 2, 65535 * 8 * 32 + 40
    rng = np.random.default_rng(2)
    co = cohort.Cohort(t, S)
    for s in range(S):
        co.load_counts(s, _KIND_COUNTS[rng.integers(0, 4, t.num_sv)])
    idx = (np.arange(n) % t.num_sv).astype(np.uint32)
    ty = rng.choice(_TYPES, n)
    n_words = -(-n // 32)
    assert -(-n_words // 8) > 65535 and n % 32 == 8
    capi.check(capi.lib.svjg_cohort_qc_begin(co._h, n_words, 1))
    blk = cohort._Block(n * S)
    gt = cohort._genotype_block(co, idx, ty, 3, genotype.ERR, blk)[0]
    capi.check(capi.lib.svjg_cohort_qc_add(co._h, n))
    codes = gt.reshape(n, S).copy()
    del blk, gt
    assert {0, 1, 2, 3} <= set(np.unique(codes).tolist())
    h, p = _hist_and_planes(co, n_words)
    assert (h == sample_counts_fast(codes, ty)).all()
    assert (p == planes_fast(codes, [n])).all()
    assert (p[:, :, -1] >> 8 == 0).all() and p[0, :, -1].any()        # the last word holds 8 records
    assert (_device_pairs(co) == pair_counts_at(codes, np.array([0]), np.array([1]))).all()
    pi, pj = np.array([0, 0, 1]), np.array([0, 1, 1])
    for min_maf in (0.0, 0.05):
        G, N = grm_at(codes, min_maf, pi, pj)
        assert (N > 0).all()
        g, nn = _device_grm(co, min_maf)
        assert (nn == N).all() and (_bits(g) == _bits(G)).all(), min_maf
    co.close()


@pytest.mark.gpu
@pytest.mark.parametrize("S,n", [(65, 300), (100, 300), (128, 300), (129, 2000), (1000, 2000)])
def test_posterior_instances(S, n):
    """cohort_posterior_kernel<4> (S = 65 to 128: a lane's fourth register cell is used from S = 97 on) and <0> over
    many warps and blocks, both ploidy modes, with the record whose EM runs to SVJG_POST_MAX_ITERS; bit for bit
    against the statement."""
    t, _rows = _tables(8000)
    rng = np.random.default_rng(S)
    for ploidy in (False, True):
        co, idx, ty, rclass = _kernel_case(t, S, n, rng, ploidy)
        blk = cohort._Block(n * S, post_records=n)
        gt, fl, _ad, pl = (a.copy() for a in cohort._genotype_block(co, idx, ty, 3, genotype.ERR, blk, rclass))
        need = blk.need.copy()
        assert need.size > 0
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
        assert (iters == capi.POST_MAX_ITERS).any() and ((iters > 0) & (iters < capi.POST_MAX_ITERS)).any()
        kinds = cell_kinds(gt, fl).reshape(n, S)
        assert (kinds[:, S - 1] > 0).any()                            # the last lane's last cell contributes
        if S > 96:
            assert (kinds[:, 96:] > 0).sum() > n                      # and so do the fourth cells of the lanes
        if ploidy:
            assert (kinds == 1).any() and (gt == capi.GT_NO_CALL).any()
        co.close()


@pytest.mark.gpu
def test_ploidy_table_at_its_limits():
    """255 classes x 64 sexes (SVJG_PLOIDY_MAX_CLASSES x SVJG_PLOIDY_MAX_SEXES), a random 0/1/2 table, every sex and
    every class in use: each cell against the statement of its ploidy, and the ploidy site statistics."""
    t, _rows = _tables(8000)
    S, n = 200, 600
    n_classes, n_sexes = capi.PLOIDY_MAX_CLASSES, capi.PLOIDY_MAX_SEXES
    rng = np.random.default_rng(255)
    co = cohort.Cohort(t, S)
    counts = []
    for s in range(S):
        c = rng.integers(0, 601, (t.num_sv, 2)).astype(np.uint32)
        c[rng.random(t.num_sv) < 0.2] = 0
        c[rng.random((t.num_sv, 2)) < 0.5] %= 40
        co.load_counts(s, c)
        counts.append(c)
    idx = rng.integers(0, t.num_sv, n).astype(np.uint32)
    idx[rng.random(n) < 0.05] = capi.NO_SV
    ty = rng.choice([0, 1, 2, 3, 255, 0x80, 0x81], size=n).astype(np.uint8)
    table = rng.integers(0, 3, (n_classes, n_sexes)).astype(np.uint8)
    sex = np.concatenate([np.arange(n_sexes), rng.integers(0, n_sexes, S - n_sexes)]).astype(np.uint8)
    rclass = np.concatenate([np.arange(n_classes), rng.integers(0, n_classes, n - n_classes)]).astype(np.uint8)
    rng.shuffle(sex)
    rng.shuffle(rclass)
    _set_ploidy(co, table, sex)
    blk = cohort._Block(n * S, n, ploidy=True)
    gt, fl, ad, pl = (a.copy() for a in cohort._genotype_block(co, idx, ty, 3, genotype.ERR, blk, rclass))
    gcount, hwe, exc = (a.copy() for a in cohort._site_stats(co, n, blk, ploidy=True))
    ploidy = table[rclass][:, sex].reshape(-1)                                   # [n * S], record-major
    n_hap = 0
    for s in range(S):
        w_gt, w_fl, w_ad, w_pl = genotype.genotype_host(counts[s], idx, ty, 3, genotype.ERR)
        p = ploidy[s::S]
        assert (fl[s::S] == w_fl).all() and (ad[s::S] == w_ad).all(), s
        dip, hap, zero = p == 2, p == 1, p == 0
        assert (gt[s::S][dip] == w_gt[dip]).all() and (pl[s::S][dip] == w_pl[dip]).all(), s
        assert (pl[s::S][hap][:, [0, 2]] == w_pl[hap][:, [0, 2]]).all(), s
        assert (gt[s::S][zero] == capi.GT_NO_CALL).all(), s
        assert (gt[s::S][hap & ((w_fl & capi.GT_GENOTYPED) == 0)] == capi.GT_HAP_MISSING).all(), s
        for i in np.nonzero(hap & ((w_fl & capi.GT_GENOTYPED) != 0))[0]:
            n0, n1 = (int(x) for x in counts[s][idx[i]])
            want, pl0, pl2 = haploid_call(n0, n1, SVTYPE_NAME[int(ty[i]) & 0x3F], 3, genotype.ERR)
            assert "01."[gt[i * S + s] - capi.GT_HAP_REF] == want, (i, s, n0, n1)
            assert [str(pl[i * S + s, 0]), str(pl[i * S + s, 2])] == [pl0, pl2]
            n_hap += 1
    assert n_hap > 10000 and (np.bincount(gt, minlength=8)[4:8] > 100).all()
    w = _stats6(gt, fl, S)
    assert (gcount == w[0]).all()
    assert (_bits(hwe) == _bits(w[1])).all() and (_bits(exc) == _bits(w[2])).all()
    co.close()


@pytest.mark.gpu
def test_product_block_loop(monkeypatch):
    """genotype_cohort_vcf with its own block step (from BLOCK_BYTES: odd, not a multiple of 32) and every switch on:
    the text of one block, and tables that follow the VCF's GT fields."""
    from svjg import synth
    t, rows = _tables(3400)
    v = genotype.NativeVcf.from_input(synth.vcf_text(rows).encode())
    S, n = 150, v.n
    cell_bytes = cohort.CELL_BYTES + cohort.POST_CELL_BYTES
    monkeypatch.setattr(cohort, "BLOCK_BYTES", cell_bytes * S * 1001 + cell_bytes * S // 2)
    step = cohort.BLOCK_BYTES // (cell_bytes * S)
    assert step == 1001 and 3000 < n and -(-n // step) >= 3
    rng = np.random.default_rng(150)
    co = cohort.Cohort(t, S)
    for s in range(S):
        c = _KIND_COUNTS[rng.integers(0, 5, t.num_sv)].copy()
        c[1::9] = [300, 280]                                          # beyond the log10 C(n, k) table: NEED_K
        co.load_counts(s, c)
    names = [f"s{k}" for k in range(S)]
    begun = []
    begin = capi.lib.svjg_cohort_qc_begin

    def qc_begin(h, n_words, want_pairs):
        begun.append((n_words, want_pairs))
        return begin(h, n_words, want_pairs)

    monkeypatch.setattr(capi.lib, "svjg_cohort_qc_begin", qc_begin)
    kw = dict(info_tags=cohort.INFO_TAGS, posteriors=True, sample_qc=True, relatedness=True, grm=True)
    res = cohort.genotype_cohort_vcf(t, co, v, names, **kw)
    one = cohort.genotype_cohort_vcf(t, co, v, names, block_records=n, **kw)
    assert begun == [(_words(_blocks(n, step)), 1), (-(-n // 32), 1)]
    assert res[0] == one[0] and res[1] == one[1]
    assert (res[2] == one[2]).all() and (res[3] == one[3]).all()
    assert _bits(res[4][0]).tobytes() == _bits(one[4][0]).tobytes() and (res[4][1] == one[4][1]).all()
    codes = _vcf_codes(res[0])
    assert codes.shape == (n, S) and {0, 1, 2, 3} <= set(np.unique(codes).tolist())
    assert (res[2] == sample_counts_fast(codes, v.svtype)).all()
    assert (res[3] == pair_counts_fast(codes)).all()
    i, j = np.triu_indices(S)
    G, N = grm_at(codes, cohort.GRM_MIN_MAF, i, j)
    assert (_bits(res[4][0][i, j]) == _bits(G)).all() and (res[4][1][i, j] == N).all()
    assert (_bits(res[4][0][j, i]) == _bits(G)).all()
    co.close()


@pytest.mark.gpu
def test_exact_tests_at_large_n():
    """svjg_cohort_site_stats with S = 50 000: records whose rare-allele count runs from 1 to S, with het, hom and
    missing mixes; HWE and ExcHet bit for bit against the streaming statement."""
    t, _rows = _tables(600)
    S = 50000
    specs = [(1, 0, 0), (2, 0, 0), (0, 1, 0), (3, 0, 5), (7, 0, 0), (50, 0, 0), (10, 20, 0), (333, 0, 0),
             (1000, 0, 100), (0, 500, 0), (4999, 0, 0), (12345, 0, 2000), (3000, 4000, 0), (25000, 0, 0),
             (20000, 2500, 0), (0, 12500, 0), (30000, 0, 0), (37000, 0, 1000), (49999, 0, 0), (50000, 0, 0),
             (0, 25000, 0), (1, 24999, 0), (2, 0, 49998), (25000, 12500, 0)]       # (het, hom-alt, missing)
    n = len(specs)
    rng = np.random.default_rng(50000)
    want_g = np.zeros((n, S), np.int64)
    for r, (h, a, m) in enumerate(specs):
        row = np.array([1] * h + [2] * a + [3] * m + [0] * (S - h - a - m))
        want_g[r] = rng.permutation(row)
    co = cohort.Cohort(t, S)
    for s in range(S):
        c = np.zeros((t.num_sv, 2), np.uint32)
        c[:n] = _GT_COUNTS[want_g[:, s]]
        co.load_counts(s, c)
    idx = np.arange(n, dtype=np.uint32)
    ty = np.full(n, 2, np.uint8)                                      # INV: no halving
    blk = cohort._Block(n * S, n)
    gt, fl, _ad, _pl = cohort._genotype_block(co, idx, ty, 3, genotype.ERR, blk)
    gcount, hwe, exc = (a.copy() for a in cohort._site_stats(co, n, blk))
    want = np.stack([(want_g == g).sum(1) for g in range(4)], axis=1)
    assert (gcount == want).all()
    rare = 2 * np.minimum(want[:, 0], want[:, 2]) + want[:, 1]
    assert rare.min() == 1 and rare.max() == S
    w = np.array([hwe_exchet(int(a), int(b), int(c)) for a, b, c, _m in gcount])
    assert (_bits(hwe) == _bits(w[:, 0])).all() and (_bits(exc) == _bits(w[:, 1])).all()
    assert (hwe < 1e-300).any() and (hwe > 0.5).any()
    co.close()
