"""Cohort genotyping: one SV catalogue genotyped in many samples by one process.  The counters of every sample
stay on the device ([S][num_sv][2], svjg_cohort_*), the genotype kernel runs over the (record x sample) grid block
by block, and each block's text (one column per sample) is written as it is made.  Column s of the VCF is byte for
byte what filter-alignments.py + predict-genotype.py write for sample s alone.  No tensor library: this is the
command-line front-end's path, like genotype.genotype_host."""
from __future__ import annotations

import ctypes as C
import math
import re

import numpy as np

from . import alnfilter, capi, genotype

CELL_BYTES = 24 + 1 + 8 + 1          # pl, gt, ad2, flags of one cell
POST_CELL_BYTES = 24 + 1             # gp, gq of one cell (genotype posteriors)
BLOCK_BYTES = 256 << 20              # cell arrays of one block of records, at most
# population INFO tags of --info-tags, in the order they are written: bit k of svjg_vcf_format_cohort_tags's mask
INFO_TAGS = ("NS", "AN", "AC", "AF", "AC_Het", "AC_Hom", "F_MISSING", "HWE", "ExcHet")
# with ploidy rules (svjg_vcf_format_cohort_ploidy): one more, bit 9
PLOIDY_INFO_TAGS = INFO_TAGS + ("AC_Hemi",)


def parse_info_tags(text, ploidy=False):
    """--info-tags: a comma list of tag names (any order), or "all": INFO_TAGS, or PLOIDY_INFO_TAGS with ``ploidy``.
    Returns the names in the order they are written; ValueError for an unknown or repeated name, an empty list, or
    AC_Hemi without ploidy rules."""
    tags = PLOIDY_INFO_TAGS if ploidy else INFO_TAGS
    if text == "all":
        return tags
    names = text.split(",")
    for nm in names:
        if nm == "AC_Hemi" and not ploidy:
            raise ValueError("AC_Hemi counts haploid calls: it needs --ploidy-file and --sample-sex")
        if nm not in tags:
            raise ValueError(f"unknown INFO tag {nm!r} (tags: {','.join(tags)}, or all)")
    if len(set(names)) != len(names):
        raise ValueError("an INFO tag is named twice")
    return tuple(t for t in tags if t in names)


def info_tags_mask(names):
    """The tag mask of svjg_vcf_format_cohort_tags / _ploidy for PLOIDY_INFO_TAGS names."""
    mask = 0
    for nm in names:
        if nm not in PLOIDY_INFO_TAGS:
            raise ValueError(f"unknown INFO tag {nm!r}")
        mask |= 1 << PLOIDY_INFO_TAGS.index(nm)
    return mask


# rows of the sample QC table (svjg_cohort_qc_sample_counts): every record, then the records of each SVTYPE code
QC_TYPES = ("ALL", "DEL", "INS", "INV", "BND")
SAMPLE_QC_HEADER = "#SAMPLE\tSVTYPE\tHOM_REF\tHET\tHOM_ALT\tHAP_REF\tHAP_ALT\tMISSING\tNO_PLOIDY\tCALL_RATE\tHET_HOM_RATIO\n"
RELATEDNESS_PIECE_PAIRS = 1 << 22          # pairs formatted per svjg_format_relatedness call


def _ratio(a, b):
    return "." if b == 0 else "%.6g" % (a / b)


def sample_qc_text(names, hist):
    """The sample QC table of the samples ``names`` from their histograms ``hist`` [S][5][8] (rows QC_TYPES, columns
    the gt codes 0-7): per sample and row, HOM_REF HET HOM_ALT HAP_REF HAP_ALT (codes 0, 1, 2, 4, 5), MISSING (3 and
    6), NO_PLOIDY (7), CALL_RATE = called / (called + MISSING) and HET_HOM_RATIO = HET / HOM_ALT ("." over 0)."""
    lines = [SAMPLE_QC_HEADER]
    for nm, h in zip(names, hist):
        for ty, row in zip(QC_TYPES, h):
            c = [int(x) for x in row]
            called, missing = c[0] + c[1] + c[2] + c[4] + c[5], c[3] + c[6]
            lines.append(f"{nm}\t{ty}\t{c[0]}\t{c[1]}\t{c[2]}\t{c[4]}\t{c[5]}\t{missing}\t{c[7]}\t"
                         f"{_ratio(called, called + missing)}\t{_ratio(c[1], c[2])}\n")
    return "".join(lines)


def write_relatedness(out, names, pairs, min_kinship=None):
    """Writes the relatedness table of the samples ``names`` from svjg_cohort_relatedness's counts ``pairs``
    [S (S - 1) / 2][5] to the binary file object ``out`` (svjg_format_relatedness, a range of rows per call).  With
    ``min_kinship``, only the pairs whose KINSHIP is at least that."""
    S = len(names)
    pairs = np.ascontiguousarray(pairs, np.uint32)
    if pairs.shape != (S * (S - 1) // 2, 5):
        raise ValueError(f"pair counts of shape {pairs.shape} for {S} samples")
    joined = "\t".join(names).encode()
    i = 0
    while True:
        lo, n_pairs = i, 0
        while i < S and n_pairs < RELATEDNESS_PIECE_PAIRS:
            n_pairs += S - 1 - i
            i += 1
        buf, n_out = C.c_void_p(), C.c_uint64()
        capi.check(capi.lib.svjg_format_relatedness(S, joined, len(joined), pairs.ctypes.data if pairs.size else None,
                                                    lo, i, int(min_kinship is not None),
                                                    0.0 if min_kinship is None else float(min_kinship), C.byref(buf),
                                                    C.byref(n_out)))
        try:
            if n_out.value:
                out.write(memoryview((C.c_char * n_out.value).from_address(buf.value)))
        finally:
            capi.lib.svjg_buffer_free(buf)
        if i >= S:
            return


GRM_MIN_MAF = 0.01                         # --grm-min-maf default
PCA_COMPONENTS = 10                        # --pca-components default


def grm_square(packed, S, dtype):
    """The symmetric [S][S] matrix of svjg_cohort_grm's packed upper triangle (pair i <= j at i (2 S - i + 1) / 2 +
    j - i), filled row by row so that no index arrays of S^2 entries are made."""
    out = np.zeros((S, S), dtype)
    o = 0
    for i in range(S):
        row = packed[o:o + S - i]
        out[i, i:] = row
        out[i:, i] = row
        o += S - i
    return out


def pca(G, k):
    """The k leading principal components of the symmetric relationship matrix G [S][S] (numpy.linalg.eigh): the k
    largest eigenvalues in descending order and their unit eigenvectors [S][k], each eigenvector's sign flipped so that
    its component of largest absolute value (the first such one on ties) is positive."""
    G = np.asarray(G, np.float64)
    if not 1 <= k <= G.shape[0]:
        raise ValueError(f"{k} principal components of {G.shape[0]} samples")
    vals, vecs = np.linalg.eigh(G)
    vals, vecs = vals[::-1][:k].copy(), vecs[:, ::-1][:, :k].copy()
    lead = vecs[np.argmax(np.abs(vecs), axis=0), np.arange(k)]
    vecs[:, lead < 0] *= -1.0
    return vals, vecs


def write_grm(bin_out, n_out, id_out, names, G, N):
    """GCTA's binary relationship matrix: the lower triangle with the diagonal, row by row (i from 0, j <= i), of G
    (``bin_out``) and of N (``n_out``) as little-endian float32, and one "NAME\\tNAME" line per sample (``id_out``).
    All three are binary file objects."""
    S = len(names)
    if np.shape(G) != (S, S) or np.shape(N) != (S, S):
        raise ValueError(f"relationship matrices of shape {np.shape(G)} / {np.shape(N)} for {S} samples")
    rows = max(1, (1 << 22) // max(S, 1))                      # about 4 M entries per write
    for lo in range(0, S, rows):
        hi = min(S, lo + rows)
        for M, out in ((G, bin_out), (N, n_out)):
            out.write(np.concatenate([M[i, :i + 1] for i in range(lo, hi)]).astype("<f4").tobytes())
    id_out.write("".join(f"{nm}\t{nm}\n" for nm in names).encode())


def write_pca(vec_out, val_out, names, vals, vecs):
    """The eigenvectors [S][K] (header "#IID\\tPC1 ... PCK", then one line per sample) and the eigenvalues [K] (one per
    line) of pca(), "%.6g", to the binary file objects ``vec_out`` and ``val_out``."""
    K = len(vals)
    if np.shape(vecs) != (len(names), K):
        raise ValueError(f"eigenvectors of shape {np.shape(vecs)} for {len(names)} samples and {K} components")
    lines = ["#IID" + "".join(f"\tPC{k + 1}" for k in range(K)) + "\n"]
    lines += [nm + "".join("\t%.6g" % x for x in row) + "\n" for nm, row in zip(names, vecs.tolist())]
    vec_out.write("".join(lines).encode())
    val_out.write("".join("%.6g\n" % x for x in vals.tolist()).encode())


_phred_weights = None


def phred_weights():
    """T[k] = 10.0 ** (-k / 10) for k < capi.POST_PLW_N, the weight of a genotype whose PL is k above the cell's
    smallest (svjg_cohort_posteriors).  Built by Python's own float power, so the device and the statement in the
    tests use the same doubles; T underflows to 0.0 long before the last entry."""
    global _phred_weights
    if _phred_weights is None:
        _phred_weights = np.array([10.0 ** (-k / 10) for k in range(capi.POST_PLW_N)], np.float64)
    return _phred_weights


def _table_lines(text):
    """(line number, whitespace-split columns) of the lines of a rule file that are not blank or '#' comments."""
    for k, line in enumerate(text.splitlines(), 1):
        cols = line.split()
        if cols and not cols[0].startswith("#"):
            yield k, cols


_DECIMAL = re.compile(r"[0-9]+")


class PloidyRules:
    """Sex-chromosome ploidy of a cohort's cells (DESIGN.md §8a).  ``ploidy_text``: the rules in the format of
    ``bcftools call --ploidy-file``, one ``CHROM FROM TO SEX PLOIDY`` per line (1-based, inclusive), ``* * * SEX
    PLOIDY`` for the default of a sex.  ``sex_text``: ``NAME SEX`` lines; every name of ``names`` (the cohort) must be
    listed exactly once, other names are ignored.  Both take '#' comments and blank lines.  ValueError, naming the
    file and the line, for a file the contract refuses.

    The ploidy of cell (record, sample) is that of the rule for the sample's sex whose CHROM is the record's CHROM
    column and whose [FROM, TO] holds the record's POS column, else the sex's default, else 2.  The record's CHROM and
    POS alone decide: an SV that starts in a PAR and ends outside it follows its POS."""

    def __init__(self, ploidy_text, sex_text, names, ploidy_source="ploidy file", sex_source="sample-sex file"):
        self.rules = {}                   # (chrom, sex) -> (from [k], to [k], ploidy [k]) sorted by from
        self.defaults = {}                # sex -> ploidy
        labels = set()
        spans = {}
        for k, cols in _table_lines(ploidy_text):
            where = f"{ploidy_source} line {k}"
            if len(cols) != 5:
                raise ValueError(f"{where}: {len(cols)} columns, a rule is CHROM FROM TO SEX PLOIDY")
            chrom, lo, hi, sex, ploidy = cols
            if ploidy not in ("0", "1", "2"):
                raise ValueError(f"{where}: ploidy {ploidy!r}, it must be 0, 1 or 2")
            labels.add(sex)
            if chrom == "*" and lo == "*" and hi == "*":
                if sex in self.defaults:
                    raise ValueError(f"{where}: a second default ('* * *') for sex {sex!r}")
                self.defaults[sex] = int(ploidy)
                continue
            if not (_DECIMAL.fullmatch(lo) and _DECIMAL.fullmatch(hi)):
                raise ValueError(f"{where}: FROM and TO must be decimal integers ('* * *' for a default)")
            lo, hi = int(lo), int(hi)
            if lo > hi:
                raise ValueError(f"{where}: FROM {lo} > TO {hi}")
            spans.setdefault((chrom, sex), []).append((lo, hi, int(ploidy), k))
        for (chrom, sex), rs in spans.items():
            rs.sort()
            for a, b in zip(rs, rs[1:]):
                if b[0] <= a[1]:
                    raise ValueError(f"{ploidy_source} lines {a[3]} and {b[3]}: two rules for {chrom} and sex {sex!r} "
                                     "overlap")
            self.rules[chrom, sex] = tuple(np.array([r[q] for r in rs], np.int64) for q in range(3))
        cohort = {nm: None for nm in names}
        for k, cols in _table_lines(sex_text):
            if len(cols) != 2:
                raise ValueError(f"{sex_source} line {k}: {len(cols)} columns, a line is NAME SEX")
            nm, sex = cols
            if nm in cohort:
                if cohort[nm] is not None:
                    raise ValueError(f"{sex_source} line {k}: sample {nm!r} is listed twice")
                cohort[nm] = sex
        missing = [nm for nm, sex in cohort.items() if sex is None]
        if missing:
            raise ValueError(f"{sex_source}: no sex for sample {missing[0]!r}" +
                             (f" and {len(missing) - 1} more" if len(missing) > 1 else ""))
        self.sample_sex = [cohort[nm] for nm in names]
        labels.update(self.sample_sex)
        if len(labels) > capi.PLOIDY_MAX_SEXES:
            raise ValueError(f"{len(labels)} sex labels in the two files: at most {capi.PLOIDY_MAX_SEXES}")
        self.sexes = sorted(set(self.sample_sex))                 # the columns of the class table
        self.sex_index = np.array([self.sexes.index(x) for x in self.sample_sex], np.uint8)

    def record_classes(self, v):
        """(rclass [n] uint8, table [n_classes][len(sexes)] uint8) of the records of NativeVcf ``v``: record i has
        ploidy table[rclass[i]][k] in a sample of sex sexes[k].  VcfError for a POS that is not a decimal integer,
        ValueError beyond 255 classes."""
        chrom, pos, names = v.loci()
        order = np.argsort(chrom, kind="stable")
        bounds = np.searchsorted(chrom[order], np.arange(len(names) + 1))
        where = {nm: k for k, nm in enumerate(names)}
        cols = []
        for sex in self.sexes:
            col = np.full(v.n, self.defaults.get(sex, 2), np.uint8)
            for (c, x), (lo, hi, pl) in self.rules.items():
                if x != sex or c not in where:
                    continue
                recs = order[bounds[where[c]]:bounds[where[c] + 1]]
                p = pos[recs]
                j = np.searchsorted(lo, p, side="right") - 1           # the last rule that starts at or before POS
                inside = (j >= 0) & (p <= hi[np.maximum(j, 0)])
                col[recs[inside]] = pl[j[inside]]
            cols.append(col)
        rows = np.ascontiguousarray(np.stack(cols, axis=1)) if v.n else np.full((1, len(self.sexes)), 2, np.uint8)
        table, rclass = np.unique(rows.view(np.dtype((np.void, rows.shape[1]))).ravel(), return_inverse=True)
        if len(table) > capi.PLOIDY_MAX_CLASSES:
            raise ValueError(f"the ploidy rules give the catalogue's records {len(table)} distinct ploidy vectors: "
                             f"at most {capi.PLOIDY_MAX_CLASSES}")
        table = np.frombuffer(table.tobytes(), np.uint8).reshape(len(table), len(self.sexes))
        return np.ascontiguousarray(rclass.reshape(-1)[:v.n], np.uint8), np.ascontiguousarray(table)


class Cohort:
    """Counters of ``n_samples`` samples against ``tables`` (on its device), all zero at the start."""

    def __init__(self, tables, n_samples):
        if tables.device is None:
            raise RuntimeError("tables.to_device() first")
        self.tables = tables                    # the handle keeps using the tables' device image
        self.n_samples = int(n_samples)
        self.num_sv = tables.num_sv
        self._h = C.c_void_p()
        capi.check(capi.lib.svjg_cohort_create(tables._h, self.n_samples, C.byref(self._h)))

    def filter(self, s, gaf, d_over=alnfilter.D_OVER):
        """The filter of filter-alignments.py over GAF bytes in host memory, ADDED to sample ``s``'s counters.
        Returns the stats; alnfilter.InputError (offset within ``gaf``) where the reference raises."""
        a = alnfilter._as_u8(gaf)
        stats = capi.FilterStats()
        rc = capi.lib.svjg_cohort_filter(self._h, int(s), a.ctypes.data if a.size else None, a.size, int(d_over),
                                         C.byref(stats))
        st = stats.as_dict()
        if rc == capi.E_INPUT:
            alnfilter._raise_input(st)
        capi.check(rc)
        return st

    def counts(self, s):
        """Sample ``s``'s counters, numpy uint32 [num_sv, 2]."""
        out = np.zeros((max(self.num_sv, 1), 2), np.uint32)
        capi.check(capi.lib.svjg_cohort_read_counts(self._h, int(s), out.ctypes.data))
        return out[:self.num_sv]

    def load_counts(self, s, counts):
        """Replaces sample ``s``'s counters with ``counts`` [num_sv, 2]."""
        c = np.ascontiguousarray(counts, dtype=np.uint32).reshape(-1, 2)
        if c.shape[0] != self.num_sv:
            raise ValueError(f"counts for {c.shape[0]} SVs, the catalogue has {self.num_sv}")
        capi.check(capi.lib.svjg_cohort_load_counts(self._h, int(s), c.ctypes.data if c.size else None))

    def close(self):
        if self._h:
            capi.lib.svjg_cohort_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Block:
    """Page-locked result arrays of one block of records: the copies from the device run at PCIe speed.  With
    ``n_records``, also the site statistics of that many records (svjg_cohort_site_stats, 32 B per record; with
    ``ploidy``, svjg_cohort_site_stats_ploidy, 40 B).  With ``post_records``, the genotype posteriors of that many
    records (svjg_cohort_posteriors: af, 8 B per record; gp and gq, 25 B per cell)."""

    def __init__(self, n_cells, n_records=0, ploidy=False, post_records=0):
        n_cells = max(int(n_cells), 1)
        self._mem = [alnfilter.PinnedBytes(n_cells * b) for b in (24, 1, 8, 1)]
        self.pl = self._mem[0].array.view(np.int64).reshape(n_cells, 3)
        self.gt = self._mem[1].array
        self.ad2 = self._mem[2].array.view(np.uint32).reshape(n_cells, 2)
        self.flags = self._mem[3].array
        if n_records:
            n_records = int(n_records)
            g = 6 if ploidy else 4
            self._mem += [alnfilter.PinnedBytes(n_records * b) for b in (4 * g, 8, 8)]
            self.gcount = self._mem[4].array.view(np.uint32).reshape(n_records, g)
            self.hwe = self._mem[5].array.view(np.float64)
            self.exchet = self._mem[6].array.view(np.float64)
        if post_records:
            mem = [alnfilter.PinnedBytes(b) for b in (int(post_records) * 8, n_cells * 24, n_cells)]
            self._mem += mem
            self.af = mem[0].array.view(np.float64)
            self.gp = mem[1].array.view(np.float64).reshape(n_cells, 3)
            self.gq = mem[2].array
        self.need = np.zeros(0, np.int64)           # the NEED_K cells the last _genotype_block patched


def _genotype_block(cohort, idx, ty, min_support, e, blk, rclass=None):
    """(gt, flags, ad2, pl) of the records ``idx`` / ``ty`` in every sample, [n * S] cells in record-major order;
    with ``rclass``, the ploidy classes of the records (svjg_cohort_genotype_ploidy, after svjg_cohort_set_ploidy).
    Cells whose rounded counts are beyond the LUT are recomputed by genotype.genotype_host from their counters,
    which ad2 and the halving flags give back exactly.  A haploid cell keeps the device's code: the device fixes the
    call before it looks up log10 C(n, k), so only PL (of which the text shows PL0 and PL2) comes from the host."""
    n, S = len(idx), cohort.n_samples
    cells = n * S
    gt, fl, ad, pl = blk.gt[:cells], blk.flags[:cells], blk.ad2[:cells], blk.pl[:cells]
    la, lb, lh = math.log10(1 - e), math.log10(e), math.log10(1 / 2)
    lut = genotype.log10comb_lut()
    if rclass is None:
        capi.check(capi.lib.svjg_cohort_genotype(cohort._h, idx.ctypes.data, ty.ctypes.data, n, int(min_support), la, lb,
                                                 lh, lut.ctypes.data, genotype.LUT_NMAX, pl.ctypes.data, gt.ctypes.data,
                                                 ad.ctypes.data, fl.ctypes.data))
    else:
        capi.check(capi.lib.svjg_cohort_genotype_ploidy(cohort._h, idx.ctypes.data, ty.ctypes.data, rclass.ctypes.data, n,
                                                        int(min_support), la, lb, lh, lut.ctypes.data, genotype.LUT_NMAX,
                                                        pl.ctypes.data, gt.ctypes.data, ad.ctypes.data, fl.ctypes.data))
    need = np.nonzero(fl & capi.GT_NEED_K)[0]
    if need.size:
        f = fl[need]
        n0 = np.where(f & capi.GT_HALVED_0, ad[need, 0], ad[need, 0] >> 1)
        n1 = np.where(f & capi.GT_HALVED_1, ad[need, 1], ad[need, 1] >> 1)
        g2, f2, a2, p2 = genotype.genotype_host(np.stack([n0, n1], axis=1), np.arange(need.size, dtype=np.uint32),
                                                ty[need // S], min_support, e)
        gt[need] = np.where(gt[need] >= capi.GT_HAP_REF, gt[need], g2)
        fl[need], ad[need], pl[need] = f2, a2, p2
    blk.need = need
    return gt, fl, ad, pl


def _site_stats(cohort, n, blk, ploidy=False):
    """(gcount [n][4] = r0, h, r2, missing, or with ``ploidy`` [n][6] = r0, h, r2, a0, a1, missing; hwe [n];
    exchet [n]) of the block _genotype_block genotyped last, from the gt codes on the device.  Those are final: the
    NEED_K patch above recomputes PL and flags, never the genotype, which genotype_one fixes before it looks up
    log10 C(n, k)."""
    g, hw, ex = blk.gcount[:n], blk.hwe[:n], blk.exchet[:n]
    fn = capi.lib.svjg_cohort_site_stats_ploidy if ploidy else capi.lib.svjg_cohort_site_stats
    capi.check(fn(cohort._h, n, g.ctypes.data, hw.ctypes.data, ex.ctypes.data))
    return g, hw, ex


def _posteriors(cohort, n, blk, iters=None):
    """(af [n], gp [n * S][3], gq [n * S]) of the block _genotype_block genotyped last (svjg_cohort_posteriors), with
    the PLs that block's NEED_K patch computed on the host sent to the device first.  ``iters``: a uint8 [n] array
    that receives the EM steps per record."""
    cells = n * cohort.n_samples
    af, gp, gq = blk.af[:n], blk.gp[:cells], blk.gq[:cells]
    need = blk.need
    pcell = np.ascontiguousarray(need, np.uint32)
    ppl = np.ascontiguousarray(blk.pl[need], np.int64)
    T = phred_weights()
    capi.check(capi.lib.svjg_cohort_posteriors(cohort._h, n, need.size, pcell.ctypes.data if need.size else None,
                                               ppl.ctypes.data if need.size else None, T.ctypes.data, T.size,
                                               af.ctypes.data, gp.ctypes.data, gq.ctypes.data,
                                               None if iters is None else iters.ctypes.data))
    return af, gp, gq


def genotype_cohort_vcf(tables, cohort, vcf_bytes, names, min_support=genotype.MIN_SUPPORT, e=genotype.ERR, out=None,
                        block_records=None, info_tags=(), ploidy=None, posteriors=False, sample_qc=False,
                        relatedness=False, grm=False, grm_min_maf=GRM_MIN_MAF):
    """predict-genotype.py's decision_vcf for every sample of ``cohort``: the multi-sample VCF, whose column s is
    the SAMPLE column of sample s's single-sample VCF.  ``vcf_bytes``: the catalogue VCF's bytes (or lines, or a
    genotype.NativeVcf of them).
    ``names``: one column name per sample.  Returns (text, [genotyped SVs per sample]); with ``out`` (a binary file
    object) each block's text is written there as it is made and the text returned is None.  ``block_records``:
    records per block (default: cell arrays of about 256 MiB); the bytes do not depend on it.  ``info_tags``: INFO_TAGS
    names; their values are computed on the device from each block's genotypes (svjg_cohort_site_stats) and written
    into the INFO column, and their ##INFO lines in front of the ##FORMAT lines (svjg_vcf_format_cohort_tags).
    ``ploidy``: a PloidyRules for the samples of ``names``; the cells are called with their ploidy and the text is
    that of svjg_vcf_format_cohort_ploidy (PL Number=G, AC_Hemi available).  ``posteriors``: the allele frequency of
    every record by EM over its cells' likelihoods (INFO AF_EM), and each cell's GP and GQ under the Hardy-Weinberg
    prior at it (svjg_cohort_posteriors, svjg_vcf_format_cohort_post); GT stays the likelihood call.
    ``sample_qc`` / ``relatedness``: the genotype codes of every block are also counted on the device
    (svjg_cohort_qc_add), and the result is (text, counts, hist, pairs): hist [S][5][8] (svjg_cohort_qc_sample_counts)
    or None, pairs [S (S - 1) / 2][5] (svjg_cohort_relatedness) or None; the text is the same.
    ``grm``: the bit planes are kept as for ``relatedness``, and the result is (text, counts, hist, pairs, (G, N)): the
    relationship matrix over the records whose minor allele frequency is at least ``grm_min_maf`` (svjg_cohort_grm),
    G [S][S] float64 and N [S][S] uint32, both symmetric."""
    S = cohort.n_samples
    mask = info_tags_mask(info_tags)
    if len(names) != S:
        raise ValueError(f"{len(names)} names for {S} samples")
    if ploidy is None and "AC_Hemi" in info_tags:
        raise ValueError("AC_Hemi counts haploid calls: it needs ploidy rules")
    if relatedness and S > capi.QC_MAX_PAIR_SAMPLES:
        raise ValueError(f"relatedness takes at most {capi.QC_MAX_PAIR_SAMPLES} samples")
    if grm and S > capi.QC_MAX_PAIR_SAMPLES:
        raise ValueError(f"the relationship matrix takes at most {capi.QC_MAX_PAIR_SAMPLES} samples")
    if grm and not 0.0 <= grm_min_maf <= 0.5:
        raise ValueError(f"grm_min_maf {grm_min_maf!r} is not in [0, 0.5]")
    v = vcf_bytes if isinstance(vcf_bytes, genotype.NativeVcf) else genotype.NativeVcf.from_input(vcf_bytes)
    if v is None:
        raise genotype.VcfError("the VCF has non-ASCII bytes or a POS/END of more than 18 digits: "
                                "cohort genotyping takes only VCFs the native parser reads")
    idx = np.ascontiguousarray(v.index_tables(tables))
    ty = np.ascontiguousarray(v.svtype)
    n = v.n
    rclass = None
    if ploidy is not None:
        rclass, table = ploidy.record_classes(v)
        capi.check(capi.lib.svjg_cohort_set_ploidy(cohort._h, table.shape[0], table.shape[1], table.ctypes.data,
                                                   ploidy.sex_index.ctypes.data))
    cell_bytes = CELL_BYTES + (POST_CELL_BYTES if posteriors else 0)
    step = int(block_records) if block_records else max(1, BLOCK_BYTES // (cell_bytes * S))
    rows = min(step, max(n, 1))
    blk = _Block(rows * S, rows if mask else 0, ploidy is not None, rows if posteriors else 0)
    if not 0 < e < 1:
        # math.log10 raises inside likelihood() only once a record passes the gate (predict-genotype.py:216), as in
        # genotype.genotype_host: a cohort in which no cell passes it is written with "./." everywhere.  A cell of
        # ploidy 0 computes no likelihood, so it does not count.
        for lo in range(0, n, step):
            gt, fl = _genotype_block(cohort, idx[lo:lo + step], ty[lo:lo + step], min_support, genotype.ERR, blk,
                                     None if rclass is None else rclass[lo:lo + step])[:2]
            if ((fl & capi.GT_GENOTYPED).astype(bool) & (gt != capi.GT_NO_CALL)).any():
                raise genotype.VcfError("error rate must be in (0, 1)")
        e = genotype.ERR
    qc = sample_qc or relatedness or grm
    if qc:
        # every block starts a new word of the bit planes
        n_words = n // step * -(-step // 32) + -(-(n % step) // 32)
        capi.check(capi.lib.svjg_cohort_qc_begin(cohort._h, n_words, int(bool(relatedness or grm))))
    joined = "\t".join(names).encode()
    n_gt = np.zeros(S, np.uint64)
    pieces = []
    for lo in range(0, n, step) if n else [0]:
        hi = min(n, lo + step)
        gt, fl, ad, pl = _genotype_block(cohort, idx[lo:hi], ty[lo:hi], min_support, e, blk,
                                         None if rclass is None else rclass[lo:hi])
        if qc:
            capi.check(capi.lib.svjg_cohort_qc_add(cohort._h, hi - lo))
        site = [None] * 3
        if mask:
            site = [a.ctypes.data for a in _site_stats(cohort, hi - lo, blk, rclass is not None)]
        buf, n_out = C.c_void_p(), C.c_uint64()
        if posteriors:
            post = [a.ctypes.data for a in _posteriors(cohort, hi - lo, blk)]
            capi.check(capi.lib.svjg_vcf_format_cohort_post(
                v._h, lo, hi, S, joined, len(joined), gt.ctypes.data, fl.ctypes.data, ad.ctypes.data, pl.ctypes.data,
                int(rclass is not None), mask, *site, *post, C.byref(buf), C.byref(n_out), n_gt.ctypes.data))
        else:
            fmt = capi.lib.svjg_vcf_format_cohort_ploidy if rclass is not None else capi.lib.svjg_vcf_format_cohort_tags
            capi.check(fmt(v._h, lo, hi, S, joined, len(joined), gt.ctypes.data, fl.ctypes.data, ad.ctypes.data,
                           pl.ctypes.data, mask, *site, C.byref(buf), C.byref(n_out), n_gt.ctypes.data))
        try:
            if out is not None:
                if n_out.value:
                    out.write(memoryview((C.c_char * n_out.value).from_address(buf.value)))
            else:
                pieces.append(C.string_at(buf.value, n_out.value))
        finally:
            capi.lib.svjg_buffer_free(buf)
    text = None if out is not None else b"".join(pieces).decode("ascii")
    if not qc:
        return text, [int(x) for x in n_gt]
    hist = pairs = None
    if sample_qc:
        hist = np.zeros((S, len(QC_TYPES), 8), np.uint32)
        capi.check(capi.lib.svjg_cohort_qc_sample_counts(cohort._h, hist.ctypes.data))
    if relatedness:
        pairs = np.zeros((S * (S - 1) // 2, 5), np.uint32)
        capi.check(capi.lib.svjg_cohort_relatedness(cohort._h, pairs.ctypes.data if pairs.size else None))
    if not grm:
        return text, [int(x) for x in n_gt], hist, pairs
    g = np.zeros(S * (S + 1) // 2, np.float64)
    nn = np.zeros(S * (S + 1) // 2, np.uint32)
    capi.check(capi.lib.svjg_cohort_grm(cohort._h, float(grm_min_maf), g.ctypes.data if S else None,
                                        nn.ctypes.data if S else None))
    return text, [int(x) for x in n_gt], hist, pairs, (grm_square(g, S, np.float64), grm_square(nn, S, np.uint32))
