"""Cohort genotyping: one SV catalogue genotyped in many samples by one process.  The counters of every sample
stay on the device ([S][num_sv][2], svjg_cohort_*), the genotype kernel runs over the (record x sample) grid block
by block, and each block's text (one column per sample) is written as it is made.  Column s of the VCF is byte for
byte what filter-alignments.py + predict-genotype.py write for sample s alone.  No tensor library: this is the
command-line front-end's path, like genotype.genotype_host."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import alnfilter, capi, genotype

CELL_BYTES = 24 + 1 + 8 + 1          # pl, gt, ad2, flags of one cell
BLOCK_BYTES = 256 << 20              # cell arrays of one block of records, at most
# population INFO tags of --info-tags, in the order they are written: bit k of svjg_vcf_format_cohort_tags's mask
INFO_TAGS = ("NS", "AN", "AC", "AF", "AC_Het", "AC_Hom", "F_MISSING", "HWE", "ExcHet")


def parse_info_tags(text):
    """--info-tags: a comma list of INFO_TAGS names (any order), or "all".  Returns the names in the order they are
    written; ValueError for an unknown or repeated name or an empty list."""
    if text == "all":
        return INFO_TAGS
    names = text.split(",")
    for nm in names:
        if nm not in INFO_TAGS:
            raise ValueError(f"unknown INFO tag {nm!r} (tags: {','.join(INFO_TAGS)}, or all)")
    if len(set(names)) != len(names):
        raise ValueError("an INFO tag is named twice")
    return tuple(t for t in INFO_TAGS if t in names)


def info_tags_mask(names):
    """The tag mask of svjg_vcf_format_cohort_tags for INFO_TAGS names."""
    mask = 0
    for nm in names:
        if nm not in INFO_TAGS:
            raise ValueError(f"unknown INFO tag {nm!r}")
        mask |= 1 << INFO_TAGS.index(nm)
    return mask


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
    ``n_records``, also the site statistics of that many records (svjg_cohort_site_stats, 32 B per record)."""

    def __init__(self, n_cells, n_records=0):
        n_cells = max(int(n_cells), 1)
        self._mem = [alnfilter.PinnedBytes(n_cells * b) for b in (24, 1, 8, 1)]
        self.pl = self._mem[0].array.view(np.int64).reshape(n_cells, 3)
        self.gt = self._mem[1].array
        self.ad2 = self._mem[2].array.view(np.uint32).reshape(n_cells, 2)
        self.flags = self._mem[3].array
        if n_records:
            n_records = int(n_records)
            self._mem += [alnfilter.PinnedBytes(n_records * b) for b in (16, 8, 8)]
            self.gcount = self._mem[4].array.view(np.uint32).reshape(n_records, 4)
            self.hwe = self._mem[5].array.view(np.float64)
            self.exchet = self._mem[6].array.view(np.float64)


def _genotype_block(cohort, idx, ty, min_support, e, blk):
    """(gt, flags, ad2, pl) of the records ``idx`` / ``ty`` in every sample, [n * S] cells in record-major order.
    Cells whose rounded counts are beyond the LUT are recomputed by genotype.genotype_host from their counters,
    which ad2 and the halving flags give back exactly."""
    n, S = len(idx), cohort.n_samples
    cells = n * S
    gt, fl, ad, pl = blk.gt[:cells], blk.flags[:cells], blk.ad2[:cells], blk.pl[:cells]
    la, lb, lh = math.log10(1 - e), math.log10(e), math.log10(1 / 2)
    lut = genotype.log10comb_lut()
    capi.check(capi.lib.svjg_cohort_genotype(cohort._h, idx.ctypes.data, ty.ctypes.data, n, int(min_support), la, lb, lh,
                                             lut.ctypes.data, genotype.LUT_NMAX, pl.ctypes.data, gt.ctypes.data,
                                             ad.ctypes.data, fl.ctypes.data))
    need = np.nonzero(fl & capi.GT_NEED_K)[0]
    if need.size:
        f = fl[need]
        n0 = np.where(f & capi.GT_HALVED_0, ad[need, 0], ad[need, 0] >> 1)
        n1 = np.where(f & capi.GT_HALVED_1, ad[need, 1], ad[need, 1] >> 1)
        g2, f2, a2, p2 = genotype.genotype_host(np.stack([n0, n1], axis=1), np.arange(need.size, dtype=np.uint32),
                                                ty[need // S], min_support, e)
        gt[need], fl[need], ad[need], pl[need] = g2, f2, a2, p2
    return gt, fl, ad, pl


def _site_stats(cohort, n, blk):
    """(gcount [n][4] = r0, h, r2, missing; hwe [n]; exchet [n]) of the block _genotype_block genotyped last, from
    the gt codes on the device.  Those are final: the NEED_K patch above recomputes PL and flags, never the genotype,
    which genotype_one fixes before it looks up log10 C(n, k)."""
    g, hw, ex = blk.gcount[:n], blk.hwe[:n], blk.exchet[:n]
    capi.check(capi.lib.svjg_cohort_site_stats(cohort._h, n, g.ctypes.data, hw.ctypes.data, ex.ctypes.data))
    return g, hw, ex


def genotype_cohort_vcf(tables, cohort, vcf_bytes, names, min_support=genotype.MIN_SUPPORT, e=genotype.ERR, out=None,
                        block_records=None, info_tags=()):
    """predict-genotype.py's decision_vcf for every sample of ``cohort``: the multi-sample VCF, whose column s is
    the SAMPLE column of sample s's single-sample VCF.  ``vcf_bytes``: the catalogue VCF's bytes (or lines).
    ``names``: one column name per sample.  Returns (text, [genotyped SVs per sample]); with ``out`` (a binary file
    object) each block's text is written there as it is made and the text returned is None.  ``block_records``:
    records per block (default: cell arrays of about 256 MiB); the bytes do not depend on it.  ``info_tags``: INFO_TAGS
    names; their values are computed on the device from each block's genotypes (svjg_cohort_site_stats) and written
    into the INFO column, and their ##INFO lines in front of the ##FORMAT lines (svjg_vcf_format_cohort_tags)."""
    S = cohort.n_samples
    mask = info_tags_mask(info_tags)
    if len(names) != S:
        raise ValueError(f"{len(names)} names for {S} samples")
    v = genotype.NativeVcf.from_input(vcf_bytes)
    if v is None:
        raise genotype.VcfError("the VCF has non-ASCII bytes or a POS/END of more than 18 digits: "
                                "cohort genotyping takes only VCFs the native parser reads")
    idx = np.ascontiguousarray(v.index_tables(tables))
    ty = np.ascontiguousarray(v.svtype)
    n = v.n
    step = int(block_records) if block_records else max(1, BLOCK_BYTES // (CELL_BYTES * S))
    blk = _Block(min(step, max(n, 1)) * S, min(step, max(n, 1)) if mask else 0)
    if not 0 < e < 1:
        # math.log10 raises inside likelihood() only once a record passes the gate (predict-genotype.py:216), as in
        # genotype.genotype_host: a cohort in which no cell passes it is written with "./." everywhere
        for lo in range(0, n, step):
            if (_genotype_block(cohort, idx[lo:lo + step], ty[lo:lo + step], min_support, genotype.ERR, blk)[1]
                    & capi.GT_GENOTYPED).any():
                raise genotype.VcfError("error rate must be in (0, 1)")
        e = genotype.ERR
    joined = "\t".join(names).encode()
    n_gt = np.zeros(S, np.uint64)
    pieces = []
    for lo in range(0, n, step) if n else [0]:
        hi = min(n, lo + step)
        gt, fl, ad, pl = _genotype_block(cohort, idx[lo:hi], ty[lo:hi], min_support, e, blk)
        site = [None] * 3
        if mask:
            site = [a.ctypes.data for a in _site_stats(cohort, hi - lo, blk)]
        buf, n_out = C.c_void_p(), C.c_uint64()
        capi.check(capi.lib.svjg_vcf_format_cohort_tags(v._h, lo, hi, S, joined, len(joined), gt.ctypes.data,
                                                        fl.ctypes.data, ad.ctypes.data, pl.ctypes.data, mask, *site,
                                                        C.byref(buf), C.byref(n_out), n_gt.ctypes.data))
        try:
            if out is not None:
                if n_out.value:
                    out.write(memoryview((C.c_char * n_out.value).from_address(buf.value)))
            else:
                pieces.append(C.string_at(buf.value, n_out.value))
        finally:
            capi.lib.svjg_buffer_free(buf)
    text = None if out is not None else b"".join(pieces).decode("ascii")
    return text, [int(x) for x in n_gt]
