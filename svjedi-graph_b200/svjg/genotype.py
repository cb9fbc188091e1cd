"""Host mirror of predict-genotype.py (reference :29-72, :89-346): VCF keys on
the host, likelihood / GT / PL on the device (kernel 4), VCF text out."""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import capi

MIN_SUPPORT = 3     # predict-genotype.py:46
ERR = 0.00005       # predict-genotype.py:61
LUT_NMAX = 256

SVTYPE_CODE = {"DEL": 0, "INS": 1, "INV": 2, "BND": 3}
GT_TEXT = ("0/0", "0/1", "1/1", "./.")

_FORMAT_LINES = (
    '##FORMAT=<ID=GT,Number=1,Type=String,Description="Genotype">\n'
    '##FORMAT=<ID=DP,Number=1,Type=Float,Description="Total number of informative read alignments across all alleles (after normalization for unbalanced SVs)">\n'
    '##FORMAT=<ID=AD,Number=2,Type=Float,Description="Number of informative read alignments supporting each allele (after normalization by breakpoint number for unbalanced SVs)">\n'
    '##FORMAT=<ID=PL,Number=3,Type=Integer,Description="Phred-scaled likelihood for each genotype">\n'
    "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tSAMPLE\n"
)


class VcfError(Exception):
    """The reference raises on this VCF line (exit status 1)."""


_lut_cache = {}


def log10comb_lut(nmax=LUT_NMAX):
    """log10(C(n,k)) for 0<=k<=n<=nmax at [n(n+1)/2 + k], from CPython's own
    math.log10(math.comb()) so it is bit-equal to predict-genotype.py:313."""
    lut = _lut_cache.get(nmax)
    if lut is None:
        lut = np.empty((nmax + 1) * (nmax + 2) // 2, dtype=np.float64)
        i = 0
        for n in range(nmax + 1):
            for k in range(n + 1):
                lut[i] = math.log10(math.comb(n, k))
                i += 1
        _lut_cache[nmax] = lut
    return lut


def _info(info, label):
    # predict-genotype.py:77-87
    fields = info.split(";")
    tag = label + "="
    try:
        if fields[0].startswith(tag):
            return info.split(tag)[1].split(";")[0]
        rest = info.split(";" + tag)[1]
    except IndexError:
        raise VcfError(f"INFO has no {label}=") from None
    return rest if fields[-1].startswith(tag) else rest.split(";")[0]


def parse_vcf(lines):
    """Splits a VCF into output header text and body records.
    Each record: (head_text, svtype_code|0x80 if short, key or None).
    Mirrors predict-genotype.py:100-211 and the column cut at :250-256."""
    header, recs = [], []
    seen_ins = {}
    for line in lines:
        if line.startswith("##FORMAT"):
            continue
        if line.startswith("##"):
            header.append((len(recs), line))
            continue
        if line.startswith("#C"):
            header.append((len(recs), _FORMAT_LINES))
            continue
        cols = line.rstrip("\n").split("\t")
        if len(cols) < 8:
            raise VcfError("VCF line with fewer than 8 columns")
        chrom, pos, alt, info = cols[0], cols[1], cols[4], cols[7]
        svtype = ""
        if "SVTYPE" in info:
            parts = info.split("SVTYPE=")
            if len(parts) < 2:
                raise VcfError("SVTYPE without a value")
            svtype = parts[1] if info.split(";")[-1].startswith("SVTYPE=") else parts[1].split(";")[0]
        key, length = None, 0
        if svtype not in ("BND", "INS"):
            end = _info(info, "END")
            if svtype in ("DEL", "INV"):
                try:
                    length = int(end) - int(pos)
                except ValueError:
                    raise VcfError("non-integer POS/END") from None
                key = f"{chrom}:{svtype}-{pos}-{end}"
        elif svtype == "INS":
            k = seen_ins.get(pos, 0) + 1          # running count per POS string, any chromosome (:151-155)
            seen_ins[pos] = k
            key, length = f"{chrom}:INS-{pos}-{k}", len(alt)
        else:
            length = 50
            key = "wrong_format"
            for br in "[]":
                if br in alt:
                    pieces = [p for p in alt.split(br) if p]
                    if len(pieces) < 2:
                        raise VcfError("malformed BND ALT")
                    key = (f"{chrom}:BND-{pos}{br}{pieces[1]}{br}" if ":" in pieces[1]
                           else f"{chrom}:BND-{br}{pieces[0]}{br}{pos}")
                    break
        code = SVTYPE_CODE.get(svtype, 255)
        if code != 255 and abs(length) < 50:
            code |= 0x80
        n_tabs = line.count("\t")
        head = line.rstrip("\n") if n_tabs + 1 <= 8 else "\t".join(line.split("\t")[:8])
        recs.append((head, code, key))
    return header, recs


class VcfText:
    """genotype.vcf text in a buffer of the library (svjg_vcf_format); ``.view`` until the object goes away."""

    def __init__(self, ptr, nbytes):
        self._p, self.nbytes = ptr, nbytes
        self.view = memoryview((C.c_char * nbytes).from_address(ptr.value)) if nbytes else memoryview(b"")

    def __del__(self):
        try:
            if self._p:
                self.view = None
                capi.lib.svjg_buffer_free(self._p)
                self._p = None
        except Exception:
            pass


class NativeVcf:
    """svjg_vcf_* (csrc/vcf.cpp): the keys, svtype codes and output text of a whole VCF without a
    Python-level loop over its records.  :func:`parse_vcf` / :func:`format_vcf` state the same rules
    line by line and take over for the spellings the library declines (non-ASCII bytes, POS/END of
    more than 18 digits)."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle)
        self.n = int(capi.lib.svjg_vcf_num_records(self._h))

    @classmethod
    def parse(cls, data, translate_cr=True):
        """``data``: bytes of the file.  None if the library declines the file; VcfError where the
        reference raises."""
        h = C.c_void_p()
        if isinstance(data, np.ndarray):                 # the file's bytes where they lie (no copy)
            a = np.ascontiguousarray(data, dtype=np.uint8)
            rc = capi.lib.svjg_vcf_parse(a.ctypes.data if a.size else None, a.size, 1 if translate_cr else 0, C.byref(h))
        else:
            rc = capi.lib.svjg_vcf_parse(data, len(data), 1 if translate_cr else 0, C.byref(h))
        if rc == capi.E_UNSUPPORTED:
            return None
        if rc == capi.E_INPUT:
            raise VcfError(capi.lib.svjg_last_error().decode("utf-8", "replace"))
        capi.check(rc)
        return cls(h.value)

    @classmethod
    def from_input(cls, vcf):
        """From what the callers hold: the file's bytes (bytes / bytearray / uint8 array: read as text
        mode reads them) or a list of lines as ``readlines()`` gives them."""
        if isinstance(vcf, np.ndarray):
            return cls.parse(vcf, True)
        if isinstance(vcf, (bytes, bytearray, memoryview)):
            return cls.parse(bytes(vcf), True)
        lines = vcf if isinstance(vcf, list) else list(vcf)
        for i, line in enumerate(lines):
            # joined and cut at "\n" again these must give the same lines
            if not line or (line.find("\n") != len(line) - 1 and not (i == len(lines) - 1 and "\n" not in line)):
                return None
        try:
            data = "".join(lines).encode("ascii")
        except UnicodeEncodeError:
            return None
        return cls.parse(data, False)

    @property
    def svtype(self):
        if not self.n:
            return np.zeros(0, np.uint8)
        p = capi.lib.svjg_vcf_svtype(self._h)
        return np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(self.n,)).copy()

    def key(self, i):
        n = C.c_uint32()
        p = capi.lib.svjg_vcf_key(self._h, i, C.byref(n))
        return None if not p else C.string_at(p, n.value).decode("ascii")

    def loci(self):
        """(chrom [n] uint32: index into the names, pos [n] int64, [distinct CHROM names in order of first appearance])
        from the CHROM and POS columns; VcfError for a POS that is not 1 to 18 decimal digits."""
        chrom, pos = np.empty(max(self.n, 1), np.uint32), np.empty(max(self.n, 1), np.int64)
        buf, n_bytes, n_chroms = C.c_void_p(), C.c_uint64(), C.c_uint32()
        rc = capi.lib.svjg_vcf_loci(self._h, chrom.ctypes.data, pos.ctypes.data, C.byref(buf), C.byref(n_bytes),
                                    C.byref(n_chroms))
        if rc == capi.E_INPUT:
            raise VcfError(capi.lib.svjg_last_error().decode("utf-8", "replace"))
        capi.check(rc)
        try:
            names = C.string_at(buf.value, n_bytes.value).decode("ascii").split("\n") if n_chroms.value else []
        finally:
            capi.lib.svjg_buffer_free(buf)
        return chrom[:self.n], pos[:self.n], names

    def index_tables(self, tables):
        idx = np.empty(max(self.n, 1), np.uint32)
        capi.check(capi.lib.svjg_vcf_index_tables(self._h, tables._h, idx.ctypes.data))
        return idx[:self.n]

    def index_counts(self, aln_counts):
        idx = np.empty(max(self.n, 1), np.uint32)
        ty = np.empty(max(self.n, 1), np.uint8)
        rc = capi.lib.svjg_vcf_index_counts(self._h, aln_counts._h, idx.ctypes.data, ty.ctypes.data)
        if rc == capi.E_INPUT:
            raise VcfError(capi.lib.svjg_last_error().decode("utf-8", "replace"))
        capi.check(rc)
        return idx[:self.n], ty[:self.n]

    def format(self, gt, flags, ad2, pl, out=None):
        """(text, number of genotyped SVs) — predict-genotype.py:248-275.  With ``out`` (a binary
        file object) the bytes go straight to it and the text returned is None."""
        gt = np.ascontiguousarray(gt, dtype=np.uint8)
        flags = np.ascontiguousarray(flags, dtype=np.uint8)
        ad2 = np.ascontiguousarray(ad2, dtype=np.uint32)
        pl = np.ascontiguousarray(pl, dtype=np.int64)
        if not (len(gt) == len(flags) == len(ad2) == len(pl) == self.n):
            raise ValueError("result arrays do not match the number of VCF records")
        buf, n_out, n_gt = C.c_void_p(), C.c_uint64(), C.c_uint64()
        capi.check(capi.lib.svjg_vcf_format(self._h, gt.ctypes.data, flags.ctypes.data, ad2.ctypes.data, pl.ctypes.data,
                                            C.byref(buf), C.byref(n_out), C.byref(n_gt)))
        try:
            if out is not None:
                text = None
                if n_out.value:
                    out.write(memoryview((C.c_char * n_out.value).from_address(buf.value)))
            else:
                text = C.string_at(buf.value, n_out.value).decode("ascii")
        finally:
            capi.lib.svjg_buffer_free(buf)
        return text, int(n_gt.value)

    def format_buffer(self, gt, flags, ad2, pl):
        """(VcfText, number of genotyped SVs): the text where the library put it, without a Python copy."""
        gt = np.ascontiguousarray(gt, dtype=np.uint8)
        flags = np.ascontiguousarray(flags, dtype=np.uint8)
        ad2 = np.ascontiguousarray(ad2, dtype=np.uint32)
        pl = np.ascontiguousarray(pl, dtype=np.int64)
        if not (len(gt) == len(flags) == len(ad2) == len(pl) == self.n):
            raise ValueError("result arrays do not match the number of VCF records")
        buf, n_out, n_gt = C.c_void_p(), C.c_uint64(), C.c_uint64()
        capi.check(capi.lib.svjg_vcf_format(self._h, gt.ctypes.data, flags.ctypes.data, ad2.ctypes.data, pl.ctypes.data,
                                            C.byref(buf), C.byref(n_out), C.byref(n_gt)))
        return VcfText(buf, int(n_out.value)), int(n_gt.value)

    def close(self):
        if self._h:
            capi.lib.svjg_vcf_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _as_lines(vcf):
    """Lines as ``open(path).readlines()`` gives them, for the line-by-line statement of the rules."""
    if isinstance(vcf, np.ndarray):
        vcf = vcf.tobytes()
    if isinstance(vcf, (bytes, bytearray, memoryview)):
        import io
        return io.TextIOWrapper(io.BytesIO(bytes(vcf))).readlines()
    return vcf


def _num(twice, halved):
    if not halved:
        return str(twice >> 1)
    return f"{twice >> 1}.5" if twice & 1 else f"{twice >> 1}.0"


def _k_overrides(flags, ad, n):
    """log10 C(n,k) from CPython for exactly the SVs whose counts are beyond the table."""
    need = np.nonzero(flags & capi.GT_NEED_K)[0]
    if not need.size:
        return None
    kov = np.full(n, np.nan)
    memo = {}
    for i in need:
        t1, t2 = int(ad[i, 0]), int(ad[i, 1])
        r1 = (t1 >> 1) + ((t1 >> 1) & 1 if t1 & 1 else 0)
        r2 = (t2 >> 1) + ((t2 >> 1) & 1 if t2 & 1 else 0)
        v = memo.get((r1, r2))
        if v is None:
            v = memo[(r1, r2)] = math.log10(math.comb(r1 + r2, r1))
        kov[i] = v
    return kov


def genotype_host(counts, sv_index, svtype, min_support=MIN_SUPPORT, e=ERR):
    """Kernel 4 from host arrays (svjg_genotype_host): ``counts`` numpy uint32 [num, 2].  Returns
    numpy (gt, flags, ad2, pl).  Needs no tensor library -- the path of the command-line front-ends."""
    n = int(len(sv_index))
    if not 0 < e < 1:
        # math.log10 raises inside likelihood() (predict-genotype.py:295-299), i.e. only once a record passes the gate
        # at :216; a VCF without such a record is written out with "./." everywhere
        out = genotype_host(counts, sv_index, svtype, min_support, ERR)
        if (out[1] & capi.GT_GENOTYPED).any():
            raise VcfError("error rate must be in (0, 1)")
        return out
    la, lb, lh = math.log10(1 - e), math.log10(e), math.log10(1 / 2)
    lut = log10comb_lut()
    counts = np.ascontiguousarray(counts, dtype=np.uint32).reshape(-1, 2)
    idx = np.ascontiguousarray(sv_index, dtype=np.uint32)
    ty = np.ascontiguousarray(svtype, dtype=np.uint8)
    pl = np.zeros((max(n, 1), 3), np.int64)
    gt = np.zeros(max(n, 1), np.uint8)
    ad = np.zeros((max(n, 1), 2), np.uint32)
    fl = np.zeros(max(n, 1), np.uint8)

    def launch(kov):
        capi.check(capi.lib.svjg_genotype_host(
            counts.ctypes.data if counts.size else None, counts.shape[0], idx.ctypes.data, ty.ctypes.data, n, int(min_support),
            la, lb, lh, lut.ctypes.data, LUT_NMAX, kov.ctypes.data if kov is not None else None,
            pl.ctypes.data, gt.ctypes.data, ad.ctypes.data, fl.ctypes.data))

    if n:
        launch(None)
        kov = _k_overrides(fl[:n], ad[:n], n)
        if kov is not None:
            launch(kov)
            if (fl[:n] & capi.GT_NEED_K).any():
                raise RuntimeError("genotype kernel could not represent a likelihood exactly")
    return gt[:n], fl[:n], ad[:n], pl[:n]


_dev_lut = {}


def genotype_device(d_counts, sv_index, svtype, min_support=MIN_SUPPORT, e=ERR, device=None):
    """Runs kernel 4 for len(sv_index) SVs; returns numpy (gt, flags, ad2, pl).
    ``d_counts``: torch int32 [num_sv, 2] on the device (the filter's counters).  ``sv_index`` /
    ``svtype``: numpy arrays, or torch tensors already on the device (int32 view of the uint32
    indices / uint8) when the same catalogue is genotyped again and again."""
    import torch
    dev = d_counts.device if device is None else device
    n = int(len(sv_index))
    if not 0 < e < 1:
        # as in genotype_host: the reference raises only when some record passes the gate (:216)
        out = genotype_device(d_counts, sv_index, svtype, min_support, ERR, device)
        if (out[1] & capi.GT_GENOTYPED).any():
            raise VcfError("error rate must be in (0, 1)")
        return out
    la, lb, lh = math.log10(1 - e), math.log10(e), math.log10(1 / 2)
    lut = _dev_lut.get(str(dev))
    if lut is None:
        lut = _dev_lut[str(dev)] = torch.from_numpy(log10comb_lut()).to(dev)      # constant table: uploaded once
    d_idx = sv_index if isinstance(sv_index, torch.Tensor) else \
        torch.from_numpy(np.ascontiguousarray(sv_index, dtype=np.uint32).view(np.int32)).to(dev)
    d_ty = svtype if isinstance(svtype, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(svtype, dtype=np.uint8)).to(dev)
    d_pl = torch.empty((max(n, 1), 3), dtype=torch.int64, device=dev)
    d_gt = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
    d_ad = torch.empty((max(n, 1), 2), dtype=torch.int32, device=dev)
    d_fl = torch.empty(max(n, 1), dtype=torch.uint8, device=dev)
    stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)

    def launch(k_override):
        capi.check(capi.lib.svjg_genotype_device(
            d_counts.data_ptr(), d_idx.data_ptr(), d_ty.data_ptr(), n, int(min_support), la, lb, lh,
            lut.data_ptr(), LUT_NMAX, k_override.data_ptr() if k_override is not None else None,
            d_pl.data_ptr(), d_gt.data_ptr(), d_ad.data_ptr(), d_fl.data_ptr(), stream))

    launch(None)
    flags = d_fl.cpu().numpy()[:n]
    if (flags & capi.GT_NEED_K).any():
        kov = _k_overrides(flags, d_ad.cpu().numpy().view(np.uint32)[:n], n)
        launch(torch.from_numpy(kov).to(dev))
        flags = d_fl.cpu().numpy()[:n]
        if (flags & capi.GT_NEED_K).any():
            raise RuntimeError("genotype kernel could not represent a likelihood exactly")
    return (d_gt.cpu().numpy()[:n], flags, d_ad.cpu().numpy().view(np.uint32)[:n], d_pl.cpu().numpy()[:n])


def format_vcf(header, recs, gt, flags, ad2, pl):
    """predict-genotype.py:248-271."""
    out = []
    hi = 0
    genotyped = 0
    for i, (head, _code, _key) in enumerate(recs):
        while hi < len(header) and header[hi][0] <= i:
            out.append(header[hi][1])
            hi += 1
        f = int(flags[i])
        if f & capi.GT_GENOTYPED:
            genotyped += 1
            t1, t2 = int(ad2[i, 0]), int(ad2[i, 1])
            h0, h1 = bool(f & capi.GT_HALVED_0), bool(f & capi.GT_HALVED_1)
            sample = (f"{GT_TEXT[gt[i]]}:{_num(t1 + t2, h0 or h1)}:{_num(t1, h0)},{_num(t2, h1)}:"
                      f"{pl[i, 0]},{pl[i, 1]},{pl[i, 2]}")
        else:
            sample = "./.:0:0,0:.,.,."
        out.append(f"{head}\tGT:DP:AD:PL\t{sample}\n")
    while hi < len(header):
        out.append(header[hi][1])
        hi += 1
    return "".join(out), genotyped


def _run_kernel(counts, idx, ty, n, min_support, e):
    if not n:
        return np.zeros(0, np.uint8), np.zeros(0, np.uint8), np.zeros((0, 2), np.uint32), np.zeros((0, 3), np.int64)
    if isinstance(counts, np.ndarray):                            # counters on the host: no tensor library needed
        return genotype_host(counts, idx, ty, min_support, e)
    return genotype_device(counts, idx, ty, min_support, e)


def _emit(text_n, out):
    """The line-by-line statement returns text: written as the text-mode file of the reference would."""
    text, n = text_n
    if out is None:
        return text, n
    import io
    w = io.TextIOWrapper(out, write_through=True)
    w.write(text)
    w.detach()
    return None, n


def genotype_vcf(tables, d_counts, vcf_lines, min_support=MIN_SUPPORT, e=ERR, out=None):
    """decision_vcf (predict-genotype.py:89-279).  ``d_counts``: the filter's counters, a torch int32
    tensor on the device or a numpy uint32 array on the host.  ``vcf_lines``: the VCF as a list of
    lines, or the bytes of the file.  Returns (vcf text, number of genotyped SVs); with ``out`` (a
    binary file object) the text is written there instead of being returned."""
    v = NativeVcf.from_input(vcf_lines)
    if v is not None:
        gt, flags, ad2, pl = _run_kernel(d_counts, v.index_tables(tables), v.svtype, v.n, min_support, e)
        return v.format(gt, flags, ad2, pl, out)
    header, recs = parse_vcf(_as_lines(vcf_lines))
    idx = np.fromiter((capi.NO_SV if r[2] is None else (lambda j: capi.NO_SV if j is None else j)(tables.find_sv(r[2]))
                       for r in recs), dtype=np.uint32, count=len(recs))
    ty = np.fromiter((r[1] for r in recs), dtype=np.uint8, count=len(recs))
    gt, flags, ad2, pl = _run_kernel(d_counts, idx, ty, len(recs), min_support, e)
    return _emit(format_vcf(header, recs, gt, flags, ad2, pl), out)


class AlnCounts:
    """Per-key list lengths of an informative_aln.json (predict-genotype.py:67-68, :219-226),
    read by libsvjg's streaming JSON reader."""

    def __init__(self, handle):
        self._h = C.c_void_p(handle)
        self.num = int(capi.lib.svjg_aln_counts_num(self._h))
        p = capi.lib.svjg_aln_counts_data(self._h)
        if self.num:
            self.counts = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint32)), shape=(self.num, 2)).copy()
        else:
            self.counts = np.zeros((0, 2), np.uint32)

    @classmethod
    def load(cls, path):
        import os
        h = C.c_void_p()
        capi.check(capi.lib.svjg_aln_counts_load(os.fsencode(path), C.byref(h)))
        return cls(h.value)

    @classmethod
    def from_memory(cls, text):
        b = text.encode() if isinstance(text, str) else bytes(text)
        h = C.c_void_p()
        capi.check(capi.lib.svjg_aln_counts_from_memory(b, len(b), C.byref(h)))
        return cls(h.value)

    def key(self, i):
        n = C.c_uint32()
        p = capi.lib.svjg_aln_counts_key(self._h, i, C.byref(n))
        if not p:
            raise IndexError(i)
        return C.string_at(p, n.value).decode("utf-8")

    def find(self, key):
        b = key.encode("utf-8")
        i = capi.lib.svjg_aln_counts_find(self._h, b, len(b))
        return None if i == capi.NO_SV else int(i)

    def close(self):
        if self._h:
            capi.lib.svjg_aln_counts_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def genotype_vcf_from_json(aln_counts, vcf_lines, min_support=MIN_SUPPORT, e=ERR, device=0, out=None):
    """decision_vcf (predict-genotype.py:89-279) with the counters taken from an
    informative_aln.json, as the stand-alone reference stage does.  A key that is
    present gates the SV in even when both of its lists are empty (:216)."""
    counts = aln_counts.counts if aln_counts.num else np.zeros((1, 2), np.uint32)
    v = NativeVcf.from_input(vcf_lines)
    if v is not None:
        idx, ty = v.index_counts(aln_counts)
        gt, flags, ad2, pl = _run_kernel(counts, idx, ty, v.n, min_support, e)
        return v.format(gt, flags, ad2, pl, out)
    header, recs = parse_vcf(_as_lines(vcf_lines))
    n = len(recs)
    idx = np.full(n, capi.NO_SV, dtype=np.uint32)
    ty = np.fromiter((r[1] for r in recs), dtype=np.uint8, count=n)
    for i, r in enumerate(recs):
        if r[2] is None:
            continue
        j = aln_counts.find(r[2])
        if j is None:
            continue
        gated = (ty[i] & 0x3F) <= 3 and not (ty[i] & 0x80) and ty[i] != 255
        if gated and aln_counts.counts[j, 0] == capi.NO_SV:
            raise VcfError(f"informative_aln entry of {r[2]!r} is not a pair of lists (the reference raises here)")
        idx[i] = j
        if ty[i] != 255:
            ty[i] |= 0x40
    gt, flags, ad2, pl = _run_kernel(counts, idx, ty, n, min_support, e)
    return _emit(format_vcf(header, recs, gt, flags, ad2, pl), out)
