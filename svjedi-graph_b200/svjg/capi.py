"""ctypes binding of libsvjg.so (include/svjg.h).  No fallback: if the CUDA
library is missing this module raises, and every product path imports it."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), "lib", "libsvjg.so")

OK, E_CUDA, E_ARG, E_IO, E_JSON, E_INPUT, E_HITS_OVERFLOW, E_NOMEM, E_UNSUPPORTED = range(9)
GT_GENOTYPED, GT_HALVED_0, GT_HALVED_1, GT_NEED_K = 1, 2, 4, 8
NO_SV = 0xFFFFFFFF
FLAG_EXACT_CHECKS, FLAG_FORCE_GENERAL = 1, 2
TUNE_TILE_BYTES, TUNE_TILE_LINES, TUNE_SCAN_BLOCKS, TUNE_SCAN_ONLY, TUNE_POOL_UNITS = 1, 2, 3, 4, 5

BAD_REASONS = {
    1: "blank line or fewer than 12 columns",
    2: "non-integer numeric column",
    3: "Alen == 0 without an id:f: tag",
    4: "empty or malformed path column",
    5: "alt node missing from the GFA",
    6: "reference-node name without start-end coordinates",
    7: "svs_edges entry without ':' in the sv id or with a bad allele",
    8: "line shorter than 16 bytes",
    9: "integer with more than 18 digits",
}


class SvjgError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libsvjg error {code}: {message}")
        self.code = code


class FilterStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in
                ("n_hits", "n_records", "n_multi", "n_checks", "status", "err_offset", "n_generic", "n_exact")]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n, _ in self._fields_}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C svjedi-graph_b200/csrc`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, u8p, u32p, u64p, i64p, f64p = (C.c_void_p,) * 6
    sig = {
        "svjg_version": (C.c_char_p, []),
        "svjg_last_error": (C.c_char_p, []),
        "svjg_tables_load": (C.c_int, [C.c_char_p, C.c_char_p, C.POINTER(C.c_void_p)]),
        "svjg_tables_from_memory": (C.c_int, [C.c_char_p, C.c_size_t, C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p)]),
        "svjg_tables_free": (None, [vp]),
        "svjg_tables_num_sv": (C.c_uint32, [vp]),
        "svjg_tables_num_links": (C.c_uint32, [vp]),
        "svjg_tables_num_alt_nodes": (C.c_uint32, [vp]),
        "svjg_tables_device_bytes": (C.c_uint64, [vp]),
        "svjg_tables_alt_node_len": (C.c_int64, [vp, C.c_char_p, C.c_uint32]),
        "svjg_tables_image_hash": (C.c_uint64, [vp]),
        "svjg_tables_sv_id": (C.c_void_p, [vp, C.c_uint32, C.POINTER(C.c_uint32)]),
        "svjg_tables_find_sv": (C.c_uint32, [vp, C.c_char_p, C.c_uint32]),
        "svjg_tables_clone": (C.c_int, [vp, C.POINTER(C.c_void_p)]),
        "svjg_tables_to_device": (C.c_int, [vp, C.c_int]),
        "svjg_tables_set_flags": (C.c_int, [vp, C.c_uint32]),
        "svjg_filter_reset": (C.c_int, [u32p, C.c_uint32, vp, vp]),
        "svjg_filter_device": (C.c_int, [vp, u8p, C.c_uint64, C.c_uint64, C.c_int64, u32p, u32p, u32p, u32p,
                                         C.c_uint64, vp, vp]),
        "svjg_filter_host": (C.c_int, [vp, u8p, C.c_uint64, C.c_int64, u32p, u32p, u64p, u32p, C.c_uint64,
                                       C.POINTER(FilterStats)]),
        "svjg_filter_json_host": (C.c_int, [vp, u8p, C.c_uint64, C.c_int64, u32p, C.POINTER(FilterStats), C.POINTER(C.c_void_p),
                                            C.POINTER(C.c_uint64)]),
        "svjg_hits_min_identity": (C.c_int, [u8p, C.c_uint64, u32p, u64p, u32p, C.POINTER(C.c_uint64), C.c_double, u32p, C.c_uint32]),
        "svjg_translate_newlines": (C.c_uint64, [u8p, C.c_uint64]),
        "svjg_filter_json_begin": (C.c_int, [vp, u8p, C.c_uint64, C.c_int64, u32p, C.POINTER(FilterStats)]),
        "svjg_filter_json_finish": (C.c_int, [vp, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
        "svjg_filter_json_write": (C.c_int, [vp, C.c_char_p, C.c_uint64, C.POINTER(C.c_uint64)]),
        "svjg_filter_json_begin_at": (C.c_int, [vp, u8p, C.c_uint64, C.c_uint64, C.c_int64, u32p, C.POINTER(FilterStats)]),
        "svjg_filter_json_gather": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, u32p]),
        "svjg_filter_tune": (C.c_int, [C.c_int, C.c_int]),
        "svjg_filter_profile": (C.c_int, [C.c_int]),
        "svjg_filter_scan_ms": (C.c_int, [C.POINTER(C.c_float)]),
        "svjg_genotype_device": (C.c_int, [u32p, u32p, u8p, C.c_uint32, C.c_int64, C.c_double, C.c_double,
                                           C.c_double, f64p, C.c_uint32, f64p, i64p, u8p, u32p, u8p, vp]),
        "svjg_genotype_host": (C.c_int, [u32p, C.c_uint32, u32p, u8p, C.c_uint32, C.c_int64, C.c_double, C.c_double,
                                         C.c_double, f64p, C.c_uint32, f64p, i64p, u8p, u32p, u8p]),
        "svjg_cohort_create": (C.c_int, [vp, C.c_uint32, C.POINTER(C.c_void_p)]),
        "svjg_cohort_free": (None, [vp]),
        "svjg_cohort_filter": (C.c_int, [vp, C.c_uint32, u8p, C.c_uint64, C.c_int64, C.POINTER(FilterStats)]),
        "svjg_cohort_read_counts": (C.c_int, [vp, C.c_uint32, u32p]),
        "svjg_cohort_load_counts": (C.c_int, [vp, C.c_uint32, u32p]),
        "svjg_cohort_genotype": (C.c_int, [vp, u32p, u8p, C.c_uint32, C.c_int64, C.c_double, C.c_double, C.c_double, f64p,
                                           C.c_uint32, i64p, u8p, u32p, u8p]),
        "svjg_cohort_site_stats": (C.c_int, [vp, C.c_uint32, u32p, f64p, f64p]),
        "svjg_host_alloc": (C.c_int, [C.c_uint64, C.POINTER(C.c_void_p)]),
        "svjg_host_free": (C.c_int, [vp]),
        "svjg_host_register": (C.c_int, [vp, C.c_uint64]),
        "svjg_host_unregister": (C.c_int, [vp]),
        "svjg_device_init": (C.c_int, [C.c_int]),
        "svjg_xchg_create": (C.c_int, [C.c_uint32, C.POINTER(C.c_void_p), C.c_char_p]),
        "svjg_xchg_open": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
        "svjg_xchg_close": (C.c_int, [vp]),
        "svjg_xchg_free": (C.c_int, [vp]),
        "svjg_xchg_counts": (C.c_void_p, [vp, C.c_uint32, C.c_uint32]),
        "svjg_xchg_signal": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32, vp]),
        "svjg_genotype_xchg": (C.c_int, [C.POINTER(C.c_void_p), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32,
                                         C.c_int, u32p, u8p, C.c_uint32, C.c_int64, C.c_double, C.c_double, C.c_double, f64p,
                                         C.c_uint32, f64p, i64p, u8p, u32p, u8p, vp]),
        "svjg_xchg_timed_out": (C.c_int, [vp, C.POINTER(C.c_uint32)]),
        "svjg_aln_counts_load": (C.c_int, [C.c_char_p, C.POINTER(C.c_void_p)]),
        "svjg_aln_counts_from_memory": (C.c_int, [C.c_char_p, C.c_size_t, C.POINTER(C.c_void_p)]),
        "svjg_aln_counts_free": (None, [vp]),
        "svjg_aln_counts_num": (C.c_uint32, [vp]),
        "svjg_aln_counts_key": (C.c_void_p, [vp, C.c_uint32, C.POINTER(C.c_uint32)]),
        "svjg_aln_counts_data": (C.c_void_p, [vp]),
        "svjg_aln_counts_find": (C.c_uint32, [vp, C.c_char_p, C.c_uint32]),
        "svjg_vcf_parse": (C.c_int, [vp, C.c_size_t, C.c_int, C.POINTER(C.c_void_p)]),
        "svjg_vcf_free": (None, [vp]),
        "svjg_vcf_num_records": (C.c_uint32, [vp]),
        "svjg_vcf_svtype": (C.c_void_p, [vp]),
        "svjg_vcf_key": (C.c_void_p, [vp, C.c_uint32, C.POINTER(C.c_uint32)]),
        "svjg_vcf_index_tables": (C.c_int, [vp, vp, u32p]),
        "svjg_vcf_index_counts": (C.c_int, [vp, vp, u32p, u8p]),
        "svjg_vcf_format": (C.c_int, [vp, u8p, u8p, u32p, i64p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64),
                                      C.POINTER(C.c_uint64)]),
        "svjg_vcf_format_cohort": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_char_p, C.c_uint64, u8p, u8p, u32p,
                                             i64p, C.POINTER(C.c_void_p), C.POINTER(C.c_uint64), u64p]),
        "svjg_vcf_format_cohort_tags": (C.c_int, [vp, C.c_uint32, C.c_uint32, C.c_uint32, C.c_char_p, C.c_uint64, u8p, u8p,
                                                  u32p, i64p, C.c_uint32, u32p, f64p, f64p, C.POINTER(C.c_void_p),
                                                  C.POINTER(C.c_uint64), u64p]),
        "svjg_buffer_free": (None, [vp]),
        "svjg_emit_informative_json": (C.c_int, [vp, u8p, C.c_uint64, u32p, u64p, u32p, C.c_uint64, C.c_char_p]),
        "svjg_emit_informative_json_mem": (C.c_int, [vp, u8p, C.c_uint64, u32p, u64p, u32p, C.c_uint64,
                                                     C.POINTER(C.c_void_p), C.POINTER(C.c_uint64)]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib, tuple(sig)


lib, EXPORTS = _load()


def check(rc):
    if rc != OK:
        raise SvjgError(rc, lib.svjg_last_error().decode("utf-8", "replace"))
