"""ctypes binding of ``include/sai_b200.h`` (the C-ABI drop-in boundary).

The product path has no CPU fallback: if ``libsai_b200.so`` is missing it is
built with nvcc; if that fails, importing this module raises.
"""

from __future__ import annotations

import ctypes as C
from pathlib import Path

from . import build as _build

MAX_POPS = 16
MAX_SRC = 8
MAX_JOBS = 8
TILE_SITES = 32

OK, E_ARG, E_CUDA, E_DOMAIN, E_CAPACITY, E_NOMEM, E_CORRUPT, E_ORDER = 0, -1, -2, -3, -4, -5, -6, -7
MAX_CHROMS = 1024  # SAI_VCF_MAX_CHROMS: chromosomes of one genome ingest
OPS = {"=": 0, "<": 1, ">": 2, "<=": 3, ">=": 4}


class PopLayout(C.Structure):
    _fields_ = [
        ("n_samples", C.c_int32),
        ("ploidy", C.c_int32),
        ("bits", C.c_int32),
        ("pair_off", C.c_int32),
        ("n_pairs", C.c_int32),
        ("n_groups", C.c_int32),
    ]


class Layout(C.Structure):
    _fields_ = [
        ("n_pops", C.c_int32),
        ("pairs_per_site", C.c_int32),
        ("pop", PopLayout * MAX_POPS),
    ]


class Cond(C.Structure):
    _fields_ = [
        ("w", C.c_double),
        ("y", C.c_double * MAX_SRC),
        ("one_minus_y", C.c_double * MAX_SRC),
        ("op", C.c_int32 * MAX_SRC),
        ("enabled", C.c_int32),
        ("pad_", C.c_int32),
    ]


class Job(C.Structure):
    _fields_ = [
        ("ref_pop", C.c_int32),
        ("tgt_pop", C.c_int32),
        ("n_src", C.c_int32),
        ("src_pop", C.c_int32 * MAX_SRC),
        ("anc_allele_available", C.c_int32),
        ("u", Cond),
        ("x", C.c_double),
        ("q", Cond),
        ("quantile", C.c_double),
    ]


class HostResults(C.Structure):
    _fields_ = [
        ("nsnps", C.c_void_p),
        ("u", C.c_void_p),
        ("q", C.c_void_p),
        ("q_cnt", C.c_void_p),
        ("u_start", C.c_void_p),
        ("q_start", C.c_void_p),
        ("totals", C.c_void_p),
        ("u_cand", C.c_void_p),
        ("q_cand", C.c_void_p),
        ("cap_u", C.c_int64),
        ("cap_q", C.c_int64),
    ]


class VcfQuery(C.Structure):
    _fields_ = [
        ("lay", Layout),
        ("sample_column", C.c_void_p),
        ("anc_pos", C.c_void_p),
        ("anc_allele", C.c_void_p),
        ("n_anc", C.c_int64),
        ("start", C.c_int64),
        ("end", C.c_int64),
        ("max_column", C.c_int32),
        ("chrom_len", C.c_int32),
        ("chrom", C.c_char * 256),
    ]


class VcfState(C.Structure):
    _fields_ = [
        ("n_sites", C.c_int64),
        ("overflow", C.c_int32),
        ("pad_", C.c_int32),
        ("vmax", C.c_int32 * MAX_POPS),
    ]


class VcfChrom(C.Structure):
    _fields_ = [
        ("first_pos", C.c_int64),
        ("last_pos", C.c_int64),
        ("n_records", C.c_int64),
        ("first_site", C.c_int64),
        ("n_sites", C.c_int64),
    ]


class FormatInput(C.Structure):
    """``sai_format_input``: the blocks of score rows ``sai_engine_format_scores`` formats."""

    _fields_ = [
        ("n_blocks", C.c_int64),
        ("n_rows", C.c_int64),
        ("block_rows", C.c_void_p),
        ("block_str", C.c_void_p),
        ("strings", C.c_void_p),
        ("strings_len", C.c_int64),
        ("start", C.c_void_p),
        ("end", C.c_void_p),
        ("nsnps", C.c_void_p),
        ("u", C.c_void_p),
        ("u_start", C.c_void_p),
        ("q", C.c_void_p),
        ("q_start", C.c_void_p),
        ("q_cnt", C.c_void_p),
        ("u_cand", C.c_void_p),
        ("q_cand", C.c_void_p),
        ("n_u_cand", C.c_int64),
        ("n_q_cand", C.c_int64),
        ("field", C.c_void_p),
        ("vals", C.c_void_p),
        ("n_fields", C.c_int32),
        ("n_vals", C.c_int32),
    ]


FMT_U, FMT_Q = -1, -2  # SAI_FMT_U / SAI_FMT_Q: the U and Q fields of a score row

TABLE_MAX_COLS = 128  # SAI_TABLE_MAX_COLS
TABLE_TEXT, TABLE_INT, TABLE_FLOAT = 0, 1, 2  # SAI_TABLE_*: a column's dtype
CELL_INT, CELL_FLOAT, CELL_NA, CELL_TEXT, CELL_UNSURE, CELL_BIGINT, CELL_NEGZERO = 1, 2, 4, 8, 16, 32, 64  # SAI_CELL_*
#: SAI_TABLE_* flags of sai_engine_table_load: what the device outlier path does not reproduce
TABLE_FLAGS = {1: "a '\\r' or '\"' in the file", 2: "a byte >= 0x80", 4: "a blank line", 8: "a row without one field per column",
               16: "a line longer than 65535 bytes"}

#: every symbol include/sai_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_I32, _I64, _U64 = C.c_int32, C.c_int64, C.c_uint64
_LAY = C.POINTER(Layout)
_JOB = C.POINTER(Job)
SYMBOLS = {
    "sai_version": (C.c_char_p, []),
    "sai_last_error": (C.c_char_p, []),
    "sai_layout_init": (C.c_int, [_LAY, _I32, _P, _P, _P]),
    "sai_bits_for_max_value": (_I32, [_I32]),
    "sai_num_tiles": (_I64, [_I64]),
    "sai_packed_bytes": (_U64, [_LAY, _I64]),
    "sai_pack_i8": (C.c_int, [_LAY, _I32, _P, _I64, _I64, _P, _I32]),
    "sai_pack_i8_all": (C.c_int, [_LAY, _P, _P, _I64, _P, _I32]),
    "sai_pack_isa": (C.c_char_p, []),
    "sai_pack_i8_isa": (C.c_int, [_LAY, _I32, _P, _I64, _I64, _P, _I32, _I32]),
    "sai_unpack_i8": (C.c_int, [_LAY, _I32, _P, _I64, _I64, _I64, _P, _I64]),
    "sai_neg_table_i8": (_I64, [_P, _I64, _I32, _I64, _P, _P, _P, _I64, _I32]),
    "sai_vcf_parse_gt": (
        _I64,
        [_P, _I64, C.c_char_p, _I64, _I64, _P, _P, _I32, _P, _P, _I64, _P, _P, _I64, _I64, C.POINTER(_I64), _I32],
    ),
    "sai_vcf_chrom_span": (C.c_int, [_P, _I64, C.c_char_p, C.POINTER(_I64), C.POINTER(_I64), C.POINTER(_I64), C.POINTER(_I64), _I32]),
    "sai_is_bgzf": (_I32, [_P, _I64]),
    "sai_bgzf_scan": (_I64, [_P, _I64, _I64, _I64, _P, _P, C.POINTER(_I64)]),
    "sai_bgzf_inflate": (C.c_int, [_P, _P, _P, _I64, _P, _I32]),
    "sai_bgzf_parse_gt": (_I64, [_P, _P, _P, _I64, _I64, C.c_char_p, _I64, _I64, _P, _P, _I32, _P, _P, _I64, _P, _P, _I64, _I64, _I32, _I32]),
    "sai_gzip_inflate": (_I64, [_P, _I64, _P, _I64]),
    "sai_inflate_raw": (_I32, [_P, _I64, _P, _I64]),
    "sai_crc32": (C.c_uint32, [_P, _I64, _I32]),
    "sai_bgzf_inflate_device": (C.c_int, [_P, _P, _I64, _P, _P, _P]),
    "sai_bgzf_descriptors": (C.c_int, [_P, _P, _P, _I64, _I64, _I64, _P]),
    "sai_site_counts": (C.c_int, [_LAY, _P, _I64, _I64, _P, _P, _I64, _I32, _P]),
    "sai_site_flags": (
        C.c_int,
        [_LAY, _P, _I64, _I64, _I64, _JOB, _I32, _P, _P, _P, _I64, _P, _P, _I64, _I32, _P],
    ),
    "sai_flags_from_counts": (C.c_int, [_LAY, _P, _P, _I64, _I64, _JOB, _I32, _P, _P, _P, _I64, _P]),
    "sai_window_stats": (
        C.c_int,
        [_P, _I64, _P, _P, _I64, _JOB, _I32, _P, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _P, _I64, _P],
    ),
    "sai_window_stats_pieces": (
        C.c_int,
        [_P, _I64, _P, _P, _P, _P, _I64, _JOB, _I32, _P, _P, _P, _I64, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _P, _I64, _P],
    ),
    "sai_column_quantiles": (C.c_int, [_P, _I32, _I32, _I64, _I64, _I64, C.c_double, _P, _P]),
    "sai_window_patterns": (
        C.c_int,
        [_LAY, _P, _I64, _P, _P, _I64, _P, _P, _I64, _I32, _I32, _I32, _P, _I32, _P, _P],
    ),
    "sai_engine_pattern_sums": (C.c_int, [_P, _LAY, _I32, _I32, _I32, _P, _I32, _P]),
    "sai_hist_rows": (_I64, [_LAY, _P, _I32]),
    "sai_site_hist": (C.c_int, [_LAY, _P, _I64, _P, _I32, _P, _I64, _P, _P]),
    "sai_window_dd": (
        C.c_int,
        [_LAY, _P, _P, _I64, _P, _P, _I64, _P, _I64, _I32, _I32, _P, _I32, _P, _P, _P, _P, _P, _P, _I32, _P, _P],
    ),
    "sai_engine_dd_sums": (C.c_int, [_P, _LAY, _I32, _I32, _P, _I32, _P, _P, _P, _P, _P, _P, _I32]),
    "sai_engine_create": (C.c_int, [_I32, C.POINTER(_P)]),
    "sai_engine_destroy": (None, [_P]),
    "sai_engine_score_host": (
        C.c_int,
        [_P, _LAY, _P, _P, _I64, _P, _P, _I64, _JOB, _I32, C.POINTER(HostResults)],
    ),
    "sai_engine_score_host_zt": (
        C.c_int,
        [_P, _LAY, _P, _P, _P, _I64, _P, _P, _I64, _JOB, _I32, C.POINTER(HostResults)],
    ),
    "sai_engine_score_host_i8": (
        C.c_int,
        [_P, _LAY, _P, _P, _P, _I64, _P, _P, _I64, _JOB, _I32, C.POINTER(HostResults)],
    ),
    "sai_engine_set_host_threads": (C.c_int, [_P, _I32]),
    "sai_engine_set_i8_wire": (C.c_int, [_P, _I32]),
    "sai_engine_i8_wire_bytes": (_U64, [_P]),
    "sai_engine_score_resident": (C.c_int, [_P, _JOB, _I32, C.POINTER(HostResults)]),
    "sai_engine_rescore_windows": (C.c_int, [_P, C.POINTER(HostResults)]),
    "sai_zt_bound": (_U64, [_LAY, _I64]),
    "sai_zt_encode": (_I64, [_LAY, _P, _I64, _P, _U64, _P, _I32]),
    "sai_zt_encode_isa": (_I64, [_LAY, _P, _I64, _P, _U64, _P, _I32, _I32]),
    "sai_zt_isa": (C.c_char_p, []),
    "sai_zt_pack_i8": (_I64, [_LAY, _P, _P, _I64, _P, _U64, _P, _I32]),
    "sai_zt_decode_host": (C.c_int, [_LAY, _P, _P, _I64, _P]),
    "sai_zt_decode": (C.c_int, [_LAY, _P, _U64, _P, _I64, _I64, _P, _P]),
    "sai_synth_fill": (C.c_int, [_LAY, _P, _I64, _I64, _I64, _P, _U64, C.c_double, _P]),
    "sai_vcf_scratch_bytes": (_U64, [C.POINTER(VcfQuery), _I64]),
    "sai_vcf_tiles_device": (C.c_int, [C.POINTER(VcfQuery), _P, _I64, _P, _U64, _P, _P, _I64, _P, _P]),
    "sai_engine_vcf_begin": (
        C.c_int, [_P, _LAY, C.c_char_p, _I64, _I64, _P, _I32, _P, _P, _I64, _I32, _I64, _I64]),
    "sai_engine_vcf_feed": (C.c_int, [_P, _P, _I64, C.POINTER(_I64)]),
    "sai_engine_vcf_feed_bgzf": (C.c_int, [_P, _P, _P, _P, _I64, _I64]),
    "sai_engine_vcf_feed_bgzf_device": (C.c_int, [_P, _P, _P, _P, _I64, _I64, _I32]),
    "sai_engine_vcf_stats": (C.c_int, [_P, _P, _I32]),
    "sai_engine_vcf_finish": (C.c_int, [_P, C.POINTER(_I64), _P, _P, _I64]),
    "sai_engine_score_loaded": (C.c_int, [_P, _P, _P, _I64, _JOB, _I32, C.POINTER(HostResults)]),
    "sai_engine_set_vcf_slicing": (C.c_int, [_P, _I64, _I32]),
    "sai_engine_vcf_slices": (_I64, [_P]),
    "sai_engine_loaded_tiles": (C.c_int, [_P, _P, _U64]),
    "sai_engine_vcf_genome_begin": (
        C.c_int, [_P, _LAY, _P, _P, _I32, _P, _I32, _P, _P, _P, _I32, _I64, _I64]),
    "sai_engine_vcf_genome_finish": (C.c_int, [_P, C.POINTER(_I64), _P, C.POINTER(VcfChrom), _P, _I64]),
    "sai_engine_score_loaded_pieces": (C.c_int, [_P, _P, _P, _P, _I32, _JOB, _I32, C.POINTER(HostResults)]),
    "sai_engine_set_vcf_neg_table": (C.c_int, [_P, _I32, _I64]),
    "sai_engine_loaded_neg_table": (_I64, [_P, _P, _P, _P, _P, _I64]),
    "sai_engine_dd_sums_loaded": (C.c_int, [_P, _I32, _I32, _P, _I32, _P, _P, _I32]),
    "sai_engine_format_scores": (C.c_int, [_P, C.POINTER(FormatInput), _P]),
    "sai_engine_format_text": (C.c_int, [_P, _I32, _P, _I64]),
    "sai_engine_format_stats": (C.c_int, [_P, _P, _I32]),
    "sai_engine_format_doubles": (C.c_int, [_P, _P, _I64, _P]),
    "sai_format_double": (_I32, [C.c_double, C.c_char_p]),
    "sai_format_doubles": (C.c_int, [_P, _I64, _P]),
    "sai_engine_table_load": (C.c_int, [_P, _P, _I64, _I32, _I64, _P]),
    "sai_engine_table_classes": (C.c_int, [_P, _P, _I64]),
    "sai_engine_table_parse": (C.c_int, [_P, _P, _I32, _I32, _I32, _I32, _P, _P, _P]),
    "sai_engine_table_runs": (C.c_int, [_P, _P, _P, _I64]),
    "sai_engine_table_order": (C.c_int, [_P, _P, _I64]),
    "sai_engine_table_build": (C.c_int, [_P, _P, _P, _P]),
    "sai_engine_table_text": (C.c_int, [_P, _P, _I64]),
    "sai_engine_table_stats": (C.c_int, [_P, _P, _I32]),
    "sai_engine_parse_doubles": (C.c_int, [_P, _P, _P, _I64, _P, _P]),
    "sai_parse_doubles": (C.c_int, [_P, _P, _I64, _P, _P]),
    "sai_classify_cells": (C.c_int, [_P, _P, _I64, _P]),
}

_lib = None


def lib_path() -> Path:
    return _build.LIB


def load() -> C.CDLL:
    """Loads (building if necessary) the C-ABI library and sets prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    import os

    override = os.environ.get("SAI_B200_LIB")  # tools/ A/B scripts: the -DSAI_EXPERIMENTS build
    path = Path(override) if override else _build.build()
    lib = C.CDLL(str(path))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library diverge
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class SaiError(RuntimeError):
    pass


def check(rc: int) -> None:
    """Maps a status code to the exception the reference raises for the same
    condition (``ValueError`` for argument errors)."""
    if rc == OK:
        return
    msg = load().sai_last_error().decode(errors="replace")
    if rc == E_ARG:
        raise ValueError(msg)
    if rc == E_DOMAIN:
        raise ValueError(msg)
    if rc == E_NOMEM:
        raise MemoryError(msg)
    raise SaiError(f"sai_b200 error {rc}: {msg}")
