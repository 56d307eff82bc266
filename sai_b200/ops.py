"""``torch.ops.sai_b200.*``: the kernels of the hot path as PyTorch custom ops.

A thin registration over the C ABI (``include/sai_b200.h``) for callers that live in a
torch program: tensors own the memory, the ops run on torch's current stream, and the
``sai_layout`` / ``sai_job`` structs travel as CPU uint8 tensors (their raw bytes).  No
computation happens here; ``DeviceScorer`` (scoring.py) calls the same entry points
directly through ctypes.

    import sai_b200.ops                      # registers the ops
    lay = ops.struct_tensor(layout); jb = ops.jobs_tensor(jobs)
    torch.ops.sai_b200.site_flags(packed, lay, jb, n_sites, mask_u, mask_q, qval, 0)
    torch.ops.sai_b200.window_stats(pos, ws, we, jb, mask_u, mask_q, qval, nsnps, u, q, q_cnt,
                                    u_start, q_start, totals, u_cand, q_cand)
    torch.ops.sai_b200.window_stats_pieces(pos, ws, we, first_site, last_site, jb, ...)   # several chromosomes, one launch
    torch.ops.sai_b200.column_quantiles(cols, 0.99, out)                                  # `sai outlier` thresholds
    table, n_text = ops.bgzf_scan_table(bgzip_bytes)                                     # bgzip blocks in HBM
    torch.ops.sai_b200.bgzf_inflate(comp, table, out, status)
"""

from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np
import torch
from torch import Tensor

from . import _cabi


def struct_tensor(obj) -> Tensor:
    """Raw bytes of a ctypes struct / array as a CPU uint8 tensor."""
    return torch.from_numpy(np.frombuffer(bytes(obj), dtype=np.uint8).copy())


def jobs_tensor(jobs: Sequence["_cabi.Job"]) -> Tensor:
    if not 1 <= len(jobs) <= _cabi.MAX_JOBS:
        raise ValueError(f"between 1 and {_cabi.MAX_JOBS} jobs per call")
    return struct_tensor((_cabi.Job * len(jobs))(*jobs))


def _layout_of(t: Tensor) -> "_cabi.Layout":
    if t.device.type != "cpu" or t.dtype != torch.uint8 or t.numel() != C.sizeof(_cabi.Layout):
        raise ValueError("layout must be a CPU uint8 tensor of sizeof(sai_layout) bytes")
    return _cabi.Layout.from_buffer_copy(t.numpy().tobytes())


def _jobs_of(t: Tensor):
    n, rem = divmod(t.numel(), C.sizeof(_cabi.Job))
    if t.device.type != "cpu" or t.dtype != torch.uint8 or rem or not 1 <= n <= _cabi.MAX_JOBS:
        raise ValueError("jobs must be a CPU uint8 tensor of 1..8 sai_job structs")
    return (_cabi.Job * n).from_buffer_copy(t.numpy().tobytes()), n


def _stream(t: Tensor):
    return C.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


@torch.library.custom_op("sai_b200::site_flags", mutates_args=("mask_u", "mask_q", "qval"), device_types="cuda")
def site_flags(packed: Tensor, layout: Tensor, jobs: Tensor, n_sites: int, mask_u: Tensor, mask_q: Tensor,
               qval: Tensor, variant: int) -> None:
    """K1: genotype pass + fused site conditions (sai_site_flags)."""
    lay = _layout_of(layout)
    jarr, n_jobs = _jobs_of(jobs)
    n_tiles = (n_sites + _cabi.TILE_SITES - 1) // _cabi.TILE_SITES
    if mask_u.shape != (n_jobs, max(1, n_tiles)) or mask_q.shape != mask_u.shape or qval.shape[0] != n_jobs:
        raise ValueError("mask_u / mask_q must be [n_jobs, n_tiles] int32 and qval [n_jobs, >= 32 * n_tiles] float64")
    with torch.cuda.device(packed.device):
        _cabi.check(_cabi.load().sai_site_flags(
            C.byref(lay), packed.data_ptr(), 0, n_tiles, n_tiles, jarr, n_jobs, mask_u.data_ptr(), mask_q.data_ptr(),
            qval.data_ptr(), qval.shape[1], None, None, 0, variant, _stream(packed)))


@torch.library.custom_op(
    "sai_b200::window_stats",
    mutates_args=("nsnps", "u", "q", "q_cnt", "u_start", "q_start", "totals", "u_cand", "q_cand"), device_types="cuda")
def window_stats(pos: Tensor, win_start: Tensor, win_end: Tensor, jobs: Tensor, mask_u: Tensor, mask_q: Tensor,
                 qval: Tensor, nsnps: Tensor, u: Tensor, q: Tensor, q_cnt: Tensor, u_start: Tensor, q_start: Tensor,
                 totals: Tensor, u_cand: Tensor, q_cand: Tensor) -> None:
    """K4: per-window N(Variants), U, Q and candidate lists (sai_window_stats)."""
    jarr, n_jobs = _jobs_of(jobs)
    with torch.cuda.device(pos.device):
        _cabi.check(_cabi.load().sai_window_stats(
            pos.data_ptr(), pos.numel(), win_start.data_ptr(), win_end.data_ptr(), win_start.numel(), jarr, n_jobs,
            mask_u.data_ptr(), mask_q.data_ptr(), qval.data_ptr(), qval.shape[1], nsnps.data_ptr(), u.data_ptr(),
            q.data_ptr(), q_cnt.data_ptr(), u_start.data_ptr(), q_start.data_ptr(), totals.data_ptr(),
            u_cand.data_ptr(), u_cand.shape[1], q_cand.data_ptr(), q_cand.shape[1], _stream(pos)))


@torch.library.custom_op(
    "sai_b200::window_stats_pieces",
    mutates_args=("nsnps", "u", "q", "q_cnt", "u_start", "q_start", "totals", "u_cand", "q_cand"), device_types="cuda")
def window_stats_pieces(pos: Tensor, win_start: Tensor, win_end: Tensor, win_first_site: Tensor, win_last_site: Tensor,
                        jobs: Tensor, mask_u: Tensor, mask_q: Tensor, qval: Tensor, nsnps: Tensor, u: Tensor, q: Tensor,
                        q_cnt: Tensor, u_start: Tensor, q_start: Tensor, totals: Tensor, u_cand: Tensor,
                        q_cand: Tensor) -> None:
    """K4 over several chromosome pieces laid side by side: window i is searched only among the
    sites [win_first_site[i], win_last_site[i]) of its own piece (sai_window_stats_pieces)."""
    jarr, n_jobs = _jobs_of(jobs)
    if win_first_site.dtype != torch.int32 or win_last_site.dtype != torch.int32 or \
            win_first_site.numel() != win_start.numel() or win_last_site.numel() != win_start.numel():
        raise ValueError("win_first_site / win_last_site must be int32, one per window")
    with torch.cuda.device(pos.device):
        _cabi.check(_cabi.load().sai_window_stats_pieces(
            pos.data_ptr(), pos.numel(), win_start.data_ptr(), win_end.data_ptr(), win_first_site.data_ptr(),
            win_last_site.data_ptr(), win_start.numel(), jarr, n_jobs, mask_u.data_ptr(), mask_q.data_ptr(),
            qval.data_ptr(), qval.shape[1], nsnps.data_ptr(), u.data_ptr(), q.data_ptr(), q_cnt.data_ptr(),
            u_start.data_ptr(), q_start.data_ptr(), totals.data_ptr(), u_cand.data_ptr(), u_cand.shape[1],
            q_cand.data_ptr(), q_cand.shape[1], _stream(pos)))


@torch.library.custom_op("sai_b200::column_quantiles", mutates_args=("out",), device_types="cuda")
def column_quantiles(cols: Tensor, quantile: float, out: Tensor) -> None:
    """N1: exact linear quantile of every score column (sai_column_quantiles).  ``cols`` is float64
    ``[n_chunks, n_columns, length]`` (the output of one all_gather_into_tensor; NaN = no value) or
    ``[n_columns, length]``; ``out`` float64 ``[n_columns, 4]`` = threshold (NaN if undefined),
    number of values, minimum, maximum."""
    if cols.dtype != torch.float64 or out.dtype != torch.float64 or cols.dim() not in (2, 3) or not cols.is_contiguous():
        raise ValueError("cols must be a contiguous float64 tensor [chunks, columns, length] or [columns, length]")
    n_chunks = cols.shape[0] if cols.dim() == 3 else 1
    n_cols, length = int(cols.shape[-2]), int(cols.shape[-1])
    if tuple(out.shape) != (n_cols, 4) or not out.is_contiguous():
        raise ValueError("out must be a contiguous float64 tensor [columns, 4]")
    with torch.cuda.device(cols.device):
        _cabi.check(_cabi.load().sai_column_quantiles(cols.data_ptr(), n_cols, n_chunks, n_cols * length, length, length,
                                                      float(quantile), out.data_ptr(), _stream(cols)))


BGZF_BLOCK = np.dtype([("comp_off", "<i8"), ("text_off", "<i8"), ("comp_bytes", "<i4"), ("isize", "<i4"), ("crc", "<u4"),
                       ("pad_", "<i4")])  # sai_bgzf_block


def bgzf_scan_table(data) -> tuple[Tensor, int]:
    """Descriptors of every complete BGZF block at the start of ``data`` (bytes-like or a uint8 array:
    the members as they lie in a bgzip file; ``comp`` = the same bytes on the device) and the bytes of
    text they inflate to, laid out block after block.  Built by ``sai_bgzf_scan`` and
    ``sai_bgzf_descriptors``: the payload offsets come from the library's gzip header walk."""
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else np.ascontiguousarray(data, np.uint8)
    lib = _cabi.load()
    tables, at, text = [], 0, 0
    cap = 1 << 16
    boff, ooff, used = np.empty(cap, np.int64), np.empty(cap + 1, np.int64), C.c_int64(0)
    while at < buf.size:
        n = int(lib.sai_bgzf_scan(buf.ctypes.data + at, buf.size - at, cap, 1 << 62, boff.ctypes.data, ooff.ctypes.data,
                                  C.byref(used)))
        _cabi.check(min(n, 0))
        if n == 0:
            break
        t = np.zeros(n, dtype=BGZF_BLOCK)
        _cabi.check(lib.sai_bgzf_descriptors(buf.ctypes.data + at, boff.ctypes.data, ooff.ctypes.data, n, at, text,
                                             t.ctypes.data))
        tables.append(t)
        text += int(ooff[n])
        at += used.value
    t = np.concatenate(tables) if tables else np.zeros(0, dtype=BGZF_BLOCK)
    return torch.from_numpy(t.view(np.uint8).copy()), text


@torch.library.custom_op("sai_b200::bgzf_inflate", mutates_args=("out", "status"), device_types="cuda")
def bgzf_inflate(comp: Tensor, blocks: Tensor, out: Tensor, status: Tensor) -> None:
    """Device inflate of BGZF blocks (sai_bgzf_inflate_device): ``comp`` uint8 CUDA holds the raw
    deflate payloads, ``blocks`` the CPU uint8 descriptor table of ``bgzf_scan_table`` (checked
    against the buffers here), ``out`` uint8 CUDA receives the text, ``status`` int32 CUDA one value
    per block (0 = exact size and matching CRC-32)."""
    n, rem = divmod(blocks.numel(), BGZF_BLOCK.itemsize)
    if blocks.device.type != "cpu" or blocks.dtype != torch.uint8 or rem:
        raise ValueError("blocks must be a CPU uint8 tensor of sai_bgzf_block descriptors")
    if comp.dtype != torch.uint8 or out.dtype != torch.uint8 or status.dtype != torch.int32 or status.numel() < n:
        raise ValueError("comp / out uint8, status int32 with one value per block")
    t = blocks.numpy().view(BGZF_BLOCK)
    if n and ((t["comp_off"] < 0).any() or (t["comp_bytes"] < 0).any() or (t["isize"] < 0).any() or (t["isize"] > 65536).any()
              or (t["text_off"] < 0).any() or (t["comp_off"] + t["comp_bytes"] > comp.numel()).any()
              or (t["text_off"] + t["isize"] > out.numel()).any()):
        raise ValueError("a block descriptor points outside comp / out or claims more than 64 KB of text")
    if n == 0:
        return
    with torch.cuda.device(comp.device):
        d_blocks = blocks.to(comp.device)
        _cabi.check(_cabi.load().sai_bgzf_inflate_device(comp.data_ptr(), d_blocks.data_ptr(), n, out.data_ptr(),
                                                         status.data_ptr(), _stream(comp)))


def vcf_query_tensor(layout, chrom: str, start: int = 1, end: int = 0) -> Tensor:
    """A ``sai_vcf_query`` (the device tables and ``max_column`` are filled in by ``vcf_tiles`` from its
    tensor arguments) as a CPU uint8 tensor; ``start > end`` = no region filter."""
    q = _cabi.VcfQuery()
    q.lay = layout
    q.start, q.end = int(start), int(end)
    name = chrom.encode()
    if not 1 <= len(name) <= 255:
        raise ValueError("chromosome name must be 1..255 bytes")
    q.chrom_len, q.chrom = len(name), name
    return struct_tensor(q)


def vcf_scratch_bytes(query: Tensor, text_bytes: int, sample_column: Tensor) -> int:
    """Bytes of the ``scratch`` tensor ``vcf_tiles`` needs for a text of ``text_bytes`` with these
    sample columns (the genotype pass keeps a row of field offsets up to the largest column)."""
    q = _cabi.VcfQuery.from_buffer_copy(query.numpy().tobytes())
    q.max_column = int(sample_column.max().item()) if sample_column.numel() else 0
    return int(_cabi.load().sai_vcf_scratch_bytes(C.byref(q), int(text_bytes)))


@torch.library.custom_op("sai_b200::vcf_tiles", mutates_args=("scratch", "tiles", "pos", "state"), device_types="cuda")
def vcf_tiles(text: Tensor, query: Tensor, sample_column: Tensor, anc_pos: Tensor, anc_allele: Tensor, scratch: Tensor,
              tiles: Tensor, pos: Tensor, state: Tensor) -> None:
    """Device VCF parse of one slice of complete lines (sai_vcf_tiles_device): ``text`` uint8 CUDA,
    ``query`` from ``vcf_query_tensor``, ``sample_column`` int32 (one VCF column per individual of
    the layout), ``anc_pos`` int32 / ``anc_allele`` uint8 ``[n, 8]`` (empty: no table), ``tiles``
    uint8 of ``sai_packed_bytes`` for ``pos.numel()`` sites (a multiple of 32), ``state`` the 88-byte
    ``sai_vcf_state`` as uint8 (zeroed before the first slice; slices chain through it)."""
    q = _cabi.VcfQuery.from_buffer_copy(query.numpy().tobytes())
    if text.dtype != torch.uint8 or sample_column.dtype != torch.int32 or pos.dtype != torch.int32:
        raise ValueError("text uint8, sample_column / pos int32")
    if state.numel() != C.sizeof(_cabi.VcfState) or sample_column.numel() < 1:
        raise ValueError("state must hold one sai_vcf_state; sample_column one column per individual")
    n_ind = sum(int(q.lay.pop[p].n_samples) for p in range(q.lay.n_pops))
    if sample_column.numel() != n_ind:
        raise ValueError("sample_column must hold one column per individual of the layout")
    q.sample_column = sample_column.data_ptr()
    q.max_column = int(sample_column.max().item())
    q.n_anc = int(anc_pos.numel())
    if q.n_anc:
        if anc_pos.dtype != torch.int32 or anc_allele.numel() != 8 * q.n_anc:
            raise ValueError("anc_pos int32 and anc_allele 8 bytes per entry")
        q.anc_pos, q.anc_allele = anc_pos.data_ptr(), anc_allele.data_ptr()
    with torch.cuda.device(text.device):
        _cabi.check(_cabi.load().sai_vcf_tiles_device(
            C.byref(q), text.data_ptr() if text.numel() else None, text.numel(), scratch.data_ptr(), scratch.numel(),
            tiles.data_ptr(), pos.data_ptr(), pos.numel(), state.data_ptr(), _stream(text)))
