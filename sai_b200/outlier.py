"""Genome-wide outlier thresholds (``sai outlier``), single- and multi-GPU.

Mirrors ``outlier()`` (sai/sai.py:154-230): for every metric column (everything
after ``N(Variants)``) the threshold is the linear quantile of the column's
non-NaN values; rows are kept with ``>`` for columns whose name starts with
"U" and ``>=`` otherwise; a column that is empty or has one unique value gives
an empty table (with a warning); output rows are naturally sorted by
Chrom/Start/End and written as ``{prefix}.{column}.{q}.outliers.tsv``.

Multi-GPU: every rank holds the score rows of its own window ranges; the
genome-wide threshold is the same on all ranks after ONE small all-gather of
the per-rank column values.  On GPUs (``device_thresholds``) the score arrays
never leave the device: one ``all_gather_into_tensor`` over NVLink for ALL
columns, then ``sai_column_quantiles`` selects the order statistics exactly
(radix select on the float64 bit patterns) -- no host copy, no sort.  The gloo
path (CPU tests) gathers U counts as a histogram and Q values as padded arrays.
"""

from __future__ import annotations

import ctypes
import re
import warnings
from typing import Optional, Sequence

import numpy as np


# --------------------------------------------------------------------------
# thresholds
# --------------------------------------------------------------------------
def linear_quantile_sorted(v: np.ndarray, q: float) -> float:
    """numpy 'linear' quantile of an already sorted, NaN-free float64 vector
    (pandas ``Series.quantile`` reduces to this; see oracle.quantile_linear)."""
    n = v.size
    vi = np.float64(n - 1) * np.float64(q)
    if vi >= n - 1:
        # numpy lerps the last value with itself: top for a finite top, NaN for +inf
        top = np.float64(v[-1])
        with np.errstate(invalid="ignore"):
            return float(top + (top - top))
    lo = int(np.floor(vi))
    g = np.float64(vi - lo)
    a, b = np.float64(v[lo]), np.float64(v[lo + 1])
    d = np.float64(b - a)
    return float(b - np.float64(d * np.float64(1 - g))) if g >= 0.5 else float(a + np.float64(d * g))


def threshold_from_values(values: np.ndarray, q: float) -> Optional[float]:
    v = np.asarray(values, dtype=np.float64)
    v = np.sort(v[~np.isnan(v)])
    if v.size == 0 or v[0] == v[-1]:
        return None
    return linear_quantile_sorted(v, q)


def threshold_from_histogram(counts: np.ndarray, q: float) -> Optional[float]:
    """Exact linear quantile of integer data given ``counts[k]`` = number of
    values equal to ``k``."""
    counts = np.asarray(counts, dtype=np.int64)
    n = int(counts.sum())
    if n == 0 or np.count_nonzero(counts) == 1:
        return None
    cum = np.cumsum(counts)
    vi = np.float64(n - 1) * np.float64(q)
    if vi >= n - 1:
        return float(np.flatnonzero(counts)[-1])
    lo = int(np.floor(vi))
    g = np.float64(vi - lo)
    a = np.float64(np.searchsorted(cum, lo, side="right"))  # value of the lo-th order statistic
    b = np.float64(np.searchsorted(cum, lo + 1, side="right"))
    d = np.float64(b - a)
    return float(b - np.float64(d * np.float64(1 - g))) if g >= 0.5 else float(a + np.float64(d * g))


def device_thresholds(cols, q: float, group=None, max_len: Optional[int] = None) -> list[Optional[float]]:
    """Genome-wide thresholds of ``C`` score columns resident on the GPU.

    ``cols``: float64 CUDA tensor ``[C, n_local]`` -- this rank's values of every column (U counts
    as exact doubles, Q values; NaN = window without a value).  With an initialised NCCL group the
    ranks' arrays are padded to ``max_len`` (the largest ``n_local``; found with one tiny MAX
    all-reduce unless the caller knows it from the sharding) and exchanged with ONE
    ``all_gather_into_tensor``; ``sai_column_quantiles`` then computes every column's linear
    quantile on the device, identically on every rank.  One 32-byte-per-column read comes back.
    ``None`` = empty or single-valued column (the reference writes an empty table, sai.py:195-207)."""
    import ctypes as C

    import torch
    import torch.distributed as dist

    from . import _cabi

    if cols.dtype != torch.float64 or cols.dim() != 2 or not cols.is_cuda:
        raise ValueError("cols must be a float64 CUDA tensor [columns, values]")
    n_cols, n_local = int(cols.shape[0]), int(cols.shape[1])
    world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
    out = torch.empty((max(n_cols, 1), 4), dtype=torch.float64, device=cols.device)
    stream = C.c_void_p(torch.cuda.current_stream(cols.device).cuda_stream)
    lib = _cabi.load()
    if world == 1:
        src = cols.contiguous()
        _cabi.check(lib.sai_column_quantiles(src.data_ptr(), n_cols, 1, 0, n_local, n_local, float(q), out.data_ptr(), stream))
    else:
        if max_len is None:
            m = torch.tensor([n_local], dtype=torch.int64, device=cols.device)
            dist.all_reduce(m, op=dist.ReduceOp.MAX, group=group)
            max_len = int(m.item())
        if n_local == max_len:
            mine = cols.contiguous()
        else:
            mine = torch.full((n_cols, max_len), float("nan"), dtype=torch.float64, device=cols.device)
            mine[:, :n_local] = cols
        gathered = torch.empty((world, n_cols, max_len), dtype=torch.float64, device=cols.device)
        dist.all_gather_into_tensor(gathered, mine, group=group)
        _cabi.check(lib.sai_column_quantiles(gathered.data_ptr(), n_cols, world, n_cols * max_len, max_len, max_len,
                                             float(q), out.data_ptr(), stream))
    thr = out[:n_cols, 0].cpu().numpy()  # the one host read (synchronises)
    return [None if np.isnan(t) else float(t) for t in thr]


def distributed_threshold(local_values: np.ndarray, q: float, column: str, group=None, device=None) -> Optional[float]:
    """Genome-wide threshold of one metric column whose rows are spread over
    the ranks of ``group``; identical on every rank.  Host-array interface (the file-level
    ``outlier``); with an NCCL group the values go through ``device_thresholds``."""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return threshold_from_values(local_values, q)
    world = dist.get_world_size(group)
    if dist.get_backend(group) == "nccl":
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else device
        v = torch.from_numpy(np.ascontiguousarray(local_values, dtype=np.float64)).to(dev)
        return device_thresholds(v.reshape(1, -1), q, group)[0]
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    v = np.asarray(local_values, dtype=np.float64)
    v = v[~np.isnan(v)]
    is_count = column.startswith("U") and (v.size == 0 or np.all(v == np.floor(v)))
    # one tiny reduction fixes the message size, then ONE all-gather carries the data
    meta = torch.tensor([v.size, int(v.max()) + 1 if (is_count and v.size) else 0, 0 if is_count else 1],
                        dtype=torch.int64, device=device)
    dist.all_reduce(meta, op=dist.ReduceOp.MAX, group=group)
    max_n, n_bins, any_float = (int(x) for x in meta.tolist())
    if not any_float:
        hist = torch.zeros(max(n_bins, 1), dtype=torch.int64, device=device)
        if v.size:
            hist += torch.from_numpy(np.bincount(v.astype(np.int64), minlength=max(n_bins, 1))).to(device)
        gathered = [torch.empty_like(hist) for _ in range(world)]
        dist.all_gather(gathered, hist, group=group)
        return threshold_from_histogram(torch.stack(gathered).sum(0).cpu().numpy(), q)
    buf = torch.full((max(max_n, 1),), float("nan"), dtype=torch.float64, device=device)
    if v.size:
        buf[: v.size] = torch.from_numpy(v).to(device)
    gathered = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(gathered, buf, group=group)
    return threshold_from_values(torch.cat(gathered).cpu().numpy(), q)


def outlier_mask(values: np.ndarray, thr: Optional[float], column: str) -> np.ndarray:
    v = np.asarray(values, dtype=np.float64)
    if thr is None:
        return np.zeros(v.shape, dtype=bool)
    with np.errstate(invalid="ignore"):
        return (v > thr) if column.startswith("U") else (v >= thr)


# --------------------------------------------------------------------------
# file level (sai/sai.py:154-230)
# --------------------------------------------------------------------------
def _natural_key(s: str):
    return [int(t) if t.isdigit() else t for t in re.split(r"(\d+)", str(s))]


class ScoreTable:
    """A score TSV read exactly like the reference reads it
    (``pd.read_csv(sep="\\t", na_values=["nan"], index_col=False)``,
    sai/sai.py:175 -- including pandas' default float parser, whose last-digit
    rounding shows in the output text) and written back cell by cell the way
    ``DataFrame.astype(str).to_csv`` of the pinned pandas 2.2.1 does: integer
    columns as integers, float columns as ``str(float)`` with ``nan`` for
    missing cells, text columns unchanged with ``nan`` for missing cells
    (that is why the reference's outlier tables show ``nan`` under Outgroup)."""

    def __init__(self, path: str):
        import pandas as pd

        self.pd = pd
        self.df = pd.read_csv(path, sep="\t", na_values=["nan"], index_col=False)
        self.columns = list(self.df.columns)
        self.n_rows = len(self.df)
        self._cols = [self.df[c].to_numpy(dtype=object) for c in self.columns]
        self._kind = [self.df[c].dtype.kind if hasattr(self.df[c].dtype, "kind") else "O" for c in self.columns]

    def numeric(self, col: str) -> np.ndarray:
        return self.pd.to_numeric(self.df[col], errors="coerce").to_numpy(dtype=np.float64)

    def cell(self, r: int, col: str):
        return self._cols[self.columns.index(col)][r]

    def format_cell(self, r: int, c: int) -> str:
        v = self._cols[c][r]
        k = self._kind[c]
        if k in "iu":
            return str(int(v))
        if k == "b":
            return str(bool(v))
        if self.pd.isna(v):
            return "nan"
        if k == "f":
            return str(float(v))
        return str(v)


TEXT_MODES = ("host", "device")


def pandas_chunk_rows(n_cols: int) -> int:
    """Rows per chunk of pandas' C parser (``low_memory=True``) for a table of ``n_cols`` columns: it
    infers one dtype per chunk and column and concatenates the chunks, so a column that is int64 in
    one chunk and text in another holds Python ints and strings (with a DtypeWarning)."""
    heuristic = 2**20 // n_cols
    rows = 1
    while rows * 2 < heuristic:
        rows *= 2
    return rows


def column_kinds(classes: np.ndarray) -> tuple[Optional[list[int]], Optional[str]]:
    """pandas' dtype of every column (``_cabi.TABLE_TEXT`` / ``_INT`` / ``_FLOAT``) from the OR of its
    cells' ``SAI_CELL_*`` classes per parse chunk, ``[chunks, columns]``; or the reason the device
    path cannot reproduce it.  A chunk with a text cell is text, one of integers only int64, any
    other float64 (an all-NA chunk too); int64 and float64 chunks concatenate to float64; text with
    anything else is a column of mixed objects.  pandas reads the integers of a float64 column either
    as int64 (cast) or with its float parser, which differ beyond 2^53, past 17 digits (leading zeros
    included) and on "-0"; such a column is left to the host path."""
    from . import _cabi

    odd_int = _cabi.CELL_BIGINT | _cabi.CELL_NEGZERO
    kinds = []
    for c in range(classes.shape[1]):
        col = classes[:, c]
        if np.any(col & _cabi.CELL_UNSURE):
            return None, f"column {c + 1} has a cell whose pandas type or value is not reproduced"
        chunk = {(_cabi.TABLE_TEXT if m & _cabi.CELL_TEXT else
                  _cabi.TABLE_INT if m & ~odd_int == _cabi.CELL_INT else _cabi.TABLE_FLOAT) for m in col.tolist()}
        if chunk == {_cabi.TABLE_INT, _cabi.TABLE_FLOAT}:
            chunk = {_cabi.TABLE_FLOAT}
        if len(chunk) > 1:
            return None, f"column {c + 1} has parse chunks of different pandas types"
        kinds.append(chunk.pop())
        if kinds[-1] == _cabi.TABLE_FLOAT and np.any(col & odd_int):
            return None, f"column {c + 1} is float64 with an integer beyond 2^53, of more than 17 digits or -0"
    return kinds, None


class _DeviceFile:
    """A score file loaded and classified on the device (``_load_device``)."""

    def __init__(self, data: bytes, names: list[str], engine, n_rows: int, kinds: list[int]):
        self.data, self.names, self.engine, self.n_rows, self.kinds = data, names, engine, n_rows, kinds
        self.first_metric = names.index("N(Variants)") + 1
        self.chrom, self.start, self.end = (names.index(c) for c in ("Chrom", "Start", "End"))


def _load_device(data: bytes, quantile: float, group, device: int, timings: Optional[dict]):
    """(reason, None) when the file has to be read on the host, else (None, ``_DeviceFile``)."""
    import torch.distributed as dist

    if not 0.0 <= quantile <= 1.0:
        return "quantile outside [0, 1]", None
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1 \
            and dist.get_backend(group) != "nccl":
        return "a process group that is not NCCL", None
    nl = data.find(b"\n")
    if nl < 0:
        return "no data rows", None
    names_b = data[:nl].split(b"\t")
    if any(not n for n in names_b):
        return "an empty column name", None
    if len(set(names_b)) != len(names_b):
        return "duplicate column names", None
    if any(b < 0x21 or b > 0x7E for n in names_b for b in n):
        return "a column name with bytes outside printable ASCII", None
    if len(names_b) > 128:
        return "more than 128 columns", None
    names = [n.decode() for n in names_b]
    if "N(Variants)" not in names:
        return "no N(Variants) column", None
    if names[-1] == "N(Variants)":
        return "no metric columns", None
    if not {"Chrom", "Start", "End"} <= set(names):
        return "no Chrom, Start or End column", None
    from . import _cabi
    from .scoring import HostEngine

    eng = HostEngine(device)
    n_rows, n_chunks, flags = eng.table_load(data, len(names), pandas_chunk_rows(len(names)))
    if timings is not None:
        timings.update(eng.table_stats())
    reason = next((why for bit, why in _cabi.TABLE_FLAGS.items() if flags & bit), None)
    if reason is None and n_rows == 0:
        reason = "no data rows"
    kinds = None
    if reason is None:
        classes = eng.table_classes(n_chunks, len(names))
        kinds, reason = column_kinds(classes)
    if reason is None:
        f = _DeviceFile(data, names, eng, n_rows, kinds)
        chrom_cls = int(np.bitwise_or.reduce(classes[:, f.chrom]))
        if any(k == _cabi.TABLE_TEXT for k in kinds[f.first_metric:]):
            reason = "a text metric column"
        elif kinds[f.start] != _cabi.TABLE_INT or kinds[f.end] != _cabi.TABLE_INT:
            reason = "Start or End is not int64"
        elif kinds[f.chrom] == _cabi.TABLE_FLOAT or chrom_cls & _cabi.CELL_NA:
            reason = "Chrom has NA cells or is float64"
        else:
            return None, f
    eng.close()
    return reason, None


def fallback_reason(score_file: str, quantile: float, group=None, device: int = 0) -> Optional[str]:
    """Why ``outlier(..., text="device")`` reads ``score_file`` on the host (``None``: it builds the
    tables on the device), for this rank alone.  The host path takes every file whose pandas
    dtypes, values or errors the device path does not reproduce exactly."""
    with open(score_file, "rb") as fh:
        data = fh.read()
    reason, f = _load_device(data, quantile, group, device, None)
    if f is not None:
        f.engine.close()
    return reason


def _ranks_agree(ok: bool, header: bytes, group, device: int) -> bool:
    """With an NCCL group of several ranks: True when every rank takes the device path and all read
    the same column names (one MIN all-reduce), so that no rank waits in a collective another rank
    never enters."""
    import zlib

    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1 \
            or dist.get_backend(group) != "nccl":
        return ok
    h = (zlib.crc32(header) << 20) | min(len(header), (1 << 20) - 1)
    t = torch.tensor([int(ok), h, -h], dtype=torch.int64, device=torch.device("cuda", device))
    dist.all_reduce(t, op=dist.ReduceOp.MIN, group=group)
    ok_all, lo, neg_hi = t.tolist()
    return ok_all == 1 and lo == -neg_hi


def device_outlier(score_file: str, output_prefix: str, quantile: float, group=None, device: int = 0,
                   timings: Optional[dict] = None) -> bool:
    """``outlier`` with the score file parsed and the tables built as text on the GPU; returns False
    (having written nothing) when the file needs the host path (``fallback_reason``).  ``timings``,
    if given, receives the seconds of every phase."""
    import time

    import torch
    import torch.distributed as dist

    from . import _cabi

    t0 = time.perf_counter()
    with open(score_file, "rb") as fh:
        data = fh.read()
    t_read = time.perf_counter() - t0
    reason, f = _load_device(data, quantile, group, device, timings)
    nl = data.find(b"\n")
    if not _ranks_agree(reason is None, data[:nl] if nl >= 0 else data, group, device):
        if f is not None:
            f.engine.close()
        return False
    eng = f.engine
    try:
        dev = torch.device("cuda", device)
        metric = f.names[f.first_metric:]
        n_metric = len(metric)
        with torch.cuda.device(dev):
            vals = torch.empty((n_metric, f.n_rows), dtype=torch.float64, device=dev)
            first, n_runs = eng.table_parse(f.kinds, f.first_metric, f.chrom, f.start, f.end, vals)
            # natural order of the chromosome names: ranked on the host with the host path's key
            off, ln = eng.table_runs(n_runs)
            names = [data[o:o + n].decode() for o, n in zip(off.tolist(), ln.tolist())]
            if f.kinds[f.chrom] == _cabi.TABLE_INT:
                names = [str(int(n)) for n in names]
            keys = {n: _natural_key(n) for n in set(names)}
            rank, last = {}, None
            for n in sorted(keys, key=keys.get):
                rank[n] = rank[last] + (keys[n] != keys[last]) if last is not None else 0
                last = n
            eng.table_order(np.array([rank[n] for n in names], dtype=np.int32))
            t1 = time.perf_counter()
            if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
                found = device_thresholds(vals, quantile, group)  # one all-gather for every column
                none = [t is None for t in found]
                thr = [np.nan if t is None else t for t in found]
            else:
                out = torch.empty((n_metric, 4), dtype=torch.float64, device=dev)
                stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                _cabi.check(_cabi.load().sai_column_quantiles(vals.data_ptr(), n_metric, 1, 0, f.n_rows, f.n_rows,
                                                              float(quantile), out.data_ptr(), stream))
                o = out.cpu().numpy()
                # threshold_from_values: no threshold for an empty or single-valued column
                none = [bool(o[m, 1] == 0 or o[m, 2] == o[m, 3]) for m in range(n_metric)]
                thr = [np.nan if none[m] else float(o[m, 0]) for m in range(n_metric)]
            t_thr = time.perf_counter() - t1
            text, offs = eng.table_build(thr, [c.startswith("U") for c in metric])
        if timings is not None:
            timings.update(eng.table_stats())
        t2 = time.perf_counter()
        view = memoryview(text)
        for m, col in enumerate(metric):
            if none[m]:
                if np.isnan(first[m]):
                    warnings.warn(f"Column '{col}' has no numeric values; writing empty result.", UserWarning)
                else:
                    warnings.warn(f"Column '{col}' has only one unique value ({np.float64(first[m])}); writing empty result.",
                                  UserWarning)
            with open(f"{output_prefix}.{col}.{quantile}.outliers.tsv", "wb") as fh:
                fh.write(view[offs[m]:offs[m + 1]])
        if timings is not None:
            timings.update(read_s=t_read, thresholds_s=t_thr, write_s=time.perf_counter() - t2)
    finally:
        eng.close()
    return True


def outlier(score_file: str, output_prefix: str, quantile: float, group=None, text: str = "host",
            device: int = 0) -> None:
    """Reads a score TSV, writes one ``{prefix}.{column}.{quantile}.outliers.tsv``
    per metric column.  With an initialised process group every rank passes the
    score file of its own shard and all ranks use the same genome-wide
    thresholds (one small all-gather per column); each rank writes the outlier
    rows of its own shard.

    ``text="device"`` parses the file and builds the tables as text on GPU ``device``
    (``device_outlier``): the same files, warnings and errors, with one all-gather for all
    columns under NCCL.  A file whose pandas reading it does not reproduce exactly, and a gloo
    group, take the host path (``fallback_reason``)."""
    if text not in TEXT_MODES:
        raise ValueError(f"text must be 'host' or 'device', not {text!r}")
    if text == "device" and device_outlier(score_file, output_prefix, quantile, group, device):
        return
    tab = ScoreTable(score_file)
    cols = tab.columns
    if "N(Variants)" in cols:
        metric_cols = cols[cols.index("N(Variants)") + 1 :]
    else:
        non_metrics = {"Chrom", "Start", "End", "Ref", "Tgt", "Src"}
        metric_cols = [c for c in cols if c not in non_metrics and not np.all(np.isnan(tab.numeric(c)))]
    if not metric_cols:
        raise ValueError("No metric columns found.")
    ci = {name: cols.index(name) for name in ("Chrom", "Start", "End") if name in cols}
    for col in metric_cols:
        vals = tab.numeric(col)
        thr = distributed_threshold(vals, quantile, col, group)
        keep: list[int] = []
        if thr is None:
            finite = vals[~np.isnan(vals)]
            if finite.size == 0:
                warnings.warn(f"Column '{col}' has no numeric values; writing empty result.", UserWarning)
            else:
                warnings.warn(f"Column '{col}' has only one unique value ({finite[0]}); writing empty result.", UserWarning)
        else:
            keep = [int(i) for i in np.flatnonzero(outlier_mask(vals, thr, col))]
            if keep:
                if len(ci) < 3:
                    missing = {"Chrom", "Start", "End"} - set(ci)
                    raise ValueError(f"Missing required columns: {', '.join(missing)}")
                keep.sort(key=lambda i: (_natural_key(tab.cell(i, "Chrom")), int(tab.cell(i, "Start")),
                                         int(tab.cell(i, "End"))))
        with open(f"{output_prefix}.{col}.{quantile}.outliers.tsv", "w") as f:
            f.write("\t".join(cols) + "\n")
            for i in keep:
                f.write("\t".join(tab.format_cell(i, c) for c in range(len(cols))) + "\n")
