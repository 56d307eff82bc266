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


def outlier(score_file: str, output_prefix: str, quantile: float, group=None) -> None:
    """Reads a score TSV, writes one ``{prefix}.{column}.{quantile}.outliers.tsv``
    per metric column.  With an initialised process group every rank passes the
    score file of its own shard and all ranks use the same genome-wide
    thresholds (one small all-gather per column); each rank writes the outlier
    rows of its own shard."""
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
