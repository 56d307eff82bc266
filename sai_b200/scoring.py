"""Python host layer over the C ABI: jobs, the host-buffer engine and the
device-resident scorer.

Nothing here computes a statistic on the CPU -- every number comes from the
CUDA kernels behind ``libsai_b200.so``.
"""

from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _cabi
from .encode import MatrixGenotypes, PackedGenotypes, ZtGenotypes


# --------------------------------------------------------------------------
# jobs
# --------------------------------------------------------------------------
def _fill_cond(cond: "_cabi.Cond", w: float, y_list: Sequence[tuple[str, float]]) -> None:
    # same checks, same messages as compute_matching_loci (stat_utils.py:99-108)
    if not (0 <= w <= 1):
        raise ValueError("Parameters w must be within the range [0, 1].")
    for op, y in y_list:
        if not (0 <= y <= 1):
            raise ValueError(f"Invalid value in y_list: {y}. within the range [0, 1].")
        if op not in _cabi.OPS:
            raise ValueError(
                f"Invalid operator in y_list: {op}. Must be '=', '<', '>', '<=', or '>='."
            )
    cond.w = float(w)
    for k, (op, y) in enumerate(y_list):
        cond.y[k] = float(y)
        cond.one_minus_y[k] = 1 - y  # Python float arithmetic, as stat_utils.py:149
        cond.op[k] = _cabi.OPS[op]
    cond.enabled = 1


def make_job(
    ref_pop: int,
    tgt_pop: int,
    src_pops: Sequence[int],
    anc_allele_available: bool,
    u: Optional[dict] = None,
    q: Optional[dict] = None,
) -> "_cabi.Job":
    """``u = {"w", "x", "y_list"}``, ``q = {"w", "quantile", "y_list"}`` -- the
    keyword arguments ``UStatistic.compute`` / ``QStatistic.compute`` receive
    (sai/preprocessors/feature_preprocessor.py:163-186)."""
    if len(src_pops) > _cabi.MAX_SRC:
        raise ValueError(f"at most {_cabi.MAX_SRC} source populations")
    job = _cabi.Job()
    job.ref_pop, job.tgt_pop, job.n_src = int(ref_pop), int(tgt_pop), len(src_pops)
    for k, s in enumerate(src_pops):
        job.src_pop[k] = int(s)
    job.anc_allele_available = 1 if anc_allele_available else 0
    for name, spec in (("u", u), ("q", q)):
        if spec is None:
            continue
        if len(spec["y_list"]) != len(src_pops):
            raise ValueError("The length of src_gts_list and y_list must match.")
        _fill_cond(getattr(job, name), spec["w"], spec["y_list"])
    if u is not None:
        job.x = float(u["x"])
    if q is not None:
        qq = float(q["quantile"])
        if not (0 <= qq <= 1):
            raise ValueError("Quantiles must be in the range [0, 1]")
        job.quantile = qq
    return job


def _job_array(jobs: Sequence["_cabi.Job"]):
    if not 1 <= len(jobs) <= _cabi.MAX_JOBS:
        raise ValueError(f"between 1 and {_cabi.MAX_JOBS} jobs per call")
    return (_cabi.Job * len(jobs))(*jobs)


def _bounds(windows: Sequence[tuple[int, int]]) -> tuple[np.ndarray, np.ndarray]:
    """The windows' starts and ends as two int64 arrays."""
    ws = np.ascontiguousarray([w[0] for w in windows], dtype=np.int64)
    we = np.ascontiguousarray([w[1] for w in windows], dtype=np.int64)
    return ws, we


def _ptr(a: np.ndarray):
    return a.ctypes.data if a.size else None


# --------------------------------------------------------------------------
# results
# --------------------------------------------------------------------------
@dataclass
class WindowResults:
    """Per job ``j`` and window ``i``.  A window's candidate positions are the
    ``u[j, i]`` (resp. ``q_cnt[j, i]``) entries of ``u_cand[j]`` (``q_cand[j]``)
    starting at ``u_start[j, i]`` (``q_start[j, i]``), in genome order."""

    nsnps: np.ndarray  # int32 [J, W]
    u: np.ndarray  # int64 [J, W]
    q: np.ndarray  # float64 [J, W], NaN where no site matches
    q_cnt: np.ndarray  # int32 [J, W]
    u_start: np.ndarray  # int64 [J, W]
    q_start: np.ndarray  # int64 [J, W]
    totals: np.ndarray  # int64 [J, 2]
    u_cand: np.ndarray  # int32 [J, cap_u] positions
    q_cand: np.ndarray

    def u_positions(self, j: int, i: int) -> np.ndarray:
        s = int(self.u_start[j, i])
        return self.u_cand[j, s : s + int(self.u[j, i])]

    def q_positions(self, j: int, i: int) -> np.ndarray:
        s = int(self.q_start[j, i])
        return self.q_cand[j, s : s + int(self.q_cnt[j, i])]


# --------------------------------------------------------------------------
# host-buffer engine (HOST pointers in, HOST results out)
# --------------------------------------------------------------------------
class HostEngine:
    """One per GPU / worker process.  Created lazily so that an object holding
    it can be pickled to worker processes before any CUDA context exists
    (the reference pickles its preprocessor, sai/multiprocessing/mp_manager.py:153-164)."""

    def __init__(self, device: int = 0):
        self.device = int(device)
        self._h = None

    def _handle(self):
        if self._h is None:
            h = C.c_void_p()
            _cabi.check(_cabi.load().sai_engine_create(self.device, C.byref(h)))
            self._h = h
        return self._h

    def close(self):
        if self._h is not None:
            _cabi.load().sai_engine_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __getstate__(self):
        return {"device": self.device}

    def __setstate__(self, st):
        self.device = st["device"]
        self._h = None

    def score(
        self,
        pg: PackedGenotypes,
        windows: Sequence[tuple[int, int]],
        jobs: Sequence["_cabi.Job"],
        cap_u: Optional[int] = None,
        cap_q: Optional[int] = None,
    ) -> WindowResults:
        return self.score_arrays(pg, *_bounds(windows), jobs, cap_u, cap_q)

    def set_host_threads(self, n_threads: int) -> None:
        """Host threads of the int8 pipeline (``score_matrices``); <= 0: all cores."""
        _cabi.check(_cabi.load().sai_engine_set_host_threads(self._handle(), int(n_threads)))

    def set_i8_wire(self, mode: str = "auto") -> None:
        """Wire format of the int8 pipeline: ``"zt"`` records built by the packers, ``"dense"`` tiles
        (data without a hom-ref majority) or ``"auto"`` (default: zt when the CPU has the vector
        record encoder).  Same results either way."""
        _cabi.check(_cabi.load().sai_engine_set_i8_wire(self._handle(), {"auto": 0, "dense": 1, "zt": 2}[mode]))

    def i8_wire_bytes(self) -> int:
        """Tile bytes the last int8 call copied to the GPU."""
        return int(_cabi.load().sai_engine_i8_wire_bytes(self._handle()))

    def score_arrays(self, pg, ws, we, jobs, cap_u=None, cap_q=None) -> WindowResults:
        """``pg``: ``PackedGenotypes`` (dense tiles), ``ZtGenotypes`` (zero-suppressed wire format)
        or ``MatrixGenotypes`` (int8 matrices: packed by host threads slice by slice while earlier
        slices are on the wire and in the genotype pass, ``sai_engine_score_host_i8``)."""
        pos = np.ascontiguousarray(pg.pos, dtype=np.int32)
        if isinstance(pg, ZtGenotypes):  # zero-suppressed wire format: expanded on the device
            entry = "sai_engine_score_host_zt"
            tiles = (_ptr(pg.stream), pg.tile_off.ctypes.data)
        elif isinstance(pg, MatrixGenotypes):  # int8 matrices: host pack | copy | genotype pass, pipelined
            entry = "sai_engine_score_host_i8"
            n = len(pg.mats)
            ptrs = (C.c_void_p * n)(*[m.ctypes.data for m in pg.mats])
            strides = (C.c_int64 * n)(*[m.strides[0] if m.shape[0] > 1 else max(1, m.shape[1]) for m in pg.mats])
            tiles = (ptrs, strides)
        else:
            entry = "sai_engine_score_host"
            tiles = (_ptr(pg.packed),)
        W = int(ws.shape[0])
        return self._score_call(entry, W, jobs, cap_u, cap_q, C.byref(pg.layout), *tiles, _ptr(pos), pg.n_sites,
                                _ptr(ws), _ptr(we), W)

    def set_vcf_slicing(self, slice_bytes: int = 0, ring: int = 0) -> None:
        """Slice size and ring depth of device ingest (<= 0: default).  Tests force many slices."""
        _cabi.check(_cabi.load().sai_engine_set_vcf_slicing(self._handle(), int(slice_bytes), int(ring)))

    def vcf_stats(self) -> dict:
        """Stages of the last finished device ingest (``sai_engine_vcf_stats``): host seconds staging /
        inflating into the pinned ring and waiting for a free slot, H2D and parse seconds summed over
        the slices (CUDA events), the device span from the first copy to the last parse, slices,
        text bytes, the seconds the final synchronise waited, host seconds enqueueing copies and
        kernels, host seconds inside the feed calls; with ``inflate="device"`` also the inflate
        kernel seconds (CUDA events), the compressed bytes copied and the host seconds spent
        inflating the groups' boundary blocks, and the slices inflated on the device."""
        out = (C.c_double * 14)()
        _cabi.check(_cabi.load().sai_engine_vcf_stats(self._handle(), out, 14))
        keys = ("stage_s", "wait_s", "h2d_s", "parse_s", "device_span_s", "slices", "text_bytes", "finish_wait_s",
                "launch_s", "feed_s", "inflate_s", "comp_bytes", "boundary_s",
                "inflated_slices")
        return dict(zip(keys, list(out)))

    def vcf_slices(self) -> int:
        """Text slices the last device ingest parsed."""
        return int(_cabi.load().sai_engine_vcf_slices(self._handle()))

    def loaded_tiles(self, layout, n_sites: int) -> np.ndarray:
        """Host copy of the tiles the last device ingest left resident (tests, tools)."""
        lib = _cabi.load()
        out = np.empty(max(1, int(lib.sai_packed_bytes(C.byref(layout), int(n_sites)))), dtype=np.uint8)
        _cabi.check(lib.sai_engine_loaded_tiles(self._handle(), out.ctypes.data, out.nbytes))
        return out[: int(lib.sai_packed_bytes(C.byref(layout), int(n_sites)))]

    def loaded_neg_table(self, n_chrom: int, n_pops: int):
        """Host copy of the negative-value table the last device ingest kept (``neg_table=True``):
        ``(neg_off, site, ind, val)``, ``neg_off`` int64 ``[n_chrom, n_pops + 1]`` -- chromosome
        ``c``'s population ``p`` holds entries ``neg_off[c, p] .. neg_off[c, p + 1] - 1`` (tests, tools)."""
        lib = _cabi.load()
        off = np.zeros((n_chrom, n_pops + 1), dtype=np.int64)
        n = int(lib.sai_engine_loaded_neg_table(self._handle(), off.ctypes.data, None, None, None, 0))
        if n < 0:
            _cabi.check(n)
        site, ind, val = (np.zeros(n, dtype=np.int32) for _ in range(3))
        if n:
            _cabi.check(min(0, int(lib.sai_engine_loaded_neg_table(self._handle(), off.ctypes.data, site.ctypes.data,
                                                                    ind.ctypes.data, val.ctypes.data, n))))
        return off, site, ind, val

    def score_loaded(self, windows, jobs, cap_u=None, cap_q=None) -> WindowResults:
        """K1 + K4 on the chunk the last device ingest (``vcf_device.read_loaded``) left resident;
        ``score_resident`` / ``pattern_sums`` then work on it like after ``score``."""
        ws, we = _bounds(windows)
        return self._score_call("sai_engine_score_loaded", len(ws), jobs, cap_u, cap_q, _ptr(ws), _ptr(we), len(ws))

    def score_loaded_pieces(self, pieces, jobs, cap_u=None, cap_q=None) -> WindowResults:
        """``score_loaded`` over pieces of the resident tiles (``vcf_device.read_genome``): ``pieces``
        = ``[(windows, first site, sites), ...]``, the results' windows piece after piece.  One genotype
        pass and one window launch; ``score_resident`` / ``pattern_sums`` then work on the same pieces."""
        ws, we = _bounds([w for p in pieces for w in p[0]])
        table = np.ascontiguousarray([[len(w), lo, n] for w, lo, n in pieces], dtype=np.int64)
        return self._score_call("sai_engine_score_loaded_pieces", len(ws), jobs, cap_u, cap_q, _ptr(ws), _ptr(we),
                                table.ctypes.data, int(table.shape[0]))

    def score_resident(self, jobs, cap_u=None, cap_q=None) -> WindowResults:
        """Another batch of jobs over the chunk of the last ``score*`` call, still resident on the
        device (no upload): a population product of more than 8 combinations costs one transfer."""
        return self._score_call("sai_engine_score_resident", self._last_W, jobs, cap_u, cap_q)

    def _score_call(self, entry: str, W: int, jobs, cap_u, cap_q, *head) -> WindowResults:
        """``entry(engine, *head, jobs, n_jobs, results)`` into new results of ``W`` windows, the windows
        that ``pattern_sums`` / ``dd_sums`` then see.  After SAI_E_CAPACITY the totals say what is
        needed: the candidate lists are regrown and only the window kernel is re-run."""
        lib = _cabi.load()
        J = len(jobs)
        self._last_W = W
        cap_u = max(1, 4 * W + 1024) if cap_u is None else int(cap_u)
        cap_q = max(1, 4 * W + 1024) if cap_q is None else int(cap_q)
        jarr = _job_array(jobs)
        r = WindowResults(
            nsnps=np.zeros((J, W), dtype=np.int32), u=np.zeros((J, W), dtype=np.int64),
            q=np.full((J, W), np.nan, dtype=np.float64), q_cnt=np.zeros((J, W), dtype=np.int32),
            u_start=np.zeros((J, W), dtype=np.int64), q_start=np.zeros((J, W), dtype=np.int64),
            totals=np.zeros((J, 2), dtype=np.int64), u_cand=np.zeros((J, cap_u), dtype=np.int32),
            q_cand=np.zeros((J, cap_q), dtype=np.int32),
        )

        def c_results():
            h = _cabi.HostResults()
            for name in ("nsnps", "u", "q", "q_cnt", "u_start", "q_start", "totals", "u_cand", "q_cand"):
                setattr(h, name, getattr(r, name).ctypes.data)
            h.cap_u, h.cap_q = r.u_cand.shape[1], r.q_cand.shape[1]
            return h

        res = c_results()
        rc = getattr(lib, entry)(self._handle(), *head, jarr, J, C.byref(res))
        if rc == _cabi.E_CAPACITY:
            r.u_cand = np.zeros((J, max(1, int(r.totals[:, 0].max()))), dtype=np.int32)
            r.q_cand = np.zeros((J, max(1, int(r.totals[:, 1].max()))), dtype=np.int32)
            res = c_results()
            rc = lib.sai_engine_rescore_windows(self._handle(), C.byref(res))
        _cabi.check(rc)
        return r

    def score_matrices(self, mats, ploidy, pos, windows, jobs, bits=None, keep_negatives: bool = False,
                       cap_u=None, cap_q=None):
        """Scores int8 (or any integer) per-individual allele-sum matrices -- one per population,
        all over ``pos`` -- without a separate packing pass.  Returns ``(results, genotypes)``;
        ``genotypes`` (layout, negative-value table) is what ``pattern_sums`` / ``dd_sums`` take.
        The bit-planes are chosen from the ploidies; data with larger values (the reference's
        flipped-missing quirk, sai/utils/utils.py:555) is detected by the packer and the call is
        repeated with planes chosen from the data."""
        from .encode import MatrixGenotypes, _as_i8, bits_for, make_layout, negative_table

        neg = negative_table(mats) if keep_negatives else (None, None, None, None)
        m8 = [_as_i8(m) for m in mats]
        pos = np.ascontiguousarray(np.asarray(pos), dtype=np.int32)
        for m in m8:
            if m.shape[0] != pos.shape[0]:
                raise ValueError("every population must have one row per position")
        ws, we = _bounds(windows)
        lay = make_layout([m.shape[1] for m in m8], ploidy, bits)
        mg = MatrixGenotypes(lay, int(pos.shape[0]), pos, m8, [], *neg)
        try:
            return self.score_arrays(mg, ws, we, jobs, cap_u, cap_q), mg
        except ValueError as e:
            if bits is not None or "does not fit" not in str(e):
                raise
        mg.layout = make_layout([m.shape[1] for m in m8], ploidy, [bits_for(m, p) for m, p in zip(m8, ploidy)])
        return self.score_arrays(mg, ws, we, jobs, cap_u, cap_q), mg

    def pattern_sums(self, pg, ref_pop: int, tgt_pop: int, out_pop: int, src_pops: Sequence[int]) -> np.ndarray:
        """Site-pattern sums ``[n_src, W, 7]`` (abba, baba, baaa, abaa, bbaa,
        abba_d, baba_d) of the chunk scored by the last ``score`` call."""
        lib = _cabi.load()
        W = self._last_W
        sums = np.zeros((len(src_pops), W, 7), dtype=np.float64)
        src = (C.c_int32 * len(src_pops))(*[int(x) for x in src_pops])
        _cabi.check(lib.sai_engine_pattern_sums(self._handle(), C.byref(pg.layout), int(ref_pop), int(tgt_pop),
                                                int(out_pop), src, len(src_pops), sums.ctypes.data))
        return sums


    def dd_sums(self, pg, ref_pop: int, tgt_pop: int, src_pops: Sequence[int]):
        """Exact integer distance sums of the DD statistic for the chunk scored by
        the last ``score`` call: ``(ref_sum, tgt_sum)``, int64 ``[n_src, W, m_max]``
        with ``ref_sum[k, i, a] = sum_j sum_sites |src_a - ref_j|``
        (sai/stats/dd_statistic.py:70-71).  ``pg`` must carry the negative-value
        table (``pack_populations(..., keep_negatives=True)``), or be a device-parsed
        chunk or genome whose table is resident (``LoadedChunk.neg``): then neither the
        tiles nor the table cross PCIe (``sai_engine_dd_sums_loaded``)."""
        lib = _cabi.load()
        W = self._last_W
        m_max = max(int(pg.layout.pop[int(s)].n_samples) for s in src_pops)
        ref_sum = np.zeros((len(src_pops), W, m_max), dtype=np.int64)
        tgt_sum = np.zeros_like(ref_sum)
        src = (C.c_int32 * len(src_pops))(*[int(x) for x in src_pops])
        if getattr(pg, "neg", False):
            _cabi.check(lib.sai_engine_dd_sums_loaded(self._handle(), int(ref_pop), int(tgt_pop), src, len(src_pops),
                                                      ref_sum.ctypes.data, tgt_sum.ctypes.data, m_max))
            return ref_sum, tgt_sum
        if getattr(pg, "neg_off", None) is None:
            raise ValueError("DD needs the raw values of missing calls: pack with keep_negatives=True")
        _cabi.check(lib.sai_engine_dd_sums(self._handle(), C.byref(pg.layout), int(ref_pop), int(tgt_pop), src,
                                           len(src_pops), pg.neg_off.ctypes.data, _ptr(pg.neg_site), _ptr(pg.neg_ind),
                                           _ptr(pg.neg_val), ref_sum.ctypes.data, tgt_sum.ctypes.data, m_max))
        return ref_sum, tgt_sum

    #: ``format_scores`` calls made by any engine of this process (which writer produced a file)
    format_calls = 0

    def format_scores(self, inp: "_cabi.FormatInput") -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        """The score rows, ``.U.log`` and ``.Q.log`` text of ``inp`` formatted on the device
        (``sai_engine_format_scores``), each copied back in one D2H copy: three uint8 arrays (empty for
        a log that does not exist)."""
        lib = _cabi.load()
        sizes = np.zeros(3, dtype=np.int64)
        _cabi.check(lib.sai_engine_format_scores(self._handle(), C.byref(inp), sizes.ctypes.data))
        HostEngine.format_calls += 1
        out = []
        for k in range(3):
            text = np.empty(int(sizes[k]), dtype=np.uint8)
            if text.size:
                _cabi.check(lib.sai_engine_format_text(self._handle(), k, text.ctypes.data, text.size))
            out.append(text)
        return tuple(out)

    def format_stats(self) -> dict:
        """Seconds of the last ``format_scores`` (CUDA events): input copy, length + scan kernels,
        write kernels."""
        out = (C.c_double * 3)()
        _cabi.check(_cabi.load().sai_engine_format_stats(self._handle(), out, 3))
        return dict(zip(("copy_s", "length_s", "write_s"), list(out)))

    def format_doubles(self, x: np.ndarray) -> np.ndarray:
        """``repr(float(v))`` of every value, formatted by the device in one launch: ``[n, 32]``
        uint8, NUL-padded (tests)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.zeros((x.size, 32), dtype=np.uint8)
        _cabi.check(_cabi.load().sai_engine_format_doubles(self._handle(), x.ctypes.data, x.size, out.ctypes.data))
        return out

    #: ``table_build`` calls made by any engine of this process (which path wrote the outlier tables)
    outlier_calls = 0

    def table_load(self, data: bytes, n_cols: int, chunk_rows: int) -> tuple[int, int, int]:
        """Copies a score file to the device, finds its cells and classifies them
        (``sai_engine_table_load``): (data rows, parse chunks, ``SAI_TABLE_*`` flags)."""
        info = np.zeros(3, dtype=np.int64)
        _cabi.check(_cabi.load().sai_engine_table_load(self._handle(), data, len(data), int(n_cols), int(chunk_rows),
                                                       info.ctypes.data))
        return int(info[0]), int(info[1]), int(info[2])

    def table_classes(self, n_chunks: int, n_cols: int) -> np.ndarray:
        """``[n_chunks, n_cols]`` uint32: the OR of the ``SAI_CELL_*`` classes of every column's cells
        per pandas parse chunk of the loaded file."""
        out = np.zeros((n_chunks, n_cols), dtype=np.uint32)
        _cabi.check(_cabi.load().sai_engine_table_classes(self._handle(), out.ctypes.data, out.size))
        return out

    def table_parse(self, kinds: Sequence[int], first_metric: int, chrom: int, start: int, end: int,
                    vals) -> tuple[np.ndarray, int]:
        """Parses the loaded file with the column dtypes ``kinds``: the metric columns into the float64
        CUDA tensor ``vals`` ``[n_metric, rows]``.  Returns each metric column's first value in file
        order (NaN: none) and the number of runs of equal Chrom text."""
        k = np.ascontiguousarray(kinds, dtype=np.int32)
        first = np.zeros(int(vals.shape[0]), dtype=np.float64)
        n_runs = C.c_int64()
        _cabi.check(_cabi.load().sai_engine_table_parse(self._handle(), k.ctypes.data, int(first_metric), int(chrom),
                                                        int(start), int(end), vals.data_ptr(), first.ctypes.data,
                                                        C.byref(n_runs)))
        return first, int(n_runs.value)

    def table_runs(self, n_runs: int) -> tuple[np.ndarray, np.ndarray]:
        """Byte offset and length of each Chrom run's name within the loaded file."""
        off = np.zeros(n_runs, dtype=np.int64)
        ln = np.zeros(n_runs, dtype=np.int64)
        _cabi.check(_cabi.load().sai_engine_table_runs(self._handle(), off.ctypes.data, ln.ctypes.data, n_runs))
        return off, ln

    def table_order(self, run_rank: np.ndarray) -> None:
        """Sorts the rows stably on (rank of their Chrom run, Start, End)."""
        r = np.ascontiguousarray(run_rank, dtype=np.int32)
        _cabi.check(_cabi.load().sai_engine_table_order(self._handle(), r.ctypes.data, r.size))

    def table_build(self, thr: Sequence[float], strict: Sequence[bool]) -> tuple[np.ndarray, np.ndarray]:
        """Every metric column's outlier table as text, copied back in one D2H copy: (uint8 text,
        int64 offsets ``[n_metric + 1]``; table m is ``text[offsets[m]:offsets[m + 1]]``)."""
        lib = _cabi.load()
        t = np.ascontiguousarray(thr, dtype=np.float64)
        s = np.ascontiguousarray(strict, dtype=np.int32)
        offs = np.zeros(t.size + 1, dtype=np.int64)
        _cabi.check(lib.sai_engine_table_build(self._handle(), t.ctypes.data, s.ctypes.data, offs.ctypes.data))
        HostEngine.outlier_calls += 1
        text = np.empty(int(offs[-1]), dtype=np.uint8)
        _cabi.check(lib.sai_engine_table_text(self._handle(), text.ctypes.data, text.size))
        return text, offs

    def table_stats(self) -> dict:
        """Seconds of the last table calls (CUDA events)."""
        out = (C.c_double * 6)()
        _cabi.check(_cabi.load().sai_engine_table_stats(self._handle(), out, 6))
        return dict(zip(("copy_in_s", "tokenise_s", "parse_s", "sort_s", "format_s", "copy_back_s"), list(out)))

    def parse_doubles(self, strings: Sequence[bytes]) -> tuple[np.ndarray, np.ndarray]:
        """pandas' float parser on every string, run by the device in one launch (tests): (values,
        bool "pandas reads it as a float")."""
        text, offs = _joined(strings)
        out = np.zeros(len(strings), dtype=np.float64)
        ok = np.zeros(len(strings), dtype=np.uint8)
        _cabi.check(_cabi.load().sai_engine_parse_doubles(self._handle(), text, offs.ctypes.data, len(strings),
                                                          out.ctypes.data, ok.ctypes.data))
        return out, ok.astype(bool)


def _joined(strings: Sequence[bytes]) -> tuple[bytes, np.ndarray]:
    offs = np.zeros(len(strings) + 1, dtype=np.int64)
    offs[1:] = np.cumsum([len(s) for s in strings])
    return b"".join(strings), offs


def parse_doubles_host(strings: Sequence[bytes]) -> tuple[np.ndarray, np.ndarray]:
    """pandas' float parser (``precise_xstrtod``) on every string, from the host build of the device
    parser: (values, bool "pandas reads it as a float")."""
    text, offs = _joined(strings)
    out = np.zeros(len(strings), dtype=np.float64)
    ok = np.zeros(len(strings), dtype=np.uint8)
    _cabi.check(_cabi.load().sai_parse_doubles(text, offs.ctypes.data, len(strings), out.ctypes.data, ok.ctypes.data))
    return out, ok.astype(bool)


def classify_cells_host(strings: Sequence[bytes]) -> np.ndarray:
    """The ``SAI_CELL_*`` class of every string as a score-file cell (host build of the device code)."""
    text, offs = _joined(strings)
    out = np.zeros(len(strings), dtype=np.uint8)
    _cabi.check(_cabi.load().sai_classify_cells(text, offs.ctypes.data, len(strings), out.ctypes.data))
    return out


def format_doubles_host(x: np.ndarray) -> np.ndarray:
    """``repr(float(v))`` of every value from the host build of the device formatter: ``[n, 32]``
    uint8, NUL-padded."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.zeros((x.size, 32), dtype=np.uint8)
    _cabi.check(_cabi.load().sai_format_doubles(x.ctypes.data, x.size, out.ctypes.data))
    return out


def dd_values(ref_sum: np.ndarray, tgt_sum: np.ndarray, n_ref: int, n_tgt: int, n_src_samples: Sequence[int]) -> list:
    """DD per source population and window from the integer sums, with the
    reference's float64 operations (dd_statistic.py:74-77): the row means are one
    division of an exactly representable integer sum, then ``np.mean`` of the
    differences.  Returns ``[n_src][W]`` numpy float64 scalars."""
    out = []
    for k, m in enumerate(n_src_samples):
        mean_src_ref = ref_sum[k, :, :m].astype(np.float64) / n_ref
        mean_src_tgt = tgt_sum[k, :, :m].astype(np.float64) / n_tgt
        diff = mean_src_ref - mean_src_tgt
        out.append([np.mean(np.ascontiguousarray(row)) for row in diff])
    return out


def four_pop_values(sums: np.ndarray) -> dict:
    """Danc / Dplus / df / fd per source population and window from the seven
    pattern sums, with the reference's formulas and its ``denominator != 0``
    rule (danc_statistic.py:74-80, dplus_statistic.py:76-83, df_statistic.py:75-81,
    fd_statistic.py:83-86).  Returns ``{name: [n_src][W] Python floats}``."""
    out = {"Danc": [], "Dplus": [], "df": [], "fd": []}
    ratio = lambda n, d: n / d if d != 0 else float("nan")
    for k in range(sums.shape[0]):
        rows = {name: [] for name in out}
        for abba, baba, baaa, abaa, bbaa, abba_d, baba_d in sums[k].tolist():
            rows["Danc"].append(ratio(baaa - abaa, baaa + abaa))
            rows["Dplus"].append(ratio(abba - baba + baaa - abaa, abba + baba + baaa + abaa))
            rows["df"].append(ratio(abba - baba, abba + baba + 2 * bbaa))
            rows["fd"].append(ratio(abba - baba, abba_d - baba_d))
        for name in out:
            out[name].append(rows[name])
    return out


# --------------------------------------------------------------------------
# device-resident scorer (torch tensors own the memory; C ABI gets raw pointers)
# --------------------------------------------------------------------------
class DeviceScorer:
    """Runs the kernels on data already resident in HBM, on torch's current
    stream.  torch is used for allocation and streams only."""

    def __init__(self, layout, n_sites: int, n_windows: int, n_jobs: int, device=None, cap_u=None, cap_q=None,
                 _share: Optional["DeviceScorer"] = None):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("sai_b200 needs a CUDA device (no CPU fallback)")
        self.torch = torch
        self.lib = _cabi.load()
        self.layout = layout
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.n_sites, self.W, self.J = int(n_sites), int(n_windows), int(n_jobs)
        self.n_tiles = (self.n_sites + _cabi.TILE_SITES - 1) // _cabi.TILE_SITES
        self.stride = self.n_tiles * _cabi.TILE_SITES
        d = self.device
        J, W = self.J, self.W
        if _share is not None:
            self.mask_u, self.mask_q, self.qval = _share.mask_u, _share.mask_q, _share.qval
        else:
            self.mask_u = torch.zeros((J, max(1, self.n_tiles)), dtype=torch.int32, device=d)
            self.mask_q = torch.zeros((J, max(1, self.n_tiles)), dtype=torch.int32, device=d)
            self.qval = torch.zeros((J, max(1, self.stride)), dtype=torch.float64, device=d)
        self.nsnps = torch.zeros((J, W), dtype=torch.int32, device=d)
        self.u = torch.zeros((J, W), dtype=torch.int64, device=d)
        self.q = torch.zeros((J, W), dtype=torch.float64, device=d)
        self.q_cnt = torch.zeros((J, W), dtype=torch.int32, device=d)
        self.u_start = torch.zeros((J, W), dtype=torch.int64, device=d)
        self.q_start = torch.zeros((J, W), dtype=torch.int64, device=d)
        self.totals = torch.zeros((J, 2), dtype=torch.int64, device=d)
        self.cap_u = max(1, 4 * W + 1024) if cap_u is None else int(cap_u)
        self.cap_q = max(1, 4 * W + 1024) if cap_q is None else int(cap_q)
        self.u_cand = torch.zeros((J, self.cap_u), dtype=torch.int32, device=d)
        self.q_cand = torch.zeros((J, self.cap_q), dtype=torch.int32, device=d)
        self.num = None if _share is None else _share.num
        self.called = None if _share is None else _share.called

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def sibling(self, n_windows: int, cap_u=None, cap_q=None) -> "DeviceScorer":
        """A scorer over the SAME site masks / Q values / cached counts with result buffers for
        another window list: a window-shape sweep flags the sites once and scores every
        (win-len, step) grid from the same masks."""
        other = DeviceScorer(self.layout, self.n_sites, n_windows, self.J, device=self.device, cap_u=cap_u, cap_q=cap_q,
                             _share=self)
        return other

    def site_counts(self, d_packed, variant: int = 0):
        """K1 alone: returns ``(num, called)`` int32 tensors ``[n_pops, stride]``."""
        torch = self.torch
        n_pops = self.layout.n_pops
        if self.num is None:
            self.num = torch.zeros((n_pops, max(1, self.stride)), dtype=torch.int32, device=self.device)
            self.called = torch.zeros_like(self.num)
        _cabi.check(
            self.lib.sai_site_counts(
                C.byref(self.layout), d_packed.data_ptr(), 0, self.n_tiles, self.num.data_ptr(),
                self.called.data_ptr(), self.stride, variant, self._stream(),
            )
        )
        return self.num, self.called

    def site_flags(self, d_packed, jobs, variant: int = 0, with_counts: bool = False, tile0: int = 0, n_tiles=None):
        """K1 fused: genotype pass + site conditions for ``jobs``."""
        jarr = _job_array(jobs)
        num = called = None
        if with_counts:
            if self.num is None:
                torch = self.torch
                self.num = torch.zeros((self.layout.n_pops, max(1, self.stride)), dtype=torch.int32, device=self.device)
                self.called = torch.zeros_like(self.num)
            num, called = self.num.data_ptr(), self.called.data_ptr()
        _cabi.check(
            self.lib.sai_site_flags(
                C.byref(self.layout), d_packed.data_ptr(), tile0, self.n_tiles - tile0 if n_tiles is None else n_tiles,
                self.n_tiles, jarr, len(jobs), self.mask_u.data_ptr(), self.mask_q.data_ptr(),
                self.qval.data_ptr(), self.qval.shape[1], num, called, self.stride if with_counts else 0,
                variant, self._stream(),
            )
        )

    def flags_from_counts(self, jobs):
        """Site conditions from the cached counts (threshold sweeps)."""
        if self.num is None:
            raise RuntimeError("site_counts() has not been run")
        jarr = _job_array(jobs)
        _cabi.check(
            self.lib.sai_flags_from_counts(
                C.byref(self.layout), self.num.data_ptr(), self.called.data_ptr(), self.stride, self.n_sites,
                jarr, len(jobs), self.mask_u.data_ptr(), self.mask_q.data_ptr(), self.qval.data_ptr(),
                self.qval.shape[1], self._stream(),
            )
        )

    def window_stats(self, d_pos, d_ws, d_we, jobs, d_first_site=None, d_last_site=None):
        """K4.  ``d_first_site`` / ``d_last_site`` (int32 per window): the site range of the
        window's own chromosome piece when several pieces are laid side by side
        (``sai_window_stats_pieces``, see sai_b200.genome)."""
        jarr = _job_array(jobs)
        self._last = (d_pos, d_ws, d_we, jobs, d_first_site, d_last_site)
        head = (d_pos.data_ptr(), self.n_sites, d_ws.data_ptr(), d_we.data_ptr())
        tail = (
            self.W, jarr, len(jobs),
            self.mask_u.data_ptr(), self.mask_q.data_ptr(), self.qval.data_ptr(), self.qval.shape[1],
            self.nsnps.data_ptr(), self.u.data_ptr(), self.q.data_ptr(), self.q_cnt.data_ptr(),
            self.u_start.data_ptr(), self.q_start.data_ptr(), self.totals.data_ptr(),
            self.u_cand.data_ptr(), self.cap_u, self.q_cand.data_ptr(), self.cap_q, self._stream(),
        )
        if d_first_site is None:
            _cabi.check(self.lib.sai_window_stats(*head, *tail))
        else:
            _cabi.check(self.lib.sai_window_stats_pieces(*head, d_first_site.data_ptr(), d_last_site.data_ptr(), *tail))

    def pattern_sums(self, d_pos, d_ws, d_we, ref_pop: int, tgt_pop: int, out_pop: int, src_pops: Sequence[int]):
        """N3 from the cached counts (``site_counts`` / ``site_flags(with_counts=True)`` first):
        float64 tensor ``[n_src, W, 7]``."""
        if self.num is None:
            raise RuntimeError("site_counts() has not been run")
        torch = self.torch
        sums = torch.zeros((len(src_pops), self.W, 7), dtype=torch.float64, device=self.device)
        src = (C.c_int32 * len(src_pops))(*[int(x) for x in src_pops])
        _cabi.check(
            self.lib.sai_window_patterns(
                C.byref(self.layout), d_pos.data_ptr(), self.n_sites, d_ws.data_ptr(), d_we.data_ptr(), self.W,
                self.num.data_ptr(), self.called.data_ptr(), self.stride, int(ref_pop), int(tgt_pop), int(out_pop),
                src, len(src_pops), sums.data_ptr(), self._stream(),
            )
        )
        return sums

    def site_hist(self, d_packed, pops: Sequence[int]):
        """N4 genotype pass: per-site value histograms of ``pops`` -> int32 ``[rows, stride]``
        and the missing-call totals (uint64 as int64 tensor ``[len(pops)]``)."""
        torch = self.torch
        arr = (C.c_int32 * len(pops))(*[int(x) for x in pops])
        rows = int(self.lib.sai_hist_rows(C.byref(self.layout), arr, len(pops)))
        hist = torch.zeros((rows, max(1, self.stride)), dtype=torch.int32, device=self.device)
        missing = torch.zeros(len(pops), dtype=torch.int64, device=self.device)
        _cabi.check(
            self.lib.sai_site_hist(C.byref(self.layout), d_packed.data_ptr(), self.n_sites, arr, len(pops),
                                   hist.data_ptr(), self.stride, missing.data_ptr(), self._stream())
        )
        return hist, missing

    def dd_sums(self, d_packed, d_pos, d_ws, d_we, hist, ref_pop: int, tgt_pop: int, src_pops: Sequence[int],
                neg_off: np.ndarray, d_neg_site, d_neg_ind, d_neg_val):
        """N4 window kernel on ``hist = site_hist(d_packed, [ref_pop, tgt_pop])[0]``: int64 tensors
        ``(ref_sum, tgt_sum)`` ``[n_src, W, m_max]`` and the int32 error flag tensor."""
        torch = self.torch
        m_max = max(int(self.layout.pop[int(s)].n_samples) for s in src_pops)
        ref_sum = torch.zeros((len(src_pops), self.W, m_max), dtype=torch.int64, device=self.device)
        tgt_sum = torch.zeros_like(ref_sum)
        err = torch.zeros(1, dtype=torch.int32, device=self.device)
        src = (C.c_int32 * len(src_pops))(*[int(x) for x in src_pops])
        off = np.ascontiguousarray(neg_off, dtype=np.int64)
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None
        _cabi.check(
            self.lib.sai_window_dd(
                C.byref(self.layout), d_packed.data_ptr(), d_pos.data_ptr(), self.n_sites, d_ws.data_ptr(),
                d_we.data_ptr(), self.W, hist.data_ptr(), self.stride, int(ref_pop), int(tgt_pop), src, len(src_pops),
                off.ctypes.data, ptr(d_neg_site), ptr(d_neg_ind), ptr(d_neg_val), ref_sum.data_ptr(),
                tgt_sum.data_ptr(), m_max, err.data_ptr(), self._stream(),
            )
        )
        return ref_sum, tgt_sum, err

    def step(self, d_packed, d_pos, d_ws, d_we, jobs, variant: int = 0):
        """One pass of the hot path over device-resident inputs: the genotype
        pass and the window kernel (2 launches + one 16-byte memset)."""
        self.site_flags(d_packed, jobs, variant)
        self.window_stats(d_pos, d_ws, d_we, jobs)

    def results(self) -> WindowResults:
        """Copies the results to the host (synchronises).  If the candidate
        buffers were too small they are grown and the window kernel is re-run
        on the flags still resident on the device."""
        torch = self.torch
        totals = self.totals.cpu().numpy()
        need_u, need_q = (int(totals[:, 0].max()), int(totals[:, 1].max())) if self.J else (0, 0)
        if need_u > self.cap_u or need_q > self.cap_q:
            if getattr(self, "_last", None) is None:
                raise _cabi.SaiError(
                    f"candidate capacity too small (need cap_u>={need_u}, cap_q>={need_q})"
                )
            self.cap_u, self.cap_q = max(self.cap_u, need_u), max(self.cap_q, need_q)
            self.u_cand = torch.zeros((self.J, self.cap_u), dtype=torch.int32, device=self.device)
            self.q_cand = torch.zeros((self.J, self.cap_q), dtype=torch.int32, device=self.device)
            self.window_stats(*self._last)
            totals = self.totals.cpu().numpy()
        return WindowResults(
            self.nsnps.cpu().numpy(), self.u.cpu().numpy(), self.q.cpu().numpy(), self.q_cnt.cpu().numpy(),
            self.u_start.cpu().numpy(), self.q_start.cpu().numpy(), totals,
            self.u_cand.cpu().numpy(), self.q_cand.cpu().numpy(),
        )


def synth_fill(layout, d_packed, n_sites: int, roles: Sequence[int], seed: int, missing_rate: float = 0.0,
               tile0: int = 0, n_tiles: Optional[int] = None, stream=None):
    """Bench/test helper: synthetic packed genotypes generated on the device."""
    import torch

    lib = _cabi.load()
    nt = (n_sites + _cabi.TILE_SITES - 1) // _cabi.TILE_SITES
    role = (C.c_int32 * len(roles))(*[int(r) for r in roles])
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream if stream is None else stream)
    _cabi.check(
        lib.sai_synth_fill(C.byref(layout), d_packed.data_ptr(), tile0, nt - tile0 if n_tiles is None else n_tiles,
                           n_sites, role, seed, float(missing_rate), st)
    )
