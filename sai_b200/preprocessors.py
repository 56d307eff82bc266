"""GPU-backed mirrors of the reference's batched entry points.

``ChunkPreprocessor`` has the constructor and ``run(chr_name, start, end)`` /
``process_items(items)`` contract of the reference class
(sai/preprocessors/chunk_preprocessor.py:38-147) and returns item dicts with
the schema of ``FeaturePreprocessor.run``
(sai/preprocessors/feature_preprocessor.py:119-191), in the reference's order
(population product outermost, windows innermost,
sai/generators/window_generator.py:164-167) -- but the per-window Python loop
is replaced by one call into the CUDA library per chunk.
"""

from __future__ import annotations

import locale
from itertools import combinations, product
from pathlib import Path
from typing import Any, Optional

import numpy as np

from . import _cabi
from .encode import PopData
from .scoring import HostEngine, dd_values, four_pop_values, make_job
from .windows import chunk_windows, split_genome


def _same_positions(members: list[PopData]) -> bool:
    first = members[0].POS
    return all(m.POS.shape == first.shape and np.array_equal(m.POS, first) for m in members[1:])


def _common_rows(members: list[PopData]) -> tuple[np.ndarray, list[np.ndarray]]:
    """Positions present in every member (window_generator.py:193-197) and each
    member's genotype rows at those positions (:217-231)."""
    if _same_positions(members):
        return members[0].POS, [m.GT for m in members]
    common = members[0].POS
    for m in members[1:]:
        common = np.intersect1d(common, m.POS)
    return common, [m.GT.compress(np.isin(m.POS, common), axis=0) for m in members]


def score_populations(
    chr_name: str,
    windows_by_tgt: dict[str, list[tuple[int, int]]],
    ref_data: dict[str, PopData],
    tgt_data: dict[str, PopData],
    src_data: dict[str, PopData],
    ploidy_config,
    stat_config,
    anc_allele_available: bool,
    engine: HostEngine,
    out_data: Optional[dict[str, PopData]] = None,
    num_src: Optional[int] = None,
    loaded=None,
    sink=None,
) -> list[dict[str, Any]]:
    """Item dicts for every (ref, tgt, src-combination, outgroup) x window.

    When every population sits on the same positions and every target population has the same
    windows (always the case for ``ChunkPreprocessor.run(chr, start, end)`` on one VCF), ALL
    populations are packed once and the population product becomes up to ``SAI_MAX_JOBS`` jobs per
    genotype pass, instead of one pack + one transfer + one pass per combination.

    ``loaded`` (a ``vcf_device.LoadedChunk``): the populations were parsed on the device into one
    layout resident in ``engine``; the ``*_data`` dicts then only name the populations (their
    values are not read) and every combination is scored from that layout.  A
    ``vcf_device.LoadedGenome`` holds several chromosomes, each with its own windows
    (``windows_by_tgt`` maps every target population to the list of them, one per chromosome;
    ``chr_name`` is not used): all chromosomes are scored with one genotype pass and one window
    launch per batch of combinations, and the items come out chromosome by chromosome.

    ``sink`` (e.g. a ``DeviceRows``): each run of windows of one combination is handed to
    ``sink(combo, windows, pos, res, j, four_vals, dd_vals, chrom, at)`` instead of being turned into
    item dicts, and the returned list stays empty."""
    stats = [s for s in stat_config.root.keys() if s in ("U", "Q")]
    four = [s for s in stat_config.root.keys() if s in ("Danc", "Dplus", "df", "fd") and stat_config.root[s] is True]
    dd = any(s == "DD" and stat_config.root[s] is True for s in stat_config.root.keys())
    num_src = len(src_data) if num_src is None else num_src
    src_combos = list(combinations(src_data.keys(), num_src))
    outs = list(out_data.keys()) if out_data else [None]
    src_ploidies = ploidy_config.get_ploidy("src")
    combos = list(product(ref_data, tgt_data, src_combos, outs))
    items: list[dict[str, Any]] = []
    if not combos:
        return items

    def job_for(ref_pop, tgt_pop, ref_idx, tgt_idx, src_idx):
        specs = {}
        for s in stats:
            prm = stat_config.get_parameters(s)
            spec = {"w": prm["ref"][ref_pop], "y_list": list(prm["src"].values())}
            spec["x" if s == "U" else "quantile"] = prm["tgt"][tgt_pop]
            specs[s] = spec
        return make_job(ref_idx, tgt_idx, src_idx, anc_allele_available, specs.get("U"), specs.get("Q"))

    def src_ploidy_list(n_src):
        # positional zip of src genotypes / y_list / ploidies, exactly as
        # feature_preprocessor.py:160,168-170 and stat_utils.py:116-119 do
        pl = list(src_ploidies[:n_src])
        if len(pl) != n_src:
            raise ValueError("The length of src_gts_list and src ploidies must match.")
        return pl

    stat_order = [s for s in stat_config.root.keys() if s in stats or s in four or (dd and s == "DD")]
    empty_cdd = np.array([])

    def emit(combo, windows, pos, res, j, four_vals, dd_vals, chrom=chr_name, at=0):
        """One item dict per window (feature_preprocessor.py:119-191).  A chromosome-scale chunk has
        tens of thousands of windows, so the per-window work is kept to plain Python objects: the
        result columns are turned into lists once and the candidate lists are views into one
        converted array.  ``windows`` are the result columns ``at, at + 1, ...``."""
        if sink is not None:
            return sink(combo, windows, pos, res, j, four_vals, dd_vals, chrom, at)
        ref_pop, tgt_pop, src_comb, out_pop = combo
        n_src = len(src_comb)
        out_name = "NA" if out_pop is None else out_pop
        pos_dtype = np.asarray(pos).dtype
        cols = slice(at, at + len(windows))
        if res is not None:
            nsnps_l = res.nsnps[j, cols].tolist()
        else:
            nsnps_l = [int(np.count_nonzero((pos >= s_) & (pos <= e_))) for s_, e_ in windows]
        want_u, want_q = "U" in stats, "Q" in stats
        if want_u:
            u_l, us_l = res.u[j, cols].tolist(), res.u_start[j, cols].tolist()
            u_cand = res.u_cand[j].astype(pos_dtype, copy=False)
        if want_q:
            q_col = res.q[j, cols]  # q_col[i] is a numpy.float64, like np.nanquantile's
            qnan_l = np.isnan(q_col).tolist()
            qs_l, qc_l = res.q_start[j, cols].tolist(), res.q_cnt[j, cols].tolist()
            q_cand = res.q_cand[j].astype(pos_dtype, copy=False)
        nan_list = [np.nan for _ in range(n_src)] if n_src > 1 else np.nan
        for i, (start, end) in enumerate(windows):
            nsnps = nsnps_l[i]
            cdd = {}
            item = {
                "chr_name": chrom,
                "start": start,
                "end": end,
                "ref_pop": ref_pop,
                "tgt_pop": tgt_pop,
                "src_pop_list": src_comb,
                "out_pop": out_name,
                "nsnps": nsnps,
                "cdd_pos": cdd,
            }
            for s in stat_order:
                if s == "U":
                    if nsnps == 0:  # empty window: feature_preprocessor.py:131-144
                        item[s] = np.nan
                        cdd[s] = empty_cdd
                    else:
                        n = u_l[i]
                        item[s] = n
                        cdd[s] = u_cand[us_l[i] : us_l[i] + n]
                elif s == "Q":
                    if nsnps == 0 or qnan_l[i]:  # q_statistic.py:96-98
                        item[s] = np.nan
                        cdd[s] = empty_cdd
                    else:
                        item[s] = q_col[i]
                        cdd[s] = q_cand[qs_l[i] : qs_l[i] + qc_l[i]]
                elif nsnps == 0:  # feature_preprocessor.py:137-141
                    item[s] = list(nan_list) if n_src > 1 else np.nan
                elif s == "DD":
                    item[s] = [dd_vals[k][at + i] for k in range(n_src)]
                else:
                    item[s] = [four_vals[s][k][at + i] for k in range(n_src)]
            items.append(item)

    def extras(pg, ref_idx, tgt_idx, src_idx, out_idx, n_ref, n_tgt, n_srcs):
        four_vals = dd_vals = None
        if four:
            four_vals = four_pop_values(engine.pattern_sums(pg, ref_idx, tgt_idx, out_idx, src_idx))
        if dd:
            ref_sum, tgt_sum = engine.dd_sums(pg, ref_idx, tgt_idx, src_idx)
            dd_vals = dd_values(ref_sum, tgt_sum, n_ref, n_tgt, n_srcs)
        return four_vals, dd_vals

    use_out = bool(out_data) and bool(four)

    # ---- populations parsed on the device, resident in `engine`: one chunk, or a genome in pieces ----
    if loaded is not None:
        win_lists = next(iter(windows_by_tgt.values()))
        if hasattr(loaded, "first_site"):  # a LoadedGenome: one piece per chromosome
            chroms = list(zip(loaded.names, win_lists, loaded.pos))
            pieces = [(w, max(f, 0), n) for w, f, n in zip(win_lists, loaded.first_site, loaded.n_sites)]
        else:
            chroms, pieces = [(chr_name, win_lists, loaded.pos)], None
        at = np.cumsum([0] + [len(w) for _, w, _ in chroms]).tolist()
        index, n_of = loaded.index, lambda i: int(loaded.layout.pop[i].n_samples)
        batches = []
        for b0 in range(0, len(combos), _cabi.MAX_JOBS):
            batch = combos[b0 : b0 + _cabi.MAX_JOBS]
            jobs = []
            for r, t, sc, _ in batch:
                src_ploidy_list(len(sc))  # same check as the host path
                jobs.append(job_for(r, t, index[("ref", r)], index[("tgt", t)], [index[("src", s)] for s in sc]))
            if b0 > 0:
                res = engine.score_resident(jobs)
            elif pieces is None:
                res = engine.score_loaded(win_lists, jobs)
            else:
                res = engine.score_loaded_pieces(pieces, jobs)
            four_by_job = []
            for r, t, sc, o in batch:
                src_idx = [index[("src", s)] for s in sc]
                four_by_job.append(extras(loaded, index[("ref", r)], index[("tgt", t)], src_idx,
                                          index[("out", o)] if (use_out and o is not None) else -1,
                                          n_of(index[("ref", r)]), n_of(index[("tgt", t)]), [n_of(i) for i in src_idx]))
            batches.append((batch, res, four_by_job))
        for (chrom, windows, pos), a in zip(chroms, at):
            for batch, res, four_by_job in batches:
                for j, combo in enumerate(batch):
                    emit(combo, windows, pos, res, j, *four_by_job[j], chrom=chrom, at=a)
        return items

    # ---- all populations in one packed matrix, the product as fused jobs ------------------
    everyone = list(ref_data.values()) + list(tgt_data.values()) + list(src_data.values())
    if use_out:
        everyone += list(out_data.values())
    win_lists = list(windows_by_tgt.values())
    fused = (
        len(combos) > 1
        and len(src_combos) == 1
        and len(everyone) <= _cabi.MAX_POPS
        and _same_positions(everyone)
        and all(w == win_lists[0] for w in win_lists[1:])
        and (stats or four or dd)
    )
    if fused:
        index, mats, ploidy = {}, [], []
        for group, data in (("ref", ref_data), ("tgt", tgt_data)):
            for name, d in data.items():
                index[(group, name)] = len(mats)
                mats.append(d.GT)
                ploidy.append(ploidy_config.get_ploidy(group, name))
        src_comb = src_combos[0]
        for name, pl in zip(src_comb, src_ploidy_list(len(src_comb))):
            index[("src", name)] = len(mats)
            mats.append(src_data[name].GT)
            ploidy.append(pl)
        if use_out:
            for name, d in out_data.items():
                index[("out", name)] = len(mats)
                mats.append(d.GT)
                ploidy.append(ploidy_config.get_ploidy("outgroup", name))
        pos = everyone[0].POS
        pg = None
        windows = win_lists[0]
        n_of = lambda i: int(pg.layout.pop[i].n_samples)
        for b0 in range(0, len(combos), _cabi.MAX_JOBS):
            batch = combos[b0 : b0 + _cabi.MAX_JOBS]
            jobs = []
            for r, t, sc, _ in batch:
                jobs.append(job_for(r, t, index[("ref", r)], index[("tgt", t)], [index[("src", s)] for s in sc]))
            if pg is None:  # int8 matrices -> pack | copy | genotype pass, pipelined; ONE upload for all batches
                res, pg = engine.score_matrices(mats, ploidy, pos, windows, jobs, keep_negatives=dd)
            else:
                res = engine.score_resident(jobs)
            for j, combo in enumerate(batch):
                r, t, sc, o = combo
                src_idx = [index[("src", s)] for s in sc]
                four_vals, dd_vals = extras(
                    pg, index[("ref", r)], index[("tgt", t)], src_idx, index[("out", o)] if (use_out and o is not None) else -1,
                    n_of(index[("ref", r)]), n_of(index[("tgt", t)]), [n_of(i) for i in src_idx])
                emit(combo, windows, pos, res, j, four_vals, dd_vals)
        return items

    # ---- general case: one packed matrix per combination ----------------------------------
    for combo in combos:
        ref_pop, tgt_pop, src_comb, out_pop = combo
        windows = windows_by_tgt[tgt_pop]
        members = [ref_data[ref_pop], tgt_data[tgt_pop]] + [src_data[s] for s in src_comb]
        if out_pop is not None:
            members.append(out_data[out_pop])
        pos, rows = _common_rows(members)
        n_src = len(src_comb)
        ploidy = [ploidy_config.get_ploidy("ref", ref_pop), ploidy_config.get_ploidy("tgt", tgt_pop)]
        ploidy += src_ploidy_list(n_src)
        src_idx = list(range(2, 2 + n_src))
        job = job_for(ref_pop, tgt_pop, 0, 1, src_idx)
        n_pack = 2 + n_src
        if out_pop is not None and four:
            ploidy.append(ploidy_config.get_ploidy("outgroup", out_pop))
            n_pack += 1
        res = pg = None
        if stats or four or dd:
            res, pg = engine.score_matrices(rows[:n_pack], ploidy[:n_pack], pos, windows, [job], keep_negatives=dd)
        four_vals, dd_vals = extras(pg, 0, 1, src_idx, 2 + n_src if (out_pop is not None and four) else -1,
                                    rows[0].shape[1], rows[1].shape[1], [rows[2 + k].shape[1] for k in range(n_src)])
        emit(combo, windows, pos, res, 0, four_vals, dd_vals)
    return items


def write_items(output_file: str, items: list[dict[str, Any]], stat_config) -> None:
    """Appends score rows and ``.U.log`` / ``.Q.log`` rows with the reference's
    text layout (feature_preprocessor.py:193-258); lines are assembled in memory and written
    with one call per file."""
    names = [s for s in stat_config.root.keys() if s in ("U", "Q") or stat_config.root[s] is True]
    rows = []
    for it in items:
        parts = []
        n_src = len(it["src_pop_list"])
        for s in names:
            v = it.get(s)
            if isinstance(v, list) and len(v) == n_src:
                parts.extend("" if x is None else str(x) for x in v)
            else:
                if isinstance(v, list):
                    v = v[0] if v else ""
                parts.append("" if v is None else str(v))
        rows.append(
            f"{it['chr_name']}\t{it['start']}\t{it['end']}\t{it['ref_pop']}\t{it['tgt_pop']}\t"
            f"{','.join(it['src_pop_list'])}\t{it['out_pop']}\t{it['nsnps']}\t" + "\t".join(parts) + "\n"
        )
    with open(output_file, "a") as f:
        f.write("".join(rows))
    for key in ("U", "Q"):
        if key not in stat_config.root:
            continue
        rows = []
        for it in items:
            c = it["cdd_pos"][key]
            if c.size == 0:
                txt = "NA"
            else:
                prefix = f"{it['chr_name']}:"
                txt = ",".join([prefix + p for p in map(str, c.tolist())])
            rows.append(f"{it['chr_name']}\t{it['start']}\t{it['end']}\t{txt}\n")
        with open(Path(output_file).with_suffix(f".{key}.log"), "a") as f:
            f.write("".join(rows))


class DeviceRows:
    """A ``score_populations`` sink for ``write="device"``: the score rows kept as numpy columns, one
    block per (chromosome, combination) run of windows in the order ``write_items`` writes them, and
    formatted on the GPU by ``write``.  No per-window Python object is made; the values are the ones
    ``emit`` puts in the item dicts (``four_pop_values`` / ``dd_values`` lists as float64 arrays), so the
    text is byte for byte that of ``write_items``."""

    def __init__(self, stat_config):
        root = stat_config.root
        self.names = [s for s in root.keys() if s in ("U", "Q") or root[s] is True]  # write_items' columns
        self.logs = [k for k in ("U", "Q") if k in root]
        self.blocks: list[dict] = []
        self._seen: dict = {}  # (id, what) -> (object, its array): a list or result converted once

    def _once(self, obj, what, make):
        hit = self._seen.get((id(obj), what))
        if hit is None or hit[0] is not obj:
            hit = self._seen[(id(obj), what)] = (obj, make())
        return hit[1]

    def __call__(self, combo, windows, pos, res, j, four_vals, dd_vals, chrom, at=0):
        ref_pop, tgt_pop, src_comb, out_pop = combo
        n = len(windows)
        cols = slice(at, at + n)
        out_name = "NA" if out_pop is None else out_pop
        b = {"chrom": f"{chrom}", "combo": f"{ref_pop}\t{tgt_pop}\t{','.join(src_comb)}\t{out_name}",
             "bounds": self._once(windows, "bounds", lambda: np.asarray(windows, dtype=np.int64).reshape(-1, 2))}
        if res is not None:
            b["nsnps"] = res.nsnps[j, cols]
        else:  # as emit: no statistic scored, or a region without data (empty positions)
            b["nsnps"] = np.array([int(np.count_nonzero((pos >= s_) & (pos <= e_))) for s_, e_ in windows], dtype=np.int32)
        zeros = np.zeros(n, dtype=np.int64)
        for key in ("u", "q"):
            if key.upper() not in self.names:
                continue
            if res is None:  # every window has nsnps == 0: no candidates are read
                b[key] = np.full(n, np.nan) if key == "q" else zeros
                b[key + "_start"], b[key + "_pool"] = zeros, None
                if key == "q":
                    b["q_cnt"] = zeros
                continue
            b[key] = getattr(res, key)[j, cols]
            b[key + "_start"] = getattr(res, key + "_start")[j, cols]
            if key == "q":
                b["q_cnt"] = res.q_cnt[j, cols]
            cand = getattr(res, key + "_cand")
            used = cand.shape[1]
            if getattr(res, "totals", None) is not None:
                used = min(int(res.totals[j, 0 if key == "u" else 1]), used)
            # (identity of job j's list, the list, the results: kept alive so that no later results share the id)
            b[key + "_pool"] = ((id(res), key, j), cand[j, :used], res)
        n_src = len(src_comb)
        field, vals = [], []
        for s in self.names:
            if s in ("U", "Q"):
                field.append(_cabi.FMT_U if s == "U" else _cabi.FMT_Q)
                continue
            for k in range(max(n_src, 1)):  # one per source; a row with nsnps == 0 prints nan in each
                src = dd_vals if s == "DD" else (four_vals[s] if four_vals is not None else None)
                if src is None or k >= n_src:
                    vals.append(np.full(n, np.nan))
                else:
                    vals.append(self._once(src[k], "f64", lambda: np.asarray(src[k], dtype=np.float64))[cols])
                field.append(len(vals) - 1)
        b["field"] = field
        b["vals"] = np.stack(vals, axis=1) if vals else np.zeros((n, 0))
        self.blocks.append(b)

    def format(self, engine, encoding: str):
        """The three texts (score rows, ``.U.log``, ``.Q.log``) as uint8 arrays, from the GPU."""
        blocks = [b for b in self.blocks if len(b["bounds"])]
        if not blocks:
            return [np.zeros(0, dtype=np.uint8)] * 3
        field = blocks[0]["field"]
        if any(b["field"] != field for b in blocks):
            raise ValueError("every combination of one score file has the same number of source populations")
        strings, block_str, at = [], [], 0
        for b in blocks:
            for key in ("chrom", "combo"):
                raw = b[key].encode(encoding)
                block_str += [at, len(raw)]
                strings.append(raw)
                at += len(raw)
        strings = b"".join(strings)
        cat = lambda key, dt: np.ascontiguousarray(np.concatenate([b[key] for b in blocks]), dtype=dt)
        bounds = np.concatenate([b["bounds"] for b in blocks])
        keep = {
            "block_rows": np.cumsum([0] + [len(b["bounds"]) for b in blocks], dtype=np.int64),
            "block_str": np.asarray(block_str, dtype=np.int64),
            "start": np.ascontiguousarray(bounds[:, 0]), "end": np.ascontiguousarray(bounds[:, 1]),
            "nsnps": cat("nsnps", np.int32), "field": np.asarray(field, dtype=np.int32),
            "vals": cat("vals", np.float64),
        }
        for key in ("u", "q"):
            if key.upper() not in self.names:
                continue
            pools, base, n_pool = [], {}, 0
            starts = []
            for b in blocks:
                p = b[key + "_pool"]
                if p is not None and p[0] not in base:
                    base[p[0]] = n_pool
                    pools.append(p[1])
                    n_pool += len(p[1])
                starts.append(b[key + "_start"] + (0 if p is None else base[p[0]]))
            keep[key] = cat(key, np.float64 if key == "q" else np.int64)
            keep[key + "_start"] = np.ascontiguousarray(np.concatenate(starts), dtype=np.int64)
            keep[key + "_cand"] = np.ascontiguousarray(np.concatenate(pools) if pools else np.zeros(0), dtype=np.int32)
            if key == "q":
                keep["q_cnt"] = cat("q_cnt", np.int32)
        inp = _cabi.FormatInput()
        inp.n_blocks, inp.n_rows = len(blocks), len(bounds)
        keep["strings"] = np.frombuffer(strings, dtype=np.uint8)
        inp.strings_len = len(strings)
        for name, arr in keep.items():
            setattr(inp, name, arr.ctypes.data if arr.size else None)
        inp.n_u_cand = keep["u_cand"].size if "u_cand" in keep else 0
        inp.n_q_cand = keep["q_cand"].size if "q_cand" in keep else 0
        inp.n_fields, inp.n_vals = len(field), keep["vals"].shape[1]
        return engine.format_scores(inp)

    def write(self, output_file: str, engine) -> None:
        """Appends the rows to the score file and the ``.U.log`` / ``.Q.log`` files: one write each."""
        rows, u_log, q_log = self.format(engine, locale.getpreferredencoding(False))
        with open(output_file, "ab") as f:
            f.write(memoryview(rows))
        for key, text in (("U", u_log), ("Q", q_log)):
            if key in self.logs:
                with open(Path(output_file).with_suffix(f".{key}.log"), "ab") as f:
                    f.write(memoryview(text))


class ChunkPreprocessor:
    """Drop-in for ``sai.preprocessors.ChunkPreprocessor`` on the U/Q path."""

    def __init__(
        self,
        vcf_file: str,
        ref_ind_file: str,
        tgt_ind_file: str,
        src_ind_file: str,
        out_ind_file: Optional[str],
        win_len: int,
        win_step: int,
        output_file: str,
        ploidy_config,
        stat_config,
        anc_allele_file: Optional[str] = None,
        num_src: int = 1,
        device: int = 0,
        ingest: str = "host",
        inflate: str = "host",
        dd_ingest: str = "host",
    ):
        """``ingest="device"`` parses the VCF on the GPU (``vcf_device``): the text is copied to the
        device and parsed there straight into the packed tiles, which all combinations are scored
        from.  The items are identical to ``"host"``; chunks the device reader does not cover (DD,
        more than 16 populations, ancestral alleles longer than 7 bytes, source ploidies that differ
        from their positions in a combination) are read on the host automatically.
        ``inflate="device"`` (with ``ingest="device"``) also inflates a bgzip file on the GPU: only
        the compressed blocks cross PCIe.  Plain text and single-member gzip are read as before.
        ``dd_ingest="device"`` (with ``ingest="device"``) reads DD chunks on the device too: the
        genotype pass keeps the raw values of missing calls DD needs (the negative-value table) in
        HBM next to the tiles, so DD no longer sends the chunk to host ingest; same items."""
        from .vcf import parse_ind_file

        if ingest not in ("host", "device"):
            raise ValueError(f"ingest must be 'host' or 'device', not {ingest!r}")
        if inflate not in ("host", "device"):
            raise ValueError(f"inflate must be 'host' or 'device', not {inflate!r}")
        if inflate == "device" and ingest != "device":
            raise ValueError("inflate='device' needs ingest='device'")
        if dd_ingest not in ("host", "device"):
            raise ValueError(f"dd_ingest must be 'host' or 'device', not {dd_ingest!r}")
        if dd_ingest == "device" and ingest != "device":
            raise ValueError("dd_ingest='device' needs ingest='device'")
        self.ingest = ingest
        self.inflate = inflate
        self.dd_ingest = dd_ingest

        self.vcf_file = vcf_file
        self.ref_ind_file = ref_ind_file
        self.tgt_ind_file = tgt_ind_file
        self.src_ind_file = src_ind_file
        self.out_ind_file = out_ind_file
        self.win_len = win_len
        self.win_step = win_step
        self.output_file = output_file
        self.ploidy_config = ploidy_config
        self.stat_config = stat_config
        self.anc_allele_file = anc_allele_file
        self.num_src = len(parse_ind_file(src_ind_file).keys())
        self.anc_allele_available = anc_allele_file is not None
        self.engine = HostEngine(device)  # picklable; CUDA context created in run()

    def run(self, chr_name: str, start: int, end: int) -> list[dict[str, Any]]:
        return self.run_into(chr_name, start, end, None)

    def run_into(self, chr_name: str, start: int, end: int, sink) -> list[dict[str, Any]]:
        """``run``, with the rows handed to ``sink`` (see ``score_populations``) when it is given."""
        from .vcf import read_data

        if self.win_len <= 0:
            raise ValueError("`win_len` must be greater than 0.")
        if self.win_step < 0:
            raise ValueError("`win_step` must be non-negative.")
        if self.ingest == "device":
            items = self._run_device(chr_name, start, end, sink)
            if items is not None:
                return items
        groups = read_data(
            vcf_file=self.vcf_file,
            chr_name=chr_name,
            ploidy_config=self.ploidy_config,
            ref_ind_file=self.ref_ind_file,
            tgt_ind_file=self.tgt_ind_file,
            src_ind_file=self.src_ind_file,
            out_ind_file=self.out_ind_file,
            anc_allele_file=self.anc_allele_file,
            start=start,
            end=end,
        )
        ref_data, ref_samples = groups["ref"]
        tgt_data, tgt_samples = groups["tgt"]
        src_data, src_samples = groups["src"]
        out_data, out_samples = groups["outgroup"]
        if start is None and end is None:
            windows = {t: split_genome(tgt_data[t].POS, self.win_len, self.win_step) for t in tgt_samples}
        else:
            wins = chunk_windows(start, end, self.win_len, self.win_step)
            windows = {t: wins for t in tgt_samples}
        if ref_data is None or tgt_data is None or src_data is None:
            return self._empty_items(chr_name, windows, ref_samples, tgt_samples, src_samples, out_samples, sink)
        return score_populations(
            chr_name, windows, ref_data, tgt_data, src_data, self.ploidy_config, self.stat_config,
            self.anc_allele_available, self.engine, out_data=out_data, num_src=self.num_src, sink=sink,
        )

    def device_fallback(self, chr_name: str, start=None, end=None) -> Optional[str]:
        """Why ``run(chr_name, start, end)`` reads this chunk on the host although ``ingest="device"``
        (``None``: it is read on the device)."""
        from .vcf import read_anc_or_error
        from .vcf_device import fallback_reason, read_plan

        plan, _, _ = read_plan(self.vcf_file, chr_name, self.ploidy_config, self.ref_ind_file, self.tgt_ind_file,
                               self.src_ind_file, self.out_ind_file)
        anc, _ = read_anc_or_error(self.anc_allele_file, chr_name, start, end)
        return fallback_reason(self.stat_config, self.ploidy_config, plan, anc, chr_name, self.num_src,
                               self.dd_ingest)

    def _run_device(self, chr_name, start, end, sink=None):
        import warnings

        from .vcf import read_anc_or_error
        from .vcf_device import _wants_outgroup, fallback_reason, read_loaded, read_plan, wants_dd

        with warnings.catch_warnings(record=True) as caught:  # warned once, by the read that is used
            warnings.simplefilter("always")
            plan, requests, out = read_plan(self.vcf_file, chr_name, self.ploidy_config, self.ref_ind_file,
                                            self.tgt_ind_file, self.src_ind_file, self.out_ind_file)
        anc, anc_error = read_anc_or_error(self.anc_allele_file, chr_name, start, end)
        if fallback_reason(self.stat_config, self.ploidy_config, plan, anc, chr_name, self.num_src,
                           self.dd_ingest) is not None:
            return None
        for w in caught:
            warnings.warn_explicit(w.message, w.category, w.filename, w.lineno)
        try:
            loaded = read_loaded(self.engine, self.vcf_file, chr_name, plan, requests, out, anc, anc_error, start, end,
                                 with_outgroup=_wants_outgroup(self.stat_config), inflate=self.inflate,
                                 neg_table=self.dd_ingest == "device" and wants_dd(self.stat_config))
        except (KeyError, OSError) as e:
            region = chr_name if start is None and end is None else f"{chr_name}:{start}-{end}"
            raise ValueError(f"Failed to read VCF file {self.vcf_file} from {region}: {e}") from e
        if loaded is None:  # no #CHROM line: the host reader decides what that means
            return None
        (ref_pops, ref_samples), (tgt_pops, tgt_samples) = loaded.groups["ref"], loaded.groups["tgt"]
        (src_pops, src_samples), (out_pops, out_samples) = loaded.groups["src"], loaded.groups["outgroup"]
        if start is None and end is None:
            windows = {t: split_genome(loaded.pos, self.win_len, self.win_step) for t in tgt_samples}
        else:
            wins = chunk_windows(start, end, self.win_len, self.win_step)
            windows = {t: wins for t in tgt_samples}
        if ref_pops is None or tgt_pops is None or src_pops is None:
            return self._empty_items(chr_name, windows, ref_samples, tgt_samples, src_samples, out_samples, sink)
        names = lambda pops: {p: None for p in pops} if pops else None
        return score_populations(
            chr_name, windows, names(ref_pops), names(tgt_pops), names(src_pops), self.ploidy_config, self.stat_config,
            self.anc_allele_available, self.engine, out_data=names(out_pops), num_src=self.num_src, loaded=loaded,
            sink=sink,
        )

    def _empty_items(self, chr_name, windows, ref_samples, tgt_samples, src_samples, out_samples=None, sink=None):
        # no data in the region: window_generator.py:249-289 (product over the outgroup populations
        # too, :269-273) + feature_preprocessor.py:131-144
        stats = [s for s in self.stat_config.root.keys() if s in ("U", "Q")]
        four = [s for s in self.stat_config.root.keys() if s in ("Danc", "Dplus", "df", "fd", "DD")]
        items = []
        for ref_pop, tgt_pop, src_comb, out_pop in product(
            ref_samples, tgt_samples, list(combinations(src_samples.keys(), self.num_src)), out_samples or [None]
        ):
            if sink is not None:  # no positions: every window has nsnps == 0
                sink((ref_pop, tgt_pop, src_comb, out_pop), windows[tgt_pop], np.zeros(0, dtype=np.int64), None, 0,
                     None, None, chr_name)
                continue
            for start, end in windows[tgt_pop]:
                it = {
                    "chr_name": chr_name, "start": start, "end": end, "ref_pop": ref_pop, "tgt_pop": tgt_pop,
                    "src_pop_list": src_comb, "out_pop": "NA" if out_pop is None else out_pop, "nsnps": 0,
                    "cdd_pos": {},
                }
                for s in four:
                    it[s] = [np.nan for _ in src_comb] if len(src_comb) > 1 else np.nan
                for s in stats:
                    it[s] = np.nan
                    it["cdd_pos"][s] = np.array([])
                items.append(it)
        return items

    def process_items(self, items: list[dict[str, Any]]) -> None:
        write_items(self.output_file, items, self.stat_config)
