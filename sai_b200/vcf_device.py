"""Device VCF ingest: the VCF text goes to the GPU and is parsed there straight into the packed
tiles (``sai_engine_vcf_*``, ``vcf_device.cu``), which stay resident in the engine for scoring.

The host only reads or inflates bytes and copies them: ``_scan_text`` / ``_scan_sorted_region``
hand their text buffers to ``sai_engine_vcf_feed`` exactly as they hand them to the host parser,
so plain, bgzip and gzip files and region reads all work the same way.  With ``inflate="device"``
a bgzip file's blocks go over compressed instead and are inflated on the device
(``sai_engine_vcf_feed_bgzf_device``); a corrupt block repeats the read with host inflate, which
raises the host path's error.  The records and values
are those of ``read_data`` (the host parser is the specification); the layout is the one the host
path packs, so the tiles are comparable byte for byte.

With ``neg_table=True`` (DD with ``dd_ingest="device"``) the genotype pass also keeps the raw value
of every missing call: the negative-value table DD reads next to the tiles (``sai_b200.h``, N4),
equal entry for entry to ``encode.negative_table`` of ``read_data``'s matrices and resident in the
engine for ``HostEngine.dd_sums``.
"""

from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _cabi
from .encode import make_layout
from .vcf import _scan_sorted_region, _scan_text, anc_table, population_plan, read_anc_or_error

GROUPS = ("ref", "tgt", "src", "outgroup")


class LoadedChunk:
    """One VCF region parsed on the device: its tiles, positions and windows live in ``engine``.
    ``index[(group, population)]`` = population index in ``layout``; ``groups[group] =
    (population names or None, samples)`` mirrors what ``read_data`` returns per group.  ``neg``:
    the engine also holds the chunk's negative-value table (``read_loaded(..., neg_table=True)``)."""

    def __init__(self, layout, pos, index, groups, neg=False):
        self.layout, self.pos, self.index, self.groups, self.neg = layout, pos, index, groups, neg

    @property
    def n_sites(self) -> int:
        return int(self.pos.shape[0])


def fallback_reason(stat_config, ploidy_config, plan, anc, chr_name: str, num_src: int,
                    dd_ingest: str = "host") -> Optional[str]:
    """Why a chunk has to be read on the host (``None``: it can be read on the device).
    DD needs the raw values of missing calls: with ``dd_ingest="host"`` that table is built by the
    host, with ``"device"`` the genotype pass keeps it (``read_loaded(..., neg_table=True)``); one
    layout holds at most ``SAI_MAX_POPS`` populations; the native parsers take ancestral alleles of at most 7 bytes;
    a source population is scored with the ploidy of its position in the combination
    (feature_preprocessor.py:160,168-170), which one layout can only hold when that is its own."""
    if dd_ingest not in ("host", "device"):
        raise ValueError(f"dd_ingest must be 'host' or 'device', not {dd_ingest!r}")
    if dd_ingest == "host" and wants_dd(stat_config):
        return "DD is enabled"
    if sum(len(pops) for group, _, pops in plan if group != "outgroup" or _wants_outgroup(stat_config)) > _cabi.MAX_POPS:
        return f"more than {_cabi.MAX_POPS} populations"
    if anc is not None and anc_table(anc) is None:
        return "an ancestral allele is longer than 7 bytes"
    if not 1 <= len(chr_name.encode()) <= 255:
        return "chromosome name outside 1..255 bytes"
    src = [pops for group, _, pops in plan if group == "src"]
    if src:
        from itertools import combinations

        positional = list(ploidy_config.get_ploidy("src"))
        for comb in combinations([p for p, _, _ in src[0]], num_src):
            if [ploidy_config.get_ploidy("src", name) for name in comb] != positional[: len(comb)]:
                return "source ploidies differ from their positions in a combination"
    return None


def wants_dd(stat_config) -> bool:
    return any(s == "DD" and stat_config.root[s] is True for s in stat_config.root)


def _wants_outgroup(stat_config) -> bool:
    return any(s in ("Danc", "Dplus", "df", "fd") and stat_config.root[s] is True for s in stat_config.root)


def read_plan(vcf_file, chr_name, ploidy_config, ref_ind_file, tgt_ind_file, src_ind_file, out_ind_file):
    """The population plan of ``read_data`` (same errors and warnings)."""
    files = (ref_ind_file, tgt_ind_file, src_ind_file, out_ind_file)
    return population_plan(tuple(zip(GROUPS, files)), ploidy_config)


def _pops_and_groups(plan, out, with_outgroup):
    pops = [(group, name, a, b) for group, _, gp in plan for name, a, b in gp
            if group != "outgroup" or with_outgroup]
    groups = dict(out)
    for group, samples, gp in plan:
        groups[group] = ([name for name, _, _ in gp] or None, samples)
    index = {(group if group != "outgroup" else "out", name): i for i, (group, name, _, _) in enumerate(pops)}
    return pops, groups, index


def _ingest(engine, vcf_file: str, pops, requests, label: str, inflate: str, begin_session, finish_session,
            region=None, neg_table: bool = False):
    """The device parse shared by ``read_loaded`` and ``read_genome``: header columns, the text fed
    to the engine's session (``region = (chr_name, start, end)``: a sorted-region read when the file
    allows it), then the finish and its retries -- a wider layout (``SAI_E_DOMAIN``), more sites
    (``SAI_E_CAPACITY``: and a larger negative-value table with ``neg_table``), host inflate after a
    corrupt block (``SAI_E_CORRUPT``).
    ``begin_session(lay, cols, n_file_samples, text_bytes_hint, min_sites)`` opens the session;
    ``finish_session(pos)`` returns ``(rc, n_sites, vmax, extra)``.  Returns ``(layout, pos,
    extra)``; ``pos`` is ``None`` when the file has no ``#CHROM`` line, ``extra`` is ``None`` when it
    has no record line."""
    if inflate not in ("host", "device"):
        raise ValueError(f"inflate must be 'host' or 'device', not {inflate!r}")
    lib = _cabi.load()
    n_samples = [b - a for _, _, a, b in pops]
    ploidy = [requests[a][1] for _, _, a, _ in pops]
    empty = np.empty(0, dtype=np.int32)
    bits, min_sites, min_entries = None, 0, 0
    for _attempt in range(5):
        lay = make_layout(n_samples, ploidy, bits)
        state = {"cols": None, "n_file": 0, "hint": 0, "begun": False, "fed": 0}
        consumed = C.c_int64(0)

        def on_header(line: bytes):
            names = line.decode().rstrip("\r").split("\t")[9:]
            col = {n: i for i, n in enumerate(names)}
            try:
                every = [col[name] for name, _ in requests]  # every population's samples, parsed or not (read_data's errors)
                state["cols"] = np.ascontiguousarray([every[i] for _, _, a, b in pops for i in range(a, b)],
                                                     dtype=np.int32)
            except KeyError as e:
                raise ValueError(f"Failed to read VCF file {vcf_file} from {label}: {e}") from e
            state["n_file"] = len(names)

        def on_size_hint(text_bytes: int):
            state["hint"] = int(text_bytes)

        def begin(length: int) -> None:
            if not state["begun"]:
                _cabi.check(lib.sai_engine_set_vcf_neg_table(engine._handle(), int(neg_table), min_entries))
                begin_session(lay, state["cols"], state["n_file"], max(state["hint"], length), min_sites)
                state["begun"] = True

        def on_lines(addr: int, length: int) -> int:
            begin(length)
            _cabi.check(lib.sai_engine_vcf_feed(engine._handle(), addr, length, C.byref(consumed)))
            state["fed"] += int(consumed.value)
            return int(consumed.value)

        def on_bgzf(base: int, block_off, out_off, n_blocks: int, skip: int) -> None:
            """A whole bgzip file: inflated by the engine's threads straight into its pinned ring."""
            if inflate == "device":
                return on_bgzf_device(base, block_off, out_off, n_blocks, skip, True)
            text = int(out_off[n_blocks]) - skip
            begin(text)
            _cabi.check(lib.sai_engine_vcf_feed_bgzf(engine._handle(), base, block_off.ctypes.data, out_off.ctypes.data,
                                                     n_blocks, skip))
            state["fed"] += text + 1

        def on_bgzf_device(base: int, block_off, out_off, n_blocks: int, skip: int, at_eof: bool) -> None:
            """bgzip blocks (whole file or region): copied compressed and inflated on the device.  A
            corrupt block fails in the finish (SAI_E_CORRUPT), like one the device finds."""
            text = int(out_off[n_blocks]) - skip
            begin(text)
            rc = lib.sai_engine_vcf_feed_bgzf_device(engine._handle(), base, block_off.ctypes.data, out_off.ctypes.data,
                                                     n_blocks, skip, int(at_eof))
            if rc != _cabi.E_CORRUPT:
                _cabi.check(rc)
            state["fed"] += text + 1

        handled = False
        if region is not None:
            handled = _scan_sorted_region(vcf_file, region[0], int(region[1]), int(region[2]), on_header, on_lines,
                                          on_bgzf=on_bgzf_device if inflate == "device" else None)
        if not handled:
            _scan_text(vcf_file, on_header, on_lines, on_size_hint=on_size_hint, on_bgzf=on_bgzf)
        if state["cols"] is None:
            return lay, None, None
        if not state["begun"]:  # no record lines at all
            return lay, empty, None
        # a kept record is >= 11 bytes (CHROM, nine tabs, newline): room for every one (np.empty commits
        # no pages); a genome parse adds up to a tile of padding per chromosome
        pos = np.empty(state["fed"] // 11 + 1024 + 32 * _cabi.MAX_CHROMS, dtype=np.int32)
        rc, n_sites, vmax, extra = finish_session(pos)
        if rc == _cabi.E_DOMAIN:  # the host path's retry rule (encode.bits_for)
            bits = [int(lib.sai_bits_for_max_value(int(v))) for v in vmax]
            continue
        if rc == _cabi.E_CAPACITY:
            min_sites = int(n_sites)
            if neg_table:  # the entries the table needs (its first capacity is an estimate)
                need = int(lib.sai_engine_loaded_neg_table(engine._handle(), None, None, None, None, 0))
                if need < 0:
                    _cabi.check(need)
                min_entries = max(min_entries, need)
            continue
        if rc == _cabi.E_CORRUPT:  # read again with host inflate: it raises the host path's error
            inflate = "host"
            continue
        if rc == _cabi.E_ORDER:
            return lay, pos[:0], rc
        _cabi.check(rc)
        n = int(n_sites)
        return lay, (pos[:n].copy() if n * 4 < pos.shape[0] else pos[:n]), extra
    raise _cabi.SaiError("device ingest did not converge on a layout")


def read_loaded(engine, vcf_file: str, chr_name: str, plan, requests, out, anc, anc_error, start=None, end=None,
                with_outgroup: bool = True, inflate: str = "host", neg_table: bool = False) -> Optional[LoadedChunk]:
    """Parses the records of ``chr_name`` (``start <= POS <= end`` when both are given) on the
    device into ``engine``'s resident tiles, one layout for every population of ``plan`` (the
    outgroup only with ``with_outgroup``).  ``None`` when the file has no ``#CHROM`` line.
    ``inflate="device"``: bgzip blocks are inflated on the device.  ``neg_table``: the engine also
    keeps the negative-value table DD reads (``LoadedChunk.neg``)."""
    lib = _cabi.load()
    pops, groups, index = _pops_and_groups(plan, out, with_outgroup)
    if not pops:
        return LoadedChunk(None, np.empty(0, dtype=np.int32), index, groups)
    anc_pos, anc_buf, n_anc = (None, None, 0) if anc is None else anc_table(anc)
    region = (int(start), int(end)) if (start is not None and end is not None) else (1, 0)

    def begin_session(lay, cols, n_file, hint, min_sites):
        _cabi.check(lib.sai_engine_vcf_begin(
            engine._handle(), C.byref(lay), chr_name.encode(), region[0], region[1], cols.ctypes.data,
            int(cols.shape[0]), anc_pos.ctypes.data if n_anc else None, anc_buf if n_anc else None,
            n_anc, n_file, hint, min_sites))

    def finish_session(pos):
        n_sites, vmax = C.c_int64(0), (C.c_int32 * len(pops))()
        rc = lib.sai_engine_vcf_finish(engine._handle(), C.byref(n_sites), vmax, pos.ctypes.data, pos.shape[0])
        return rc, n_sites.value, vmax, True

    label = chr_name if start is None and end is None else f"{chr_name}:{start}-{end}"
    lay, pos, extra = _ingest(engine, vcf_file, pops, requests, label, inflate, begin_session, finish_session,
                              (chr_name, start, end) if (start is not None and end is not None) else None, neg_table)
    if pos is None:
        return None
    if anc_error is not None and pos.size:  # records but no ancestral allele in the region: the reference raises
        raise anc_error
    if pos.size == 0:
        groups = {g: (None, v[1]) for g, v in groups.items()}
    return LoadedChunk(lay, pos, index, groups, neg=neg_table and extra is not None)


class LoadedGenome:
    """Every chromosome of a table parsed in one device pass: the tiles of all of them resident in
    ``engine``, chromosome ``c``'s sites at ``[first_site[c], first_site[c] + n_sites[c])`` (a tile
    boundary; ``first_site`` -1: no site), ``pos[c]`` its positions.  ``span[c] = (first POS, last POS,
    records)`` in file order over all its records, as ``vcf.chromosome_span`` counts them (``None``:
    no record).  ``index`` / ``groups`` / ``neg`` as ``LoadedChunk``'s; chromosome ``c``'s rows of
    the negative-value table count sites from ``first_site[c]``."""

    def __init__(self, layout, chroms, pos_all, index, groups, names, neg=False):
        self.layout, self.index, self.groups, self.names, self.neg = layout, index, groups, list(names), neg
        self.first_site = [int(c.first_site) for c in chroms]
        self.n_sites = [int(c.n_sites) for c in chroms]
        self.span = [(int(c.first_pos), int(c.last_pos), int(c.n_records)) if c.n_records > 0 else None for c in chroms]
        self.pos = [pos_all[f : f + n] if n else pos_all[:0] for f, n in zip(self.first_site, self.n_sites)]
        self.total_sites = int(pos_all.shape[0])


def genome_tables(chr_names, anc_allele_file):
    """The chromosome table (names back to back + offsets) and the ancestral-allele tables of all
    chromosomes concatenated (``anc_off[c] .. anc_off[c + 1]`` = chromosome ``c``'s entries, each
    slice equal to ``anc_table(read_anc_arrays(file, c, None, None))``).  The BED file is read once.
    Returns ``(names, name_off, anc)``: ``anc = (pos int32, alleles as 8-byte records, anc_off)``, or
    ``None`` without a file or when an allele is longer than 7 bytes (``fallback_reason``)."""
    from .vcf import AncAlleles

    enc = [c.encode() for c in chr_names]
    names = b"".join(enc)
    name_off = np.zeros(len(enc) + 1, dtype=np.int32)
    name_off[1:] = np.cumsum([len(e) for e in enc])
    if not anc_allele_file:
        return names, name_off, None
    import pandas as pd

    try:
        df = pd.read_csv(anc_allele_file, sep=r"\s+", header=None, usecols=[0, 2, 3], names=["chrom", "pos", "allele"],
                         dtype={"chrom": str, "pos": np.int64, "allele": str}, engine="c", comment=None,
                         keep_default_na=False)
    except FileNotFoundError as exc:
        raise FileNotFoundError(f"File {anc_allele_file} not found.") from exc
    except pd.errors.EmptyDataError:
        df = pd.DataFrame({"chrom": [], "pos": np.array([], dtype=np.int64), "allele": []})
    chrom, pos_all, allele_all = df["chrom"].to_numpy(), df["pos"].to_numpy(), df["allele"].to_numpy()
    parts_pos, parts_all, anc_off = [], [], [0]
    for c in chr_names:
        keep = chrom == c
        pos, allele = pos_all[keep], allele_all[keep]
        if pos.size == 0:
            anc_off.append(anc_off[-1])
            continue
        _, first_of_reversed = np.unique(pos[::-1], return_index=True)  # read_anc_arrays: last occurrence wins
        idx = pos.size - 1 - first_of_reversed
        t = anc_table(AncAlleles(pos[idx], allele[idx]))
        if t is None:
            return names, name_off, None
        parts_pos.append(t[0])
        parts_all.append(t[1])
        anc_off.append(anc_off[-1] + t[2])
    anc_pos = np.concatenate(parts_pos) if parts_pos else np.empty(0, dtype=np.int32)
    return names, name_off, (np.ascontiguousarray(anc_pos), b"".join(parts_all), np.asarray(anc_off, dtype=np.int64))


def read_genome(engine, vcf_file: str, chr_names, plan, requests, out, tables, with_outgroup: bool = True,
                inflate: str = "host", neg_table: bool = False):
    """Parses every chromosome of ``chr_names`` in one pass over ``vcf_file`` into ``engine``'s
    resident tiles (``sai_engine_vcf_genome_*``).  ``tables`` = ``genome_tables(chr_names, file)``
    (its ``anc`` ``None`` without an ancestral-allele file).  Returns a
    ``LoadedGenome``; ``None`` when the file has no ``#CHROM`` line, no populations are parsed, or a
    chromosome's records resume after another chromosome's (``SAI_E_ORDER``): such files are read
    one chromosome at a time.  ``neg_table`` as ``read_loaded``'s."""
    lib = _cabi.load()
    names, name_off, anc = tables
    pops, groups, index = _pops_and_groups(plan, out, with_outgroup)
    if not pops:
        return None
    n = len(chr_names)
    chroms = (_cabi.VcfChrom * n)()

    def begin_session(lay, cols, n_file, hint, min_sites):
        anc_pos, anc_buf, anc_off = anc if anc is not None else (None, None, None)
        has = anc is not None and int(anc_off[-1]) > 0
        _cabi.check(lib.sai_engine_vcf_genome_begin(
            engine._handle(), C.byref(lay), names, name_off.ctypes.data, n, cols.ctypes.data, int(cols.shape[0]),
            anc_pos.ctypes.data if has else None, anc_buf if has else None, anc_off.ctypes.data if has else None,
            n_file, hint, min_sites))

    def finish_session(pos):
        n_sites, vmax = C.c_int64(0), (C.c_int32 * len(pops))()
        rc = lib.sai_engine_vcf_genome_finish(engine._handle(), C.byref(n_sites), vmax, chroms, pos.ctypes.data,
                                              pos.shape[0])
        return rc, n_sites.value, vmax, chroms

    lay, pos, extra = _ingest(engine, vcf_file, pops, requests, ",".join(chr_names), inflate, begin_session,
                              finish_session, neg_table=neg_table)
    if pos is None or extra == _cabi.E_ORDER:
        return None
    neg = neg_table and extra is not None
    if extra is None:  # no record line: nothing found
        chroms = (_cabi.VcfChrom * n)(*[_cabi.VcfChrom(0, 0, 0, -1, 0) for _ in range(n)])
    return LoadedGenome(lay, chroms, pos, index, groups, chr_names, neg=neg)


def read_region(engine, vcf_file, chr_name, ploidy_config, ref_ind_file, tgt_ind_file, src_ind_file, out_ind_file,
                anc_allele_file, start=None, end=None, with_outgroup=True):
    """Plan, ancestral-allele table and device parse in one call (tests, tools)."""
    plan, requests, out = read_plan(vcf_file, chr_name, ploidy_config, ref_ind_file, tgt_ind_file, src_ind_file,
                                    out_ind_file)
    anc, anc_error = read_anc_or_error(anc_allele_file, chr_name, start, end)
    return read_loaded(engine, vcf_file, chr_name, plan, requests, out, anc, anc_error, start, end, with_outgroup)
