"""Top-level ``score`` with the signature and file outputs of the reference's
``sai.sai.score`` (sai/sai.py:33-151), running the U/Q path on the GPU.

Every statistic of the reference's registry is computed on the GPU: U, Q, the
four site-pattern statistics (Danc, Dplus, df, fd) and DD.  In a reference-side integration ``score`` itself stays
untouched and only the ``ChunkPreprocessor`` it constructs is swapped
(INTEGRATION.md).
"""

from __future__ import annotations

import os
import warnings
from pathlib import Path
from typing import Sequence

import numpy as np

from .configs import load_config
from .preprocessors import ChunkPreprocessor, DeviceRows
from .generators import ChunkGenerator


def _load_checked_config(config: str, anc_allele_file):
    """The configuration, refused as the reference refuses it (sai/sai.py:79-84) and for statistics
    this port does not compute."""
    cfg = load_config(config)
    stat_config = cfg.statistics
    others = [s for s in stat_config.root if s not in ("U", "Q", "Danc", "Dplus", "df", "fd", "DD") and stat_config.root[s] is not False]
    if others:
        raise NotImplementedError(
            f"sai_b200 covers U, Q, Danc, Dplus, df, fd and DD; the configuration also enables {others}."
        )
    if anc_allele_file is None:  # sai/sai.py:79-84
        for stat_name in stat_config.root.keys():
            if stat_name in ["fd", "df", "Danc", "Dplus"]:
                raise ValueError(
                    f"The {stat_name} statistic requires polarized data, please provide the ancestral allele information with `--anc-alleles`."
                )
    return cfg


def _preprocessor(vcf_file, cfg, win_len, win_step, anc_allele_file, output_file, device, ingest, inflate, dd_ingest):
    pop_config = cfg.populations
    return ChunkPreprocessor(
        vcf_file=vcf_file,
        ref_ind_file=pop_config.get_population("ref"),
        tgt_ind_file=pop_config.get_population("tgt"),
        src_ind_file=pop_config.get_population("src"),
        out_ind_file=pop_config.get_population("outgroup"),
        win_len=win_len,
        win_step=win_step,
        output_file=output_file,
        ploidy_config=cfg.ploidies,
        stat_config=cfg.statistics,
        anc_allele_file=anc_allele_file,
        device=device,
        ingest=ingest,
        inflate=inflate,
        dd_ingest=dd_ingest,
    )


def _check_write(write: str) -> None:
    if write not in ("host", "device"):
        raise ValueError(f"write must be 'host' or 'device', not {write!r}")


def _run_and_write(pre: ChunkPreprocessor, chunks, output_file: str, write: str) -> None:
    """Scores the chunks and appends their rows: item dicts written by ``process_items``
    (``write="host"``), or blocks of rows formatted on the GPU (``write="device"``)."""
    if write == "host":
        items = []
        for params in chunks:
            items.extend(pre.run(**params))
        pre.process_items(items)
        return
    rows = DeviceRows(pre.stat_config)
    for params in chunks:
        pre.run_into(sink=rows, **params)
    rows.write(output_file, pre.engine)


def _write_headers(output_file: str, stat_config, ploidy_config) -> None:
    """The header lines of the score file and of the ``.U.log`` / ``.Q.log`` files (sai/sai.py:122-142)."""
    header = ["Chrom", "Start", "End", "Ref", "Tgt", "Src", "Outgroup", "N(Variants)"]
    src_pops = list(ploidy_config.root["src"].keys())
    for stat_name in stat_config.root.keys():  # sai/sai.py:122-129
        if stat_name not in ("U", "Q") and stat_config.root[stat_name] is False:
            continue
        if stat_name in ("U", "Q") or len(src_pops) <= 1:
            header.append(stat_name)
        else:
            header.extend(f"{stat_name}.{sp}" for sp in src_pops)
    directory = os.path.dirname(output_file)
    if directory:
        os.makedirs(directory, exist_ok=True)
    with open(output_file, "w") as f:
        f.write("\t".join(header) + "\n")
    for key in ("U", "Q"):
        if key in stat_config.root:
            with open(Path(output_file).with_suffix(f".{key}.log"), "w") as f:
                f.write(f"Chrom\tStart\tEnd\t{key}_SNP\n")


def score(
    vcf_file: str,
    chr_name: str,
    win_len: int,
    win_step: int,
    anc_allele_file: str,
    output_file: str,
    config: str,
    num_workers: int = 1,
    device: int = 0,
    ingest: str = "host",
    inflate: str = "host",
    dd_ingest: str = "host",
    write: str = "host",
) -> None:
    """``ingest="device"`` parses the VCF on the GPU (``ChunkPreprocessor(ingest=...)``),
    ``inflate="device"`` also inflates a bgzip file there, and ``dd_ingest="device"`` reads a DD
    configuration there too (the raw values of missing calls are kept in HBM); same output.
    ``write="device"`` formats the score file and the ``.U.log`` / ``.Q.log`` files on the GPU from the
    scoring results (``DeviceRows``: no per-window Python object, one copy back and one write per
    file); same bytes."""
    _check_write(write)
    cfg = _load_checked_config(config, anc_allele_file)
    # ONE chunk, as sai.py:86-93 (num_chunks=1; `num_workers` is accepted and ignored there too):
    # rows come out product-major / windows-inner, identical to the reference's text.  Real
    # parallelism is sai_b200.multiprocessing.mp_pool (one worker per GPU) or sai_b200.distributed.
    generator = ChunkGenerator(vcf_file=vcf_file, chr_name=chr_name, window_size=win_len, step_size=win_step,
                               num_chunks=1)
    pre = _preprocessor(vcf_file, cfg, win_len, win_step, anc_allele_file, output_file, device, ingest, inflate,
                        dd_ingest)
    _write_headers(output_file, cfg.statistics, cfg.ploidies)
    _run_and_write(pre, generator.get(), output_file, write)  # sai.py:148-149


def score_genome(
    vcf_file: str,
    chr_names: Sequence[str],
    win_len: int,
    win_step: int,
    anc_allele_file: str,
    output_file: str,
    config: str,
    device: int = 0,
    inflate: str = "host",
    dd_ingest: str = "host",
    write: str = "host",
) -> None:
    """Scores every chromosome of ``chr_names`` of one (multi-chromosome) VCF: the score file and the
    ``.U.log`` / ``.Q.log`` files are byte for byte those of ``score(vcf_file, c, ...)`` run for each
    ``c`` in turn and concatenated (header lines once), and so are the errors -- but the file is read
    once.  Its text is parsed on the GPU (``vcf_device.read_genome``; ``inflate="device"`` also
    inflates a bgzip file there) into one resident layout in which every chromosome starts on a tile
    boundary, and all chromosomes are scored with one genotype pass and one window launch.

    With ``dd_ingest="device"`` a DD configuration takes the one-pass read too: the genotype pass
    keeps the raw values of missing calls (the negative-value table) per chromosome in HBM, and DD is
    computed per chromosome from the resident tiles and table.

    Files the one-pass reader does not take -- where ``vcf_device.fallback_reason`` names a reason
    (DD with ``dd_ingest="host"``, more than 16 populations, long ancestral alleles, positional
    source ploidies), more than
    ``SAI_VCF_MAX_CHROMS`` (1024) chromosomes, or chromosomes whose records are not contiguous in
    the file -- are scored one chromosome at a time by the ``score`` path, with the same output.

    ``write="device"`` formats the rows on the GPU as ``score(..., write="device")`` does, on both
    paths."""
    from . import _cabi
    from .preprocessors import score_populations, write_items
    from .vcf import read_anc_or_error
    from .vcf_device import _wants_outgroup, fallback_reason, genome_tables, read_genome, read_plan, wants_dd
    from .windows import chunk_windows, split_genome, split_windows_ranges

    _check_write(write)
    cfg = _load_checked_config(config, anc_allele_file)
    stat_config, ploidy_config = cfg.statistics, cfg.ploidies
    chr_names = list(chr_names)
    pre = _preprocessor(vcf_file, cfg, win_len, win_step, anc_allele_file, output_file, device, "device", inflate,
                        dd_ingest)

    def each_chromosome() -> None:
        generators = [ChunkGenerator(vcf_file=vcf_file, chr_name=c, window_size=win_len, step_size=win_step, num_chunks=1)
                      for c in chr_names]
        _write_headers(output_file, stat_config, ploidy_config)
        for generator in generators:
            _run_and_write(pre, generator.get(), output_file, write)

    if not chr_names or len(set(chr_names)) != len(chr_names) or len(chr_names) > _cabi.MAX_CHROMS:
        return each_chromosome()
    with warnings.catch_warnings(record=True) as caught:  # warned once, by the read that is used
        warnings.simplefilter("always")
        plan, requests, out = read_plan(vcf_file, chr_names[0], ploidy_config, pre.ref_ind_file, pre.tgt_ind_file,
                                        pre.src_ind_file, pre.out_ind_file)
    if any(fallback_reason(stat_config, ploidy_config, plan, None, c, pre.num_src, dd_ingest) is not None
           for c in chr_names):
        return each_chromosome()
    tables = genome_tables(chr_names, anc_allele_file)
    if anc_allele_file and tables[2] is None:  # an ancestral allele longer than 7 bytes
        return each_chromosome()
    for w in caught:
        warnings.warn_explicit(w.message, w.category, w.filename, w.lineno)
    try:
        loaded = read_genome(pre.engine, vcf_file, chr_names, plan, requests, out, tables,
                             with_outgroup=_wants_outgroup(stat_config), inflate=inflate,
                             neg_table=dd_ingest == "device" and wants_dd(stat_config))
    except (KeyError, OSError) as e:
        raise ValueError(f"Failed to read VCF file {vcf_file} from {','.join(chr_names)}: {e}") from e
    if loaded is None:  # no #CHROM line, or a chromosome's records are not contiguous
        return each_chromosome()
    windows = []
    for c, name in enumerate(chr_names):
        span = loaded.span[c]
        if span is None:
            raise ValueError(f"Chromosome {name} not found in VCF.")
        chunks = split_windows_ranges(split_genome([span[0], span[1]], win_len, win_step), 1)
        if not chunks:  # no window (last POS before the first): score() runs no chunk
            return each_chromosome()
        start, end = chunks[0]
        pos = loaded.pos[c]
        if pos.size and (int(pos.min()) < start or int(pos.max()) > end):  # score() reads [start, end] only
            return each_chromosome()
        if anc_allele_file:
            anc_pos, _, anc_off = tables[2]
            mine = anc_pos[anc_off[c] : anc_off[c + 1]]
            if not np.any((mine >= start) & (mine <= end)):  # records but no ancestral allele: the reference raises
                raise read_anc_or_error(anc_allele_file, name, start, end)[1]
        windows.append(chunk_windows(start, end, win_len, win_step))
    (ref_pops, _), (tgt_pops, tgt_samples) = loaded.groups["ref"], loaded.groups["tgt"]
    (src_pops, _), (out_pops, _) = loaded.groups["src"], loaded.groups["outgroup"]
    if ref_pops is None or tgt_pops is None or src_pops is None:
        return each_chromosome()
    _write_headers(output_file, stat_config, ploidy_config)
    names = lambda pops: {p: None for p in pops} if pops else None
    rows = DeviceRows(stat_config) if write == "device" else None
    items = score_populations(
        chr_names[0], {t: windows for t in tgt_samples}, names(ref_pops), names(tgt_pops), names(src_pops),
        ploidy_config, stat_config, anc_allele_file is not None, pre.engine, out_data=names(out_pops),
        num_src=pre.num_src, loaded=loaded, sink=rows)
    if rows is not None:
        rows.write(output_file, pre.engine)
    else:
        write_items(output_file, items, stat_config)
