"""Top-level ``score`` with the signature and file outputs of the reference's
``sai.sai.score`` (sai/sai.py:33-151), running the U/Q path on the GPU.

Every statistic of the reference's registry is computed on the GPU: U, Q, the
four site-pattern statistics (Danc, Dplus, df, fd) and DD.  In a reference-side integration ``score`` itself stays
untouched and only the ``ChunkPreprocessor`` it constructs is swapped
(INTEGRATION.md).
"""

from __future__ import annotations

import os
from pathlib import Path

from .configs import load_config
from .preprocessors import ChunkPreprocessor
from .generators import ChunkGenerator


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
) -> None:
    """``ingest="device"`` parses the VCF on the GPU (``ChunkPreprocessor(ingest=...)``), and
    ``inflate="device"`` also inflates a bgzip file there; same output."""
    cfg = load_config(config)
    stat_config, ploidy_config, pop_config = cfg.statistics, cfg.ploidies, cfg.populations
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
    # ONE chunk, as sai.py:86-93 (num_chunks=1; `num_workers` is accepted and ignored there too):
    # rows come out product-major / windows-inner, identical to the reference's text.  Real
    # parallelism is sai_b200.multiprocessing.mp_pool (one worker per GPU) or sai_b200.distributed.
    generator = ChunkGenerator(vcf_file=vcf_file, chr_name=chr_name, window_size=win_len, step_size=win_step,
                               num_chunks=1)
    pre = ChunkPreprocessor(
        vcf_file=vcf_file,
        ref_ind_file=pop_config.get_population("ref"),
        tgt_ind_file=pop_config.get_population("tgt"),
        src_ind_file=pop_config.get_population("src"),
        out_ind_file=pop_config.get_population("outgroup"),
        win_len=win_len,
        win_step=win_step,
        output_file=output_file,
        ploidy_config=ploidy_config,
        stat_config=stat_config,
        anc_allele_file=anc_allele_file,
        device=device,
        ingest=ingest,
        inflate=inflate,
    )
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
    items = []
    for params in generator.get():  # sai.py:148-149
        items.extend(pre.run(**params))
    pre.process_items(items)
