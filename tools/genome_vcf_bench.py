#!/usr/bin/env python
"""One pass over a whole-genome bgzip VCF against one pass per chromosome (needs a GPU).

    python tools/genome_vcf_bench.py [--chroms 22] [--sites 10000] [--samples 64] [--inflate device]

Writes (untimed) a synthetic bgzip VCF of ``--chroms`` chromosomes with ``--sites`` diploid, phased
GT-only records each and an ancestral table that lists every site, then times
  * ``score_genome`` over all chromosomes (one device pass: the text is read, inflated and parsed once);
  * the loop of ``score(..., ingest="device")`` per chromosome, what a genome costs without it (a
    multi-chromosome file is scanned whole for every chromosome);
and checks that the two produce the same files byte for byte.  It also reports the text bytes each
leg's device sessions parsed (``HostEngine.vcf_stats``), read with the same ingest calls the legs
make.  U and Q, one ref / tgt / src population.  Prints one JSON line, the card's name and power
limit included.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def write_genome(d, n_chroms, n_sites, n_samples, seed=1):
    from sai_b200.vcf import write_bgzf

    rng = np.random.default_rng(seed)
    tokens = np.frombuffer(b"0|0\t0|1\t1|0\t1|1\t", dtype=np.uint8).reshape(4, 4)
    samples = [f"s{i}" for i in range(n_samples)]
    parts = ["##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(samples) + "\n"]
    bed, names = [], [f"chr{c + 1}" for c in range(n_chroms)]
    parts = [parts[0].encode()]
    for name in names:
        pos = np.cumsum(rng.integers(50, 400, size=n_sites)) + 1000
        codes = rng.choice(4, size=(n_sites, n_samples), p=[0.7, 0.1, 0.1, 0.1])
        geno = tokens[codes].reshape(n_sites, 4 * n_samples)
        geno[:, -1] = ord("\n")
        rows = geno.tobytes()
        w = 4 * n_samples
        parts.append(b"".join(f"{name}\t{p}\t.\tA\tG\t.\tPASS\t.\tGT\t".encode() + rows[i * w : (i + 1) * w]
                              for i, p in enumerate(pos.tolist())))
        bed.append("".join(f"{name}\t{p - 1}\t{p}\tA\n" for p in pos.tolist()))
    text = b"".join(parts)
    write_bgzf(os.path.join(d, "g.vcf.gz"), text)
    with open(os.path.join(d, "anc.bed"), "w") as f:
        f.write("".join(bed))
    lists = {}
    third = n_samples // 3
    for g, sl in (("ref", slice(0, third)), ("tgt", slice(third, 2 * third)), ("src", slice(2 * third, n_samples))):
        lists[g] = os.path.join(d, f"{g}.list")
        with open(lists[g], "w") as f:
            f.writelines(f"{g.upper()}\t{s}\n" for s in samples[sl])
    return names, lists, len(text)


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def texts(out):
    return [open(p, "rb").read() for p in (out, out[:-4] + ".U.log", out[:-4] + ".Q.log")]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chroms", type=int, default=22)
    ap.add_argument("--sites", type=int, default=10000, help="records per chromosome")
    ap.add_argument("--samples", type=int, default=64)
    ap.add_argument("--win-len", type=int, default=50000)
    ap.add_argument("--win-step", type=int, default=10000)
    ap.add_argument("--inflate", choices=("host", "device"), default="device")
    ap.add_argument("--out", default=None, help="directory for the JSON line (default: print only)")
    a = ap.parse_args()

    import torch
    import yaml

    if not torch.cuda.is_available():
        raise SystemExit("genome_vcf_bench.py needs a CUDA device")
    from sai_b200.configs import PloidyConfig
    from sai_b200.score import score, score_genome
    from sai_b200.scoring import HostEngine
    from sai_b200.vcf import read_anc_or_error
    from sai_b200.vcf_device import genome_tables, read_genome, read_loaded, read_plan
    from sai_b200.windows import split_genome, split_windows_ranges

    with tempfile.TemporaryDirectory() as d:
        names, lists, text_bytes = write_genome(d, a.chroms, a.sites, a.samples)
        vcf, anc = os.path.join(d, "g.vcf.gz"), os.path.join(d, "anc.bed")
        ploidies = {"ref": {"REF": 2}, "tgt": {"TGT": 2}, "src": {"SRC": 2}}
        stats = {"U": {"ref": {"REF": 0.3}, "tgt": {"TGT": 0.5}, "src": {"SRC": "=1"}},
                 "Q": {"ref": {"REF": 0.3}, "tgt": {"TGT": 0.95}, "src": {"SRC": "=1"}}}
        cfg = os.path.join(d, "cfg.yaml")
        with open(cfg, "w") as f:
            yaml.safe_dump({"statistics": stats, "ploidies": ploidies, "populations": lists}, f)

        # warm-up: CUDA context, library, allocations
        score(vcf, names[0], a.win_len, a.win_step, anc, os.path.join(d, "warm", "s.tsv"), cfg, ingest="device",
              inflate=a.inflate)

        t0 = time.perf_counter()
        score_genome(vcf, names, a.win_len, a.win_step, anc, os.path.join(d, "genome", "s.tsv"), cfg, inflate=a.inflate)
        t_genome = time.perf_counter() - t0

        t0 = time.perf_counter()
        parts = []
        for i, c in enumerate(names):
            out = os.path.join(d, f"loop{i}", "s.tsv")
            score(vcf, c, a.win_len, a.win_step, anc, out, cfg, ingest="device", inflate=a.inflate)
            parts.append(texts(out))
        t_loop = time.perf_counter() - t0
        want = [parts[0][k] + b"".join(p[k].split(b"\n", 1)[1] for p in parts[1:]) for k in range(3)]
        same = texts(os.path.join(d, "genome", "s.tsv")) == want

        # the text bytes each leg's device sessions parse (the ingest calls the legs make)
        e = HostEngine(0)
        pc = PloidyConfig(ploidies)
        plan, requests, out = read_plan(vcf, names[0], pc, lists["ref"], lists["tgt"], lists["src"], None)
        read_genome(e, vcf, names, plan, requests, out, genome_tables(names, anc), with_outgroup=False, inflate=a.inflate)
        genome_text = e.vcf_stats()["text_bytes"]
        loop_text = 0
        for c in names:
            g = read_genome(e, vcf, [c], plan, requests, out, genome_tables([c], anc), with_outgroup=False,
                            inflate=a.inflate)
            start, end = split_windows_ranges(split_genome(g.span[0][:2], a.win_len, a.win_step), 1)[0]
            tab, err = read_anc_or_error(anc, c, start, end)
            read_loaded(e, vcf, c, plan, requests, out, tab, err, start, end, with_outgroup=False, inflate=a.inflate)
            loop_text += e.vcf_stats()["text_bytes"]
        e.close()

    res = {"chroms": a.chroms, "sites_per_chrom": a.sites, "samples": a.samples, "inflate": a.inflate,
           "text_bytes": text_bytes, "score_genome_s": round(t_genome, 4), "score_loop_s": round(t_loop, 4),
           "speedup": round(t_loop / t_genome, 3), "genome_parsed_text_bytes": int(genome_text),
           "loop_parsed_text_bytes": int(loop_text), "identical_outputs": bool(same), "gpu": gpu_info()}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "genome_vcf_bench.json"), "w") as f:
            f.write(line + "\n")
    if not same:
        raise SystemExit("score_genome and the per-chromosome loop differ")


if __name__ == "__main__":
    main()
