#!/usr/bin/env python
"""``score_genome`` with ``write="host"`` against ``write="device"`` on a synthetic 22-chromosome bgzip VCF
with about 288 000 windows (hg19 autosome lengths, 50 kb windows every 10 kb), sparse sites and few
samples so that ingest is not the subject, with 1 and 8 target populations.

Per leg: the seconds of ingest, scoring (genotype pass, window kernels, pattern / DD sums), item or
block building (``score_populations`` minus scoring), formatting (``write_items``' text, or
``DeviceRows.format``: the copy in, the format kernels and the copies back) and the file writes; the
format kernels alone from CUDA events.  The files of the two legs are compared byte for byte.  Prints
one JSON line per target count, with the card's name and power limit.

    python tools/write_bench.py [--reps 3]
"""

from __future__ import annotations

import argparse
import filecmp
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HG19_MB = [249, 243, 198, 191, 181, 171, 159, 146, 141, 136, 135, 134, 115, 107, 103, 90, 81, 78, 59, 63, 48, 51]
WIN_LEN, WIN_STEP = 50_000, 10_000


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": limit}
    except Exception as e:  # the numbers are still reported, without the card
        return {"gpu": f"unknown ({e})", "power_limit": "unknown"}


def write_case(d: str, n_tgt: int, seed: int = 1) -> tuple[str, str]:
    """bgzip VCF (one site every ~20 kb, 2 samples per population) and a U + Q configuration."""
    import yaml

    from sai_b200.vcf import write_bgzf

    rng = np.random.default_rng(seed)
    pops = {"ref": ["R"], "tgt": [f"T{i}" for i in range(n_tgt)], "src": ["S"]}
    samples = [(g, p, f"{p}_{i}") for g in pops for p in pops[g] for i in range(2)]
    gts = np.array(["0|0", "0|1", "1|0", "1|1", "0|0"])
    chunks = ["##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
              + "\t".join(s for _, _, s in samples) + "\n"]
    for c, mb in enumerate(HG19_MB):
        pos = np.cumsum(rng.integers(1, 40_000, size=mb * 1_000_000 // 20_000))
        g = rng.choice(gts, size=(pos.size, len(samples)))
        body = ["\t".join(row) for row in g.tolist()]
        chunks.append("".join(f"chr{c + 1}\t{p}\t.\tA\tG\t.\tPASS\t.\tGT\t{b}\n" for p, b in zip(pos.tolist(), body)))
    vcf = os.path.join(d, "g.vcf.gz")
    write_bgzf(vcf, "".join(chunks).encode())
    lists = {}
    for grp, names in pops.items():
        lists[grp] = os.path.join(d, f"{grp}.list")
        with open(lists[grp], "w") as f:
            f.writelines(f"{p}\t{s}\n" for g, p, s in samples if g == grp)
    stats = {s: {"ref": {"R": 0.3}, "tgt": {t: (0.2 if s == "U" else 0.9) for t in pops["tgt"]}, "src": {"S": "=1"}}
             for s in ("U", "Q")}
    cfg = os.path.join(d, "cfg.yaml")
    with open(cfg, "w") as f:
        yaml.safe_dump({"statistics": stats, "ploidies": {g: {p: 2 for p in ps} for g, ps in pops.items()},
                        "populations": lists}, f)
    return vcf, cfg


class Phases:
    """Seconds spent inside wrapped functions, by phase."""

    def __init__(self):
        self.t: dict[str, float] = {}
        self.undo = []

    def wrap(self, owner, name, phase):
        fn = getattr(owner, name)

        def timed(*a, **k):
            t0 = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                self.t[phase] = self.t.get(phase, 0.0) + time.perf_counter() - t0

        setattr(owner, name, timed)
        self.undo.append((owner, name, fn))

    def restore(self):
        for owner, name, fn in reversed(self.undo):
            setattr(owner, name, fn)


def leg(vcf, cfg, out, write, chroms, fmt_stats):
    from sai_b200 import preprocessors, vcf_device
    from sai_b200.score import score_genome
    from sai_b200.scoring import HostEngine

    ph = Phases()
    ph.wrap(vcf_device, "read_genome", "ingest")
    for m in ("score_loaded_pieces", "score_resident", "pattern_sums", "dd_sums"):
        ph.wrap(HostEngine, m, "scoring")
    ph.wrap(preprocessors, "score_populations", "populations")
    ph.wrap(preprocessors, "write_items", "format_and_write")
    ph.wrap(preprocessors.DeviceRows, "format", "format")
    ph.wrap(preprocessors.DeviceRows, "write", "format_and_write")
    fmt = {}
    orig_format = preprocessors.DeviceRows.format

    def format_and_time(self, engine, encoding):
        r = orig_format(self, engine, encoding)
        fmt.update(engine.format_stats())
        return r

    preprocessors.DeviceRows.format = format_and_time
    t0 = time.perf_counter()
    try:
        score_genome(vcf, chroms, WIN_LEN, WIN_STEP, None, out, cfg, inflate="device", write=write)
    finally:
        preprocessors.DeviceRows.format = orig_format
        ph.restore()
    total = time.perf_counter() - t0
    t = ph.t
    build = t.get("populations", 0.0) - t.get("scoring", 0.0)
    formatting = t.get("format", 0.0)
    writes = t.get("format_and_write", 0.0) - formatting
    if write == "host":  # write_items builds the text and writes it in one call
        formatting, writes = t.get("format_and_write", 0.0), 0.0
    fmt_stats.append(fmt)
    return {"total_s": total, "ingest_s": t.get("ingest", 0.0), "scoring_s": t.get("scoring", 0.0),
            "items_or_blocks_s": build, "format_s": formatting, "file_write_s": writes}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--targets", default="1,8")
    args = ap.parse_args()
    info = card()
    chroms = [f"chr{c + 1}" for c in range(len(HG19_MB))]
    with tempfile.TemporaryDirectory() as d:
        for n_tgt in [int(x) for x in args.targets.split(",")]:
            vcf, cfg = write_case(d, n_tgt)
            best: dict[str, dict] = {}
            fmt_stats: list = []
            for rep in range(args.reps + 1):  # the first repetition warms up
                for write in ("host", "device"):
                    out = os.path.join(d, f"{write}{n_tgt}", "s.tsv")
                    r = leg(vcf, cfg, out, write, chroms, fmt_stats if write == "device" else [])
                    if rep and (write not in best or r["total_s"] < best[write]["total_s"]):
                        best[write] = r
            same = all(filecmp.cmp(os.path.join(d, f"host{n_tgt}", f), os.path.join(d, f"device{n_tgt}", f), shallow=False)
                       for f in ("s.tsv", "s.U.log", "s.Q.log"))
            size = sum(os.path.getsize(os.path.join(d, f"device{n_tgt}", f)) for f in ("s.tsv", "s.U.log", "s.Q.log"))
            rows = sum(1 for _ in open(os.path.join(d, f"device{n_tgt}", "s.tsv"))) - 1
            kern = min(fmt_stats[1:] or fmt_stats, key=lambda s: s.get("length_s", 0) + s.get("write_s", 0))
            print(json.dumps({"bench": "write", "targets": n_tgt, "rows": rows, "text_MB": round(size / 1e6, 1),
                              "identical": same, **info,
                              "host": {k: round(v, 4) for k, v in best["host"].items()},
                              "device": {k: round(v, 4) for k, v in best["device"].items()},
                              "format_kernels_ms": {k: round(1e3 * v, 3) for k, v in kern.items()}}), flush=True)
            if not same:
                sys.exit(1)


if __name__ == "__main__":
    main()
