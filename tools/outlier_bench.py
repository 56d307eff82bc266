#!/usr/bin/env python
"""``outlier`` with ``text="host"`` against ``text="device"`` on a seeded synthetic score file the size of
a whole-genome scan of 8 target populations: 2 302 496 rows (22 chromosomes, 50 kb windows every
10 kb), with Ref / Tgt / Src text, an all-NA Outgroup, an integer U column with NaN rows, and Q and
four float columns (NaN rows, negative values, 17-digit reprs).

Both legs run at q = 0.99 and 0.9, best of ``--reps`` after one warm-up run.  The device leg's phases:
file read, copy in, tokenise + classify, parse, thresholds, sort, format, copy back, file writes (the
copies and kernels from CUDA events).  The files of the two legs are compared byte for byte.  Prints
one JSON line per quantile, with the card's name and power limit.

    python tools/outlier_bench.py [--reps 3]
"""

from __future__ import annotations

import argparse
import filecmp
import json
import os
import sys
import tempfile
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from write_bench import HG19_MB, WIN_LEN, WIN_STEP, card  # noqa: E402

FLOATS = ["Q", "Dplus", "Danc", "df", "fd"]


def write_scores(path: str, n_tgt: int = 8, seed: int = 1) -> int:
    rng = np.random.default_rng(seed)
    parts = ["\t".join(["Chrom", "Start", "End", "Ref", "Tgt", "Src", "Outgroup", "N(Variants)", "U"] + FLOATS) + "\n"]
    rows = 0
    for c, mb in enumerate(HG19_MB):
        starts = np.arange(0, mb * 1_000_000 - WIN_LEN + 1, WIN_STEP)
        n = starts.size
        for t in range(n_tgt):
            nsnps = rng.integers(0, 40, size=n)
            empty = nsnps == 0
            u = rng.poisson(3.0, size=n).astype(str).astype(object)
            u[empty] = "nan"
            cols = [np.full(n, f"chr{c + 1}", dtype=object), starts.astype(str), (starts + WIN_LEN).astype(str),
                    np.full(n, "AFR", dtype=object), np.full(n, f"T{t}", dtype=object), np.full(n, "NEA", dtype=object),
                    np.full(n, "NA", dtype=object), nsnps.astype(str), u]
            for k, _ in enumerate(FLOATS):
                v = rng.random(n) * (1.0 if k < 2 else 2.0) - (0.0 if k < 2 else 1.0)
                s = np.array([repr(x) for x in v.tolist()], dtype=object)
                s[empty | (rng.random(n) < 0.02)] = "nan"
                cols.append(s)
            parts.append("\n".join("\t".join(r) for r in zip(*cols)) + "\n")
            rows += n
    with open(path, "w") as f:
        f.writelines(parts)
    return rows


def host_leg(path, prefix, q) -> dict:
    from sai_b200.outlier import outlier

    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        outlier(path, prefix, q, text="host")
    return {"total_s": time.perf_counter() - t0}


def device_leg(path, prefix, q) -> dict:
    from sai_b200.outlier import device_outlier

    timings: dict = {}
    t0 = time.perf_counter()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        assert device_outlier(path, prefix, q, timings=timings), "the device path refused the file"
    timings["total_s"] = time.perf_counter() - t0
    return timings


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    info = card()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "scores.tsv")
        rows = write_scores(path)
        for q in (0.99, 0.9):
            best: dict[str, dict] = {}
            for rep in range(args.reps + 1):  # the first repetition warms up
                for text, leg in (("host", host_leg), ("device", device_leg)):
                    r = leg(path, os.path.join(d, f"{text}"), q)
                    if rep and (text not in best or r["total_s"] < best[text]["total_s"]):
                        best[text] = r
            cols = open(path).readline().rstrip("\n").split("\t")
            cols = cols[cols.index("N(Variants)") + 1:]
            names = [f"{c}.{q}.outliers.tsv" for c in cols]
            same = all(filecmp.cmp(os.path.join(d, f"host.{f}"), os.path.join(d, f"device.{f}"), shallow=False) for f in names)
            out_mb = sum(os.path.getsize(os.path.join(d, f"device.{f}")) for f in names) / 1e6
            print(json.dumps({"bench": "outlier", "q": q, "rows": rows, "file_MB": round(os.path.getsize(path) / 1e6, 1),
                              "tables_MB": round(out_mb, 1), "identical": same, **info,
                              "host": {k: round(v, 4) for k, v in best["host"].items()},
                              "device": {k: round(v, 4) for k, v in best["device"].items()},
                              "speedup": round(best["host"]["total_s"] / best["device"]["total_s"], 1)}), flush=True)
            if not same:
                sys.exit(1)


if __name__ == "__main__":
    main()
