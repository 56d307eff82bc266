#!/usr/bin/env python
"""K1 alone (the genotype pass, `DeviceScorer.site_flags`) at bench.py's layout and size, timed with
CUDA events.  Uses only the public DeviceScorer API, so the same script times an older tree too.

    python tools/k1_gate_bench.py [--sites 6000000] [--reps 50] [--out FILE]

Two jobs on bench.py's data (rank 0's shard):
  bench     U + Q of bench.py (src "=1", w = 0.01, ancestral alleles): K1 time, the share of tiles
            whose reference and target a pass that reads the sources first must read, and the
            bytes such a pass reads over K1 time.  The shares come from `site_counts` on the same
            data with the gate predicates in numpy (reporting only, not a correctness check).
  all_live  src ">= 0", w = 1.0: every tile is live, so every byte is read as by a pass without
            gates; the worst case of the staged pass.
Prints the card's name, power limit and maximum SM clock, then one JSON line.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
from bench import WORKLOAD, make_job_for  # noqa: E402


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def time_k1(torch, sc, d_packed, job, reps: int, warmup: int = 5):
    for _ in range(warmup):
        sc.site_flags(d_packed, [job])
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        sc.site_flags(d_packed, [job])
        b.record()
    torch.cuda.synchronize()
    ms = np.array([a.elapsed_time(b) for a, b in ev])
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()), "reps": reps}


def gate_shares(num, called, lay, n_sites: int, wl):
    """Tiles whose reference / target the staged pass reads for bench.py's job (one source, "=" y,
    ancestral alleles): src_freq == y, then ref_freq < w, in float64 as the kernels decide."""
    freq = lambda p: np.divide(num[p, :n_sites], called[p, :n_sites] * lay.pop[p].ploidy,
                               out=np.full(n_sites, np.nan), where=called[p, :n_sites] > 0)
    assert wl["y"][0] == "=" and wl["anc"]
    src = freq(2) == wl["y"][1]
    ref = src & (freq(0) < wl["w"])
    n_tiles = (n_sites + 31) // 32
    tiles = lambda m: np.pad(m, (0, n_tiles * 32 - n_sites)).reshape(n_tiles, 32).any(1)
    return float(tiles(src).mean()), float(tiles(ref).mean()), float(src.mean()), float(ref.mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=WORKLOAD["n_sites"])
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    from sai_b200 import _cabi
    from sai_b200.encode import make_layout
    from sai_b200.scoring import DeviceScorer, make_job, synth_fill

    if not torch.cuda.is_available():
        raise SystemExit("k1_gate_bench.py needs a CUDA device")
    print(card(), flush=True)
    wl = dict(WORKLOAD, n_sites=args.sites)
    S = wl["n_sites"]
    lay = make_layout(list(wl["n_ind"]), list(wl["ploidy"]), [2, 2, 2])
    d_packed = torch.empty(int(_cabi.load().sai_packed_bytes(C.byref(lay), S)), dtype=torch.uint8, device="cuda")
    synth_fill(lay, d_packed, S, [0, 1, 2], wl["seed"], 0.0)  # bench.py's rank-0 shard
    sc = DeviceScorer(lay, S, 1, 1)
    pair_bytes = [256 * lay.pop[p].n_pairs for p in range(3)]  # per tile: ref, tgt, src
    n_tiles = sc.n_tiles
    full_bytes = n_tiles * sum(pair_bytes)

    num, called = (t.cpu().numpy() for t in sc.site_counts(d_packed))
    tile_ref, tile_tgt, site_src, site_ref = gate_shares(num, called, lay, S, wl)
    gated_bytes = n_tiles * (pair_bytes[2] + tile_ref * pair_bytes[0] + tile_tgt * pair_bytes[1])

    bench = time_k1(torch, sc, d_packed, make_job_for(wl), args.reps)
    all_live_job = make_job(0, 1, [2], wl["anc"], u=dict(w=1.0, x=wl["x"], y_list=[(">=", 0.0)]),
                            q=dict(w=1.0, quantile=wl["quantile"], y_list=[(">=", 0.0)]))
    all_live = time_k1(torch, sc, d_packed, all_live_job, args.reps)

    bench.update(tiles_reading_ref=tile_ref, tiles_reading_tgt=tile_tgt, sites_src_pass=site_src,
                 sites_src_ref_pass=site_ref, bytes_read=int(gated_bytes),
                 tb_s_bytes_read=gated_bytes / (bench["median_ms"] / 1e3) / 1e12,
                 tb_s_all_bytes=full_bytes / (bench["median_ms"] / 1e3) / 1e12)
    all_live.update(bytes_read=int(full_bytes), tb_s_bytes_read=full_bytes / (all_live["median_ms"] / 1e3) / 1e12)
    line = json.dumps({"sites": S, "tiles": n_tiles, "card": card().splitlines()[-1], "bench": bench,
                       "all_live": all_live})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
