#!/usr/bin/env python
"""K1 alone (the genotype pass, `DeviceScorer.site_flags`) at bench.py's layout and size, timed with
CUDA events.  Uses only the public DeviceScorer API, so the same script times an older tree too.

    python tools/k1_gate_bench.py [--sites 6000000] [--reps 50] [--out FILE] [--profile]

Three jobs on bench.py's data (rank 0's shard):
  bench     U + Q of bench.py (src "=1", w = 0.01, ancestral alleles): K1 time, the share of tiles
            on which the staged pass reads the reference and the target, and its bytes over K1 time.
  sparse    src ">= y", w = 0.05, with y the smallest of 1, 7/8, ..., 1/8 for which at most half of
            the tiles hold a source-live site: many tiles with a few live sites each, the middle of
            the range between the bench job and the all-live job.
  all_live  src ">= 0", w = 1.0: every tile is live, so every byte is read as by a pass without
            gates; the worst case of the staged pass.
The shares and bytes come from `site_counts` on the same data with the gate predicates in numpy
(reporting only, not a correctness check).  Bytes are modelled for the pass as it reads: the source
pairs of every tile, then per tile the reference at the sites where the source gate holds and the
target where the reference gate holds too -- gathered (the distinct 32-byte sectors, 4 sites of
one pair, or 64-byte blocks of 8 sites) at up to GATHER_SITES such sites, the whole tile above.
`bytes_tile_granular` is the same pass reading every live tile whole.  `live_tiles` is the number of
tiles where the source gate holds at some site: the tiles on which the pass reads more than the sources.
--profile times nothing with events; it runs each job under torch.profiler (CUDA activities) and
reports the mean device time per launch of each kernel and memset of the pass (`split`).
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

GATHER_SITES = 8  # kGatherSites, sai_b200/csrc/site_kernels.cu


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


def split_k1(torch, sc, d_packed, job, reps: int):
    """Mean device time per K1 call of each kernel / memset it launches, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    for _ in range(5):
        sc.site_flags(d_packed, [job])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            sc.site_flags(d_packed, [job])
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and e.count > 0:
            us = getattr(e, "device_time_total", None)
            if us is None:
                us = e.cuda_time_total
            out[e.key[:60]] = {"us_per_call": us / reps, "launches_per_call": e.count / reps}
    return out


def freqs(num, called, lay, n_sites: int):
    return [np.divide(num[p, :n_sites], called[p, :n_sites] * lay.pop[p].ploidy, out=np.full(n_sites, np.nan),
                      where=called[p, :n_sites] > 0) for p in range(3)]


def gates(f, op: str, y: float, w: float):
    """Per site: the source gate, and the source + reference gates, of a one-source job with
    ancestral alleles (src 2, ref 0), in float64 as the kernels decide."""
    src = {"=": f[2] == y, ">=": f[2] >= y}[op]
    return src, src & (f[0] < w)


def pass_model(src, ref, lay, n_sites: int):
    """Tile shares and modelled bytes of the staged pass for the per-site gate masks src, ref."""
    n_tiles = (n_sites + 31) // 32
    tiles = lambda m: np.pad(m, (0, n_tiles * 32 - n_sites)).reshape(n_tiles, 32)
    pair_bytes = [256 * lay.pop[p].n_pairs for p in range(3)]  # per tile: ref, tgt, src
    out = {"live_tiles": int(tiles(src).any(1).sum()),
           "tiles_reading_ref": float(tiles(src).any(1).mean()), "tiles_reading_tgt": float(tiles(ref).any(1).mean()),
           "sites_src_pass": float(src.mean()), "sites_src_ref_pass": float(ref.mean())}
    tile_gran = n_tiles * pair_bytes[2]
    model = {32: tile_gran, 64: tile_gran}
    for pop, m in ((0, tiles(src)), (1, tiles(ref))):
        live = m.sum(1)
        tile_gran += int((live > 0).sum()) * pair_bytes[pop]
        whole = int((live > GATHER_SITES).sum()) * pair_bytes[pop]
        g = m[(live > 0) & (live <= GATHER_SITES)]
        for sector in (32, 64):
            blocks = int(g.reshape(g.shape[0], 32 * 8 // sector, sector // 8).any(2).sum())
            model[sector] += whole + blocks * lay.pop[pop].n_pairs * sector
    out.update(bytes_read=int(model[32]), bytes_read_64B=int(model[64]), bytes_tile_granular=int(tile_gran))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=WORKLOAD["n_sites"])
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    ap.add_argument("--profile", action="store_true", help="per-kernel split from torch.profiler instead of events")
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
    f = freqs(num, called, lay, S)
    n_tiles = sc.n_tiles
    full_bytes = n_tiles * sum(256 * lay.pop[p].n_pairs for p in range(3))
    assert wl["y"][0] == "=" and wl["anc"]
    bench_model = pass_model(*gates(f, "=", wl["y"][1], wl["w"]), lay, S)
    sparse_y = next(y / 8 for y in range(8, 0, -1)
                    if pass_model(*gates(f, ">=", (y - 1) / 8, 0.05), lay, S)["tiles_reading_ref"] > 0.5 or y == 1)
    sparse_model = pass_model(*gates(f, ">=", sparse_y, 0.05), lay, S)

    timer = (lambda *a: {"split": split_k1(*a)}) if args.profile else time_k1
    bench = timer(torch, sc, d_packed, make_job_for(wl), args.reps)
    sparse_job = make_job(0, 1, [2], wl["anc"], u=dict(w=0.05, x=wl["x"], y_list=[(">=", sparse_y)]),
                          q=dict(w=0.05, quantile=wl["quantile"], y_list=[(">=", sparse_y)]))
    sparse = timer(torch, sc, d_packed, sparse_job, args.reps)
    all_live_job = make_job(0, 1, [2], wl["anc"], u=dict(w=1.0, x=wl["x"], y_list=[(">=", 0.0)]),
                            q=dict(w=1.0, quantile=wl["quantile"], y_list=[(">=", 0.0)]))
    all_live = timer(torch, sc, d_packed, all_live_job, args.reps)

    for r, model in ((bench, bench_model), (sparse, sparse_model)):
        r.update(model)
        if not args.profile:
            r.update(tb_s_bytes_read=model["bytes_read"] / (r["median_ms"] / 1e3) / 1e12,
                     tb_s_all_bytes=full_bytes / (r["median_ms"] / 1e3) / 1e12)
    sparse["src_y"] = sparse_y
    all_live.update(bytes_read=int(full_bytes), live_tiles=int(n_tiles))
    if not args.profile:
        all_live.update(tb_s_bytes_read=full_bytes / (all_live["median_ms"] / 1e3) / 1e12)
    line = json.dumps({"sites": S, "tiles": n_tiles, "card": card().splitlines()[-1], "bench": bench,
                       "sparse": sparse, "all_live": all_live})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
