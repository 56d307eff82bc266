#!/usr/bin/env python
"""K4 alone (the window pass, `DeviceScorer.window_stats` after one `site_flags`) timed with CUDA
events.  Uses only the public DeviceScorer API, so the same script times an older tree too.

    python tools/k4_bench.py [--reps 50] [--legs bench,strong,dense,unsorted] [--genome-sites 80000000]
                             [--compare-lib SO] [--out FILE]

Legs (K1 runs once per leg; the window pass is then timed on its masks):
  bench     bench.py's job, data (rank 0's shard, 6 M sites) and windows (50 kb every 10 kb).
  strong    the whole genome of bench.py's `strong` record on one GPU: 22 pieces, one
            `sai_window_stats_pieces` launch over all their windows.
  dense     the all-live job of tools/k1_gate_bench.py (src ">= 0", w = 1.0) on the bench data:
            every site is flagged, so every window holds far more than 32 Q-flagged sites.
  unsorted  the bench job with its window list in a fixed random order: no run of consecutive
            windows is sorted, so every window takes the per-window path.
The bench and strong legs also time K1 (`site_flags`), so K4's share of the step is reported.
`--compare-lib` binds a second scorer over the same masks to another build of the library (an older
tree) and alternates the two rep by rep; every output array must be equal: N(Variants), U, Q (bit
patterns), q_cnt, the totals and the candidate positions of every window in window order (the
offsets into the candidate buffers are layout, not results).
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
from bench import HG19_MB, WORKLOAD, make_job_for, make_positions, make_windows  # noqa: E402


def card() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f"nvidia-smi unavailable: {e}"


def load_lib(path: str):
    from sai_b200 import _cabi

    lib = C.CDLL(path)
    for name, (res, args) in _cabi.SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def stats(ms):
    ms = np.asarray(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()), "reps": len(ms)}


def outputs(res) -> dict:
    """What a caller receives, job by job: per-window arrays and the candidates in window order."""
    def concat(cand, start, cnt):
        cnt = cnt.astype(np.int64)
        first = np.cumsum(cnt) - cnt
        return cand[np.arange(int(cnt.sum())) + np.repeat(start - first, cnt)]

    out = {}
    for j in range(res.nsnps.shape[0]):
        out.update({f"nsnps{j}": res.nsnps[j], f"u{j}": res.u[j], f"q{j}": res.q[j].view(np.int64),
                    f"q_cnt{j}": res.q_cnt[j], f"totals{j}": res.totals[j],
                    f"u_pos{j}": concat(res.u_cand[j], res.u_start[j], res.u[j]),
                    f"q_pos{j}": concat(res.q_cand[j], res.q_start[j], res.q_cnt[j])})
    return out


def run_leg(torch, sc, call, other_lib, reps: int, k1=None):
    """Times `call(scorer)` (one window pass) with events; with `other_lib`, alternates a sibling
    scorer on the same masks bound to it and checks every output equal."""
    scorers = {"change": sc}
    if other_lib is not None:
        scorers["compare"] = sc.sibling(sc.W, cap_u=sc.cap_u, cap_q=sc.cap_q)
        scorers["compare"].lib = other_lib
    res = {}
    for name, s in scorers.items():  # warm-up; results() also regrows the candidate buffers if needed
        for _ in range(3):
            call(s)
        res[name] = outputs(s.results())
    if other_lib is not None:
        a, b = res["change"], res["compare"]
        assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a), \
            [k for k in a if not np.array_equal(a[k], b[k])]
    times = {name: [] for name in scorers}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(reps):  # alternated rep by rep
        for name, s in scorers.items():
            ev[0].record()
            call(s)
            ev[1].record()
            torch.cuda.synchronize()
            times[name].append(ev[0].elapsed_time(ev[1]))
    r0 = res["change"]
    out = {name: stats(t) for name, t in times.items()}
    out.update(windows=int(sc.W), u_total=int(sum(r0[k].sum() for k in r0 if k.startswith("u") and k[1:].isdigit())),
               outputs_equal=None if other_lib is None else True)
    if k1 is not None:
        kt = []
        for _ in range(reps):
            ev[0].record()
            k1()
            ev[1].record()
            torch.cuda.synchronize()
            kt.append(ev[0].elapsed_time(ev[1]))
        out["k1"] = stats(kt)
        out["k4_share_of_step"] = out["change"]["median_ms"] / (out["change"]["median_ms"] + out["k1"]["median_ms"])
    return out


def strong_batch(torch, lay, wl, total: int):
    """bench.py's `strong` genome on one GPU (shard_genome(..., 1)): 22 pieces in one batch."""
    from sai_b200.genome import GenomeBatch, piece_site_range, shard_genome, synth_fill_piece
    from sai_b200.windows import split_genome

    chrom_sites = [max(64, int(total * mb / sum(HG19_MB)) // 32 * 32) for mb in HG19_MB]
    chrom_pos = [make_positions(n, mb * 1e6 / n, 100 + c) for c, (n, mb) in enumerate(zip(chrom_sites, HG19_MB))]
    chrom_wins = [split_genome([int(p[0]), int(p[-1])], wl["win_len"], wl["win_step"]) for p in chrom_pos]
    pieces = shard_genome(chrom_wins, 1)[0]
    ranges = [piece_site_range(chrom_pos[p.chrom], chrom_wins[p.chrom], p) for p in pieces]
    wins = [chrom_wins[p.chrom][p.win_lo : p.win_hi] for p in pieces]
    n_w = sum(len(w) for w in wins)
    batch = GenomeBatch(lay, [hi - lo for lo, hi in ranges], wins, 1, cap_u=max(8 * n_w, 1 << 16), cap_q=max(32 * n_w, 1 << 18))
    for k, (p, (lo, hi)) in enumerate(zip(pieces, ranges)):
        synth_fill_piece(batch, k, lo, chrom_sites[p.chrom], [0, 1, 2], 777 + p.chrom, 0.0)
        batch.pos_view(k).copy_(torch.from_numpy(chrom_pos[p.chrom][lo:hi]))
    torch.cuda.synchronize()
    return batch


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--legs", default="bench,strong,dense,unsorted")
    ap.add_argument("--genome-sites", type=int, default=80_000_000, help="sites of the strong leg's genome")
    ap.add_argument("--compare-lib", default=None, help="another build of libsai_b200.so, alternated on every leg")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    from sai_b200 import _cabi
    from sai_b200.encode import make_layout
    from sai_b200.scoring import DeviceScorer, make_job, synth_fill

    if not torch.cuda.is_available():
        raise SystemExit("k4_bench.py needs a CUDA device")
    print(card(), flush=True)
    legs = args.legs.split(",")
    other = load_lib(args.compare_lib) if args.compare_lib else None
    wl = dict(WORKLOAD)
    lay = make_layout(list(wl["n_ind"]), list(wl["ploidy"]), [2, 2, 2])
    job = make_job_for(wl)
    out = {}

    if {"bench", "dense", "unsorted"} & set(legs):
        S = wl["n_sites"]
        d_packed = torch.empty(int(_cabi.load().sai_packed_bytes(C.byref(lay), S)), dtype=torch.uint8, device="cuda")
        synth_fill(lay, d_packed, S, [0, 1, 2], wl["seed"], 0.0)  # bench.py's rank-0 shard
        pos = make_positions(S, wl["mean_gap"], wl["seed"])
        ws, we = make_windows(pos, wl["win_len"], wl["win_step"])
        W = int(ws.shape[0])
        d_pos, d_ws, d_we = (torch.from_numpy(a).cuda() for a in (pos, ws, we))
        perm = np.random.default_rng(4).permutation(W)
        d_ws_u, d_we_u = torch.from_numpy(ws[perm]).cuda(), torch.from_numpy(we[perm]).cuda()
        all_live = make_job(0, 1, [2], wl["anc"], u=dict(w=1.0, x=wl["x"], y_list=[(">=", 0.0)]),
                            q=dict(w=1.0, quantile=wl["quantile"], y_list=[(">=", 0.0)]))
        for leg, jb, a, b in (("bench", job, d_ws, d_we), ("dense", all_live, d_ws, d_we),
                              ("unsorted", job, d_ws_u, d_we_u)):
            if leg not in legs:
                continue
            sc = DeviceScorer(lay, S, W, 1, cap_u=max(4 * W, 1 << 16), cap_q=max(16 * W, 1 << 18))
            sc.site_flags(d_packed, [jb])
            k1 = (lambda: sc.site_flags(d_packed, [jb])) if leg == "bench" else None
            out[leg] = run_leg(torch, sc, lambda s: s.window_stats(d_pos, a, b, [jb]), other, args.reps, k1)
            print(leg, json.dumps(out[leg]), flush=True)
            del sc
        del d_packed
        torch.cuda.empty_cache()

    if "strong" in legs:
        batch = strong_batch(torch, lay, wl, args.genome_sites)
        batch.score([job])
        calls = lambda s: s.window_stats(batch.d_pos, batch.d_ws, batch.d_we, [job], batch.d_first, batch.d_last)
        k1 = lambda: batch.score([job])  # K1 + K4: the step; K1 alone = step - K4
        out["strong"] = run_leg(torch, batch.scorer, calls, other, args.reps, None)
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        st = []
        for _ in range(args.reps):
            ev[0].record()
            k1()
            ev[1].record()
            torch.cuda.synchronize()
            st.append(ev[0].elapsed_time(ev[1]))
        out["strong"]["step"] = stats(st)
        out["strong"]["k4_share_of_step"] = out["strong"]["change"]["median_ms"] / out["strong"]["step"]["median_ms"]
        print("strong", json.dumps(out["strong"]), flush=True)
        del batch
        torch.cuda.empty_cache()

    line = json.dumps({"card": card().splitlines()[-1], "legs": out})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
