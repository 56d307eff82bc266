#!/usr/bin/env python
"""DD kernels (N4) timed with CUDA events at the layout of `tests/run_configs.py --config 6`:
1 M sites, ref 1500, tgt 1000, one source of 4 (plus a 2-individual outgroup the DD job does not
read), all diploid, 0.2 % missing calls with raw values -1 / -2, 50 kb windows every 10 kb.  The
packed matrix (0.64 GB at 2 planes) is larger than the 126 MB L2.

    python tools/dd_bench.py [--sites 1000000] [--reps 20] [--legs a,b,c] [--compare-lib SO] [--out FILE]

Legs (the same calls, with values changed and the layout widened):
  a  2 planes everywhere: the common layout.
  b  0.1 % of the ref / tgt calls become values 15..30, so ref and tgt take 5 planes.
  c  every call of ref, tgt and the source is a value 15..127: 8 planes, the worst case.
Per leg: `site_hist` (k_site_hist over ref, tgt and the source, as `HostEngine.dd_sums` runs it)
and `dd_sums` (k_site_dd + k_entry_dd + k_window_dd) through `DeviceScorer`, each bracketed by
CUDA events, median over `--reps`; and `HostEngine.dd_sums` from call to return (table upload,
kernels, result download).  `--compare-lib` binds a second DeviceScorer to another build of the
library (an older tree) and alternates the two rep by rep on leg a; its sums must equal ours.
Every leg checks DeviceScorer against HostEngine and a few windows against the oracle.
Prints the card's name, power limit and maximum SM clock, then one JSON line.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.dont_write_bytecode = True

N_IND, PLOIDY, ROLES, SEED, MISSING = [1500, 1000, 4, 2], [2, 2, 2, 2], [0, 1, 2, 0], 20261018 + 6, 0.002
LEG_BITS = {"a": [2, 2, 2, 2], "b": [5, 5, 2, 2], "c": [8, 8, 8, 2]}


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


def base_matrices(S: int, rng):
    """Device-generated diploid calls (bench's site model), decoded to int8 on the host; the
    missing calls get raw values -1 ("0/.") or -2 ("./.")."""
    import torch

    from sai_b200 import _cabi
    from sai_b200.encode import PackedGenotypes, make_layout, unpack_population
    from sai_b200.scoring import synth_fill

    lay = make_layout(N_IND, PLOIDY, LEG_BITS["a"])
    d = torch.empty(int(_cabi.load().sai_packed_bytes(C.byref(lay), S)), dtype=torch.uint8, device="cuda")
    synth_fill(lay, d, S, ROLES, SEED, MISSING)
    pg = PackedGenotypes(lay, S, np.zeros(S, np.int32), d.cpu().numpy())
    del d
    mats = [unpack_population(pg, p) for p in range(lay.n_pops)]
    for m in mats:
        neg = m < 0
        m[neg] = np.where(rng.random(int(neg.sum())) < 0.5, -1, -2)
    return mats


def widen(mats, leg: str, rng):
    """Leg b: 0.1 % of the ref / tgt calls set to 15..30.  Leg c: every call of ref, tgt and the
    source set to 15..127.  Missing calls stay missing."""
    if leg == "a":
        return mats, 0
    out, n_wide = list(mats), 0
    for p in (0, 1) if leg == "b" else (0, 1, 2):
        m = mats[p].copy()
        if leg == "b":
            idx = rng.integers(0, m.size, size=m.size // 1000)
            idx = idx[m.flat[idx] >= 0]
            m.flat[idx] = rng.integers(15, 31, size=idx.size)
        else:  # one pool of values 15..127, read at a different offset per block of sites
            rows = 1 << 16
            pool = (np.frombuffer(rng.bytes((rows + 4096) * m.shape[1]), np.uint8) % 113 + 15).astype(np.int8)
            pool = pool.reshape(rows + 4096, m.shape[1])
            for a in range(0, m.shape[0], rows):
                blk = m[a : a + rows]
                off = int(rng.integers(0, 4096))
                np.copyto(blk, pool[off : off + blk.shape[0]], where=blk >= 0)
        n_wide += int((m >= 15).sum())
        out[p] = m
    return out, n_wide


def stats(ms):
    ms = np.asarray(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()), "reps": len(ms)}


def run_leg(leg, mats, pos, wins, engine, args, other_lib, rng):
    import torch

    import sai_oracle as orc
    from sai_b200.encode import pack_populations
    from sai_b200.scoring import DeviceScorer, make_job

    pg = pack_populations(mats, PLOIDY, pos, bits=LEG_BITS[leg], keep_negatives=True)
    job = make_job(0, 1, [2], True)
    engine.score(pg, wins, [job])
    want = engine.dd_sums(pg, 0, 1, [2])  # warm-up, reference integers
    host_ms = []
    for _ in range(3):
        t0 = time.perf_counter()
        engine.dd_sums(pg, 0, 1, [2])
        host_ms.append((time.perf_counter() - t0) * 1e3)

    dev = torch.device("cuda")
    d_packed = torch.from_numpy(pg.packed).to(dev)
    d_pos = torch.from_numpy(pg.pos).to(dev)
    d_ws = torch.tensor([w[0] for w in wins], dtype=torch.int64, device=dev)
    d_we = torch.tensor([w[1] for w in wins], dtype=torch.int64, device=dev)
    d_neg = [torch.from_numpy(a).to(dev) for a in (pg.neg_site, pg.neg_ind, pg.neg_val)]
    scorers = {"change": DeviceScorer(pg.layout, pg.n_sites, len(wins), 1)}
    if other_lib is not None and leg == "a":
        scorers["compare"] = DeviceScorer(pg.layout, pg.n_sites, len(wins), 1)
        scorers["compare"].lib = other_lib

    def once(sc, times=None):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        ev[0].record()
        hist, _ = sc.site_hist(d_packed, [0, 1, 2])
        ev[1].record()
        r, t, err = sc.dd_sums(d_packed, d_pos, d_ws, d_we, hist, 0, 1, [2], pg.neg_off, *d_neg)
        ev[2].record()
        torch.cuda.synchronize()
        if times is not None:
            times[0].append(ev[0].elapsed_time(ev[1]))
            times[1].append(ev[1].elapsed_time(ev[2]))
        return r, t, err

    times = {k: ([], []) for k in scorers}
    for name, sc in scorers.items():  # warm-up, and the results
        r, t, err = once(sc)
        assert int(err.item()) == 0, name
        assert np.array_equal(r.cpu().numpy(), want[0]) and np.array_equal(t.cpu().numpy(), want[1]), name
    for _ in range(args.reps):  # alternated rep by rep
        for name, sc in scorers.items():
            once(sc, times[name])

    checked = 0
    for i in np.linspace(0, len(wins) - 1, 4).astype(int):
        keep = (pos >= wins[i][0]) & (pos <= wins[i][1])
        if keep.any():
            src = mats[2][keep].astype(np.int64)
            for p, got in ((0, want[0]), (1, want[1])):
                exp = orc.cityblock_sums(src, mats[p][keep].astype(np.int64)).sum(axis=1)
                assert np.array_equal(got[0, i, : N_IND[2]], exp), (leg, i, p)
            checked += 1
    out = {"bits": LEG_BITS[leg], "table_entries": int(pg.neg_off[3]), "host_dd_sums": stats(host_ms),
           "oracle_windows_checked": checked}
    for name, (h, d) in times.items():
        out[name] = {"site_hist": stats(h), "dd_sums": stats(d), "total_median_ms": float(np.median(np.add(h, d)))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--legs", default="a,b,c")
    ap.add_argument("--compare-lib", default=None, help="another build of libsai_b200.so, alternated on leg a")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    from sai_b200.scoring import HostEngine
    from sai_b200.windows import split_genome

    if not torch.cuda.is_available():
        raise SystemExit("dd_bench.py needs a CUDA device")
    print(card(), flush=True)
    rng = np.random.default_rng(6)
    S = args.sites
    pos = np.cumsum(rng.geometric(1.0 / 41.5, size=S).astype(np.int64)).astype(np.int32)
    wins = split_genome([int(pos[0]), int(pos[-1])], 50_000, 10_000)
    base = base_matrices(S, rng)
    other = load_lib(args.compare_lib) if args.compare_lib else None
    engine = HostEngine(0)
    legs = {}
    try:
        for leg in args.legs.split(","):
            mats, n_wide = widen(base, leg, rng)
            legs[leg] = run_leg(leg, mats, pos, wins, engine, args, other, rng)
            legs[leg]["wide_calls"] = n_wide
            print(leg, json.dumps(legs[leg]), flush=True)
    finally:
        engine.close()
    line = json.dumps({"sites": S, "windows": len(wins), "card": card().splitlines()[-1], "legs": legs})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
