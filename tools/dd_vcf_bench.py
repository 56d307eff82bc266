#!/usr/bin/env python
"""DD read on the device (``dd_ingest="device"``) against host ingest (needs a GPU).

    python tools/dd_vcf_bench.py [--sites 600000] [--samples 2504] [--chroms 22] [--genome-sites 10000]

Writes (untimed) synthetic bgzip VCFs of diploid, phased GT-only records with about 1 % missing
calls (``./.``) and times three legs, checking on each that both sides give identical outputs:
  (a) ``score`` of one chromosome of ``--sites`` x ``--samples`` with U + Q + DD: host ingest
      against ``ingest="device", inflate="device", dd_ingest="device"``;
  (b) ``score_genome`` of ``--chroms`` chromosomes with DD: one device pass (``dd_ingest="device"``)
      against the per-chromosome loop a DD configuration takes with ``dd_ingest="host"``;
  (c) ``HostEngine.dd_sums`` of leg (a)'s chunk from the resident table against the call that copies
      the host-built table (``pack_populations(..., keep_negatives=True)``), best of ``--reps``.
Prints one JSON line, the card's name and power limit included.
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


def write_vcf(path, names, n_sites, n_samples, seed):
    from sai_b200.vcf import write_bgzf

    rng = np.random.default_rng(seed)
    tokens = np.frombuffer(b"0|0\t0|1\t1|0\t1|1\t./.\t", dtype=np.uint8).reshape(5, 4)
    head = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
    parts = [(head + "\t".join(f"s{i}" for i in range(n_samples)) + "\n").encode()]
    bed = []
    for name in names:
        pos = np.cumsum(rng.integers(50, 400, size=n_sites)) + 1000
        for a in range(0, n_sites, 20000):  # bounded memory: 20 000 records at a time
            p = pos[a : a + 20000]
            codes = rng.choice(5, size=(p.shape[0], n_samples), p=[0.69, 0.1, 0.1, 0.1, 0.01])
            geno = tokens[codes].reshape(p.shape[0], 4 * n_samples)
            geno[:, -1] = ord("\n")
            rows, w = geno.tobytes(), 4 * n_samples
            parts.append(b"".join(f"{name}\t{q}\t.\tA\tG\t.\tPASS\t.\tGT\t".encode() + rows[i * w : (i + 1) * w]
                                  for i, q in enumerate(p.tolist())))
        bed.append("".join(f"{name}\t{q - 1}\t{q}\tA\n" for q in pos.tolist()))
    text = b"".join(parts)
    write_bgzf(path, text)
    return "".join(bed), len(text)


def setup(d, tag, names, n_sites, n_samples, seed, win_len, win_step):
    import yaml

    sub = os.path.join(d, tag)
    os.makedirs(sub)
    vcf = os.path.join(sub, "g.vcf.gz")
    bed, text_bytes = write_vcf(vcf, names, n_sites, n_samples, seed)
    with open(os.path.join(sub, "anc.bed"), "w") as f:
        f.write(bed)
    lists, third = {}, n_samples // 3
    for g, sl in (("ref", range(0, third)), ("tgt", range(third, 2 * third)), ("src", range(2 * third, n_samples))):
        lists[g] = os.path.join(sub, f"{g}.list")
        with open(lists[g], "w") as f:
            f.writelines(f"{g.upper()}\ts{i}\n" for i in sl)
    ploidies = {"ref": {"REF": 2}, "tgt": {"TGT": 2}, "src": {"SRC": 2}}
    stats = {"U": {"ref": {"REF": 0.3}, "tgt": {"TGT": 0.5}, "src": {"SRC": "=1"}},
             "Q": {"ref": {"REF": 0.3}, "tgt": {"TGT": 0.95}, "src": {"SRC": "=1"}}, "DD": True}
    cfg = os.path.join(sub, "cfg.yaml")
    with open(cfg, "w") as f:
        yaml.safe_dump({"statistics": stats, "ploidies": ploidies, "populations": lists}, f)
    return sub, vcf, os.path.join(sub, "anc.bed"), cfg, lists, ploidies, text_bytes


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown"


def texts(out):
    return [open(p, "rb").read() for p in (out, out[:-4] + ".U.log", out[:-4] + ".Q.log")]


def timed(f):
    t0 = time.perf_counter()
    f()
    return time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=600000, help="records of leg (a)'s chromosome")
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--chroms", type=int, default=22, help="chromosomes of leg (b)")
    ap.add_argument("--genome-sites", type=int, default=10000, help="records per chromosome of leg (b)")
    ap.add_argument("--genome-samples", type=int, default=64)
    ap.add_argument("--win-len", type=int, default=50000)
    ap.add_argument("--win-step", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for the JSON line (default: print only)")
    a = ap.parse_args()

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("dd_vcf_bench.py needs a CUDA device")
    from sai_b200.configs import PloidyConfig
    from sai_b200.encode import pack_populations
    from sai_b200.score import score, score_genome
    from sai_b200.scoring import HostEngine, make_job
    from sai_b200.vcf import read_anc_or_error, read_data
    from sai_b200.vcf_device import read_loaded, read_plan
    from sai_b200.windows import split_genome

    res = {"gpu": gpu_info()}
    with tempfile.TemporaryDirectory() as d:
        # (a) one chromosome, host ingest against device ingest with the device table
        sub, vcf, anc, cfg, lists, ploidies, text_bytes = setup(d, "a", ["chr1"], a.sites, a.samples, 1, a.win_len,
                                                                a.win_step)
        run = lambda tag, **k: score(vcf, "chr1", a.win_len, a.win_step, anc, os.path.join(sub, tag, "s.tsv"), cfg, **k)
        dev = dict(ingest="device", inflate="device", dd_ingest="device")
        run("warm", **dev)  # CUDA context, library, allocations
        t_dev = timed(lambda: run("dev", **dev))
        t_host = timed(lambda: run("host"))
        same_a = texts(os.path.join(sub, "dev", "s.tsv")) == texts(os.path.join(sub, "host", "s.tsv"))
        res["a"] = {"sites": a.sites, "samples": a.samples, "text_bytes": text_bytes, "host_ingest_s": round(t_host, 4),
                    "device_ingest_s": round(t_dev, 4), "speedup": round(t_host / t_dev, 3), "identical_outputs": same_a}

        # (c) dd_sums of that chunk: resident table against the host-built table
        pc = PloidyConfig(ploidies)
        data = read_data(vcf, "chr1", pc, lists["ref"], lists["tgt"], lists["src"], None, anc)
        mats = [data[g][0][n].GT for g, n in (("ref", "REF"), ("tgt", "TGT"), ("src", "SRC"))]
        pos = data["ref"][0]["REF"].POS
        windows = split_genome(pos, a.win_len, a.win_step)
        job = make_job(0, 1, [2], True)
        e_host, e_dev = HostEngine(0), HostEngine(0)
        pg = pack_populations(mats, [2, 2, 2], pos, keep_negatives=True)
        e_host.score(pg, windows, [job])
        plan, requests, out = read_plan(vcf, "chr1", pc, lists["ref"], lists["tgt"], lists["src"], None)
        tab, err = read_anc_or_error(anc, "chr1", None, None)
        loaded = read_loaded(e_dev, vcf, "chr1", plan, requests, out, tab, err, with_outgroup=False, inflate="device",
                             neg_table=True)
        e_dev.score_loaded(windows, [job])
        got, want = e_dev.dd_sums(loaded, 0, 1, [2]), e_host.dd_sums(pg, 0, 1, [2])
        same_c = all(np.array_equal(x, y) for x, y in zip(got, want))
        t_res = min(timed(lambda: e_dev.dd_sums(loaded, 0, 1, [2])) for _ in range(a.reps))
        t_tab = min(timed(lambda: e_host.dd_sums(pg, 0, 1, [2])) for _ in range(a.reps))
        res["c"] = {"sites": int(pos.shape[0]), "windows": len(windows), "table_entries": int(pg.neg_off[-1]),
                    "host_table_s": round(t_tab, 5), "resident_table_s": round(t_res, 5), "identical_sums": same_c}
        e_host.close()
        e_dev.close()

        # (b) a genome with DD: one device pass against the per-chromosome loop
        names = [f"chr{c + 1}" for c in range(a.chroms)]
        sub, vcf, anc, cfg, _, _, text_bytes = setup(d, "b", names, a.genome_sites, a.genome_samples, 2, a.win_len,
                                                     a.win_step)
        gen = lambda tag, dd: score_genome(vcf, names, a.win_len, a.win_step, anc, os.path.join(sub, tag, "s.tsv"), cfg,
                                           inflate="device", dd_ingest=dd)
        gen("warm", "device")
        t_one = timed(lambda: gen("one", "device"))
        t_loop = timed(lambda: gen("loop", "host"))
        same_b = texts(os.path.join(sub, "one", "s.tsv")) == texts(os.path.join(sub, "loop", "s.tsv"))
        res["b"] = {"chroms": a.chroms, "sites_per_chrom": a.genome_sites, "samples": a.genome_samples,
                    "text_bytes": text_bytes, "one_pass_s": round(t_one, 4), "per_chromosome_s": round(t_loop, 4),
                    "speedup": round(t_loop / t_one, 3), "identical_outputs": same_b}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "dd_vcf_bench.json"), "w") as f:
            f.write(line + "\n")
    if not (same_a and same_b and same_c):
        raise SystemExit("a leg's outputs differ")


if __name__ == "__main__":
    main()
