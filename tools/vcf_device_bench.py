#!/usr/bin/env python
"""Device VCF ingest against host ingest, file -> results (needs a GPU).

    python tools/vcf_device_bench.py [--sites 600000] [--samples 2504] [--reps 2] [--level 6]

Writes (untimed) a synthetic VCF of diploid, phased GT-only records in plain text and bgzip form
(zlib level ``--level``), then times ``ChunkPreprocessor.run`` over the whole chromosome with
``ingest="host"`` and ``ingest="device"`` -- for bgzip also ``ingest="device", inflate="device"``
(U and Q, one ref / tgt / src population each), checks that the items are identical, and breaks the
device path into stages:
  * the device session's own stages (``HostEngine.vcf_stats``): host seconds staging the text into
    the pinned ring (plain) or inflating the blocks into it (bgzip), host seconds waiting for a free
    ring slot, H2D and parse seconds summed over the real slices (CUDA events), the device span from
    the first copy to the last parse, and the seconds the final synchronise waited;
  * H2D: a pinned host -> device copy of 1 GB (the PCIe bound of plain text);
  * parse: ``torch.ops.sai_b200.vcf_tiles`` on a device-resident 256 MB slice, CUDA events;
  * K1 + K4: ``score_loaded`` on the resident tiles;
  * the layout retry: the plain file with an ancestral table that flips every site (a flipped
    missing call is 4 in a diploid: the parse is repeated with 3 planes) against one that flips none;
  * inflate: ``torch.ops.sai_b200.bgzf_inflate`` on every block of ~256 MB of text whose compressed
    members are resident in HBM, CUDA events; GB/s of text out and of compressed bytes in.
Prints one JSON line (GPU name and power limit included).
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
from sai_b200.configs import PloidyConfig, StatConfig  # noqa: E402
from sai_b200.preprocessors import ChunkPreprocessor  # noqa: E402


def write_vcf(path, n_sites, n_samples, seed=1, block=20000):
    """Fixed-width records (POS zero-padded to 10 digits) assembled as byte matrices."""
    rng = np.random.default_rng(seed)
    tokens = np.frombuffer(b"0|0\t0|1\t1|0\t1|1\t./.\t", dtype=np.uint8).reshape(5, 4)
    pos = np.cumsum(rng.geometric(1 / 40.0, size=n_sites))
    with open(path, "wb") as f:
        f.write(b"##fileformat=VCFv4.1\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
                + "\t".join(f"i{k}" for k in range(n_samples)).encode() + b"\n")
        for b0 in range(0, n_sites, block):
            p = pos[b0 : b0 + block]
            fq = rng.beta(0.2, 2.0, size=(p.size, 1))
            g = (rng.random((p.size, n_samples)) < fq).astype(np.int8) * 2 + (rng.random((p.size, n_samples)) < fq)
            g[rng.random((p.size, n_samples)) < 1e-4] = 4  # rare missing calls
            body = tokens[g].reshape(p.size, 4 * n_samples)
            body[:, -1] = ord("\n")
            head = np.frombuffer(b"".join(b"1\t%010d\t.\tA\tT\t.\tPASS\t.\tGT\t" % x for x in p.tolist()),
                                 dtype=np.uint8).reshape(p.size, -1)
            f.write(np.concatenate([head, body], axis=1).tobytes())
    return pos


def write_bgzf_parallel(path, data: bytes, block=0xFF00, level=6):
    """``vcf.write_bgzf`` with the blocks compressed by a thread pool (zlib releases the GIL)."""
    import struct
    import zlib
    from concurrent.futures import ThreadPoolExecutor

    def member(at):
        chunk = data[at : at + block] if at is not None else b""
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        payload = co.compress(chunk) + co.flush()
        return (struct.pack("<BBBBIBBH", 31, 139, 8, 4, 0, 0, 255, 6) + b"BC" + struct.pack("<HH", 2, 25 + len(payload))
                + payload + struct.pack("<II", zlib.crc32(chunk) & 0xFFFFFFFF, len(chunk)))

    with open(path, "wb") as f, ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        for m in ex.map(member, list(range(0, len(data), block)) + [None], chunksize=64):
            f.write(m)


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def same_items(a, b):
    if len(a) != len(b):
        return False
    for x, y in zip(a, b):
        for k in x:
            if k == "cdd_pos":
                if any(not np.array_equal(x[k][s], y[k][s]) for s in x[k]):
                    return False
            elif repr(x[k]) != repr(y[k]):
                return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sites", type=int, default=600000)
    ap.add_argument("--samples", type=int, default=2504)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--level", type=int, default=6, help="zlib level of the bgzip file")
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("vcf_device_bench needs a CUDA device")
    import sai_b200.ops as ops
    from sai_b200 import _cabi
    from sai_b200.scoring import make_job
    from sai_b200.vcf_device import read_region

    n_ref, n_tgt = int(a.samples * 0.6), int(a.samples * 0.4) - 4
    out = {"gpu": gpu_info(), "sites": a.sites, "samples": a.samples, "level": a.level}
    with tempfile.TemporaryDirectory() as tmp:
        vcf = os.path.join(tmp, "s.vcf")
        pos = write_vcf(vcf, a.sites, a.samples)
        bgz = os.path.join(tmp, "s.vcf.gz")
        write_bgzf_parallel(bgz, open(vcf, "rb").read(), level=a.level)
        text_bytes = os.path.getsize(vcf)
        out["text_GB"] = round(text_bytes / 1e9, 3)
        out["bgzip_GB"] = round(os.path.getsize(bgz) / 1e9, 3)
        groups = {"ref": (0, n_ref, "REF"), "tgt": (n_ref, n_ref + n_tgt, "TGT"), "src": (n_ref + n_tgt, a.samples, "SRC")}
        for g, (lo, hi, name) in groups.items():
            with open(os.path.join(tmp, f"{g}.list"), "w") as f:
                f.writelines(f"{name}\ti{k}\n" for k in range(lo, hi))
        lists = [os.path.join(tmp, f"{g}.list") for g in ("ref", "tgt", "src")]
        pc = PloidyConfig({"ref": {"REF": 2}, "tgt": {"TGT": 2}, "src": {"SRC": 2}})
        stats = {"U": {"ref": {"REF": 0.01}, "tgt": {"TGT": 0.2}, "src": {"SRC": "=1"}},
                 "Q": {"ref": {"REF": 0.01}, "tgt": {"TGT": 0.95}, "src": {"SRC": "=1"}}}
        end = int(pos[-1]) + 1
        for kind, path in (("plain", vcf), ("bgzip", bgz)):
            items, times = {}, {}
            legs = [("host", "host", "host"), ("device", "device", "host")]
            if kind == "bgzip":
                legs.append(("device_inflate", "device", "device"))
            for leg, ingest, inflate in legs:
                pre = ChunkPreprocessor(path, *lists, None, 50000, 10000, os.path.join(tmp, "o.tsv"), pc,
                                        StatConfig(json.loads(json.dumps(stats))), ingest=ingest, inflate=inflate)
                best = None
                for _ in range(a.reps + 1):  # the first run warms the page cache and the engine's buffers
                    t0 = time.perf_counter()
                    items[leg] = pre.run("1", 1, end)
                    dt = time.perf_counter() - t0
                    best = dt if best is None else min(best, dt)
                times[leg] = best
                if ingest == "device":
                    out[f"{kind}_{leg}_stages"] = {k: round(v, 4) for k, v in pre.engine.vcf_stats().items()}
                pre.engine.close()
            out[kind] = {
                "host_s": round(times["host"], 4), "device_s": round(times["device"], 4),
                "speedup": round(times["host"] / times["device"], 3),
                "device_text_GB_s": round(text_bytes / times["device"] / 1e9, 2),
                "device_Ggenotypes_s": round(a.sites * a.samples / times["device"] / 1e9, 3),
                "host_text_GB_s": round(text_bytes / times["host"] / 1e9, 2),
                "identical": same_items(items["host"], items["device"]),
            }
            if kind == "bgzip":
                out[kind].update({
                    "device_inflate_s": round(times["device_inflate"], 4),
                    "device_inflate_speedup": round(times["host"] / times["device_inflate"], 3),
                    "device_inflate_vs_device": round(times["device"] / times["device_inflate"], 3),
                    "device_inflate_identical": same_items(items["host"], items["device_inflate"]),
                })

        # the layout retry: every site flipped (the rare missing calls become 4) against none flipped
        with open(os.path.join(tmp, "ref.bed"), "w") as f_ref, open(os.path.join(tmp, "alt.bed"), "w") as f_alt:
            f_ref.writelines(f"1\t{p - 1}\t{p}\tA\n" for p in pos.tolist())
            f_alt.writelines(f"1\t{p - 1}\t{p}\tT\n" for p in pos.tolist())
        retry = {}
        for name in ("ref", "alt"):
            pre = ChunkPreprocessor(vcf, *lists, None, 50000, 10000, os.path.join(tmp, "o.tsv"), pc,
                                    StatConfig(json.loads(json.dumps(stats))), os.path.join(tmp, f"{name}.bed"),
                                    ingest="device")
            best = None
            for _ in range(a.reps + 1):
                t0 = time.perf_counter()
                pre.run("1", 1, end)
                best = min(best or 1e9, time.perf_counter() - t0)
            retry[f"anc_{name}_device_s"] = round(best, 4)
            pre.engine.close()
        retry["retry_cost"] = round(retry["anc_alt_device_s"] / retry["anc_ref_device_s"], 3)
        out["layout_retry"] = retry

        # H2D: pinned -> device, 1 GB
        h = torch.empty(1 << 30, dtype=torch.uint8).pin_memory()
        d = torch.empty_like(h, device="cuda")
        d.copy_(h, non_blocking=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            d.copy_(h, non_blocking=True)
        e1.record()
        torch.cuda.synchronize()
        out["h2d_GB_s"] = round(3 * (1 << 30) / (e0.elapsed_time(e1) / 1e3) / 1e9, 1)
        del h, d

        # parse kernels on a device-resident slice, and K1 + K4 on the resident tiles
        from sai_b200.scoring import HostEngine

        eng = HostEngine(0)
        loaded = read_region(eng, vcf, "1", pc, *lists, None, None)
        windows = [(s, s + 49999) for s in range(1, end, 10000)]
        job = make_job(0, 1, [2], False, {"w": 0.01, "x": 0.2, "y_list": [("=", 1.0)]},
                       {"w": 0.01, "quantile": 0.95, "y_list": [("=", 1.0)]})
        eng.score_loaded(windows, [job])
        t0 = time.perf_counter()
        for _ in range(3):
            eng.score_loaded(windows, [job])
        out["k1_k4_s"] = round((time.perf_counter() - t0) / 3, 5)
        raw = open(vcf, "rb").read()
        body0 = raw.index(b"\n", raw.index(b"#CHROM")) + 1
        cut = raw.rindex(b"\n", body0, body0 + min(256 << 20, len(raw) - body0)) + 1
        d_text = torch.frombuffer(bytearray(raw[body0:cut]), dtype=torch.uint8).cuda()
        n_cap = (cut - body0) // (4 * a.samples) + 64
        n_cap = (n_cap + 31) // 32 * 32
        q = ops.vcf_query_tensor(loaded.layout, "1")
        cols = torch.arange(a.samples, dtype=torch.int32, device="cuda")  # ref, tgt, src: columns in file order
        scratch = torch.empty(ops.vcf_scratch_bytes(q, d_text.numel(), cols), dtype=torch.uint8, device="cuda")
        tiles = torch.empty(int(_cabi.load().sai_packed_bytes(ops.C.byref(loaded.layout), n_cap)), dtype=torch.uint8,
                            device="cuda")
        pos_d = torch.empty(n_cap, dtype=torch.int32, device="cuda")
        state = torch.zeros(ops.C.sizeof(_cabi.VcfState), dtype=torch.uint8, device="cuda")
        none = torch.empty(0, dtype=torch.int32, device="cuda")

        def parse():
            state.zero_()
            torch.ops.sai_b200.vcf_tiles(d_text, q, cols, none, none, scratch, tiles, pos_d, state)

        parse()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            parse()
        e1.record()
        torch.cuda.synchronize()
        t_parse = e0.elapsed_time(e1) / 1e3 / 5
        n_parsed = int(np.frombuffer(state.cpu().numpy().tobytes()[:8], dtype=np.int64)[0])
        out["parse_slice_MB"] = round(d_text.numel() / 1e6, 1)
        out["parse_sites"] = n_parsed
        out["parse_TB_s"] = round(d_text.numel() / t_parse / 1e12, 3)
        eng.close()

        # the inflate kernel alone: every block of the first ~256 MB of text, members resident in HBM
        mm = np.memmap(bgz, dtype=np.uint8, mode="r")
        table, _ = ops.bgzf_scan_table(mm)
        n = min(table.numel() // ops.BGZF_BLOCK.itemsize, (256 << 20) // 0xFF00 + 1)
        t = table.numpy().view(ops.BGZF_BLOCK)
        comp_bytes = int(t["comp_bytes"][:n].sum())  # the deflate payloads the kernel reads
        text_bytes = int(t["text_off"][n - 1] + t["isize"][n - 1])
        raw = mm[: int(t["comp_off"][n - 1] + t["comp_bytes"][n - 1]) + 8].tobytes()
        table = table[: n * ops.BGZF_BLOCK.itemsize].clone()
        d_comp = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
        d_out = torch.empty(text_bytes, dtype=torch.uint8, device="cuda")
        status = torch.empty(n, dtype=torch.int32, device="cuda")

        def inflate():
            torch.ops.sai_b200.bgzf_inflate(d_comp, table, d_out, status)

        inflate()
        torch.cuda.synchronize()
        ok = bool((status == 0).all()) and d_out[: 1 << 20].cpu().numpy().tobytes() == open(vcf, "rb").read(1 << 20)
        e0.record()
        for _ in range(5):
            inflate()
        e1.record()
        torch.cuda.synchronize()
        t_inf = e0.elapsed_time(e1) / 1e3 / 5
        out["inflate_kernel"] = {"blocks": n, "text_MB": round(text_bytes / 1e6, 1), "comp_MB": round(comp_bytes / 1e6, 1),
                                 "s": round(t_inf, 5), "text_GB_s": round(text_bytes / t_inf / 1e9, 2),
                                 "comp_GB_s": round(comp_bytes / t_inf / 1e9, 3), "ok": ok}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
