"""bgzip inflated on the GPU (``inflate="device"``): the block kernel against the host decoder, corrupt
blocks, and the ingest session's tiles and items against host inflate."""

from __future__ import annotations

import json
import os
import struct
import zlib

import numpy as np
import pytest

from helpers import GOLDEN, SimplePloidy, vcf_case_names

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from sai_b200.scoring import HostEngine

    e = HostEngine(0)
    yield e
    e.close()


def _member(data: bytes, level: int, strategy: int, flush_at=None) -> bytes:
    co = zlib.compressobj(level, zlib.DEFLATED, -15, 9, strategy)
    if flush_at is None:
        payload = co.compress(data) + co.flush()
    else:  # several deflate blocks in one member
        payload = co.compress(data[:flush_at]) + co.flush(zlib.Z_FULL_FLUSH) + co.compress(data[flush_at:]) + co.flush()
    if 26 + len(payload) > 65536:  # a BGZF member is at most 64 KB: incompressible 64 KB of text does not fit
        return None
    return (struct.pack("<BBBBIBBH", 31, 139, 8, 4, 0, 0, 255, 6) + b"BC" + struct.pack("<HH", 2, 25 + len(payload))
            + payload + struct.pack("<II", zlib.crc32(data) & 0xFFFFFFFF, len(data)))


def _sources():
    rng = np.random.default_rng(5)
    gt = np.frombuffer(b"0|0\t" * 16384, dtype=np.uint8).copy()
    gt[rng.random(gt.size) < 0.02] = ord("1")
    fixtures = b"".join(open(os.path.join(GOLDEN, f), "rb").read() for f in sorted(os.listdir(GOLDEN))
                        if f.endswith(".vcf"))
    return {"random": rng.integers(0, 256, 65536, dtype=np.uint8).tobytes(), "one byte": b"A" * 65536,
            "gt runs": gt.tobytes(), "fixtures": (fixtures * (1 + 65536 // len(fixtures)))[:65536]}


def _inflate_on_device(members):
    """All members in one launch: (text per member, status per member)."""
    import torch

    import sai_b200.ops as ops
    from sai_b200 import _cabi

    lib = _cabi.load()
    raw = b"".join(members)
    table, n_text = ops.bgzf_scan_table(raw)
    t = table.numpy().view(ops.BGZF_BLOCK)
    assert len(t) == len(members)
    d_comp = torch.frombuffer(bytearray(raw), dtype=torch.uint8).cuda()
    out = torch.zeros(max(1, n_text), dtype=torch.uint8, device="cuda")
    status = torch.full((len(members),), -1, dtype=torch.int32, device="cuda")
    torch.ops.sai_b200.bgzf_inflate(d_comp, table, out, status)
    text = out.cpu().numpy().tobytes()
    boff = np.ascontiguousarray(np.cumsum([0] + [len(m) for m in members[:-1]]), dtype=np.int64)
    ooff = np.ascontiguousarray(np.append(t["text_off"], n_text), dtype=np.int64)
    return [text[a : a + n] for a, n in zip(t["text_off"], t["isize"])], status.cpu().numpy(), (lib, raw, boff, ooff)


def test_kernel_matches_host_inflate():
    strategies = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]
    members, want = [], []
    for src in _sources().values():
        for size in (0, 1, 257, 258, 32768, 32769, 65280, 65536):
            data = src[:size]
            for level in range(10):
                for strategy in strategies:
                    m = _member(data, level, strategy)
                    if m is not None:
                        members.append(m)
                        want.append(data)
            m = _member(data, 6, zlib.Z_DEFAULT_STRATEGY, flush_at=size // 3) if size > 2 else None
            if m is not None:
                members.append(m)
                want.append(data)
    got, status, (lib, raw, boff, ooff) = _inflate_on_device(members)
    assert (status == 0).all(), np.flatnonzero(status)[:10]
    host = np.empty(int(ooff[-1]) + 1, dtype=np.uint8)
    buf = np.frombuffer(raw, dtype=np.uint8)
    assert lib.sai_bgzf_inflate(buf.ctypes.data, boff.ctypes.data, ooff.ctypes.data, len(members), host.ctypes.data, 0) == 0
    for i, (g, w) in enumerate(zip(got, want)):
        assert g == w, i
        assert g == host[ooff[i] : ooff[i + 1]].tobytes(), i
        assert lib.sai_crc32(host[ooff[i]:].ctypes.data, len(w), 0) == (zlib.crc32(w) & 0xFFFFFFFF)


def test_corrupt_blocks_fail_alone():
    src = _sources()
    members = [_member(s[: 20000 + 1000 * i], 6, zlib.Z_DEFAULT_STRATEGY) for i, s in enumerate(src.values())] * 3
    bad = {}
    m = bytearray(members[1])  # CRC byte
    m[-6] ^= 0x40
    bad[1] = bytes(m)
    m = bytearray(members[5])  # a payload bit
    m[40] ^= 0x10
    bad[5] = bytes(m)
    m = members[10]  # a truncated payload: the BC size shrinks with it
    cut = m[: len(m) - 8 - 200] + m[-8:]
    bad[10] = cut[:16] + struct.pack("<H", len(cut) - 1) + cut[18:]
    corrupted = [bad.get(i, x) for i, x in enumerate(members)]
    good, st_good, _ = _inflate_on_device(members)
    got, status, _ = _inflate_on_device(corrupted)
    assert (st_good == 0).all()
    for i in range(len(members)):
        if i in bad:
            assert status[i] != 0, i
            assert got[i] == b"\n" * len(good[i]), i
        else:
            assert status[i] == 0 and got[i] == good[i], i


def _device_tiles_check(engine, vcf, chrom, pc, lists, anc=None, start=None, end=None):
    """Tiles and positions of inflate="device" equal host ingest's (test_gpu_vcf_ingest._check_tiles)."""
    from test_gpu_vcf_ingest import _host_tiles

    from sai_b200.vcf import _is_bgzf, read_anc_or_error
    from sai_b200.vcf_device import read_loaded, read_plan

    want = _host_tiles(vcf, chrom, pc, lists, anc, start, end)
    plan, requests, out = read_plan(vcf, chrom, pc, *lists)
    a, a_err = read_anc_or_error(anc, chrom, start, end)
    got = read_loaded(engine, vcf, chrom, plan, requests, out, a, a_err, start, end, inflate="device")
    if want is None:
        assert got.n_sites == 0
        return 0
    assert np.array_equal(got.pos, want.pos), (vcf, start, end)
    tiles = engine.loaded_tiles(got.layout, got.n_sites)
    assert tiles.tobytes() == want.packed.tobytes()
    if _is_bgzf(vcf) and got.n_sites:  # whole file or region: the blocks went over compressed
        st = engine.vcf_stats()
        assert st["comp_bytes"] > 0 and st["inflated_slices"] >= 1, st
    return got.n_sites


@pytest.mark.parametrize("name", vcf_case_names())
def test_fixture_tiles_device_inflate(name, engine, tmp_path):
    from test_gpu_vcf_ingest import _fixture_lists

    from sai_b200.vcf import _is_gzip, write_bgzf

    case = json.load(open(os.path.join(GOLDEN, f"vcf_{name}.json")))
    vcf = os.path.join(GOLDEN, case["vcf"])
    pc = SimplePloidy(case["ploidies"])
    anc = os.path.join(GOLDEN, f"vcf_{name}.anc.bed") if case["anc"] else None
    text = open(vcf, "rb").read() if not _is_gzip(vcf) else __import__("gzip").open(vcf).read()
    files = [vcf] if _is_gzip(vcf) else []
    for block in (64, 500):  # 64: the header spans blocks, most blocks hold no newline
        bgz = str(tmp_path / f"x{block}.vcf.gz")
        write_bgzf(bgz, text, block=block)
        files.append(bgz)
    s, e = case["start"], case["end"]
    for f in files:
        for a in {None, anc}:
            for region in ((None, None), (s, e), (s, (s + e) // 2), ((s + e) // 3, e)):
                _device_tiles_check(engine, f, case["chr_name"], pc, _fixture_lists(name), a, *region)
                if region == (None, None) and f != vcf:  # bgzip written here: the blocks went over compressed
                    assert engine.vcf_stats()["comp_bytes"] > 0


@pytest.mark.parametrize("seed, crlf, final_newline", [(21, False, True), (22, True, True), (23, False, False)])
def test_random_vcf_tiles_device_inflate(seed, crlf, final_newline, engine, tmp_path):
    from test_gpu_vcf_ingest import _random_case

    _, bgz, anc, pc, lists, recs = _random_case(tmp_path, seed, crlf, final_newline)
    n = 0
    for a in (None, anc):
        for region in ((None, None), (recs[40][1], recs[300][1])):
            n += _device_tiles_check(engine, bgz, "7", pc, lists, a, *region)
    assert n > 500


def test_single_chromosome_regions_and_tiny_slices(engine, tmp_path):
    """Region reads of a one-chromosome file (the bisection hands its blocks over): starting mid-block,
    ending before the end of the file, at the end, with 64-byte blocks and tiny slices (lines cross
    groups, whole groups hold no newline), with and without a final newline."""
    from sai_b200.configs import PloidyConfig
    from sai_b200.vcf import write_bgzf

    rng = np.random.default_rng(31)
    for final_newline in (True, False):
        vcf = tmp_path / f"one{final_newline}.vcf"
        lines = open(_write_one_chrom(vcf, rng, final_newline), "rb").read()
        (tmp_path / "ref.list").write_text("".join(f"R\ts{i}\n" for i in range(0, 20)))
        (tmp_path / "tgt.list").write_text("".join(f"T\ts{i}\n" for i in range(20, 38)))
        (tmp_path / "src.list").write_text("S\ts38\nS\ts39\n")
        pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 2}, "src": {"S": 2}})
        lists = [str(tmp_path / f"{g}.list") for g in ("ref", "tgt", "src")] + [None]
        pos = [int(x.split(b"\t")[1]) for x in lines.split(b"\n") if x and not x.startswith(b"#")]
        for block, slicing in ((64, (700, 2)), (64, (0, 0)), (3000, (1000, 3))):
            bgz = str(tmp_path / f"one{final_newline}{block}.vcf.gz")
            write_bgzf(bgz, lines, block=block)
            try:
                engine.set_vcf_slicing(*slicing)
                for region in ((pos[0], pos[-1]), (pos[10] + 1, pos[60]), (pos[70], pos[-1] + 10), (pos[-1] + 5, pos[-1] + 50),
                               (None, None)):
                    _device_tiles_check(engine, bgz, "1", pc, lists, None, *region)
                st = engine.vcf_stats()  # the whole file: most groups are inflated on the device
                assert st["inflated_slices"] >= max(1, st["slices"] / 2), st
            finally:
                engine.set_vcf_slicing(0, 0)


def test_deeper_ring_after_a_shallow_one(tmp_path):
    """A fresh engine inflates with a ring of 2 slots, then of 6 and of 3: the compressed ring is rebuilt
    for each depth."""
    from sai_b200.configs import PloidyConfig
    from sai_b200.scoring import HostEngine
    from sai_b200.vcf import write_bgzf

    vcf = _write_one_chrom(tmp_path / "d.vcf", np.random.default_rng(3), True, n_rec=300)
    (tmp_path / "ref.list").write_text("".join(f"R\ts{i}\n" for i in range(0, 20)))
    (tmp_path / "tgt.list").write_text("".join(f"T\ts{i}\n" for i in range(20, 38)))
    (tmp_path / "src.list").write_text("S\ts38\nS\ts39\n")
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 2}, "src": {"S": 2}})
    lists = [str(tmp_path / f"{g}.list") for g in ("ref", "tgt", "src")] + [None]
    bgz = str(tmp_path / "d.vcf.gz")
    write_bgzf(bgz, open(vcf, "rb").read(), block=500)
    eng = HostEngine(0)
    try:
        for ring in (2, 6, 3):
            eng.set_vcf_slicing(1500, ring)
            assert _device_tiles_check(eng, bgz, "1", pc, lists) == 300
            st = eng.vcf_stats()
            assert st["inflated_slices"] > 2 * ring, st
    finally:
        eng.close()


def _write_one_chrom(path, rng, final_newline, n_rec=120, n_smp=40):
    pos = np.sort(rng.choice(np.arange(1, 100 * n_rec), size=n_rec, replace=False))
    rows = ["##fileformat=VCFv4.1", "##a=" + "x" * 300,
            "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(f"s{i}" for i in range(n_smp))]
    for p in pos:
        rows.append("\t".join(["1", str(p), ".", "A", "T", ".", "PASS", ".", "GT"]
                              + [f"{rng.integers(2)}|{rng.integers(2)}" for _ in range(n_smp)]))
    open(path, "w").write("\n".join(rows) + ("\n" if final_newline else ""))
    return path


def test_wide_values_and_ancestral_table(engine, tmp_path):
    from sai_b200.configs import PloidyConfig
    from sai_b200.vcf import write_bgzf

    hdr = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\ta\tb\tc\n"
    rows = ["1\t10\t.\tA\tT\t.\t.\t.\tGT\t0|1\t./.\t1|1", "1\t20\t.\tA\tT\t.\t.\t.\tGT\t9|9\t0|0\t1|0",
            "1\t30\t.\tG\tC\t.\t.\t.\tGT\t0|0\t./.\t1|1"]
    write_bgzf(str(tmp_path / "t.vcf.gz"), (hdr + "\n".join(rows) + "\n").encode(), block=40)
    (tmp_path / "anc.bed").write_text("1\t9\t10\tT\n1\t19\t20\tA\n1\t29\t30\tG\n")
    for g, pop in (("ref", "R a"), ("tgt", "T b"), ("src", "S c")):
        (tmp_path / f"{g}.list").write_text(pop.replace(" ", "\t") + "\n")
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 2}, "src": {"S": 2}})
    lists = [str(tmp_path / f"{g}.list") for g in ("ref", "tgt", "src")] + [None]
    for anc in (str(tmp_path / "anc.bed"), None):
        for region in ((None, None), (1, 25)):
            assert _device_tiles_check(engine, str(tmp_path / "t.vcf.gz"), "1", pc, lists, anc, *region) >= 2


def _pre(vcf, tmp_path, pc, stats, anc, inflate):
    from sai_b200.configs import StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor

    return ChunkPreprocessor(vcf, str(tmp_path / "ref.list"), str(tmp_path / "tgt.list"), str(tmp_path / "src.list"), None,
                             4000, 2000, str(tmp_path / "o.tsv"), pc, StatConfig(json.loads(json.dumps(stats))), anc,
                             ingest="device" if inflate == "device" else "host", inflate=inflate)


def test_items_dd_and_corrupt_file_match_host(tmp_path):
    from test_gpu_vcf_ingest import _random_case, _same_items

    from sai_b200.vcf import write_bgzf

    vcf, bgz, anc, pc, _, recs = _random_case(tmp_path, 41, n_rec=300, n_smp=45, wide=False)
    u = {"ref": {"R1": 0.3, "R2": 0.3}, "tgt": {"T": 0.2}, "src": {"S1": "=1", "S2": ">=0.5"}}
    q = {"ref": {"R1": 0.3, "R2": 0.3}, "tgt": {"T": 0.9}, "src": {"S1": "=1", "S2": ">=0.5"}}
    last = recs[-1][1]
    for stats in ({"U": u, "Q": q}, {"U": u, "DD": True}):
        for region in ((1, last + 5000), (recs[50][1], recs[200][1])):
            got = {i: _pre(bgz, tmp_path, pc, stats, anc, i).run("7", *region) for i in ("host", "device")}
            assert len(got["host"]) > 0
            _same_items(got["device"], got["host"])
    # one corrupt block in the middle: the same exception and message as host inflate
    text = open(vcf, "rb").read()
    write_bgzf(str(tmp_path / "c.vcf.gz"), text, block=3000)
    raw = bytearray(open(tmp_path / "c.vcf.gz", "rb").read())
    at = 0
    for _ in range(len(text) // 3000 // 2):
        at += struct.unpack("<H", raw[at + 16 : at + 18])[0] + 1
    raw[at + 60] ^= 0x08
    (tmp_path / "c.vcf.gz").write_bytes(bytes(raw))
    errors = {}
    for inflate in ("host", "device"):
        with pytest.raises(Exception) as ei:
            _pre(str(tmp_path / "c.vcf.gz"), tmp_path, pc, {"U": u}, None, inflate).run("7", 1, last + 5000)
        errors[inflate] = (type(ei.value), str(ei.value))
    assert errors["device"] == errors["host"]


def test_score_entry_point_device_inflate(tmp_path):
    import yaml

    from sai_b200.score import score
    from sai_b200.vcf import write_bgzf

    case = json.load(open(os.path.join(GOLDEN, "vcf_example_q.json")))
    bgz = str(tmp_path / "q.vcf.gz")
    write_bgzf(bgz, open(os.path.join(GOLDEN, case["vcf"]), "rb").read(), block=300)
    cfg = tmp_path / "cfg.yaml"
    cfg.write_text(yaml.safe_dump({
        "statistics": case["stats"], "ploidies": case["ploidies"],
        "populations": {g: os.path.join(GOLDEN, f"vcf_example_q.{g}.list") for g in ("ref", "tgt", "src")}}))
    texts = {}
    for ingest, inflate in (("host", "host"), ("device", "device")):
        out = tmp_path / inflate / "s.tsv"
        score(bgz, case["chr_name"], case["win_len"], case["win_step"], None, str(out), str(cfg), ingest=ingest,
              inflate=inflate)
        texts[inflate] = [open(out.parent / f).read() for f in sorted(os.listdir(out.parent))]
    assert texts["device"] == texts["host"] and len(texts["host"]) == 2
