"""Device VCF ingest (``ingest="device"``): VCF text parsed on the GPU into the packed tiles.

The host parser is the specification: the device tiles and positions must equal, byte for byte,
``pack_populations`` over what ``read_data`` returns, and the scored items and text outputs must
equal those of ``ingest="host"``.
"""

from __future__ import annotations

import json
import os

import numpy as np
import pytest

from helpers import GOLDEN, SimplePloidy, SimpleStats, check_items, vcf_case_names

pytestmark = pytest.mark.gpu

GROUPS = ("ref", "tgt", "src", "outgroup")


@pytest.fixture(scope="module")
def engine():
    from sai_b200.scoring import HostEngine

    e = HostEngine(0)
    yield e
    e.close()


def _host_tiles(vcf, chrom, pc, lists, anc, start, end, with_outgroup=True):
    from sai_b200.encode import pack_populations
    from sai_b200.vcf import read_data

    d = read_data(vcf, chrom, pc, *lists, anc, start, end)
    mats, ploidy, pos = [], [], None
    for g in GROUPS:
        data = d[g][0]
        if data is None or (g == "outgroup" and not with_outgroup):
            continue
        for name, pdat in data.items():
            mats.append(pdat.GT)
            ploidy.append(pc.root[g][name])
            pos = pdat.POS
    if not mats:
        return None
    return pack_populations(mats, ploidy, pos)


def _check_tiles(engine, vcf, chrom, pc, lists, anc=None, start=None, end=None):
    from sai_b200.vcf_device import read_region

    want = _host_tiles(vcf, chrom, pc, lists, anc, start, end)
    got = read_region(engine, vcf, chrom, pc, *lists, anc, start, end)
    if want is None:
        assert got.n_sites == 0
        return 0
    assert np.array_equal(got.pos, want.pos), (vcf, start, end)
    for p in range(want.layout.n_pops):
        assert bytes(got.layout.pop[p]) == bytes(want.layout.pop[p]), p
    tiles = engine.loaded_tiles(got.layout, got.n_sites)
    assert tiles.tobytes() == want.packed.tobytes()
    return got.n_sites


def _fixture_lists(name):
    f = lambda g: os.path.join(GOLDEN, f"vcf_{name}.{g}.list")
    return [f("ref"), f("tgt"), f("src"), f("outgroup") if os.path.exists(f("outgroup")) else None]


@pytest.mark.parametrize("name", vcf_case_names())
def test_fixture_tiles_match_host_pack(name, engine, tmp_path):
    from sai_b200.vcf import write_bgzf, _is_gzip

    case = json.load(open(os.path.join(GOLDEN, f"vcf_{name}.json")))
    vcf = os.path.join(GOLDEN, case["vcf"])
    pc = SimplePloidy(case["ploidies"])
    anc = os.path.join(GOLDEN, f"vcf_{name}.anc.bed") if case["anc"] else None
    files = [vcf]
    if not _is_gzip(vcf):
        bgz = str(tmp_path / "x.vcf.gz")
        write_bgzf(bgz, open(vcf, "rb").read(), block=500)
        files.append(bgz)
    for f in files:
        for a in {None, anc}:
            for region in ((None, None), (case["start"], case["end"]), (case["start"], (case["start"] + case["end"]) // 2)):
                _check_tiles(engine, f, case["chr_name"], pc, _fixture_lists(name), a, *region)


def _random_vcf(path, rng, n_rec, n_smp, crlf=False, final_newline=True, wide=True):
    """Records of every shape the host parser handles: GT:DP and GT-not-first formats, multi-digit
    and junk alleles, haploid / triploid fields, '.', './.', '1/.', missing trailing columns,
    comment and blank lines, other contigs, records cut inside the fixed columns."""
    lines = ["##fileformat=VCFv4.1", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
             + "\t".join(f"s{i}" for i in range(n_smp))]
    pos = np.sort(rng.choice(np.arange(1, 40 * n_rec), size=n_rec, replace=False))
    recs = []
    for p in pos:
        r = rng.random()
        if r < 0.02:
            lines.append("# a comment line")
        elif r < 0.03:
            lines.append("")
        chrom = "7" if rng.random() < 0.85 else rng.choice(["77", "x7"])
        ref = "ACGT"[rng.integers(4)]
        alt = "ACGT"[(("ACGT".index(ref)) + 1 + rng.integers(3)) % 4] + (",<DEL>" if rng.random() < 0.1 else "")
        if wide and rng.random() < 0.03:  # cut inside the fixed columns
            cols = [chrom, str(p), ".", ref, alt, ".", "PASS", "AA=x", "GT"]
            lines.append("\t".join(cols[: rng.integers(1, 9)]))
            continue
        fmt = rng.choice(["GT", "GT", "GT", "GT:DP", "DP:GT:GQ"])
        fields = []
        for _ in range(n_smp):
            pl = int(rng.choice([1, 2, 2, 2, 2, 3]))
            al = []
            for _k in range(pl):
                x = rng.random()
                if not wide and 0.08 <= x < 0.105:  # no values above 14 (DD's limit) and no junk (the Python reader)
                    x = 0.5
                al.append("." if x < 0.08 else ("12" if x < 0.09 else ("9" if x < 0.1 else ("1a" if x < 0.105 else str(int(x > 0.6))))))
            gt = al[0] + "".join(("|" if rng.random() < 0.5 else "/") + a for a in al[1:])
            fields.append({"GT": gt, "GT:DP": gt + ":12", "DP:GT:GQ": "7:" + gt + ":30"}[fmt])
        if wide and rng.random() < 0.05:
            fields = fields[: rng.integers(0, n_smp)]  # missing trailing columns
        lines.append("\t".join([chrom, str(p), ".", ref, alt, ".", "PASS", "AA=x", fmt] + fields))
        recs.append((chrom, int(p), ref, alt.split(",")[0]))
    nl = "\r\n" if crlf else "\n"
    text = nl.join(lines) + (nl if final_newline else "")
    open(path, "w", newline="").write(text)
    return recs


def _random_case(tmp_path, seed, crlf=False, final_newline=True, n_rec=500, n_smp=45, wide=True):
    from sai_b200.configs import PloidyConfig
    from sai_b200.vcf import write_bgzf

    rng = np.random.default_rng(seed)
    vcf = tmp_path / f"r{seed}.vcf"
    recs = _random_vcf(vcf, rng, n_rec, n_smp, crlf, final_newline, wide)
    (tmp_path / "ref.list").write_text("".join(f"R1\ts{i}\n" for i in range(0, 40)) + "".join(f"R2\ts{i}\n" for i in range(5, 12)))
    (tmp_path / "tgt.list").write_text("".join(f"T\ts{i}\n" for i in range(12, 44)))
    (tmp_path / "src.list").write_text("S1\ts40\nS1\ts44\nS2\ts42\n")
    anc = tmp_path / "anc.bed"
    with open(anc, "w") as f:
        for chrom, p, ref, alt in recs:
            r = rng.random()
            if r < 0.1:
                continue
            f.write(f"{chrom}\t{p - 1}\t{p}\t{ref if r < 0.4 else (alt if r < 0.9 else 'N')}\n")
    bgz = tmp_path / f"r{seed}.vcf.gz"
    write_bgzf(str(bgz), vcf.read_bytes(), block=3000)
    pc = PloidyConfig({"ref": {"R1": 2, "R2": 4}, "tgt": {"T": 2}, "src": {"S1": 1, "S2": 3}})
    lists = [str(tmp_path / f"{g}.list") for g in ("ref", "tgt", "src")] + [None]
    return str(vcf), str(bgz), str(anc), pc, lists, recs


@pytest.mark.parametrize("seed, crlf, final_newline", [(1, False, True), (2, True, True), (3, False, False)])
def test_random_vcf_tiles_match_host_pack(seed, crlf, final_newline, engine, tmp_path):
    vcf, bgz, anc, pc, lists, recs = _random_case(tmp_path, seed, crlf, final_newline)
    n = 0
    for f in (vcf, bgz):
        for a in (None, anc):
            for region in ((None, None), (recs[40][1], recs[300][1])):
                n += _check_tiles(engine, f, "7", pc, lists, a, *region)
    assert n > 500


def test_tiny_slices_straddle_records_and_tiles(engine, tmp_path):
    vcf, bgz, anc, pc, lists, _ = _random_case(tmp_path, 5, n_rec=300, n_smp=45)
    try:
        engine.set_vcf_slicing(700, 3)  # a record is ~180 bytes: records and 32-site tiles cross slices
        for f in (vcf, bgz):
            for a in (None, anc):
                assert _check_tiles(engine, f, "7", pc, lists, a) > 100
                # plain: ~700-byte slices; bgzip (inflated straight into the ring): one 3000-byte block per slice
                assert engine.vcf_slices() > (3 * 10 if f == vcf else 3 * 5)
    finally:
        engine.set_vcf_slicing(0, 0)


def test_bgzf_feed_tiny_blocks_and_header_inside_a_block(engine, tmp_path):
    """The bgzip feed with blocks far smaller than a record (a line spans many blocks, the header ends
    inside a block) and with one block larger than the slice size."""
    from sai_b200.vcf import write_bgzf

    vcf, _, anc, pc, lists, _ = _random_case(tmp_path, 7, n_rec=200, n_smp=45, final_newline=False)
    text = open(vcf, "rb").read()
    for block, slicing in ((97, (700, 2)), (60000, (700, 2)), (5000, (0, 0))):
        bgz = str(tmp_path / f"b{block}.vcf.gz")
        write_bgzf(bgz, text, block=block)
        try:
            engine.set_vcf_slicing(*slicing)
            assert _check_tiles(engine, bgz, "7", pc, lists, anc) > 50
        finally:
            engine.set_vcf_slicing(0, 0)


def test_missing_outgroup_sample_raises_like_host(tmp_path):
    """A sample of a population that is not parsed (the outgroup without a four-population statistic)
    missing from the VCF: the same ValueError as host ingest."""
    from sai_b200.configs import PloidyConfig, StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor

    vcf, _, _, _, _, recs = _random_case(tmp_path, 17, n_rec=100, n_smp=45, wide=False)
    (tmp_path / "r.list").write_text("R\ts0\nR\ts1\n")
    (tmp_path / "t.list").write_text("T\ts2\n")
    (tmp_path / "s.list").write_text("S\ts3\n")
    (tmp_path / "o.list").write_text("O\tnobody\n")
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 2}, "src": {"S": 2}, "outgroup": {"O": 2}})
    u = {"U": {"ref": {"R": 0.3}, "tgt": {"T": 0.2}, "src": {"S": "=1"}}}
    for ingest in ("host", "device"):
        pre = ChunkPreprocessor(vcf, str(tmp_path / "r.list"), str(tmp_path / "t.list"), str(tmp_path / "s.list"),
                                str(tmp_path / "o.list"), 5000, 5000, str(tmp_path / "o.tsv"), pc, StatConfig(u),
                                ingest=ingest)
        with pytest.raises(ValueError, match="Failed to read VCF file"):
            pre.run("7", 1, recs[-1][1])


def test_wide_values_take_the_retry_path(engine, tmp_path):
    """Flipped missing calls (4 in a diploid) and values above 14 do not fit the ploidy's planes:
    the parse is repeated with the host's layout and the tiles are identical."""
    from sai_b200.configs import PloidyConfig

    hdr = "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\ta\tb\tc\n"
    rows = ["1\t10\t.\tA\tT\t.\t.\t.\tGT\t0|1\t./.\t1|1", "1\t20\t.\tA\tT\t.\t.\t.\tGT\t9|9\t0|0\t1|0",
            "1\t30\t.\tG\tC\t.\t.\t.\tGT\t0|0\t./.\t1|1"]
    (tmp_path / "t.vcf").write_text(hdr + "\n".join(rows) + "\n")
    (tmp_path / "anc.bed").write_text("1\t9\t10\tT\n1\t19\t20\tA\n1\t29\t30\tG\n")
    for g, pop in (("ref", "R a"), ("tgt", "T b"), ("src", "S c")):
        (tmp_path / f"{g}.list").write_text(pop.replace(" ", "\t") + "\n")
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 2}, "src": {"S": 2}})
    lists = [str(tmp_path / f"{g}.list") for g in ("ref", "tgt", "src")] + [None]
    _check_tiles(engine, str(tmp_path / "t.vcf"), "1", pc, lists, str(tmp_path / "anc.bed"))
    _check_tiles(engine, str(tmp_path / "t.vcf"), "1", pc, lists, None)


def _preprocessor(name, out, ingest, stats=None):
    from sai_b200.preprocessors import ChunkPreprocessor

    case = json.load(open(os.path.join(GOLDEN, f"vcf_{name}.json")))
    lists = _fixture_lists(name)
    return case, ChunkPreprocessor(
        vcf_file=os.path.join(GOLDEN, case["vcf"]), ref_ind_file=lists[0], tgt_ind_file=lists[1], src_ind_file=lists[2],
        out_ind_file=lists[3], win_len=case["win_len"], win_step=case["win_step"], output_file=str(out),
        ploidy_config=SimplePloidy(case["ploidies"]), stat_config=SimpleStats(stats or case["stats"]),
        anc_allele_file=os.path.join(GOLDEN, f"vcf_{name}.anc.bed") if case["anc"] else None, ingest=ingest)


def _texts(out):
    return {p: open(p).read() for p in (str(out), str(out)[:-4] + ".U.log", str(out)[:-4] + ".Q.log") if os.path.exists(p)}


@pytest.mark.parametrize("name", vcf_case_names())
def test_fixture_items_device_ingest(name, tmp_path):
    case, pre = _preprocessor(name, tmp_path / "d.tsv", "device")
    assert pre.device_fallback(case["chr_name"], case["start"], case["end"]) is None
    items = pre.run(case["chr_name"], case["start"], case["end"])
    check_items(items, case["items"], q_tol=0.0, four_tol=1e-12)
    pre.process_items(items)
    assert open(tmp_path / "d.tsv").read() == case["text"]["tsv"]
    _, host = _preprocessor(name, tmp_path / "h.tsv", "host")
    host.process_items(host.run(case["chr_name"], case["start"], case["end"]))
    assert list(_texts(tmp_path / "d.tsv").values()) == list(_texts(tmp_path / "h.tsv").values())
    if name == "example_q":
        assert float(items[0]["Q"]) == 0.9
    if name == "example_u":
        assert items[0]["U"] == 3
    if name == "mixed_ploidy":
        assert [it["U"] for it in items] == [0, 1]
    if name == "outgroup_stats":
        want = dict(fd=0.0012826844929596443, df=0.0012417913767941238, Danc=-0.12498082112760132, Dplus=-0.12149240420484364)
        for k, v in want.items():
            assert items[0][k][0] == v


def _same_items(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert x.keys() == y.keys()
        for k in x:
            if k == "cdd_pos":
                assert x[k].keys() == y[k].keys()
                for s in x[k]:
                    assert np.array_equal(x[k][s], y[k][s]) and np.asarray(x[k][s]).dtype == np.asarray(y[k][s]).dtype
            else:
                assert repr(x[k]) == repr(y[k]), (k, x[k], y[k])


def test_many_combinations_empty_region_and_gap(tmp_path):
    """More than 8 (ref, tgt, src) combinations (score_resident batches), an empty region and a
    gap chunk with an ancestral table: identical items to the host path."""
    from sai_b200.configs import PloidyConfig, StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor

    vcf, bgz, anc, _, _, recs = _random_case(tmp_path, 11, n_rec=400, n_smp=45)
    (tmp_path / "ref3.list").write_text("".join(f"R{k}\ts{i}\n" for k in range(3) for i in range(k, 30, 3)))
    (tmp_path / "tgt3.list").write_text("".join(f"T{k}\ts{i}\n" for k in range(3) for i in range(30 + k, 42, 3)))
    (tmp_path / "src3.list").write_text("S1\ts42\nS2\ts43\nS3\ts44\n")
    pc = PloidyConfig({"ref": {f"R{k}": 2 for k in range(3)}, "tgt": {f"T{k}": 2 for k in range(3)},
                       "src": {"S1": 2, "S2": 2, "S3": 2}})
    y = {"S1": "=1", "S2": ">=0.5", "S3": "<0.5"}
    sc = {"U": {"ref": {f"R{k}": 0.3 for k in range(3)}, "tgt": {f"T{k}": 0.2 for k in range(3)}, "src": y},
          "Q": {"ref": {f"R{k}": 0.3 for k in range(3)}, "tgt": {f"T{k}": 0.9 for k in range(3)}, "src": y}}
    last = recs[-1][1]
    for f in (vcf, bgz):
        for a in (None, anc):
            for region in ((1, last + 5000), (last + 100, last + 20000)):
                got = {}
                for ingest in ("host", "device"):
                    pre = ChunkPreprocessor(f, str(tmp_path / "ref3.list"), str(tmp_path / "tgt3.list"),
                                            str(tmp_path / "src3.list"), None, 4000, 2000, str(tmp_path / "o.tsv"),
                                            pc, StatConfig(json.loads(json.dumps(sc))), a, ingest=ingest)
                    got[ingest] = pre.run("7", *region)
                assert len(got["host"]) >= 27
                _same_items(got["device"], got["host"])


def test_fallbacks_give_host_output(tmp_path):
    """DD, more than 16 populations and long ancestral alleles are read on the host."""
    from sai_b200.configs import PloidyConfig, StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor

    vcf, _, anc, _, _, recs = _random_case(tmp_path, 13, n_rec=200, n_smp=45, wide=False)
    (tmp_path / "r.list").write_text("".join(f"R\ts{i}\n" for i in range(20)))
    (tmp_path / "t.list").write_text("".join(f"T\ts{i}\n" for i in range(20, 40)))
    (tmp_path / "s.list").write_text("S\ts40\nS\ts41\n")
    (tmp_path / "many.list").write_text("".join(f"T{i}\ts{i}\n" for i in range(20)))
    long_anc = tmp_path / "long.bed"
    long_anc.write_text(open(anc).read() + f"7\t{recs[0][1] + 1}\t{recs[0][1] + 2}\tACGTACGTA\n")
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 2}, "src": {"S": 2}})
    pc_many = PloidyConfig({"ref": {"R": 2}, "tgt": {f"T{i}": 2 for i in range(20)}, "src": {"S": 2}})
    u = {"ref": {"R": 0.3}, "tgt": {"T": 0.2}, "src": {"S": "=1"}}
    cases = [
        ("DD", "t.list", pc, {"U": u, "DD": True}, str(anc)),
        ("populations", "many.list", pc_many, {"U": {**u, "tgt": {f"T{i}": 0.2 for i in range(20)}}}, str(anc)),
        ("longer than 7", "t.list", pc, {"U": u}, str(long_anc)),
    ]
    for reason, tgt, ploidy, stats, a in cases:
        got = {}
        for ingest in ("host", "device"):
            pre = ChunkPreprocessor(vcf, str(tmp_path / "r.list"), str(tmp_path / tgt), str(tmp_path / "s.list"), None,
                                    5000, 5000, str(tmp_path / "o.tsv"), ploidy, StatConfig(json.loads(json.dumps(stats))), a,
                                    ingest=ingest)
            if ingest == "device":
                assert reason in pre.device_fallback("7", 1, recs[-1][1])
            got[ingest] = pre.run("7", 1, recs[-1][1])
        _same_items(got["device"], got["host"])


def test_score_entry_point_device_ingest(tmp_path):
    import yaml

    from sai_b200.score import score

    case = json.load(open(os.path.join(GOLDEN, "vcf_example_q.json")))
    cfg = tmp_path / "cfg.yaml"
    cfg.write_text(yaml.safe_dump({
        "statistics": case["stats"], "ploidies": case["ploidies"],
        "populations": {g: os.path.join(GOLDEN, f"vcf_example_q.{g}.list") for g in ("ref", "tgt", "src")}}))
    texts = {}
    for ingest in ("host", "device"):
        out = tmp_path / ingest / "s.tsv"
        score(os.path.join(GOLDEN, case["vcf"]), case["chr_name"], case["win_len"], case["win_step"], None, str(out),
              str(cfg), ingest=ingest)
        texts[ingest] = list(_texts(out).values())
    assert texts["device"] == texts["host"] and len(texts["host"]) == 2


def test_torch_op_matches_engine(engine, tmp_path):
    import torch

    import sai_b200.ops as ops
    from sai_b200 import _cabi
    from sai_b200.vcf import anc_table, read_anc_arrays
    from sai_b200.vcf_device import read_region

    vcf, _, anc, pc, lists, _ = _random_case(tmp_path, 21, n_rec=300, n_smp=45)
    loaded = read_region(engine, vcf, "7", pc, *lists, anc)
    want = engine.loaded_tiles(loaded.layout, loaded.n_sites)
    text = open(vcf, "rb").read()
    body = text[text.index(b"\n", text.index(b"#CHROM")) + 1 :]
    body = body if body.endswith(b"\n") else body + b"\n"
    names = text[text.index(b"#CHROM") :].split(b"\n", 1)[0].decode().split("\t")[9:]
    cols = []
    for g in ("ref", "tgt", "src"):
        for line in open(lists[("ref", "tgt", "src").index(g)]):
            cols.append((line.split()[0], names.index(line.split()[1])))
    order = [p for g in ("ref", "tgt", "src") for p in pc.root[g]]
    sample_column = torch.tensor([c for p in order for name, c in cols if name == p], dtype=torch.int32, device="cuda")
    apos, abuf, n = anc_table(read_anc_arrays(anc, "7"))
    n_sites_cap = (loaded.n_sites + 31) // 32 * 32
    q = ops.vcf_query_tensor(loaded.layout, "7")
    half = body.rindex(b"\n", 0, len(body) // 2) + 1  # two slices chained through `state`
    d_text = torch.frombuffer(bytearray(body), dtype=torch.uint8).cuda()
    scratch = torch.empty(ops.vcf_scratch_bytes(q, max(half, len(body) - half), sample_column), dtype=torch.uint8,
                          device="cuda")  # sized for the larger slice only
    tiles = torch.empty(int(_cabi.load().sai_packed_bytes(ops.C.byref(loaded.layout), n_sites_cap)), dtype=torch.uint8,
                        device="cuda")
    pos = torch.empty(n_sites_cap, dtype=torch.int32, device="cuda")
    state = torch.zeros(ops.C.sizeof(_cabi.VcfState), dtype=torch.uint8, device="cuda")
    for a, b in ((0, half), (half, len(body))):
        torch.ops.sai_b200.vcf_tiles(d_text[a:b].clone(), q, sample_column, torch.from_numpy(apos).cuda(),
                                     torch.frombuffer(bytearray(abuf), dtype=torch.uint8).cuda(), scratch, tiles, pos, state)
    torch.cuda.synchronize()
    st = _cabi.VcfState.from_buffer_copy(state.cpu().numpy().tobytes())
    assert st.n_sites == loaded.n_sites and st.overflow == 0
    assert np.array_equal(pos[: loaded.n_sites].cpu().numpy(), loaded.pos)
    assert tiles[: want.size].cpu().numpy().tobytes() == want.tobytes()
