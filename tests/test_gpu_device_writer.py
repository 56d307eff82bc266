"""``write="device"``: the score file and the ``.U.log`` / ``.Q.log`` files formatted on the GPU are byte
for byte those of the host writer (``write_items``), on every path ``score`` and ``score_genome`` take,
and the device's float64 digits are the host build's.  Each comparison checks which writer ran through
``HostEngine.format_calls``."""

from __future__ import annotations

import json
import os
import types

import numpy as np
import pytest

from helpers import vcf_case_names
from test_gpu_genome_vcf import REQUESTED, WIN_LEN, WIN_STEP, _config, _stats, _write_case

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _files(out):
    base = str(out)[:-4]
    return {s: open(base + s, "rb").read() for s in (".tsv", ".U.log", ".Q.log") if os.path.exists(base + s)}


def _both(tmp_path, run):
    """``run(output_file, write)`` with each writer: the files of both, after checking which writer ran."""
    from sai_b200.scoring import HostEngine

    got = {}
    for write in ("host", "device"):
        out = tmp_path / write / "s.tsv"
        before = HostEngine.format_calls
        run(str(out), write)
        calls = HostEngine.format_calls - before
        assert (calls > 0) if write == "device" else (calls == 0), (write, calls)
        got[write] = _files(out)
    assert got["device"].keys() == got["host"].keys()
    for k in got["host"]:
        assert got["device"][k] == got["host"][k], k
    return got["host"]


def test_device_digits_equal_host_build():
    from sai_b200.scoring import HostEngine, format_doubles_host

    rng = np.random.default_rng(99)
    lo, hi, g = rng.random(2_000_000), rng.random(2_000_000), rng.random(2_000_000)
    x = np.concatenate([rng.integers(0, 2**64, size=5_000_000, dtype=np.uint64, endpoint=False).view(np.float64),
                        rng.random(1_000_000), lo + (hi - lo) * g,
                        [0.0, -0.0, np.nan, np.inf, -np.inf, 5e-324, 1e16, 9999999999999998.0, 1e-4, 9.999999999999999e-05]])
    eng = HostEngine(0)
    try:
        dev = eng.format_doubles(x)
    finally:
        eng.close()
    assert np.array_equal(dev, format_doubles_host(x))
    for i in (0, 5_000_000, len(x) - 1, len(x) - 4):
        assert bytes(dev[i]).rstrip(b"\0").decode() == repr(float(x[i]))


def _golden_config(tmp_path, name):
    import yaml

    case = json.load(open(os.path.join(GOLDEN, f"vcf_{name}.json")))
    lists = {g: os.path.join(GOLDEN, f"vcf_{name}.{g}.list") for g in ("ref", "tgt", "src", "outgroup")}
    lists = {g: p for g, p in lists.items() if os.path.exists(p)}
    cfg = tmp_path / "cfg.yaml"
    cfg.write_text(yaml.safe_dump({"statistics": case["stats"], "ploidies": case["ploidies"], "populations": lists}))
    anc = os.path.join(GOLDEN, f"vcf_{name}.anc.bed") if case["anc"] else None
    return case, str(cfg), anc


@pytest.mark.parametrize("ingest", ["host", "device"])
@pytest.mark.parametrize("name", vcf_case_names())
def test_golden_vcfs_through_score(name, ingest, tmp_path):
    from sai_b200.score import score

    case, cfg, anc = _golden_config(tmp_path, name)
    vcf = os.path.join(GOLDEN, case["vcf"])
    _both(tmp_path, lambda out, write: score(vcf, case["chr_name"], case["win_len"], case["win_step"], anc, out, cfg,
                                             ingest=ingest, write=write))


@pytest.mark.parametrize("ingest,dd_ingest", [("host", "host"), ("device", "device")])
def test_all_statistics_two_sources_outgroup_many_combinations(ingest, dd_ingest, tmp_path):
    """Seven statistics, two sources (``Danc.S1`` columns), outgroups: 2 x 3 x 2 = 12 combinations, more
    than one batch of 8 jobs; DD from host ingest and from the device's negative-value table."""
    from sai_b200.score import score

    lists, _ = _write_case(tmp_path)
    cfg = _config(tmp_path, lists, _stats(with_four=True, dd=True))
    files = _both(tmp_path, lambda out, write: score(str(tmp_path / "g.vcf"), "1", WIN_LEN, WIN_STEP,
                                                     str(tmp_path / "anc.bed"), out, cfg, ingest=ingest,
                                                     dd_ingest=dd_ingest, write=write))
    head, *rows = files[".tsv"].decode().splitlines()
    assert "Danc.S1\tDanc.S2" in head and "DD.S2" in head
    assert len({tuple(r.split("\t")[3:7]) for r in rows}) == 12
    assert any("\tnan\tnan" in r for r in rows)  # windows without a site


def test_no_statistic_scored_per_combination(tmp_path):
    """No statistic enabled: the per-combination path scores nothing and counts sites on the host."""
    from sai_b200.score import score

    lists, _ = _write_case(tmp_path)
    cfg = _config(tmp_path, lists, {"Danc": False})
    files = _both(tmp_path, lambda out, write: score(str(tmp_path / "g.vcf"), "10", WIN_LEN, WIN_STEP,
                                                     str(tmp_path / "anc.bed"), out, cfg, write=write))
    assert files[".tsv"].count(b"\n") > 12


@pytest.mark.parametrize("ingest", ["host", "device"])
def test_region_without_data_and_single_combination(ingest, tmp_path):
    """A region past the last record (``_empty_items``) and one combination (the general path)."""
    from sai_b200.configs import PloidyConfig, StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor, DeviceRows, write_items
    from sai_b200.scoring import HostEngine

    lists, _ = _write_case(tmp_path)
    (tmp_path / "r1.list").write_text("R1\tR1_0\nR1\tR1_1\n")
    (tmp_path / "t1.list").write_text("T1\tT1_0\nT1\tT1_1\nT1\tT1_2\n")
    (tmp_path / "s1.list").write_text("S1\tS1_0\n")
    pc = PloidyConfig({"ref": {"R1": 2}, "tgt": {"T1": 2}, "src": {"S1": 2}})
    st = {"Q": {"ref": {"R1": 0.3}, "tgt": {"T1": 0.9}, "src": {"S1": "=1"}},
          "U": {"ref": {"R1": 0.3}, "tgt": {"T1": 0.2}, "src": {"S1": "=1"}}}
    for region in ((1, 20_000), (900_000, 930_000)):
        texts = {}
        for write in ("host", "device"):
            out = tmp_path / write / "o.tsv"
            out.parent.mkdir(exist_ok=True)
            pre = ChunkPreprocessor(str(tmp_path / "g.vcf"), str(tmp_path / "r1.list"), str(tmp_path / "t1.list"),
                                    str(tmp_path / "s1.list"), None, 3000, 1000, str(out), pc,
                                    StatConfig(json.loads(json.dumps(st))), ingest=ingest)
            for p in (out, out.with_suffix(".U.log"), out.with_suffix(".Q.log")):
                p.write_bytes(b"")
            if write == "host":
                write_items(str(out), pre.run("1", *region), pre.stat_config)
            else:
                rows = DeviceRows(pre.stat_config)
                before = HostEngine.format_calls
                assert pre.run_into("1", *region, rows) == []
                rows.write(str(out), pre.engine)
                assert HostEngine.format_calls == before + 1
            texts[write] = _files(out)
        assert texts["device"] == texts["host"]
        assert texts["host"][".U.log"].count(b"NA\n") > 0


@pytest.mark.parametrize("interleave", [False, True])
def test_score_genome_one_pass_and_fallback(interleave, tmp_path):
    from sai_b200.score import score_genome

    lists, _ = _write_case(tmp_path, interleave=interleave)
    cfg = _config(tmp_path, lists, _stats(with_four=True))
    _both(tmp_path, lambda out, write: score_genome(str(tmp_path / "g.vcf"), REQUESTED, WIN_LEN, WIN_STEP,
                                                    str(tmp_path / "anc.bed"), out, cfg, write=write))


def test_score_genome_dd_device_ingest(tmp_path):
    from sai_b200.score import score_genome

    lists, _ = _write_case(tmp_path)
    cfg = _config(tmp_path, lists, _stats(with_four=False, dd=True))
    _both(tmp_path, lambda out, write: score_genome(str(tmp_path / "g.vcf.gz"), REQUESTED, WIN_LEN, WIN_STEP, None, out,
                                                    cfg, inflate="device", dd_ingest="device", write=write))


def test_chromosome_names_of_1_4_and_255_bytes(tmp_path):
    from sai_b200.score import score_genome

    names = ["7", "chrA", "c" * 255]
    lists, _ = _write_case(tmp_path, chroms=[(n, 60, True, "all") for n in names])
    cfg = _config(tmp_path, lists, _stats(with_four=False))
    files = _both(tmp_path, lambda out, write: score_genome(str(tmp_path / "g.vcf"), names, WIN_LEN, WIN_STEP, None, out,
                                                            cfg, write=write))
    for f in (".tsv", ".U.log", ".Q.log"):
        assert b"\n" + b"c" * 255 + b"\t" in files[f] and b"\nchrA\t" in files[f] and b"\n7\t" in files[f]


def test_bad_write_value_raises_before_writing(tmp_path):
    from sai_b200.score import score, score_genome

    lists, _ = _write_case(tmp_path)
    cfg = _config(tmp_path, lists, _stats())
    out = tmp_path / "x" / "s.tsv"
    with pytest.raises(ValueError, match="write must be 'host' or 'device'"):
        score(str(tmp_path / "g.vcf"), "1", WIN_LEN, WIN_STEP, str(tmp_path / "anc.bed"), str(out), cfg, write="gpu")
    with pytest.raises(ValueError, match="write must be 'host' or 'device'"):
        score_genome(str(tmp_path / "g.vcf"), REQUESTED, WIN_LEN, WIN_STEP, None, str(out), cfg, write="Device")
    # a configuration error is raised before any file is written, with either writer
    with pytest.raises(ValueError, match="polarized"):
        score(str(tmp_path / "g.vcf"), "1", WIN_LEN, WIN_STEP, None, str(out), cfg, write="device")
    assert not out.parent.exists()


# ---- formatted rows of chosen values: dense candidate lists and every float64 layout -----------------
class _Res:
    pass


def _results(rng, n_jobs, W, q_values):
    r = _Res()
    r.nsnps = rng.integers(0, 4, size=(n_jobs, W)).astype(np.int32)
    r.nsnps[:, 0] = 5
    r.u = rng.integers(0, 3, size=(n_jobs, W))
    r.u[:, 1] = 1500  # a dense window
    r.u[:, 2] = 0
    r.q_cnt = rng.integers(0, 3, size=(n_jobs, W)).astype(np.int32)
    r.q_cnt[:, 3] = 2500
    r.q = np.resize(q_values, (n_jobs, W)).astype(np.float64)
    for a, n in (("u_start", r.u), ("q_start", r.q_cnt)):
        s = np.zeros((n_jobs, W), dtype=np.int64)
        s[:, 1:] = np.cumsum(n, axis=1)[:, :-1]
        setattr(r, a, s)
    r.totals = np.stack([r.u.sum(1), r.q_cnt.sum(1)], 1)
    r.u_cand = rng.integers(1, 2**31 - 1, size=(n_jobs, int(r.totals[:, 0].max()) + 7)).astype(np.int32)
    r.q_cand = rng.integers(1, 9, size=(n_jobs, int(r.totals[:, 1].max()) + 7)).astype(np.int32)
    return r


def test_dense_windows_and_float_layouts(tmp_path):
    """Windows of 1 500 / 2 500 candidates next to windows of none, and Q / DD / Danc values that need 17
    significant digits or the exponent form, through the one-pass path's block order."""
    from sai_b200.configs import PloidyConfig, StatConfig
    from sai_b200.preprocessors import DeviceRows, score_populations, write_items
    from sai_b200.scoring import HostEngine

    q_values = [0.30000000000000004, 1e-05, 1.2345678901234568e-300, 1e16, 9999999999999998.0, 0.1, np.nan,
                2.5e-7, 123456789012345.67, 0.0001, 9.999999999999999e-05, -0.0, 1.7976931348623157e308]
    names = ["chr1", "2", "c" * 255]
    W_each = 40
    W = W_each * len(names)
    tg, srcs = [f"T{i}" for i in range(10)], ["S1", "S2"]  # 10 combinations: two batches

    class Stub(HostEngine):
        def __init__(self, seed):
            super().__init__(0)
            self.rng = np.random.default_rng(seed)

        def score_loaded_pieces(self, pieces, jobs):
            return _results(self.rng, len(jobs), W, q_values)

        score_resident = lambda self, jobs: _results(self.rng, len(jobs), W, q_values)

        def pattern_sums(self, pg, r, t, o, src):
            s = self.rng.integers(0, 5, size=(len(src), W, 7)).astype(np.float64)
            s[:, ::3, 2] = 1.0 / 3e7  # ratios in exponent form
            return s

        def dd_sums(self, pg, r, t, src):
            s = self.rng.integers(0, 1 << 40, size=(len(src), W, 3))
            return s, s[:, :, ::-1].copy()

    index = {("ref", "R"): 0, ("src", "S1"): 1, ("src", "S2"): 2, ("out", "O"): 3,
             **{("tgt", t): 4 + i for i, t in enumerate(tg)}}
    loaded = types.SimpleNamespace(
        first_site=[0] * len(names), n_sites=[10] * len(names), names=names, pos=[np.arange(10, dtype=np.int32)] * 3,
        index=index, layout=types.SimpleNamespace(pop=[types.SimpleNamespace(n_samples=3)] * 16))
    wins = [[(1 + 1000 * i, 3000 + 1000 * i) for i in range(W_each)] for _ in names]
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {t: 2 for t in tg}, "src": {s: 2 for s in srcs}, "outgroup": {"O": 2}})
    sc = StatConfig({"Q": {"ref": {"R": 0.3}, "tgt": {t: 0.9 for t in tg}, "src": {s: "=1" for s in srcs}},
                     "DD": True, "Danc": True,
                     "U": {"ref": {"R": 0.3}, "tgt": {t: 0.2 for t in tg}, "src": {s: "=1" for s in srcs}}})
    texts = {}
    for write in ("host", "device"):
        out = tmp_path / f"{write}.tsv"
        eng = Stub(3)
        rows = DeviceRows(sc) if write == "device" else None
        items = score_populations("chr1", {t: wins for t in tg}, {"R": None}, {t: None for t in tg},
                                  {s: None for s in srcs}, pc, sc, True, eng, out_data={"O": None}, num_src=2,
                                  loaded=loaded, sink=rows)
        if rows is None:
            write_items(str(out), items, sc)
        else:
            before = HostEngine.format_calls
            rows.write(str(out), eng)
            assert HostEngine.format_calls == before + 1
        eng.close()
        texts[write] = _files(out)
    assert texts["device"] == texts["host"]
    tsv = texts["host"][".tsv"].decode()
    for v in ("0.30000000000000004", "1e-05", "1.2345678901234568e-300", "1e+16", "9999999999999998.0", "\tnan"):
        assert v in tsv, v
    longest = max(line.count(b",") for line in texts["host"][".Q.log"].split(b"\n"))
    assert longest >= 2499 and b"\tNA\n" in texts["host"][".U.log"]
