"""DD on device-parsed VCFs (``dd_ingest="device"``): the genotype pass keeps the raw value of
every missing call, the negative-value table DD reads next to the tiles.

The host is the specification: the resident table must equal ``encode.negative_table`` of
``read_data``'s matrices entry for entry (per chromosome for a genome read), and items and text
outputs must equal those of host ingest, DD compared bit for bit.  The retries of the read are
asserted from the return codes of every finish call.
"""

from __future__ import annotations

import numpy as np
import pytest

import sai_oracle as orc
from test_gpu_vcf_ingest import _random_case, _same_items
from test_gpu_genome_vcf import (REQUESTED, WIN_LEN, WIN_STEP, _config, _per_chromosome, _stats, _texts,
                                 _write_case)

pytestmark = pytest.mark.gpu

GROUP_OF = {"ref": "ref", "tgt": "tgt", "src": "src", "out": "outgroup"}


@pytest.fixture(scope="module")
def engine():
    from sai_b200.scoring import HostEngine

    e = HostEngine(0)
    yield e
    e.close()


@pytest.fixture
def finish_codes(monkeypatch):
    """Return codes of every sai_engine_vcf_finish / _genome_finish: the retries made visible."""
    from sai_b200 import _cabi

    lib = _cabi.load()
    codes = []
    for name in ("sai_engine_vcf_finish", "sai_engine_vcf_genome_finish"):
        real = getattr(lib, name)

        def spy(*args, real=real):
            rc = real(*args)
            codes.append(int(rc))
            return rc

        monkeypatch.setattr(lib, name, spy, raising=False)
    return codes


@pytest.fixture
def device_only(monkeypatch):
    """``device_only(slicing)``: from then on the per-chromosome path may not run (``score_genome``
    must take the one-pass read), and the ingest session it opens uses ``slicing``."""
    from sai_b200 import preprocessors

    def arm(slicing=None):
        def run(self, *a, **k):
            raise AssertionError("the per-chromosome path ran")

        init = preprocessors.ChunkPreprocessor.__init__

        def init_with_slicing(self, *a, **k):
            init(self, *a, **k)
            if slicing:
                self.engine.set_vcf_slicing(*slicing)

        monkeypatch.setattr(preprocessors.ChunkPreprocessor, "run", run)
        monkeypatch.setattr(preprocessors.ChunkPreprocessor, "__init__", init_with_slicing)

    return arm


def _host_table(loaded, data):
    """``negative_table`` of the host matrices in the device layout's population order."""
    from sai_b200.encode import negative_table

    order = sorted(loaded.index.items(), key=lambda kv: kv[1])
    return negative_table([data[GROUP_OF[g]][0][name].GT for (g, name), _ in order])


def _check_table(off, site, ind, val, c, want):
    w_off, w_site, w_ind, w_val = want
    lo = int(off[c, 0])
    assert np.array_equal(off[c] - lo, w_off)
    hi = lo + int(w_off[-1])
    assert np.array_equal(site[lo:hi], w_site)
    assert np.array_equal(ind[lo:hi], w_ind)
    assert np.array_equal(val[lo:hi], w_val)
    return hi - lo


PLOIDIES = {"mixed": {"ref": {"R1": 2, "R2": 4}, "tgt": {"T": 2}, "src": {"S1": 1, "S2": 3}},
            "ploidy8": {"ref": {"R1": 2, "R2": 8}, "tgt": {"T": 3}, "src": {"S1": 1, "S2": 2}}}


def _read(engine, vcf, anc, pc, lists, start, end, inflate, neg=True):
    from sai_b200.vcf import read_anc_or_error
    from sai_b200.vcf_device import read_loaded, read_plan

    plan, requests, out = read_plan(vcf, "7", pc, *lists)
    a, a_err = read_anc_or_error(anc, "7", start, end)
    return read_loaded(engine, vcf, "7", plan, requests, out, a, a_err, start, end, inflate=inflate, neg_table=neg)


@pytest.mark.parametrize("seed, ploidy", [(1, "mixed"), (2, "ploidy8"), (3, "mixed")])
def test_table_equals_host_negative_table(seed, ploidy, engine, tmp_path):
    from sai_b200.configs import PloidyConfig
    from sai_b200.vcf import read_data

    vcf, bgz, anc, _, lists, recs = _random_case(tmp_path, seed)
    pc = PloidyConfig(PLOIDIES[ploidy])
    n = 0
    for f, inflate in ((vcf, "host"), (bgz, "host"), (bgz, "device")):
        for a in (None, anc):
            for start, end in ((None, None), (recs[40][1], recs[300][1])):
                for slicing in ((0, 0), (700, 3)):
                    engine.set_vcf_slicing(*slicing)
                    try:
                        got = _read(engine, f, a, pc, lists, start, end, inflate)
                    finally:
                        engine.set_vcf_slicing(0, 0)
                    assert got.neg
                    data = read_data(f, "7", pc, *lists, a, start, end)
                    tab = engine.loaded_neg_table(1, got.layout.n_pops)
                    n += _check_table(*tab, 0, _host_table(got, data))
    assert n > 10000
    vals = engine.loaded_neg_table(1, got.layout.n_pops)[3]
    assert set(np.unique(vals).tolist()) >= {-1, -2}


def test_capacity_and_layout_repeats_rebuild_the_table(engine, tmp_path, finish_codes):
    """The first capacity (1/64 of the site capacity per individual) is far below this file's
    missing calls: the finish reports SAI_E_CAPACITY and the read repeats with the true count; the
    wide values then take the SAI_E_DOMAIN repeat in the same read."""
    from sai_b200 import _cabi
    from sai_b200.configs import PloidyConfig
    from sai_b200.vcf import read_data

    pc = PloidyConfig(PLOIDIES["mixed"])
    for wide, want in ((False, [_cabi.E_CAPACITY, 0]), (True, [_cabi.E_CAPACITY, _cabi.E_DOMAIN, 0])):
        (tmp_path / f"w{wide}").mkdir()
        vcf, _, _, _, lists, _ = _random_case(tmp_path / f"w{wide}", 4, n_rec=600, wide=wide)
        finish_codes.clear()
        got = _read(engine, vcf, None, pc, lists, None, None, "host")
        assert finish_codes == want
        data = read_data(vcf, "7", pc, *lists, None, None, None)
        assert _check_table(*engine.loaded_neg_table(1, got.layout.n_pops), 0, _host_table(got, data)) > 5000


def _pre(vcf, lists, out, pc, stats, anc, ingest, dd_ingest="host", inflate="host"):
    from sai_b200.configs import StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor

    return ChunkPreprocessor(vcf, *lists, 3000, 1000, str(out), pc, StatConfig(stats), anc, ingest=ingest,
                             inflate=inflate, dd_ingest=dd_ingest)


def _run_text(pre, chrom, start, end):
    items = pre.run(chrom, start, end)
    pre.process_items(items)
    out = pre.output_file
    return items, [open(p).read() for p in (out, out[:-4] + ".U.log", out[:-4] + ".Q.log")]


@pytest.mark.parametrize("fmt, inflate", [("vcf", "host"), ("vcf.gz", "host"), ("vcf.gz", "device")])
def test_items_and_files_equal_host_ingest(fmt, inflate, tmp_path, finish_codes):
    from sai_b200.configs import PloidyConfig

    vcf, bgz, anc, _, lists, recs = _random_case(tmp_path, 7, n_rec=700)
    f = vcf if fmt == "vcf" else bgz
    pc = PloidyConfig(PLOIDIES["mixed"])
    stats = {"U": {"ref": {"R1": 0.3, "R2": 0.3}, "tgt": {"T": 0.1}, "src": {"S1": ">=0.5", "S2": ">0"}},
             "Q": {"ref": {"R1": 0.3, "R2": 0.3}, "tgt": {"T": 0.9}, "src": {"S1": ">=0.5", "S2": ">0"}}, "DD": True}
    n_dd = 0
    for a in (None, anc):
        for start, end in ((1, recs[-1][1] + 100), (recs[100][1], recs[500][1])):
            dev = _pre(f, lists, tmp_path / "d.tsv", pc, stats, a, "device", "device", inflate)
            assert dev.device_fallback("7", start, end) is None
            assert "DD" in _pre(f, lists, tmp_path / "x.tsv", pc, stats, a, "device").device_fallback("7", start, end)
            finish_codes.clear()
            got, got_text = _run_text(dev, "7", start, end)
            assert finish_codes and finish_codes[-1] == 0  # the device read ran
            want, want_text = _run_text(_pre(f, lists, tmp_path / "h.tsv", pc, stats, a, "host"), "7", start, end)
            _same_items(got, want)
            for g, w in zip(got, want):
                if g["nsnps"]:
                    assert [float(x).hex() for x in g["DD"]] == [float(x).hex() for x in w["DD"]]
                    n_dd += 1
            assert got_text == want_text
            for p in (tmp_path / "d.tsv", tmp_path / "h.tsv"):
                p.unlink()
                for s in (".U.log", ".Q.log"):
                    p.with_suffix(s).unlink()
    assert n_dd > 50


def test_wide_values_on_the_device_path_match_the_oracle(tmp_path):
    """The 5-8-plane DD case (values >= 16, flipped ``./././././././.``) read on the device."""
    from sai_b200.configs import PloidyConfig, StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor
    from sai_b200.vcf import read_data
    from test_gpu_dd_wide import _write_vcf

    rng = np.random.default_rng(21)
    n_r, n_t, n_s1, n_s2 = 40, 35, 2, 3
    vcf = tmp_path / "m.vcf"
    samples, recs = _write_vcf(vcf, rng, 400, n_r, n_t, n_s1, n_s2)
    groups = {"r.list": ("R", 0, n_r), "t.list": ("T", n_r, n_t), "s.list": [("S1", n_r + n_t, n_s1), ("S2", n_r + n_t + n_s1, n_s2)]}
    for fname, spec in groups.items():
        spec = spec if isinstance(spec, list) else [spec]
        (tmp_path / fname).write_text("".join(f"{pop}\t{samples[i]}\n" for pop, a, n in spec for i in range(a, a + n)))
    anc = tmp_path / "anc.bed"
    anc.write_text("".join(f"1\t{p - 1}\t{p}\t{alt if rng.random() < 0.4 else ref}\n" for p, ref, alt in recs
                           if rng.random() < 0.95))
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 8}, "src": {"S1": 2, "S2": 4}})
    stats = {"U": {"ref": {"R": 0.3}, "tgt": {"T": 0.1}, "src": {"S1": ">=0.5", "S2": ">0"}}, "DD": True}
    lists = [str(tmp_path / g) for g in ("r.list", "t.list", "s.list")]
    start, end, win_len, win_step = 1, int(recs[-1][0]) + 3000, 2000, 1000
    n_dd = 0
    for a in (None, str(anc)):
        data = read_data(str(vcf), "1", pc, *lists, None, a, start, end)
        mk = lambda g: {p: orc.PopData(d.POS, d.GT.astype(np.int64)) for p, d in data[g][0].items()}
        ref_d, tgt_d, src_d = mk("ref"), mk("tgt"), mk("src")
        if a is not None:
            assert (tgt_d["T"].GT == 16).any()  # flipped "./././././././."
        exp = orc.score_chunk("1", start, end, win_len, win_step, ref_d, tgt_d, src_d, pc, StatConfig(stats), a is not None)
        rows, logs = orc.format_items(exp, ["U", "DD"])
        out = tmp_path / f"d.{a is not None}.tsv"
        pre = ChunkPreprocessor(str(vcf), *lists, None, win_len, win_step, str(out), pc, StatConfig(stats), a,
                                ingest="device", dd_ingest="device")
        assert pre.device_fallback("1", start, end) is None
        items = pre.run("1", start, end)
        assert len(items) == len(exp)
        for g, e in zip(items, exp):
            assert (g["start"], g["end"], g["nsnps"]) == (e["start"], e["end"], e["nsnps"])
            if e["nsnps"]:
                assert [float(x).hex() for x in g["DD"]] == [float(x).hex() for x in e["DD"]]
                n_dd += 1
        pre.process_items(items)
        assert out.read_text() == "".join(rows)
        assert out.with_suffix(".U.log").read_text() == "".join(logs["U"])
    assert n_dd > 20


@pytest.mark.parametrize("fmt, inflate, slicing", [("vcf", "host", None), ("vcf", "host", (400, 3)),
                                                   ("vcf.gz", "host", (1000, 2)), ("vcf.gz", "device", None),
                                                   ("vcf.gz", "device", (700, 4))])
def test_score_genome_with_dd_equals_per_chromosome_score(fmt, inflate, slicing, tmp_path, device_only):
    from sai_b200.score import score_genome

    lists, _ = _write_case(tmp_path)
    cfg = _config(tmp_path, lists, _stats(dd=True))
    vcf, anc = str(tmp_path / f"g.{fmt}"), str(tmp_path / "anc.bed")
    want = _per_chromosome(vcf, REQUESTED, anc, tmp_path / "want" / "s.tsv", cfg)
    device_only(slicing)
    out = tmp_path / "got" / "s.tsv"
    score_genome(vcf, REQUESTED, WIN_LEN, WIN_STEP, anc, str(out), cfg, inflate=inflate, dd_ingest="device")
    got = _texts(out)
    assert got == want
    assert "DD" in got[0].split(b"\n", 1)[0].decode()


@pytest.mark.parametrize("fmt, inflate, slicing", [("vcf", "host", (300, 3)), ("vcf.gz", "device", (700, 4))])
def test_genome_table_per_chromosome_equals_host(fmt, inflate, slicing, engine, tmp_path, finish_codes):
    from sai_b200.vcf import read_data
    from sai_b200.vcf_device import genome_tables, read_genome, read_plan
    from helpers import SimplePloidy
    from test_gpu_genome_vcf import GROUPS, PLOIDY

    lists, _ = _write_case(tmp_path, seed=1)
    vcf, anc = str(tmp_path / f"g.{fmt}"), str(tmp_path / "anc.bed")
    pc = SimplePloidy(PLOIDY)
    plan, requests, out = read_plan(vcf, REQUESTED[0], pc, lists["ref"], lists["tgt"], lists["src"], lists["outgroup"])
    engine.set_vcf_slicing(*slicing)
    try:
        g = read_genome(engine, vcf, REQUESTED, plan, requests, out, genome_tables(REQUESTED, anc), inflate=inflate,
                        neg_table=True)
    finally:
        engine.set_vcf_slicing(0, 0)
    assert g.neg and finish_codes[-1] == 0
    tab = engine.loaded_neg_table(len(REQUESTED), g.layout.n_pops)
    n = 0
    for c, name in enumerate(REQUESTED):
        d = read_data(vcf, name, pc, lists["ref"], lists["tgt"], lists["src"], lists["outgroup"], anc)
        if d["ref"][0] is None:
            assert tab[0][c, -1] == tab[0][c, 0], name
            continue
        n += _check_table(*tab, c, _host_table(g, d))
    assert n > 500
    assert tab[0][-1, -1] == tab[1].shape[0]
