"""DD and pattern sums after scoring, on tiles already resident in HBM: one chunk or a genome in pieces.

A single chunk is the one-piece case of a genome scored in pieces, so every route must give the
same numbers.  Pinned here:
- the int64 DD sums and the float64 pattern sums, bit for bit, of three routes: the host-packed
  matrices of each chromosome with the host-built negative-value table (``sai_engine_dd_sums``),
  a single-chromosome device read with its resident table (``sai_engine_dd_sums_loaded``), and a
  genome read scored in pieces.  The file has missing calls, a chromosome of one record, a
  chromosome the genome route gives no windows and a source population of 5 bit-planes;
- the refusals of the two DD entry points, with their messages.
Every file is generated here from a seed.
"""

from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from helpers import SimplePloidy
from test_gpu_genome_vcf import PLOIDY, REQUESTED, WIN_LEN, WIN_STEP, _samples, _write_case

pytestmark = pytest.mark.gpu

GROUP_OF = {"ref": "ref", "tgt": "tgt", "src": "src", "out": "outgroup"}
WIDE = ("1", "chrX")  # chromosomes where S1 has calls of 12, 16 and 24: 5 bit-planes
NO_WINDOWS = "10"  # the genome route scores this chromosome as a piece without windows
# (ref, tgt, sources, outgroup) of the DD and pattern-sum calls
COMBOS = [("R1", "T1", ("S1", "S2"), "O1"), ("R2", "T3", ("S2",), "O2"), ("R1", "T2", ("S1",), "O2")]


@pytest.fixture(scope="module")
def engine():
    from sai_b200.scoring import HostEngine

    e = HostEngine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def case(tmp_path_factory):
    return _make_case(tmp_path_factory.mktemp("resident"))


def _make_case(d):
    """The genome test file under ``d`` with wide source calls written into S1 on the ``WIDE`` chromosomes."""
    lists, _ = _write_case(d, seed=5)
    rng = np.random.default_rng(5)
    s1 = [9 + i for i, s in enumerate(_samples()) if s.startswith("S1_")]
    lines = (d / "g.vcf").read_text().splitlines(keepends=True)
    for i, line in enumerate(lines):
        f = line.split("\t")
        if line.startswith("#") or f[0] not in WIDE:
            continue
        for k in s1:
            if rng.random() < 0.25:
                f[k] = str(rng.choice(["0|12", "7|9", "12|12"]))
        lines[i] = "\t".join(f)
    (d / "g.vcf").write_text("".join(lines))
    return str(d / "g.vcf"), [lists[g] for g in ("ref", "tgt", "src", "outgroup")]


def _plan(vcf, lists):
    from sai_b200.vcf_device import read_plan

    return read_plan(vcf, REQUESTED[0], SimplePloidy(PLOIDY), *lists)


def _windows(pos):
    top = int(pos[-1])
    return [(s, s + WIN_LEN - 1) for s in range(1, top + 1, WIN_STEP)] + [(top + 1, top + 50)]


def _job(index):
    from sai_b200.scoring import make_job

    r, t, src, _ = COMBOS[0]
    return make_job(index[("ref", r)], index[("tgt", t)], [index[("src", s)] for s in src], False)


def _sums(engine, pg, index):
    """Per combination: the pattern sums ``[n_src, W, 7]`` and the DD sums ``[n_src, W, m_max]``."""
    out = []
    for r, t, src, o in COMBOS:
        ri, ti, si = index[("ref", r)], index[("tgt", t)], [index[("src", s)] for s in src]
        out.append((engine.pattern_sums(pg, ri, ti, index[("out", o)], si), *engine.dd_sums(pg, ri, ti, si)))
    return out


def _host_route(engine, vcf, lists, name, layout, index):
    from sai_b200.encode import pack_populations
    from sai_b200.vcf import read_data

    d = read_data(vcf, name, SimplePloidy(PLOIDY), *lists, None)
    order = sorted(index.items(), key=lambda kv: kv[1])
    mats = [d[GROUP_OF[g]][0][p].GT for (g, p), _ in order]
    pos = d["ref"][0]["R1"].POS
    pg = pack_populations(mats, [2] * len(mats), pos, bits=[int(layout.pop[i].bits) for i in range(len(mats))],
                          keep_negatives=True)
    assert int(pg.neg_off[-1]) > 0  # missing calls
    wins = _windows(pos)
    engine.score(pg, wins, [_job(index)])
    return wins, pg, _sums(engine, pg, index)


def _genome(engine, vcf, lists, neg=True):
    from sai_b200.vcf_device import genome_tables, read_genome

    plan, requests, out = _plan(vcf, lists)
    g = read_genome(engine, vcf, REQUESTED, plan, requests, out, genome_tables(REQUESTED, None), neg_table=neg)
    assert g is not None and g.neg == neg
    return g


def _read_chunk(engine, vcf, lists, name, neg=True):
    from sai_b200.vcf_device import read_loaded

    plan, requests, out = _plan(vcf, lists)
    c = read_loaded(engine, vcf, name, plan, requests, out, None, None, neg_table=neg)
    assert c is not None and c.neg == neg
    return c


def _same(got, want, name):
    for (gp, gr, gt), (wp, wr, wt) in zip(got, want):
        assert gp.tobytes() == wp.tobytes(), name
        assert np.array_equal(gr, wr) and np.array_equal(gt, wt), name


def test_dd_and_pattern_sums_equal_across_routes(engine, case):
    vcf, lists = case
    g = _genome(engine, vcf, lists)
    assert int(g.layout.pop[g.index[("src", "S1")]].bits) == 5
    host = {name: _host_route(engine, vcf, lists, name, g.layout, g.index) for name in REQUESTED}
    assert sum(int(s[1].any()) for h in host.values() for s in h[2]) > 10  # nonzero DD sums
    # the genome read, scored in pieces (one of them without windows)
    g = _genome(engine, vcf, lists)
    pieces = [([] if name == NO_WINDOWS else host[name][0], max(f, 0), n)
              for name, f, n in zip(REQUESTED, g.first_site, g.n_sites)]
    engine.score_loaded_pieces(pieces, [_job(g.index)])
    whole = _sums(engine, g, g.index)
    at = 0
    for name, (w, _, _) in zip(REQUESTED, pieces):
        cols = slice(at, at + len(w))
        at += len(w)
        if name != NO_WINDOWS:
            _same([tuple(a[:, cols] for a in s) for s in whole], host[name][2], name)
    assert at == whole[0][0].shape[1]
    # one chromosome read on the device, scored as one chunk
    for name in REQUESTED:
        c = _read_chunk(engine, vcf, lists, name)
        assert c.index == g.index
        engine.score_loaded(host[name][0], [_job(c.index)])
        _same(_sums(engine, c, c.index), host[name][2], name)


def test_refusals(engine, case):
    from sai_b200 import _cabi

    vcf, lists = case
    # the host-table entry on tiles scored in pieces
    g = _genome(engine, vcf, lists)
    wins, pg, _ = _host_route(engine, vcf, lists, "1", g.layout, g.index)
    g = _genome(engine, vcf, lists)
    engine.score_loaded_pieces([(wins, 0, g.n_sites[0])], [_job(g.index)])
    with pytest.raises(ValueError, match="scored in pieces"):
        engine.dd_sums(pg, 0, 1, [g.index[("src", "S1")]])
    # a piece that is not a chromosome of the session
    assert g.first_site[0] == 0 and g.n_sites[0] > 32
    engine.score_loaded_pieces([(wins, 0, 32)], [_job(g.index)])
    with pytest.raises(ValueError, match="is not a chromosome"):
        engine.dd_sums(g, 0, 1, [g.index[("src", "S1")]])
    # the resident-table entry after a session that kept no table
    c = _read_chunk(engine, vcf, lists, "1", neg=False)
    engine.score_loaded(wins, [_job(c.index)])
    sums = np.zeros((1, len(wins), 8), dtype=np.int64)
    src = (C.c_int32 * 1)(c.index[("src", "S1")])
    with pytest.raises(ValueError, match="kept no negative-value table"):
        _cabi.check(_cabi.load().sai_engine_dd_sums_loaded(engine._handle(), 0, 1, src, 1, sums.ctypes.data,
                                                           sums.ctypes.data, 8))
