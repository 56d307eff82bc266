"""Site-granular stages of the staged genotype pass (k_site_gated): a tile with at most K sites
where a job is still live reads the reference / target only at those sites (a gather), a tile with
more reads them whole.  Inputs are hand-planted so that the number of live sites per tile is
exact; every case is checked against the read-everything path (``_check``: U / Q mask words bit
for bit, Q values by bit pattern, untouched tiles outside the range)."""

import numpy as np
import pytest

from test_gpu_site_gating import _check

pytestmark = pytest.mark.gpu

K = 8  # kGatherSites in sai_b200/csrc/site_kernels.cu


def _pop(rng, n_sites, n, fixed=(), low=(), absent=(), missing=0.0):
    """n diploid individuals.  Background sites are neither all 0 nor all 2 (no source matches
    "=1", nor its 1 - y, by chance) and have a frequency near 0.5; `fixed` sites are all 2, `low`
    sites all 0 but one 1 (frequency 1 / 2n), `absent` sites all missing; then `missing` of all
    calls are set missing."""
    g = rng.integers(0, 3, size=(n_sites, n), dtype=np.int8)
    g[:, 0], g[:, 1] = 0, 2
    fixed, low, absent = (np.asarray(sorted(s), dtype=np.int64) for s in (fixed, low, absent))
    g[fixed] = 2
    g[low] = 0
    g[low, rng.integers(0, n, size=low.size)] = 1
    if missing > 0:
        g[rng.random(g.shape) < missing] = -1
    g[absent] = -1
    return g


def _pack(mats, bits=None):
    import torch

    from sai_b200.encode import pack_populations

    n_sites = mats[0].shape[0]
    pg = pack_populations(mats, [2] * len(mats), np.arange(1, n_sites + 1), bits=bits)
    return pg.layout, torch.from_numpy(pg.packed).cuda()


def _job(ref, tgt, srcs, anc=True, w=0.05):
    from sai_b200.scoring import make_job

    y = [("=", 1.0)] * len(srcs)
    return make_job(ref, tgt, srcs, anc, u=dict(w=w, x=0.5, y_list=y), q=dict(w=w, quantile=0.95, y_list=y))


def _plant(rng, n_tiles, n_src, n_ref, lanes=None):
    """Per tile, n_src source-live sites (random lanes, or `lanes`), the first n_ref of them also
    reference-live."""
    src, ref = set(), set()
    for t in range(n_tiles):
        ls = list(lanes) if lanes is not None else list(rng.choice(32, size=n_src, replace=False))
        src.update(32 * t + int(s) for s in ls[:n_src])
        ref.update(32 * t + int(s) for s in ls[:n_ref])
    return src, ref


def _three_pops(rng, n_sites, src, ref, n=(150, 90, 9), missing=0.0, bits=None, tgt_absent=(), ref_absent=()):
    R = _pop(rng, n_sites, n[0], low=ref, absent=ref_absent, missing=missing)
    T = _pop(rng, n_sites, n[1], absent=tgt_absent, missing=missing)
    S = _pop(rng, n_sites, n[2], fixed=src, missing=missing)
    return _pack([R, T, S], bits)


@pytest.mark.parametrize("n_src,n_ref", [(K, K), (K + 1, K + 1), (K, 1), (K + 1, 2), (20, K), (20, K + 1),
                                         (32, K), (32, K + 1)])
def test_gather_switch(n_src, n_ref):
    """Both sides of the gather / whole-tile switch: K and K + 1 source-live sites (the reference
    gathered, or read whole together with the target), and K and K + 1 reference-live sites on
    tiles with fewer or more source-live sites (the target gathered, or read whole in stage 2)."""
    rng = np.random.default_rng(100 * n_src + n_ref)
    n_tiles = 64
    src, ref = _plant(rng, n_tiles, n_src, n_ref)
    lay, d_packed = _three_pops(rng, 32 * n_tiles, src, ref)
    n_u, n_q = _check(lay, d_packed, 32 * n_tiles, [_job(0, 1, [2]), _job(0, 1, [2], anc=False)])
    assert n_q == 2 * len(ref) and n_u > 0


def test_shared_sectors():
    """Live sites that share one 32-byte sector (4 sites of a pair): lanes 0-3, lanes 28-31, and
    the last sites of a ragged last tile."""
    rng = np.random.default_rng(7)
    n_sites = 32 * 40 + 30
    src = {0, 1, 2, 3, 5 * 32 + 28, 5 * 32 + 29, 5 * 32 + 30, 5 * 32 + 31, 9 * 32 + 31, 10 * 32,
           n_sites - 6, n_sites - 5, n_sites - 4, n_sites - 3, n_sites - 2, n_sites - 1}
    ref = src - {2, 5 * 32 + 29}
    lay, d_packed = _three_pops(rng, n_sites, src, ref)
    n_u, n_q = _check(lay, d_packed, n_sites, [_job(0, 1, [2])])
    assert n_q == len(ref)


@pytest.mark.parametrize("bits", [[2, 2, 2], [3, 3, 2], [4, 4, 2], [8, 8, 2], [3, 4, 8], [8, 3, 4]])
def test_wide_reference(bits):
    """A reference of 2100 individuals (66 groups: three groups on some lanes) and targets of 70;
    2-, 3-, 4- and 8-plane populations on the gather path."""
    rng = np.random.default_rng(sum(bits))
    n_tiles = 48
    src, ref = _plant(rng, n_tiles, 3, 2)
    s2, r2 = _plant(rng, n_tiles, K + 3, K + 1)  # whole-tile reads in the same pass
    src |= {s + 32 * n_tiles for s in s2}
    ref |= {s + 32 * n_tiles for s in r2}
    n_sites = 64 * n_tiles - 11
    src, ref = {s for s in src if s < n_sites}, {s for s in ref if s < n_sites}
    lay, d_packed = _three_pops(rng, n_sites, src, ref, n=(2100, 70, 12), missing=0.01, bits=bits)
    n_u, n_q = _check(lay, d_packed, n_sites, [_job(0, 1, [2])])
    assert n_q > len(ref) // 2


def test_missing_populations():
    """Missing calls everywhere, and whole populations missing at live sites: the reference at
    source-live sites, the target at reference-live sites."""
    rng = np.random.default_rng(11)
    n_tiles = 80
    src, ref = _plant(rng, n_tiles, 4, 3)
    ref_absent = {s for s in src - ref if rng.random() < 0.5}
    tgt_absent = {s for s in ref if rng.random() < 0.3}
    lay, d_packed = _three_pops(rng, 32 * n_tiles, src, ref, missing=0.03, ref_absent=ref_absent,
                                tgt_absent=tgt_absent)
    n_u, n_q = _check(lay, d_packed, 32 * n_tiles, [_job(0, 1, [2]), _job(0, 1, [2], anc=False)])
    assert 0 < n_q < 2 * len(ref)


def test_fused_jobs_differing_gates():
    """Job A live at site 3 and job B at site 17 of the same tiles; B's reference is A's target and
    A's reference is B's source, so one population is read by stage 2 for B and used by stage 3
    for A, and another is read in stage 1 for B and used as A's reference."""
    rng = np.random.default_rng(13)
    n_tiles = 50
    n_sites = 32 * n_tiles
    a = {32 * t + 3 for t in range(n_tiles)}
    b = {32 * t + 17 for t in range(n_tiles)} | {32 * t + s for t in range(0, n_tiles, 5) for s in range(20, 32)}
    P0 = _pop(rng, n_sites, 60, fixed=b, low=a, missing=0.01)
    P1 = _pop(rng, n_sites, 45, low=b, missing=0.01)
    P2 = _pop(rng, n_sites, 6, fixed=a)
    P3 = _pop(rng, n_sites, 33)
    lay, d_packed = _pack([P0, P1, P2, P3])
    jobs = [_job(0, 1, [2]), _job(1, 3, [0]), _job(1, 3, [0, 2], anc=False, w=0.5)]
    n_u, n_q = _check(lay, d_packed, n_sites, jobs)
    assert n_q >= len(a) + len(b)


def test_gather_tile_subranges():
    rng = np.random.default_rng(17)
    n_tiles = 120
    src, ref = _plant(rng, n_tiles, 2, 1)
    s2, r2 = _plant(rng, n_tiles, K + 1, K)
    src |= {s for s in s2 if (s // 32) % 3 == 0}
    ref |= {s for s in r2 if (s // 32) % 3 == 0}
    n_sites = 32 * n_tiles - 5
    src, ref = {s for s in src if s < n_sites}, {s for s in ref if s < n_sites}
    lay, d_packed = _three_pops(rng, n_sites, src, ref, missing=0.01)
    jobs = [_job(0, 1, [2])]
    for tile0, nt in [(0, 1), (1, 6), (5, 50), (n_tiles // 3, n_tiles // 2), (n_tiles - 3, 3), (n_tiles - 1, 1)]:
        _check(lay, d_packed, n_sites, jobs, tile0=tile0, n_tiles=nt)
