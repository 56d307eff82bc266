"""The staged genotype pass (k_site_gated: sources first, then the references and targets of the
jobs still live on a tile) against the pass that reads every population: ``site_counts`` followed
by ``flags_from_counts``.  The U and Q mask words must agree bit for bit for every job and tile,
and the Q values at every Q-flagged site."""

import numpy as np
import pytest

import synth

pytestmark = pytest.mark.gpu


def _check(lay, d_packed, n_sites, jobs, tile0=0, n_tiles=None):
    """Gated site_flags over tiles [tile0, tile0 + n_tiles) == the read-everything path there;
    tiles outside the range are left untouched.  Returns the number of flagged (U, Q) sites."""
    import torch

    from sai_b200.scoring import DeviceScorer

    ref = DeviceScorer(lay, n_sites, 1, len(jobs))
    ref.site_counts(d_packed)
    ref.flags_from_counts(jobs)
    got = DeviceScorer(lay, n_sites, 1, len(jobs))
    sentinel = 0x5A5A5A5A
    got.mask_u.fill_(sentinel)
    got.mask_q.fill_(sentinel)
    got.qval.fill_(-7.0)
    got.site_flags(d_packed, jobs, tile0=tile0, n_tiles=n_tiles)
    torch.cuda.synchronize()
    nt = got.n_tiles
    t1 = nt if n_tiles is None else tile0 + n_tiles
    mu, mq = got.mask_u.cpu().numpy(), got.mask_q.cpu().numpy()
    eu, eq = ref.mask_u.cpu().numpy(), ref.mask_q.cpu().numpy()
    assert np.array_equal(mu[:, tile0:t1], eu[:, tile0:t1])
    assert np.array_equal(mq[:, tile0:t1], eq[:, tile0:t1])
    assert (mu[:, :tile0] == sentinel).all() and (mu[:, t1:nt] == sentinel).all()
    assert (mq[:, :tile0] == sentinel).all() and (mq[:, t1:nt] == sentinel).all()
    qg, qe = got.qval.cpu().numpy(), ref.qval.cpu().numpy()
    n_u = n_q = 0
    for j in range(len(jobs)):
        bits = np.unpackbits(eq[j, tile0:t1].astype(np.uint32).view(np.uint8), bitorder="little").astype(bool)
        sites = np.flatnonzero(bits) + tile0 * 32
        assert np.array_equal(qg[j, sites].view(np.int64), qe[j, sites].view(np.int64)), j
        n_q += sites.size
        n_u += int(np.unpackbits(eu[j, tile0:t1].astype(np.uint32).view(np.uint8)).sum())
    return n_u, n_q


def _bench_job(anc=True):
    from sai_b200.scoring import make_job

    return make_job(0, 1, [2], anc, u=dict(w=0.01, x=0.5, y_list=[("=", 1.0)]),
                    q=dict(w=0.01, quantile=0.95, y_list=[("=", 1.0)]))


@pytest.mark.parametrize("missing", [0.0, 0.01])
def test_bench_generator(missing):
    import torch

    from sai_b200 import _cabi
    from sai_b200.encode import make_layout
    from sai_b200.scoring import synth_fill
    import ctypes as C

    n = 65536
    lay = make_layout([1500, 1000, 4], [2, 2, 2], [2, 2, 2])
    d_packed = torch.empty(int(_cabi.load().sai_packed_bytes(C.byref(lay), n)), dtype=torch.uint8, device="cuda")
    synth_fill(lay, d_packed, n, [0, 1, 2], 20261020, missing)
    n_u, n_q = _check(lay, d_packed, n, [_bench_job(True), _bench_job(False)])
    assert n_u > 0 and n_q > 0


def _random_case(seed, n_sites, bits, missing, src_all_missing=0.0):
    """Seven populations: R, T1, T2 (haploid), S1, S2 (haploid), S3, and X, which no job uses."""
    import torch

    from sai_b200.encode import pack_populations

    pops = {"ref": {"R": (150, 2), "X": (40, 2)}, "tgt": {"T1": (90, 2), "T2": (70, 1)},
            "src": {"S1": (3, 2), "S2": (5, 1), "S3": (33, 2)}}
    pos, mats = synth.make_populations(seed, n_sites, pops, mean_gap=30.0, introgressed=0.03, missing=missing,
                                       src_all_missing=src_all_missing)
    order = [mats["ref"]["R"], mats["tgt"]["T1"], mats["tgt"]["T2"], mats["src"]["S1"], mats["src"]["S2"],
             mats["src"]["S3"], mats["ref"]["X"]]
    if src_all_missing > 0:  # the reference population too, at other sites
        rng = np.random.default_rng(seed + 1)
        order[0][rng.random(n_sites) < src_all_missing] = -1
    ploidy = [2, 2, 1, 2, 1, 2, 2]
    pg = pack_populations(order, ploidy, pos, bits=bits)
    return pg, torch.from_numpy(pg.packed).cuda()


R, T1, T2, S1, S2, S3, X = range(7)


def _fused_jobs():
    from sai_b200.scoring import make_job

    u = lambda w, x, ys: dict(w=w, x=x, y_list=ys)
    q = lambda w, ys: dict(w=w, quantile=0.95, y_list=ys)
    return [
        make_job(R, T1, [S1], True, u=u(0.05, 0.2, [("=", 1.0)]), q=q(0.05, [("=", 1.0)])),
        # U and Q with different w and y; two sources; no ancestral alleles (1 - y, inversion)
        make_job(R, T2, [S1, S2], False, u=u(0.3, 0.1, [(">=", 0.5), ("<", 0.5)]), q=q(0.5, [("<", 0.5), (">", 0.2)])),
        # U only; T1 is a target above and the reference here, S2 a source above and here
        make_job(T1, R, [S2], False, u=u(0.6, 0.1, [("<", 0.2)])),
        # Q only; S1 is a source above and the reference here, T2 a target above and a source here
        make_job(S1, T1, [T2], True, q=q(0.4, [(">", 0.3)])),
        make_job(R, T1, [S1, S2, S3], False, u=u(0.5, 0.0, [("=", 1.0), ("<=", 0.8), (">", 0.1)]),
                 q=q(0.5, [("=", 1.0), ("<=", 0.8), (">", 0.1)])),
        make_job(T2, T1, [S3], True, u=u(0.9, 0.3, [(">=", 0.05)]), q=q(0.2, [("<=", 0.05)])),
        make_job(R, S3, [S1, T2], False, q=q(1.0, [("<=", 0.0), (">=", 0.5)])),
        make_job(R, T1, [S2], False, u=u(0.1, 0.5, [("=", 1.0)]), q=q(0.2, [(">", 0.5)])),
    ]


@pytest.mark.parametrize("bits", [[2] * 7, [3, 2, 4, 3, 2, 8, 2], [4, 3, 2, 2, 8, 4, 3], [8] * 7])
@pytest.mark.parametrize("missing", [0.0, 0.02])
def test_fused_jobs(bits, missing):
    n = 20000 + 13  # n_sites % 32 != 0
    pg, d_packed = _random_case(11 + bits[0] + int(100 * missing), n, bits, missing)
    jobs = _fused_jobs()
    n_u, n_q = _check(pg.layout, d_packed, n, jobs)
    assert n_u > 0 and n_q > 0


def test_population_missing_at_some_sites():
    n = 12345
    pg, d_packed = _random_case(5, n, None, 0.01, src_all_missing=0.05)
    n_u, n_q = _check(pg.layout, d_packed, n, _fused_jobs())
    assert n_u > 0 and n_q > 0


def test_tile_subranges():
    """Slice by slice, as the host engine calls the pass."""
    n = 40000 + 7
    pg, d_packed = _random_case(23, n, None, 0.01)
    nt = (n + 31) // 32
    jobs = _fused_jobs()[:5]
    for tile0, n_tiles in [(0, 1), (3, 100), (nt // 3, nt // 2), (nt - 5, 5), (nt - 1, 1), (17, 0)]:
        _check(pg.layout, d_packed, n, jobs, tile0=tile0, n_tiles=n_tiles)


@pytest.mark.parametrize("anc", [True, False])
def test_every_tile_live(anc):
    from sai_b200.scoring import make_job

    n = 9000 + 5
    pg, d_packed = _random_case(31, n, None, 0.01)
    job = make_job(R, T1, [S3], anc, u=dict(w=1.0, x=0.0, y_list=[(">=", 0.0)]),
                   q=dict(w=1.0, quantile=0.95, y_list=[(">=", 0.0)]))
    n_u, n_q = _check(pg.layout, d_packed, n, [job])
    assert n_q > n // 2


def test_no_tile_live():
    import torch

    from sai_b200.encode import pack_populations
    from sai_b200.scoring import make_job

    n = 5000
    rng = np.random.default_rng(3)
    gts = [rng.integers(0, 3, size=(n, 60)).astype(np.int8), rng.integers(0, 3, size=(n, 50)).astype(np.int8),
           np.zeros((n, 4), np.int8)]
    pg = pack_populations(gts, [2, 2, 2], np.arange(1, n + 1))
    job = make_job(0, 1, [2], True, u=dict(w=1.0, x=0.0, y_list=[("=", 1.0)]),
                   q=dict(w=1.0, quantile=0.95, y_list=[("=", 1.0)]))
    n_u, n_q = _check(pg.layout, torch.from_numpy(pg.packed).cuda(), n, [job])
    assert n_u == 0 and n_q == 0
