"""The live-tile queue of the staged genotype pass: k_site_scan stores the zero mask words of tiles
where no job's source gate holds and queues the others, k_site_live runs the reference / target
stages over batches of queued tiles.  Inputs are planted so that the set of live tiles is exact;
every case is checked against the read-everything path (``_check``: U / Q mask words bit for bit,
Q values by bit pattern, tiles outside the range untouched)."""

import numpy as np
import pytest

from test_gpu_site_gather import K, _job, _three_pops
from test_gpu_site_gating import _check

pytestmark = pytest.mark.gpu

BATCH = 4  # kGateTiles in sai_b200/csrc/site_kernels.cu (three populations fit 4 tiles per batch)


def _live_tiles(rng, tiles, n_sites, n_src=1, n_ref=1, whole=()):
    """Source-live sites on each tile of `tiles` (n_src random lanes, the first n_ref of them also
    reference-live; K + 3 / K + 1 on the tiles of `whole`, which are read whole), clipped to
    n_sites."""
    src, ref = set(), set()
    for t in tiles:
        ns, nr = (K + 3, K + 1) if t in whole else (n_src, n_ref)
        lanes = rng.choice(32, size=ns, replace=False)
        src.update(32 * t + int(s) for s in lanes)
        ref.update(32 * t + int(s) for s in lanes[:nr])
    return {s for s in src if s < n_sites}, {s for s in ref if s < n_sites}


def _case(seed, n_tiles, tiles, ragged=0, **kw):
    rng = np.random.default_rng(seed)
    n_sites = 32 * n_tiles - ragged
    src, ref = _live_tiles(rng, tiles, n_sites, **kw)
    lay, d_packed = _three_pops(rng, n_sites, src, ref)
    return lay, d_packed, n_sites, src, ref


def _jobs():
    return [_job(0, 1, [2]), _job(0, 1, [2], anc=False)]


def test_no_tile_and_every_tile_live():
    lay, d_packed, n_sites, src, ref = _case(1, 70, [])
    assert _check(lay, d_packed, n_sites, _jobs()) == (0, 0)
    lay, d_packed, n_sites, src, ref = _case(2, 70, range(70), n_src=2, n_ref=1)
    n_u, n_q = _check(lay, d_packed, n_sites, _jobs())
    assert n_q == 2 * len(ref)


@pytest.mark.parametrize("n_live", [BATCH - 1, BATCH, BATCH + 1, 2 * BATCH + 1])
def test_ragged_last_batch(n_live):
    rng = np.random.default_rng(n_live)
    n_tiles = 200
    tiles = sorted(rng.choice(n_tiles, size=n_live, replace=False).tolist())
    lay, d_packed, n_sites, src, ref = _case(10 + n_live, n_tiles, tiles, n_src=2, n_ref=1)
    n_u, n_q = _check(lay, d_packed, n_sites, _jobs())
    assert n_q == 2 * len(ref)


def test_live_at_subrange_ends():
    """Live tiles only at the first and last tile of sub-ranges that start past tile 0, a 1-tile
    range, and the ragged last tile of the chromosome."""
    rng = np.random.default_rng(3)
    n_tiles = 150
    n_sites = 32 * n_tiles - 13
    ranges = [(5, 40), (45, 1), (70, 33), (n_tiles - 20, 20)]
    tiles = sorted({t for t0, nt in ranges for t in (t0, t0 + nt - 1)} - {n_tiles - 1})
    src, ref = _live_tiles(rng, tiles, n_sites, n_src=3, n_ref=2)
    src |= {n_sites - 5, n_sites - 1}
    ref |= {n_sites - 1}
    lay, d_packed = _three_pops(rng, n_sites, src, ref)
    for tile0, nt in ranges:
        n_u, n_q = _check(lay, d_packed, n_sites, _jobs(), tile0=tile0, n_tiles=nt)
        assert n_q == 2 * len({s for s in ref if tile0 <= s // 32 < tile0 + nt})


def test_distant_tiles_mixed_with_whole_reads():
    """Isolated live tiles far apart (a batch spans distant tiles) and, among them, tiles with more
    than K live sites, read whole inside the same batches."""
    n_tiles = 3000
    tiles = list(range(7, n_tiles, 211))
    whole = set(tiles[1::3])
    lay, d_packed, n_sites, src, ref = _case(4, n_tiles, tiles, n_src=1, n_ref=1, whole=whole)
    n_u, n_q = _check(lay, d_packed, n_sites, _jobs())
    assert n_q == 2 * len(ref)


def test_many_warps_race_on_the_queue():
    """~1e5 tiles, ~20 % of them live at random: thousands of warps append to and claim from the
    queue.  Two runs store identical outputs."""
    import torch

    from sai_b200.scoring import DeviceScorer

    rng = np.random.default_rng(5)
    n_tiles = 100_000
    tiles = np.flatnonzero(rng.random(n_tiles) < 0.2).tolist()
    whole = set(tiles[::50])
    src, ref = _live_tiles(rng, tiles, 32 * n_tiles, n_src=2, n_ref=1, whole=whole)
    lay, d_packed = _three_pops(rng, 32 * n_tiles, src, ref, n=(40, 33, 3))
    jobs = _jobs()
    n_u, n_q = _check(lay, d_packed, 32 * n_tiles, jobs)
    assert n_q == 2 * len(ref)
    runs = []
    for _ in range(2):
        sc = DeviceScorer(lay, 32 * n_tiles, 1, len(jobs))
        sc.qval.zero_()
        sc.site_flags(d_packed, jobs)
        torch.cuda.synchronize()
        runs.append([sc.mask_u.cpu().numpy(), sc.mask_q.cpu().numpy(), sc.qval.cpu().numpy().view(np.int64)])
    for a, b in zip(*runs):
        assert np.array_equal(a, b)
