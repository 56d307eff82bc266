"""The window and quantile kernels at every size where they switch code paths, bit for bit
against numpy and the oracle.

K4 ``k_window_stats`` (window_kernels.cu) takes a batched fast path for windows of at most
``kFastTiles = 64`` tiles with at most ``kFastN = 32`` U- and Q-flagged sites and
``window_generic`` otherwise, which ranks up to 32 values by all-pairs comparison, radix-selects
up to ``kBufCap = 256`` buffered values and above that selects from the global masks; its second
walk takes the masks of the first ``kMaskCache = 64`` tiles from shared memory and re-reads the
rest with ``range_mask`` applied again.  N3 ``k_window_patterns`` reproduces numpy's pairwise
summation (eight accumulators below 128 sites, recursion with ``n2`` rounded down to a multiple of
8 above), N4 ``k_window_dd`` sums int64 per-site distances with a 128-site unrolled loop, and N1
``k_column_quantile`` gathers the selected bin into shared memory once it holds at most
``kQCap = 4096`` keys and re-reads the column when the successor of the k-th key is not among them.

Every case builds its data so that the side of the threshold it lands on is known, and the CPU
tests at the end check that the sweeps reach both sides and that a plausible wrong summation order
or lerp would be caught."""

from __future__ import annotations

import numpy as np
import pytest

import sai_oracle as orc


@pytest.fixture(scope="module")
def engine():
    from sai_b200.scoring import HostEngine

    e = HostEngine(0)
    yield e
    e.close()


def _same(a: float, b: float) -> bool:
    """Bit-identical, any NaN equal to any NaN."""
    a, b = float(a), float(b)
    return (a != a and b != b) or a.hex() == b.hex()


# =====================================================================================================
# K4: U, Q and candidates with a known number of flagged sites per window
# =====================================================================================================
K4_COUNTS = (0, 1, 31, 32, 33, 255, 256, 257, 1000)  # around kFastN = 32 and kBufCap = 256
K4_FAST_TILES = 64  # kFastTiles == kMaskCache
K4_U = dict(w=0.5, x=0.0, y_list=[("=", 1.0)])
K4_Q = dict(w=0.5, y_list=[("=", 1.0)])
# (want U, want Q, quantile): U + Q at four quantiles, a U-only job and a Q-only job
K4_JOBS = [(True, True, 0.0), (True, True, 0.5), (True, True, 0.95), (True, True, 1.0), (True, False, None),
           (False, True, 0.5)]
N_TGT = 10  # diploid target individuals: frequencies k / 20, many ties


def _k4_jobs():
    from sai_b200.scoring import make_job

    return [make_job(0, 1, [2], True, u=K4_U if wu else None, q=dict(K4_Q, quantile=qq) if wq else None)
            for wu, wq, qq in K4_JOBS]


def _k4_matrices(derived: np.ndarray, k_tgt: np.ndarray) -> list:
    """ref all ancestral (frequency 0 < w), the one source individual derived exactly at ``derived``
    (frequency 1 == y), the target carrying ``k_tgt`` derived alleles (frequency k / 20).  So a site
    is Q-flagged iff it is derived, and U-flagged iff it is derived and k > 0 (x = 0)."""
    n = derived.size
    ref = np.zeros((n, 4), np.int8)
    tgt = np.clip(k_tgt[:, None] - 2 * np.arange(N_TGT)[None, :], 0, 2).astype(np.int8)
    src = np.where(derived, 2, 0).astype(np.int8)[:, None]
    return [ref, tgt, src]


def _k4_genome(seed: int = 11):
    """Regions of known flag density: dense (62 %), a gap without flags, sparse (one flag per 2100
    sites: a window of more than 64 tiles with at most 32 flags), medium (10 %).  The site count is a
    multiple of 32 so that a second copy starts on a tile boundary."""
    rng = np.random.default_rng(seed)
    sparse = np.zeros(40 * 2100, bool)
    sparse[np.arange(40) * 2100 + rng.integers(0, 2000, size=40)] = True
    parts = [("dense", rng.random(6000) < 0.62), ("gap", np.zeros(4000, bool)), ("sparse", sparse),
             ("medium", rng.random(24000) < 0.1)]
    n = sum(p.size for _, p in parts)
    parts.append(("tail", np.zeros((-n) % 32 + 64, bool)))
    regions, at = {}, 0
    for name, p in parts:
        regions[name] = (at, at + p.size)
        at += p.size
    derived = np.concatenate([p for _, p in parts])
    k = rng.integers(0, 21, size=derived.size)
    k[derived & (rng.random(derived.size) < 0.1)] = 0  # derived in the source, absent from the target: Q only
    return derived, k, regions


def _tiles(lo: int, hi: int) -> int:
    return (hi - 1) // 32 - lo // 32 + 1 if hi > lo else 0


def _k4_site_windows(derived, k, regions):
    """Site ranges [lo, hi): every tile count 0..70 at every start offset lo % 32 (hi % 32 varies
    with them) in the dense and the sparse region, and windows holding exactly each count of
    K4_COUNTS U- or Q-flagged sites, ending right after the last one, right before the next one and
    in between.  Ordered so that fast-path and generic windows alternate, odd in number."""
    n = derived.size
    wins = set()
    for name in ("dense", "sparse"):
        t0 = regions[name][0] // 32 + 1
        for t in range(71):
            for off in range(32):
                T0 = t0 + (5 * t + off) % 23
                lo = 32 * T0 + off
                if t == 0:
                    wins.add((lo, lo))
                    continue
                end = off + (7 + off) % (32 - off) if t == 1 else (off + 7 * t + 3) % 32
                wins.add((lo, 32 * (T0 + t - 1) + end + 1))
    for flags in (derived, derived & (k > 0)):
        idx = np.flatnonzero(flags)
        for a, b in regions.values():
            for lo in (a, a + 17, (a + b) // 2):
                j = int(np.searchsorted(idx, lo))
                for c in K4_COUNTS:
                    if j + c > idx.size:
                        continue
                    hi_min = int(idx[j + c - 1]) + 1 if c else lo + 1
                    hi_max = int(idx[j + c]) if j + c < idx.size else n
                    if hi_max < hi_min:
                        continue
                    for hi in (hi_min, (hi_min + hi_max) // 2, hi_max):
                        wins.add((lo, hi))
    cu = np.concatenate([[0], np.cumsum(derived & (k > 0))])
    cq = np.concatenate([[0], np.cumsum(derived)])
    fast, slow = [], []
    for lo, hi in sorted(wins):
        f = _tiles(lo, hi) <= K4_FAST_TILES and cu[hi] - cu[lo] <= 32 and cq[hi] - cq[lo] <= 32
        (fast if f else slow).append((lo, hi))
    out = []
    while fast or slow:
        for lst in (fast, slow):
            if lst:
                out.append(lst.pop())
    if len(out) % 2 == 0:
        out.pop()
    return np.array(out, dtype=np.int64)


def _k4_case():
    derived, k, regions = _k4_genome()
    pos = np.arange(1, derived.size + 1, dtype=np.int32)  # window [lo + 1, hi] holds the sites lo..hi-1
    sw = _k4_site_windows(derived, k, regions)
    return dict(derived=derived, k=k, pos=pos, mats=_k4_matrices(derived, k), ws=sw[:, 0] + 1, we=sw[:, 1],
                regions=regions)


def _k4_expected(pos, derived, k, ws, we):
    """Per window: N(Variants), and per job U, Q, candidate positions -- from the construction:
    U is a count, Q is np.quantile (linear) of the flagged target frequencies, candidates are the
    positions in site order."""
    lo = np.searchsorted(pos, ws, side="left")
    hi = np.maximum(lo, np.searchsorted(pos, we, side="right"))
    tf = k / (2.0 * N_TGT)
    uidx, qidx = np.flatnonzero(derived & (k > 0)), np.flatnonzero(derived)
    ua, ub = np.searchsorted(uidx, lo), np.searchsorted(uidx, hi)
    qa, qb = np.searchsorted(qidx, lo), np.searchsorted(qidx, hi)
    qs = sorted({qq for _, wq, qq in K4_JOBS if wq})
    J, W = len(K4_JOBS), ws.size
    e = dict(nsnps=(hi - lo).astype(np.int64), u=np.zeros((J, W), np.int64), q=np.full((J, W), np.nan),
             u_pos=[[None] * W for _ in range(J)], q_pos=[[None] * W for _ in range(J)], lo=lo, hi=hi,
             n_u=ub - ua, n_q=qb - qa)
    empty = np.zeros(0, np.int32)
    for i in range(W):
        up = pos[uidx[ua[i] : ub[i]]]
        sites = qidx[qa[i] : qb[i]]
        vals = tf[sites]
        thr = {qq: float(np.quantile(vals, qq)) for qq in qs} if vals.size else {}
        for j, (wu, wq, qq) in enumerate(K4_JOBS):
            e["u"][j, i] = up.size if wu else 0
            e["u_pos"][j][i] = up if wu else empty
            if wq and vals.size:
                e["q"][j, i] = thr[qq]
                e["q_pos"][j][i] = pos[sites[vals >= thr[qq]]]
            else:
                e["q_pos"][j][i] = empty
    return e


def _k4_oracle_check(mats, pos, exp, ws, we, picks):
    """The construction agrees with orc.u_statistic / orc.q_statistic on the picked windows."""
    m64 = [m.astype(np.int64) for m in mats]
    for i in picks:
        keep = (pos >= ws[i]) & (pos <= we[i])
        assert keep.sum() == exp["nsnps"][i]
        if not keep.any():
            continue
        sub = [m[keep] for m in m64]
        for j, (wu, wq, qq) in enumerate(K4_JOBS):
            if wu:
                eu = orc.u_statistic(sub[0], sub[1], [sub[2]], 2, 2, [2], pos=pos[keep], anc_allele_available=True, **K4_U)
                assert eu["value"] == exp["u"][j, i] and np.array_equal(eu["cdd_pos"], exp["u_pos"][j][i]), (i, j)
            if wq:
                eq = orc.q_statistic(sub[0], sub[1], [sub[2]], 2, 2, [2], pos=pos[keep], anc_allele_available=True,
                                     quantile=qq, **K4_Q)
                assert _same(eq["value"], exp["q"][j, i]), (i, j)
                assert np.array_equal(np.asarray(eq["cdd_pos"], np.int64), exp["q_pos"][j][i]), (i, j)


def _k4_compare(res, exp, what):
    W = exp["nsnps"].size
    for j in range(len(K4_JOBS)):
        assert np.array_equal(res.nsnps[j], exp["nsnps"]), (what, j)
        assert np.array_equal(res.u[j], exp["u"][j]), (what, j)
        qn = np.isnan(exp["q"][j])
        assert np.array_equal(np.isnan(res.q[j]), qn), (what, j)
        assert np.array_equal(res.q[j][~qn].view(np.int64), exp["q"][j][~qn].view(np.int64)), (what, j)
        assert res.totals[j, 0] == exp["u"][j].sum() and res.totals[j, 1] == sum(p.size for p in exp["q_pos"][j])
        for i in range(W):
            assert np.array_equal(res.u_positions(j, i), exp["u_pos"][j][i]), (what, j, i)
            assert np.array_equal(res.q_positions(j, i), exp["q_pos"][j][i]), (what, j, i)


def _k4_device(pg, ws, we, cap_u, cap_q, first=None, last=None):
    """K1 flags + K4 through DeviceScorer with candidate buffers of cap_u / cap_q entries per job."""
    import torch

    from sai_b200.scoring import DeviceScorer

    dev = torch.device("cuda")
    d_packed, d_pos = torch.from_numpy(pg.packed).to(dev), torch.from_numpy(pg.pos).to(dev)
    d_ws, d_we = torch.from_numpy(ws).to(dev), torch.from_numpy(we).to(dev)
    jobs = _k4_jobs()
    sc = DeviceScorer(pg.layout, pg.n_sites, ws.size, len(jobs), cap_u=cap_u, cap_q=cap_q)
    sc.site_flags(d_packed, jobs)
    if first is None:
        sc.window_stats(d_pos, d_ws, d_we, jobs)
    else:
        sc.window_stats(d_pos, d_ws, d_we, jobs, torch.from_numpy(first).to(dev), torch.from_numpy(last).to(dev))
    return sc.results(), sc


@pytest.mark.gpu
def test_k4_fast_and_generic_paths_at_every_threshold(engine):
    """kFastTiles / kMaskCache = 64 tiles, kFastN = 32 and kBufCap = 256 flagged sites, every
    lo % 32 and hi % 32, U-only and Q-only jobs, quantiles 0, 0.5, 0.95, 1; an odd number of windows
    (not a multiple of the experiments build's batch of 2 or 4) with fast and generic windows
    alternating.  The same windows then run over two tile-aligned pieces (the genome twice side by
    side, window i searching piece i % 2, ``sai_window_stats_pieces``).  Candidate buffers are
    sized to exactly the need (no retry) and, for the pieces, to the need - 1 (DeviceScorer.results
    grows them and re-runs the window kernel)."""
    from sai_b200.encode import pack_populations

    c = _k4_case()
    ws, we, pos = c["ws"], c["we"], c["pos"]
    exp = _k4_expected(pos, c["derived"], c["k"], ws, we)
    _k4_oracle_check(c["mats"], pos, exp, ws, we, np.linspace(0, ws.size - 1, 40).astype(int))
    need_u = int(exp["u"].sum(axis=1).max())
    need_q = max(sum(p.size for p in exp["q_pos"][j]) for j in range(len(K4_JOBS)))

    pg = pack_populations(c["mats"], [2, 2, 2], pos)
    res, sc = _k4_device(pg, ws, we, need_u, need_q)
    assert (sc.cap_u, sc.cap_q) == (need_u, need_q)  # exactly enough: no second launch
    _k4_compare(res, exp, "one piece")

    n = pos.size
    assert n % 32 == 0
    pg2 = pack_populations([np.concatenate([m, m]) for m in c["mats"]], [2, 2, 2], np.concatenate([pos, pos]))
    first = np.where(np.arange(ws.size) % 2 == 1, n, 0).astype(np.int32)
    res2, sc2 = _k4_device(pg2, ws, we, need_u - 1, need_q - 1, first, first + n)
    assert (sc2.cap_u, sc2.cap_q) == (need_u, need_q)  # grown by the retry
    _k4_compare(res2, exp, "two pieces")

    # the host-buffer engine runs the same kernel with its own capacity handling
    _k4_compare(engine.score(pg, list(zip(ws.tolist(), we.tolist())), _k4_jobs()), exp, "HostEngine")


@pytest.mark.gpu
def test_k4_duplicate_positions_up_to_int32_max(engine):
    """Split multi-allelic records (one position on up to three consecutive sites) near and at
    2^31 - 1, windows starting and ending on duplicated positions, ending at 2^31 - 1 and beyond it;
    fast and generic windows of 1..100 tiles."""
    from sai_b200.encode import pack_populations

    rng = np.random.default_rng(23)
    top = 2**31 - 1
    uniq = np.append(np.sort(rng.choice(np.arange(top - 300_000, top), size=3999, replace=False)), top)
    pos = np.repeat(uniq, rng.choice([1, 1, 1, 2, 3], size=uniq.size)).astype(np.int32)
    n = pos.size
    derived = rng.random(n) < np.where(np.arange(n) < n // 2, 0.012, 0.5)  # sparse half, dense half
    k = rng.integers(0, 21, size=n)
    mats = _k4_matrices(derived, k)
    dup = np.flatnonzero(np.diff(pos) == 0)
    wins = []
    for lo in list(rng.choice(dup, size=40)) + list(rng.integers(0, n, size=40)):
        for length in (1, 31, 33, 32 * 64 - 5, 32 * 64 + 40, 32 * 100):
            hi = min(n, int(lo) + length)
            wins.append((int(pos[lo]), int(pos[hi - 1])))
    wins += [(int(pos[-300]), top), (int(pos[-5]), 2**40), (top, top), (top, 2**40), (top - 10, top - 1),
             (int(pos[dup[-1]]), int(pos[dup[-1]])), (1, 2**40), (2**33, 2**34)]
    ws = np.array([w[0] for w in wins], np.int64)
    we = np.array([w[1] for w in wins], np.int64)
    exp = _k4_expected(pos, derived, k, ws, we)
    tiles = np.array([_tiles(a, b) for a, b in zip(exp["lo"], exp["hi"])])
    assert (tiles > K4_FAST_TILES).any() and ((tiles <= K4_FAST_TILES) & (exp["n_q"] <= 32) & (exp["n_q"] > 0)).any()
    assert (exp["n_q"] > 256).any() and (exp["hi"] == n).any()
    _k4_oracle_check(mats, pos, exp, ws, we, range(0, ws.size, 8))
    pg = pack_populations(mats, [2, 2, 2], pos)
    res, _ = _k4_device(pg, ws, we, None, None)
    _k4_compare(res, exp, "device scorer")
    _k4_compare(engine.score(pg, wins, _k4_jobs()), exp, "HostEngine")


# =====================================================================================================
# N3: window sums in numpy's pairwise order
# =====================================================================================================
N3_PLOIDY = [2, 2, 2, 2]  # ref, tgt, src, outgroup
N3_SIZES = (24, 20, 16, 8)


def _n3_lengths(max_pow: int) -> list:
    """Every n in 0..600 (L < 8, the 4-deep unrolled loop ``i + 24 < body`` with its 8-step and
    L % 8 tails, the leaf size 128 and the first recursion levels) and 2^k - 8, -1, +0, +1, +8."""
    ns = set(range(601))
    for k in range(3, max_pow + 1):
        ns |= {2**k - 8, 2**k - 1, 2**k, 2**k + 1, 2**k + 8}
    return sorted(ns)


def _n3_genome(n_sites: int, n_nan: int, seed: int = 5):
    """Per-site derived-allele probabilities spread over three decades (products from ~1e-6 to 1,
    so the summation order changes the last bits); the last ``n_nan`` sites of the tail hold sites
    where nobody in the target is called (frequency NaN)."""
    rng = np.random.default_rng(seed)
    p = 10.0 ** rng.uniform(-3, 0, size=n_sites)
    mats = [rng.binomial(pl, p[:, None], size=(n_sites, m)).astype(np.int8) for pl, m in zip(N3_PLOIDY, N3_SIZES)]
    for m in mats:
        m[rng.random(m.shape) < 0.01] = -1
    if n_nan:
        mats[1][n_sites - 64 + rng.choice(64, size=n_nan, replace=False)] = -1
    return mats


def _n3_freqs(mats):
    return [orc.site_frequency(m.astype(np.int64), pl) for m, pl in zip(mats, N3_PLOIDY)]


def _n3_expected(freqs, lo, hi) -> list:
    """The seven sums of sites [lo, hi): five plain patterns from orc.pattern_sum, abba_d / baba_d with
    dnr = max(tgt, src) as orc.four_pop_statistics forms them."""
    fr, ft, fs, fo = (f[lo:hi] for f in freqs)
    four = (fr, ft, fs, fo)
    dnr = np.maximum(ft, fs)
    out = [orc.pattern_sum(four, p) for p in ("abba", "baba", "baaa", "abaa", "bbaa")]
    out += [orc.pattern_sum((fr, dnr, dnr, fo), "abba"), orc.pattern_sum((fr, dnr, dnr, fo), "baba")]
    return out


def _n3_windows(lengths, n_main, rng):
    starts = [int(rng.integers(0, n_main - n + 1)) for n in lengths]
    return [(s, s + n) for s, n in zip(starts, lengths)]


@pytest.mark.gpu
def test_n3_pattern_sums_pairwise_order():
    """Every window length 0..600, 2^k +- {0, 1, 8} up to 2^17 and one window of ~10^6 sites (n2
    rounded down to a multiple of 8 at every recursion level), plus windows over sites with
    frequency NaN: all seven sums bit-identical to np.sum of the oracle's per-site products."""
    import torch

    from sai_b200.encode import pack_populations
    from sai_b200.scoring import DeviceScorer

    rng = np.random.default_rng(8)
    n_main = 1_000_003
    mats = _n3_genome(n_main + 1000, n_nan=3)
    n = mats[0].shape[0]
    freqs = _n3_freqs(mats)
    assert not np.isnan(freqs[1][:n_main]).any() and np.isnan(freqs[1][n_main:]).sum() == 3
    wins = _n3_windows(_n3_lengths(17), n_main, rng) + [(0, n_main), (7, n_main)]
    wins += [(n - 64 - a, n - b) for a, b in ((0, 0), (5, 0), (10, 40), (30, 60), (200, 0))]
    pos = np.arange(1, n + 1, dtype=np.int32)
    pg = pack_populations(mats, N3_PLOIDY, pos)
    dev = torch.device("cuda")
    d_packed, d_pos = torch.from_numpy(pg.packed).to(dev), torch.from_numpy(pos).to(dev)
    d_ws = torch.tensor([lo + 1 for lo, _ in wins], dtype=torch.int64, device=dev)
    d_we = torch.tensor([hi for _, hi in wins], dtype=torch.int64, device=dev)
    sc = DeviceScorer(pg.layout, n, len(wins), 1)
    sc.site_counts(d_packed)
    got = sc.pattern_sums(d_pos, d_ws, d_we, 0, 1, 3, [2]).cpu().numpy()[0]
    n_nan = 0
    for i, (lo, hi) in enumerate(wins):
        want = _n3_expected(freqs, lo, hi)
        for t in range(7):
            assert _same(got[i, t], want[t]), (hi - lo, t, float(got[i, t]).hex(), float(want[t]).hex())
        n_nan += np.isnan(want[0])
    assert 0 < n_nan < 10


# =====================================================================================================
# N4: int64 window sums of the per-site DD distances
# =====================================================================================================
def _dd_device(pg, ws, we, src_pops=(2,)):
    import torch

    from sai_b200.scoring import DeviceScorer

    dev = torch.device("cuda")
    d_packed, d_pos = torch.from_numpy(pg.packed).to(dev), torch.from_numpy(pg.pos).to(dev)
    d_ws, d_we = torch.from_numpy(ws).to(dev), torch.from_numpy(we).to(dev)
    d_neg = [torch.from_numpy(a).to(dev) for a in (pg.neg_site, pg.neg_ind, pg.neg_val)]
    sc = DeviceScorer(pg.layout, pg.n_sites, ws.size, 1)
    hist, _ = sc.site_hist(d_packed, [0, 1])
    ref_sum, tgt_sum, err = sc.dd_sums(d_packed, d_pos, d_ws, d_we, hist, 0, 1, list(src_pops), pg.neg_off, *d_neg)
    assert int(err.item()) == 0
    return ref_sum.cpu().numpy(), tgt_sum.cpu().numpy()


@pytest.mark.gpu
def test_n4_window_sums_around_the_unrolled_loop():
    """Window lengths 0..300 (the ``s + 96 < hi`` loop of 128 sites per trip and its 32-site tail) at
    start offsets 0, 1, 31, 33 and 517, missing calls included: equal to orc.cityblock_sums."""
    from sai_b200.encode import pack_populations

    rng = np.random.default_rng(41)
    n = 1000
    f = rng.beta(0.5, 1.0, size=n)
    mats = [rng.binomial(2, f[:, None], size=(n, m)).astype(np.int8) for m in (30, 20, 3)]
    for m in mats:
        hole = rng.random(m.shape) < 0.03
        m[hole] = -rng.integers(1, 3, size=int(hole.sum()))
    pos = np.arange(1, n + 1, dtype=np.int32)
    pg = pack_populations(mats, [2, 2, 2], pos, keep_negatives=True)
    wins = [(s, s + L) for s in (0, 1, 31, 33, 517) for L in range(301) if s + L <= n]
    ws = np.array([lo + 1 for lo, _ in wins], np.int64)
    we = np.array([hi for _, hi in wins], np.int64)
    ref_sum, tgt_sum = _dd_device(pg, ws, we)
    m64 = [m.astype(np.int64) for m in mats]
    for i, (lo, hi) in enumerate(wins):
        src = m64[2][lo:hi]
        assert np.array_equal(ref_sum[0, i], orc.cityblock_sums(src, m64[0][lo:hi]).sum(axis=1)), (lo, hi)
        assert np.array_equal(tgt_sum[0, i], orc.cityblock_sums(src, m64[1][lo:hi]).sum(axis=1)), (lo, hi)


@pytest.mark.gpu
def test_n4_window_sum_above_int32():
    """8000 ref individuals with per-individual values of 118..127 against sources near 0 over 2400
    sites: per-window distance sums above 2^31 need the int64 accumulation; DD from them (the host's
    float64 step) equals orc.dd_statistic bit for bit."""
    from sai_b200.encode import pack_populations
    from sai_b200.scoring import dd_values

    rng = np.random.default_rng(43)
    n = 2400
    ref = rng.integers(118, 128, size=(n, 8000)).astype(np.int8)
    tgt = rng.integers(0, 3, size=(n, 40)).astype(np.int8)
    src = rng.integers(0, 3, size=(n, 2)).astype(np.int8)
    tgt[rng.random(tgt.shape) < 0.02] = -1
    src[rng.random(src.shape) < 0.02] = -2
    mats = [ref, tgt, src]
    pos = np.arange(1, n + 1, dtype=np.int32)
    pg = pack_populations(mats, [2, 2, 2], pos, keep_negatives=True)
    wins = [(0, n), (0, 1500), (700, n)]
    ws = np.array([lo + 1 for lo, _ in wins], np.int64)
    we = np.array([hi for _, hi in wins], np.int64)
    ref_sum, tgt_sum = _dd_device(pg, ws, we)
    got = dd_values(ref_sum, tgt_sum, 8000, 40, [2])
    m64 = [m.astype(np.int64) for m in mats]
    for i, (lo, hi) in enumerate(wins):
        want = orc.cityblock_sums(m64[2][lo:hi], m64[0][lo:hi]).sum(axis=1)
        assert np.array_equal(ref_sum[0, i], want), i
        assert np.array_equal(tgt_sum[0, i], orc.cityblock_sums(m64[2][lo:hi], m64[1][lo:hi]).sum(axis=1)), i
        exp = orc.dd_statistic(m64[0][lo:hi], m64[1][lo:hi], [m64[2][lo:hi]])
        assert _same(got[0][i], exp[0]), i
    assert ref_sum[0, 0].min() > 2**31


# =====================================================================================================
# N1: the outlier threshold (radix select of a column, numpy's lerp)
# =====================================================================================================
ULP1 = np.nextafter(1.0, 2.0) - 1.0


def _n1_columns() -> dict:
    rng = np.random.default_rng(17)

    def mix(*parts):
        v = np.concatenate(parts)
        return v[rng.permutation(v.size)]

    one_two = lambda k: 1.0 + rng.random(k)  # [1, 2): one top-byte bin of the ordered keys
    cols = {
        # the bin the k-th key falls in holds exactly 4096 (gathered at pass 0) / 4097 keys (a later pass)
        "bin_4096": mix(one_two(4096), 2.0 + 2.0 * rng.random(3000), -rng.random(3000)),
        "bin_4097": mix(one_two(4097), 2.0 + 2.0 * rng.random(3000), -rng.random(3000)),
        "n_4096": rng.normal(size=4096),
        "n_100": rng.normal(size=100),
        "n_5": rng.normal(size=5),
        "n_101": rng.normal(size=101),
        # never gathered: 10 000 ties, and 6000 keys that share their top 7 bytes
        "ties_10000": mix(np.full(10_000, 0.5), np.full(5, 0.1), np.full(5, 0.9)),
        "ulp_256": mix(1.0 + np.arange(256) * ULP1),
        "ulp_6000": mix(1.0 + (np.arange(6000) % 256) * ULP1),
        # the k-th key can be the largest of its gathered bin: 1.0 - 2.0 straddles a top-byte boundary,
        # 1.0625 a second-byte boundary of 5000 keys in [1, 2)
        "straddle_2": mix(one_two(3000), 2.0 + 2.0 * rng.random(3000)),
        "straddle_1.0625": mix(one_two(5000), 2.0 + rng.random(100)),
        "signed_zeros": mix(np.full(30, -0.0), np.zeros(30), -rng.random(20), rng.random(20)),
        "subnormals": mix(np.array([5e-324, -5e-324, 1e-310, -1e-310, 2.2250738585072014e-308, 0.0, -0.0, 1e-320]),
                          rng.normal(size=8) * 1e-300),
        "inf": mix(np.array([-np.inf, -np.inf, np.inf, np.inf]), rng.normal(size=12)),
        "inf_max": mix(np.array([np.inf]), rng.normal(size=50)),
        "neg_inf_min": mix(np.array([-np.inf]), rng.normal(size=50)),
    }
    return cols


def _n1_quantiles(cols) -> list:
    """0, 1, values with g == 0 and g == 0.5 exactly, q just below 1 (k = n - 2: (n - 1) q < n - 1 for
    every double q < 1, so vi >= n - 1 only at q = 1), and the q that puts k on the largest key of
    a bin in the straddle columns."""
    qs = {0.0, 0.25, 0.375, 0.5, 0.75, 0.95, 0.99, 1.0 - 2.0**-53, 1.0}
    for name, border in (("straddle_2", 2.0), ("straddle_1.0625", 1.0625), ("bin_4096", 2.0)):
        v = cols[name]
        k = int((v < border).sum()) - 1
        qs.add((k + 0.25) / (v.size - 1))
        qs.add((k + 0.75) / (v.size - 1))
    n = cols["ties_10000"].size
    qs.add((n - 6 + 0.5) / (n - 1))  # k = the last of the ties: successor outside, never gathered
    return sorted(qs)


def _ordered_keys(v: np.ndarray) -> np.ndarray:
    b = (np.asarray(v, np.float64) + 0.0).view(np.uint64)
    return np.where(b >> np.uint64(63) == 1, ~b, b | np.uint64(1 << 63))


def _n1_path(v: np.ndarray, q: float):
    """(pass at which the k-th key's bin is gathered or None, whether the successor is re-read from
    the column), as k_column_quantile decides them; None when no select runs."""
    v = v[~np.isnan(v)]
    keys = np.sort(_ordered_keys(v))
    n = keys.size
    if n == 0 or keys[0] == keys[-1]:
        return None
    vi = np.float64(n - 1) * np.float64(q)
    if vi >= n - 1:
        return None
    k = int(np.floor(vi))
    ka = keys[k]
    gathered = None
    for p in range(7):
        sh = np.uint64(56 - 8 * p)
        if ((keys >> sh) == (ka >> sh)).sum() <= 4096:
            gathered = p
            break
    reread = False
    if k + 1 >= int((keys <= ka).sum()):
        if gathered is None:
            reread = True
        else:
            sh = np.uint64(56 - 8 * gathered)
            reread = not ((keys > ka) & ((keys >> sh) == (ka >> sh))).any()
    return gathered, reread


def _n1_check(got, v, q, what) -> int:
    """got == the oracle's threshold bit for bit; returns 1 if they differ only in the sign of zero."""
    want = orc.outlier_threshold(v, q)
    if want is None:
        assert np.isnan(got), (what, q, got)
        return 0
    if want == 0.0 and got == 0.0 and _same(-want, got):
        # -0.0 vs +0.0: the kernel reads -0.0 as +0.0, np.quantile may hand back either zero of a tie.
        # The sign cannot reach `sai outlier`'s output: the threshold is only compared (v >= thr, or
        # v > thr for U), where -0.0 == +0.0 selects the same rows, and it is never written.
        assert got == want
        return 1
    assert _same(got, want), (what, q, float(got).hex(), float(want).hex())
    return 0


@pytest.mark.gpu
@pytest.mark.parametrize("n_chunks", [1, 3, 8])
def test_n1_column_quantiles_at_select_paths(n_chunks):
    """Every column of _n1_columns at every q of _n1_quantiles through
    torch.ops.sai_b200.column_quantiles, the columns cut into n_chunks pieces padded with NaN."""
    import torch

    import sai_b200.ops  # noqa: F401  (registers torch.ops.sai_b200)

    cols = _n1_columns()
    names = list(cols)
    L = -(-max(v.size for v in cols.values()) // n_chunks) + 5
    buf = np.full((n_chunks, len(names), L), np.nan)
    for c, name in enumerate(names):
        v = cols[name]
        per = -(-v.size // n_chunks)
        for r in range(n_chunks):
            part = v[r * per : (r + 1) * per]
            buf[r, c, : part.size] = part
    d = torch.from_numpy(buf).cuda()
    out = torch.empty((len(names), 4), dtype=torch.float64, device="cuda")
    signs = 0
    for q in _n1_quantiles(cols):
        torch.ops.sai_b200.column_quantiles(d, q, out)
        o = out.cpu().numpy()
        for c, name in enumerate(names):
            signs += _n1_check(o[c, 0], cols[name], q, name)
            assert o[c, 1] == cols[name].size, name
    assert signs < len(names) * 4


@pytest.mark.gpu
@pytest.mark.parametrize("n_chunks", [1, 3, 8])
def test_n1_chunk_lengths_around_the_load_loop(n_chunks):
    """Piece lengths 32768 k - 1, 32768 k, 32768 k + 1 (the kInFlight = 4 loads of 8192-element
    strides and their tail) with NaN padding at the end of some pieces; the column's extremes sit at
    the last index of the last piece, so a skipped tail changes the result."""
    import torch

    import sai_b200.ops  # noqa: F401

    rng = np.random.default_rng(29)
    for L in (32767, 32768, 32769, 65535, 65537):
        buf = rng.normal(size=(n_chunks, 2, L))
        buf[:, 1] = np.round(buf[:, 1] * 4)  # ties
        for r in range(0, n_chunks, 2):
            buf[r, :, L - int(rng.integers(1, 50)) :] = np.nan
        buf[-1, 0, -1], buf[-1, 1, -1] = 50.0, -50.0
        d = torch.from_numpy(buf).cuda()
        out = torch.empty((2, 4), dtype=torch.float64, device="cuda")
        for q in (0.0, 0.5, 0.95, 1.0, 1.0 / (n_chunks * L)):
            torch.ops.sai_b200.column_quantiles(d, q, out)
            o = out.cpu().numpy()
            for c in range(2):
                v = buf[:, c].ravel()
                _n1_check(o[c, 0], v, q, (L, c))
                assert o[c, 1] == np.count_nonzero(~np.isnan(v)) and o[c, 2] == np.nanmin(v) and o[c, 3] == np.nanmax(v)


# =====================================================================================================
# CPU: the sweeps reach both sides of every threshold, and would catch a wrong order or lerp
# =====================================================================================================
def test_k4_construction_matches_oracle_and_covers_thresholds():
    """Every count of K4_COUNTS occurs as a U and as a Q count in windows of at most and of more than
    64 tiles; every lo % 32 and hi % 32 occurs on both sides; fast and generic windows alternate;
    48 windows agree with orc.u_statistic / orc.q_statistic."""
    c = _k4_case()
    ws, we, pos = c["ws"], c["we"], c["pos"]
    exp = _k4_expected(pos, c["derived"], c["k"], ws, we)
    lo, hi = exp["lo"], exp["hi"]
    tiles = np.array([_tiles(a, b) for a, b in zip(lo, hi)])
    big = tiles > K4_FAST_TILES
    for cnt in K4_COUNTS:
        for side in (False, True):
            assert ((exp["n_q"] == cnt) & (big == side)).any(), ("Q", cnt, side)
            assert ((exp["n_u"] == cnt) & (big == side)).any(), ("U", cnt, side)
    nonempty = hi > lo
    for side in (False, True):
        sel = nonempty & (big == side)
        assert set((lo[sel] % 32).tolist()) == set(range(32)) and set((hi[sel] % 32).tolist()) == set(range(32))
    assert set(tiles.tolist()) >= set(range(71))
    # > 64 tiles with 1..32 flags whose last flag lies beyond the 64 cached tiles: the global-mask branch
    qidx = np.flatnonzero(c["derived"])
    last_flag = np.array([qidx[np.searchsorted(qidx, b) - 1] if n else -1 for b, n in zip(hi, exp["n_q"])])
    assert (big & (exp["n_q"] >= 1) & (exp["n_q"] <= 32) & (last_flag // 32 - lo // 32 >= K4_FAST_TILES)).any()
    fast = (tiles <= K4_FAST_TILES) & (exp["n_u"] <= 32) & (exp["n_q"] <= 32)
    assert ws.size % 2 == 1 and (fast[:-1] != fast[1:]).sum() > 0.4 * ws.size
    assert all(((exp["n_q"] > a) & (exp["n_q"] <= b)).any() for a, b in ((0, 32), (32, 256), (256, 10**6)))
    _k4_oracle_check(c["mats"], pos, exp, ws, we, np.linspace(0, ws.size - 1, 48).astype(int))


def _pairwise_n2_unrounded(a) -> float:
    """orc.pairwise_sum_model with the wrong split n2 = n // 2 (not rounded down to a multiple of 8)."""
    a = [float(x) for x in a]

    def pw(lo, n):
        if n < 8:
            res = 0.0
            for i in range(lo, lo + n):
                res = res + a[i]
            return res
        if n <= 128:
            r = a[lo : lo + 8]
            i = 8
            while i < n - (n % 8):
                for j in range(8):
                    r[j] = r[j] + a[lo + i + j]
                i += 8
            res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]))
            while i < n:
                res = res + a[lo + i]
                i += 1
            return res
        n2 = n // 2
        return pw(lo, n2) + pw(lo + n2, n - n2)

    return pw(0, len(a))


def test_n3_sweep_tells_pairwise_order_from_wrong_ones():
    """On the N3 data and window lengths (up to 2^14 + 8 here), a sequential sum and a pairwise sum
    whose split is not rounded to 8 both differ from np.sum in many windows, while the oracle's
    model of numpy's order agrees in all of them."""
    rng = np.random.default_rng(8)
    mats = _n3_genome(40_000, n_nan=0)
    freqs = _n3_freqs(mats)
    fr, ft, fs, fo = freqs
    prod = (1 - fr) * ft * fs * (1 - fo)  # abba, multiplied in the order of orc.pattern_sum
    lengths = _n3_lengths(14)
    seq_diff = pw_diff = pw_cases = 0
    for lo, hi in _n3_windows(lengths, mats[0].shape[0], rng):
        a = prod[lo:hi]
        want = orc.pattern_sum((fr[lo:hi], ft[lo:hi], fs[lo:hi], fo[lo:hi]), "abba")
        assert _same(orc.pairwise_sum_model(a), want)
        if a.size:
            seq_diff += not _same(np.cumsum(a)[-1], want)
        if a.size > 128 and (a.size // 2) % 8:
            pw_cases += 1
            pw_diff += not _same(_pairwise_n2_unrounded(a), want)
    assert seq_diff > 0.3 * len(lengths), seq_diff
    assert pw_diff > 0.15 * pw_cases and pw_diff > 50, (pw_diff, pw_cases)


def test_n1_columns_reach_every_select_path():
    """The N1 columns and quantiles reach: gather at pass 0, at a later pass, never; the successor
    found among the gathered keys and re-read from the column (after a gather and without one);
    g == 0, g == 0.5 exactly and vi >= n - 1."""
    cols = _n1_columns()
    qs = _n1_quantiles(cols)
    paths = {_n1_path(v, q) for v in cols.values() for q in qs} - {None}
    gathered = {g for g, _ in paths}
    assert 0 in gathered and None in gathered and any(g is not None and g > 0 for g in gathered)
    assert (None, True) in paths and any(g is not None and r for g, r in paths)
    assert any(g is not None and not r for g, r in paths)
    assert _n1_path(cols["bin_4096"], 0.5) == (0, False) and _n1_path(cols["bin_4097"], 0.5)[0] > 0
    assert _n1_path(cols["ulp_6000"], 0.5)[0] is None
    for name in ("straddle_2", "straddle_1.0625", "bin_4096"):
        assert any(_n1_path(cols[name], q)[1] for q in qs if _n1_path(cols[name], q)), name
    gs = {float(np.float64(v.size - 1) * np.float64(q) % 1.0) for v in cols.values() for q in qs}
    assert 0.0 in gs and 0.5 in gs


def test_n1_sweep_tells_lerp_branches_apart():
    """A lerp without numpy's g >= 0.5 branch (always a + (b - a) g) differs from np.quantile on many
    of the N1 cases, so the device comparison would notice a kernel that dropped it."""
    cols = _n1_columns()
    rng = np.random.default_rng(3)
    cols.update({f"normal_{i}": rng.normal(size=int(rng.integers(10, 3000))) for i in range(20)})
    qs = _n1_quantiles(cols) + list(rng.random(40))
    wrong = upper = 0
    for v in cols.values():
        s = np.sort(v[~np.isnan(v)])
        for q in qs:
            want = orc.outlier_threshold(v, q)
            vi = np.float64(s.size - 1) * np.float64(q)
            if want is None or vi >= s.size - 1:
                continue
            k = int(np.floor(vi))
            g = np.float64(vi - k)
            a, b = s[k], s[k + 1]
            with np.errstate(invalid="ignore"):
                alt = float(a + np.float64(np.float64(b - a) * g))
            if g >= 0.5:
                upper += 1
                wrong += not _same(alt, want)
    assert wrong > 20, (wrong, upper)


def test_host_threshold_of_infinite_columns_matches_numpy():
    """The host threshold of `sai outlier` (threshold_from_values) on columns with +-inf: numpy's
    lerp of inf with inf is NaN, at q = 1 too."""
    from sai_b200.outlier import threshold_from_values

    cols = _n1_columns()
    for name in ("inf", "inf_max", "neg_inf_min", "signed_zeros", "subnormals", "n_5"):
        for q in _n1_quantiles(cols):
            got = threshold_from_values(cols[name], q)
            want = orc.outlier_threshold(cols[name], q)
            if want is None:
                assert got is None
            elif want == 0.0:
                assert got == 0.0
            else:
                assert _same(got, want), (name, q, got, want)
