"""K4's span path, bit for bit against numpy and the oracle.

``k_window_spans`` (window_kernels.cu) takes a span of ``kSpan = 32`` consecutive windows (window
``32 s`` to ``32 s + 31``) through shared memory when the span's starts and ends + 1 are
non-decreasing, all its windows share one piece, and its site range R (the sites of all its windows)
covers at most ``kSpanTiles = 512`` tiles holding at most ``kSpanFlags = 1024`` U- and Q-flagged sites.
Any other span runs the per-window code.  Every case here says from its data which path each span
takes (``_span_path`` restates the rule in numpy), and the results must not depend on it."""

from __future__ import annotations

import numpy as np
import pytest

from test_gpu_kernel_boundaries import (_k4_compare, _k4_device, _k4_expected, _k4_genome, _k4_jobs, _k4_matrices,
                                        _k4_oracle_check, _tiles)

SPAN, SPAN_TILES, SPAN_FLAGS = 32, 512, 1024  # kSpan, kSpanTiles, kSpanFlags


def _span_path(pos, derived, k, ws, we, first=None, last=None) -> np.ndarray:
    """Per span: True where the kernel takes the span path (for every job: the flag counts are
    those of a job with both U and Q)."""
    n = pos.size
    first = np.zeros(ws.size, np.int64) if first is None else first
    last = np.full(ws.size, n, np.int64) if last is None else last
    u_flag, q_flag = derived & (k > 0), derived
    out = []
    for s in range(0, ws.size, SPAN):
        a, b = ws[s : s + SPAN], we[s : s + SPAN] + 1
        f, l = first[s : s + SPAN], last[s : s + SPAN]
        ok = bool((np.diff(a) >= 0).all() and (np.diff(b) >= 0).all() and (f == f[0]).all() and (l == l[0]).all())
        if ok:
            p = pos[f[0] : l[0]]
            lo = int(f[0] + np.searchsorted(p, min(a[0], b[0])))
            hi = max(lo, int(f[0] + np.searchsorted(p, max(a[-1], b[-1]))))
            ok = _tiles(lo, hi) <= SPAN_TILES and u_flag[lo:hi].sum() <= SPAN_FLAGS and q_flag[lo:hi].sum() <= SPAN_FLAGS
        out.append(ok)
    return np.array(out)


def _windows(pos, ranges):
    """Site ranges [lo, hi) -> inclusive position windows; an empty range becomes end = start - 1."""
    ws = np.array([pos[lo] for lo, _ in ranges], np.int64)
    we = np.array([pos[hi - 1] if hi > lo else pos[lo] - 1 for lo, hi in ranges], np.int64)
    return ws, we


def _run_and_compare(engine, pg, mats, pos, derived, k, ws, we):
    exp = _k4_expected(pos, derived, k, ws, we)
    _k4_oracle_check(mats, pos, exp, ws, we, np.linspace(0, ws.size - 1, min(ws.size, 24)).astype(int))
    need_u = int(exp["u"].sum(axis=1).max())
    need_q = max(sum(p.size for p in exp["q_pos"][j]) for j in range(exp["u"].shape[0]))
    res, sc = _k4_device(pg, ws, we, need_u, need_q)
    assert (sc.cap_u, sc.cap_q) == (need_u, need_q)  # exactly enough: no second launch
    _k4_compare(res, exp, "device scorer")
    return exp, need_u, need_q


@pytest.fixture(scope="module")
def engine():
    from sai_b200.scoring import HostEngine

    e = HostEngine(0)
    yield e
    e.close()


def _genome():
    """_k4_genome's regions (dense 0-6000, gap, sparse, medium from 94 000) with positions 1, 2, ...
    that jump by 1000 at site 100 000, so that windows there hold no site."""
    derived, k, regions = _k4_genome()
    n = derived.size
    pos = (np.arange(1, n + 1) + 1000 * (np.arange(n) >= 100_000)).astype(np.int32)
    return derived, k, regions, pos


def _groups(derived, k, pos):
    """Groups of 32 windows, each filling one span: name -> site ranges (or position windows)."""
    idx = np.flatnonzero(derived)  # Q-flagged sites
    g = {}
    # exactly c Q-flagged sites per window, ranges from right after the previous flag / right on a flag
    # to right on the last one / right before the next one: 0 .. 257 around the n <= 32 selection
    g["gap_0"] = [(6000 + 40 * i, 6000 + 40 * i + 50) for i in range(SPAN)]
    for c in (32, 33, 256, 257):
        j0 = int(np.searchsorted(idx, 100))
        rs = []
        for i in range(SPAN):
            j = j0 + 7 * i
            lo = int(idx[j - 1]) + 1 if i % 2 else int(idx[j])
            hi = int(idx[j + c]) if i % 2 else int(idx[j + c - 1]) + 1
            rs.append((lo, hi))
        g[f"q{c}"] = rs
    # equal starts, windows selecting nothing (end < start), windows between the positions around the jump
    b = 99_980
    p = lambda s: int(pos[s])
    g["edges"] = ("pos", [(p(b), p(b + 3)), (p(b), p(b + 3)), (p(b), p(b + 9)), (p(b + 5), p(b + 9)),
                          (p(b + 12), p(b + 10)), (p(b + 12), p(b + 10)), (p(b + 19), p(b + 19)),
                          (p(b + 19) + 1, p(b + 19) + 999), (p(b + 19) + 1, p(b + 19) + 999),
                          (p(b + 19) + 400, p(b + 19) + 999), (p(b + 19) + 500, p(b + 20)),
                          (p(b + 20), p(b + 20)), (p(b + 20), p(b + 25))]
                 + [(p(b + 30 + 3 * i), p(b + 40 + 9 * i)) for i in range(SPAN - 13)])
    # fallbacks: R over more than 512 tiles; more than 1024 U- and Q-flagged sites; an unsorted span
    g["long"] = [(10_000 + 100 * i, 27_000 + 100 * i) for i in range(SPAN)]
    g["flags"] = [(50 * i, 2200 + 50 * i) for i in range(SPAN)]
    g["unsorted"] = g["q33"][::-1]
    return g


def _assemble(pos, groups, tail):
    names, ws, we = [], [], []
    for name, rs in groups.items():
        if isinstance(rs, tuple):
            a = np.array([w[0] for w in rs[1]], np.int64)
            b = np.array([w[1] for w in rs[1]], np.int64)
        else:
            a, b = _windows(pos, rs)
        assert a.size == SPAN, name
        names.append(name)
        ws.append(a)
        we.append(b)
    a, b = _windows(pos, tail)
    return names, np.concatenate(ws + [a]), np.concatenate(we + [b])


FALLBACK = {"long", "flags", "unsorted"}


@pytest.mark.gpu
def test_k4_span_path_cases_one_piece_and_pieces(engine):
    """Spans of windows with 0, 32, 33, 256 and 257 Q-flagged sites, equal starts, end < start and
    windows without sites, next to spans over the shared-memory budget (tiles, flags) and an unsorted
    span; six jobs (U + Q at four quantiles, U-only, Q-only) in one launch; a partial last span.
    Candidate buffers exactly as large as needed.  Then the same windows over two tile-aligned pieces
    (the genome twice), span s in piece s % 2, with one sorted span whose windows cross from the
    first piece to the second; candidate buffers one short (DeviceScorer.results grows them and
    re-runs the window kernel)."""
    from sai_b200.encode import pack_populations

    derived, k, _, pos = _genome()
    mats = _k4_matrices(derived, k)
    groups = _groups(derived, k, pos)
    names, ws, we = _assemble(pos, groups, [(94_000 + 50 * i, 94_000 + 50 * i + 700) for i in range(5)])
    span = _span_path(pos, derived, k, ws, we)
    assert span.size == len(names) + 1
    assert [bool(s) for s in span[:-1]] == [nm not in FALLBACK for nm in names] and span[-1]
    pg = pack_populations(mats, [2, 2, 2], pos)
    exp, need_u, need_q = _run_and_compare(engine, pg, mats, pos, derived, k, ws, we)
    at = {nm: slice(SPAN * i, SPAN * (i + 1)) for i, nm in enumerate(names)}
    for c in (32, 33, 256, 257):
        assert (exp["n_q"][at[f"q{c}"]] == c).all()
    assert (exp["n_q"][at["gap_0"]] == 0).all() and (exp["nsnps"][at["edges"]] == 0).sum() >= 5
    assert (we[at["edges"]] < ws[at["edges"]]).any() and (np.diff(ws[at["edges"]]) == 0).any()

    n = pos.size
    assert n % 32 == 0
    pg2 = pack_populations([np.concatenate([m, m]) for m in mats], [2, 2, 2], np.concatenate([pos, pos]))
    cross_name = "cross"
    names2 = names + [cross_name]
    ws2 = np.concatenate([ws[: SPAN * len(names)], ws[at["q32"]], ws[SPAN * len(names) :]])
    we2 = np.concatenate([we[: SPAN * len(names)], we[at["q32"]], we[SPAN * len(names) :]])
    first = (n * ((np.arange(ws2.size) // SPAN) % 2)).astype(np.int32)
    first[SPAN * len(names) : SPAN * len(names) + SPAN // 2] = 0
    first[SPAN * len(names) + SPAN // 2 : SPAN * (len(names) + 1)] = n
    span2 = _span_path(np.concatenate([pos, pos]), np.concatenate([derived, derived]), np.concatenate([k, k]),
                       ws2, we2, first.astype(np.int64), first.astype(np.int64) + n)
    assert [bool(s) for s in span2[:-1]] == [nm not in FALLBACK | {cross_name} for nm in names2] and span2[-1]
    exp2 = _k4_expected(pos, derived, k, ws2, we2)
    nu2 = int(exp2["u"].sum(axis=1).max())
    nq2 = max(sum(p.size for p in exp2["q_pos"][j]) for j in range(exp2["u"].shape[0]))
    res2, sc2 = _k4_device(pg2, ws2, we2, nu2 - 1, nq2 - 1, first, first + n)
    assert (sc2.cap_u, sc2.cap_q) == (nu2, nq2)  # grown by the retry
    _k4_compare(res2, exp2, "two pieces")

    # the host-buffer engine runs the same kernel with its own capacity handling
    _k4_compare(engine.score(pg, list(zip(ws.tolist(), we.tolist())), _k4_jobs()), exp, "HostEngine")


@pytest.mark.gpu
@pytest.mark.parametrize("W", [1, SPAN - 1, SPAN, SPAN + 1, 3 * SPAN])
def test_k4_span_path_window_counts(W):
    """Sorted sliding windows (600 sites every 45) over the medium region: every span, full or
    partial, takes the span path."""
    from sai_b200.encode import pack_populations

    derived, k, regions, pos = _genome()
    mats = _k4_matrices(derived, k)
    lo0 = regions["medium"][0]
    ws, we = _windows(pos, [(lo0 + 45 * i, lo0 + 45 * i + 600) for i in range(W)])
    assert _span_path(pos, derived, k, ws, we).all()
    pg = pack_populations(mats, [2, 2, 2], pos)
    _run_and_compare(None, pg, mats, pos, derived, k, ws, we)


@pytest.mark.gpu
def test_k4_span_path_duplicates_and_int32_max(engine):
    """Split multi-allelic records (one position on up to three consecutive sites) up to 2^31 - 1:
    sorted windows starting and ending on duplicated positions, windows ending at 2^31 - 1 and beyond
    it, starting at 2^31 - 1 and beyond it -- all through the span path."""
    from sai_b200.encode import pack_populations

    rng = np.random.default_rng(29)
    top = 2**31 - 1
    uniq = np.append(np.sort(rng.choice(np.arange(top - 300_000, top), size=3999, replace=False)), top)
    pos = np.repeat(uniq, rng.choice([1, 1, 1, 2, 3], size=uniq.size)).astype(np.int32)
    n = pos.size
    derived = rng.random(n) < np.where(np.arange(n) < n // 2, 0.012, 0.5)  # sparse half, dense half
    k = rng.integers(0, 21, size=n)
    mats = _k4_matrices(derived, k)
    dup = np.flatnonzero(np.diff(pos) == 0)
    wins = []
    h = n // 2
    # spans of 32 windows whose starts (then ends) are sorted duplicates of one stretch of sites:
    # short windows in the dense half, windows of 1500 sites in the sparse half
    for length, a, b in ((40, h, h + 600), (1500, 0, 1000)):
        for d in np.sort(rng.choice(dup[(dup >= a) & (dup < b)], size=SPAN, replace=False)):
            wins.append((int(pos[d]), int(pos[d + length])))  # from the first copy of a duplicate
    for length, a, b in ((40, h + 600, h + 1200), (1500, 1500, 2500)):
        for d in np.sort(rng.choice(dup[(dup >= a) & (dup < b)], size=SPAN, replace=False)):
            wins.append((int(pos[d - length]), int(pos[d])))  # ending on it
    wins += [(int(pos[-300]), int(pos[-200])), (int(pos[-300]), top), (int(pos[-5]), top), (int(pos[-5]), 2**40),
             (top, 2**40), (2**33, 2**40), (2**33, 2**41)]
    ws = np.array([w[0] for w in wins], np.int64)
    we = np.array([w[1] for w in wins], np.int64)
    assert _span_path(pos, derived, k, ws, we).all()
    pg = pack_populations(mats, [2, 2, 2], pos)
    exp, _, _ = _run_and_compare(engine, pg, mats, pos, derived, k, ws, we)
    assert (exp["hi"] == n).sum() >= 4 and (exp["n_q"] > 32).any() and ((exp["n_q"] > 0) & (exp["n_q"] <= 32)).any()
    _k4_compare(engine.score(pg, wins, _k4_jobs()), exp, "HostEngine")
