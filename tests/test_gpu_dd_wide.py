"""DD on populations of 5-8 bit-planes: per-individual values of 15..127 (multi-allelic genotype
indices, high ploidy, the reference's flipped-missing alleles) score exactly like the oracle,
from the kernels through the stat class to a VCF chunk."""

from __future__ import annotations

import numpy as np
import pytest

import sai_oracle as orc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    from sai_b200.scoring import HostEngine

    e = HostEngine(0)
    yield e
    e.close()


def _population(rng, f, n, ploidy, bits, wide, miss):
    """Binomial calls that fit ``bits`` planes, a share ``miss`` missing with raw values -ploidy..-1;
    in a population of 5+ planes a share ``wide`` of the calls (``"one"``: a single call) becomes a
    value in 15..max, and a rate below 1 adds three 14s and three 15s (the last value row and the
    first wide value)."""
    top = min(127, (1 << bits) - 2)
    g = np.minimum(rng.binomial(ploidy, f[:, None], size=(f.shape[0], n)), top)
    hole = rng.random(g.shape) < miss
    hit = np.zeros(g.shape, bool)
    if bits > 4 and wide == "one":
        hit.flat[rng.choice(np.flatnonzero(~hole))] = True
    elif bits > 4:
        hit = (rng.random(g.shape) < wide) & ~hole
    g[hit] = rng.integers(15, top + 1, size=int(hit.sum()))
    if bits > 4 and wide != "one" and 0 < wide < 1:
        g.flat[rng.choice(np.flatnonzero(~hole), size=6, replace=False)] = [14, 14, 14, 15, 15, 15]
    g[hole] = -rng.integers(1, ploidy + 1, size=int(hole.sum()))
    return g.astype(np.int8)


# (ploidy, bit-planes, individuals) of ref, tgt, src1, src2; wide-call rate; missing rate
CASES = {
    "one-wide-call": ([2, 8, 4, 2], [2, 8, 5, 2], [40, 70, 3, 45], "one", 0.03),
    "wide-0.1%": ([8, 1, 8, 8], [5, 2, 8, 4], [90, 20, 41, 5], 0.001, 0.0),
    "ploidy-16": ([16, 16, 1, 16], [5, 5, 2, 5], [60, 45, 34, 3], 0, 0.03),  # ordinary calls of 15 and 16
    "wide-5%": ([4, 2, 2, 4], [6, 5, 2, 6], [33, 64, 70, 2], 0.05, 0.3),
    "every-call-wide": ([16, 8, 8, 16], [8, 8, 5, 8], [50, 35, 3, 33], 1.0, 0.03),
    "wide-sources-only": ([2, 4, 8, 2], [2, 4, 8, 6], [37, 29, 36, 7], 0.05, 0.03),
}


def _case(name, seed):
    from sai_b200.encode import pack_populations

    ploidy, bits, n_ind, wide, miss = CASES[name]
    rng = np.random.default_rng(seed)
    n_sites = int(rng.integers(200, 500))
    f = rng.beta(0.4, 1.0, size=n_sites)
    mats = []
    for k, (p, b, n) in enumerate(zip(ploidy, bits, n_ind)):
        one = wide == "one" and k != 1  # "one": the single wide call of the matrix is in tgt
        mats.append(_population(rng, f, n, p, b, 0 if one else wide, miss))
    pos = np.cumsum(rng.integers(1, 30, size=n_sites)).astype(np.int32)
    pg = pack_populations(mats, ploidy, pos, bits=bits, keep_negatives=True)
    assert [pg.layout.pop[i].bits for i in range(4)] == bits
    top = int(pos[-1])
    wins = [(1, top), (int(pos[3]), int(pos[n_sites // 2])), (top + 1, top + 50), (int(pos[10]), int(pos[10])),
            (int(pos[-1]), int(pos[-1]))]
    wins += [(s, s + 999) for s in range(1, top, 500)]
    return mats, pos, pg, wins, n_ind


@pytest.mark.parametrize("name", list(CASES))
@pytest.mark.parametrize("seed", [0, 1])
def test_dd_wide_random_vs_oracle(name, seed, engine):
    """ref_sum / tgt_sum equal the oracle's cityblock sums and DD is bit-identical, on layouts that
    mix 5-8-plane populations with 2- and 4-plane ones."""
    from sai_b200.scoring import dd_values, make_job

    mats, pos, pg, wins, n_ind = _case(name, 300 + seed)
    wide_calls = sum(int((m >= 15).sum()) for m in mats)
    assert wide_calls == 1 if CASES[name][3] == "one" else wide_calls > 0
    engine.score(pg, wins, [make_job(0, 1, [2, 3], True)])
    ref_sum, tgt_sum = engine.dd_sums(pg, 0, 1, [2, 3])
    got = dd_values(ref_sum, tgt_sum, n_ind[0], n_ind[1], n_ind[2:])
    m64 = [m.astype(np.int64) for m in mats]
    for i, (a, b) in enumerate(wins):
        keep = (pos >= a) & (pos <= b)
        if not keep.any():
            assert not ref_sum[:, i].any() and not tgt_sum[:, i].any()
            continue
        exp = orc.dd_statistic(m64[0][keep], m64[1][keep], [m64[2][keep], m64[3][keep]])
        for k in range(2):
            src = m64[2 + k][keep]
            assert np.array_equal(ref_sum[k, i, : n_ind[2 + k]], orc.cityblock_sums(src, m64[0][keep]).sum(axis=1)), (i, k)
            assert np.array_equal(tgt_sum[k, i, : n_ind[2 + k]], orc.cityblock_sums(src, m64[1][keep]).sum(axis=1)), (i, k)
            assert float(got[k][i]).hex() == float(exp[k]).hex(), (i, k)


def test_device_scorer_wide_hist_and_sums(engine):
    """DeviceScorer.site_hist + dd_sums on the tiles HostEngine scores give its integers; the
    histogram of a 5-8-plane population is the 15 values 0..14 and one row of wide calls."""
    import torch

    from sai_b200.scoring import DeviceScorer, make_job

    mats, pos, pg, wins, _ = _case("wide-5%", 7)
    engine.score(pg, wins, [make_job(0, 1, [2, 3], True)])
    want_ref, want_tgt = engine.dd_sums(pg, 0, 1, [2, 3])
    dev = torch.device("cuda")
    d_packed = torch.from_numpy(pg.packed).to(dev)
    d_pos = torch.from_numpy(pg.pos).to(dev)
    d_ws = torch.tensor([w[0] for w in wins], dtype=torch.int64, device=dev)
    d_we = torch.tensor([w[1] for w in wins], dtype=torch.int64, device=dev)
    d_neg = [torch.from_numpy(a).to(dev) for a in (pg.neg_site, pg.neg_ind, pg.neg_val)]
    sc = DeviceScorer(pg.layout, pg.n_sites, len(wins), 1)
    hist, missing = sc.site_hist(d_packed, [0, 1])
    ref_sum, tgt_sum, err = sc.dd_sums(d_packed, d_pos, d_ws, d_we, hist, 0, 1, [2, 3], pg.neg_off, *d_neg)
    torch.cuda.synchronize()
    assert int(err.item()) == 0
    assert np.array_equal(ref_sum.cpu().numpy(), want_ref) and np.array_equal(tgt_sum.cpu().numpy(), want_tgt)
    assert missing.cpu().tolist() == [int(pg.neg_off[1] - pg.neg_off[0]), int(pg.neg_off[2] - pg.neg_off[1])]
    h = hist.cpu().numpy()[:, : pg.n_sites]
    assert h.shape[0] == 32  # 6 and 5 planes: 16 rows each
    for p in range(2):
        m = mats[p]
        for u in range(15):
            assert np.array_equal(h[16 * p + u], (m == u).sum(axis=1)), (p, u)
        assert np.array_equal(h[16 * p + 15], (m >= 15).sum(axis=1)), p
        assert (m == 15).any() and (m == 14).any()


def test_dd_stat_class_values_above_14():
    """STAT_REGISTRY's DD on int64 matrices: multi-allelic diploid calls (0/12 = 12, 7/9 = 16) and
    octoploid data where a flipped all-missing call counts 16, bit for bit like the oracle."""
    from sai_b200.stats import STAT_REGISTRY

    cls = STAT_REGISTRY.get("DD")
    rng = np.random.default_rng(5)
    n = 300
    f = rng.beta(0.5, 1.0, size=n)
    # multi-allelic diploid: a few sums of two genotype indices up to 40, missing as -1 / -2
    mk = lambda k: rng.binomial(2, f[:, None], size=(n, k)).astype(np.int64)
    ref, tgt, s1, s2 = mk(40), mk(33), mk(2), mk(35)
    for m in (ref, tgt, s1, s2):
        hit = rng.random(m.shape) < 0.01
        m[hit] = rng.integers(3, 41, size=int(hit.sum()))
        hole = rng.random(m.shape) < 0.02
        m[hole] = -rng.integers(1, 3, size=int(hole.sum()))
    ref[0, 0], tgt[1, 1], s2[2, 2] = 12, 16, 15
    cases = [(ref, tgt, [s1, s2], 2, 2, [2, 2])]
    # octoploid with ancestral flips: |a - 1| per allele, so "./././././././." counts 16
    mk8 = lambda k: rng.binomial(8, f[:, None], size=(n, k)).astype(np.int64)
    ref8, tgt8, src8 = mk8(45), mk8(30), mk8(3)
    for m in (ref8, tgt8, src8):
        m[rng.random(m.shape) < 0.03] = 16
        hole = rng.random(m.shape) < 0.02
        m[hole] = -rng.integers(1, 9, size=int(hole.sum()))
    cases.append((ref8, tgt8, [src8], 8, 8, [8]))
    for r, t, srcs, pr, pt, ps in cases:
        res = cls(ref_gts=r, tgt_gts=t, src_gts_list=srcs, ref_ploidy=pr, tgt_ploidy=pt, src_ploidy_list=ps).compute()
        exp = orc.dd_statistic(r, t, srcs)
        assert res["name"] == "DD" and [float(v).hex() for v in res["value"]] == [float(v).hex() for v in exp]


def _write_vcf(path, rng, n_rec, n_r, n_t, n_s1, n_s2):
    """Diploid ref R and sources S1 with multi-allelic calls (0/12, 7/9, 3/.), octoploid tgt T with
    whole missing calls, tetraploid source S2."""
    samples = [f"r{i}" for i in range(n_r)] + [f"t{i}" for i in range(n_t)] + [f"a{i}" for i in range(n_s1)] + \
        [f"b{i}" for i in range(n_s2)]
    lines = ["##fileformat=VCFv4.2", "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(samples)]
    pos = np.sort(rng.choice(np.arange(1, 40 * n_rec), size=n_rec, replace=False))
    recs = []

    def gt(ploidy, p_alt):
        if ploidy == 2 and rng.random() < 0.04:
            return str(rng.choice(["0/12", "7/9", "3/.", "./.", "12/12"]))
        if ploidy == 8 and rng.random() < 0.03:
            return "/".join(["."] * 8)
        al = ["." if rng.random() < 0.02 else str(int(rng.random() < p_alt)) for _ in range(ploidy)]
        return "/".join(al)

    for p in pos:
        ref = "ACGT"[rng.integers(4)]
        alt = "ACGT"[("ACGT".index(ref) + 1 + rng.integers(3)) % 4]
        fa = float(rng.beta(0.4, 1.0))
        fields = [gt(2, fa) for _ in range(n_r)] + [gt(8, fa) for _ in range(n_t)] + [gt(2, fa) for _ in range(n_s1)] + \
            [gt(4, fa) for _ in range(n_s2)]
        lines.append("\t".join(["1", str(p), ".", ref, alt, ".", "PASS", ".", "GT"] + fields))
        recs.append((int(p), ref, alt))
    open(path, "w").write("\n".join(lines) + "\n")
    return samples, recs


def test_vcf_chunk_with_values_above_14(tmp_path):
    """A VCF with multi-allelic and octoploid calls (values up to 24 without and 16 from flipped
    missing calls with an ancestral-allele BED) scored by ChunkPreprocessor: items and TSV text equal
    the oracle's.  ingest="device" reads such a chunk on the host (DD) and writes the same text."""
    from sai_b200.configs import PloidyConfig, StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor
    from sai_b200.vcf import read_data

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
        vmax = max(int(d.GT.max()) for g in (ref_d, tgt_d, src_d) for d in g.values())
        assert vmax >= 16
        if a is not None:
            assert (tgt_d["T"].GT == 16).any()  # flipped "./././././././."
        exp = orc.score_chunk("1", start, end, win_len, win_step, ref_d, tgt_d, src_d, pc, StatConfig(stats), a is not None)
        rows, logs = orc.format_items(exp, ["U", "DD"])
        for ingest in ("host", "device"):
            out = tmp_path / f"{ingest}.{a is not None}.tsv"
            pre = ChunkPreprocessor(str(vcf), *lists, None, win_len, win_step, str(out), pc, StatConfig(stats), a,
                                    ingest=ingest)
            if ingest == "device":
                assert "DD" in pre.device_fallback("1", start, end)
            items = pre.run("1", start, end)
            assert len(items) == len(exp)
            for g, e in zip(items, exp):
                assert (g["start"], g["end"], g["nsnps"]) == (e["start"], e["end"], e["nsnps"])
                assert np.array_equal(g["cdd_pos"]["U"], e["cdd_pos"]["U"])
                if e["nsnps"]:
                    assert g["U"] == e["U"]
                    assert [float(x).hex() for x in g["DD"]] == [float(x).hex() for x in e["DD"]]
                    n_dd += 1
            pre.process_items(items)
            assert out.read_text() == "".join(rows)
            assert out.with_suffix(".U.log").read_text() == "".join(logs["U"])
    assert n_dd > 20


def test_dd_coverage_checks_on_wide_layout(engine):
    """The safety checks hold on 5-8-plane layouts: no negative-value table is refused, and a table
    that lacks one missing call raises the engine's coverage error."""
    from sai_b200 import _cabi
    from sai_b200.encode import pack_populations
    from sai_b200.scoring import make_job

    mats, pos, pg, wins, _ = _case("wide-5%", 11)
    ploidy, bits = CASES["wide-5%"][:2]
    bare = pack_populations(mats, ploidy, pos, bits=bits)
    engine.score(bare, wins, [make_job(0, 1, [2, 3], True)])
    with pytest.raises(ValueError, match="keep_negatives"):
        engine.dd_sums(bare, 0, 1, [2, 3])
    for pop in (0, 3):  # a 6-plane ref, a 6-plane source
        lo, hi = int(pg.neg_off[pop]), int(pg.neg_off[pop + 1])
        assert hi - lo > 3
        keep = np.ones(pg.neg_site.shape[0], bool)
        keep[lo + 1] = False
        cut = pack_populations(mats, ploidy, pos, bits=bits, keep_negatives=True)
        cut.neg_site, cut.neg_ind, cut.neg_val = cut.neg_site[keep].copy(), cut.neg_ind[keep].copy(), cut.neg_val[keep].copy()
        cut.neg_off = cut.neg_off.copy()
        cut.neg_off[pop + 1 :] -= 1
        engine.score(cut, wins, [make_job(0, 1, [2, 3], True)])
        with pytest.raises((_cabi.SaiError, ValueError), match="missing calls but .* entries in the negative-value table"):
            engine.dd_sums(cut, 0, 1, [2, 3])
