"""``score_genome``: every chromosome of a multi-chromosome VCF scored from one device pass.

The specification is ``score`` run once per chromosome with the outputs concatenated (header lines
once): the score file and the ``.U.log`` / ``.Q.log`` files must be equal byte for byte, and so must
the errors.  Below that, the one-pass read (``vcf_device.read_genome``) is pinned chromosome by
chromosome against ``chromosome_span`` and against the host read packed with ``pack_populations``:
each chromosome's tile range, padding sites included, is the host pack of that chromosome alone.
Every file is generated here from a seed.
"""

from __future__ import annotations

import numpy as np
import pytest

from helpers import SimplePloidy

pytestmark = pytest.mark.gpu

GROUPS = ("ref", "tgt", "src", "outgroup")
POPS = {"ref": {"R1": 4, "R2": 3}, "tgt": {"T1": 4, "T2": 3, "T3": 3}, "src": {"S1": 3, "S2": 2},
        "outgroup": {"O1": 2, "O2": 2}}
PLOIDY = {g: {p: 2 for p in pops} for g, pops in POPS.items()}
WIN_LEN, WIN_STEP = 2000, 1000
# (name, records, requested, ancestral table): "all" = every record (the REF allele), "most" = a
# random 85% with REF or ALT and a few alleles matching neither, "not_first" = "most" without the
# first record, "none_match" = entries at positions without a record only (nothing kept)
CHROMS = [("1", 70, True, "most"), ("10", 64, True, "all"), ("chrUn", 20, False, "most"), ("chr1", 1, True, "all"),
          ("chr1_alt", 45, True, "not_first"), ("chrE", 30, True, "none_match"), ("chrX", 50, True, "most")]
REQUESTED = [c[0] for c in CHROMS if c[2]]


def _samples():
    return [s for g in GROUPS for p, n in POPS[g].items() for s in (f"{p}_{i}" for i in range(n))]


def _write_case(d, seed=0, chroms=CHROMS, interleave=False):
    """VCF (plain and bgzip), ancestral BED and population lists under ``d``."""
    from sai_b200.vcf import write_bgzf

    rng = np.random.default_rng(seed)
    samples = _samples()
    gts = np.array(["0|0", "0|1", "1|0", "1|1", "./.", "0|0", "0|0"])
    lines, bed = [], []
    per_chrom = []
    for name, n, _, anc in chroms:
        pos = np.cumsum(rng.integers(40, 160, size=n)) + int(rng.integers(1, 500))
        rows = []
        for i, p in enumerate(pos.tolist()):
            ref, alt = rng.choice(list("ACGT"), size=2, replace=False)
            g = "\t".join(rng.choice(gts, size=len(samples)).tolist())
            rows.append(f"{name}\t{p}\t.\t{ref}\t{alt}\t.\tPASS\t.\tGT\t{g}\n")
            if anc == "all":
                bed.append(f"{name}\t{p - 1}\t{p}\t{ref}\n")
            elif anc in ("most", "not_first") and not (anc == "not_first" and i == 0) and rng.random() < 0.85:
                bed.append(f"{name}\t{p - 1}\t{p}\t{rng.choice([ref, alt, 'T' if ref != 'T' and alt != 'T' else 'G'], p=[0.6, 0.35, 0.05])}\n")
        if anc == "none_match":
            bed.extend(f"{name}\t{p}\t{p + 1}\tA\n" for p in (pos[:-1] + 1).tolist())
        per_chrom.append(rows)
    if interleave:  # the first chromosome's last records after the second chromosome's
        a, b = per_chrom[0], per_chrom[1]
        per_chrom[0], per_chrom[1] = a[: len(a) // 2], b + a[len(a) // 2 :]
    for rows in per_chrom:
        lines.extend(rows)
    head = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(samples) + "\n"
    text = (head + "".join(lines)).encode()
    (d / "g.vcf").write_bytes(text)
    write_bgzf(str(d / "g.vcf.gz"), text, block=997)  # small blocks: records and chromosomes straddle them
    (d / "anc.bed").write_text("".join(bed))
    lists = {}
    for g in GROUPS:
        lists[g] = str(d / f"{g}.list")
        with open(lists[g], "w") as f:
            for p, n in POPS[g].items():
                f.writelines(f"{p}\t{p}_{i}\n" for i in range(n))
    return lists, len(text) - len(head)


def _config(d, lists, stats):
    import yaml

    cfg = d / "cfg.yaml"
    cfg.write_text(yaml.safe_dump({"statistics": stats, "ploidies": PLOIDY, "populations": lists}))
    return str(cfg)


def _stats(with_four=True, dd=False):
    ref = {p: 0.3 for p in POPS["ref"]}
    st = {"U": {"ref": ref, "tgt": {p: 0.5 for p in POPS["tgt"]}, "src": {"S1": "=1", "S2": "=1"}},
          "Q": {"ref": ref, "tgt": {p: 0.95 for p in POPS["tgt"]}, "src": {"S1": "=1", "S2": "=1"}}}
    if with_four:
        st.update({"Danc": True, "Dplus": True, "df": True, "fd": True})
    if dd:
        st["DD"] = True
    return st


def _texts(out):
    return [open(p, "rb").read() for p in (str(out), str(out)[:-4] + ".U.log", str(out)[:-4] + ".Q.log")]


def _per_chromosome(vcf, names, anc, out, cfg):
    """The specification: ``score`` per chromosome (host ingest), outputs concatenated, headers once."""
    from sai_b200.score import score

    parts = []
    for i, c in enumerate(names):
        o = out.parent / f"part{i}" / out.name
        score(vcf, c, WIN_LEN, WIN_STEP, anc, str(o), cfg)
        parts.append(_texts(o))
    return [parts[0][k] + b"".join(p[k].split(b"\n", 1)[1] for p in parts[1:]) for k in range(3)]


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


@pytest.mark.parametrize("fmt", ["vcf", "vcf.gz"])
@pytest.mark.parametrize("inflate", ["host", "device"])
@pytest.mark.parametrize("slicing", [None, (400, 3)])
def test_score_genome_equals_per_chromosome_score(fmt, inflate, slicing, tmp_path, device_only):
    from sai_b200.score import score_genome

    lists, _ = _write_case(tmp_path)
    cfg = _config(tmp_path, lists, _stats())
    vcf, anc = str(tmp_path / f"g.{fmt}"), str(tmp_path / "anc.bed")
    want = _per_chromosome(vcf, REQUESTED, anc, tmp_path / "want" / "s.tsv", cfg)
    device_only(slicing)
    out = tmp_path / "got" / "s.tsv"
    score_genome(vcf, REQUESTED, WIN_LEN, WIN_STEP, anc, str(out), cfg, inflate=inflate)
    got = _texts(out)
    assert got == want
    rows = got[0].decode().splitlines()[1:]
    assert {r.split("\t")[0] for r in rows} == set(REQUESTED)
    assert any(r.startswith("chrE\t") and "\tnan" in r for r in rows)  # the chromosome left empty: NaN rows


def test_requested_order_and_no_outgroup_statistics(tmp_path, device_only):
    from sai_b200.score import score_genome

    lists, _ = _write_case(tmp_path, seed=3)
    cfg = _config(tmp_path, lists, _stats(with_four=False))
    names = ["chrX", "10", "chr1", "1"]
    vcf, anc = str(tmp_path / "g.vcf.gz"), str(tmp_path / "anc.bed")
    want = _per_chromosome(vcf, names, anc, tmp_path / "want" / "s.tsv", cfg)
    device_only()
    score_genome(vcf, names, WIN_LEN, WIN_STEP, anc, str(tmp_path / "got" / "s.tsv"), cfg)
    assert _texts(tmp_path / "got" / "s.tsv") == want


@pytest.fixture(scope="module")
def engine():
    from sai_b200.scoring import HostEngine

    e = HostEngine(0)
    yield e
    e.close()


def _plan(vcf, lists):
    from sai_b200.vcf_device import read_plan

    return read_plan(vcf, REQUESTED[0], SimplePloidy(PLOIDY), lists["ref"], lists["tgt"], lists["src"],
                     lists["outgroup"])


@pytest.mark.parametrize("fmt,inflate,slicing", [("vcf", "host", None), ("vcf", "host", (300, 3)),
                                                 ("vcf.gz", "host", (1000, 2)), ("vcf.gz", "device", (700, 4))])
def test_read_genome_spans_and_tiles_per_chromosome(fmt, inflate, slicing, engine, tmp_path):
    from sai_b200 import _cabi
    from sai_b200.encode import pack_populations
    from sai_b200.vcf import chromosome_span, read_data
    from sai_b200.vcf_device import genome_tables, read_genome

    lists, text_bytes = _write_case(tmp_path, seed=1)
    vcf, anc = str(tmp_path / f"g.{fmt}"), str(tmp_path / "anc.bed")
    plan, requests, out = _plan(vcf, lists)
    engine.set_vcf_slicing(*(slicing or (0, 0)))
    try:
        g = read_genome(engine, vcf, REQUESTED, plan, requests, out, genome_tables(REQUESTED, anc), inflate=inflate)
        slices = engine.vcf_slices()
        fed = engine.vcf_stats()["text_bytes"]
    finally:
        engine.set_vcf_slicing(0, 0)
    # one session, one pass over the text
    assert fed <= text_bytes + 1
    if slicing:
        assert slices <= text_bytes // (slicing[0] // 2) + 2
    else:
        assert slices == 1
    tiles = engine.loaded_tiles(g.layout, g.total_sites)
    tile_bytes = int(g.layout.pairs_per_site) * 32 * 8
    pc = SimplePloidy(PLOIDY)
    for c, name in enumerate(REQUESTED):
        first, last, n = chromosome_span(vcf, name)
        assert g.span[c][:2] == (first, last), name
        if n != -1:
            assert g.span[c][2] == n, name
        d = read_data(vcf, name, pc, lists["ref"], lists["tgt"], lists["src"], lists["outgroup"], anc)
        if d["ref"][0] is None:  # every record dropped by the ancestral table
            assert g.n_sites[c] == 0 and g.first_site[c] == -1, name
            continue
        mats = [pdat.GT for grp in GROUPS for pdat in d[grp][0].values()]
        ploidy = [2] * len(mats)
        host = pack_populations(mats, ploidy, d["ref"][0]["R1"].POS, bits=[int(g.layout.pop[p].bits) for p in range(len(mats))])
        assert g.first_site[c] % _cabi.TILE_SITES == 0, name
        assert np.array_equal(g.pos[c], host.pos), name
        t0 = g.first_site[c] // 32
        got = tiles[t0 * tile_bytes : (t0 + (g.n_sites[c] + 31) // 32) * tile_bytes]
        assert got.tobytes() == host.packed.tobytes(), name
    assert g.n_sites[REQUESTED.index("10")] == 64
    assert g.n_sites[REQUESTED.index("chr1")] == 1


def test_interleaved_file_and_dd_fall_back_with_identical_output(tmp_path):
    from sai_b200.score import score_genome

    lists, _ = _write_case(tmp_path, seed=2, interleave=True)
    vcf, anc = str(tmp_path / "g.vcf.gz"), str(tmp_path / "anc.bed")
    for i, stats in enumerate((_stats(), _stats(with_four=False, dd=True))):
        cfg = _config(tmp_path, lists, stats)
        want = _per_chromosome(vcf, REQUESTED, anc, tmp_path / f"want{i}" / "s.tsv", cfg)
        score_genome(vcf, REQUESTED, WIN_LEN, WIN_STEP, anc, str(tmp_path / f"got{i}" / "s.tsv"), cfg, inflate="device")
        assert _texts(tmp_path / f"got{i}" / "s.tsv") == want


def test_interleaved_file_is_reported_by_the_device(engine, tmp_path):
    from sai_b200.vcf_device import genome_tables, read_genome

    lists, _ = _write_case(tmp_path, seed=2, interleave=True)
    vcf = str(tmp_path / "g.vcf")
    plan, requests, out = _plan(vcf, lists)
    assert read_genome(engine, vcf, REQUESTED, plan, requests, out, genome_tables(REQUESTED, None)) is None
    g = read_genome(engine, vcf, REQUESTED[2:], plan, requests, out, genome_tables(REQUESTED[2:], None))
    assert g is not None and g.n_sites[0] == 1  # the chromosomes after the interleaved pair are contiguous


def test_errors_match_score(tmp_path):
    from sai_b200.score import score, score_genome

    lists, _ = _write_case(tmp_path, seed=4)
    cfg = _config(tmp_path, lists, _stats())
    vcf, anc = str(tmp_path / "g.vcf"), str(tmp_path / "anc.bed")
    out = tmp_path / "e" / "s.tsv"
    with pytest.raises(ValueError, match="Chromosome chr2 not found in VCF."):
        score_genome(vcf, ["1", "chr2"], WIN_LEN, WIN_STEP, anc, str(out), cfg)
    assert not out.exists()
    # chrUn has records but no ancestral allele
    bed = [l for l in open(anc) if not l.startswith("chrUn\t")]
    (tmp_path / "anc_no_un.bed").write_text("".join(bed))
    with pytest.raises(ValueError) as want:
        score(vcf, "chrUn", WIN_LEN, WIN_STEP, str(tmp_path / "anc_no_un.bed"), str(tmp_path / "w" / "s.tsv"), cfg)
    with pytest.raises(ValueError) as got:
        score_genome(vcf, ["1", "chrUn"], WIN_LEN, WIN_STEP, str(tmp_path / "anc_no_un.bed"), str(out), cfg)
    assert str(got.value) == str(want.value) and "No ancestral allele" in str(got.value)
    assert not out.exists()
