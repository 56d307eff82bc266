"""CPU side of device VCF ingest: the population plan shared with ``read_data`` and the choice
between device and host ingest."""

from __future__ import annotations

import warnings

import pytest

from sai_b200.configs import PloidyConfig, StatConfig


def _lists(tmp_path):
    (tmp_path / "ref.list").write_text("R\ta\nR\tb\nX\tc\n")
    (tmp_path / "tgt.list").write_text("T\td\n")
    (tmp_path / "src.list").write_text("S1\te\nS2\tf\n")
    return [str(tmp_path / f"{g}.list") for g in ("ref", "tgt", "src")] + [None]


def test_population_plan_matches_read_data_rules(tmp_path):
    from sai_b200.vcf import population_plan

    files = _lists(tmp_path)
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 4}, "src": {"S1": 1, "S2": 2}})
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        plan, requests, out = population_plan(tuple(zip(("ref", "tgt", "src", "outgroup"), files)), pc)
    assert any("'X' found in sample file" in str(x.message) for x in w)
    assert out == {"outgroup": (None, None)}
    assert [(g, pops) for g, _, pops in plan] == [("ref", [("R", 0, 2)]), ("tgt", [("T", 2, 3)]),
                                                  ("src", [("S1", 3, 4), ("S2", 4, 5)])]
    assert requests == [("a", 2), ("b", 2), ("d", 4), ("e", 1), ("f", 2)]
    with pytest.raises(ValueError, match="not found in sample file"):
        population_plan((("ref", files[0]),), PloidyConfig({"ref": {"Q": 2}, "tgt": {"T": 2}, "src": {"S1": 2}}))


def test_device_ingest_fallback_selection(tmp_path):
    from sai_b200.vcf import AncAlleles, population_plan
    from sai_b200.vcf_device import fallback_reason

    import numpy as np

    files = _lists(tmp_path)
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 4}, "src": {"S1": 1, "S2": 2}})
    plan, _, _ = population_plan(tuple(zip(("ref", "tgt", "src", "outgroup"), files)), pc)
    u = {"U": {"ref": {"R": 0.1}, "tgt": {"T": 0.2}, "src": {"S1": "=1", "S2": "=1"}}}
    sc = StatConfig(u)
    short = AncAlleles(np.array([5, 9]), np.array(["A", "ACGTACG"], dtype=object))
    long = AncAlleles(np.array([5, 9]), np.array(["A", "ACGTACGT"], dtype=object))
    assert fallback_reason(sc, pc, plan, None, "21", 2) is None
    assert fallback_reason(sc, pc, plan, short, "21", 2) is None
    assert "longer than 7" in fallback_reason(sc, pc, plan, long, "21", 2)
    assert "DD" in fallback_reason(StatConfig({**u, "DD": True}), pc, plan, None, "21", 2)
    assert "chromosome" in fallback_reason(sc, pc, plan, None, "c" * 256, 2)
    # one source at a time: S2 would be scored with S1's ploidy (the position in the combination)
    assert "ploidies" in fallback_reason(sc, pc, plan, None, "21", 1)
    many = [(g, s, pops * 6) for g, s, pops in plan]
    assert "populations" in fallback_reason(sc, pc, many, None, "21", 2)
