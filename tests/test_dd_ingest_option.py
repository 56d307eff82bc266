"""CPU side of DD on device-parsed VCFs (``dd_ingest="device"``): the option's checks and the
choice between device and host ingest."""

from __future__ import annotations

import numpy as np
import pytest

from sai_b200.configs import PloidyConfig, StatConfig


def _lists(tmp_path):
    (tmp_path / "ref.list").write_text("R\ta\nR\tb\n")
    (tmp_path / "tgt.list").write_text("T\td\n")
    (tmp_path / "src.list").write_text("S1\te\nS2\tf\n")
    return [str(tmp_path / f"{g}.list") for g in ("ref", "tgt", "src")] + [None]


def test_dd_ingest_device_needs_device_ingest(tmp_path):
    from sai_b200.preprocessors import ChunkPreprocessor

    files = _lists(tmp_path)
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 2}, "src": {"S1": 2, "S2": 2}})
    sc = StatConfig({"DD": True})
    make = lambda **k: ChunkPreprocessor("x.vcf", *files, 100, 50, str(tmp_path / "o.tsv"), pc, sc, **k)
    with pytest.raises(ValueError, match="dd_ingest='device' needs ingest='device'"):
        make(dd_ingest="device")
    with pytest.raises(ValueError, match="dd_ingest must be"):
        make(ingest="device", dd_ingest="gpu")
    assert make().dd_ingest == "host"
    assert make(ingest="device", dd_ingest="device").dd_ingest == "device"


def test_fallback_reason_with_device_dd(tmp_path):
    from sai_b200.vcf import AncAlleles, population_plan
    from sai_b200.vcf_device import fallback_reason

    files = _lists(tmp_path)
    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 4}, "src": {"S1": 1, "S2": 2}})
    plan, _, _ = population_plan(tuple(zip(("ref", "tgt", "src", "outgroup"), files)), pc)
    u = {"U": {"ref": {"R": 0.1}, "tgt": {"T": 0.2}, "src": {"S1": "=1", "S2": "=1"}}}
    dd = StatConfig({**u, "DD": True})
    long = AncAlleles(np.array([5, 9]), np.array(["A", "ACGTACGT"], dtype=object))
    assert "DD" in fallback_reason(dd, pc, plan, None, "21", 2)
    assert "DD" in fallback_reason(dd, pc, plan, None, "21", 2, "host")
    assert fallback_reason(dd, pc, plan, None, "21", 2, "device") is None
    # every other reason is still named
    assert "longer than 7" in fallback_reason(dd, pc, plan, long, "21", 2, "device")
    assert "chromosome" in fallback_reason(dd, pc, plan, None, "c" * 256, 2, "device")
    assert "ploidies" in fallback_reason(dd, pc, plan, None, "21", 1, "device")
    many = [(g, s, pops * 6) for g, s, pops in plan]
    assert "populations" in fallback_reason(dd, pc, many, None, "21", 2, "device")
    with pytest.raises(ValueError, match="dd_ingest must be"):
        fallback_reason(dd, pc, plan, None, "21", 2, "gpu")


def test_neg_table_entry_points_in_abi():
    from sai_b200 import _cabi

    for name in ("sai_engine_set_vcf_neg_table", "sai_engine_loaded_neg_table", "sai_engine_dd_sums_loaded"):
        assert name in _cabi.SYMBOLS
    assert _cabi.SYMBOLS["sai_engine_loaded_neg_table"][0] is _cabi.C.c_int64
