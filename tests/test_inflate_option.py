"""The ``inflate`` option and the bgzip region hand-over of ``_scan_sorted_region`` (no GPU needed)."""

from __future__ import annotations

import ctypes as C
import os

import numpy as np
import pytest

from helpers import GOLDEN


def _lists():
    return [os.path.join(GOLDEN, f"vcf_example_q.{g}.list") for g in ("ref", "tgt", "src")]


@pytest.mark.parametrize("ingest, inflate", [("host", "device"), ("device", "gpu"), ("host", "HOST"), ("device", None)])
def test_bad_inflate_arguments_raise(ingest, inflate):
    from sai_b200.configs import PloidyConfig, StatConfig
    from sai_b200.preprocessors import ChunkPreprocessor

    pc = PloidyConfig({"ref": {"R": 2}, "tgt": {"T": 2}, "src": {"S": 2}})
    with pytest.raises(ValueError, match="inflate"):
        ChunkPreprocessor(os.path.join(GOLDEN, "vcf_example_q.vcf"), *_lists(), None, 100, 100, "o.tsv", pc,
                          StatConfig({"U": {"ref": {"R": 0.3}, "tgt": {"T": 0.2}, "src": {"S": "=1"}}}),
                          ingest=ingest, inflate=inflate)


def _one_chrom_vcf(rng, n_rec, n_smp, final_newline):
    pos = np.sort(rng.choice(np.arange(1, 50 * n_rec), size=n_rec, replace=False))
    rows = ["##fileformat=VCFv4.1", "##x=" + "y" * 200,
            "#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(f"s{i}" for i in range(n_smp))]
    for p in pos:
        rows.append("\t".join(["1", str(p), ".", "A", "T", ".", "PASS", ".", "GT"]
                              + [f"{rng.integers(2)}|{rng.integers(2)}" for _ in range(n_smp)]))
    return ("\n".join(rows) + ("\n" if final_newline else "")).encode(), pos


def _lines_of(path, start, end, hook):
    """Text the region read hands over: `on_lines` buffers (complete lines consumed), or with `hook`
    the blocks it receives, host-inflated and cut the way the device feed cuts them."""
    from sai_b200 import _cabi
    from sai_b200.vcf import _scan_sorted_region

    got = []

    def on_lines(addr, length):
        b = C.string_at(addr, length)
        done = b.rfind(b"\n") + 1
        got.append(b[:done])
        return done

    def on_bgzf(base, block_off, out_off, n, skip, at_eof):
        assert out_off[0] == 0 and 0 <= skip <= out_off[n]
        text = np.empty(int(out_off[n]) + 1, dtype=np.uint8)
        b_off = np.ascontiguousarray(block_off - block_off[0]) if n else block_off
        if n:
            _cabi.check(_cabi.load().sai_bgzf_inflate(base + int(block_off[0]), b_off.ctypes.data, out_off.ctypes.data, n,
                                                      text.ctypes.data, 1))
        t = text[skip : int(out_off[n])].tobytes()
        if at_eof:
            t += b"\n" if t and not t.endswith(b"\n") else b""
        else:
            t = t[: t.rfind(b"\n") + 1]
        got.append(t)
        hooked.append(at_eof)

    hooked = []
    assert _scan_sorted_region(path, "1", start, end, lambda line: None, on_lines, on_bgzf=on_bgzf if hook else None)
    assert bool(hooked) == hook
    return b"".join(got)


@pytest.mark.parametrize("block, final_newline", [(64, True), (300, False), (5000, True)])
def test_region_hook_hands_over_the_same_text(tmp_path, block, final_newline):
    from sai_b200.vcf import write_bgzf

    rng = np.random.default_rng(block)
    text, pos = _one_chrom_vcf(rng, 150, 20, final_newline)
    path = str(tmp_path / "x.vcf.gz")
    write_bgzf(path, text, block=block)
    regions = [(1, int(pos[20])), (int(pos[40]) + 1, int(pos[90])), (int(pos[120]), int(pos[-1]) + 100),
               (int(pos[-1]) + 10, int(pos[-1]) + 90), (int(pos[0]), int(pos[-1]))]
    for start, end in regions:
        want = _lines_of(path, start, end, hook=False)
        assert _lines_of(path, start, end, hook=True) == want, (start, end)
        if start <= pos[0] and end >= pos[-1]:
            assert want.count(b"\n") == len(pos)
