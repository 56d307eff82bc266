"""`outlier(..., text="device")`: the score file parsed and the outlier tables built as text on the GPU
give the files, warnings and errors of the host path, byte for byte; files the device path does not
reproduce go to the host path.  HostEngine.outlier_calls tells which path ran."""

import os
import socket
import warnings

import numpy as np
import pytest

from helpers import GOLDEN

pytestmark = pytest.mark.gpu

QS = [0, 0.25, 0.5, 0.9, 0.99, 1]


def _run(path, prefix, q, text):
    from sai_b200.outlier import outlier

    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        try:
            outlier(str(path), str(prefix), q, text=text)
            err = None
        except Exception as e:  # noqa: BLE001 -- compared between the two paths
            err = (type(e), str(e))
    files = {}
    d, base = os.path.split(str(prefix))
    for f in sorted(os.listdir(d)):
        if f.startswith(base + "."):
            files[f[len(base):]] = open(os.path.join(d, f), "rb").read()
    return files, [str(x.message) for x in w if issubclass(x.category, UserWarning)], err


def _both(tmp_path, path, q, device_path=True):
    from sai_b200.outlier import fallback_reason
    from sai_b200.scoring import HostEngine

    assert (fallback_reason(str(path), q) is None) == device_path, fallback_reason(str(path), q)

    (tmp_path / "h").mkdir(exist_ok=True)
    (tmp_path / "d").mkdir(exist_ok=True)
    for sub in ("h", "d"):
        for f in os.listdir(tmp_path / sub):
            os.remove(tmp_path / sub / f)
    host = _run(path, tmp_path / "h" / "o", q, "host")
    calls = HostEngine.outlier_calls
    dev = _run(path, tmp_path / "d" / "o", q, "device")
    assert HostEngine.outlier_calls == calls + device_path  # counts the tables built on the device
    assert dev[2] == host[2]
    assert dev[1] == host[1]
    assert dev[0].keys() == host[0].keys()
    for k in host[0]:
        assert dev[0][k] == host[0][k], k
    return host


def test_device_parser_equals_host_build():
    from sai_b200.scoring import HostEngine, parse_doubles_host

    rng = np.random.default_rng(8)
    bits = rng.integers(0, 2**64, size=4_000_000, dtype=np.uint64).view(np.float64)
    strings = [repr(float(v)).encode() for v in bits[np.isfinite(bits)]]
    strings += [repr(float(v)).encode() for v in rng.random(3_000_000)]
    m = rng.integers(0, 10**18, size=3_000_000, dtype=np.int64)
    e = rng.integers(-330, 311, size=m.size)
    strings += [f"{a}.{a % 1000}e{b}".encode() for a, b in zip(m.tolist(), e.tolist())]
    eng = HostEngine(0)
    got, ok = eng.parse_doubles(strings)
    eng.close()
    exp, eok = parse_doubles_host(strings)
    assert np.array_equal(ok, eok)
    assert np.array_equal(got.view(np.uint64), exp.view(np.uint64))


def test_reference_golden_tables(tmp_path):
    d = os.path.join(GOLDEN, "outlier_example")
    files, _, err = _both(tmp_path, os.path.join(d, "scores.tsv"), 0.9)
    assert err is None
    expected = sorted(f for f in os.listdir(d) if f.startswith("expected."))
    assert len(expected) == 12
    for f in expected:
        col = f[len("expected."): -len(".0.9.outliers.tsv")]
        assert files[f".{col}.0.9.outliers.tsv"] == open(os.path.join(d, f), "rb").read(), col


@pytest.mark.parametrize("q", [0.25, 0.75])
def test_reference_unit_test_file(tmp_path, q):
    _both(tmp_path, os.path.join(GOLDEN, "outlier_q.scores"), q)


def test_degenerate_columns_warn_alike(tmp_path):
    p = tmp_path / "s.tsv"
    p.write_text("Chrom\tStart\tEnd\tRef\tTgt\tSrc\tOutgroup\tN(Variants)\tU\tQ\tZ\tW\n"
                 "1\t1\t10\tA\tB\tC\tNA\t5\t2\tnan\tnan\t-0.0\n"
                 "1\t11\t20\tA\tB\tC\tNA\t5\t2\tnan\t-0.0\t0.0\n"
                 "1\t21\t30\tA\tB\tC\tNA\t5\t2\tnan\t0.0\t-0.0\n")
    _, warned, _ = _both(tmp_path, p, 0.99)
    assert len(warned) == 4 and "(-0.0)" in warned[2] and "(-0.0)" in warned[3]


NAMES = ["chr1", "1", "chr10", "chr2", "chrUn_gl000220", "chrX", "2", "10", "chr01"]


def _adversarial(path, rng, n_runs=60, n_tgt=3):
    """Runs of mixed-order chromosome names, rows tied on (Chrom, Start, End) across targets,
    integer columns with one NaN, all-NaN and NA text columns, inf, 17+ digit floats."""
    lines = ["Chrom\tStart\tEnd\tRef\tTgt\tSrc\tOutgroup\tN(Variants)\tU\tQ\tUint\tNoVal\tDplus\tfd\tBig"]
    for _ in range(n_runs):
        chrom = NAMES[int(rng.integers(len(NAMES)))]
        starts = rng.integers(0, 10**6, size=int(rng.integers(1, 40)))
        for tgt in range(n_tgt):
            for s in starts.tolist():
                u = int(rng.integers(0, 30))
                q = rng.random()
                qs = ["nan", "inf", repr(q), f"{q:.20f}", "5.", ".5", "1e-5", "0"][int(rng.integers(8)) if rng.random() < 0.3 else 2]
                lines.append("\t".join([chrom, str(s), str(s + int(rng.integers(0, 3)) * 1000), "AFR", f"T{tgt}", "NEA", "NA",
                                        str(int(rng.integers(0, 99))), str(u) if rng.random() > 0.01 else "nan", qs,
                                        str(u), "nan", repr(-rng.random()), f"{rng.normal() * 1e5:.17g}",
                                        f"{rng.random():.25f}"]))
    path.write_text("\n".join(lines) + "\n")


@pytest.mark.parametrize("q", QS)
def test_adversarial_files(tmp_path, q):
    rng = np.random.default_rng(int(q * 100))
    p = tmp_path / "s.tsv"
    _adversarial(p, rng)
    from sai_b200.outlier import fallback_reason

    assert fallback_reason(str(p), q) is None
    files, _, err = _both(tmp_path, p, q)
    assert err is None and len(files) == 7


def test_multi_chromosome_file_larger_than_a_parse_chunk(tmp_path):
    """~300 k rows: several pandas parse chunks, thousands of radix tiles."""
    rng = np.random.default_rng(9)
    n = 300_000
    chrom = np.repeat([f"chr{i}" for i in (1, 2, 10, 11, 3, 22, 4)], n // 7 + 1)[:n]
    start = rng.integers(0, 2**40, size=n)
    vals = rng.random((n, 3))
    vals[rng.random(n) < 0.05, 1] = np.nan
    start, vals = start.tolist(), vals.tolist()  # Python ints and floats: repr() prints the bare number
    with open(tmp_path / "s.tsv", "w") as f:
        f.write("Chrom\tStart\tEnd\tRef\tTgt\tSrc\tN(Variants)\tU\tQ\tD\n")
        for i in range(n):
            f.write(f"{chrom[i]}\t{start[i]}\t{start[i] + 50000}\tAFR\tEUR\tNEA\t{i % 97}\t{int(vals[i][0] * 40)}\t"
                    f"{vals[i][1]!r}\t{vals[i][2] - 0.5!r}\n")
    for q in (0.9, 0.99):
        _both(tmp_path, tmp_path / "s.tsv", q)


HEADER = "Chrom\tStart\tEnd\tRef\tTgt\tSrc\tN(Variants)\tU\tQ\n"
ROWS = ["chr1\t1\t10\tA\tB\tC\t5\t2\t0.5\n", "chr2\t11\t20\tA\tB\tC\t5\t3\t0.7\n", "chr1\t21\t30\tA\tB\tC\t5\t4\t0.9\n"]
FALLBACKS = {
    "unsure cell": HEADER + ROWS[0] + ROWS[1].replace("\t3\t", "\t+3\t") + ROWS[2],
    "bool cell": HEADER + ROWS[0] + ROWS[1].replace("\t3\t", "\tTrue\t") + ROWS[2],
    "ragged row": HEADER + ROWS[0] + ROWS[1].replace("\n", "\t1\n") + ROWS[2],
    "short row": HEADER + ROWS[0] + ROWS[1].replace("\t0.7\n", "\n") + ROWS[2],
    "blank line": HEADER + ROWS[0] + "\n" + ROWS[1] + ROWS[2],
    "carriage return": (HEADER + "".join(ROWS)).replace("\n", "\r\n"),
    "quote": HEADER + ROWS[0] + ROWS[1].replace("\tA\t", '\t"A"\t') + ROWS[2],
    "high byte": HEADER + ROWS[0] + ROWS[1].replace("\tA\t", "\té\t") + ROWS[2],
    "duplicate names": HEADER.replace("Ref", "Tgt") + "".join(ROWS),
    "empty name": HEADER.replace("Ref", "") + "".join(ROWS),
    "no N(Variants)": HEADER.replace("N(Variants)", "N") + "".join(ROWS),
    "Chrom with NA": HEADER + ROWS[0] + ROWS[1].replace("chr2", "NA") + ROWS[2],
    "Start not int64": HEADER + ROWS[0] + ROWS[1].replace("\t11\t", "\t11.5\t") + ROWS[2],
    "no Chrom": HEADER.replace("Chrom", "Chr") + "".join(ROWS),
    "long line": HEADER + ROWS[0] + ROWS[1].replace("\tA\t", "\t" + "A" * 70000 + "\t") + ROWS[2],
    "text metric": HEADER + ROWS[0] + ROWS[1].replace("\t0.7\n", "\tx\n") + ROWS[2],
    "header only": HEADER,
    "zero-padded integer in a float column": HEADER + ROWS[0].replace("\t2\t", "\t0000000000000000012\t")
    + ROWS[1].replace("\t3\t", "\tnan\t") + ROWS[2].replace("\t4\t", "\t3\t"),
}


@pytest.mark.parametrize("case", sorted(FALLBACKS))
def test_fallbacks_take_the_host_path(tmp_path, case):
    from sai_b200.outlier import device_outlier, fallback_reason

    p = tmp_path / "s.tsv"
    p.write_bytes(FALLBACKS[case].encode())
    assert fallback_reason(str(p), 0.5) is not None
    assert not device_outlier(str(p), str(tmp_path / "x"), 0.5)
    assert not any(f.startswith("x.") for f in os.listdir(tmp_path))
    _both(tmp_path, p, 0.5, device_path=False)


def test_plain_file_without_final_newline_and_int_chrom(tmp_path):
    from sai_b200.outlier import fallback_reason

    p = tmp_path / "s.tsv"
    p.write_text(HEADER + "".join(r.replace("chr", "") for r in ROWS + ROWS).rstrip("\n"))
    assert fallback_reason(str(p), 0.5) is None
    _both(tmp_path, p, 0.5)


def test_bad_text_value_raises():
    from sai_b200.outlier import outlier

    with pytest.raises(ValueError, match="text must be"):
        outlier("unused", "unused", 0.5, text="gpu")


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _nccl_worker(rank, world, port, d):
    import torch
    import torch.distributed as dist

    from sai_b200.outlier import outlier
    from sai_b200.scoring import HostEngine

    torch.cuda.set_device(rank)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        shard = os.path.join(d, f"shard{rank}.tsv")
        for text in ("host", "device"):
            calls = HostEngine.outlier_calls
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                outlier(shard, os.path.join(d, f"{text}{rank}"), 0.9, text=text, device=rank)
            assert (HostEngine.outlier_calls > calls) == (text == "device")
    finally:
        dist.destroy_process_group()


def test_nccl_two_gpus_match_host_path(tmp_path):
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    rng = np.random.default_rng(4)
    for r in range(2):
        _adversarial(tmp_path / f"shard{r}.tsv", rng, n_runs=30 + 20 * r)
    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    for r in range(2):
        host = sorted(f for f in os.listdir(tmp_path) if f.startswith(f"host{r}."))
        assert len(host) == 7
        for f in host:
            assert (tmp_path / f).read_bytes() == (tmp_path / f.replace("host", "device", 1)).read_bytes(), f
