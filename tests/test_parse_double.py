"""The score-file cell parser of the device outlier path (sai_b200/csrc/parse_double.cuh), host build:
its float parser gives read_csv's bits (pandas' precise_xstrtod, which does not round correctly), and
its cell classes give pandas' dtype of a column, or say that they cannot."""

import io
import warnings

import numpy as np
import pandas as pd

from sai_b200 import _cabi
from sai_b200.outlier import column_kinds, pandas_chunk_rows
from sai_b200.scoring import classify_cells_host, parse_doubles_host


def _read_column(strings):
    text = "x\n" + "\n".join(s.decode() for s in strings) + "\n"
    return pd.read_csv(io.StringIO(text), sep="\t", na_values=["nan"], index_col=False, low_memory=False)["x"]


def _check_bits(strings):
    got, ok = parse_doubles_host(strings)
    assert ok.all(), [s for s, k in zip(strings, ok) if not k][:10]
    col = _read_column(strings)
    assert col.dtype == np.float64
    exp = col.to_numpy()
    bad = np.flatnonzero(got.view(np.uint64) != exp.view(np.uint64))
    assert bad.size == 0, [(strings[i], got[i], exp[i]) for i in bad[:10]]


def test_repr_of_random_bit_patterns_and_unit_interval():
    rng = np.random.default_rng(20261022)
    bits = rng.integers(0, 2**64, size=1_000_000, dtype=np.uint64).view(np.float64)
    bits = bits[np.isfinite(bits)]
    _check_bits([repr(float(v)).encode() for v in bits])
    _check_bits([repr(float(v)).encode() for v in rng.random(1_000_000)])


def test_long_digit_strings():
    rng = np.random.default_rng(3)
    out = []
    for _ in range(600_000):
        nd = int(rng.integers(18, 26))
        digits = "".join(map(str, rng.integers(0, 10, size=nd)))
        point = int(rng.integers(0, nd + 1))
        s = digits[:point] + "." + digits[point:]
        if rng.random() < 0.5:
            s += f"e{int(rng.integers(-40, 40))}"
        out.append(("-" if rng.random() < 0.3 else "") + s)
    _check_bits([s.encode() for s in out])


def test_exponents_across_subnormals_and_overflow():
    rng = np.random.default_rng(11)
    strings = []
    for e in range(-330, 311):
        for _ in range(1500):
            m = rng.random() * 10
            strings.append(f"{m:.{int(rng.integers(1, 19))}f}e{e}".encode())
    got, ok = parse_doubles_host(strings)
    _check_bits([s for s, k in zip(strings, ok) if k])
    # a value that overflows is a range error of the parser, which pandas turns into an infinity;
    # the device path leaves such cells to the host (they classify as unsure)
    over = [s for s, k in zip(strings, ok) if not k]
    assert over and all(np.isinf(got[~ok]))
    assert np.isinf(_read_column(over).to_numpy()).all()
    assert set(classify_cells_host(over[:2000]).tolist()) == {_cabi.CELL_UNSURE}


def test_spellings_and_big_integers():
    rng = np.random.default_rng(5)
    big = [str(int(v)).encode() for v in rng.integers(2**53, 2**63 - 1, size=200_000, dtype=np.int64)]
    big += [b"-" + s for s in big[:50_000]]
    fixed = [b"0", b"-0", b"-0.0", b"5.", b".5", b"-.5", b"-5.", b"000123", b"00.00100", b"1e3", b"1E3", b"1e+3",
             b"1e-3", b"0e0", b"12345678901234567890123", b"0.000000000000000000000000001",
             b"9007199254740993", b"99999999999999999", b"1.7976931348623157e308", b"4.9e-324", b"2e-324",
             b"1e-400", b"-1e-700"]
    _check_bits(big + fixed + [b"0.5"])


CELLS = {
    "int": [b"5", b"-3", b"005", b"-0", b"9223372036854775807", b"-9223372036854775808", b"9007199254740993", b"12",
            b"0000000000000000012", b"-000000000000000000000123", b"00000000000000000"],
    "float": [b"1.5", b"-2e-3", b"5.", b".5", b"1E3", b"inf", b"-inf", b"0.1234567890123456789", b"1e-320"],
    "na": [b"", b"nan", b"NA", b"NaN", b"null", b"-nan", b"#N/A", b"N/A", b"<NA>", b"None", b"1.#IND"],
    "text": [b"chr1", b"0x10", b"1d3", b"abc", b"1e5x", b"X", b"chrUn_gl000220", b"--1x"],
    "unsure": [b"+5", b" 5", b"5 ", b"True", b"false", b"TRUE", b"Infinity", b"INF", b"-Inf", b"9223372036854775808",
               b"1.#INF", b"e", b"1e", b"-", b"NAN", b"1e+", b"1e99999", b"1e309", b"--1", b"1.2.3"],
}


def test_cell_classes():
    cls = {k: classify_cells_host(v) for k, v in CELLS.items()}
    assert set(cls["int"].tolist()) == {_cabi.CELL_INT, _cabi.CELL_INT | _cabi.CELL_BIGINT, _cabi.CELL_INT | _cabi.CELL_NEGZERO}
    assert set(cls["float"].tolist()) == {_cabi.CELL_FLOAT}
    assert set(cls["na"].tolist()) == {_cabi.CELL_NA}
    assert set(cls["text"].tolist()) == {_cabi.CELL_TEXT}
    assert set(cls["unsure"].tolist()) == {_cabi.CELL_UNSURE}


def test_random_columns_get_pandas_dtype():
    rng = np.random.default_rng(17)
    pool = [(k, s) for k, v in CELLS.items() for s in v]
    kind_of = {_cabi.TABLE_INT: "i", _cabi.TABLE_FLOAT: "f", _cabi.TABLE_TEXT: "O"}
    checked = unsure = 0
    for _ in range(3000):
        cells = [pool[i][1] for i in rng.integers(0, len(pool), size=int(rng.integers(1, 7)))]
        classes = classify_cells_host(cells).astype(np.uint32)
        kinds, reason = column_kinds(np.bitwise_or.reduce(classes)[None, None])
        text = "k\tx\n" + "".join(f"{i}\t{c.decode()}\n" for i, c in enumerate(cells))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            col = pd.read_csv(io.StringIO(text), sep="\t", na_values=["nan"], index_col=False)["x"]
        if kinds is None:
            unsure += 1
            continue
        checked += 1
        dt = col.dtype.kind if hasattr(col.dtype, "kind") else "O"
        assert dt == kind_of[kinds[0]], (cells, col.dtype)
        if kinds[0] == _cabi.TABLE_FLOAT:
            vals, _ = parse_doubles_host(cells)
            vals[[c == b"inf" for c in cells]] = np.inf  # spelled out, not parsed
            vals[[c == b"-inf" for c in cells]] = -np.inf
            na = np.array([c in CELLS["na"] for c in cells])
            vals[na] = np.nan
            assert np.array_equal(vals.view(np.uint64)[~na], col.to_numpy()[~na].view(np.uint64)), cells
            assert np.isnan(col.to_numpy()[na]).all()
    assert checked > 500 and unsure > 100


def test_chunk_rows_is_pandas_parse_chunk():
    # an int64 chunk followed by one with a text cell: pandas keeps the ints as ints, with a DtypeWarning
    for n_cols in (3, 13):
        rows = pandas_chunk_rows(n_cols)
        hdr = "\t".join(f"c{i}" for i in range(n_cols))
        tail = "\t1" * (n_cols - 1)
        for n_int, mixed in ((rows - 1, False), (rows, True)):
            text = hdr + "\n" + f"5{tail}\n" * n_int + f"x{tail}\n"
            with warnings.catch_warnings(record=True) as w:
                warnings.simplefilter("always")
                col = pd.read_csv(io.StringIO(text), sep="\t", na_values=["nan"], index_col=False)["c0"]
            assert isinstance(col.iloc[0], int) == mixed
            assert any(issubclass(x.category, pd.errors.DtypeWarning) for x in w) == mixed


def test_zero_padded_integers_leave_float_columns_to_the_host():
    # more than 17 digits: pandas' float parser drops the digits after the 17th, its int64 path does
    # not, and which one a float64 column's integers go through depends on the chunk
    cells = [b"0000000000000000012", b"nan", b"3"]
    assert classify_cells_host(cells)[0] == _cabi.CELL_INT | _cabi.CELL_BIGINT
    assert parse_doubles_host(cells[:1])[0][0] == 0.0 and _read_column(cells).iloc[0] == 12.0
    assert column_kinds(np.bitwise_or.reduce(classify_cells_host(cells).astype(np.uint32))[None, None])[0] is None
    assert column_kinds(classify_cells_host([b"0000000000000000012"]).astype(np.uint32)[None, :])[0] == [_cabi.TABLE_INT]


def test_column_kinds_across_chunks():
    I, F, N, T, B = _cabi.CELL_INT, _cabi.CELL_FLOAT, _cabi.CELL_NA, _cabi.CELL_TEXT, _cabi.CELL_BIGINT
    kinds, _ = column_kinds(np.array([[I, I | N, N, T | N], [I, F, N, T]], dtype=np.uint32))
    assert kinds == [_cabi.TABLE_INT, _cabi.TABLE_FLOAT, _cabi.TABLE_FLOAT, _cabi.TABLE_TEXT]
    assert column_kinds(np.array([[I], [I | F]], dtype=np.uint32))[0] == [_cabi.TABLE_FLOAT]
    assert column_kinds(np.array([[I | B], [F]], dtype=np.uint32))[0] is None
    assert column_kinds(np.array([[I | B | N]], dtype=np.uint32))[0] is None
    assert column_kinds(np.array([[I | B]], dtype=np.uint32))[0] == [_cabi.TABLE_INT]
    assert column_kinds(np.array([[I | _cabi.CELL_NEGZERO], [I]], dtype=np.uint32))[0] == [_cabi.TABLE_INT]
    assert column_kinds(np.array([[I | _cabi.CELL_NEGZERO], [F]], dtype=np.uint32))[0] is None
    assert column_kinds(np.array([[I], [T]], dtype=np.uint32))[0] is None
    assert column_kinds(np.array([[N], [T]], dtype=np.uint32))[0] is None
    assert column_kinds(np.array([[I | _cabi.CELL_UNSURE]], dtype=np.uint32))[0] is None
