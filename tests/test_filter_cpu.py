"""Milvus `filter` expressions (engine/filter_expr.py) on the host: grammar, errors, bit packing, and the masks over the
real ICD-10 table against plain-Python predicates over the records."""
import importlib
import os
import re

import numpy as np
import pytest

from oracle import text as otext

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = importlib.import_module("rag-project-icd10_b200.engine.filter_expr")
S = importlib.import_module("rag-project-icd10_b200.engine.store")


def _table(rows):
    t = S.ColumnTable(None, 4)
    n = len(rows)
    t.stage(rows, np.zeros((n, 4), np.float32), np.zeros((n, 4), np.uint16), np.ones(n, np.uint8))
    t.commit()
    return t


@pytest.fixture(scope="module")
def records():
    return otext.load_records(os.path.join(ROOT, "data", "ICD_10v601.csv"))


@pytest.fixture(scope="module")
def icd(records):
    return _table(records)


SMALL = [
    dict(code="A00", preferred_zh="霍乱", level=1, has_complication=False, parent_code="", main_code="A00"),
    dict(code="A00.0", preferred_zh="古典生物型霍乱", level=2, has_complication=False, parent_code="A00"),
    dict(code="A01.0+G01*", preferred_zh='引号"和\\反斜杠', level=3, has_complication=True, parent_code="A01"),
    dict(code="J18.9", preferred_zh="肺炎", level=2, has_complication=False, parent_code="J18"),
    dict(code="", preferred_zh="", level=3, has_complication=True, parent_code="J18"),
]


@pytest.fixture(scope="module")
def small():
    return _table(SMALL)


def _ids(pred, table):
    return np.nonzero(pred.mask(table))[0].tolist()


@pytest.mark.parametrize("expr,want", [
    ("level == 2", [1, 3]), ("level != 2", [0, 2, 4]), ("level < 2", [0]), ("level <= 2", [0, 1, 3]),
    ("level > 2", [2, 4]), ("level >= 3", [2, 4]), ("level in [1, 3]", [0, 2, 4]), ("level not in [1, 3]", [1, 3]),
    ("level in []", []), ("level == 2.0", [1, 3]),
    ("id == 3", [3]), ("id != 3", [0, 1, 2, 4]), ("id < 2", [0, 1]), ("id <= 2", [0, 1, 2]), ("id > 2", [3, 4]),
    ("id >= 2", [2, 3, 4]), ("id in [4, 0, 99, -1]", [0, 4]), ("id not in [1]", [0, 2, 3, 4]), ("id > 1.5", [2, 3, 4]),
    ("id < -1", []), ("id >= 100", []),
    ('code == "A00"', [0]), ("code == 'A00'", [0]), ('code != "A00"', [1, 2, 3, 4]), ('code == ""', [4]),
    ('code in ["J18.9", "A00", "nope"]', [0, 3]), ('code not in ["J18.9", "A00"]', [1, 2, 4]),
    ('code like "A0%"', [0, 1, 2]), ('code like "%.9"', [3]), ('code like "%1.0%"', [2]), ('code like "A00"', [0]),
    ('code like "%"', [0, 1, 2, 3, 4]), ('code like "%%"', [0, 1, 2, 3, 4]), ('code like "%G01*"', [2]),
    ('preferred_zh like "%霍乱"', [0, 1]), ('preferred_zh == "肺炎"', [3]), ('preferred_zh like "古典%"', [1]),
    (r'preferred_zh == "引号\"和\\反斜杠"', [2]), (r"preferred_zh like '%\"和%'", [2]), (r'code == "A00"', [0]),
    ("has_complication == true", [2, 4]), ("has_complication == false", [0, 1, 3]), ("has_complication != true", [0, 1, 3]),
    ("has_complication == TRUE", [2, 4]),
    # logic, precedence (not > and > or), parentheses, keyword case and the symbolic forms
    ("level == 2 or level == 3 and has_complication == false", [1, 3]),
    ("(level == 2 or level == 3) and has_complication == false", [1, 3]),
    ("level == 1 or level == 3 and has_complication == true", [0, 2, 4]),
    ("(level == 1 or level == 3) and has_complication == true", [2, 4]),
    ("not level == 2 and id < 3", [0, 2]), ("not (level == 2 and id < 3)", [0, 2, 3, 4]),
    ("NOT level == 2 AND id < 3", [0, 2]), ("Not level == 2 Or id == 1", [0, 1, 2, 4]),
    ("!(level == 2) && id < 3", [0, 2]), ("level == 1 || id == 4", [0, 4]), ("!!(id == 1)", [1]),
    ('parent_code == "J18" && !(code like "J%")', [4]),
    ("  level == 1  ", [0]), ("((((id == 0))))", [0]),
])
def test_operators(small, expr, want):
    assert _ids(F.compile(expr), small) == want


@pytest.mark.parametrize("expr", ["", "   ", "\n\t", None])
def test_empty_expression_is_no_filter(small, expr):
    p = F.compile(expr)
    assert p.is_all and _ids(p, small) == [0, 1, 2, 3, 4]


@pytest.mark.parametrize("expr,msg", [
    ("foo == 1", "unknown field"), ("extra == 1", "unknown field"), ("vector == 1", "unknown field"),
    ("color == 'red'", "dynamic fields"),
    ('level == "3"', "type mismatch"), ("code == 3", "type mismatch"), ("has_complication == 1", "type mismatch"),
    ("level == true", "type mismatch"), ('level in [1, "2"]', "type mismatch"), ("code in ['A', 1]", "type mismatch"),
    ('code like "A_0%"', "'_' wildcard"), ('code like "A%0"', "start and/or the end"), ('code like "%A%0%"', "start and/or"),
    ('level like "3%"', "string field"), ("code < 'B'", "not supported"), ("has_complication > false", "bool field"),
    ("has_complication in [true]", "bool field"),
    ("level == 3 level == 2", "trailing"), ("level == 3)", "trailing"), ("(level == 3", "')'"), ("level ==", "end of expression"),
    ("level 3", "comparison operator"), ("== 3", "field name"), ("level == 3 and", "end of expression"),
    ('code == "A00', "unterminated"), ("level == 3 ; drop", "unexpected character"), ("level in 1", "'['"),
    ("level in [1 2]", "',' or ']'"), ("level not == 3", "'in' after 'not'"), ("level == level", "literal"),
    (r'code == "\u12"', "\\u escape"),
])
def test_errors_name_the_problem(expr, msg):
    with pytest.raises(ValueError, match=re.escape(msg)):
        F.compile(expr)


def test_pack_bits_layout():
    for n in (0, 1, 31, 32, 33, 64, 100, 1000):
        rng = np.random.default_rng(n)
        m = rng.random(n) < 0.5
        w = F.pack_bits(m)
        assert w.dtype == np.uint32 and w.shape == ((n + 31) // 32,)
        back = np.array([(w[i >> 5] >> (i & 31)) & 1 for i in range(n)], bool)
        assert np.array_equal(back, m)
        if n % 32:
            assert w[-1] >> (n % 32) == 0          # bits at or above n are clear
    assert F.pack_bits(np.array([1, 0, 0, 0, 0, 0, 0, 0, 0, 1] + [0] * 22 + [1], bool)).tolist() == [0x201, 1]
    assert F.pack_bits(np.ones(40, bool)).tolist() == [0xFFFFFFFF, 0xFF]


def test_icd_level_counts(icd):
    assert len(icd) == 40474
    for lv, n in ((1, 5031), (2, 12106), (3, 23337)):
        assert int(F.compile(f"level == {lv}").mask(icd).sum()) == n


ICD_EXPRS = [
    ('code like "J%"', lambda r, i: r["code"].startswith("J")),
    ("level == 3", lambda r, i: r["level"] == 3),
    ('parent_code == "A00.0"', lambda r, i: r["parent_code"] == "A00.0"),
    ("has_complication == false", lambda r, i: not r["has_complication"]),
    ('level == 3 and has_complication == false', lambda r, i: r["level"] == 3 and not r["has_complication"]),
    ('code like "%.9"', lambda r, i: r["code"].endswith(".9")),
    ('preferred_zh like "%结核%"', lambda r, i: "结核" in r["preferred_zh"]),
    ('semantic_text like "%ICD-10: A0%"', lambda r, i: "ICD-10: A0" in r["semantic_text"]),
    ('category_path like "A00 >%"', lambda r, i: r["category_path"].startswith("A00 >")),
    ('secondary_code != "" or main_code in ["A00", "B99"]', lambda r, i: r["secondary_code"] != "" or r["main_code"] in ("A00", "B99")),
    ('id >= 20000 and not (level in [2]) || code == "A00"', lambda r, i: (i >= 20000 and r["level"] != 2) or r["code"] == "A00"),
    ('preferred_zh == "霍乱"', lambda r, i: r["preferred_zh"] == "霍乱"),
]


@pytest.mark.parametrize("expr,fn", ICD_EXPRS, ids=[e for e, _ in ICD_EXPRS])
def test_icd_masks_equal_python_predicates(icd, records, expr, fn):
    want = np.array([bool(fn(r, i)) for i, r in enumerate(records)])
    got = F.compile(expr).mask(icd)
    assert got.dtype == bool and np.array_equal(got, want)
    assert want.any()


@pytest.mark.parametrize("expr", [e for e, _ in ICD_EXPRS])
def test_shard_ranges_are_slices_of_the_global_mask(icd, expr):
    p = F.compile(expr)
    full = p.mask(icd)
    n = len(icd)
    for lo, hi in ((0, 1), (0, n // 3), (n // 3, 2 * n // 3), (2 * n // 3, n), (12345, 12345), (777, 40001), (n - 1, n)):
        assert np.array_equal(p.mask(icd, lo, hi), full[lo:hi]), (lo, hi)
    with pytest.raises(ValueError):
        p.mask(icd, 0, n + 1)


def test_large_table_is_vectorised():
    """No per-row Python: a 4 M-row table (ints, id ranges, strings) evaluates in well under a second per expression."""
    import time
    n = 4_000_000
    t = S.ColumnTable(None, 1)
    t.n = n
    t.ints["level"]._map = np.tile(np.array([1, 2, 3, 3], "<i4"), n // 4)
    codes = np.frombuffer(b"J18.9A00.0", np.uint8)
    col = t.strs["code"]
    col.data._map = np.tile(codes, n // 2)
    col.off._map = (np.arange(1, n + 1, dtype=np.uint64) * 5)
    for expr, count in (("level == 3", n // 2), ("id >= 1000000", n - 1_000_000), ('code like "J%"', n // 2),
                        ('code == "A00.0"', n // 2), ('code like "%8.9%"', n // 2)):
        t0 = time.perf_counter()
        m = F.compile(expr).mask(t)
        dt = time.perf_counter() - t0
        assert int(m.sum()) == count, expr
        assert dt < 1.0, (expr, dt)
