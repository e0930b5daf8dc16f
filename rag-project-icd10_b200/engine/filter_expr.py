"""Milvus boolean ``filter`` expressions over the scalar columns of a collection (GPU-free).

``compile(expr)`` parses the subset of the Milvus expression grammar that the ICD schema needs; ``Predicate.mask(table,
lo, hi)`` evaluates it over rows [lo, hi) of an ``engine.store.ColumnTable`` as one bool per row, vectorised over the
mapped columns (no per-row Python: strings are compared as UTF-8 bytes gathered from the ``.str`` / ``.off`` arrays);
``pack_bits`` turns that into the row bitmap the scan kernels read (bit i & 31 of little-endian uint32 word i >> 5 =
row i may be returned; include/icdrag.h, icd_index_search_filtered).

Supported:
  fields     the schema's scalar fields and the primary key ``id`` (= row id); dynamic fields are not
  numeric    level, id:      == != < <= > >=, in [...], not in [...]
  string     code, ...:      == !=, in [...], not in [...], like "p%" / "%s" / "%i%" / "exact" (no ``_``, no inner ``%``)
  bool       has_complication:  == / != true | false
  logic      and / && , or / || , not / ! (keywords in any case), parentheses; precedence not > and > or
  literals   strings in " or ' with backslash escapes, integers and decimals, true / false
Anything else raises ValueError naming the problem.  An empty or all-blank expression is "no filter".
"""
from __future__ import annotations

import re
from typing import List, Optional, Sequence

import numpy as np

STR_FIELDS = ("code", "preferred_zh", "main_code", "secondary_code", "parent_code", "category_path", "semantic_text")
INT_FIELDS = ("level", "id")
BOOL_FIELDS = ("has_complication",)

_TOKEN = re.compile(r"""
    (?P<ws>\s+)
  | (?P<num>-?\d+(?:\.\d+)?(?:[eE][+-]?\d+)?)
  | (?P<str>"(?:[^"\\]|\\.)*"|'(?:[^'\\]|\\.)*')
  | (?P<op>==|!=|<=|>=|&&|\|\||<|>|!|\(|\)|\[|\]|,)
  | (?P<name>[A-Za-z_][A-Za-z0-9_]*)
""", re.VERBOSE | re.DOTALL)
_ESCAPES = {"n": "\n", "t": "\t", "r": "\r", "\\": "\\", "'": "'", '"': '"', "0": "\0"}
_KEYWORDS = {"and", "or", "not", "in", "like", "true", "false"}


class _Tok:
    __slots__ = ("kind", "value", "pos")

    def __init__(self, kind: str, value, pos: int):
        self.kind, self.value, self.pos = kind, value, pos

    def __repr__(self) -> str:
        return repr(self.value) if self.kind == "str" else str(self.value)


def _unescape(body: str, pos: int) -> str:
    out, i = [], 0
    while i < len(body):
        c = body[i]
        if c != "\\":
            out.append(c)
            i += 1
            continue
        e = body[i + 1]
        if e == "u":
            hexd = body[i + 2:i + 6]
            if not re.fullmatch(r"[0-9A-Fa-f]{4}", hexd):
                raise ValueError(f"filter: bad \\u escape in the string at offset {pos}")
            out.append(chr(int(hexd, 16)))
            i += 6
        else:
            out.append(_ESCAPES.get(e, e))
            i += 2
    return "".join(out)


def _tokenize(expr: str) -> List[_Tok]:
    toks, i = [], 0
    while i < len(expr):
        m = _TOKEN.match(expr, i)
        if m is None:
            if expr[i] in "\"'":
                raise ValueError(f"filter: unterminated string literal at offset {i}")
            raise ValueError(f"filter: unexpected character {expr[i]!r} at offset {i}")
        kind = m.lastgroup
        text = m.group(kind)
        if kind == "num":
            toks.append(_Tok("num", float(text) if any(c in text for c in ".eE") else int(text), i))
        elif kind == "str":
            toks.append(_Tok("str", _unescape(text[1:-1], i), i))
        elif kind == "op":
            toks.append(_Tok("op", text, i))
        elif kind == "name":
            low = text.lower()
            if low in _KEYWORDS:
                toks.append(_Tok("kw", low, i))
            else:
                toks.append(_Tok("name", text, i))
        i = m.end()
    return toks


# ---------------------------------------------------------------------------------------------- predicates
class Predicate:
    """A compiled filter.  ``mask(table, lo, hi)`` -> bool[hi - lo] for rows [lo, hi) of a ColumnTable."""

    is_all = False   # True only for the empty expression (no filter)

    def mask(self, table, lo: int = 0, hi: Optional[int] = None) -> np.ndarray:
        hi = len(table) if hi is None else int(hi)
        lo = int(lo)
        if not 0 <= lo <= hi <= len(table):
            raise ValueError(f"row range [{lo}, {hi}) outside the table's {len(table)} rows")
        return self._eval(table, lo, hi)

    def _eval(self, table, lo: int, hi: int) -> np.ndarray:
        raise NotImplementedError


class _All(Predicate):
    is_all = True

    def _eval(self, table, lo, hi):
        return np.ones(hi - lo, bool)


class _Not(Predicate):
    def __init__(self, a: Predicate):
        self.a = a

    def _eval(self, table, lo, hi):
        return ~self.a._eval(table, lo, hi)


class _And(Predicate):
    def __init__(self, a: Predicate, b: Predicate):
        self.a, self.b = a, b

    def _eval(self, table, lo, hi):
        return self.a._eval(table, lo, hi) & self.b._eval(table, lo, hi)


class _Or(Predicate):
    def __init__(self, a: Predicate, b: Predicate):
        self.a, self.b = a, b

    def _eval(self, table, lo, hi):
        return self.a._eval(table, lo, hi) | self.b._eval(table, lo, hi)


_NUM_OPS = {"==": np.equal, "!=": np.not_equal, "<": np.less, "<=": np.less_equal, ">": np.greater,
            ">=": np.greater_equal}


class _IntCmp(Predicate):
    """level / id against a number (op in _NUM_OPS) or a list of numbers (op 'in')."""

    def __init__(self, field: str, op: str, value):
        self.field, self.op, self.value = field, op, value

    def _eval(self, table, lo, hi):
        if self.field == "id":
            return self._eval_id(lo, hi)
        col = table.ints[self.field].view()[lo:hi]
        if self.op == "in":
            return np.isin(col, np.asarray(self.value, np.float64)) if self.value else np.zeros(hi - lo, bool)
        return _NUM_OPS[self.op](col, self.value)

    def _eval_id(self, lo, hi):
        # the row id is the position: ranges and index sets instead of a materialised arange
        out = np.zeros(hi - lo, bool)
        if self.op == "in":
            ids = np.asarray([v for v in self.value if float(v).is_integer()], np.int64)
            ids = ids[(ids >= lo) & (ids < hi)] - lo
            out[ids] = True
            return out
        v = self.value
        if self.op in ("==", "!="):
            if float(v).is_integer() and lo <= v < hi:
                out[int(v) - lo] = True
            return ~out if self.op == "!=" else out
        # smallest row id that satisfies id > v / id >= v, or one past the largest for < / <=
        import math
        if self.op == ">":
            first = math.floor(v) + 1
        elif self.op == ">=":
            first = math.ceil(v)
        elif self.op == "<":
            first = math.ceil(v)
        else:  # "<="
            first = math.floor(v) + 1
        cut = min(max(first - lo, 0), hi - lo)
        if self.op in (">", ">="):
            out[cut:] = True
        else:
            out[:cut] = True
        return out


class _BoolCmp(Predicate):
    def __init__(self, field: str, want: bool):
        self.field, self.want = field, want

    def _eval(self, table, lo, hi):
        col = table.bools[self.field].view()[lo:hi]
        return (col != 0) if self.want else (col == 0)


def _str_bounds(table, field: str, lo: int, hi: int):
    """(UTF-8 bytes of the column, start offsets [hi - lo], end offsets [hi - lo]) of rows [lo, hi)."""
    c = table.strs[field]
    off = c.off.view()
    data = c.data.view()
    ends = np.asarray(off[lo:hi], np.int64)
    starts = np.empty_like(ends)
    if hi > lo:
        starts[1:] = ends[:-1]
        starts[0] = int(off[lo - 1]) if lo > 0 else 0
    return data, starts, ends


def _match_at(data, pos: np.ndarray, pat: bytes, rows: np.ndarray) -> np.ndarray:
    """Rows of `rows` whose bytes at pos[...] equal `pat` (pos: byte offset of each candidate)."""
    for j, b in enumerate(pat):
        keep = data[pos + j] == b
        rows, pos = rows[keep], pos[keep]
        if rows.size == 0:
            break
    return rows


class _StrMatch(Predicate):
    """kind: 'eq' (the whole value), 'prefix', 'suffix', 'infix' against one UTF-8 pattern."""

    def __init__(self, field: str, kind: str, pat: str):
        self.field, self.kind, self.pat = field, kind, pat.encode("utf-8")

    def _eval(self, table, lo, hi):
        data, starts, ends = _str_bounds(table, self.field, lo, hi)
        lens = ends - starts
        L = len(self.pat)
        out = np.zeros(hi - lo, bool)
        if self.kind == "infix":
            return self._infix(data, starts, ends) if L else np.ones(hi - lo, bool)
        rows = np.nonzero(lens == L if self.kind == "eq" else lens >= L)[0]
        pos = ends[rows] - L if self.kind == "suffix" else starts[rows]
        out[_match_at(data, pos, self.pat, rows)] = True
        return out

    def _infix(self, data, starts, ends):
        n = starts.shape[0]
        out = np.zeros(n, bool)
        if n == 0:
            return out
        b0, b1 = int(starts[0]), int(ends[-1])
        L = len(self.pat)
        # every byte offset where the pattern starts, over the whole byte range of the rows at once
        pos = np.nonzero(data[b0:b1] == self.pat[0])[0].astype(np.int64) + b0
        pos = pos[pos + L <= b1]
        cand = np.arange(pos.size)
        hit = _match_at(data, pos, self.pat, cand)
        pos = pos[hit]
        row = np.searchsorted(ends, pos, side="right")          # the row whose bytes hold offset pos
        ok = pos + L <= ends[np.minimum(row, n - 1)]
        out[row[ok]] = True
        return out


class _StrIn(Predicate):
    def __init__(self, field: str, values: Sequence[str]):
        self.field = field
        self.parts = [_StrMatch(field, "eq", v) for v in dict.fromkeys(values)]

    def _eval(self, table, lo, hi):
        out = np.zeros(hi - lo, bool)
        for p in self.parts:
            out |= p._eval(table, lo, hi)
        return out


# ---------------------------------------------------------------------------------------------- parser
class _Parser:
    def __init__(self, expr: str):
        self.toks = _tokenize(expr)
        self.i = 0

    def peek(self) -> Optional[_Tok]:
        return self.toks[self.i] if self.i < len(self.toks) else None

    def take(self) -> _Tok:
        t = self.peek()
        if t is None:
            raise ValueError("filter: unexpected end of expression")
        self.i += 1
        return t

    def accept(self, kind: str, *values) -> Optional[_Tok]:
        t = self.peek()
        if t is not None and t.kind == kind and (not values or t.value in values):
            self.i += 1
            return t
        return None

    def expect(self, kind: str, value, what: str) -> _Tok:
        t = self.accept(kind, value)
        if t is None:
            got = self.peek()
            raise ValueError(f"filter: expected {what}, got {'end of expression' if got is None else repr(got)}"
                             + ("" if got is None else f" at offset {got.pos}"))
        return t

    def parse(self) -> Predicate:
        p = self.or_()
        t = self.peek()
        if t is not None:
            raise ValueError(f"filter: unexpected trailing token {t!r} at offset {t.pos}")
        return p

    def or_(self) -> Predicate:
        p = self.and_()
        while self.accept("kw", "or") or self.accept("op", "||"):
            p = _Or(p, self.and_())
        return p

    def and_(self) -> Predicate:
        p = self.not_()
        while self.accept("kw", "and") or self.accept("op", "&&"):
            p = _And(p, self.not_())
        return p

    def not_(self) -> Predicate:
        if self.accept("kw", "not") or self.accept("op", "!"):
            return _Not(self.not_())
        if self.accept("op", "("):
            p = self.or_()
            self.expect("op", ")", "')'")
            return p
        return self.comparison()

    def literal(self):
        t = self.take()
        if t.kind in ("num", "str"):
            return t.value
        if t.kind == "kw" and t.value in ("true", "false"):
            return t.value == "true"
        raise ValueError(f"filter: expected a literal, got {t!r} at offset {t.pos}")

    def literal_list(self) -> list:
        self.expect("op", "[", "'[' after 'in'")
        vals = []
        if self.accept("op", "]"):
            return vals
        while True:
            vals.append(self.literal())
            if self.accept("op", "]"):
                return vals
            self.expect("op", ",", "',' or ']' in the list")

    def comparison(self) -> Predicate:
        t = self.take()
        if t.kind != "name":
            raise ValueError(f"filter: expected a field name, got {t!r} at offset {t.pos}")
        field = t.value
        if field not in STR_FIELDS + INT_FIELDS + BOOL_FIELDS:
            raise ValueError(f"filter: unknown field {field!r} (dynamic fields cannot be filtered; scalar fields: "
                             f"{', '.join(('id',) + STR_FIELDS + ('level',) + BOOL_FIELDS)})")
        negate = False
        if self.accept("kw", "not"):
            self.expect("kw", "in", "'in' after 'not'")
            op, negate = "in", True
        elif self.accept("kw", "in"):
            op = "in"
        elif self.accept("kw", "like"):
            op = "like"
        else:
            o = self.take()
            if o.kind != "op" or o.value not in _NUM_OPS:
                raise ValueError(f"filter: expected a comparison operator after {field!r}, got {o!r} at offset {o.pos}")
            op = o.value
        value = self.literal_list() if op == "in" else self.literal()
        p = self._build(field, op, value)
        return _Not(p) if negate else p

    @staticmethod
    def _build(field: str, op: str, value) -> Predicate:
        vals = value if op == "in" else [value]
        if field in INT_FIELDS:
            if op == "like":
                raise ValueError(f"filter: 'like' needs a string field, {field!r} is numeric")
            bad = [v for v in vals if isinstance(v, (bool, str))]
            if bad:
                raise ValueError(f"filter: type mismatch: {field!r} is numeric, compared with {bad[0]!r}")
            return _IntCmp(field, op, list(value) if op == "in" else value)
        if field in BOOL_FIELDS:
            if op not in ("==", "!="):
                raise ValueError(f"filter: {field!r} is a bool field: only == and != with true / false")
            if not isinstance(value, bool):
                raise ValueError(f"filter: type mismatch: {field!r} is bool, compared with {value!r}")
            return _BoolCmp(field, value == (op == "=="))
        # string fields
        bad = [v for v in vals if not isinstance(v, str)]
        if bad:
            raise ValueError(f"filter: type mismatch: {field!r} is a string field, compared with {bad[0]!r}")
        if op == "in":
            return _StrIn(field, value)
        if op in ("==", "!="):
            p = _StrMatch(field, "eq", value)
            return _Not(p) if op == "!=" else p
        if op != "like":
            raise ValueError(f"filter: {op!r} is not supported on the string field {field!r} (== != in like)")
        if "_" in value:
            raise ValueError(f"filter: 'like' pattern {value!r}: the '_' wildcard is not supported")
        head, tail = value.startswith("%"), value.endswith("%") and len(value) > 1
        core = value[1 if head else 0:len(value) - (1 if tail else 0)]
        if "%" in core:
            raise ValueError(f"filter: 'like' pattern {value!r}: '%' is supported only at the start and/or the end")
        kind = "infix" if head and tail else "suffix" if head else "prefix" if tail else "eq"
        return _StrMatch(field, kind, core)


def compile(expr: Optional[str]) -> Predicate:   # noqa: A001 -- the name the module documents
    """Parse a filter expression; ValueError on anything outside the supported subset."""
    if expr is None or not str(expr).strip():
        return _All()
    if not isinstance(expr, str):
        raise ValueError(f"filter must be a string, got {type(expr).__name__}")
    return _Parser(expr).parse()


def pack_bits(bool_mask) -> np.ndarray:
    """bool[n] -> uint32[ceil(n / 32)]: bit i & 31 of word i >> 5 = row i (the scan kernels' row mask)."""
    m = np.ascontiguousarray(bool_mask, bool).reshape(-1)
    words = (m.size + 31) // 32
    b = np.zeros(words * 4, np.uint8)
    packed = np.packbits(m, bitorder="little")
    b[:packed.size] = packed
    return b.view("<u4").astype(np.uint32, copy=False)
