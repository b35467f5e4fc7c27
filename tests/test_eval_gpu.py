"""dbx_eval_scalar (one fused kernel per expression) against the reference's printed results
(tests/golden/arithmetic.json) and against the CPU oracle on seeded random blocks: result type,
validity and every valid value bit for bit; first failing row and message for per-row errors."""
import json
import math
import os

import numpy as np
import pytest

from databend_b200 import abi
from databend_b200 import scalar_expr as sx
from databend_b200.block import Column, DataBlock, pack_bitmap

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "arithmetic.json")
DT = {"I8": abi.I8, "I16": abi.I16, "I32": abi.I32, "I64": abi.I64, "U8": abi.U8, "U16": abi.U16, "U32": abi.U32, "U64": abi.U64,
      "F32": abi.F32, "F64": abi.F64, "BOOL": abi.BOOL}
NAME = {v: k for k, v in DT.items()}
NP = {"I8": np.int8, "I16": np.int16, "I32": np.int32, "I64": np.int64, "U8": np.uint8, "U16": np.uint16, "U32": np.uint32, "U64": np.uint64,
      "F32": np.float32, "F64": np.float64}


def oracle():
    from oracle import eval_oracle
    return eval_oracle


@pytest.fixture(params=["jit", "interp"])
def eval_mode(request, monkeypatch):
    """Both builds of the evaluator: a straight-line kernel generated and compiled per expression
    (the default; run strict, DBX_EVAL_JIT=2, so that a kernel which fails to compile or launch fails
    the test instead of falling back to the interpreter), and the precompiled interpreter
    (DBX_EVAL_JIT=0)."""
    monkeypatch.setenv("DBX_EVAL_JIT", "2" if request.param == "jit" else "0")
    return request.param


def load_cases():
    with open(GOLD) as f:
        return json.load(f)


def to_sexpr(e):
    if e[0] == "col":
        return sx.col(e[1])
    if e[0] == "lit":
        return sx.lit(e[1], DT[e[2]])
    if e[0] == "cast":
        return sx.cast(to_sexpr(e[1]), DT[e[2]], bool(e[3]))
    return sx.call(e[1], *[to_sexpr(a) for a in e[2:]])


def to_tuple(e):
    if e[0] in ("col", "lit"):
        return tuple(e)
    if e[0] == "cast":
        return ("cast", to_tuple(e[1]), e[2], e[3])
    return ("call", e[1]) + tuple(to_tuple(a) for a in e[2:])


def make_column(t, values, valid):
    return Column.from_data(np.asarray(values, dtype=bool if t == "BOOL" else NP[t]), DT[t], validity=valid)


def block_of(cols, rows):
    if not cols:
        cols = [("U8", [0] * rows, None)]
    return DataBlock([make_column(t, v, valid) for t, v, valid in cols], rows)


def run_gpu(cols, rows, e):
    col, odt = sx.eval_scalar(block_of(cols, rows), to_sexpr(e))
    t = NAME[odt & ~abi.NULLABLE]
    vals = col.values()
    valid = col.valid_mask() if (col.validity is not None) else np.ones(rows, dtype=bool)
    return t, vals, valid


def assert_matches(t, vals, valid, et, evals, evalid, what):
    assert t == et, what
    np.testing.assert_array_equal(np.asarray(valid, dtype=bool), np.asarray(evalid, dtype=bool), err_msg=str(what))
    for r in range(len(evals)):
        if not evalid[r]:
            continue
        g, x = vals[r], evals[r]
        if t[0] == "F":
            x = NP[t](x)
            ok = (np.isnan(g) and np.isnan(x)) or np.asarray(g, NP[t]).tobytes() == np.asarray(x, NP[t]).tobytes() or (g == 0 and x == 0 and False)
            assert ok, (what, r, g, x)
        else:
            assert int(g) == int(x), (what, r, g, x)


@pytest.mark.parametrize("case", load_cases()["cases"], ids=lambda c: c["src"])
def test_reference_golden_outputs(gpu, eval_mode, case):
    cols = [(c["type"], [float(v) if c["type"][0] == "F" else v for v in c["values"]], c["valid"]) for c in case["columns"]]
    t, vals, valid = run_gpu(cols, case["rows"], case["expr"])
    assert t == case["out_type"], case["checked"]
    exp_valid = case["out_valid"] or [1] * case["rows"]
    np.testing.assert_array_equal(valid.astype(int), np.asarray(exp_valid[:case["rows"]], dtype=int), err_msg=case["checked"])
    for r in range(case["rows"]):
        if exp_valid[r]:
            g, x = vals[r], case["out_values"][r]
            if t[0] == "F":
                x = float(x)
                assert (math.isnan(g) and math.isnan(x)) or g == x or abs(g - x) <= 1e-12 * abs(x), (case["checked"], r, g, x)
            else:
                assert int(g) == int(x), (case["checked"], r, g, x)


@pytest.mark.parametrize("case", load_cases()["errors"], ids=lambda c: c["src"])
def test_reference_error_cases(gpu, eval_mode, case):
    cols = [(c["type"], c["values"], c["valid"]) for c in case["columns"]]
    with pytest.raises(sx.EvalError, match=case["error"]) as ei:
        run_gpu(cols, case["rows"], case["expr"])
    assert ei.value.row == case["row"]


EDGE = {"I8": [-128, 127, -1, 0, 1], "I16": [-32768, 32767, -1, 0, 1], "I32": [-2**31, 2**31 - 1, -1, 0, 1], "I64": [-2**63, 2**63 - 1, -1, 0, 1],
        "U8": [0, 1, 255, 128, 127], "U16": [0, 1, 65535, 32768], "U32": [0, 1, 2**32 - 1, 2**31], "U64": [0, 1, 2**64 - 1, 2**63, 2**63 + 1],
        "F32": [0.0, -0.0, 1.5, -2.5, 0.5, 3.4e38, float("nan"), float("inf"), -float("inf")],
        "F64": [0.0, -0.0, 1.5, -2.5, 0.5, 1e300, 9.3e18, -9.3e18, 2.5, 3.5, float("nan"), float("inf"), -float("inf")]}


def random_column(rng, t, rows, nullable):
    if t == "BOOL":
        v = rng.random(rows) < 0.5
    elif t[0] == "F":
        v = (rng.standard_normal(rows) * 10 ** rng.integers(0, 6, rows)).astype(NP[t])
    else:
        info = np.iinfo(NP[t])
        small = rng.integers(-20 if info.min < 0 else 0, 21, rows)
        wide = rng.integers(info.min, info.max, rows, dtype=NP[t], endpoint=True)
        v = np.where(rng.random(rows) < 0.6, small, wide).astype(NP[t])
    if t != "BOOL":
        k = min(rows, len(EDGE[t]))
        pos = rng.choice(rows, k, replace=False)
        v[pos] = np.asarray(EDGE[t][:k], dtype=NP[t])
    valid = (rng.random(rows) < 0.8).tolist() if nullable else None
    return (t, v.tolist(), valid)


NUM = ["I8", "I16", "I32", "I64", "U8", "U16", "U32", "U64", "F32", "F64"]


def check_against_oracle(cols, rows, e, what=None):
    eo = oracle()
    try:
        et, _, evals, evalid = eo.evaluate(to_tuple(e), cols)
    except eo.EvalFailure as f:
        with pytest.raises(sx.EvalError, match=f.msg) as ei:
            run_gpu(cols, rows, e)
        assert ei.value.row == f.row, (what or e, ei.value.row, f.row)
        return "error"
    t, vals, valid = run_gpu(cols, rows, e)
    assert_matches(t, vals, valid, et, evals, evalid, what or e)
    return "ok"


@pytest.mark.parametrize("fn", ["plus", "minus", "multiply", "divide", "div", "modulo"])
def test_binary_arithmetic_all_type_pairs(gpu, fn, eval_mode):
    """Every (left type, right type) pair of the ten numeric types, edge values and NULLs included;
    rows whose divisor is zero are exercised separately so that the value comparison runs too.
    (The generated-kernel build compiles one kernel per pair: it takes a third of the left types
    here; test_eval_matrix_gpu.py runs it on every pair.)"""
    rng = np.random.default_rng(sum(map(ord, fn)))
    rows = 257
    outcomes = set()
    for ta in (NUM if eval_mode == "interp" else ["I8", "U64", "F32"]):
        for tb in NUM:
            a = random_column(rng, ta, rows, nullable=True)
            b = random_column(rng, tb, rows, nullable=(ta != tb))
            e = ["call", fn, ["col", 0], ["col", 1]]
            outcomes.add(check_against_oracle([a, b], rows, e, (fn, ta, tb)))
            if fn in ("divide", "div", "modulo"):  # no zero divisors: values compared on every row
                bv = [x if x != 0 else 3 for x in b[1]]
                outcomes.add(check_against_oracle([a, (tb, bv, b[2])], rows, e, (fn, ta, tb, "nonzero")))
    assert "ok" in outcomes


def test_unary_and_casts_all_types(gpu, eval_mode):
    rng = np.random.default_rng(5)
    rows = 300
    for ta in (NUM if eval_mode == "interp" else ["I16", "U64", "F64"]):
        a = random_column(rng, ta, rows, nullable=True)
        check_against_oracle([a], rows, ["call", "negate", ["col", 0]], ("negate", ta))
        check_against_oracle([a], rows, ["call", "is_null", ["col", 0]])
        check_against_oracle([a], rows, ["call", "is_not_null", ["col", 0]])
        for to in NUM + ["BOOL"]:
            check_against_oracle([a], rows, ["cast", ["col", 0], to, 1], ("try_cast", ta, to))
            check_against_oracle([a], rows, ["cast", ["col", 0], to, 0], ("cast", ta, to))
    b = random_column(rng, "BOOL", rows, nullable=True)
    check_against_oracle([b], rows, ["call", "not", ["col", 0]])
    for to in NUM:
        check_against_oracle([b], rows, ["cast", ["col", 0], to, 0], ("cast bool", to))


def test_comparisons_and_three_valued_logic(gpu, eval_mode):
    rng = np.random.default_rng(6)
    rows = 500
    for t in NUM + ["BOOL"]:
        a, b = random_column(rng, t, rows, True), random_column(rng, t, rows, True)
        if t != "BOOL":
            b[1][:50] = a[1][:50]
        for fn in ("eq", "noteq", "lt", "lte", "gt", "gte"):
            check_against_oracle([a, b], rows, ["call", fn, ["col", 0], ["col", 1]], (fn, t))
    a, b = random_column(rng, "BOOL", rows, True), random_column(rng, "BOOL", rows, True)
    for fn in ("and", "or"):
        check_against_oracle([a, b], rows, ["call", fn, ["col", 0], ["col", 1]])
        check_against_oracle([a, (b[0], b[1], None)], rows, ["call", fn, ["col", 0], ["col", 1]])


def test_nested_expression_one_kernel(gpu, eval_mode):
    """(a * b + c) % 7 > cast(d / 3 as Int32) and not(is_null(c)): one launch for the tree (plus the
    bit-packing launches), inputs read once."""
    from databend_b200.lib import load

    def launch_count():
        return load().dbx_kernel_launch_count()
    rng = np.random.default_rng(8)
    rows = 100_000
    cols = [random_column(rng, "I16", rows, False), random_column(rng, "U8", rows, True), random_column(rng, "I32", rows, True),
            ("F64", (rng.standard_normal(rows) * 1000).tolist(), None)]
    e = ["call", "and",
         ["call", "gt",
          ["cast", ["call", "modulo", ["call", "plus", ["call", "multiply", ["col", 0], ["col", 1]], ["col", 2]], ["lit", 7, "U8"]], "I64", 0],
          ["cast", ["cast", ["call", "divide", ["col", 3], ["lit", 3, "U8"]], "I32", 0], "I64", 0]],
         ["call", "not", ["call", "is_null", ["col", 2]]]]
    before = launch_count()
    assert check_against_oracle(cols, rows, e) == "ok"
    assert launch_count() - before <= 3


def test_error_is_first_failing_valid_row_and_null_rows_do_not_raise(gpu, eval_mode):
    a = ("I32", [5, 6, 7, 8], None)
    b = ("I32", [1, 0, 0, 2], [1, 0, 1, 1])
    with pytest.raises(sx.EvalError, match="Division by zero") as ei:
        run_gpu([a, b], 4, ["call", "modulo", ["col", 0], ["col", 1]])
    assert ei.value.row == 2
    b = ("I32", [1, 0, 5, 2], [1, 0, 1, 1])
    t, vals, valid = run_gpu([a, b], 4, ["call", "div", ["col", 0], ["col", 1]])
    assert t == "I32" and valid.tolist() == [True, False, True, True] and [int(vals[i]) for i in (0, 2, 3)] == [5, 1, 4]
    with pytest.raises(sx.EvalError, match="number overflowed"):
        run_gpu([("F64", [1.0, 300.0], None)], 2, ["cast", ["col", 0], "U8", 0])
    t, vals, valid = run_gpu([("F64", [1.4, 300.0, 254.5, -0.4], None)], 4, ["cast", ["col", 0], "U8", 1])
    assert valid.tolist() == [True, False, True, True] and [int(vals[0]), int(vals[2]), int(vals[3])] == [1, 255, 0]


def test_empty_block_and_device_resident_input(gpu, eval_mode):
    from databend_b200.transforms import to_device
    t, vals, valid = run_gpu([("I32", [], None)], 0, ["call", "plus", ["col", 0], ["lit", 1, "U8"]])
    assert t == "I64" and len(vals) == 0
    rng = np.random.default_rng(9)
    rows = 70_001
    a = rng.integers(-1000, 1000, rows).astype(np.int32)
    b = rng.integers(1, 1000, rows).astype(np.int64)
    blk = DataBlock([to_device(Column(abi.I32, rows, data=a)), to_device(Column(abi.I64, rows, data=b))], rows)
    col, odt = sx.eval_scalar(blk, sx.col(0) % sx.col(1))
    exp = np.fmod(a.astype(np.int64), b)
    np.testing.assert_array_equal(col.values(), exp)
