"""The expression oracle (oracle/eval_oracle.py) against the reference's own printed results:
tests/golden/arithmetic.json is transcribed from functions/tests/it/scalars/testdata/
{arithmetic,cast,boolean,comparison}.txt by tests/golden/make_arith_golden.py."""
import json
import math
import os

import pytest

from oracle import eval_oracle as eo

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "arithmetic.json")


def load_cases():
    with open(GOLD) as f:
        return json.load(f)


def tree(e):
    """json lists -> the tuples eval_oracle takes."""
    if e[0] == "col":
        return ("col", e[1])
    if e[0] == "lit":
        return ("lit", e[1], e[2])
    if e[0] == "cast":
        return ("cast", tree(e[1]), e[2], e[3])
    return ("call", e[1]) + tuple(tree(a) for a in e[2:])


def columns_of(case):
    cols = [(c["type"], [float(v) if c["type"][0] == "F" else v for v in c["values"]], c["valid"]) for c in case["columns"]]
    if not cols:
        cols = [("U8", [0] * case["rows"], None)]
    return cols


def same_value(t, got, exp):
    if t[0] == "F":
        exp = float(exp)
        return (math.isnan(got) and math.isnan(exp)) or got == exp or abs(got - exp) <= 1e-12 * abs(exp)  # the golden prints shortest round-trip digits
    return int(got) == int(exp)


@pytest.mark.parametrize("case", load_cases()["cases"], ids=lambda c: c["src"])
def test_oracle_matches_reference_output(case):
    t, nullable, vals, oks = eo.evaluate(tree(case["expr"]), columns_of(case))
    assert t == case["out_type"], case["checked"]
    exp_valid = case["out_valid"] or [1] * case["rows"]
    assert [int(o) for o in oks] == [int(v) for v in exp_valid[:case["rows"]]], case["checked"]
    for r in range(case["rows"]):
        if exp_valid[r]:
            assert same_value(t, vals[r], case["out_values"][r]), (case["checked"], r, vals[r], case["out_values"][r])


@pytest.mark.parametrize("case", load_cases()["errors"], ids=lambda c: c["src"])
def test_oracle_raises_reference_errors(case):
    with pytest.raises(eo.EvalFailure) as ei:
        eo.evaluate(tree(case["expr"]), columns_of(case))
    assert ei.value.msg == case["error"] and ei.value.row == case["row"]


def test_result_type_table():
    """arithmetics_type.rs:240-265 spot checks (the golden outputs' types cover the rest)."""
    assert eo.t_add_mul("I8", "I16") == "I32" and eo.t_add_mul("U8", "U8") == "U16" and eo.t_add_mul("U64", "I8") == "I64"
    assert eo.t_minus("U8", "U8") == "I16" and eo.t_minus("U32", "F64") == "F64"
    assert eo.t_intdiv("U32", "F64") == "I64" and eo.t_intdiv("U8", "U32") == "U32"
    assert eo.t_modulo("I8", "I8") == "I16" and eo.t_modulo("U16", "U8") == "U8" and eo.t_modulo("U8", "I8") == "U8"
    assert eo.t_negate("U8") == "I16" and eo.t_negate("F32") == "F32" and eo.t_negate("U64") == "I64"


def test_sort_oracle_matches_reference_golden_permutations():
    """oracle/sort_oracle.py (multi-column ORDER BY restatement) on the reference's single-key sort
    goldens (tests/golden/sort.json, from expression/tests/it/sort.rs)."""
    import numpy as np
    from oracle import sort_oracle
    with open(os.path.join(os.path.dirname(GOLD), "sort.json")) as f:
        cases = json.load(f)["cases"]
    np_dt = {"I64": np.int64, "F64": np.float64, "I32": np.int32, "U64": np.uint64, "F32": np.float32}
    for c in cases:
        vals = c["values"]
        valid = None
        if any(v is None for v in vals):
            valid = [v is not None for v in vals]
            vals = [0 if v is None else v for v in vals]
        arr = np.asarray(vals, dtype=np_dt.get(c["dtype"], np.float64))
        perm = sort_oracle.sort_permutation([(arr, valid, c["asc"], c["nulls_first"])], c["limit"] or 0)
        if c.get("rows") is not None:
            assert perm.tolist() == c["rows"], c["src"]


def test_spill_oracle_states_finalize_to_the_c_oracle_results():
    """oracle/spill_oracle.py (serialised partial states, restated from the reference's StateSerde) has no
    reference golden; this ties it to the pinned C oracle instead: finalising its states (sum, count,
    sum / count, min / max with the NULL flags) must give exactly the C oracle's final results."""
    import numpy as np
    from databend_b200 import abi
    from databend_b200.block import Column, DataBlock
    from databend_b200.transforms import AggregatorParams
    from oracle import oracle as orc
    from oracle import spill_oracle
    rng = np.random.default_rng(4)
    n = 50_000
    k = rng.integers(-3, 200, n).astype(np.int32)
    kv = rng.random(n) > 0.05
    v = rng.integers(-10**6, 10**6, n).astype(np.int64)
    vv = rng.random(n) > 0.3
    x = rng.integers(0, 1 << 20, n).astype(np.float64)
    f = (rng.integers(-500, 500, n) * 0.25).astype(np.float32)
    fv = rng.random(n) > 0.5
    blk = DataBlock([Column.from_data(k, validity=kv), Column.from_data(v, validity=vv), Column.from_data(x), Column.from_data(f, validity=fv)])
    kinds = ["sum", "count", "count", "avg", "min", "max", "avg"]
    args = [1, None, 1, 2, 1, 3, 3]
    params = AggregatorParams([0], list(zip(kinds, args)))
    cols = {1: (v, vv), 2: (x, None), 3: (f, fv)}
    fields, arity, okeys = spill_oracle.group_states([(k, kv)], [None if a is None else cols[a] for a in args], kinds)
    keys, kvalid, aggs, avalid, _ = orc.filter_group_agg(blk, params.to_c(None), threads=2)
    exp = {}
    for i in range(len(aggs[0])):
        key = int(keys[0].view(np.int64)[i]) if kvalid[0][i] else None
        exp[key] = [(aggs[a][i].item() if avalid[a][i] else None) for a in range(len(kinds))]
    assert len(okeys[0][0]) == len(exp)
    for g in range(len(okeys[0][0])):
        key = int(okeys[0][0][g]) if okeys[0][1][g] else None
        got = []
        for a, kind in enumerate(kinds):
            fs = [fld[g] for fld in fields[a]]
            if kind == "count":
                got.append(int(fs[0]))
            elif kind == "sum":
                got.append(fs[0].item() if fs[-1] else None)
            elif kind == "avg":
                got.append(float(np.float64(fs[0]) / np.float64(fs[1])) if fs[-1] else None)
            else:
                got.append(fs[1].item() if fs[0] else None)
        assert got == exp[key], (key, got, exp[key])


def test_expression_builder_flattens_to_postfix():
    """Host logic of databend_b200/scalar_expr.py (no GPU): operator overloads build the tree, flatten()
    emits the postfix program the C-ABI takes, oversized trees and unknown functions are refused."""
    from databend_b200 import abi, scalar_expr as sx
    from databend_b200.lib import DbxError
    e = sx.call("and", sx.call("gt", sx.cast((sx.col(0) * sx.col(1) + sx.col(1)) % sx.lit(7, abi.U8), abi.I64), sx.lit(3, abi.I64)), sx.call("not", sx.call("is_null", sx.col(2))))
    prog = sx.flatten(e)
    kinds = [prog.nodes[i].kind for i in range(prog.n_nodes)]
    funcs = [prog.nodes[i].func for i in range(prog.n_nodes) if prog.nodes[i].kind == abi.EXPR_CALL]
    assert kinds == [abi.EXPR_COLUMN, abi.EXPR_COLUMN, abi.EXPR_CALL, abi.EXPR_COLUMN, abi.EXPR_CALL, abi.EXPR_CONST, abi.EXPR_CALL, abi.EXPR_CAST,
                     abi.EXPR_CONST, abi.EXPR_CALL, abi.EXPR_COLUMN, abi.EXPR_CALL, abi.EXPR_CALL, abi.EXPR_CALL]
    assert funcs == [abi.FN_MULTIPLY, abi.FN_PLUS, abi.FN_MODULO, abi.FN_GT, abi.FN_IS_NULL, abi.FN_NOT, abi.FN_AND]
    assert prog.nodes[7].cast_to == abi.I64 and prog.nodes[5].c.dtype == abi.U8 and prog.nodes[5].c.v.u64 == 7
    big = sx.col(0)
    for _ in range(abi.MAX_EXPR_NODES):
        big = big + sx.col(0)
    with pytest.raises(DbxError, match="too large"):
        sx.flatten(big)
    with pytest.raises(DbxError, match="not built"):
        sx.call("sqrt", sx.col(0))


# ---- the oracle's numeric conversions against exact rational arithmetic (fractions.Fraction)

INT_TYPES = ["I8", "I16", "I32", "I64", "U8", "U16", "U32", "U64"]
# 64-bit integers whose correctly rounded f32 differs from the f32 of their f64 (double rounding)
F32_WITNESSES = {1152921573326323713: 2.0 ** 60 + 2.0 ** 37, -1152921573326323713: -(2.0 ** 60 + 2.0 ** 37),
                 4611686293305294849: 2.0 ** 62 + 2.0 ** 39, 9223372586610589697: 2.0 ** 63 + 2.0 ** 40}


def nearest_even(v, ftype):
    """`v` (int or Fraction) rounded to the nearest value of ftype, ties to the even significand: the
    candidates around a first guess are compared by exact distance."""
    import numpy as np
    from fractions import Fraction
    ft, ut = (np.float32, np.uint32) if ftype == "F32" else (np.float64, np.uint64)
    c = [ft(float(v))]
    for _ in range(2):
        c = [np.nextafter(c[0], ft(-np.inf))] + c + [np.nextafter(c[-1], ft(np.inf))]
    dist = [abs(Fraction(float(x)) - Fraction(v)) for x in c]
    best = [x for x, d in zip(c, dist) if d == min(dist)]
    if len(best) == 2:
        best = [x for x in best if not int(np.asarray(x, ft).view(ut)) & 1]
    assert len(best) == 1
    return float(best[0])


def round_half_away_exact(x):
    from fractions import Fraction
    q = Fraction(x)
    r = math.floor(abs(q) + Fraction(1, 2))
    return r if q >= 0 else -r


def int_range(t):
    b = int(t[1:])
    return (-(1 << (b - 1)), (1 << (b - 1)) - 1) if t[0] == "I" else (0, (1 << b) - 1)


def conversion_inputs(t):
    """Type boundaries, the double-rounding witnesses, seeded uniform values and seeded values at and
    next to the f32 / f64 rounding ties, all inside the range of `t`."""
    import random
    lo, hi = int_range(t)
    rng = random.Random(t)
    vals = {lo, lo + 1, hi - 1, hi, 0, 1, (1 << 24) + 1, (1 << 53) + 1, -(1 << 24) - 1, -(1 << 53) - 1}
    vals.update(F32_WITNESSES)
    vals.update(rng.randint(lo, hi) for _ in range(1000))
    bits = int(t[1:])
    for p in (p for p in (24, 53) if p < bits):
        for _ in range(300):
            n = rng.randint(p + 1, bits)
            m = rng.randrange(1 << (n - 1), 1 << n) | 1 << (n - p - 1)  # n significant bits, bit n-p-1 set ...
            m &= ~((1 << (n - p - 1)) - 1)                                # ... and nothing below it: a tie
            for d in (-1, 0, 1):
                vals.update((m + d, -(m + d)))
    return sorted(v for v in vals if lo <= v <= hi)


@pytest.mark.parametrize("t", INT_TYPES)
def test_integer_to_float_conversions_round_once_to_nearest_even(t):
    """Rust `x as f32` / `x as f64` for every integer type, through cast_as, checked_cast and a
    CAST / TRY_CAST over a column: one rounding, to nearest, ties to even."""
    vals = conversion_inputs(t)
    for to in ("F32", "F64"):
        exp = [nearest_even(v, to) for v in vals]
        assert [eo.cast_as(v, t, to) for v in vals] == exp, (t, to)
        assert [eo.checked_cast(v, t, to) for v in vals] == exp, (t, to)
        for try_cast in (0, 1):
            rt, nullable, got, oks = eo.evaluate(("cast", ("col", 0), to, try_cast), [(t, vals, None)])
            assert rt == to and all(oks) and got == exp, (t, to, try_cast)
    for v, f in F32_WITNESSES.items():
        if int_range(t)[0] <= v <= int_range(t)[1]:
            assert eo.cast_as(v, t, "F32") == f == nearest_even(v, "F32"), (t, v)


@pytest.mark.parametrize("ftype", ["F32", "F64"])
@pytest.mark.parametrize("t", INT_TYPES)
def test_float_to_integer_cast_rounds_half_away_and_accepts_exactly_min_to_max(t, ftype):
    """CAST / TRY_CAST of a float to an integer rounds half away from zero, then is checked: at every
    boundary value the cast succeeds exactly when the exactly rounded value lies in [MIN, MAX]."""
    from helpers import float_int_boundaries
    lo, hi = int_range(t)
    xs = float_int_boundaries(t, ftype)
    exp = [None if (math.isnan(x) or math.isinf(x)) else round_half_away_exact(x) for x in xs]
    exp = [r if (r is not None and lo <= r <= hi) else None for r in exp]
    assert any(r is None for r in exp) and any(r is not None for r in exp)
    for x, r in zip(xs, exp):
        assert eo.checked_cast(eo.round_half_away(x), "F64", t) == r, (t, ftype, x)
    rt, nullable, got, oks = eo.evaluate(("cast", ("col", 0), t, 1), [(ftype, xs, None)])
    assert rt == t and nullable
    assert oks == [r is not None for r in exp], (t, ftype)
    assert [g for g, ok in zip(got, oks) if ok] == [r for r in exp if r is not None], (t, ftype)
    first_bad = next(i for i, r in enumerate(exp) if r is None)
    with pytest.raises(eo.EvalFailure, match="number overflowed") as ei:
        eo.evaluate(("cast", ("col", 0), t, 0), [(ftype, xs, None)])
    assert ei.value.row == first_bad
