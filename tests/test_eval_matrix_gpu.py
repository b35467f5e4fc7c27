"""dbx_eval_scalar where expression kernels go wrong, bit for bit against the CPU oracle
(oracle/eval_oracle.py, itself pinned by tests/golden/arithmetic.json and test_eval_oracle.py):
  * the whole type matrix of the arithmetic, casts and negate in the generated-kernel build;
  * float -> integer casts at the exact boundaries of every integer type, and the 64-bit integer ->
    Float32 values that a double rounding gets wrong, in both builds;
  * const operands, BOOL data and validity at bit offsets, device-resident inputs;
  * a block of 2,000,003 rows, so every thread of the grid strides several times and the first
    failing row is reduced across CTAs.
The generated-kernel leg runs with DBX_EVAL_JIT=2: a kernel that fails to compile or launch is an
error, not a silent fall-back to the interpreter.  NaN results compare as a class; every other
float compares by its bits."""
import time

import numpy as np
import pytest

from databend_b200 import abi
from databend_b200 import scalar_expr as sx
from databend_b200.block import Column, DataBlock
from helpers import INT_TYPES, float_int_boundaries, int_type_range
from test_eval_gpu import DT, NAME, NP, NUM, assert_matches, check_against_oracle, oracle, random_column, to_sexpr, to_tuple

pytestmark = pytest.mark.gpu
ARITH = ["plus", "minus", "multiply", "divide", "div", "modulo"]
GRID_ROWS = 2_000_003  # the grid is at most 148 SMs x 8 CTAs x 256 threads: ~6.6 rows per thread


@pytest.fixture(scope="module", autouse=True)
def report_file_runtime(request):
    t0 = time.perf_counter()
    yield
    tr = request.config.pluginmanager.get_plugin("terminalreporter")
    msg = f"{__name__}: {time.perf_counter() - t0:.1f} s"
    (tr.write_line if tr else print)(msg)


@pytest.fixture
def strict_jit(monkeypatch):
    monkeypatch.setenv("DBX_EVAL_JIT", "2")


@pytest.fixture(params=["jit", "interp"])
def eval_mode(request, monkeypatch):
    """Generated kernel, strict (DBX_EVAL_JIT=2), and the precompiled interpreter (DBX_EVAL_JIT=0)."""
    monkeypatch.setenv("DBX_EVAL_JIT", "2" if request.param == "jit" else "0")
    return request.param


def column_of(t, values, valid):
    if t == "BOOL":
        return Column.from_data(np.asarray(values, dtype=bool), abi.BOOL, validity=valid)
    return Column.from_data(np.asarray(values, dtype=NP[t]), DT[t], validity=valid)


def eval_block(block, e):
    col, odt = sx.eval_scalar(block, to_sexpr(e))
    valid = col.valid_mask() if col.validity is not None else np.ones(block.num_rows, dtype=bool)
    return NAME[odt & ~abi.NULLABLE], col.values(), valid


def check_block(block, oracle_cols, e, what):
    """`block` on the device against the oracle over `oracle_cols` ((type, values, valid) of the
    same rows, as the oracle sees them)."""
    eo = oracle()
    try:
        et, _, evals, evalid = eo.evaluate(to_tuple(e), oracle_cols)
    except eo.EvalFailure as f:
        with pytest.raises(sx.EvalError, match=f.msg) as ei:
            eval_block(block, e)
        assert ei.value.row == f.row, (what, ei.value.row, f.row)
        return "error"
    t, vals, valid = eval_block(block, e)
    assert_matches(t, vals, valid, et, evals, evalid, what)
    return "ok"


# ---- 1. the full type matrix in the generated build


@pytest.mark.parametrize("fn", ARITH)
def test_generated_kernels_binary_arithmetic_every_type_pair(gpu, strict_jit, fn):
    """All 10 x 10 operand types; nullable and non-null operands; zero divisors (first failing row)
    and non-zero divisors (every value compared).  The non-null and non-zero reruns reuse the kernel
    compiled for the pair: NVRTC's cache is keyed by the program text."""
    rng = np.random.default_rng(100 + ARITH.index(fn))
    rows = 257
    outcomes = set()
    for ta in NUM:
        for tb in NUM:
            a = random_column(rng, ta, rows, nullable=True)
            b = random_column(rng, tb, rows, nullable=True)
            e = ["call", fn, ["col", 0], ["col", 1]]
            divisors = [b[1]]
            if fn in ("divide", "div", "modulo"):
                divisors.append([x if x != 0 else 3 for x in b[1]])
            for bv in divisors:
                for nullable in (True, False):
                    cols = [a, (tb, bv, b[2])] if nullable else [(ta, a[1], None), (tb, bv, None)]
                    outcomes.add(check_against_oracle(cols, rows, e, (fn, ta, tb, nullable, bv is b[1])))
    assert outcomes == ({"ok", "error"} if fn in ("divide", "div", "modulo") else {"ok"})


def test_generated_kernels_casts_and_negate_every_type(gpu, strict_jit):
    """CAST and TRY_CAST from each of the 10 numeric types and BOOL to each of the 10 numeric types
    and BOOL, and negate on every numeric type (nullable and not)."""
    rng = np.random.default_rng(200)
    rows = 300
    for ta in NUM + ["BOOL"]:
        a = random_column(rng, ta, rows, nullable=True)
        for cols in ([a], [(ta, a[1], None)]):
            if ta != "BOOL":
                check_against_oracle(cols, rows, ["call", "negate", ["col", 0]], ("negate", ta))
            for to in NUM + ["BOOL"]:
                for try_cast in (1, 0):
                    check_against_oracle(cols, rows, ["cast", ["col", 0], to, try_cast], ("cast", ta, to, try_cast))


def round_half_away(d):
    """f64::round over an array, exactly (d - trunc(d) is exact)."""
    t = np.trunc(d)
    return t + np.where(np.abs(d - t) >= 0.5, np.sign(d), 0.0)


# ---- 2. float -> integer boundaries, 3. Int64 / UInt64 -> Float32


@pytest.mark.parametrize("ftype", ["F32", "F64"])
def test_float_to_integer_cast_boundaries(gpu, eval_mode, ftype):
    """MIN - 1, MIN - 0.5 and its neighbours, MIN, MAX, MAX + 0.5 and its neighbours, MAX + 1, 2^63 and
    2^64 with their neighbours, +-0, subnormals, +-inf and NaN, to every integer type: TRY_CAST gives
    NULL exactly where the rounded value leaves [MIN, MAX], CAST reports the first such row."""
    for t in INT_TYPES:
        xs = float_int_boundaries(t, ftype)
        lo, hi = int_type_range(t)
        n = len(xs)
        col = (ftype, xs, None)
        assert check_against_oracle([col], n, ["cast", ["col", 0], t, 1], ("try_cast", ftype, t)) == "ok"
        assert check_against_oracle([col], n, ["cast", ["col", 0], t, 0], ("cast", ftype, t)) == "error"
        # the same values with every out-of-range row NULL: CAST must then succeed on all rows
        with np.errstate(invalid="ignore"):
            r = round_half_away(np.asarray(xs))
        keep = [bool(np.isfinite(v)) and lo <= int(v) <= hi for v in r]  # compared as exact integers
        assert check_against_oracle([(ftype, xs, keep)], n, ["cast", ["col", 0], t, 0], ("cast, failures NULL", ftype, t)) == "ok"


def test_int64_uint64_to_float32_round_once(gpu, eval_mode):
    """64-bit integers whose nearest f32 differs from the f32 of their nearest f64, against numpy's
    direct conversion (one cvtsi2ss) as well as the oracle, so that a kernel and an oracle that round
    twice alike cannot agree on a wrong value."""
    wit = {"I64": [1152921573326323713, -1152921573326323713, 4611686293305294849, -4611686293305294849, 2 ** 63 - 1, -2 ** 63, 0, 1],
           "U64": [9223372586610589697, 1152921573326323713, 2 ** 64 - 1, 2 ** 63, 0, 1]}
    exact = {1152921573326323713: 2.0 ** 60 + 2.0 ** 37, 4611686293305294849: 2.0 ** 62 + 2.0 ** 39, 9223372586610589697: 2.0 ** 63 + 2.0 ** 40}
    for t, vals in wit.items():
        direct = np.asarray(vals, dtype=NP[t]).astype(np.float32)
        for v, d in zip(vals, direct):
            if abs(v) in exact:
                assert float(d) == np.sign(v) * exact[abs(v)]  # numpy's conversion rounds once
        for try_cast in (0, 1):
            e = ["cast", ["col", 0], "F32", try_cast]
            assert check_against_oracle([(t, vals, None)], len(vals), e, (t, try_cast)) == "ok"
            rt, got, valid = eval_block(DataBlock([column_of(t, vals, None)]), e)
            assert rt == "F32" and valid.all()
            np.testing.assert_array_equal(got.view(np.uint32), direct.view(np.uint32), err_msg=str((t, try_cast)))


# ---- 4. const operands, bit offsets, device-resident inputs


CONSTS = {"I8": -128, "I16": 32767, "I32": -7, "I64": -2 ** 63, "U8": 255, "U16": 3, "U32": 2 ** 32 - 1, "U64": 2 ** 64 - 1,
          "F32": 0.1, "F64": -2.5, "BOOL": True}


def oracle_value(t, v):
    """What the device holds for a const of type t: an F32 const is rounded to f32."""
    return float(np.float32(v)) if t == "F32" else v


def test_const_operands_every_type(gpu, eval_mode):
    """Column.new_const of every type (a NULL const and an F32 const that is not exact in f32
    included) next to a column, on either side of each operator."""
    rng = np.random.default_rng(300)
    rows = 300
    for i, t in enumerate(NUM + ["BOOL"]):
        for value in (CONSTS[t], None):
            const = Column.new_const(DT[t], value, rows)
            cval = (t, [oracle_value(t, value if value is not None else 0)] * rows, None if value is not None else [False] * rows)
            other_t = NUM[(i + 3) % len(NUM)] if t != "BOOL" else "BOOL"
            for ot in ([t, other_t] if t != "BOOL" else ["BOOL"]):
                o = random_column(rng, ot, rows, nullable=True)
                blk = DataBlock([column_of(*o), const], rows)
                ocols = [o, cval]
                if t == "BOOL":
                    exprs = [["call", f, ["col", a], ["col", 1 - a]] for f in ("and", "or") for a in (0, 1)]
                    exprs += [["call", "not", ["col", 1]], ["cast", ["col", 1], "I32", 0]]
                else:
                    exprs = [["call", f, ["col", a], ["col", 1 - a]] for f in ("plus", "minus", "multiply", "divide", "modulo") for a in (0, 1)]
                    exprs += [["call", "negate", ["col", 1]], ["cast", ["col", 1], "F32", 0], ["cast", ["col", 1], "I16", 1]]
                    if ot == t:
                        exprs += [["call", f, ["col", 0], ["col", 1]] for f in ("eq", "lt", "gte")]
                exprs += [["call", "is_null", ["col", 1]], ["call", "is_not_null", ["col", 1]]]
                for e in exprs:
                    check_block(blk, ocols, e, (t, value, ot, e))


@pytest.mark.parametrize("device", [False, True], ids=["host", "device"])
def test_bit_offset_inputs(gpu, eval_mode, device):
    """BOOL data and validity starting at a bit offset (Column::slice), from host memory and already in
    HBM, for offsets inside the first byte and past it, and row counts that end mid-byte."""
    from databend_b200.transforms import to_device
    rng = np.random.default_rng(400)
    total = 1000
    bools = rng.random(total) < 0.5
    bvalid = rng.random(total) < 0.8
    ints = rng.integers(-2 ** 31, 2 ** 31, total).astype(np.int32)
    ivalid = rng.random(total) < 0.7
    bcol = Column.from_data(bools, abi.BOOL, validity=bvalid.tolist())
    icol = Column.from_data(ints, abi.I32, validity=ivalid.tolist())
    plain = Column.from_data(rng.random(total) < 0.5, abi.BOOL)
    for off, n in ((3, 501), (13, 250), (8, 7), (0, 999)):
        cols = [c.slice(off, off + n) for c in (bcol, icol, plain)]
        if device:
            cols = [to_device(c) for c in cols]
            assert cols[0].dev_ptr and cols[0].data_bit_offset == off and cols[1].validity_bit_offset == off
        blk = DataBlock(cols, n)
        ocols = [("BOOL", bools[off:off + n].tolist(), bvalid[off:off + n].tolist()),
                 ("I32", ints[off:off + n].tolist(), ivalid[off:off + n].tolist()),
                 ("BOOL", plain.values()[off:off + n].tolist(), None)]
        for e in (["call", "not", ["col", 0]], ["call", "and", ["col", 0], ["col", 2]], ["call", "or", ["col", 2], ["col", 0]],
                  ["cast", ["col", 0], "U8", 0], ["call", "plus", ["col", 1], ["cast", ["col", 2], "I32", 0]],
                  ["call", "is_null", ["col", 1]], ["call", "modulo", ["col", 1], ["lit", 1000, "I16"]]):
            check_block(blk, ocols, e, (off, n, device, e))


# ---- 5. grid scale


def test_grid_scale_expression_tree(gpu, eval_mode):
    """(try_cast(c0 * c1 + c2 as Int32) >= try_cast(c3 as Int32)) and (c1 % 7 != 0) over 2,000,003 rows,
    against the same arithmetic vectorised in numpy (Int64 wrapping, round half away from zero,
    three-valued and), and a seeded 20,000-row sample against the oracle."""
    rng = np.random.default_rng(500)
    n = GRID_ROWS
    wide = rng.random(n) < 0.5
    c0 = np.where(wide, rng.integers(-2 ** 63, 2 ** 63 - 1, n, dtype=np.int64, endpoint=True), rng.integers(-50_000, 50_000, n))
    c1 = np.where(rng.random(n) < 0.5, rng.integers(-2 ** 63, 2 ** 63 - 1, n, dtype=np.int64, endpoint=True), rng.integers(-50_000, 50_000, n))
    c2 = rng.integers(0, 65536, n).astype(np.uint16)
    c3 = np.round(rng.standard_normal(n) * 2e9, 1)
    c3[rng.choice(n, 1000, replace=False)] = np.nan
    v0, v3 = rng.random(n) < 0.9, rng.random(n) < 0.9
    cols = [("I64", c0, v0), ("I64", c1, None), ("U16", c2, None), ("F64", c3, v3)]
    blk = DataBlock([Column.from_data(v, DT[t], validity=m) for t, v, m in cols], n)
    e = ["call", "and",
         ["call", "gte", ["cast", ["call", "plus", ["call", "multiply", ["col", 0], ["col", 1]], ["col", 2]], "I32", 1],
          ["cast", ["col", 3], "I32", 1]],
         ["call", "noteq", ["call", "modulo", ["col", 1], ["lit", 7, "U8"]], ["lit", 0, "I16"]]]
    t, got, valid = eval_block(blk, e)
    # numpy restatement
    with np.errstate(over="ignore", invalid="ignore"):
        s = c0 * c1 + c2.astype(np.int64)  # wraps in Int64
        l_ok = v0 & (s >= -2 ** 31) & (s < 2 ** 31)
        r = round_half_away(c3)
        r_ok = v3 & np.isfinite(c3) & (r >= -2 ** 31) & (r < 2 ** 31)
        lhs = l_ok & r_ok
        gte = np.where(lhs, s >= np.where(r_ok, r, 0).astype(np.int64), False)
        rhs = np.fmod(c1, 7) != 0
    exp_valid = ~rhs | lhs  # three-valued and: a false side wins, otherwise NULL if a side is NULL (c1 has no NULLs)
    exp = lhs & gte & rhs
    assert t == "BOOL"
    assert 0.05 < lhs.mean() < 0.95 and 0.05 < exp.mean() < 0.95 and (~exp_valid).any()
    np.testing.assert_array_equal(valid, exp_valid)
    np.testing.assert_array_equal(got[exp_valid], exp[exp_valid])
    # the oracle on a sample of rows (the expression is row-local)
    idx = np.sort(np.random.default_rng(501).choice(n, 20_000, replace=False))
    ocols = [(ct, v[idx].tolist(), None if m is None else m[idx].tolist()) for ct, v, m in cols]
    et, _, evals, evalid = oracle().evaluate(to_tuple(e), ocols)
    assert_matches(t, got[idx], valid[idx], et, evals, evalid, "grid sample")


def test_grid_scale_first_failing_row(gpu, eval_mode):
    """CAST(c0 AS Int8) over 2,000,003 rows with overflowing rows planted in different CTAs and
    strides: the first one is reported; made NULL, the next one is."""
    n = GRID_ROWS
    threads = 148 * 8 * 256  # one stride of the grid on a B200
    planted = sorted([threads * 5 + 10,                 # CTA 0, sixth stride
                      threads - 256 * 12 + 77,           # one of the last CTAs, first stride
                      threads + 256 * 600 + 3,           # CTA 600, second stride
                      1_000_000, n - 1])
    vals = np.random.default_rng(600).integers(-128, 128, n).astype(np.int32)
    vals[planted] = [128, -129, 2 ** 31 - 1, -2 ** 31, 300]
    valid = np.ones(n, dtype=bool)
    for first in planted:
        blk = DataBlock([Column.from_data(vals, abi.I32, validity=valid)], n)
        with pytest.raises(sx.EvalError, match="number overflowed") as ei:
            sx.eval_scalar(blk, sx.cast(sx.col(0), abi.I8))
        assert ei.value.row == first
        valid[first] = False
    blk = DataBlock([Column.from_data(vals, abi.I32, validity=valid)], n)
    col, _ = sx.eval_scalar(blk, sx.cast(sx.col(0), abi.I8))
    np.testing.assert_array_equal(col.valid_mask(), valid)
    np.testing.assert_array_equal(col.values()[valid], vals[valid].astype(np.int8))
