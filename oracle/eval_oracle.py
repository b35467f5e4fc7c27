"""CPU ORACLE for scalar expressions (test infrastructure only — never imported by the product).

Row-by-row Python restatement of the reference's evaluator for the numeric / boolean functions
libdbx evaluates on the device.  Each rule cites the file it follows (relative to /root/reference):
  result types          src/query/codegen/src/writes/arithmetics_type.rs:240-265 (arithmetic_coercion)
  plus/minus/multiply   src/query/functions/src/scalars/numeric_basic_arithmetic/src/numeric_basic_arithmetic.rs:255-400
                        ((a as T) op (b as T), wrapping: release build, Cargo.toml:577)
  divide / div          numeric_basic_arithmetic.rs:407-482 (through f64; "divided by zero")
  modulo                .../arithmetic_modulo.rs:68-97 (in LeastSuper; "Division by zero"; MIN % -1 = 0)
  unary minus           src/query/functions/src/scalars/arithmetic/src/arithmetic.rs:210-277 (Negate type; 64-bit checked)
  to_<type> casts       src/query/functions/src/scalars/arithmetic/src/arithmetic.rs:490-600
                        (lossless `as`; float->int rounds then checked; lossy checked "number overflowed")
  NULL handling         passthrough_nullable (register.rs): NULL in -> NULL out, errors masked
  and / or              boolean.rs: three-valued logic
Pinned by tests/golden/arithmetic.json (transcribed from functions/tests/it/scalars/testdata/arithmetic.txt)."""
import math
import struct

import numpy as np

INT_BITS = {"I8": 8, "I16": 16, "I32": 32, "I64": 64, "U8": 8, "U16": 16, "U32": 32, "U64": 64, "F32": 32, "F64": 64}
NP = {"I8": np.int8, "I16": np.int16, "I32": np.int32, "I64": np.int64, "U8": np.uint8, "U16": np.uint16, "U32": np.uint32,
      "U64": np.uint64, "F32": np.float32, "F64": np.float64, "BOOL": np.bool_}


def is_float(t): return t in ("F32", "F64")
def is_signed(t): return t in ("I8", "I16", "I32", "I64")
def bits(t): return INT_BITS[t]


def make_type(b, signed, flt):
    if flt:
        return "F32" if b <= 32 else "F64"
    return ("I" if signed else "U") + str(b)


def next_bits(b): return 64 if b >= 64 else b * 2
def t_add_mul(a, b): return make_type(next_bits(max(bits(a), bits(b))), is_signed(a) or is_signed(b), is_float(a) or is_float(b))
def t_minus(a, b): return make_type(next_bits(max(bits(a), bits(b))), True, is_float(a) or is_float(b))
def t_intdiv(a, b): return make_type(max(bits(a), bits(b)), is_signed(a) or is_signed(b) or is_float(a) or is_float(b), False)  # floats count as signed (number.rs:392-404)
def t_super(a, b): return make_type(max(bits(a), bits(b)), is_signed(a) or is_signed(b), is_float(a) or is_float(b))


def t_modulo(a, b):
    if is_float(a) or is_float(b):
        return "F64"
    s = is_signed(a)
    return make_type(next_bits(bits(b)) if s else bits(b), s, False)


def t_negate(a): return a if is_float(a) else make_type(next_bits(bits(a)), True, False)


def wrap(v, t):
    """Python int -> value of integer type t with two's complement wrapping."""
    b = bits(t)
    v &= (1 << b) - 1
    if is_signed(t) and v >= 1 << (b - 1):
        v -= 1 << b
    return v


def f32(x): return struct.unpack("<f", struct.pack("<f", x))[0] if not (math.isinf(x) or math.isnan(x)) and abs(x) < 3.5e38 else float(np.float32(x))


def int_range(t):
    b = bits(t)
    return (-(1 << (b - 1)), (1 << (b - 1)) - 1) if is_signed(t) else (0, (1 << b) - 1)


def int_to_f32(v):
    """Rust `v as f32` for an integer: rounded ONCE to nearest, ties to even (through f64 a 64-bit
    integer would round twice: 2^60 + 2^36 + 1 -> 2^60 instead of 2^60 + 2^37)."""
    a = abs(v)
    if a < 1 << 24:
        return float(v)
    sh = a.bit_length() - 24
    q, r = a >> sh, a & ((1 << sh) - 1)
    half = 1 << (sh - 1)
    if r > half or (r == half and q & 1):
        q += 1
    return math.copysign(float(q << sh), v)


def round_half_away(x):
    """f64::round: half away from zero, exactly (floor(|x| + 0.5) is wrong where |x| + 0.5 rounds,
    e.g. 0.49999999999999994 and odd integers in [2^52, 2^53))."""
    if math.isnan(x) or math.isinf(x):
        return x
    t = math.trunc(x)
    if abs(x - t) >= 0.5:  # exact: x and trunc(x) are doubles within 1 of each other
        t += 1 if x > 0 else -1
    return math.copysign(float(t), x)


def cast_as(v, frm, to):
    """Rust `v as to`."""
    if is_float(to):
        if not is_float(frm):
            return int_to_f32(int(v)) if to == "F32" else float(int(v))
        x = float(v)
        return float(np.float32(x)) if to == "F32" else x
    if is_float(frm):
        if math.isnan(v):
            return 0
        lo, hi = int_range(to)
        if v <= lo:
            return lo
        if v >= hi:
            return hi
        return int(math.trunc(v))
    return wrap(int(v), to)


def checked_cast(v, frm, to):
    """num_traits::cast::cast: None when not representable."""
    if is_float(to):
        return cast_as(v, frm, to)
    if is_float(frm):
        if math.isnan(v) or math.isinf(v):
            return None
        tr = math.trunc(v)
        lo, hi = int_range(to)
        return int(tr) if lo <= tr <= hi else None
    lo, hi = int_range(to)
    return int(v) if lo <= int(v) <= hi else None


class EvalFailure(Exception):
    def __init__(self, msg, row):
        super().__init__(msg)
        self.msg, self.row = msg, row


def infer(e, col_types):
    """-> (type name, nullable) of an expression tree (tuples: ("col", i) | ("lit", value, type) |
    ("cast", e, type, try) | ("call", name, args...))."""
    k = e[0]
    if k == "col":
        return col_types[e[1]]
    if k == "lit":
        return (e[2], e[1] is None)
    if k == "cast":
        t, n = infer(e[1], col_types)
        return (e[2], n or bool(e[3]))
    name, args = e[1], [infer(a, col_types) for a in e[2:]]
    if name in ("is_null", "is_not_null"):
        return ("BOOL", False)
    if name == "not":
        return ("BOOL", args[0][1])
    if name == "negate":
        return (t_negate(args[0][0]), args[0][1])
    (ta, na), (tb, nb) = args
    n = na or nb
    if name in ("plus", "multiply"):
        return (t_add_mul(ta, tb), n)
    if name == "minus":
        return (t_minus(ta, tb), n)
    if name == "divide":
        return ("F64", n)
    if name == "div":
        return (t_intdiv(ta, tb), n)
    if name == "modulo":
        return (t_modulo(ta, tb), n)
    return ("BOOL", n)


def cmp3(a, b, t):
    if is_float(t):
        an, bn = math.isnan(a), math.isnan(b)
        if an or bn:
            return 0 if an == bn else (1 if an else -1)
    return -1 if a < b else (1 if a > b else 0)


def eval_row(e, row, col_types, r):
    """-> (value, valid); raises EvalFailure for a per-row error on a valid row."""
    k = e[0]
    if k == "col":
        v, ok = row[e[1]]
        return (v if ok else 0, ok)
    if k == "lit":
        return (e[1] if e[1] is not None else 0, e[1] is not None)
    if k == "cast":
        v, ok = eval_row(e[1], row, col_types, r)
        frm = infer(e[1], col_types)[0]
        to = e[2]
        if not ok:
            return (0, False)
        if to == "BOOL":
            return (bool(v != 0), True)
        if frm == "BOOL":
            return (cast_as(int(v), "U8", to), True)
        if is_float(frm) and not is_float(to):
            out = checked_cast(round_half_away(float(v)), "F64", to)
        else:
            out = checked_cast(v, frm, to)
        if out is None:
            if e[3]:
                return (0, False)
            raise EvalFailure("number overflowed", r)
        return (out, True)
    name = e[1]
    if name in ("is_null", "is_not_null", "not", "negate"):
        v, ok = eval_row(e[2], row, col_types, r)
        ta = infer(e[2], col_types)[0]
        if name == "is_null":
            return (not ok, True)
        if name == "is_not_null":
            return (ok, True)
        if not ok:
            return (0, False)
        if name == "not":
            return (not v, True)
        to = t_negate(ta)
        if (ta == "I64" and v == -(1 << 63)) or (ta == "U64" and v > (1 << 63)):  # arithmetic.rs:226-276: 64-bit negate is checked
            raise EvalFailure("number overflowed", r)
        return ((-float(v) if to == "F64" else float(np.float32(-np.float32(v)))) if is_float(to) else wrap(-cast_as(v, ta, to), to), True)
    (a, aok), (b, bok) = eval_row(e[2], row, col_types, r), eval_row(e[3], row, col_types, r)
    ta, tb = infer(e[2], col_types)[0], infer(e[3], col_types)[0]
    if name in ("and", "or"):
        at, af, bt, bf = aok and bool(a), aok and not a, bok and bool(b), bok and not b
        if name == "and":
            return (False, True) if (af or bf) else ((True, True) if (at and bt) else (False, False))
        return (True, True) if (at or bt) else ((False, True) if (af and bf) else (False, False))
    if not (aok and bok):
        return (0, False)
    if name in ("plus", "minus", "multiply"):
        to = t_minus(ta, tb) if name == "minus" else t_add_mul(ta, tb)
        if is_float(to):
            x, y = float(a), float(b)
            return (x + y if name == "plus" else x - y if name == "minus" else x * y, True)
        x, y = cast_as(a, ta, to), cast_as(b, tb, to)
        return (wrap(x + y if name == "plus" else x - y if name == "minus" else x * y, to), True)
    if name == "divide":
        if float(b) == 0.0:
            raise EvalFailure("divided by zero", r)
        return (float(np.float64(float(a)) / np.float64(float(b))), True)
    if name == "div":
        if float(b) == 0.0:
            raise EvalFailure("divided by zero", r)
        return (cast_as(float(np.float64(float(a)) / np.float64(float(b))), "F64", t_intdiv(ta, tb)), True)
    if name == "modulo":
        if b == 0:
            raise EvalFailure("Division by zero", r)
        tm, to = t_super(ta, tb), t_modulo(ta, tb)
        x, y = cast_as(a, ta, tm), cast_as(b, tb, tm)
        if is_float(tm):
            with np.errstate(invalid="ignore"):  # Rust f32/f64 `%` == C fmodf/fmod (inf % y = NaN)
                rem = float(np.fmod(np.float32(x), np.float32(y))) if tm == "F32" else float(np.fmod(np.float64(x), np.float64(y)))
        elif is_signed(tm):
            rem = 0 if y == -1 else (abs(x) % abs(y)) * (1 if x >= 0 else -1)  # Rust %: truncated, sign of the dividend
        else:
            rem = x % y
        return (cast_as(rem, tm, to), True)
    c = cmp3(a, b, ta)
    return ({"eq": c == 0, "noteq": c != 0, "lt": c < 0, "lte": c <= 0, "gt": c > 0, "gte": c >= 0}[name], True)


def evaluate(e, columns):
    """columns: list of (type name, values sequence, valid sequence or None).  Returns
    (type, nullable, values list, valid list); raises EvalFailure at the FIRST failing row."""
    col_types = [(t, valid is not None) for t, _, valid in columns]
    t, nullable = infer(e, col_types)
    n = len(columns[0][1]) if columns else 0
    vals, oks = [], []
    for r in range(n):
        row = []
        for ct, v, valid in columns:
            x = v[r]
            x = float(x) if is_float(ct) else (bool(x) if ct == "BOOL" else int(x))
            row.append((x, True if valid is None else bool(valid[r])))
        v, ok = eval_row(e, row, col_types, r)
        vals.append(v if ok else (False if t == "BOOL" else 0))
        oks.append(ok)
    return t, nullable, vals, oks
