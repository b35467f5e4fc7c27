// eval_kernels.cuh — device side of dbx_eval_scalar: value images, the reference's cast / arithmetic
// rules per expression node, and the two kernels built from them:
//   eval_kernel           interprets the postfix program per row (value stack in registers);
//   dbx_jit_eval (NVRTC)  the same per-node functions called with COMPILE-TIME node descriptions in a
//                         generated straight-line body (eval.cu: specialise_expr) — the interpreter's
//                         dispatch, type switches and stack traffic fold away.
// Reference semantics: see eval.cu's header.
#pragma once
#include "common.cuh"

namespace dbx {

constexpr int kMaxExprNodes = DBX_MAX_EXPR_NODES;
constexpr int kEvalStack = 8;

struct NodeDev {
  int32_t kind;      // dbx_expr_kind
  int32_t func;      // dbx_func
  int32_t col;       // COLUMN: input slot
  int32_t out;       // result dtype of this node (dbx_dtype)
  int32_t a_type;    // CALL / CAST: dtype of the (first) argument
  int32_t b_type;    // CALL with two arguments: dtype of the second
  int32_t m_type;    // MODULO: LeastSuper(L, R) in which the remainder is computed
  int32_t try_cast;  // CAST: 1 = try_cast (failure -> NULL)
  uint64_t c_bits;   // CONST: value image in the node's type
  int32_t c_null;
  int32_t pad;
};
struct EvalParams {
  NodeDev nodes[kMaxExprNodes];
  DevCol cols[16];
  int32_t n_nodes, n_cols;
  int64_t n_rows;
  void* out_data;          // out dtype values (BOOL: one byte per row, packed afterwards)
  uint8_t* out_valid;      // one byte per row or nullptr
  int32_t out_dtype, pad;
  unsigned long long* first_error;  // min over failing rows of (row << 8 | code); ~0 = none
};

__host__ __device__ inline bool is_float_t(int t) { return t == DBX_F32 || t == DBX_F64; }
__host__ __device__ inline bool is_signed_t(int t) { return t == DBX_I8 || t == DBX_I16 || t == DBX_I32 || t == DBX_I64; }
__host__ __device__ inline int bits_of_t(int t) {
  switch (t) {
    case DBX_I8: case DBX_U8: return 8;
    case DBX_I16: case DBX_U16: return 16;
    case DBX_I32: case DBX_U32: case DBX_F32: return 32;
    default: return 64;
  }
}
// value images: integers sign/zero-extended to 64 bits, F64 as its bits, F32 as the f64 bits of the
// (exactly widened) value; BOOL 0/1
__device__ __forceinline__ double as_f64(uint64_t v, int t) {
  if (is_float_t(t)) return __longlong_as_double((long long)v);
  return is_signed_t(t) ? (double)(int64_t)v : (double)v;
}
// narrow a 64-bit two's complement result to an integer type (Rust wrapping arithmetic in that type)
__device__ __forceinline__ uint64_t wrap_int(uint64_t v, int t) {
  switch (t) {
    case DBX_I8: return (uint64_t)(int64_t)(int8_t)v;
    case DBX_I16: return (uint64_t)(int64_t)(int16_t)v;
    case DBX_I32: return (uint64_t)(int64_t)(int32_t)v;
    case DBX_U8: return v & 0xFFu;
    case DBX_U16: return v & 0xFFFFu;
    case DBX_U32: return v & 0xFFFFFFFFu;
    default: return v;
  }
}
__device__ __forceinline__ double int_min_f(int t) { return is_signed_t(t) ? -ldexp(1.0, bits_of_t(t) - 1) : 0.0; }
__device__ __forceinline__ double int_max_p1_f(int t) { return ldexp(1.0, is_signed_t(t) ? bits_of_t(t) - 1 : bits_of_t(t)); }  // max + 1, exact
// Rust `f64 as <int>`: truncates toward zero, saturates, NaN -> 0.  Returns the 64-bit image
// (sign-extended for signed types).
__device__ __forceinline__ uint64_t f64_as_int(double d, int t) {
  if (d != d) return 0;
  const int w = bits_of_t(t);
  if (is_signed_t(t)) {
    if (d <= int_min_f(t)) return w == 64 ? 0x8000000000000000ULL : (uint64_t)(-(int64_t)(1ULL << (w - 1)));
    if (d >= int_max_p1_f(t)) return w == 64 ? 0x7FFFFFFFFFFFFFFFULL : ((1ULL << (w - 1)) - 1);
    return (uint64_t)(int64_t)trunc(d);
  }
  if (d <= 0.0) return 0;
  if (d >= int_max_p1_f(t)) return w == 64 ? ~0ULL : ((1ULL << w) - 1);
  return (uint64_t)trunc(d);
}
// Rust `x as T` between any two numeric types (lossy where Rust is)
__device__ __forceinline__ uint64_t cast_as(uint64_t v, int from, int to) {
  if (is_float_t(to)) {
    // 64-bit integers round once, straight to f32 (cvt.rn.f32.{s64,u64}): through f64 they would round
    // twice (2^60 + 2^36 + 1 -> 2^60 instead of 2^60 + 2^37).  Narrower integers are exact in f64.
    if (to == DBX_F32 && from == DBX_I64) return (uint64_t)__double_as_longlong((double)__ll2float_rn((long long)v));
    if (to == DBX_F32 && from == DBX_U64) return (uint64_t)__double_as_longlong((double)__ull2float_rn((unsigned long long)v));
    double d = as_f64(v, from);
    if (to == DBX_F32) d = (double)(float)d;
    return (uint64_t)__double_as_longlong(d);
  }
  if (is_float_t(from)) {
    return f64_as_int(__longlong_as_double((long long)v), to);
  }
  return wrap_int(v, to);  // integer to integer: two's complement truncation / reinterpretation
}
// num_traits::cast::cast (checked): false when the value is not representable in `to`
__device__ __forceinline__ bool checked_cast(uint64_t v, int from, int to, uint64_t* out) {
  if (is_float_t(to)) { *out = cast_as(v, from, to); return true; }
  if (is_float_t(from)) {
    const double d = __longlong_as_double((long long)v);
    if (d != d) return false;
    const double tr = trunc(d);
    if (!(tr >= int_min_f(to) && tr < int_max_p1_f(to))) return false;
    *out = is_signed_t(to) ? (uint64_t)(int64_t)tr : (uint64_t)tr;
    return true;
  }
  // integer -> integer: value must lie in the destination range
  if (is_signed_t(from)) {
    const int64_t x = (int64_t)v;
    if (is_signed_t(to)) {
      if (bits_of_t(to) < 64) { const int64_t lim = 1LL << (bits_of_t(to) - 1); if (x < -lim || x >= lim) return false; }
    } else {
      if (x < 0) return false;
      if (bits_of_t(to) < 64 && (uint64_t)x >= (1ULL << bits_of_t(to))) return false;
    }
  } else {
    if (is_signed_t(to)) { if (v >= (1ULL << (bits_of_t(to) - 1))) return false; }
    else if (bits_of_t(to) < 64 && v >= (1ULL << bits_of_t(to))) return false;
  }
  *out = v;
  return true;
}

__device__ __forceinline__ uint64_t load_image(const DevCol& c, int64_t r, int dtype) {  // dtype = c.dtype (a constant when specialised)
  if (c.is_const) return c.const_bits;
  const char* base = (const char*)c.data;
  switch (dtype) {
    case DBX_I64: case DBX_U64: case DBX_F64: return ((const uint64_t*)base)[r];
    case DBX_I32: return (uint64_t)(int64_t)((const int32_t*)base)[r];
    case DBX_U32: return ((const uint32_t*)base)[r];
    case DBX_F32: return (uint64_t)__double_as_longlong((double)((const float*)base)[r]);
    case DBX_I16: return (uint64_t)(int64_t)((const int16_t*)base)[r];
    case DBX_U16: return ((const uint16_t*)base)[r];
    case DBX_I8: return (uint64_t)(int64_t)((const int8_t*)base)[r];
    case DBX_U8: return ((const uint8_t*)base)[r];
    case DBX_BOOL: return (uint64_t)bit_test((const uint8_t*)base, c.dbit_off + r);
    default: return 0;
  }
}
// three-way compare of two values of the same dtype (OrderedFloat for floats: NaN greatest and equal to itself)
__device__ __forceinline__ int cmp_same(uint64_t a, uint64_t b, int t) {
  if (is_float_t(t)) {
    const double x = __longlong_as_double((long long)a), y = __longlong_as_double((long long)b);
    const bool xn = x != x, yn = y != y;
    if (xn | yn) return xn == yn ? 0 : (xn ? 1 : -1);
    return x < y ? -1 : (x > y ? 1 : 0);
  }
  if (is_signed_t(t)) return (int64_t)a < (int64_t)b ? -1 : ((int64_t)a > (int64_t)b ? 1 : 0);
  return a < b ? -1 : (a > b ? 1 : 0);
}
enum : int { ERR_DIV_ZERO = 1, ERR_DIVIDED_BY_ZERO = 2, ERR_OVERFLOW = 3 };

// ---- one node applied to its operand(s); `a`/`an` is the (first) operand and receives the result
__device__ __forceinline__ void apply_cast(const NodeDev& nd, uint64_t& a, bool& an, int& err) {
  uint64_t out = 0;
  bool ok = an;
  if (ok) {
    const int from = nd.a_type, to = nd.out;
    bool fits = true;
    if (to == DBX_BOOL) out = is_float_t(from) ? (as_f64(a, from) != 0.0) : (a != 0);
    else if (from == DBX_BOOL) out = cast_as(a, DBX_U8, to);
    else if (is_float_t(from) && !is_float_t(to)) {  // round cast (numeric_cast_option = rounding, the default)
      const double d = round(__longlong_as_double((long long)a));
      fits = checked_cast((uint64_t)__double_as_longlong(d), DBX_F64, to, &out);
    } else {
      fits = checked_cast(a, from, to, &out);
    }
    if (!fits) {
      out = 0;
      if (nd.try_cast) ok = false; else err = err ? err : ERR_OVERFLOW;
    }
  }
  a = out; an = ok;
}
__device__ __forceinline__ void apply_unary(const NodeDev& nd, uint64_t& a, bool& an, int& err) {
  const int f = nd.func;
  if (f == DBX_FN_IS_NULL) { a = an ? 0 : 1; an = true; }
  else if (f == DBX_FN_IS_NOT_NULL) { a = an ? 1 : 0; an = true; }
  else if (f == DBX_FN_NOT) { a = a ? 0 : 1; }
  else {  // NEGATE: -(a as Negate type); floats keep their type; 64-bit inputs are checked (arithmetic.rs:226-276)
    if (is_float_t(nd.out)) a = (uint64_t)__double_as_longlong(-as_f64(a, nd.a_type));
    else {
      if (an && ((nd.a_type == DBX_I64 && a == 0x8000000000000000ULL) || (nd.a_type == DBX_U64 && a > 0x8000000000000000ULL))) err = err ? err : ERR_OVERFLOW;
      a = wrap_int((uint64_t)0 - cast_as(a, nd.a_type, nd.out), nd.out);
    }
  }
}
__device__ __forceinline__ void apply_binary(const NodeDev& nd, uint64_t& a, bool& an, const uint64_t b, const bool bn, int& err) {
  const int f = nd.func;
  uint64_t out = 0;
  bool ok = an && bn;
  if (f == DBX_FN_AND || f == DBX_FN_OR) {  // three-valued logic (boolean.rs: and / or on nullable booleans)
    const bool at = an && a, af = an && !a, bt = bn && b, bf = bn && !b;
    if (f == DBX_FN_AND) { if (af || bf) { out = 0; ok = true; } else if (at && bt) { out = 1; ok = true; } else ok = false; }
    else { if (at || bt) { out = 1; ok = true; } else if (af && bf) { out = 0; ok = true; } else ok = false; }
  } else if (ok) {
    const int ta = nd.a_type, tb = nd.b_type, to = nd.out;
    if (f == DBX_FN_PLUS || f == DBX_FN_MINUS || f == DBX_FN_MULTIPLY) {
      if (is_float_t(to)) {
        const double x = as_f64(a, ta), y = as_f64(b, tb);
        out = (uint64_t)__double_as_longlong(f == DBX_FN_PLUS ? x + y : (f == DBX_FN_MINUS ? x - y : x * y));
      } else {  // (a as T) op (b as T), wrapping in T
        const uint64_t x = cast_as(a, ta, to), y = cast_as(b, tb, to);
        out = wrap_int(f == DBX_FN_PLUS ? x + y : (f == DBX_FN_MINUS ? x - y : x * y), to);
      }
    } else if (f == DBX_FN_DIVIDE) {
      const double y = as_f64(b, tb);
      if (y == 0.0) err = err ? err : ERR_DIVIDED_BY_ZERO;
      else out = (uint64_t)__double_as_longlong(as_f64(a, ta) / y);
    } else if (f == DBX_FN_DIV) {
      const double y = as_f64(b, tb);
      if (y == 0.0) err = err ? err : ERR_DIVIDED_BY_ZERO;
      else out = f64_as_int(as_f64(a, ta) / y, to);
    } else if (f == DBX_FN_MODULO) {
      const bool b_zero = is_float_t(tb) ? (__longlong_as_double((long long)b) == 0.0) : (b == 0);
      if (b_zero) err = err ? err : ERR_DIV_ZERO;
      else {
        const int tm = nd.m_type;
        const uint64_t x = cast_as(a, ta, tm), y = cast_as(b, tb, tm);
        uint64_t rem;
        if (is_float_t(tm)) {
          double fr = fmod(__longlong_as_double((long long)x), __longlong_as_double((long long)y));
          if (tm == DBX_F32) fr = (double)fmodf((float)__longlong_as_double((long long)x), (float)__longlong_as_double((long long)y));
          rem = (uint64_t)__double_as_longlong(fr);
        } else if (is_signed_t(tm)) {
          const int64_t xs = (int64_t)x, ys = (int64_t)y;
          rem = (ys == -1 || ys == 0) ? 0 : (uint64_t)(xs % ys);  // MIN % -1 = 0
          if (ys == 0) err = err ? err : ERR_DIV_ZERO;
        } else {
          rem = y == 0 ? 0 : x % y;
          if (y == 0) err = err ? err : ERR_DIV_ZERO;
        }
        out = cast_as(rem, tm, to);
      }
    } else {  // comparisons: both sides were cast to a common type by the type checker (a_type == b_type)
      const int c3 = cmp_same(a, b, ta);
      out = f == DBX_FN_EQ ? c3 == 0 : f == DBX_FN_NOTEQ ? c3 != 0 : f == DBX_FN_LT ? c3 < 0 : f == DBX_FN_LTE ? c3 <= 0 : f == DBX_FN_GT ? c3 > 0 : c3 >= 0;
    }
  }
  a = out; an = ok;
}
__device__ __forceinline__ void load_column(const DevCol& c, int64_t r, int dtype, uint64_t& v, bool& ok) {
  ok = c.is_const ? c.is_const != 2 : (!c.validity || bit_test(c.validity, c.vbit_off + r));
  v = ok ? load_image(c, r, dtype) : 0;
}
__device__ __forceinline__ void store_result(const EvalParams& p, int64_t r, uint64_t v, bool valid, int err) {
  // an error is raised by the CALL whose own arguments are valid on this row (passthrough_nullable masks
  // only that call's NULL rows), whatever the validity of the final value
  if (err) atomicMin(p.first_error, ((unsigned long long)r << 8) | (unsigned long long)err);
  if (!valid) v = 0;
  switch (p.out_dtype) {
    case DBX_BOOL: ((uint8_t*)p.out_data)[r] = (uint8_t)(v != 0); break;
    case DBX_I8: case DBX_U8: ((uint8_t*)p.out_data)[r] = (uint8_t)v; break;
    case DBX_I16: case DBX_U16: ((uint16_t*)p.out_data)[r] = (uint16_t)v; break;
    case DBX_I32: case DBX_U32: ((uint32_t*)p.out_data)[r] = (uint32_t)v; break;
    case DBX_F32: ((float*)p.out_data)[r] = (float)__longlong_as_double((long long)v); break;
    default: ((uint64_t*)p.out_data)[r] = v; break;
  }
  if (p.out_valid) p.out_valid[r] = valid ? 1 : 0;
}

#ifndef DBX_JIT
// The interpreter: an 8-deep value stack held in registers (push / pop shift the registers, so no
// dynamically indexed local array), top of stack in s0.
__global__ void __launch_bounds__(256) eval_kernel(const __grid_constant__ EvalParams p) {
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < p.n_rows; r += (int64_t)gridDim.x * blockDim.x) {
    uint64_t s0 = 0, s1 = 0, s2 = 0, s3 = 0, s4 = 0, s5 = 0, s6 = 0, s7 = 0;
    bool n0 = false, n1 = false, n2 = false, n3 = false, n4 = false, n5 = false, n6 = false, n7 = false;
    int err = 0;
    for (int i = 0; i < p.n_nodes; ++i) {
      const NodeDev& nd = p.nodes[i];
      if (nd.kind == DBX_EXPR_COLUMN || nd.kind == DBX_EXPR_CONST) {
        s7 = s6; s6 = s5; s5 = s4; s4 = s3; s3 = s2; s2 = s1; s1 = s0;
        n7 = n6; n6 = n5; n5 = n4; n4 = n3; n3 = n2; n2 = n1; n1 = n0;
        if (nd.kind == DBX_EXPR_COLUMN) load_column(p.cols[nd.col], r, nd.out, s0, n0);
        else { s0 = nd.c_bits; n0 = !nd.c_null; }
      } else if (nd.kind == DBX_EXPR_CAST) {
        apply_cast(nd, s0, n0, err);
      } else if (nd.func == DBX_FN_NOT || nd.func == DBX_FN_NEGATE || nd.func == DBX_FN_IS_NULL || nd.func == DBX_FN_IS_NOT_NULL) {
        apply_unary(nd, s0, n0, err);
      } else {
        apply_binary(nd, s1, n1, s0, n0, err);  // s1 op s0 -> s1, then pop
        s0 = s1; s1 = s2; s2 = s3; s3 = s4; s4 = s5; s5 = s6; s6 = s7;
        n0 = n1; n1 = n2; n2 = n3; n3 = n4; n4 = n5; n5 = n6; n6 = n7;
      }
    }
    store_result(p, r, s0, n0, err);
  }
}
#endif

}  // namespace dbx
