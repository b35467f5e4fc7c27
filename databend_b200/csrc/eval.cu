// eval.cu — dbx_eval_scalar: Evaluator::run over a DataBlock for numeric expressions.
//
// Reference replaced (paths relative to /root/reference):
//   Evaluator::{run, partial_run, eval_common_call, run_cast}   src/query/expression/src/evaluator.rs:247-465
//   ScalarFunction::eval + passthrough_nullable                  src/query/expression/src/function.rs:103, register.rs
//   plus / minus / multiply / divide / div / modulo              src/query/functions/src/scalars/numeric_basic_arithmetic/src/numeric_basic_arithmetic.rs:255-520
//   modulo semantics                                             .../arithmetic_modulo.rs:29-97
//   result types (ResultTypeOfBinary)                            src/query/codegen/src/writes/arithmetics_type.rs:240-265
//   to_<number> casts                                            src/query/functions/src/scalars/arithmetic/src/arithmetic.rs:490-600
//   comparison / boolean functions                               src/query/functions/src/scalars/comparison.rs, boolean.rs
//
// The reference walks the Expr tree and materialises one column per node (one full memory pass
// each).  Here the expression arrives as a postfix program; the host infers every node's type with
// the reference's rules, and ONE kernel evaluates the whole program per row in registers: every
// input column is read once and one output column is written.  Per-row errors (division by zero,
// number overflowed) are collected as "first failing row" like EvalContext::set_error; NULL rows
// never raise (passthrough_nullable evaluates under the validity).
#include <algorithm>
#include <cmath>
#include <vector>

#include "runtime.h"
#include "eval_kernels.cuh"
#include "agg_jit.h"

#include <sstream>

namespace dbx {
namespace {


__global__ void eval_pack_bits_kernel(const uint8_t* bytes, int64_t n, uint8_t* bits) {
  const int64_t nb = (n + 7) / 8;
  for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nb; b += (int64_t)gridDim.x * blockDim.x) {
    uint32_t v = 0;
    for (int k = 0; k < 8; ++k) {
      const int64_t i = b * 8 + k;
      if (i < n && bytes[i]) v |= 1u << k;
    }
    bits[b] = (uint8_t)v;
  }
}

// ---- the reference's type rules (arithmetics_type.rs codegen)
inline int make_type(int bits, bool is_signed, bool is_float) {
  if (is_float) return bits <= 32 ? DBX_F32 : DBX_F64;
  switch (bits) {
    case 8: return is_signed ? DBX_I8 : DBX_U8;
    case 16: return is_signed ? DBX_I16 : DBX_U16;
    case 32: return is_signed ? DBX_I32 : DBX_U32;
    default: return is_signed ? DBX_I64 : DBX_U64;
  }
}
inline int next_bits(int b) { return b >= 64 ? 64 : b * 2; }
inline int type_add_mul(int a, int b) { return make_type(next_bits(std::max(bits_of_t(a), bits_of_t(b))), is_signed_t(a) || is_signed_t(b), is_float_t(a) || is_float_t(b)); }
inline int type_minus(int a, int b) { return make_type(next_bits(std::max(bits_of_t(a), bits_of_t(b))), true, is_float_t(a) || is_float_t(b)); }
inline int type_intdiv(int a, int b) {  // NumberDataType::is_signed counts the float types as signed (number.rs:392-404)
  return make_type(std::max(bits_of_t(a), bits_of_t(b)), is_signed_t(a) || is_signed_t(b) || is_float_t(a) || is_float_t(b), false);
}
inline int type_super(int a, int b) { return make_type(std::max(bits_of_t(a), bits_of_t(b)), is_signed_t(a) || is_signed_t(b), is_float_t(a) || is_float_t(b)); }
inline int type_modulo(int a, int b) {
  if (is_float_t(a) || is_float_t(b)) return DBX_F64;
  const bool s = is_signed_t(a);
  return make_type(s ? next_bits(bits_of_t(b)) : bits_of_t(b), s, false);
}
inline int type_negate(int a) { return is_float_t(a) ? a : make_type(next_bits(bits_of_t(a)), true, false); }

// Source of the straight-line kernel for a type-checked program: every node is a constexpr
// NodeDev, every stack slot a named variable.
std::string specialised_source(const EvalParams& p) {
  std::ostringstream o;
  o << "#define DBX_JIT 1\n#include \"eval_kernels.cuh\"\nnamespace dbx {\n__device__ constexpr NodeDev jnodes[" << p.n_nodes << "] = {\n";
  for (int i = 0; i < p.n_nodes; ++i) {
    const NodeDev& n = p.nodes[i];
    char cb[40];
    snprintf(cb, sizeof(cb), "0x%llxULL", (unsigned long long)n.c_bits);
    o << " {" << n.kind << ", " << n.func << ", " << n.col << ", " << n.out << ", " << n.a_type << ", " << n.b_type << ", " << n.m_type << ", " << n.try_cast
      << ", " << cb << ", " << n.c_null << ", 0},\n";
  }
  o << "};\n}\nextern \"C\" __global__ void __launch_bounds__(256) dbx_jit_eval(const __grid_constant__ dbx::EvalParams p) {\n"
    << "  using namespace dbx;\n"
    << "  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < p.n_rows; r += (int64_t)gridDim.x * blockDim.x) {\n"
    << "    int err = 0;\n";
  for (int d = 0; d < kEvalStack; ++d) o << "    uint64_t v" << d << " = 0; bool k" << d << " = false;\n";
  int sp = 0;
  for (int i = 0; i < p.n_nodes; ++i) {
    const NodeDev& n = p.nodes[i];
    if (n.kind == DBX_EXPR_COLUMN) { o << "    load_column(p.cols[" << n.col << "], r, " << n.out << ", v" << sp << ", k" << sp << ");\n"; ++sp; }
    else if (n.kind == DBX_EXPR_CONST) { o << "    v" << sp << " = jnodes[" << i << "].c_bits; k" << sp << " = !jnodes[" << i << "].c_null;\n"; ++sp; }
    else if (n.kind == DBX_EXPR_CAST) o << "    apply_cast(jnodes[" << i << "], v" << sp - 1 << ", k" << sp - 1 << ", err);\n";
    else if (n.func == DBX_FN_NOT || n.func == DBX_FN_NEGATE || n.func == DBX_FN_IS_NULL || n.func == DBX_FN_IS_NOT_NULL)
      o << "    apply_unary(jnodes[" << i << "], v" << sp - 1 << ", k" << sp - 1 << ", err);\n";
    else { o << "    apply_binary(jnodes[" << i << "], v" << sp - 2 << ", k" << sp - 2 << ", v" << sp - 1 << ", k" << sp - 1 << ", err);\n"; --sp; }
  }
  o << "    store_result(p, r, v0, k0, err);\n  }\n}\n";
  return o.str();
}

}  // namespace
}  // namespace dbx

using namespace dbx;

extern "C" int32_t dbx_eval_scalar(int32_t device, const dbx_expr* expr, const dbx_block* block, int32_t out_mem, dbx_block* out,
                                   int32_t* out_dtype, int64_t* first_error_row) {
  ErrorSink& err = g_create_error;
  if (!expr || !block || !out || expr->n_nodes < 1 || expr->n_nodes > kMaxExprNodes || block->num_cols > 16) { err.set("dbx_eval_scalar: bad argument"); return DBX_ERR_INVALID; }
  if (first_error_row) *first_error_row = -1;
  int32_t ndev = 0;
  DBX_TRY(dbx_device_count(&ndev));
  if (device < 0 || device >= ndev) { err.set("dbx_eval_scalar: device index out of range"); return DBX_ERR_INVALID; }
  DBX_CUDA_TRY(err, cudaSetDevice(device));
  const int64_t n = block->num_rows;
  // ---- type inference over the postfix program
  EvalParams p;
  memset(&p, 0, sizeof(p));
  int tstack[kEvalStack];
  bool nstack[kEvalStack];  // nullable
  int sp = 0;
  auto numeric = [](int t) { return t != DBX_BOOL && t != DBX_VEC_F32 && dtype_size(t) > 0; };
  for (int i = 0; i < expr->n_nodes; ++i) {
    const dbx_expr_node& in = expr->nodes[i];
    NodeDev& nd = p.nodes[i];
    nd.kind = in.kind; nd.func = in.func;
    if (in.kind == DBX_EXPR_COLUMN) {
      if (in.col < 0 || in.col >= block->num_cols) { err.set("eval: column index outside the block"); return DBX_ERR_INVALID; }
      const dbx_column& c = block->cols[in.col];
      if (c.dtype == DBX_VEC_F32 || (c.dtype != DBX_BOOL && dtype_size(c.dtype) == 0)) { err.set("eval: only numeric and boolean columns"); return DBX_ERR_UNSUPPORTED; }
      if (sp >= kEvalStack) { err.set("eval: expression too deep"); return DBX_ERR_UNSUPPORTED; }
      nd.col = in.col; nd.out = c.dtype;
      tstack[sp] = c.dtype; nstack[sp] = c.validity != nullptr || (c.is_const && c.konst.is_null); ++sp;
    } else if (in.kind == DBX_EXPR_CONST) {
      if (sp >= kEvalStack) { err.set("eval: expression too deep"); return DBX_ERR_UNSUPPORTED; }
      const int t = in.c.dtype;
      nd.out = t; nd.c_null = in.c.is_null;
      if (t == DBX_F32) { const double d = (double)(float)in.c.v.f64; memcpy(&nd.c_bits, &d, 8); }
      else nd.c_bits = in.c.v.u64;
      tstack[sp] = t; nstack[sp] = in.c.is_null != 0; ++sp;
    } else if (in.kind == DBX_EXPR_CAST) {
      if (sp < 1) { err.set("eval: malformed postfix program"); return DBX_ERR_INVALID; }
      const int to = in.cast_to;
      if (to != DBX_BOOL && !numeric(to)) { err.set("eval: cast target must be numeric or boolean"); return DBX_ERR_UNSUPPORTED; }
      nd.a_type = tstack[sp - 1]; nd.out = to; nd.try_cast = in.try_cast;
      tstack[sp - 1] = to; nstack[sp - 1] = nstack[sp - 1] || in.try_cast;
    } else if (in.kind == DBX_EXPR_CALL) {
      const int f = in.func;
      const bool unary = f == DBX_FN_NOT || f == DBX_FN_NEGATE || f == DBX_FN_IS_NULL || f == DBX_FN_IS_NOT_NULL;
      if (sp < (unary ? 1 : 2)) { err.set("eval: malformed postfix program"); return DBX_ERR_INVALID; }
      if (unary) {
        const int ta = tstack[sp - 1];
        nd.a_type = ta;
        if (f == DBX_FN_NOT) { if (ta != DBX_BOOL) { err.set("eval: not() needs a Boolean argument"); return DBX_ERR_INVALID; } nd.out = DBX_BOOL; }
        else if (f == DBX_FN_NEGATE) { if (!numeric(ta)) { err.set("eval: minus() needs a numeric argument"); return DBX_ERR_INVALID; } nd.out = type_negate(ta); }
        else { nd.out = DBX_BOOL; nstack[sp - 1] = false; }
        tstack[sp - 1] = nd.out;
        continue;
      }
      const int ta = tstack[sp - 2], tb = tstack[sp - 1];
      nd.a_type = ta; nd.b_type = tb;
      const bool nullable = nstack[sp - 2] || nstack[sp - 1];
      int to;
      switch (f) {
        case DBX_FN_PLUS: case DBX_FN_MULTIPLY: case DBX_FN_MINUS: case DBX_FN_DIVIDE: case DBX_FN_DIV: case DBX_FN_MODULO:
          if (!numeric(ta) || !numeric(tb)) { err.set("eval: arithmetic needs numeric arguments"); return DBX_ERR_INVALID; }
          to = f == DBX_FN_MINUS ? type_minus(ta, tb) : f == DBX_FN_DIVIDE ? DBX_F64 : f == DBX_FN_DIV ? type_intdiv(ta, tb)
               : f == DBX_FN_MODULO ? type_modulo(ta, tb) : type_add_mul(ta, tb);
          nd.m_type = type_super(ta, tb);
          break;
        case DBX_FN_EQ: case DBX_FN_NOTEQ: case DBX_FN_LT: case DBX_FN_LTE: case DBX_FN_GT: case DBX_FN_GTE:
          if (ta != tb) { err.set("eval: comparison arguments must have one type (the type checker casts both sides to their common super type: add DBX_EXPR_CAST nodes)"); return DBX_ERR_INVALID; }
          to = DBX_BOOL;
          break;
        case DBX_FN_AND: case DBX_FN_OR:
          if (ta != DBX_BOOL || tb != DBX_BOOL) { err.set("eval: and / or need Boolean arguments"); return DBX_ERR_INVALID; }
          to = DBX_BOOL;
          break;
        default: err.set("eval: unknown function"); return DBX_ERR_INVALID;
      }
      nd.out = to;
      sp -= 1;
      tstack[sp - 1] = to; nstack[sp - 1] = nullable;
    } else { err.set("eval: unknown node kind"); return DBX_ERR_INVALID; }
  }
  if (sp != 1) { err.set("eval: postfix program does not reduce to one value"); return DBX_ERR_INVALID; }
  const int ot = tstack[0];
  const bool o_nullable = nstack[0];
  if (out_dtype) *out_dtype = ot | (o_nullable ? DBX_NULLABLE : 0);

  cudaStream_t st = nullptr;
  DBX_CUDA_TRY(err, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } guard{st};
  // ---- inputs on the device
  std::vector<DevBuf> owned;
  p.n_cols = block->num_cols;
  for (int c = 0; c < block->num_cols; ++c) {
    const dbx_column& col = block->cols[c];
    DevCol& dc = p.cols[c];
    memset(&dc, 0, sizeof(dc));
    dc.dtype = col.dtype;
    if (col.dtype == DBX_VEC_F32 || (col.dtype != DBX_BOOL && dtype_size(col.dtype) == 0)) continue;  // never referenced (checked above)
    if (col.len != n) { err.set("eval: column length differs from num_rows"); return DBX_ERR_INVALID; }
    if (col.is_const) {
      dc.is_const = col.konst.is_null ? 2 : 1;
      if (col.dtype == DBX_F32 || col.dtype == DBX_F64) { const double d = col.dtype == DBX_F32 ? (double)(float)col.konst.v.f64 : col.konst.v.f64; memcpy(&dc.const_bits, &d, 8); }
      else dc.const_bits = col.konst.v.u64;
      continue;
    }
    if (col.mem == DBX_MEM_DEVICE) { dc.data = col.data; dc.validity = col.validity; dc.vbit_off = col.validity_bit_offset; dc.dbit_off = col.data_bit_offset; continue; }
    const bool is_bool = col.dtype == DBX_BOOL;
    const int64_t b0 = is_bool ? col.data_bit_offset >> 3 : 0;
    const size_t bytes = is_bool ? (size_t)(((col.data_bit_offset + n + 7) >> 3) - b0) : (size_t)n * dtype_size(col.dtype);
    owned.emplace_back();
    DBX_CUDA_TRY(err, owned.back().ensure(bytes ? bytes : 1));
    if (bytes) DBX_CUDA_TRY(err, cudaMemcpyAsync(owned.back().p, (const char*)col.data + b0, bytes, cudaMemcpyHostToDevice, st));
    dc.data = owned.back().p;
    dc.dbit_off = is_bool ? (col.data_bit_offset & 7) : 0;
    if (col.validity) {
      const int64_t v0 = col.validity_bit_offset >> 3, v1 = (col.validity_bit_offset + n + 7) >> 3;
      owned.emplace_back();
      DBX_CUDA_TRY(err, owned.back().ensure((size_t)std::max<int64_t>(v1 - v0, 1)));
      if (v1 > v0) DBX_CUDA_TRY(err, cudaMemcpyAsync(owned.back().p, col.validity + v0, (size_t)(v1 - v0), cudaMemcpyHostToDevice, st));
      dc.validity = (const uint8_t*)owned.back().p;
      dc.vbit_off = col.validity_bit_offset & 7;
    }
  }
  // ---- output
  auto ob = std::make_unique<OwnedBlock>();
  ob->device = device;
  const size_t esz = ot == DBX_BOOL ? 1 : dtype_size(ot);
  void *od = nullptr, *ov = nullptr, *ferr = nullptr;
  DBX_CUDA_TRY(err, pool_alloc(device, st, (size_t)std::max<int64_t>(n, 1) * esz, &od));
  ob->dev_allocs.push_back(od);
  if (o_nullable) { DBX_CUDA_TRY(err, pool_alloc(device, st, (size_t)std::max<int64_t>(n, 1), &ov)); ob->dev_allocs.push_back(ov); }
  DBX_CUDA_TRY(err, pool_alloc(device, st, 8, &ferr));
  ob->dev_allocs.push_back(ferr);
  DBX_CUDA_TRY(err, cudaMemsetAsync(ferr, 0xFF, 8, st));
  p.n_nodes = expr->n_nodes; p.n_rows = n; p.out_data = od; p.out_valid = (uint8_t*)ov; p.out_dtype = ot;
  p.first_error = (unsigned long long*)ferr;
  if (n) {
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, (int64_t)kNumSMs * 8));
    // A straight-line kernel generated for this expression (NVRTC, cached per expression shape, types
    // and literals); without NVRTC, or with DBX_EVAL_JIT=0, the interpreter serves it — same results.
    // DBX_EVAL_JIT=2 is strict: a generated kernel that cannot be compiled or launched is an error
    // instead of a silent fall-back, so a caller can prove the generated kernel ran.
    cudaKernel_t jk = nullptr;
    const char* jit_env = getenv("DBX_EVAL_JIT");
    const int jit_mode = jit_env ? atoi(jit_env) : 1;
    std::string why;
    if (jit_mode != 0 && !jit_get_kernel(specialised_source(p), "dbx_jit_eval", &jk, &why)) jk = nullptr;
    bool launched = false;
    if (jk) {
      void* args[] = {(void*)&p};
      const cudaError_t ce = cudaLaunchKernel((const void*)jk, dim3(grid), dim3(256), args, 0, st);
      if (ce == cudaSuccess) launched = true;
      else { why = std::string("cudaLaunchKernel: ") + cudaGetErrorString(ce); cudaGetLastError(); }
    }
    if (!launched && jit_mode == 2) {
      cudaStreamSynchronize(st);  // the input uploads still read host memory the caller may free
      err.set("eval: DBX_EVAL_JIT=2 and the generated kernel did not run: " + why);
      return DBX_ERR_UNSUPPORTED;
    }
    if (!launched) eval_kernel<<<grid, 256, 0, st>>>(p);
    count_launch();
    DBX_CUDA_TRY(err, cudaGetLastError());
  }
  dbx_column oc;
  memset(&oc, 0, sizeof(oc));
  oc.dtype = ot; oc.mem = DBX_MEM_DEVICE; oc.len = n; oc.data = od;
  auto pack = [&](const void* bytes, const void** dst) -> int32_t {
    void* bits = nullptr;
    DBX_CUDA_TRY(err, pool_alloc(device, st, (size_t)(n + 7) / 8 + 8, &bits));
    ob->dev_allocs.push_back(bits);
    if (n) { eval_pack_bits_kernel<<<(int)std::max<int64_t>(1, std::min<int64_t>(((n + 7) / 8 + 255) / 256, (int64_t)kNumSMs * 8)), 256, 0, st>>>((const uint8_t*)bytes, n, (uint8_t*)bits); count_launch(); }
    *dst = bits;
    return DBX_OK;
  };
  if (ot == DBX_BOOL) DBX_TRY(pack(od, &oc.data));
  if (o_nullable) { const void* vb = nullptr; DBX_TRY(pack(ov, &vb)); oc.validity = (const uint8_t*)vb; oc.null_count = -1; }
  unsigned long long herr = ~0ULL;
  DBX_CUDA_TRY(err, cudaMemcpyAsync(&herr, ferr, 8, cudaMemcpyDeviceToHost, st));
  DBX_CUDA_TRY(err, cudaStreamSynchronize(st));
  if (herr != ~0ULL) {  // EvalContext::render_error: "<message>, during run expr" with the first failing row
    const int code = (int)(herr & 0xFF);
    const int64_t row = (int64_t)(herr >> 8);
    if (first_error_row) *first_error_row = row;
    const char* msg = code == ERR_DIV_ZERO ? "Division by zero" : code == ERR_DIVIDED_BY_ZERO ? "divided by zero" : "number overflowed";
    err.set(std::string(msg) + " while evaluating the expression (first failing row " + std::to_string(row) + ")");
    return DBX_ERR_BAD_ARGUMENTS;
  }
  ob->cols.push_back(oc);
  int32_t rc = pull_owned_block(ob, device, st, err, out_mem, out);
  if (rc == DBX_OK) out->num_rows = n;
  return rc;
}

// Generates and compiles (no GPU needed) the straight-line kernel of a canned program that touches
// every node kind: cast(c0 % 7 as Int64) > -cast(c1 as Int64) and not(is_null(c1)).
extern "C" int32_t dbx_eval_jit_selftest(char* msg, int32_t msg_cap) {
  EvalParams p;
  memset(&p, 0, sizeof(p));
  int i = 0;
  auto node = [&](int kind, int func, int col, int out, int a, int b, int m, uint64_t c) {
    NodeDev& n = p.nodes[i++];
    n.kind = kind; n.func = func; n.col = col; n.out = out; n.a_type = a; n.b_type = b; n.m_type = m; n.c_bits = c;
  };
  node(DBX_EXPR_COLUMN, 0, 0, DBX_I64, 0, 0, 0, 0);
  node(DBX_EXPR_CONST, 0, 0, DBX_U8, 0, 0, 0, 7);
  node(DBX_EXPR_CALL, DBX_FN_MODULO, 0, DBX_I16, DBX_I64, DBX_U8, DBX_I64, 0);
  node(DBX_EXPR_CAST, 0, 0, DBX_I64, DBX_I16, 0, 0, 0);
  node(DBX_EXPR_COLUMN, 0, 1, DBX_F64, 0, 0, 0, 0);
  node(DBX_EXPR_CAST, 0, 0, DBX_I64, DBX_F64, 0, 0, 0);
  node(DBX_EXPR_CALL, DBX_FN_NEGATE, 0, DBX_I64, DBX_I64, 0, 0, 0);
  node(DBX_EXPR_CALL, DBX_FN_GT, 0, DBX_BOOL, DBX_I64, DBX_I64, 0, 0);
  node(DBX_EXPR_COLUMN, 0, 1, DBX_F64, 0, 0, 0, 0);
  node(DBX_EXPR_CALL, DBX_FN_IS_NULL, 0, DBX_BOOL, DBX_F64, 0, 0, 0);
  node(DBX_EXPR_CALL, DBX_FN_NOT, 0, DBX_BOOL, DBX_BOOL, 0, 0, 0);
  node(DBX_EXPR_CALL, DBX_FN_AND, 0, DBX_BOOL, DBX_BOOL, DBX_BOOL, 0, 0);
  p.n_nodes = i;
  p.out_dtype = DBX_BOOL;
  std::string why;
  cudaKernel_t k = nullptr;
  const bool ok = jit_get_kernel(specialised_source(p), "dbx_jit_eval", &k, &why, /*compile_only=*/true);
  if (msg && msg_cap > 0) snprintf(msg, (size_t)msg_cap, "%s", ok ? "ok" : why.c_str());
  return ok ? DBX_OK : DBX_ERR_UNSUPPORTED;
}
