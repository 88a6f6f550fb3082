// pybind11 / torch bindings for the tutel_b200 native runtime (`tutel_b200._C`).
#include <ATen/cuda/CUDAContext.h>
#include <c10/cuda/CUDAGuard.h>
#include <torch/extension.h>

#include <string>
#include <vector>

#include "cpu_kernels.h"
#include "gemm_mx.h"
#include "gemm_sm100.h"
#include "jit_nvrtc.h"
#include "moe_kernels.h"
#include "p2p_kernels.h"
#include "symm_heap.h"

namespace {

#define TB_CHECK_CUDA(expr)                                                                          \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    TORCH_CHECK(_e == cudaSuccess, "tutel_b200 CUDA error: ", cudaGetErrorString(_e), " at ", #expr); \
  } while (0)

int gemm_dtype_of(const at::Tensor& t) {
  switch (t.scalar_type()) {
    case at::kBFloat16: return tb::DT_BF16;
    case at::kHalf: return tb::DT_FP16;
    case at::kFloat: return tb::DT_FP32;
    case at::kFloat8_e4m3fn: return tb::DT_E4M3;
    case at::kFloat8_e5m2: return tb::DT_E5M2;
    default: TORCH_CHECK(false, "unsupported dtype for tutel_b200 GEMM: ", t.scalar_type());
  }
}

int elem_type_of(const at::Tensor& t) {
  switch (t.scalar_type()) {
    case at::kFloat: return tb::ET_F32;
    case at::kHalf: return tb::ET_F16;
    case at::kBFloat16: return tb::ET_BF16;
    default: TORCH_CHECK(false, "unsupported dtype for tutel_b200 dispatch kernels: ", t.scalar_type());
  }
}

// A/B element type of the tcgen05 GEMM: 16-bit floats or 8-bit e4m3 / e5m2 (fp32 operands are refused, not reinterpreted)
int gemm_input_dtype_of(const at::Tensor& t, const char* who) {
  const int dt = gemm_dtype_of(t);
  TORCH_CHECK(dt != tb::DT_FP32, who, ": A/B must be bf16, fp16, float8_e4m3fn or float8_e5m2, got ", t.scalar_type());
  return dt;
}

cudaStream_t cur_stream() { return at::cuda::getCurrentCUDAStream().stream(); }

// a: [G, M, K] (a_mn=false) or [G, K, M] (a_mn=true); b: [Gb, N, K] (b_mn=false) or [Gb, K, N] (b_mn=true);
// d: [G, M, N].  Innermost dims contiguous.  Pointer-table / flag arguments are raw device addresses (0 = off).
void gemm_ex(const at::Tensor& a, const at::Tensor& b, at::Tensor& d, bool a_mn, bool b_mn, int64_t epilogue,
             const c10::optional<at::Tensor>& bias, const c10::optional<at::Tensor>& aux,
             const c10::optional<at::Tensor>& row_counts, double alpha, int64_t b_group_div, int64_t cta_group,
             int64_t block_n, int64_t d_ptr_table, int64_t signal_ptr_table, int64_t wait_flags,
             int64_t wait_rows_per_flag, int64_t wait_flags_per_group, int64_t wait_target, int64_t max_ctas,
             int64_t group_rot, int64_t group_mod, const c10::optional<at::Tensor>& scale_a,
             const c10::optional<at::Tensor>& scale_b, const c10::optional<at::Tensor>& colsum,
             const c10::optional<at::Tensor>& d2, int64_t act) {
  TORCH_CHECK(a.is_cuda() && b.is_cuda() && d.is_cuda(), "tutel_b200.gemm: CUDA tensors required");
  TORCH_CHECK(a.dim() == 3 && b.dim() == 3 && d.dim() == 3, "tutel_b200.gemm: expected 3-D operands");
  TORCH_CHECK(a.stride(2) == 1 && b.stride(2) == 1 && d.stride(2) == 1, "tutel_b200.gemm: innermost dim must be contiguous");
  TORCH_CHECK(a.scalar_type() == b.scalar_type(), "tutel_b200.gemm: A/B dtype mismatch");
  const c10::cuda::CUDAGuard guard(a.device());
  tb::GemmProblem p;
  p.G = static_cast<int>(a.size(0));
  p.M = static_cast<int>(a_mn ? a.size(2) : a.size(1));
  p.K = static_cast<int>(a_mn ? a.size(1) : a.size(2));
  p.N = static_cast<int>(b_mn ? b.size(2) : b.size(1));
  TORCH_CHECK((b_mn ? b.size(1) : b.size(2)) == p.K, "tutel_b200.gemm: K mismatch");
  TORCH_CHECK(d.size(0) == p.G && d.size(1) == p.M && d.size(2) == p.N, "tutel_b200.gemm: output shape mismatch");
  p.b_group_div = static_cast<int>(b_group_div > 0 ? b_group_div : 1);
  TORCH_CHECK(b.size(0) * p.b_group_div >= p.G, "tutel_b200.gemm: not enough B groups");
  const int64_t gB = (p.G + p.b_group_div - 1) / p.b_group_div;   // B groups (and rows of bias / scale_b / colsum) in use
  p.a = a.data_ptr(); p.lda = a.stride(1); p.a_group_stride = a.stride(0); p.a_mn_major = a_mn;
  p.b = b.data_ptr(); p.ldb = b.stride(1); p.b_group_stride = b.stride(0); p.b_mn_major = b_mn;
  p.in_dtype = gemm_input_dtype_of(a, "tutel_b200.gemm");
  p.d = d.data_ptr(); p.ldd = d.stride(1); p.d_group_stride = d.stride(0);
  p.out_dtype = gemm_dtype_of(d);
  TORCH_CHECK(p.out_dtype <= tb::DT_FP32, "tutel_b200.gemm: output must be bf16/fp16/fp32");
  p.epilogue = static_cast<int>(epilogue);
  p.alpha = static_cast<float>(alpha);
  if (bias.has_value() && bias->defined()) {
    TORCH_CHECK(bias->is_cuda() && bias->dim() == 2 && bias->stride(1) == 1 &&
                    (bias->scalar_type() == a.scalar_type() || (a.element_size() == 1 && bias->scalar_type() == d.scalar_type() && d.element_size() == 2)),
                "tutel_b200.gemm: bias must be [Gb, N] of the input dtype (fp8 inputs: of the 16-bit output dtype)");
    TORCH_CHECK(bias->size(1) == p.N && bias->size(0) >= gB, "tutel_b200.gemm: bias must be [>= ceil(G / b_group_div), N]");
    p.bias = bias->data_ptr();
    p.bias_group_stride = bias->stride(0);
  }
  if (aux.has_value() && aux->defined()) {
    TORCH_CHECK(aux->is_cuda() && aux->scalar_type() == d.scalar_type() && aux->dim() == 3 && aux->stride(2) == 1 &&
                    aux->element_size() == 2 && aux->size(0) == p.G && aux->size(1) == p.M && aux->size(2) == p.N,
                "tutel_b200.gemm: aux must be a 16-bit [G, M, N] tensor of the output dtype");
    p.aux = aux->data_ptr();
    p.ld_aux = aux->stride(1);
    p.aux_group_stride = aux->stride(0);
  }
  if (row_counts.has_value() && row_counts->defined()) {
    TORCH_CHECK(row_counts->is_cuda() && row_counts->scalar_type() == at::kInt && row_counts->numel() >= p.G);
    p.row_counts = row_counts->data_ptr<int>();
  }
  if (scale_a.has_value() && scale_a->defined()) {
    TORCH_CHECK(scale_a->is_cuda() && scale_a->scalar_type() == at::kFloat && scale_a->dim() == 2 && scale_a->stride(1) == 1 &&
                scale_a->size(0) == p.G && scale_a->size(1) == p.M, "tutel_b200.gemm: scale_a must be float [G, M]");
    p.scale_a = scale_a->data_ptr<float>();
    p.scale_a_group_stride = scale_a->stride(0);
  }
  if (scale_b.has_value() && scale_b->defined()) {
    TORCH_CHECK(scale_b->is_cuda() && scale_b->scalar_type() == at::kFloat && scale_b->dim() == 2 && scale_b->stride(1) == 1 &&
                scale_b->size(1) == p.N && scale_b->size(0) >= gB, "tutel_b200.gemm: scale_b must be float [>= ceil(G / b_group_div), N]");
    p.scale_b = scale_b->data_ptr<float>();
    p.scale_b_group_stride = scale_b->stride(0);
  }
  if (colsum.has_value() && colsum->defined()) {
    TORCH_CHECK(colsum->is_cuda() && colsum->scalar_type() == at::kFloat && colsum->dim() == 2 && colsum->stride(1) == 1 &&
                colsum->size(1) == p.N && colsum->size(0) >= gB, "tutel_b200.gemm: colsum must be float [>= ceil(G / b_group_div), N]");
    p.colsum = colsum->data_ptr<float>();
    p.colsum_group_stride = colsum->stride(0);
  }
  p.cta_group = static_cast<int>(cta_group);
  p.block_n = static_cast<int>(block_n);
  p.max_ctas = static_cast<int>(max_ctas);
  p.d_ptr_table = reinterpret_cast<const unsigned long long*>(d_ptr_table);
  p.signal_ptr_table = reinterpret_cast<const unsigned long long*>(signal_ptr_table);
  p.wait_flags = reinterpret_cast<const uint32_t*>(wait_flags);
  p.wait_rows_per_flag = static_cast<int>(wait_rows_per_flag);
  p.wait_flags_per_group = static_cast<int>(wait_flags_per_group);
  p.wait_target = static_cast<uint32_t>(wait_target);
  p.group_rot = static_cast<int>(group_rot);
  p.group_mod = static_cast<int>(group_mod != 0 ? group_mod : 1);
  if (d2.has_value() && d2->defined()) {
    TORCH_CHECK(d2->is_cuda() && d2->scalar_type() == d.scalar_type() && d2->sizes() == d.sizes() && d2->strides() == d.strides(),
                "tutel_b200.gemm: d2 must look like d");
    p.d2 = d2->data_ptr();
  }
  if (act != 0) p.act = static_cast<int>(act);
  const char* why = nullptr;
  cudaError_t e = tb::gemm_sm100_launch(p, cur_stream(), &why);
  TORCH_CHECK(e == cudaSuccess, "tutel_b200.gemm launch failed: ", why ? why : cudaGetErrorString(e));
}

void gemm(const at::Tensor& a, const at::Tensor& b, at::Tensor& d, bool a_mn, bool b_mn, int64_t epilogue,
          const c10::optional<at::Tensor>& bias, const c10::optional<at::Tensor>& aux,
          const c10::optional<at::Tensor>& row_counts, double alpha, int64_t b_group_div, int64_t cta_group,
          int64_t block_n, int64_t d_ptr_table, int64_t signal_ptr_table, int64_t wait_flags,
          int64_t wait_rows_per_flag, int64_t wait_flags_per_group, int64_t wait_target, int64_t max_ctas,
          int64_t group_rot, int64_t group_mod, const c10::optional<at::Tensor>& scale_a,
          const c10::optional<at::Tensor>& scale_b, const c10::optional<at::Tensor>& colsum) {
  gemm_ex(a, b, d, a_mn, b_mn, epilogue, bias, aux, row_counts, alpha, b_group_div, cta_group, block_n, d_ptr_table,
          signal_ptr_table, wait_flags, wait_rows_per_flag, wait_flags_per_group, wait_target, max_ctas, group_rot, group_mod,
          scale_a, scale_b, colsum, c10::nullopt, 0);
}

std::vector<at::Tensor> route_locations(const at::Tensor& idx, int64_t E, int64_t C) {
  TORCH_CHECK(idx.is_cuda() && idx.scalar_type() == at::kInt && idx.dim() == 2 && idx.is_contiguous());
  const c10::cuda::CUDAGuard guard(idx.device());
  const int k = static_cast<int>(idx.size(0)), S = static_cast<int>(idx.size(1));
  auto opts = idx.options();
  at::Tensor loc = at::empty({k, S}, opts);
  at::Tensor counts = at::empty({E}, opts);
  at::Tensor ws = at::empty({static_cast<int64_t>(tb::route_workspace_ints(S, static_cast<int>(E), k))}, opts);
  TB_CHECK_CUDA(tb::route_locations(idx.data_ptr<int>(), loc.data_ptr<int>(), counts.data_ptr<int>(),
                                    ws.data_ptr<int>(), S, static_cast<int>(E), k, cur_stream()));
  std::vector<at::Tensor> out{loc, counts};
  if (C > 0) {
    at::Tensor slot = at::empty({E * C}, opts);
    TB_CHECK_CUDA(tb::build_slot_map(idx.data_ptr<int>(), loc.data_ptr<int>(), slot.data_ptr<int>(), S,
                                     static_cast<int>(E), k, static_cast<int>(C), cur_stream()));
    out.push_back(slot);
  }
  return out;
}

at::Tensor build_slot_map(const at::Tensor& idx, const at::Tensor& loc, int64_t E, int64_t C) {
  TORCH_CHECK(idx.is_cuda() && loc.is_cuda() && idx.scalar_type() == at::kInt && loc.scalar_type() == at::kInt);
  TORCH_CHECK(idx.is_contiguous() && loc.is_contiguous() && idx.dim() == 2);
  const c10::cuda::CUDAGuard guard(idx.device());
  at::Tensor slot = at::empty({E * C}, idx.options());
  TB_CHECK_CUDA(tb::build_slot_map(idx.data_ptr<int>(), loc.data_ptr<int>(), slot.data_ptr<int>(),
                                   static_cast<int>(idx.size(1)), static_cast<int>(E), static_cast<int>(idx.size(0)),
                                   static_cast<int>(C), cur_stream()));
  return slot;
}

// x [S, M]; gates float [k, S] or None; slot_src int [E*C]; out [E*C, M] (ignored rows live in dst_ptr_table).
void encode_rows(const at::Tensor& x, const c10::optional<at::Tensor>& gates, const at::Tensor& slot_src,
                 at::Tensor& out, int64_t k, int64_t E, int64_t C, int64_t dst_ptr_table, int64_t signal_ptr_table,
                 int64_t signal_rows, int64_t rot_chunks, int64_t signal_value, int64_t chunk_counters,
                 const c10::optional<at::Tensor>& valid_rows) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 2 && x.is_contiguous() && slot_src.is_cuda() && slot_src.is_contiguous());
  TORCH_CHECK(slot_src.scalar_type() == at::kInt && slot_src.numel() == E * C);
  const c10::cuda::CUDAGuard guard(x.device());
  const void* g = nullptr;
  if (gates.has_value() && gates->defined()) {
    TORCH_CHECK(gates->is_cuda() && gates->scalar_type() == at::kFloat && gates->is_contiguous());
    g = gates->data_ptr();
  }
  const int* vr = nullptr;
  if (valid_rows.has_value() && valid_rows->defined()) {
    TORCH_CHECK(valid_rows->is_cuda() && valid_rows->scalar_type() == at::kInt && valid_rows->numel() >= E);
    vr = valid_rows->data_ptr<int>();
  }
  if (dst_ptr_table == 0)
    TORCH_CHECK(out.is_cuda() && out.is_contiguous() && out.scalar_type() == x.scalar_type() &&
                out.numel() == E * C * x.size(1));
  TB_CHECK_CUDA(tb::encode_rows(x.data_ptr(), g, slot_src.data_ptr<int>(), out.data_ptr(),
                                reinterpret_cast<const unsigned long long*>(dst_ptr_table),
                                reinterpret_cast<const unsigned long long*>(signal_ptr_table),
                                reinterpret_cast<unsigned int*>(chunk_counters), static_cast<int>(signal_rows), static_cast<int>(x.size(0)), static_cast<int>(E),
                                static_cast<int>(k), static_cast<int>(C), static_cast<int>(x.size(1)), elem_type_of(x),
                                static_cast<int>(rot_chunks), static_cast<int>(signal_value), vr, cur_stream()));
}

// fp8 dispatch: x [S, M] (16-bit) -> e4m3 rows + fp32 row scales.  Local: returns [q [E*C, M], scale [E*C]]; remote push
// (dst_ptr_table != 0): rows / scales / flags go through the pointer tables and nothing is returned.
std::vector<at::Tensor> encode_rows_fp8(const at::Tensor& x, const c10::optional<at::Tensor>& gates, const at::Tensor& slot_src,
                                        int64_t k, int64_t E, int64_t C, int64_t dst_ptr_table, int64_t scale_ptr_table,
                                        int64_t signal_ptr_table, int64_t signal_rows, int64_t rot_chunks, int64_t signal_value,
                                        int64_t chunk_counters) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 2 && x.is_contiguous() && slot_src.is_cuda() && slot_src.is_contiguous());
  TORCH_CHECK(slot_src.scalar_type() == at::kInt && slot_src.numel() == E * C && x.size(1) % 16 == 0 && x.element_size() == 2);
  const c10::cuda::CUDAGuard guard(x.device());
  const void* g = nullptr;
  if (gates.has_value() && gates->defined()) {
    TORCH_CHECK(gates->is_cuda() && gates->scalar_type() == at::kFloat && gates->is_contiguous());
    g = gates->data_ptr();
  }
  std::vector<at::Tensor> out;
  void* q = nullptr;
  float* sc = nullptr;
  if (dst_ptr_table == 0) {
    out.push_back(at::empty({E * C, x.size(1)}, x.options().dtype(at::kFloat8_e4m3fn)));
    out.push_back(at::empty({E * C}, x.options().dtype(at::kFloat)));
    q = out[0].data_ptr();
    sc = out[1].data_ptr<float>();
  } else {
    TORCH_CHECK(scale_ptr_table != 0, "encode_rows_fp8: a remote push needs scale_ptr_table");
  }
  TB_CHECK_CUDA(tb::encode_rows_fp8(x.data_ptr(), g, slot_src.data_ptr<int>(), q, sc,
                                    reinterpret_cast<const unsigned long long*>(dst_ptr_table),
                                    reinterpret_cast<const unsigned long long*>(scale_ptr_table),
                                    reinterpret_cast<const unsigned long long*>(signal_ptr_table),
                                    reinterpret_cast<unsigned int*>(chunk_counters), static_cast<int>(signal_rows),
                                    static_cast<int>(x.size(0)), static_cast<int>(E), static_cast<int>(k), static_cast<int>(C),
                                    static_cast<int>(x.size(1)), elem_type_of(x), static_cast<int>(rot_chunks),
                                    static_cast<int>(signal_value), cur_stream()));
  return out;
}

// buf [E*C, M]; gates float [k, S] or None; idx/loc int [k, S]; returns [S, M]
at::Tensor decode_rows(const at::Tensor& buf, const c10::optional<at::Tensor>& gates, const at::Tensor& idx,
                       const at::Tensor& loc, int64_t E, int64_t C, int64_t wait_flags, int64_t wait_target) {
  TORCH_CHECK(buf.is_cuda() && buf.is_contiguous() && idx.is_cuda() && loc.is_cuda());
  TORCH_CHECK(idx.scalar_type() == at::kInt && loc.scalar_type() == at::kInt && idx.is_contiguous() && loc.is_contiguous());
  const c10::cuda::CUDAGuard guard(buf.device());
  const int k = static_cast<int>(idx.size(0)), S = static_cast<int>(idx.size(1));
  const int M = static_cast<int>(buf.numel() / (E * C));
  const void* g = nullptr;
  if (gates.has_value() && gates->defined()) {
    TORCH_CHECK(gates->is_cuda() && gates->scalar_type() == at::kFloat && gates->is_contiguous());
    g = gates->data_ptr();
  }
  at::Tensor out = at::empty({S, M}, buf.options());
  TB_CHECK_CUDA(tb::decode_rows(buf.data_ptr(), g, idx.data_ptr<int>(), loc.data_ptr<int>(), out.data_ptr(),
                                reinterpret_cast<const uint32_t*>(wait_flags), static_cast<uint32_t>(wait_target), S,
                                static_cast<int>(E), k, static_cast<int>(C), M, elem_type_of(buf), cur_stream()));
  return out;
}

// a [S, M], buf [E*C, M] -> float [k, S]
at::Tensor gate_grad(const at::Tensor& a, const at::Tensor& buf, const at::Tensor& idx, const at::Tensor& loc,
                     int64_t E, int64_t C) {
  TORCH_CHECK(a.is_cuda() && a.is_contiguous() && buf.is_cuda() && buf.is_contiguous());
  TORCH_CHECK(a.scalar_type() == buf.scalar_type());
  const c10::cuda::CUDAGuard guard(a.device());
  const int k = static_cast<int>(idx.size(0)), S = static_cast<int>(idx.size(1));
  at::Tensor out = at::empty({k, S}, a.options().dtype(at::kFloat));
  TB_CHECK_CUDA(tb::gate_grad(a.data_ptr(), buf.data_ptr(), idx.data_ptr<int>(), loc.data_ptr<int>(), out.data_ptr(),
                              S, static_cast<int>(E), k, static_cast<int>(C), static_cast<int>(a.size(1)),
                              elem_type_of(a), cur_stream()));
  return out;
}

// logits [S, E] (fp32 / fp16 / bf16) -> [scores fp32 [S,E], idx int [k,S], top fp32 [k,S], gates fp32 [k,S], loc int [k,S],
// counts int [E], ce fp32 [E], l_aux (scalar, logits dtype), slot_src int [E*C] (only when C > 0)]   - two launches
std::vector<at::Tensor> gate_route_forward(const at::Tensor& logits, int64_t k, int64_t C, bool normalize, double eps) {
  TORCH_CHECK(logits.is_cuda() && logits.dim() == 2 && logits.is_contiguous(), "gate_route_forward: contiguous CUDA [S, E] logits expected");
  const c10::cuda::CUDAGuard guard(logits.device());
  const int S = static_cast<int>(logits.size(0)), E = static_cast<int>(logits.size(1));
  TORCH_CHECK(E <= 512 && k >= 1 && k <= 32 && k <= E, "gate_route_forward: needs E <= 512 and 1 <= k <= min(32, E)");
  const int tiles = tb::gate_route_tiles(S);
  auto f32 = logits.options().dtype(at::kFloat);
  auto i32 = logits.options().dtype(at::kInt);
  at::Tensor scores = at::empty({S, E}, f32);
  at::Tensor idx = at::empty({k, S}, i32), loc = at::empty({k, S}, i32), counts = at::empty({E}, i32);
  at::Tensor top = at::empty({k, S}, f32), gates = at::empty({k, S}, f32), ce = at::empty({E}, f32);
  at::Tensor l_aux = at::empty({}, logits.options());
  at::Tensor me = at::empty({tiles, E}, f32);
  at::Tensor hist = at::empty({tiles, k, E}, i32);
  at::Tensor slot;
  if (C > 0) slot = at::empty({E * C}, i32);
  TB_CHECK_CUDA(tb::gate_route_forward(logits.data_ptr(), scores.data_ptr<float>(), idx.data_ptr<int>(), top.data_ptr<float>(),
                                       gates.data_ptr<float>(), me.data_ptr<float>(), hist.data_ptr<int>(), loc.data_ptr<int>(),
                                       counts.data_ptr<int>(), C > 0 ? slot.data_ptr<int>() : nullptr, ce.data_ptr<float>(),
                                       l_aux.data_ptr(), S, E, static_cast<int>(k), static_cast<int>(C), normalize,
                                       static_cast<float>(eps), elem_type_of(logits), cur_stream()));
  std::vector<at::Tensor> out{scores, idx, top, gates, loc, counts, ce, l_aux};
  if (C > 0) out.push_back(slot);
  return out;
}

// -> d logits [S, E] in `like`'s dtype; dgates fp32 [k, S] or None; dl: scalar of `like`'s dtype or None      - one launch
at::Tensor gate_route_backward(const at::Tensor& scores, const at::Tensor& idx, const at::Tensor& top,
                               const c10::optional<at::Tensor>& dgates, const c10::optional<at::Tensor>& ce,
                               const c10::optional<at::Tensor>& dl, const at::Tensor& like, bool normalize, double eps) {
  TORCH_CHECK(scores.is_cuda() && scores.scalar_type() == at::kFloat && scores.dim() == 2 && scores.is_contiguous());
  const int S = static_cast<int>(scores.size(0)), E = static_cast<int>(scores.size(1));
  const int k = static_cast<int>(idx.size(0));
  TORCH_CHECK(idx.scalar_type() == at::kInt && idx.is_contiguous() && idx.size(1) == S);
  TORCH_CHECK(top.scalar_type() == at::kFloat && top.is_contiguous() && top.sizes() == idx.sizes());
  const float* dg_p = nullptr;
  const float* ce_p = nullptr;
  const void* dl_p = nullptr;
  if (dgates.has_value() && dgates->defined()) {
    TORCH_CHECK(dgates->scalar_type() == at::kFloat && dgates->is_contiguous() && dgates->sizes() == idx.sizes());
    dg_p = dgates->data_ptr<float>();
  }
  if (ce.has_value() && ce->defined() && dl.has_value() && dl->defined()) {
    TORCH_CHECK(ce->is_cuda() && ce->scalar_type() == at::kFloat && ce->is_contiguous() && ce->numel() == E);
    TORCH_CHECK(dl->is_cuda() && dl->scalar_type() == like.scalar_type() && dl->numel() == 1);
    ce_p = ce->data_ptr<float>();
    dl_p = dl->data_ptr();
  }
  const c10::cuda::CUDAGuard guard(scores.device());
  at::Tensor out = at::empty({S, E}, like.options());
  TB_CHECK_CUDA(tb::gate_route_backward(scores.data_ptr<float>(), idx.data_ptr<int>(), top.data_ptr<float>(), dg_p, ce_p, dl_p,
                                        out.data_ptr(), S, E, k, normalize, static_cast<float>(eps), elem_type_of(like),
                                        cur_stream()));
  return out;
}

// x [G, T, N] (last dim contiguous) -> [G, N] column sums in x's dtype (fp32 accumulation)
at::Tensor grouped_colsum(const at::Tensor& x) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 3 && x.stride(2) == 1, "grouped_colsum: CUDA [G, T, N] tensor expected");
  const c10::cuda::CUDAGuard guard(x.device());
  const int G = static_cast<int>(x.size(0)), T = static_cast<int>(x.size(1)), N = static_cast<int>(x.size(2));
  const int splits = tb::colsum_row_splits(G, T, N, static_cast<int>(x.element_size()));
  at::Tensor out = at::empty({G, N}, x.options());
  at::Tensor acc;
  if (splits > 1) acc = at::zeros({G, N}, x.options().dtype(at::kFloat));
  TB_CHECK_CUDA(tb::grouped_colsum(x.data_ptr(), x.stride(1), x.stride(0), out.data_ptr(),
                                   splits > 1 ? acc.data_ptr<float>() : nullptr, G, T, N, splits, elem_type_of(x), cur_stream()));
  if (splits > 1) out.copy_(acc);
  return out;
}

// int [S, E] -> cumsum along dim 0 minus one (int32)
at::Tensor cumsum_sub_one(const at::Tensor& data) {
  TORCH_CHECK(data.is_cuda() && data.dim() == 2, "cumsum_sub_one: CUDA [S, E] tensor expected");
  const c10::cuda::CUDAGuard guard(data.device());
  at::Tensor x = data.to(at::kInt).contiguous();
  const int S = static_cast<int>(x.size(0)), E = static_cast<int>(x.size(1));
  at::Tensor out = at::empty_like(x);
  at::Tensor ws = at::empty({static_cast<int64_t>(tb::cumsum_workspace_ints(S, E))}, x.options());
  TB_CHECK_CUDA(tb::cumsum_sub_one(x.data_ptr<int>(), out.data_ptr<int>(), ws.data_ptr<int>(), S, E, cur_stream()));
  return out;
}

std::vector<at::Tensor> quantize_rows(const at::Tensor& x) {
  TORCH_CHECK(x.is_cuda() && x.is_contiguous() && x.dim() >= 2, "quantize_rows: contiguous CUDA tensor [.., K] expected");
  const c10::cuda::CUDAGuard guard(x.device());
  const int K = static_cast<int>(x.size(-1));
  const int64_t R = x.numel() / K;
  at::Tensor q = at::empty(x.sizes(), x.options().dtype(at::kFloat8_e4m3fn));
  auto lead = x.sizes().vec();
  lead.pop_back();
  at::Tensor scale = at::empty(lead, x.options().dtype(at::kFloat));
  TB_CHECK_CUDA(tb::quantize_rows_e4m3(x.data_ptr(), q.data_ptr(), scale.data_ptr<float>(), R, K, elem_type_of(x), cur_stream()));
  return {q, scale};
}

// x [G, R, K] (16 bit) -> [qT e4m3 [G, K, R], scale fp32 [G, K]]   (transposed copy with one scale per output row)
std::vector<at::Tensor> quantize_transpose(const at::Tensor& x) {
  TORCH_CHECK(x.is_cuda() && x.is_contiguous() && x.dim() == 3 && x.element_size() == 2 && x.size(1) % 128 == 0 && x.size(2) % 64 == 0,
              "quantize_transpose: contiguous 16-bit CUDA tensor [G, R, K] with R % 128 == 0 and K % 64 == 0 expected");
  const c10::cuda::CUDAGuard guard(x.device());
  const int G = static_cast<int>(x.size(0)), R = static_cast<int>(x.size(1)), K = static_cast<int>(x.size(2));
  at::Tensor q = at::empty({G, K, R}, x.options().dtype(at::kFloat8_e4m3fn));
  at::Tensor scale = at::empty({G, K}, x.options().dtype(at::kFloat));
  at::Tensor ws = at::empty({G, K}, x.options().dtype(at::kFloat));
  TB_CHECK_CUDA(tb::quantize_transpose_e4m3(x.data_ptr(), q.data_ptr(), scale.data_ptr<float>(), ws.data_ptr<float>(), G, R, K,
                                            elem_type_of(x), cur_stream()));
  return {q, scale};
}

// q e4m3 [.., K], scale fp32 [..] -> 16-bit [.., K]
at::Tensor dequant_rows(const at::Tensor& q, const at::Tensor& scale, at::ScalarType dtype) {
  TORCH_CHECK(q.is_cuda() && q.is_contiguous() && q.scalar_type() == at::kFloat8_e4m3fn && scale.is_cuda() && scale.is_contiguous() &&
              scale.scalar_type() == at::kFloat && q.dim() >= 2 && scale.numel() * q.size(-1) == q.numel());
  const c10::cuda::CUDAGuard guard(q.device());
  at::Tensor y = at::empty(q.sizes(), q.options().dtype(dtype));
  TB_CHECK_CUDA(tb::dequant_rows_e4m3(q.data_ptr(), scale.data_ptr<float>(), y.data_ptr(), scale.numel(), static_cast<int>(q.size(-1)),
                                      elem_type_of(y), cur_stream()));
  return y;
}

// MX block-scaled fp8 (OCP MX: e4m3 elements, one UE8M0 scale per 32 K elements); see csrc/gemm_mx.cu.
// x [G, R, K] (16 bit, K % 128 == 0) -> [q e4m3 [G, R, K], sf uint8 (tile-ordered scale atoms, csrc/gemm_mx.h)]
std::vector<at::Tensor> mx_quantize(const at::Tensor& x) {
  TORCH_CHECK(x.is_cuda() && x.is_contiguous() && x.dim() == 3 && x.element_size() == 2 && x.size(2) % 128 == 0,
              "mx_quantize: contiguous 16-bit CUDA tensor [G, R, K] with K % 128 == 0 expected");
  const c10::cuda::CUDAGuard guard(x.device());
  const int G = static_cast<int>(x.size(0)), R = static_cast<int>(x.size(1)), K = static_cast<int>(x.size(2));
  at::Tensor q = at::empty({G, R, K}, x.options().dtype(at::kFloat8_e4m3fn));
  const long long sf_bytes = tb::mx_sf_bytes(G, R, K);
  at::Tensor sf = (R % 128 == 0) ? at::empty({sf_bytes}, x.options().dtype(at::kByte))
                                 : at::zeros({sf_bytes}, x.options().dtype(at::kByte));
  TB_CHECK_CUDA(tb::mx_quantize(x.data_ptr(), q.data_ptr(), sf.data_ptr(), G, R, K, elem_type_of(x), cur_stream()));
  return {q, sf};
}

// x [G, R, K] (16 bit, R % 128 == 0, K % 64 == 0) -> [qT e4m3 [G, K, R] quantised along R, sf]
std::vector<at::Tensor> mx_quantize_transpose(const at::Tensor& x) {
  TORCH_CHECK(x.is_cuda() && x.is_contiguous() && x.dim() == 3 && x.element_size() == 2 && x.size(1) % 128 == 0 && x.size(2) % 64 == 0,
              "mx_quantize_transpose: contiguous 16-bit CUDA tensor [G, R, K] with R % 128 == 0 and K % 64 == 0 expected");
  const c10::cuda::CUDAGuard guard(x.device());
  const int G = static_cast<int>(x.size(0)), R = static_cast<int>(x.size(1)), K = static_cast<int>(x.size(2));
  at::Tensor q = at::empty({G, K, R}, x.options().dtype(at::kFloat8_e4m3fn));
  const long long sf_bytes = tb::mx_sf_bytes(G, K, R);
  at::Tensor sf = (K % 128 == 0) ? at::empty({sf_bytes}, x.options().dtype(at::kByte))
                                 : at::zeros({sf_bytes}, x.options().dtype(at::kByte));
  TB_CHECK_CUDA(tb::mx_quantize_transpose(x.data_ptr(), q.data_ptr(), sf.data_ptr(), G, R, K, elem_type_of(x), cur_stream()));
  return {q, sf};
}

// d[g] = epilogue(a[g] * b[g]^T + bias[g]) :  a e4m3 [G, M, K], b e4m3 [G, N, K], scales from mx_quantize -> bf16 [G, M, N]
// epilogue: 0 none, 1 ReLU, 2 ReLU backward (d = aux > 0 ? acc : 0 with aux bf16 [G, M, N])
at::Tensor mx_gemm(const at::Tensor& a, const at::Tensor& sfa, const at::Tensor& b, const at::Tensor& sfb,
                   const c10::optional<at::Tensor>& bias, const c10::optional<at::Tensor>& aux, int64_t epilogue,
                   int64_t block_n, int64_t cta_group, int64_t max_ctas) {
  TORCH_CHECK(a.is_cuda() && b.is_cuda() && sfa.is_cuda() && sfb.is_cuda() && a.dim() == 3 && b.dim() == 3);
  TORCH_CHECK(a.is_contiguous() && b.is_contiguous() && sfa.is_contiguous() && sfb.is_contiguous());
  TORCH_CHECK(a.scalar_type() == at::kFloat8_e4m3fn && b.scalar_type() == at::kFloat8_e4m3fn &&
              sfa.scalar_type() == at::kByte && sfb.scalar_type() == at::kByte, "mx_gemm: e4m3 operands and uint8 scales expected");
  TORCH_CHECK(a.size(0) == b.size(0) && a.size(2) == b.size(2), "mx_gemm: a [G, M, K] and b [G, N, K] expected");
  const c10::cuda::CUDAGuard guard(a.device());
  tb::MxGemmProblem p;
  p.G = static_cast<int>(a.size(0)); p.M = static_cast<int>(a.size(1)); p.K = static_cast<int>(a.size(2));
  p.N = static_cast<int>(b.size(1));
  TORCH_CHECK(sfa.numel() == tb::mx_sf_bytes(p.G, p.M, p.K) && sfb.numel() == tb::mx_sf_bytes(p.G, p.N, p.K),
              "mx_gemm: scale arrays do not match the operand shapes");
  at::Tensor d = at::empty({p.G, p.M, p.N}, a.options().dtype(at::kBFloat16));
  p.a = a.data_ptr(); p.sfa = sfa.data_ptr(); p.b = b.data_ptr(); p.sfb = sfb.data_ptr(); p.d = d.data_ptr();
  p.ldd = p.N; p.d_group_stride = static_cast<long long>(p.M) * p.N;
  if (bias.has_value() && bias->defined()) {
    TORCH_CHECK(bias->is_cuda() && bias->scalar_type() == at::kBFloat16 && bias->is_contiguous() && bias->numel() == static_cast<long long>(p.G) * p.N,
                "mx_gemm: bias must be a contiguous bf16 [G, N]");
    p.bias = bias->data_ptr(); p.bias_group_stride = p.N;
  }
  if (aux.has_value() && aux->defined()) {
    TORCH_CHECK(aux->is_cuda() && aux->scalar_type() == at::kBFloat16 && aux->is_contiguous() && aux->numel() == d.numel(),
                "mx_gemm: aux must be a contiguous bf16 [G, M, N]");
    p.aux = aux->data_ptr(); p.ld_aux = p.N; p.aux_group_stride = p.d_group_stride;
  }
  p.epilogue = static_cast<int>(epilogue);
  p.block_n = static_cast<int>(block_n);
  p.cta_group = static_cast<int>(cta_group);
  p.max_ctas = static_cast<int>(max_ctas);
  const char* why = nullptr;
  cudaError_t e = tb::mx_gemm_launch(p, cur_stream(), &why);
  TORCH_CHECK(e == cudaSuccess, "mx_gemm: ", why ? why : cudaGetErrorString(e));
  return d;
}

// Gated-linear-unit GEMMs (SwiGLU / GeGLU / ReGLU experts; reference: tutel/experts/llama_ffn.py:38-41 runs three
// cuBLAS GEMMs plus separate activation and multiply kernels).
//   forward  (b2 given):  h = act(a*b) .* (a*b2)   [+ g = a*b -> d2, u = a*b2 -> d3 when given]   ONE launch
//   backward (aux given): acc = a*b (= dh);  d = dh .* u .* act'(g),  d2 = dh .* act(g)   with g = aux, u = aux2
void gemm_glu(const at::Tensor& a, const at::Tensor& b, const c10::optional<at::Tensor>& b2, at::Tensor& d,
              const c10::optional<at::Tensor>& d2, const c10::optional<at::Tensor>& d3,
              const c10::optional<at::Tensor>& aux, const c10::optional<at::Tensor>& aux2, bool b_mn, int64_t act,
              const c10::optional<at::Tensor>& scale_a, const c10::optional<at::Tensor>& scale_b,
              const c10::optional<at::Tensor>& scale_b2, const c10::optional<at::Tensor>& row_counts,
              int64_t b_group_div, int64_t cta_group, int64_t wait_flags, int64_t wait_rows_per_flag,
              int64_t wait_flags_per_group, int64_t wait_target, int64_t group_rot, int64_t group_mod, int64_t max_ctas) {
  TORCH_CHECK(a.is_cuda() && b.is_cuda() && d.is_cuda() && a.dim() == 3 && b.dim() == 3 && d.dim() == 3);
  TORCH_CHECK(a.stride(2) == 1 && b.stride(2) == 1 && d.stride(2) == 1 && a.scalar_type() == b.scalar_type());
  const c10::cuda::CUDAGuard guard(a.device());
  const bool fwd = b2.has_value() && b2->defined();
  tb::GemmProblem p;
  p.G = static_cast<int>(a.size(0));
  p.M = static_cast<int>(a.size(1));
  p.K = static_cast<int>(a.size(2));
  p.N = static_cast<int>(b_mn ? b.size(2) : b.size(1));
  TORCH_CHECK((b_mn ? b.size(1) : b.size(2)) == p.K, "tutel_b200.gemm_glu: K mismatch");
  p.b_group_div = static_cast<int>(b_group_div > 0 ? b_group_div : 1);
  TORCH_CHECK(b.size(0) * p.b_group_div >= p.G && d.size(0) == p.G && d.size(1) == p.M && d.size(2) == p.N && d.element_size() == 2);
  const int64_t gB = (p.G + p.b_group_div - 1) / p.b_group_div;
  p.cta_group = static_cast<int>(cta_group);
  p.max_ctas = static_cast<int>(max_ctas);
  p.wait_flags = reinterpret_cast<const uint32_t*>(wait_flags);
  p.wait_rows_per_flag = static_cast<int>(wait_rows_per_flag);
  p.wait_flags_per_group = static_cast<int>(wait_flags_per_group);
  p.wait_target = static_cast<uint32_t>(wait_target);
  p.group_rot = static_cast<int>(group_rot);
  p.group_mod = static_cast<int>(group_mod != 0 ? group_mod : 1);
  p.a = a.data_ptr(); p.lda = a.stride(1); p.a_group_stride = a.stride(0);
  p.b = b.data_ptr(); p.ldb = b.stride(1); p.b_group_stride = b.stride(0); p.b_mn_major = b_mn;
  p.in_dtype = gemm_input_dtype_of(a, "tutel_b200.gemm_glu");
  p.d = d.data_ptr(); p.ldd = d.stride(1); p.d_group_stride = d.stride(0);
  p.out_dtype = gemm_dtype_of(d);
  p.act = static_cast<int>(act);
  auto same_as_d = [&](const at::Tensor& t) {
    return t.is_cuda() && t.scalar_type() == d.scalar_type() && t.sizes() == d.sizes() && t.strides() == d.strides();
  };
  if (fwd) {
    TORCH_CHECK(b2->scalar_type() == b.scalar_type() && b2->sizes() == b.sizes() && b2->strides() == b.strides(),
                "tutel_b200.gemm_glu: b2 must have the layout of b");
    p.epilogue = tb::EPI_GLU;
    p.b2 = b2->data_ptr();
    if (d2.has_value() && d2->defined()) {
      TORCH_CHECK(d3.has_value() && d3->defined() && same_as_d(*d2) && same_as_d(*d3), "tutel_b200.gemm_glu: d2/d3 must look like d");
      p.d2 = d2->data_ptr();
      p.d3 = d3->data_ptr();
    }
  } else {
    TORCH_CHECK(aux.has_value() && aux2.has_value() && d2.has_value() && same_as_d(*d2) && same_as_d(*aux) &&
                    aux2->scalar_type() == d.scalar_type() && aux2->sizes() == aux->sizes() && aux2->strides() == aux->strides(),
                "tutel_b200.gemm_glu: backward needs aux, aux2 and d2 shaped like d");
    p.epilogue = tb::EPI_GLU_BWD;
    p.aux = aux->data_ptr(); p.ld_aux = aux->stride(1); p.aux_group_stride = aux->stride(0);
    p.aux2 = aux2->data_ptr();
    p.d2 = d2->data_ptr();
  }
  auto scale = [&](const c10::optional<at::Tensor>& t, int64_t rows, int64_t cols, const float** ptr, long long* stride) {
    if (!t.has_value() || !t->defined()) return;
    TORCH_CHECK(t->is_cuda() && t->scalar_type() == at::kFloat && t->dim() == 2 && t->stride(1) == 1 && t->size(0) >= rows &&
                    t->size(1) == cols,
                "tutel_b200.gemm_glu: scales must be float [G, M] (scale_a) or [>= ceil(G / b_group_div), N] (scale_b, scale_b2)");
    *ptr = t->data_ptr<float>();
    if (stride) *stride = t->stride(0);
  };
  scale(scale_a, p.G, p.M, &p.scale_a, &p.scale_a_group_stride);
  scale(scale_b, gB, p.N, &p.scale_b, &p.scale_b_group_stride);
  long long s2 = p.scale_b_group_stride;
  scale(scale_b2, gB, p.N, &p.scale_b2, &s2);
  TORCH_CHECK(s2 == p.scale_b_group_stride, "tutel_b200.gemm_glu: scale_b / scale_b2 stride mismatch");
  if (row_counts.has_value() && row_counts->defined()) {
    TORCH_CHECK(row_counts->is_cuda() && row_counts->scalar_type() == at::kInt && row_counts->numel() >= p.G);
    p.row_counts = row_counts->data_ptr<int>();
  }
  const char* why = nullptr;
  cudaError_t e = tb::gemm_sm100_launch(p, cur_stream(), &why);
  TORCH_CHECK(e == cudaSuccess, "tutel_b200.gemm_glu launch failed: ", why ? why : cudaGetErrorString(e));
}

at::Tensor skinny_gemm(const at::Tensor& x, const at::Tensor& w, const c10::optional<at::Tensor>& bias,
                       const c10::optional<at::Tensor>& counts, bool w_is_kn, bool relu) {
  TORCH_CHECK(x.is_cuda() && w.is_cuda() && x.dim() == 3 && w.dim() == 3 && x.is_contiguous() && w.is_contiguous());
  TORCH_CHECK(x.scalar_type() == w.scalar_type() && x.size(0) == w.size(0));
  const c10::cuda::CUDAGuard guard(x.device());
  const int G = static_cast<int>(x.size(0)), R = static_cast<int>(x.size(1)), K = static_cast<int>(x.size(2));
  const int N = static_cast<int>(w_is_kn ? w.size(2) : w.size(1));
  TORCH_CHECK((w_is_kn ? w.size(1) : w.size(2)) == K, "skinny_gemm: K mismatch");
  at::Tensor y = at::zeros({G, R, N}, x.options());
  const void* b = nullptr;
  if (bias.has_value() && bias->defined()) {
    TORCH_CHECK(bias->is_cuda() && bias->is_contiguous() && bias->scalar_type() == x.scalar_type() && bias->numel() == static_cast<int64_t>(G) * N);
    b = bias->data_ptr();
  }
  const int* c = nullptr;
  if (counts.has_value() && counts->defined()) {
    TORCH_CHECK(counts->is_cuda() && counts->scalar_type() == at::kInt && counts->numel() >= G);
    c = counts->data_ptr<int>();
  }
  TB_CHECK_CUDA(tb::skinny_grouped_gemm(x.data_ptr(), w.data_ptr(), b, y.data_ptr(), c, G, R, N, K, w_is_kn, relu,
                                        elem_type_of(x), cur_stream()));
  return y;
}

// x [G, R, K], w1 [G, H, K], w2 [G, H, N], biases [G, H] / [G, N] or None, counts int [G] or None -> fp32 [G, R, N]
at::Tensor skinny_ffn(const at::Tensor& x, const at::Tensor& w1, const c10::optional<at::Tensor>& b1, const at::Tensor& w2,
                      const c10::optional<at::Tensor>& b2, const c10::optional<at::Tensor>& counts, int64_t act) {
  TORCH_CHECK(x.is_cuda() && x.dim() == 3 && w1.dim() == 3 && w2.dim() == 3 && x.is_contiguous() && w1.is_contiguous() && w2.is_contiguous());
  TORCH_CHECK(x.scalar_type() == w1.scalar_type() && x.scalar_type() == w2.scalar_type() && x.size(0) == w1.size(0) && x.size(0) == w2.size(0));
  const c10::cuda::CUDAGuard guard(x.device());
  const int G = static_cast<int>(x.size(0)), R = static_cast<int>(x.size(1)), K = static_cast<int>(x.size(2));
  const int H = static_cast<int>(w1.size(1)), N = static_cast<int>(w2.size(2));
  TORCH_CHECK(w1.size(2) == K && w2.size(1) == H, "skinny_ffn: weight shapes do not match");
  at::Tensor y = at::zeros({G, R, N}, x.options().dtype(at::kFloat));
  auto opt_ptr = [&](const c10::optional<at::Tensor>& t, int64_t n) -> const void* {
    if (!t.has_value() || !t->defined()) return nullptr;
    TORCH_CHECK(t->is_cuda() && t->is_contiguous() && t->scalar_type() == x.scalar_type() && t->numel() == n);
    return t->data_ptr();
  };
  const int* c = nullptr;
  if (counts.has_value() && counts->defined()) {
    TORCH_CHECK(counts->is_cuda() && counts->scalar_type() == at::kInt && counts->numel() >= G);
    c = counts->data_ptr<int>();
  }
  TB_CHECK_CUDA(tb::skinny_grouped_ffn(x.data_ptr(), w1.data_ptr(), opt_ptr(b1, static_cast<int64_t>(G) * H), w2.data_ptr(),
                                       opt_ptr(b2, static_cast<int64_t>(G) * N), y.data_ptr<float>(), c, G, R, K, H, N,
                                       static_cast<int>(act), elem_type_of(x), cur_stream()));
  return y;
}

}  // namespace

void register_symm_bindings(pybind11::module& m);  // symm_heap.cpp / p2p bindings
void register_cpu_bindings(pybind11::module& m);   // cpu_kernels.cpp
void register_jit_bindings(pybind11::module& m);   // jit_nvrtc.cpp

PYBIND11_MODULE(TORCH_EXTENSION_NAME, m) {
  m.doc() = "tutel_b200 native runtime: sm_100a tcgen05 grouped GEMM, routing/dispatch kernels, symmetric heap, "
            "P2P collectives, NVRTC JIT";
  m.def("gemm", &gemm);
  m.def("gemm_ex", &gemm_ex);
  m.def("gemm_glu", &gemm_glu);
  m.def("route_locations", &route_locations);
  m.def("build_slot_map", &build_slot_map);
  m.def("encode_rows", &encode_rows);
  m.def("encode_rows_fp8", &encode_rows_fp8);
  m.def("decode_rows", &decode_rows);
  m.def("gate_grad", &gate_grad);
  m.def("gate_route_forward", &gate_route_forward);
  m.def("gate_route_backward", &gate_route_backward);
  m.def("grouped_colsum", &grouped_colsum);
  m.def("cumsum_sub_one", &cumsum_sub_one);
  m.def("skinny_gemm", &skinny_gemm);
  m.def("skinny_ffn", &skinny_ffn);
  m.def("quantize_rows", &quantize_rows);
  m.def("dequant_rows", &dequant_rows);
  m.def("quantize_transpose", &quantize_transpose);
  m.def("mx_quantize", &mx_quantize);
  m.def("mx_quantize_transpose", &mx_quantize_transpose);
  m.def("mx_gemm", &mx_gemm);
  register_symm_bindings(m);
  register_cpu_bindings(m);
  register_jit_bindings(m);
}
