// Host API of the sm_100a tcgen05 grouped GEMM family (see gemm_sm100.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace tb {

enum GemmEpilogue : int {
  EPI_NONE = 0,       // D = acc * alpha
  EPI_BIAS = 1,       // D = acc + bias[n]
  EPI_BIAS_RELU = 2,  // D = relu(acc + bias[n])        (bias optional)
  EPI_BIAS_GELU = 3,  // D = gelu_erf(acc + bias[n])      (d2, when given, receives the pre-activation acc + bias)
  EPI_BIAS_SILU = 4,  // D = silu(acc + bias[n])          (same)
  EPI_RELU_BWD = 5,   // D = aux[m,n] > 0 ? acc : 0     (aux = forward activation output)
  EPI_GLU = 6,        // dual-B: D = act(A*B) .* (A*B2); optionally also stores g = A*B -> d2 and u = A*B2 -> d3
  EPI_GLU_BWD = 7,    // acc = dh:  D = dh * u * act'(g)  and  d2 = dh * act(g)   with g = aux, u = aux2
  EPI_ADD = 8,        // D = acc + aux[m,n]
  EPI_ACT_BWD = 9,    // D = acc * act'(aux[m,n])        (aux = forward PRE-activation; act = GemmProblem::act)
};

enum GemmAct : int { ACT_RELU = 1, ACT_GELU = 2, ACT_SILU = 3 };

enum GemmDtype : int { DT_BF16 = 0, DT_FP16 = 1, DT_FP32 = 2, DT_E4M3 = 3, DT_E5M2 = 4 };

// One launch computes, for every group g in [0,G):
//     D_g[M,N] = epilogue( A_g[M,K] * B_{g / b_group_div}[K,N] )
// A is "K-major" when element (m,k) is at a + m*lda + k, "MN-major" when it is at a + k*lda + m.
// B is "K-major" when element (k,n) is at b + n*ldb + k (i.e. an [N,K] row-major weight), "MN-major" when at
// b + k*ldb + n ([K,N] row-major).  D is always row-major [M,N].
struct GemmProblem {
  int M = 0, N = 0, K = 0, G = 1;
  int b_group_div = 1;

  const void* a = nullptr;
  long long lda = 0, a_group_stride = 0;  // in elements
  bool a_mn_major = false;
  const void* b = nullptr;
  long long ldb = 0, b_group_stride = 0;
  bool b_mn_major = false;
  int in_dtype = DT_BF16;  // A and B element type
  // EPI_GLU only: second B operand with the layout / strides of `b`.  One 256-wide accumulator tile then holds 128
  // columns of A*B ("gate") and the SAME 128 columns of A*B2 ("up"); with CTA pairs each CTA stages one of the two
  // weight tiles, so the gated activation costs no extra shared-memory traffic and no separate elementwise pass.
  const void* b2 = nullptr;
  int act = ACT_SILU;      // activation of EPI_GLU / EPI_GLU_BWD

  void* d = nullptr;
  long long ldd = 0, d_group_stride = 0;
  int out_dtype = DT_BF16;
  // Optional: per-group output base pointers (device array of G uint64). Entries may point into PEER GPUs'
  // memory (NVLink P2P mapping): this is how the GEMM->combine all-to-all is fused into the epilogue.
  const unsigned long long* d_ptr_table = nullptr;
  void* d2 = nullptr;  // extra outputs of the GLU epilogues (strides / dtype of `d`)
  void* d3 = nullptr;

  int epilogue = EPI_NONE;
  float alpha = 1.0f;
  const void* bias = nullptr;  // [G / b_group_div, N], same dtype as A/B
  long long bias_group_stride = 0;
  const void* aux = nullptr;  // [G, M, N] row-major, out_dtype
  long long ld_aux = 0, aux_group_stride = 0;
  const void* aux2 = nullptr;  // EPI_GLU_BWD: the "up" pre-activation (strides of `aux`)

  // fp8 (e4m3 / e5m2, K-major) operands: optional per-row scales of A [G, M] and per-column scales of B [G/div, N]
  // (fp32); the epilogue computes D = acc * scale_a[m] * scale_b[n] before bias / activation.
  const float* scale_a = nullptr;
  long long scale_a_group_stride = 0;
  const float* scale_b = nullptr;
  long long scale_b_group_stride = 0;
  const float* scale_b2 = nullptr;  // column scales of b2 (stride of scale_b)

  // Optional: fp32 [G/div, N] accumulator that receives (atomically) the column sums of the stored result - the bias
  // gradient of the layer, fused into the dgrad GEMM instead of a separate reduction pass.  Must be zeroed by the caller.
  float* colsum = nullptr;
  long long colsum_group_stride = 0;

  // Optional: valid rows per group (device int32[G]); row tiles past the count are skipped entirely
  // (dropless / Megablocks path: no host sync, no padded FLOPs).
  const int* row_counts = nullptr;

  // Optional dispatch fusion: before the A rows [m0, m0+BM) of group g are loaded, the TMA producer
  // acquires  wait_flags[g * wait_flags_per_group + m0 / wait_rows_per_flag] >= wait_target  (system scope);
  // peers bump these counters after pushing token rows over NVLink.  ceil(M / wait_rows_per_flag) (rows per flag
  // default to the tile height) must not exceed 64 nor wait_flags_per_group.
  const uint32_t* wait_flags = nullptr;
  int wait_rows_per_flag = 0, wait_flags_per_group = 0;
  uint32_t wait_target = 0;
  // Optional combine fusion: after an output tile of group g is stored, signal_ptr_table[g] (a uint32 counter,
  // usually in a peer's memory) is incremented with release.sys semantics.
  const unsigned long long* signal_ptr_table = nullptr;
  // Tile order: group g is visited as (g/mod)*mod + (g%mod + rot)%mod, so a rank can start with the segment whose
  // rows it produced itself while the peers' rows are still in flight.  A negative mod visits the segment downwards.
  // group_rot must be >= 0; when |mod| > 1, |mod| must divide G and group_rot must be < |mod|.
  int group_rot = 0, group_mod = 1;

  // Tuning: cta_group (1 or 2, 0 = auto), BN (128 or 256, 0 = auto)
  int cta_group = 0;
  int block_n = 0;
  int max_ctas = 0;  // 0 = all SMs; at least one CTA (one pair with cta_group 2) always runs
};

// Returns cudaSuccess or the launch error; throws nothing.  `why` (optional) receives a static message on
// argument errors (misaligned strides, A/B not bf16 / fp16 / e4m3 / e5m2, group_rot / group_mod or wait-flag
// counts out of range, etc.).  The sizes of the side tensors (bias, aux, scales, colsum) are not visible here: the
// caller guarantees them (the torch bindings check them against the tensor shapes).
cudaError_t gemm_sm100_launch(const GemmProblem& p, cudaStream_t stream, const char** why = nullptr);

}  // namespace tb
