// tcgen05 / TMEM / TMA grouped GEMM for sm_100a (B200).
//
// Replaces the reference's cuBLAS `torch.matmul` expert GEMMs (tutel/experts/ffn.py:114-118,
// tutel/experts/llama_ffn.py:38-41) and its host-synchronised per-expert loop
// `sparse_bmm_infer` (tutel/custom/custom_kernel.cpp:874-889) with ONE persistent, warp-specialised kernel:
//
//   warp 0      TMA producer   cp.async.bulk.tensor (128B swizzle) -> smem ring, mbarrier complete_tx
//   warp 1      MMA issuer     one thread issues tcgen05.mma (kind::f16 / kind::f8f6f4), accumulators in TMEM,
//                              tcgen05.commit releases smem slots / publishes the accumulator
//   warp 2      TMEM allocator
//   warps 4..7  epilogue       tcgen05.ld TMEM->registers, fused bias / activation / activation-grad / GLU / bias-grad
//                              math, then swizzled smem and ONE TMA tensor store per 32x32 block (side inputs arrive
//                              the same way, by tensor loads one segment ahead) - or per-row bulk stores straight
//                              into PEER GPUs' memory plus a release.sys counter bump (GEMM -> combine all-to-all
//                              fusion) - while the MMA warp already works on the next tile in the second TMEM
//                              accumulator buffer.
//
// The producer can also acquire system-scope "rows have arrived" counters before loading an A tile, which is
// how the dispatch all-to-all is overlapped tile-by-tile with the first expert GEMM.
//
// CTA_GROUP == 2 runs CTA pairs (cluster of 2) with tcgen05.mma.cta_group::2 (UMMA_M = 256): each CTA stages
// half of A's rows and half of B's columns, halving shared-memory traffic per SM.
#include "gemm_sm100.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdio>
#include <cstdlib>
#include <mutex>

#include "ptx.cuh"

namespace tb {

struct GemmArgs {
  int M, N, K, G;
  int b_group_div;
  int tiles_m, tiles_n;
  long long num_tiles;
  uint32_t idesc;
  int elt_bytes;

  void* d;
  long long ldd, d_group_stride;
  const unsigned long long* d_ptr_table;
  int out_dtype;

  int epilogue;
  float alpha;
  const void* bias;
  long long bias_group_stride;
  int bias_is_fp32;
  int bias_is_bf16;
  const void* aux;
  long long ld_aux, aux_group_stride;
  const void* aux2;
  void* d2;
  void* d3;
  int dual;        // EPI_GLU: B tile = 128 columns of tmB + the same 128 columns of tmB2
  int act;
  const float* scale_b2;

  const int* row_counts;
  float* colsum;  // [G / b_group_div, N] fp32: += column sums of the epilogue result (bias gradient), may be null
  long long colsum_group_stride;
  const float* scale_a;  // [G, M] per-row dequantisation scales (fp8 operands), may be null
  long long scale_a_group_stride;
  const float* scale_b;  // [G / b_group_div, N] per-column scales, may be null
  long long scale_b_group_stride;

  const uint32_t* wait_flags;
  int wait_rows_per_flag, wait_flags_per_group;
  uint32_t wait_target;
  const unsigned long long* signal_ptr_table;
  int staged_store;  // 16-bit outputs: stage rows in smem and write them with cp.async.bulk (full 64 B segments)
  int tma_store;     // 16-bit local outputs: stage 32x32 blocks in smem and write them with ONE tensor store each
  int tma_side;      // side inputs (aux / aux2) arrive through tensor loads into swizzled smem, one segment ahead
  int stages;        // depth of the operand ring
  int epi_warp_bytes;
  int group_rot, group_mod;  // tile order visits group (g/mod)*mod + (g%mod + rot)%mod  (own-rank segment first)
};

namespace {

constexpr int kThreads = 256;
constexpr int kSwizzleBytes = 128;   // one swizzle row: 64 bf16 / 128 fp8
constexpr int kBlockKRows = 64;      // k-rows per stage for MN-major 16-bit operands (== BK elements)
constexpr int kSmemLimit = 232448;   // 227 KB

template <int CG, int BN>
struct Cfg {
  static constexpr int BM_CTA = 128;
  static constexpr int BM = 128 * CG;
  static constexpr int BN_CTA = BN / CG;
  static constexpr int A_BYTES = BM_CTA * kSwizzleBytes;
  static constexpr int B_BYTES = BN_CTA * kSwizzleBytes;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  // Epilogue staging per epilogue warp (the host picks the size per launch and derives the ring depth from it):
  //  - local outputs: 2 KB slots of 32 rows x 64 B in the TMA SWIZZLE_64B layout, one tensor store per slot
  //    (4 slots; with side inputs: 2 store slots + 2 stages x 2 side-input slots filled by tensor loads);
  //  - remote outputs (per-group pointer table): 3 slots of 32 padded rows, one bulk store per row.
  static constexpr int EPI_ROW_BYTES = 80;                       // 64 B of payload + 16 B pad (bank-conflict free)
  static constexpr int EPI_SLOT_BYTES = 32 * EPI_ROW_BYTES;      // one warp, one 32-column chunk
  static constexpr int EPI_ROW_SLOTS = 3;
  static constexpr int EPI_TMA_SLOT_BYTES = 32 * 64;
  static constexpr int EPI_WARP_BYTES = 8192;
  static constexpr int EPI_WARP_BYTES_SIDE = 12288;
  static_assert(EPI_ROW_SLOTS * EPI_SLOT_BYTES <= EPI_WARP_BYTES, "");
  static constexpr int BAR_BYTES = 512;
  static constexpr int MAX_STAGES = 8;
  static constexpr int stages_for(int epi_warp_bytes) {
    const int n = (kSmemLimit - 1024 - BAR_BYTES - 4 * epi_warp_bytes) / STAGE_BYTES;
    return n > MAX_STAGES ? MAX_STAGES : n;
  }
  static constexpr int smem_bytes(int stages, int epi_warp_bytes) {
    return stages * STAGE_BYTES + 1024 + BAR_BYTES + 4 * epi_warp_bytes;
  }
  static_assert(stages_for(EPI_WARP_BYTES_SIDE) >= 3, "need a real pipeline");
  // 228 KB per SM, 1 KB reserved per resident block: a dispatch block (no shared memory of its own) must still fit
  static_assert(smem_bytes(stages_for(EPI_WARP_BYTES), EPI_WARP_BYTES) + 2 * 1024 <= 228 * 1024, "no room for the push kernel");
  static constexpr int TMEM_COLS = 2 * BN;  // double-buffered fp32 accumulator
  static_assert(TMEM_COLS <= 512, "TMEM has 512 columns");
};

struct TileCoord {
  int g, m_blk, n_blk;
};

// Tiles are enumerated group-major; inside a group, bands of kBand row-blocks sweep all column blocks so that a
// wave of CTAs re-uses both its A band and its B columns out of L2.
template <int kBand>
__device__ __forceinline__ TileCoord decode_tile(long long t, int tiles_m, int tiles_n) {
  const int per_group = tiles_m * tiles_n;
  TileCoord c;
  c.g = static_cast<int>(t / per_group);
  int r = static_cast<int>(t - static_cast<long long>(c.g) * per_group);
  const int band_tiles = kBand * tiles_n;
  const int band = r / band_tiles;
  const int first_m = band * kBand;
  const int rows_in_band = min(kBand, tiles_m - first_m);
  r -= band * band_tiles;
  c.m_blk = first_m + r % rows_in_band;
  c.n_blk = r / rows_in_band;
  return c;
}

// mod > 1: ascending from `rot`;  mod < -1: descending from `rot` (matches a sender that walks destinations upwards).
__device__ __forceinline__ int rotate_group(int g, int rot, int mod) {
  if (mod > 1) {
    const int base = (g / mod) * mod;
    return base + (g - base + rot) % mod;
  }
  if (mod < -1) {
    const int m = -mod;
    const int base = (g / m) * m;
    return base + (rot + m - (g - base)) % m;
  }
  return g;
}

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
__device__ __forceinline__ float silu(float x) { return __fdividef(x, 1.0f + __expf(-x)); }

__device__ __forceinline__ void unpack8(const uint4& u, bool is_bf16, float* f) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (is_bf16) {
      f[2 * i] = __uint_as_float(w[i] << 16);
      f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
    } else {
      const __half2 h = *reinterpret_cast<const __half2*>(&w[i]);
      const float2 t = __half22float2(h);
      f[2 * i] = t.x;
      f[2 * i + 1] = t.y;
    }
  }
}
// 32 floats -> 16 packed words; the dtype branch is taken ONCE per segment (a per-element branch on a kernel argument
// serialises the unrolled loop and costs all its instruction-level parallelism).
template <bool BF16>
__device__ __forceinline__ void pack32_t(const float* v, uint32_t* w) {
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    if constexpr (BF16) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    } else {
      const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<const uint32_t*>(&h);
    }
  }
}
__device__ __forceinline__ void pack32(const float* v, uint32_t* w, bool is_bf16) {
  if (is_bf16) pack32_t<true>(v, w); else pack32_t<false>(v, w);
}
template <bool BF16>
__device__ __forceinline__ void unpack32_t(const uint4* p, float* f) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const uint32_t w[4] = {p[q].x, p[q].y, p[q].z, p[q].w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if constexpr (BF16) {
        f[q * 8 + 2 * i] = __uint_as_float(w[i] << 16);
        f[q * 8 + 2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
      } else {
        const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
        f[q * 8 + 2 * i] = t.x;
        f[q * 8 + 2 * i + 1] = t.y;
      }
    }
  }
}
__device__ __forceinline__ void unpack32(const uint4* p, float* f, bool is_bf16) {
  if (is_bf16) unpack32_t<true>(p, f); else unpack32_t<false>(p, f);
}

__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }

// GLU math on one 32-column segment, activation fixed at compile time (branch-free, fully interleavable).
template <int ACT>
__device__ __forceinline__ void glu_fwd_seg(const float* g, const float* u, float* o) {
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    float a;
    if constexpr (ACT == ACT_RELU) a = fmaxf(g[j], 0.0f);
    else if constexpr (ACT == ACT_GELU) a = gelu_erf(g[j]);
    else a = g[j] * fast_sigmoid(g[j]);
    o[j] = a * u[j];
  }
}
// in: dh (as raw accumulator bits), g, u      out: o = d gate, u = d up
template <int ACT>
__device__ __forceinline__ void glu_bwd_seg(const uint32_t* r, const float* g, float* u, float* o) {
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const float dh = __uint_as_float(r[j]);
    float a, da;
    if constexpr (ACT == ACT_RELU) {
      a = fmaxf(g[j], 0.0f);
      da = g[j] > 0.0f ? 1.0f : 0.0f;
    } else if constexpr (ACT == ACT_GELU) {
      const float cdf = 0.5f * (1.0f + erff(g[j] * 0.70710678118654752f));
      a = g[j] * cdf;
      da = cdf + g[j] * 0.3989422804014327f * __expf(-0.5f * g[j] * g[j]);
    } else {
      const float sg = fast_sigmoid(g[j]);
      a = g[j] * sg;
      da = sg * (1.0f + g[j] * (1.0f - sg));
    }
    o[j] = dh * u[j] * da;
    u[j] = dh * a;
  }
}

// Resource budget (deliberate): 256 threads x 224 registers = 57344 of the SM's 65536 registers and at most 225.5 KB of
// its 228 KB shared memory, so ONE 128-thread x 64-register block of the dispatch kernel (encode_rows, which needs no
// shared memory) always fits next to a GEMM CTA.  That is what makes the dispatch+GEMM fusion deadlock-free: a GEMM
// whose producer spins on arrival flags can never starve the kernel that publishes them, whichever gets the SMs first.
// XACT selects the (rarely used) epilogues with transcendental activations - GELU / SiLU forward with the pre-activation
// saved for training, and their gradient - in their own instantiations, so that their registers do not burden the
// common ReLU / bias / GLU kernels.
template <int CG, bool A_MN, bool B_MN, int BN, int ELT, bool XACT>
__global__ void __maxnreg__(224)
gemm_sm100_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                  const __grid_constant__ CUtensorMap tmB2, const __grid_constant__ CUtensorMap tmD,
                  const __grid_constant__ CUtensorMap tmD2, const __grid_constant__ CUtensorMap tmD3,
                  const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmX2,
                  const GemmArgs args) {
  using C = Cfg<CG, BN>;
  extern __shared__ uint8_t smem_raw[];

  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0);  // warp-uniform role id
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = (CG == 2) ? ptx::cluster_ctarank() : 0u;
  const bool is_leader = (cta_rank == 0);

  // ---- shared memory carve-up (operand ring must be 1024B aligned for the 128B swizzle) ----
  const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
  const int stages = args.stages;
  const uint32_t bar_base = smem_base + static_cast<uint32_t>(stages) * C::STAGE_BYTES;
  auto smem_a = [&](int s) { return smem_base + s * C::STAGE_BYTES; };
  auto smem_b = [&](int s) { return smem_base + s * C::STAGE_BYTES + C::A_BYTES; };
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 64u + 8u * s; };
  auto tfull_bar = [&](int a) { return bar_base + 128u + 8u * a; };
  auto tempty_bar = [&](int a) { return bar_base + 144u + 8u * a; };
  const uint32_t tmem_slot = bar_base + 160u;
  auto side_bar = [&](int w, int st) { return bar_base + 192u + 8u * (w * 2 + st); };   // epilogue warp w, stage st
  const uint32_t epi_base = bar_base + C::BAR_BYTES;  // 512-byte aligned staging of the epilogue warps
  uint32_t* tmem_slot_ptr =
      reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - ptx::smem_u32(smem_raw)));

  if (warp == 0 && ptx::elect_one()) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    if (args.dual) ptx::prefetch_tensormap(&tmB2);
    if (args.tma_store) ptx::prefetch_tensormap(&tmD);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < stages; ++s) {
      ptx::mbar_init(full_bar(s), 1);
      ptx::mbar_init(empty_bar(s), 1);
    }
    for (int w = 0; w < 8; ++w) ptx::mbar_init(side_bar(w >> 1, w & 1), 1);
    for (int a = 0; a < 2; ++a) {
      ptx::mbar_init(tfull_bar(a), 1);
      ptx::mbar_init(tempty_bar(a), 4 * CG);  // one arrival per epilogue warp of every CTA in the group
    }
    ptx::fence_mbar_init();
  }
  if (warp == 2) ptx::tmem_alloc<CG>(tmem_slot, C::TMEM_COLS);
  ptx::tc_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync(); else __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot_ptr, 0);  // keep it in a uniform register

  constexpr int kEltBytes = ELT;                             // 2: fp16/bf16 (kind::f16)   1: e4m3/e5m2 (kind::f8f6f4)
  static_assert(ELT == 2 || (!A_MN && !B_MN), "8-bit operands are K-major only");
  const int num_kb = (args.K * kEltBytes + kSwizzleBytes - 1) / kSwizzleBytes;
  constexpr int bk_elems = kSwizzleBytes / kEltBytes;        // K elements per stage
  const long long tile_step = gridDim.x / CG;
  const long long tile_first = blockIdx.x / CG;
  constexpr int kBand = (CG == 2) ? 8 : 16;
  const bool dual = args.dual != 0;
  const int tile_n = dual ? BN / 2 : BN;   // output columns per tile

  if (warp == 0) {
    // =============================== TMA producer ===============================
    int s = 0;
    uint32_t ph = 0;
    int seen_group = -1;
    unsigned long long seen_mask = 0ull;
    for (long long t = tile_first; t < args.num_tiles; t += tile_step) {
      TileCoord tc = decode_tile<kBand>(t, args.tiles_m, args.tiles_n);
      tc.g = rotate_group(tc.g, args.group_rot, args.group_mod);
      if (args.row_counts != nullptr && tc.m_blk * C::BM >= args.row_counts[tc.g]) continue;
      const int m0 = tc.m_blk * C::BM + static_cast<int>(cta_rank) * C::BM_CTA;
      const int n0 = tc.n_blk * BN + static_cast<int>(cta_rank) * C::BN_CTA;   // (non-dual) first B column of this CTA
      const int gb = tc.g / args.b_group_div;
      if (args.wait_flags != nullptr) {
        // Dispatch fusion: rows of this tile are pushed by peer GPUs; acquire their release flags - once per
        // (group, flag): consecutive tiles of a group share flags, so remember which ones were already seen.
        if (tc.g != seen_group) { seen_group = tc.g; seen_mask = 0ull; }
        const int f0 = (tc.m_blk * C::BM) / args.wait_rows_per_flag;
        const int f1 = (min(tc.m_blk * C::BM + C::BM, args.M) - 1) / args.wait_rows_per_flag;
        unsigned long long need = 0ull;
        for (int f = f0; f <= f1; ++f) need |= 1ull << (f & 63);
        if ((seen_mask & need) != need) {
          if (lane == 0) {
            for (int f = f0; f <= f1; ++f)
              if (!((seen_mask >> (f & 63)) & 1ull))
                ptx::wait_flag_ge_sys(args.wait_flags + static_cast<long long>(tc.g) * args.wait_flags_per_group + f,
                                      args.wait_target);
            ptx::fence_proxy_async_global();  // order the upcoming async-proxy (TMA) reads after the acquire
          }
          __syncwarp();
          seen_mask |= need;
        }
      }
      for (int kb = 0; kb < num_kb; ++kb) {
        ptx::mbar_wait(empty_bar(s), ph ^ 1u);
        if (ptx::elect_one()) {
          const uint32_t fb = full_bar(s);
          if constexpr (CG == 1) {
            ptx::mbar_expect_tx(fb, C::STAGE_BYTES);
          } else {
            if (is_leader) ptx::mbar_expect_tx(fb, 2 * C::STAGE_BYTES);
          }
          const int k0 = kb * bk_elems;
          // ---- A ----
          if constexpr (!A_MN) {
            if constexpr (CG == 1) ptx::tma_load_3d(smem_a(s), &tmA, fb, k0, m0, tc.g);
            else ptx::tma_load_3d_2sm(smem_a(s), &tmA, fb, k0, m0, tc.g);
          } else {
            constexpr int chunk_elems = kSwizzleBytes / kEltBytes;
            const int chunk_bytes = bk_elems * kSwizzleBytes;
            const int nchunk = C::BM_CTA / chunk_elems;
            for (int c = 0; c < nchunk; ++c) {
              if constexpr (CG == 1)
                ptx::tma_load_3d(smem_a(s) + c * chunk_bytes, &tmA, fb, m0 + c * chunk_elems, k0, tc.g);
              else
                ptx::tma_load_3d_2sm(smem_a(s) + c * chunk_bytes, &tmA, fb, m0 + c * chunk_elems, k0, tc.g);
            }
          }
          // ---- B ----
          if (!dual) {
            if constexpr (!B_MN) {
              if constexpr (CG == 1) ptx::tma_load_3d(smem_b(s), &tmB, fb, k0, n0, gb);
              else ptx::tma_load_3d_2sm(smem_b(s), &tmB, fb, k0, n0, gb);
            } else {
              constexpr int chunk_elems = kSwizzleBytes / kEltBytes;
              const int chunk_bytes = bk_elems * kSwizzleBytes;
              const int nchunk = C::BN_CTA / chunk_elems;
              for (int c = 0; c < nchunk; ++c) {
                if constexpr (CG == 1)
                  ptx::tma_load_3d(smem_b(s) + c * chunk_bytes, &tmB, fb, n0 + c * chunk_elems, k0, gb);
                else
                  ptx::tma_load_3d_2sm(smem_b(s) + c * chunk_bytes, &tmB, fb, n0 + c * chunk_elems, k0, gb);
              }
            }
          } else {
            // GLU: accumulator columns [0, BN/2) come from B, [BN/2, BN) from B2, both at weight columns nb0...
            // A CTA pair splits exactly there: rank 0 stages the B tile, rank 1 the B2 tile.
            const int nb0 = tc.n_blk * (BN / 2);
            if constexpr (!B_MN) {
              if constexpr (CG == 1) {
                ptx::tma_load_3d(smem_b(s), &tmB, fb, k0, nb0, gb);
                ptx::tma_load_3d(smem_b(s) + (BN / 2) * kSwizzleBytes, &tmB2, fb, k0, nb0, gb);
              } else {
                ptx::tma_load_3d_2sm(smem_b(s), cta_rank ? &tmB2 : &tmB, fb, k0, nb0, gb);
              }
            } else {
              constexpr int chunk_elems = kSwizzleBytes / kEltBytes;
              const int chunk_bytes = bk_elems * kSwizzleBytes;
              constexpr int half_chunks = (BN / 2) / chunk_elems;
              if constexpr (CG == 1) {
                for (int c = 0; c < 2 * half_chunks; ++c)
                  ptx::tma_load_3d(smem_b(s) + c * chunk_bytes, c < half_chunks ? &tmB : &tmB2, fb,
                                   nb0 + (c % half_chunks) * chunk_elems, k0, gb);
              } else {
                for (int c = 0; c < half_chunks; ++c)
                  ptx::tma_load_3d_2sm(smem_b(s) + c * chunk_bytes, cta_rank ? &tmB2 : &tmB, fb,
                                       nb0 + c * chunk_elems, k0, gb);
              }
            }
          }
        }
        __syncwarp();
        if (++s == stages) { s = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer ===============================
    // The whole warp walks the pipeline (keeps control flow convergent, descriptors in uniform registers);
    // one elected lane issues the tcgen05 instructions.
    if (CG == 1 || is_leader) {
      int s = 0;
      uint32_t ph = 0;
      int acc = 0;
      uint32_t acc_ph = 0;
      // Descriptor = constant high word + low word {start>>4, lbo>>4}.  Advancing along K inside a stage and
      // from stage to stage only adds to the 14-bit start-address field (smem < 256 KB, so it never carries).
      constexpr uint32_t kMnChunkBytes = 64u * kSwizzleBytes;           // BK rows * 128 B (16-bit operands)
      constexpr uint32_t kMnKStep = 16u * kSwizzleBytes;                // UMMA_K rows * 128 B
      constexpr uint32_t a_lbo = A_MN ? kMnChunkBytes : 16u;
      constexpr uint32_t b_lbo = B_MN ? kMnChunkBytes : 16u;
      constexpr uint32_t a_kstep = (A_MN ? kMnKStep : 32u) >> 4;
      constexpr uint32_t b_kstep = (B_MN ? kMnKStep : 32u) >> 4;
      constexpr uint32_t desc_hi = (1024u >> 4) | (1u << 14) | (2u << 29);  // SBO | version 1 | SWIZZLE_128B
      const uint32_t a_lo0 = ((smem_a(0) >> 4) & 0x3FFFu) | ((a_lbo >> 4) << 16);
      const uint32_t b_lo0 = ((smem_b(0) >> 4) & 0x3FFFu) | ((b_lbo >> 4) << 16);
      const uint32_t idesc = args.idesc;
      for (long long t = tile_first; t < args.num_tiles; t += tile_step) {
        TileCoord tc = decode_tile<kBand>(t, args.tiles_m, args.tiles_n);
      tc.g = rotate_group(tc.g, args.group_rot, args.group_mod);
        if (args.row_counts != nullptr && tc.m_blk * C::BM >= args.row_counts[tc.g]) continue;
        ptx::mbar_wait(tempty_bar(acc), acc_ph ^ 1u);
        ptx::tc_fence_after();
        const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * BN);
        for (int kb = 0; kb < num_kb; ++kb) {
          ptx::mbar_wait(full_bar(s), ph);
          ptx::tc_fence_after();
          const uint32_t a_lo = a_lo0 + static_cast<uint32_t>(s) * (C::STAGE_BYTES >> 4);
          const uint32_t b_lo = b_lo0 + static_cast<uint32_t>(s) * (C::STAGE_BYTES >> 4);
          if (ptx::elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const uint64_t ad = (static_cast<uint64_t>(desc_hi) << 32) | (a_lo + k * a_kstep);
              const uint64_t bd = (static_cast<uint64_t>(desc_hi) << 32) | (b_lo + k * b_kstep);
              if constexpr (ELT == 2) ptx::umma_f16<CG>(d_tmem, ad, bd, idesc, (kb | k) != 0);
              else ptx::umma_f8<CG>(d_tmem, ad, bd, idesc, (kb | k) != 0);
            }
            ptx::umma_commit<CG>(empty_bar(s));                       // smem slot reusable once these retire
            if (kb == num_kb - 1) ptx::umma_commit<CG>(tfull_bar(acc));  // accumulator complete
          }
          __syncwarp();
          if (++s == stages) { s = 0; ph ^= 1u; }
        }
        if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // =============================== epilogue ===============================
    const int ew = warp - 4;  // == warp % 4: TMEM lane quarter this warp may touch
    int acc = 0;
    uint32_t acc_ph = 0;
    const bool out16 = (args.out_dtype != DT_FP32);
    const bool out_bf16 = (args.out_dtype == DT_BF16);
    const bool glu = args.epilogue == EPI_GLU || args.epilogue == EPI_GLU_BWD;
    // Output paths: (1) local 16-bit: 32x32 blocks through swizzled smem and one tensor store per block;
    // (2) remote (NVLink) 16-bit: padded smem rows and one bulk store per row (full 64-byte segments on the wire; the
    // copy engine retires only ~50 of these small operations per microsecond and SM, fine for one output per
    // accumulator);  (3) straight from registers (fp32, row_counts tails, TUTEL_B200_EPI=direct).
    const bool tma_out = out16 && args.tma_store != 0;
    const bool staged = out16 && args.staged_store != 0 && !tma_out && !glu;
    const uint32_t epi_warp = epi_base + static_cast<uint32_t>(ew) * static_cast<uint32_t>(args.epi_warp_bytes);
    int slot_toggle = 0;
    // Side inputs (activation for the ReLU mask, pre-activations of the GLU backward, addend): lane 0 asks the TMA unit
    // for the NEXT 32x32 segment (this tile's next columns, or the first segment of the next tile) while the warp works
    // on the current one; the data lands in swizzled smem and is announced on a per-warp mbarrier, so no thread ever
    // waits on a global load (there is only one epilogue warp per scheduler - nothing else could hide that latency).
    const bool side = args.tma_side != 0;
    const bool has_x2 = args.aux2 != nullptr;
    const uint32_t side_base = epi_warp + 2u * C::EPI_TMA_SLOT_BYTES;
    int side_stage = 0;
    uint32_t side_phase = 0;
    auto side_issue = [&](int st, int n, int m0, int g) {   // one lane
      const uint32_t bar = side_bar(ew, st);
      ptx::mbar_expect_tx(bar, has_x2 ? 2u * C::EPI_TMA_SLOT_BYTES : 1u * C::EPI_TMA_SLOT_BYTES);
      ptx::tma_load_3d(side_base + static_cast<uint32_t>(st * 2) * C::EPI_TMA_SLOT_BYTES, &tmX, bar, n, m0, g);
      if (has_x2) ptx::tma_load_3d(side_base + static_cast<uint32_t>(st * 2 + 1) * C::EPI_TMA_SLOT_BYTES, &tmX2, bar, n, m0, g);
    };
    auto side_coords = [&](long long t2, int& n0, int& m0, int& g) -> bool {
      if (t2 >= args.num_tiles) return false;
      TileCoord c2 = decode_tile<kBand>(t2, args.tiles_m, args.tiles_n);
      g = rotate_group(c2.g, args.group_rot, args.group_mod);
      n0 = c2.n_blk * tile_n;
      m0 = c2.m_blk * C::BM + static_cast<int>(cta_rank) * C::BM_CTA + ew * 32;
      return true;
    };
    if (side && lane == 0) {
      int n0, m0, g;
      if (side_coords(tile_first, n0, m0, g)) side_issue(0, n0, m0, g);
    }
    // The L2 is also asked for each thread's whole row segment of the NEXT tile one tile ahead, so DRAM sees long
    // contiguous requests instead of 64-byte pieces.
    auto prefetch_side = [&](long long t2) {
      if (args.aux == nullptr || t2 >= args.num_tiles) return;
      TileCoord c2 = decode_tile<kBand>(t2, args.tiles_m, args.tiles_n);
      c2.g = rotate_group(c2.g, args.group_rot, args.group_mod);
      const int m2 = c2.m_blk * C::BM + static_cast<int>(cta_rank) * C::BM_CTA + ew * 32 + lane;
      const int n2 = c2.n_blk * tile_n;
      if (m2 >= args.M || n2 >= args.N) return;
      const uint32_t bytes = static_cast<uint32_t>(min(tile_n, args.N - n2)) * 2u;
      const long long off = (static_cast<long long>(c2.g) * args.aux_group_stride + static_cast<long long>(m2) * args.ld_aux + n2) * 2;
      ptx::prefetch_l2_bulk(reinterpret_cast<const uint8_t*>(args.aux) + off, bytes);
      if (args.aux2 != nullptr) ptx::prefetch_l2_bulk(reinterpret_cast<const uint8_t*>(args.aux2) + off, bytes);
    };
    prefetch_side(tile_first);
    for (long long t = tile_first; t < args.num_tiles; t += tile_step) {
      TileCoord tc = decode_tile<kBand>(t, args.tiles_m, args.tiles_n);
      tc.g = rotate_group(tc.g, args.group_rot, args.group_mod);
      prefetch_side(t + tile_step);
      int m_valid = args.M;
      if (args.row_counts != nullptr) {
        m_valid = min(args.M, args.row_counts[tc.g]);
        if (tc.m_blk * C::BM >= m_valid) continue;
      }
      const int m = tc.m_blk * C::BM + static_cast<int>(cta_rank) * C::BM_CTA + ew * 32 + lane;
      const bool row_ok = m < m_valid;
      const int gb = tc.g / args.b_group_div;
      uint8_t* d_base = (args.d_ptr_table != nullptr)
                            ? reinterpret_cast<uint8_t*>(args.d_ptr_table[tc.g])
                            : reinterpret_cast<uint8_t*>(args.d) +
                                  static_cast<long long>(tc.g) * args.d_group_stride * (out16 ? 2 : 4);
      uint8_t* d_row = d_base + static_cast<long long>(m) * args.ldd * (out16 ? 2 : 4);
      const uint8_t* aux_row = nullptr;
      if (args.aux != nullptr)
        aux_row = reinterpret_cast<const uint8_t*>(args.aux) +
                  (static_cast<long long>(tc.g) * args.aux_group_stride + static_cast<long long>(m) * args.ld_aux) * 2;
      const uint8_t* bias_g = nullptr;
      if (args.bias != nullptr)
        bias_g = reinterpret_cast<const uint8_t*>(args.bias) +
                 static_cast<long long>(gb) * args.bias_group_stride * (args.bias_is_fp32 ? 4 : 2);

      ptx::mbar_wait(tfull_bar(acc), acc_ph);
      ptx::tc_fence_after();
      const uint32_t t_row = tmem_base + static_cast<uint32_t>(acc * BN) + (static_cast<uint32_t>(ew * 32) << 16);

      // One 32-column segment of this thread's row -> global memory (16-bit: via a padded smem row and one bulk
      // store per row segment, or direct 16-byte stores; fp32: direct).
      const int m_warp0 = tc.m_blk * C::BM + static_cast<int>(cta_rank) * C::BM_CTA + ew * 32;
      auto store_seg = [&](const CUtensorMap* tm, uint8_t* row, int n, int ncols, const float* v) {
        uint32_t w[16];
        if (out16) pack32(v, w, out_bf16);
        if (tma_out) {
          const uint32_t slot = epi_warp + static_cast<uint32_t>(slot_toggle) * C::EPI_TMA_SLOT_BYTES;
          slot_toggle = (slot_toggle + 1) & (side ? 1 : 3);        // 2 store slots next to side-input slots, else 4
          if (lane == 0) {   // the store that used this slot has read it
            if (side) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            else asm volatile("cp.async.bulk.wait_group.read 3;" ::: "memory");
          }
          __syncwarp();
          const uint32_t my = slot + static_cast<uint32_t>(lane) * 64u;
          const uint32_t sw = (static_cast<uint32_t>(lane) >> 1) & 3u;               // SWIZZLE_64B: 16-byte unit ^= row/2 % 4
#pragma unroll
          for (int q = 0; q < 4; ++q)
            asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(my + ((static_cast<uint32_t>(q) ^ sw) << 4)),
                         "r"(w[q * 4]), "r"(w[q * 4 + 1]), "r"(w[q * 4 + 2]), "r"(w[q * 4 + 3])
                         : "memory");
          ptx::fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (m_warp0 < args.M) ptx::tma_store_3d(tm, slot, n, m_warp0, tc.g);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        } else if (staged) {
          const uint32_t slot = epi_warp + static_cast<uint32_t>(slot_toggle) * C::EPI_SLOT_BYTES +
                                static_cast<uint32_t>(lane) * C::EPI_ROW_BYTES;
          slot_toggle = slot_toggle == C::EPI_ROW_SLOTS - 1 ? 0 : slot_toggle + 1;
          asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory");  // the bulk store that used this slot has read it
#pragma unroll
          for (int q = 0; q < 4; ++q)
            asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(slot + q * 16), "r"(w[q * 4]), "r"(w[q * 4 + 1]),
                         "r"(w[q * 4 + 2]), "r"(w[q * 4 + 3])
                         : "memory");
          ptx::fence_proxy_async_smem();
          if (row_ok)
            asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(row + n * 2), "r"(slot),
                         "r"(static_cast<uint32_t>(ncols * 2))
                         : "memory");
          asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        } else if (row_ok) {
          if (out16) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              if (q * 8 < ncols) {
                *reinterpret_cast<uint4*>(row + (n + q * 8) * 2) = make_uint4(w[q * 4], w[q * 4 + 1], w[q * 4 + 2], w[q * 4 + 3]);
              }
            }
          } else {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              if (q * 4 < ncols) {
                float4 o = make_float4(v[q * 4], v[q * 4 + 1], v[q * 4 + 2], v[q * 4 + 3]);
                *reinterpret_cast<float4*>(row + (n + q * 4) * 4) = o;
              }
            }
          }
        }
      };
      // 32 values of a 16-bit [.., ld] side input (zeros for rows past the end)
      auto load_seg16 = [&](const uint8_t* row, int n, int ncols, float* f) {
        uint4 p[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
          p[q] = (row_ok && q * 8 < ncols) ? ptx::ld_nc_v4(row + (n + q * 8) * 2) : make_uint4(0u, 0u, 0u, 0u);
        unpack32(p, f, out_bf16);
      };
      const uint8_t* aux2_row = nullptr;
      if (args.aux2 != nullptr)
        aux2_row = reinterpret_cast<const uint8_t*>(args.aux2) +
                   (static_cast<long long>(tc.g) * args.aux_group_stride + static_cast<long long>(m) * args.ld_aux) * 2;
      const int nch = min(tile_n / 32, (args.N - tc.n_blk * tile_n + 31) / 32);   // 32-column segments of this tile
      int nx_n = 0, nx_m = 0, nx_g = 0;
      const bool nx_ok = side && side_coords(t + tile_step, nx_n, nx_m, nx_g);
      // segment c of this tile: side inputs -> f0 (aux) and f1 (aux2, may be null)
      auto side_fetch = [&](int c, int n, int ncols, float* f0, float* f1) {
        if (!side) {
          load_seg16(aux_row, n, ncols, f0);
          if (f1 != nullptr) load_seg16(aux2_row, n, ncols, f1);
          return;
        }
        __syncwarp();   // every lane has finished reading the stage that is refilled next
        if (lane == 0) {
          if (c + 1 < nch) side_issue(side_stage ^ 1, n + 32, m_warp0, tc.g);
          else if (nx_ok) side_issue(side_stage ^ 1, nx_n, nx_m, nx_g);
        }
        ptx::mbar_wait(side_bar(ew, side_stage), (side_phase >> side_stage) & 1u);
        const uint32_t sw = (static_cast<uint32_t>(lane) >> 1) & 3u;
#pragma unroll
        for (int a = 0; a < 2; ++a) {
          float* f = a == 0 ? f0 : f1;
          if (f == nullptr) continue;
          const uint32_t my = side_base + static_cast<uint32_t>(side_stage * 2 + a) * C::EPI_TMA_SLOT_BYTES +
                              static_cast<uint32_t>(lane) * 64u;
          uint4 p[4];
#pragma unroll
          for (int q = 0; q < 4; ++q)
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(p[q].x), "=r"(p[q].y), "=r"(p[q].z), "=r"(p[q].w)
                         : "r"(my + ((static_cast<uint32_t>(q) ^ sw) << 4))
                         : "memory");
          unpack32(p, f, out_bf16);
        }
        side_phase ^= 1u << side_stage;
        side_stage ^= 1;
      };

      if (!XACT && glu) {
        // ---------------- gated-linear-unit epilogues ----------------
        const bool fwd = args.epilogue == EPI_GLU;
        const long long row_off = (static_cast<long long>(tc.g) * args.d_group_stride + static_cast<long long>(m) * args.ldd) * 2;
        uint8_t* d2_row = args.d2 != nullptr ? reinterpret_cast<uint8_t*>(args.d2) + row_off : nullptr;
        uint8_t* d3_row = args.d3 != nullptr ? reinterpret_cast<uint8_t*>(args.d3) + row_off : nullptr;
        const float sa = (args.scale_a != nullptr && row_ok)
                             ? args.scale_a[static_cast<long long>(tc.g) * args.scale_a_group_stride + m] : 1.0f;
#pragma unroll 1
        for (int c = 0; c < nch; ++c) {
          const int n = tc.n_blk * tile_n + c * 32;
          const int ncols = min(32, args.N - n);
          uint32_t r[32];
          float g[32], u[32], o[32];
          ptx::tmem_ld_32x32(t_row + static_cast<uint32_t>(c * 32), r);
          ptx::tmem_ld_wait();
          if (fwd) {
#pragma unroll
            for (int j = 0; j < 32; ++j) g[j] = __uint_as_float(r[j]);
            ptx::tmem_ld_32x32(t_row + static_cast<uint32_t>(BN / 2 + c * 32), r);
            ptx::tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) u[j] = __uint_as_float(r[j]);
            if (args.scale_a != nullptr || args.scale_b != nullptr) {
              const float* sb = args.scale_b != nullptr ? args.scale_b + static_cast<long long>(gb) * args.scale_b_group_stride + n : nullptr;
              const float* sb2 = args.scale_b2 != nullptr ? args.scale_b2 + static_cast<long long>(gb) * args.scale_b_group_stride + n : nullptr;
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                g[j] *= (sb != nullptr && j < ncols) ? sa * sb[j] : sa;
                u[j] *= (sb2 != nullptr && j < ncols) ? sa * sb2[j] : sa;
              }
            }
            if (d2_row != nullptr) {       // training: keep the pre-activations for the backward pass
              store_seg(&tmD2, d2_row, n, ncols, g);
              store_seg(&tmD3, d3_row, n, ncols, u);
            }
            if (args.act == ACT_RELU) glu_fwd_seg<ACT_RELU>(g, u, o);
            else if (args.act == ACT_GELU) glu_fwd_seg<ACT_GELU>(g, u, o);
            else glu_fwd_seg<ACT_SILU>(g, u, o);
            store_seg(&tmD, d_row, n, ncols, o);
          } else {
            if (args.scale_a != nullptr || args.scale_b != nullptr) {     // fp8 operands: dh = acc * sa[m] * sb[n]
              const float* sb = args.scale_b != nullptr ? args.scale_b + static_cast<long long>(gb) * args.scale_b_group_stride + n : nullptr;
#pragma unroll
              for (int j = 0; j < 32; ++j)
                r[j] = __float_as_uint(__uint_as_float(r[j]) * ((sb != nullptr && j < ncols) ? sa * sb[j] : sa));
            }
            side_fetch(c, n, ncols, g, u);
            if (args.act == ACT_RELU) glu_bwd_seg<ACT_RELU>(r, g, u, o);
            else if (args.act == ACT_GELU) glu_bwd_seg<ACT_GELU>(r, g, u, o);
            else glu_bwd_seg<ACT_SILU>(r, g, u, o);
            store_seg(&tmD, d_row, n, ncols, o);
            store_seg(&tmD2, d2_row, n, ncols, u);
          }
        }
      } else {
#pragma unroll 1
      for (int c = 0; c < nch; ++c) {
        const int n = tc.n_blk * BN + c * 32;
        uint32_t r[32];
        ptx::tmem_ld_32x32(t_row + static_cast<uint32_t>(c * 32), r);
        ptx::tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
        const int ncols = min(32, args.N - n);  // multiple of 8
        if (args.scale_a != nullptr || args.scale_b != nullptr) {
          // fp8 operands were quantised with one scale per A row and per B column: D = acc * sa[m] * sb[n]
          const float sa = (args.scale_a != nullptr && row_ok)
                               ? args.scale_a[static_cast<long long>(tc.g) * args.scale_a_group_stride + m] : 1.0f;
          const float* sb = args.scale_b != nullptr ? args.scale_b + static_cast<long long>(gb) * args.scale_b_group_stride + n : nullptr;
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] *= (sb != nullptr && j < ncols) ? sa * sb[j] : sa;
        }

        if (args.epilogue == EPI_NONE) {
          if (args.alpha != 1.0f) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] *= args.alpha;
          }
        } else if (args.epilogue == EPI_RELU_BWD || args.epilogue == EPI_ADD || args.epilogue == EPI_ACT_BWD) {
          float f[32];
          side_fetch(c, n, ncols, f, nullptr);
          if (args.epilogue == EPI_RELU_BWD) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = f[j] > 0.0f ? v[j] : 0.0f;
          } else if (args.epilogue == EPI_ADD) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += f[j];
          } else if (!XACT) {
          } else if (args.act == ACT_GELU) {      // f = pre-activation: d/dx [x * Phi(x)] = Phi(x) + x * phi(x)
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float cdf = 0.5f * (1.0f + erff(f[j] * 0.70710678118654752f));
              v[j] *= cdf + f[j] * 0.3989422804014327f * __expf(-0.5f * f[j] * f[j]);
            }
          } else if (args.act == ACT_SILU) {      // d/dx [x * s(x)] = s(x) * (1 + x * (1 - s(x)))
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const float sg = fast_sigmoid(f[j]);
              v[j] *= sg * (1.0f + f[j] * (1.0f - sg));
            }
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = f[j] > 0.0f ? v[j] : 0.0f;
          }
        } else {
          if (bias_g != nullptr) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              if (q * 8 < ncols) {
                float f[8];
                if (args.bias_is_fp32) {
                  const float4 b0 = *reinterpret_cast<const float4*>(bias_g + (n + q * 8) * 4);
                  const float4 b1 = *reinterpret_cast<const float4*>(bias_g + (n + q * 8 + 4) * 4);
                  f[0] = b0.x; f[1] = b0.y; f[2] = b0.z; f[3] = b0.w;
                  f[4] = b1.x; f[5] = b1.y; f[6] = b1.z; f[7] = b1.w;
                } else {
                  unpack8(*reinterpret_cast<const uint4*>(bias_g + (n + q * 8) * 2), args.bias_is_bf16 != 0, f);
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) v[q * 8 + j] += f[j];
              }
            }
          }
          if (XACT && args.d2 != nullptr && (args.epilogue == EPI_BIAS_GELU || args.epilogue == EPI_BIAS_SILU)) {
            // training: the backward pass needs the pre-activation (ReLU gets by with the sign of its output)
            uint8_t* d2_row = reinterpret_cast<uint8_t*>(args.d2) +
                              (static_cast<long long>(tc.g) * args.d_group_stride + static_cast<long long>(m) * args.ldd) *
                                  (out16 ? 2 : 4);
            store_seg(&tmD2, d2_row, n, ncols, v);
          }
          if (args.epilogue == EPI_BIAS_RELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.0f);
          } else if (XACT && args.epilogue == EPI_BIAS_GELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
          } else if (XACT && args.epilogue == EPI_BIAS_SILU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = silu(v[j]);
          }
        }

        if (args.colsum != nullptr) {
          // Bias gradient fused into the epilogue: transpose-reduce the warp's 32 rows x 32 columns with 31 shuffles
          // (afterwards lane j holds the sum of column j) and add it to the fp32 accumulator in global memory.
          float s[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) s[j] = row_ok ? v[j] : 0.0f;
#pragma unroll
          for (int off = 16; off >= 1; off >>= 1) {
            const bool upper = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < off; ++i) {
              const float send = upper ? s[i] : s[i + off];
              const float recv = __shfl_xor_sync(0xffffffffu, send, off);
              s[i] = (upper ? s[i + off] : s[i]) + recv;
            }
          }
          if (lane < ncols)
            atomicAdd(args.colsum + static_cast<long long>(gb) * args.colsum_group_stride + n + lane, s[0]);
        }
        store_seg(&tmD, d_row, n, ncols, v);
      }
      }
      // Accumulator drained: hand the TMEM buffer back to the MMA warp.
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if constexpr (CG == 1) ptx::mbar_arrive(tempty_bar(acc));
        else ptx::mbar_arrive_cluster(tempty_bar(acc), 0);
      }
      if (args.signal_ptr_table != nullptr) {
        // Combine fusion: all 128 epilogue threads' (possibly remote) stores -> one release.sys counter bump.
        if (staged) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // this thread's bulk stores are complete
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (ew == 0 && lane == 0) {
          ptx::fence_acq_rel_sys();
          ptx::red_add_release_sys(reinterpret_cast<uint32_t*>(args.signal_ptr_table[tc.g]), 1u);
        }
      }
      if (++acc == 2) { acc = 0; acc_ph ^= 1u; }
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // staging smem must outlive the last bulk reads
  }

  // ---- teardown ----
  ptx::tc_fence_before();
  if constexpr (CG == 2) ptx::cluster_sync(); else __syncthreads();
  if (warp == 2) ptx::tmem_dealloc<CG>(tmem_base, C::TMEM_COLS);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

bool make_operand_map(CUtensorMap* map, const void* base, int dtype, bool mn_major, long long rows_mn,
                      long long k, long long ld, long long group_stride, int groups, int box_mn_kmajor,
                      const char** why) {
  EncodeTiledFn enc = get_encode_fn();
  if (enc == nullptr) { *why = "cuTensorMapEncodeTiled unavailable"; return false; }
  const int eb = (dtype == DT_E4M3 || dtype == DT_E5M2) ? 1 : 2;
  CUtensorMapDataType dt = eb == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                   : (dtype == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16);
  if ((reinterpret_cast<uintptr_t>(base) & 15) || ((ld * eb) & 15) || ((group_stride * eb) & 15)) {
    *why = "operand base/stride must be 16-byte aligned";
    return false;
  }
  cuuint64_t dims[3];
  cuuint64_t strides[2];
  cuuint32_t box[3];
  cuuint32_t estr[3] = {1, 1, 1};
  const cuuint32_t row_elems = kSwizzleBytes / eb;
  if (!mn_major) {
    dims[0] = static_cast<cuuint64_t>(k); dims[1] = static_cast<cuuint64_t>(rows_mn);
    box[0] = row_elems; box[1] = static_cast<cuuint32_t>(box_mn_kmajor);
  } else {
    dims[0] = static_cast<cuuint64_t>(rows_mn); dims[1] = static_cast<cuuint64_t>(k);
    box[0] = row_elems; box[1] = row_elems;  // BK k-rows x one 128-byte MN chunk
  }
  dims[2] = static_cast<cuuint64_t>(groups);
  box[2] = 1;
  strides[0] = static_cast<cuuint64_t>(ld) * eb;
  strides[1] = static_cast<cuuint64_t>(groups > 1 ? group_stride : (mn_major ? k : rows_mn) * ld) * eb;
  if (strides[1] == 0) strides[1] = strides[0];
  CUresult r = enc(map, dt, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { *why = "cuTensorMapEncodeTiled failed"; return false; }
  return true;
}

// 16-bit output [G, M, N] viewed in 32-column x 32-row blocks, SWIZZLE_64B (the layout the epilogue warps write).
bool make_output_map(CUtensorMap* map, const void* base, int dtype, long long rows, long long cols, long long ld,
                     long long group_stride, int groups, const char** why) {
  EncodeTiledFn enc = get_encode_fn();
  if (enc == nullptr) { *why = "cuTensorMapEncodeTiled unavailable"; return false; }
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows), static_cast<cuuint64_t>(groups)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(ld) * 2,
                           static_cast<cuuint64_t>(groups > 1 ? group_stride : rows * ld) * 2};
  if (strides[1] == 0) strides[1] = strides[0];
  cuuint32_t box[3] = {32, 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(map, dtype == DT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { *why = "cuTensorMapEncodeTiled (output) failed"; return false; }
  return true;
}

uint32_t make_idesc(int in_dtype, bool a_mn, bool b_mn, int umma_m, int umma_n) {
  uint32_t fmt;
  switch (in_dtype) {
    case DT_BF16: fmt = 1; break;
    case DT_FP16: fmt = 0; break;
    case DT_E4M3: fmt = 0; break;
    default: fmt = 1; break;  // DT_E5M2
  }
  uint32_t d = 0;
  d |= 1u << 4;                       // accumulator format: fp32
  d |= fmt << 7;                      // A format
  d |= fmt << 10;                     // B format
  d |= (a_mn ? 1u : 0u) << 15;        // A major
  d |= (b_mn ? 1u : 0u) << 16;        // B major
  d |= static_cast<uint32_t>(umma_n >> 3) << 17;
  d |= static_cast<uint32_t>(umma_m >> 4) << 24;
  return d;
}

struct OutMaps {
  CUtensorMap d, d2, d3, x, x2;   // outputs and side inputs (32x32 blocks, SWIZZLE_64B)
};

template <int CG, bool A_MN, bool B_MN, int BN, int ELT, bool XACT = false>
cudaError_t launch_inst(const CUtensorMap& ta, const CUtensorMap& tb_, const CUtensorMap& tb2, const OutMaps& om,
                        const GemmArgs& args_in, int grid, cudaStream_t stream) {
  using C = Cfg<CG, BN>;
  auto* kern = gemm_sm100_kernel<CG, A_MN, B_MN, BN, ELT, XACT>;
  static bool configured = false;
  if (!configured) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemLimit);
    if (e != cudaSuccess) return e;
    configured = true;
  }
  GemmArgs args = args_in;
  args.epi_warp_bytes = args.tma_side ? C::EPI_WARP_BYTES_SIDE : C::EPI_WARP_BYTES;
  args.stages = C::stages_for(args.epi_warp_bytes);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = C::smem_bytes(args.stages, args.epi_warp_bytes);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, ta, tb_, tb2, om.d, om.d2, om.d3, om.x, om.x2, args);
}

}  // namespace

cudaError_t gemm_sm100_launch(const GemmProblem& p, cudaStream_t stream, const char** why_out) {
  const char* why_local = nullptr;
  const char** why = why_out ? why_out : &why_local;
  *why = nullptr;
  if (p.M <= 0 || p.N <= 0 || p.K <= 0 || p.G <= 0) return cudaSuccess;
  if (p.in_dtype != DT_BF16 && p.in_dtype != DT_FP16 && p.in_dtype != DT_E4M3 && p.in_dtype != DT_E5M2) {
    *why = "A/B must be bf16, fp16, e4m3 or e5m2";
    return cudaErrorInvalidValue;
  }
  const int eb = (p.in_dtype == DT_E4M3 || p.in_dtype == DT_E5M2) ? 1 : 2;
  if (p.N % 8 != 0) { *why = "N must be a multiple of 8"; return cudaErrorInvalidValue; }
  const int ob = p.out_dtype == DT_FP32 ? 4 : 2;
  if ((reinterpret_cast<uintptr_t>(p.d) & 15) || ((p.ldd * ob) & 15) || ((p.d_group_stride * ob) & 15)) {
    *why = "output base/stride must be 16-byte aligned";
    return cudaErrorInvalidValue;
  }

  int dev = 0;
  cudaGetDevice(&dev);
  static int sm_count_cache[64] = {0};
  if (sm_count_cache[dev & 63] == 0) cudaDeviceGetAttribute(&sm_count_cache[dev & 63], cudaDevAttrMultiProcessorCount, dev);
  int sms = sm_count_cache[dev & 63];
  if (p.max_ctas > 0) sms = p.max_ctas < sms ? p.max_ctas : sms;

  const bool dual = p.epilogue == EPI_GLU;
  if (dual && (p.b2 == nullptr || p.out_dtype == DT_FP32)) { *why = "EPI_GLU needs b2 and a 16-bit output"; return cudaErrorInvalidValue; }
  if (p.epilogue == EPI_GLU_BWD && (p.aux == nullptr || p.aux2 == nullptr || p.d2 == nullptr || p.out_dtype == DT_FP32)) {
    *why = "EPI_GLU_BWD needs aux, aux2, d2 and a 16-bit output";
    return cudaErrorInvalidValue;
  }
  if ((p.epilogue == EPI_GLU || p.epilogue == EPI_GLU_BWD) && p.d_ptr_table != nullptr) { *why = "GLU epilogues write local outputs only"; return cudaErrorInvalidValue; }
  int cg = p.cta_group;
  int bn = p.block_n;
  if (bn == 0) bn = (p.N <= 128 && !dual) ? 128 : 256;
  if (dual) bn = 256;
  if (cg == 0) cg = (p.M > 128) ? 2 : 1;
  if (cg == 2 && (sms & 1)) sms -= 1;
  if (sms < cg) sms = cg;   // max_ctas = 1 with CTA pairs still runs one pair

  const int bm = 128 * cg;
  // rotate_group() maps g into [0, G) only when |group_mod| divides G and 0 <= group_rot < |group_mod|.
  const int rot_mod = p.group_mod < 0 ? -p.group_mod : p.group_mod;
  if (p.group_rot < 0 || (rot_mod > 1 && (p.G % rot_mod != 0 || p.group_rot >= rot_mod))) {
    *why = "group_mod must divide G and group_rot must lie in [0, |group_mod|)";
    return cudaErrorInvalidValue;
  }
  // The producer remembers the arrival flags of the current group in a 64-bit mask.
  if (p.wait_flags != nullptr) {
    const int rows_per_flag = p.wait_rows_per_flag > 0 ? p.wait_rows_per_flag : bm;
    const int flags = (p.M + rows_per_flag - 1) / rows_per_flag;
    if (flags > 64 || flags > p.wait_flags_per_group) {
      *why = "wait_flags: ceil(M / wait_rows_per_flag) must be at most 64 and at most wait_flags_per_group";
      return cudaErrorInvalidValue;
    }
  }
  GemmArgs a{};
  a.M = p.M; a.N = p.N; a.K = p.K; a.G = p.G;
  a.b_group_div = p.b_group_div > 0 ? p.b_group_div : 1;
  a.tiles_m = (p.M + bm - 1) / bm;
  a.tiles_n = dual ? (p.N + bn / 2 - 1) / (bn / 2) : (p.N + bn - 1) / bn;
  a.num_tiles = static_cast<long long>(a.tiles_m) * a.tiles_n * p.G;
  a.idesc = make_idesc(p.in_dtype, p.a_mn_major, p.b_mn_major, bm, bn);
  a.elt_bytes = eb;
  a.d = p.d; a.ldd = p.ldd; a.d_group_stride = p.d_group_stride; a.d_ptr_table = p.d_ptr_table;
  a.out_dtype = p.out_dtype;
  a.epilogue = p.epilogue; a.alpha = p.alpha;
  a.bias = p.bias; a.bias_group_stride = p.bias_group_stride; a.bias_is_fp32 = 0;
  a.bias_is_bf16 = (eb == 2) ? (p.in_dtype == DT_BF16) : (p.out_dtype == DT_BF16);
  a.aux = p.aux; a.ld_aux = p.ld_aux; a.aux_group_stride = p.aux_group_stride;
  a.aux2 = p.aux2; a.d2 = p.d2; a.d3 = p.d3; a.dual = dual ? 1 : 0; a.act = p.act; a.scale_b2 = p.scale_b2;
  a.row_counts = p.row_counts;
  a.colsum = p.colsum; a.colsum_group_stride = p.colsum_group_stride;
  a.scale_a = p.scale_a; a.scale_a_group_stride = p.scale_a_group_stride;
  a.scale_b = p.scale_b; a.scale_b_group_stride = p.scale_b_group_stride;
  a.wait_flags = p.wait_flags; a.wait_rows_per_flag = p.wait_rows_per_flag > 0 ? p.wait_rows_per_flag : bm;
  a.wait_flags_per_group = p.wait_flags_per_group; a.wait_target = p.wait_target;
  a.signal_ptr_table = p.signal_ptr_table;
  {
    static int staged_default = -1;
    if (staged_default < 0) {
      const char* e = getenv("TUTEL_B200_EPI");
      staged_default = (e != nullptr && (e[0] == 'd' || e[0] == '0')) ? 0 : 1;   // "direct" / "0" disables staging
    }
    a.staged_store = staged_default;
  }
  a.group_rot = p.group_rot; a.group_mod = p.group_mod;

  CUtensorMap ta, tb_;
  const int gB = (p.G + a.b_group_div - 1) / a.b_group_div;
  if (!make_operand_map(&ta, p.a, p.in_dtype, p.a_mn_major, p.M, p.K, p.lda, p.a_group_stride, p.G, 128, why))
    return cudaErrorInvalidValue;
  const int b_box = dual ? bn / 2 : bn / cg;
  if (!make_operand_map(&tb_, p.b, p.in_dtype, p.b_mn_major, p.N, p.K, p.ldb, p.b_group_stride, gB, b_box, why))
    return cudaErrorInvalidValue;
  CUtensorMap tb2 = tb_;
  if (dual && !make_operand_map(&tb2, p.b2, p.in_dtype, p.b_mn_major, p.N, p.K, p.ldb, p.b_group_stride, gB, b_box, why))
    return cudaErrorInvalidValue;

  // Local 16-bit outputs leave through tensor stores (one per 32x32 block).
  OutMaps om;
  om.d = ta; om.d2 = ta; om.d3 = ta; om.x = ta; om.x2 = ta;   // placeholders (dereferenced only when the flags are set)
  a.tma_store = 0;
  a.tma_side = 0;
  if (a.staged_store && p.out_dtype != DT_FP32 && p.d_ptr_table == nullptr && p.row_counts == nullptr && p.d != nullptr) {
    if (!make_output_map(&om.d, p.d, p.out_dtype, p.M, p.N, p.ldd, p.d_group_stride, p.G, why)) return cudaErrorInvalidValue;
    if (p.d2 != nullptr && !make_output_map(&om.d2, p.d2, p.out_dtype, p.M, p.N, p.ldd, p.d_group_stride, p.G, why))
      return cudaErrorInvalidValue;
    if (p.d3 != nullptr && !make_output_map(&om.d3, p.d3, p.out_dtype, p.M, p.N, p.ldd, p.d_group_stride, p.G, why))
      return cudaErrorInvalidValue;
    a.tma_store = 1;
    const bool uses_side = p.epilogue == EPI_RELU_BWD || p.epilogue == EPI_ADD || p.epilogue == EPI_GLU_BWD || p.epilogue == EPI_ACT_BWD;
    if (uses_side && p.aux != nullptr && ((reinterpret_cast<uintptr_t>(p.aux) | reinterpret_cast<uintptr_t>(p.aux2)) & 15) == 0 &&
        ((p.ld_aux * 2) & 15) == 0 && ((p.aux_group_stride * 2) & 15) == 0) {
      if (!make_output_map(&om.x, p.aux, p.out_dtype, p.M, p.N, p.ld_aux, p.aux_group_stride, p.G, why)) return cudaErrorInvalidValue;
      if (p.aux2 != nullptr && !make_output_map(&om.x2, p.aux2, p.out_dtype, p.M, p.N, p.ld_aux, p.aux_group_stride, p.G, why))
        return cudaErrorInvalidValue;
      a.tma_side = 1;
    }
  }

  long long want = a.num_tiles * cg;
  int grid = static_cast<int>(want < sms ? want : sms);
  if (cg == 2 && (grid & 1)) grid += 1;

  const bool xact = p.epilogue == EPI_BIAS_GELU || p.epilogue == EPI_BIAS_SILU || p.epilogue == EPI_ACT_BWD;
  if (xact && eb != 2) { *why = "GELU / SiLU epilogues need 16-bit operands"; return cudaErrorInvalidValue; }
#define TB_LAUNCH(CGv, AMN, BMN, BNv)                                                                   \
  do {                                                                                                  \
    if (xact) return launch_inst<CGv, AMN, BMN, BNv, 2, true>(ta, tb_, tb2, om, a, grid, stream);        \
    return launch_inst<CGv, AMN, BMN, BNv, 2, false>(ta, tb_, tb2, om, a, grid, stream);                 \
  } while (0)
#define TB_SWITCH_MAJOR(CGv, BNv)                                    \
  do {                                                               \
    if (!p.a_mn_major && !p.b_mn_major) TB_LAUNCH(CGv, false, false, BNv); \
    if (!p.a_mn_major && p.b_mn_major) TB_LAUNCH(CGv, false, true, BNv);   \
    if (p.a_mn_major && !p.b_mn_major) TB_LAUNCH(CGv, true, false, BNv);   \
    TB_LAUNCH(CGv, true, true, BNv);                                       \
  } while (0)
  if (eb == 1) {
    if (p.a_mn_major || p.b_mn_major) { *why = "fp8 operands must be K-major"; return cudaErrorInvalidValue; }
    if (cg == 1 && bn == 256) return launch_inst<1, false, false, 256, 1>(ta, tb_, tb2, om, a, grid, stream);
    if (cg == 1 && bn == 128) return launch_inst<1, false, false, 128, 1>(ta, tb_, tb2, om, a, grid, stream);
    if (cg == 2 && bn == 256) return launch_inst<2, false, false, 256, 1>(ta, tb_, tb2, om, a, grid, stream);
    if (cg == 2 && bn == 128) return launch_inst<2, false, false, 128, 1>(ta, tb_, tb2, om, a, grid, stream);
  }
  if (cg == 1 && bn == 256) TB_SWITCH_MAJOR(1, 256);
  if (cg == 1 && bn == 128) TB_SWITCH_MAJOR(1, 128);
  if (cg == 2 && bn == 256) TB_SWITCH_MAJOR(2, 256);
  if (cg == 2 && bn == 128) TB_SWITCH_MAJOR(2, 128);
#undef TB_SWITCH_MAJOR
#undef TB_LAUNCH
  *why = "unsupported cta_group/block_n";
  return cudaErrorInvalidValue;
}

// run-time spin-wait limit of this translation unit's kernels (ptx.cuh)
cudaError_t set_spin_timeout_gemm(unsigned long long ns) {
  return cudaMemcpyToSymbol(tb_spin_timeout_ns, &ns, sizeof(ns));
}

}  // namespace tb
