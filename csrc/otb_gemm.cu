// otter_b200 — tcgen05 / TMA GEMM with fused epilogues (the >99.9 %-of-FLOPs kernel of the hot path).
//
//   D[M,N] = epilogue( A[M,K] . B[N,K]^T ),  bf16 operands, fp32 accumulation in TMEM.
//
// Serves every nn.Linear on the path and its autograd dgrad / wgrad:
//   forward  y  = x W^T      : A = x  [M][K]  K-major,  B = W  [N][K]  K-major
//   dgrad    dx = dy W       : A = dy [M][N'] K-major,  B = W  [N'][K'] read as MN-major (no transpose copy)
//   wgrad    dW = dy^T x     : A = dy read MN-major,    B = x  read MN-major (reduction over tokens)
// (reference: modeling_otter.py:139-148,164-184,253-256,284-288,340,363-370; clip.py:106-149)
//
// Structure (one CTA per SM, persistent over output tiles, 384 threads):
//   warp 10  : TMA producer   — cp.async.bulk.tensor 128B-swizzled tiles into a kStages-deep smem ring
//   warp 11  : MMA issuer     — one thread issues tcgen05.mma (128 x BN x 16), tcgen05.commit frees smem slots
//                               (highest warp ids: the issue arbiter favours them over the math-heavy epilogue)
//   warp 8   : TMEM allocator — 2 x BN fp32 columns (double-buffered accumulator)
//   warps 0-7: epilogue       — tcgen05.ld 32 lanes x 32 columns (two warps per TMEM lane quarter, each half of
//                               the tile's columns), global operands prefetched per chunk, fused
//                               bias/GELU/gate/residual, 16 B stores
// The accumulator double buffer lets the epilogue of tile i overlap the main loop of tile i+1.
#include <cstdlib>

#include "otb_common.cuh"
#include "otb_host.h"

namespace otb {

constexpr int kBM = 128;
constexpr int kBK = 64;
constexpr int kGemmThreads = 384;   // 8 epilogue warps + 4 control warps
constexpr int kEpiWarpStage = 32 * 128;             // one epilogue warp's store stage: 32 rows x 128 B (64 bf16 columns)
constexpr int kEpiStageBytes = 8 * kEpiWarpStage;    // 32 KB, sits between the operand ring and the barriers

struct GemmEpi {
  const float* bias;
  const bf16* aux_in;
  bf16* aux_out;
  const float* scale_ptr;
  const bf16* residual;
  void* out;
  long long ld_out, ld_aux_in, ld_aux_out, ld_res;
  int act, scale_tanh, out_fp32, accumulate;
  float alpha;
  int res_fp32;   // residual is fp32 [M][N] (fp32-grade parity path)
  int tma_out;    // bf16 output leaves through a swizzled smem stage + TMA store (full 128 B lines, bounds clipped by TMA)
  int cls;        // index into kEpiCls when the options match one of the compiled classes, else -1 (run-time options)
};

template <int BN>
struct GemmCfg {
  static constexpr int kABytes = kBM * kBK * 2;            // 16 KB
  static constexpr int kBBytes = BN * kBK * 2;             // 32 KB (BN=256) / 16 KB (BN=128)
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (BN == 256) ? 4 : 6;
  static constexpr int kTmemCols = 2 * BN;                 // double-buffered accumulator
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;
};

// One epilogue warp's share of one 128 x BN accumulator tile: TMEM lane quarter q (32 rows), column half `half`.
template <int BN>
__device__ __forceinline__ void epilogue_tile(const GemmEpi& ep, float scale, uint32_t taddr, int m0, int n0, int M,
                                              int N, int q, int half, int lane) {
  const int row = m0 + q * 32 + lane;
  const bool row_ok = row < M;
  const long long lrow = row;
#pragma unroll 1
  for (int c = half * (BN / 64); c < (half + 1) * (BN / 64); ++c) {
    const int colbase = n0 + c * 32;
    const bool act_chunk = row_ok && colbase < N;
    // Issue every global read of this 32-column chunk up front (they do not depend on the accumulator):
    // each thread reads 64 B of its own row, so the loads of a warp are uncoalesced — what matters is
    // having all of them in flight together instead of one dependent load per 8 columns.
    uint4 res[4], aux[4];
    float4 old[8];
    if (act_chunk) {
      if (ep.residual != nullptr && !ep.res_fp32) {
        const uint4* pr = reinterpret_cast<const uint4*>(ep.residual + lrow * ep.ld_res + colbase);
#pragma unroll
        for (int g = 0; g < 4; ++g) if (colbase + g * 8 < N) res[g] = __ldg(pr + g);
      }
      if (ep.aux_in != nullptr) {
        const uint4* pa = reinterpret_cast<const uint4*>(ep.aux_in + lrow * ep.ld_aux_in + colbase);
#pragma unroll
        for (int g = 0; g < 4; ++g) if (colbase + g * 8 < N) aux[g] = __ldg(pa + g);
      }
      if (ep.out_fp32 && ep.accumulate) {
        const float4* po = reinterpret_cast<const float4*>(reinterpret_cast<float*>(ep.out) + lrow * ep.ld_out + colbase);
#pragma unroll
        for (int g = 0; g < 8; ++g) if (colbase + g * 4 < N) old[g] = po[g];
      }
    }
    uint32_t r[32];
    tmem_ld32(taddr + c * 32, r);
    tmem_ld_wait();
    if (act_chunk) {
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        const int col = colbase + g * 8;
        if (col >= N) break;
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[g * 8 + i]);
        if (ep.bias != nullptr) {
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(ep.bias + col));
          const float4 b1 = __ldg(reinterpret_cast<const float4*>(ep.bias + col + 4));
          v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
          v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
        }
        if (ep.aux_out != nullptr) {
          uint4 o;
          o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
          o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
          *reinterpret_cast<uint4*>(ep.aux_out + lrow * ep.ld_aux_out + col) = o;
        }
        if (ep.aux_in == nullptr) {
          if (ep.act == 1) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = gelu_fast(v[i]);
          } else if (ep.act == 2) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = quick_gelu(v[i]);
          } else if (ep.act == 3) {                     // relu^2 (Persimmon "relu2")
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float r_ = fmaxf(v[i], 0.f); v[i] = r_ * r_; }
          }
        } else {   // backward of the activation whose pre-activation is aux_in: act 3 -> 2 relu(z), otherwise gelu'(z)
          const float2 a0 = unpack_bf16x2(aux[g].x), a1 = unpack_bf16x2(aux[g].y), a2 = unpack_bf16x2(aux[g].z),
                       a3 = unpack_bf16x2(aux[g].w);
          if (ep.act == 3) {
            v[0] *= 2.f * fmaxf(a0.x, 0.f); v[1] *= 2.f * fmaxf(a0.y, 0.f);
            v[2] *= 2.f * fmaxf(a1.x, 0.f); v[3] *= 2.f * fmaxf(a1.y, 0.f);
            v[4] *= 2.f * fmaxf(a2.x, 0.f); v[5] *= 2.f * fmaxf(a2.y, 0.f);
            v[6] *= 2.f * fmaxf(a3.x, 0.f); v[7] *= 2.f * fmaxf(a3.y, 0.f);
          } else {
            v[0] *= gelu_grad_fast(a0.x); v[1] *= gelu_grad_fast(a0.y);
            v[2] *= gelu_grad_fast(a1.x); v[3] *= gelu_grad_fast(a1.y);
            v[4] *= gelu_grad_fast(a2.x); v[5] *= gelu_grad_fast(a2.y);
            v[6] *= gelu_grad_fast(a3.x); v[7] *= gelu_grad_fast(a3.y);
          }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] *= scale;
        if (ep.residual != nullptr && ep.res_fp32) {
          const float* pr = reinterpret_cast<const float*>(ep.residual) + lrow * ep.ld_res + col;
          const float4 r0 = __ldg(reinterpret_cast<const float4*>(pr)), r1 = __ldg(reinterpret_cast<const float4*>(pr + 4));
          v[0] += r0.x; v[1] += r0.y; v[2] += r0.z; v[3] += r0.w;
          v[4] += r1.x; v[5] += r1.y; v[6] += r1.z; v[7] += r1.w;
        } else if (ep.residual != nullptr) {
          const float2 a0 = unpack_bf16x2(res[g].x), a1 = unpack_bf16x2(res[g].y), a2 = unpack_bf16x2(res[g].z),
                       a3 = unpack_bf16x2(res[g].w);
          v[0] += a0.x; v[1] += a0.y; v[2] += a1.x; v[3] += a1.y;
          v[4] += a2.x; v[5] += a2.y; v[6] += a3.x; v[7] += a3.y;
        }
        if (ep.out_fp32) {
          float* o = reinterpret_cast<float*>(ep.out) + lrow * ep.ld_out + col;
          float4 o0 = make_float4(0.f, 0.f, 0.f, 0.f), o1 = o0;
          if (ep.accumulate) { o0 = old[2 * g]; o1 = old[2 * g + 1]; }
          o0.x += v[0]; o0.y += v[1]; o0.z += v[2]; o0.w += v[3];
          o1.x += v[4]; o1.y += v[5]; o1.z += v[6]; o1.w += v[7];
          *reinterpret_cast<float4*>(o) = o0;
          *reinterpret_cast<float4*>(o + 4) = o1;
        } else {
          uint4 o;
          o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
          o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
          *reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(ep.out) + lrow * ep.ld_out + col) = o;
        }
      }
    }
  }
}

// TMA-store variant of the epilogue.  The direct epilogue above has every thread write 16 B pieces of its own row:
// 32 different 128 B lines per warp store instruction, partially written sectors on the way to L2, and the
// accumulate class first READS its old fp32 values the same way.  Here a warp assembles 32 rows x 128 B (64 bf16 or
// 32 fp32 columns) in a SWIZZLE_128B smem stage — thread = row, the 16 B unit j of row r lands at unit j ^ (r & 7),
// which is bank-conflict free and exactly the layout the output tensor map expects — and one lane hands the 4 KB box
// to the TMA engine, which writes whole lines, clips rows >= M / columns >= N, and for `accumulate` performs the
// fp32 add at L2 (cp.reduce.async.bulk ... add) so the old values never travel to the SM.
// The stage is reused once the previous bulk operation has finished READING it (wait_group.read), which overlaps
// with the TMEM load and the math of the next chunk.  The pre-activation side output (aux_out) keeps direct stores.
// CLS >= 0: the epilogue options of launch class kEpiCls[CLS] are compile-time constants — the per-group option tests
// (uniform branches that cut the 32 independent element streams of a chunk into tiny basic blocks) disappear and the
// chunk becomes one block the scheduler can interleave.  ncu r02 (profiles/r02_ncu_gemm_epilogue.md): the generic code
// executes 42 instructions per output for GELU + aux at 0.36 IPC per scheduler with 2 epilogue warps each; 29 % of the
// stall samples sit on those branches.  CLS = -1: options read from `ep` at run time (any combination).
struct EpiCls { bool bias, aux_out; int act; bool aux_in, scale, res, out_f32, acc; };
constexpr int kNumEpiCls = 14;
constexpr EpiCls kEpiCls[kNumEpiCls] = {
    /* 0 plain                      */ {false, false, 0, false, false, false, false, false},
    /* 1 * gate                     */ {false, false, 0, false, true, false, false, false},
    /* 2 bias                       */ {true, false, 0, false, false, false, false, false},
    /* 3 bias + quick-GELU          */ {true, false, 2, false, false, false, false, false},
    /* 4 bias + residual            */ {true, false, 0, false, false, true, false, false},
    /* 5 residual                   */ {false, false, 0, false, false, true, false, false},
    /* 6 GELU + pre-activation      */ {false, true, 1, false, false, false, false, false},
    /* 7 branch out, * gate, + res  */ {false, true, 0, false, true, true, false, false},
    /* 8 * gelu'(aux) * gate        */ {false, false, 0, true, true, false, false, false},
    /* 9 * gelu'(aux)               */ {false, false, 0, true, false, false, false, false},
    /* 10 fp32 store                */ {false, false, 0, false, false, false, true, false},
    /* 11 fp32 store * gate         */ {false, false, 0, false, true, false, true, false},
    /* 12 fp32 accumulate           */ {false, false, 0, false, false, false, true, true},
    /* 13 fp32 accumulate * gate    */ {false, false, 0, false, true, false, true, true},
};

template <int BN, int CLS>
__device__ __forceinline__ void epilogue_tile_tma(const GemmEpi& ep, float scale, uint32_t taddr, int m0, int n0, int M,
                                                  int N, int q, int half, int lane, uint8_t* stage,
                                                  const CUtensorMap* map_d) {
  constexpr bool kS = CLS >= 0;
  constexpr EpiCls kC = kEpiCls[kS ? CLS : 0];
  const bool f_bias = kS ? kC.bias : (ep.bias != nullptr);
  const bool f_auxo = kS ? kC.aux_out : (ep.aux_out != nullptr);
  const int f_act = kS ? kC.act : ep.act;
  const bool f_auxi = kS ? kC.aux_in : (ep.aux_in != nullptr);
  const bool f_scale = kS ? kC.scale : true;
  const bool f_res = kS ? kC.res : (ep.residual != nullptr);
  const bool f_f32 = kS ? kC.out_f32 : (ep.out_fp32 != 0);
  const bool f_acc = kS ? kC.acc : (ep.accumulate != 0);
  const int row0 = m0 + q * 32;
  if (row0 >= M) return;                                      // warp-uniform: no row of this quarter is inside
  const int row = row0 + lane;
  const bool row_ok = row < M;
  const long long lrow = row;
  uint8_t* my_row = stage + lane * 128;
  const int xr = lane & 7;
#pragma unroll 1
  for (int c = half * (BN / 64); c < (half + 1) * (BN / 64); ++c) {     // 32-column chunks of this warp's half
    const int colbase = n0 + c * 32;
    if (colbase >= N) break;                                  // warp-uniform
    const bool act_chunk = row_ok;
    uint4 res[4], aux[4];
    if (act_chunk) {
      if (f_res) {
        const uint4* pr = reinterpret_cast<const uint4*>(ep.residual + lrow * ep.ld_res + colbase);
#pragma unroll
        for (int g = 0; g < 4; ++g) if (colbase + g * 8 < N) res[g] = __ldg(pr + g);
      }
      if (f_auxi) {
        const uint4* pa = reinterpret_cast<const uint4*>(ep.aux_in + lrow * ep.ld_aux_in + colbase);
#pragma unroll
        for (int g = 0; g < 4; ++g) if (colbase + g * 8 < N) aux[g] = __ldg(pa + g);
      }
    }
    uint32_t r[32];
    tmem_ld32(taddr + c * 32, r);
    tmem_ld_wait();
    // bf16: two chunks share one 128 B-wide box (units 0-3 / 4-7); fp32: one chunk is one box (units 0-7).
    const bool first_of_box = f_f32 || (c & 1) == 0;
    const bool last_of_box = f_f32 || (c & 1) == 1 || colbase + 32 >= N;
    if (first_of_box) {                                       // the previous box must have left the stage
      if (lane == 0) tma_store_wait_read<0>();
      __syncwarp();
    }
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const int col = colbase + g * 8;
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[g * 8 + i]);
      if (act_chunk && col < N) {
        if (f_bias) {
          const float4 b0 = __ldg(reinterpret_cast<const float4*>(ep.bias + col));
          const float4 b1 = __ldg(reinterpret_cast<const float4*>(ep.bias + col + 4));
          v[0] += b0.x; v[1] += b0.y; v[2] += b0.z; v[3] += b0.w;
          v[4] += b1.x; v[5] += b1.y; v[6] += b1.z; v[7] += b1.w;
        }
        if (f_auxo) {
          uint4 x;
          x.x = pack_bf16x2(v[0], v[1]); x.y = pack_bf16x2(v[2], v[3]);
          x.z = pack_bf16x2(v[4], v[5]); x.w = pack_bf16x2(v[6], v[7]);
          *reinterpret_cast<uint4*>(ep.aux_out + lrow * ep.ld_aux_out + col) = x;
        }
        if (!f_auxi) {
          if (f_act == 1) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = gelu_fast(v[i]);
          } else if (f_act == 2) {
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] = quick_gelu(v[i]);
          } else if (f_act == 3) {                     // relu^2 (Persimmon "relu2")
#pragma unroll
            for (int i = 0; i < 8; ++i) { const float r_ = fmaxf(v[i], 0.f); v[i] = r_ * r_; }
          }
        } else {   // backward of the activation whose pre-activation is aux_in: act 3 -> 2 relu(z), otherwise gelu'(z)
          const float2 a0 = unpack_bf16x2(aux[g].x), a1 = unpack_bf16x2(aux[g].y), a2 = unpack_bf16x2(aux[g].z),
                       a3 = unpack_bf16x2(aux[g].w);
          if (f_act == 3) {
            v[0] *= 2.f * fmaxf(a0.x, 0.f); v[1] *= 2.f * fmaxf(a0.y, 0.f);
            v[2] *= 2.f * fmaxf(a1.x, 0.f); v[3] *= 2.f * fmaxf(a1.y, 0.f);
            v[4] *= 2.f * fmaxf(a2.x, 0.f); v[5] *= 2.f * fmaxf(a2.y, 0.f);
            v[6] *= 2.f * fmaxf(a3.x, 0.f); v[7] *= 2.f * fmaxf(a3.y, 0.f);
          } else {
            v[0] *= gelu_grad_fast(a0.x); v[1] *= gelu_grad_fast(a0.y);
            v[2] *= gelu_grad_fast(a1.x); v[3] *= gelu_grad_fast(a1.y);
            v[4] *= gelu_grad_fast(a2.x); v[5] *= gelu_grad_fast(a2.y);
            v[6] *= gelu_grad_fast(a3.x); v[7] *= gelu_grad_fast(a3.y);
          }
        }
        if (f_scale) {
#pragma unroll
          for (int i = 0; i < 8; ++i) v[i] *= scale;
        }
        if (f_res) {
          const float2 a0 = unpack_bf16x2(res[g].x), a1 = unpack_bf16x2(res[g].y), a2 = unpack_bf16x2(res[g].z),
                       a3 = unpack_bf16x2(res[g].w);
          v[0] += a0.x; v[1] += a0.y; v[2] += a1.x; v[3] += a1.y;
          v[4] += a2.x; v[5] += a2.y; v[6] += a3.x; v[7] += a3.y;
        }
      }
      // rows >= M and columns >= N hold don't-care values: the TMA engine clips them
      if (f_f32) {
        *reinterpret_cast<float4*>(my_row + (((2 * g) ^ xr) << 4)) = make_float4(v[0], v[1], v[2], v[3]);
        *reinterpret_cast<float4*>(my_row + (((2 * g + 1) ^ xr) << 4)) = make_float4(v[4], v[5], v[6], v[7]);
      } else {
        uint4 o;
        o.x = pack_bf16x2(v[0], v[1]); o.y = pack_bf16x2(v[2], v[3]);
        o.z = pack_bf16x2(v[4], v[5]); o.w = pack_bf16x2(v[6], v[7]);
        *reinterpret_cast<uint4*>(my_row + ((((c & 1) * 4 + g) ^ xr) << 4)) = o;
      }
    }
    if (last_of_box) {
      fence_proxy_async_smem();                               // generic-proxy writes -> visible to the TMA engine
      __syncwarp();
      if (lane == 0) {
        const int box_col = f_f32 ? colbase : (colbase & ~63);
        if (f_acc) tma_reduce_add_2d(map_d, stage, box_col, row0);
        else tma_store_2d(map_d, stage, box_col, row0);
        tma_store_commit();
      }
    }
  }
}

// per-tile dispatch on the launch's epilogue class (host: epi_class_of)
template <int BN>
__device__ __forceinline__ void epilogue_dispatch_tma(const GemmEpi& ep, float scale, uint32_t taddr, int m0, int n0,
                                                      int M, int N, int q, int half, int lane, uint8_t* stage,
                                                      const CUtensorMap* map_d) {
#define OTB_EPI_CASE(C_) case C_: epilogue_tile_tma<BN, C_>(ep, scale, taddr, m0, n0, M, N, q, half, lane, stage, map_d); break;
  switch (ep.cls) {
    OTB_EPI_CASE(0) OTB_EPI_CASE(1) OTB_EPI_CASE(2) OTB_EPI_CASE(3) OTB_EPI_CASE(4) OTB_EPI_CASE(5) OTB_EPI_CASE(6)
    OTB_EPI_CASE(7) OTB_EPI_CASE(8) OTB_EPI_CASE(9) OTB_EPI_CASE(10) OTB_EPI_CASE(11) OTB_EPI_CASE(12) OTB_EPI_CASE(13)
    default: epilogue_tile_tma<BN, -1>(ep, scale, taddr, m0, n0, M, N, q, half, lane, stage, map_d); break;
  }
#undef OTB_EPI_CASE
}

// MC = true: clusters of 2 CTAs work on two vertically adjacent 128-row tiles of the same BN-wide column block;
// each CTA fetches half of the shared B tile and TMA-multicasts it to both, which cuts the L2->SM operand
// traffic per FLOP by a third (the big GEMMs are L2-bandwidth bound at one 128xBN tile per CTA).
template <int BN, bool A_MN, bool B_MN, bool MC, bool TS>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const __grid_constant__ CUtensorMap map_d, int M, int N, int K, GemmEpi ep) {
  using Cfg = GemmCfg<BN>;
  pdl_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* epi_stage = smem + Cfg::kStages * Cfg::kStageBytes;      // 8 x 4 KB (1024-aligned), TMA-store epilogue only
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_stage + (TS ? kEpiStageBytes : 0));
  uint64_t* full_bar = bars;                        // [kStages]
  uint64_t* empty_bar = bars + Cfg::kStages;        // [kStages]
  uint64_t* tfull_bar = bars + 2 * Cfg::kStages;    // [2]
  uint64_t* tempty_bar = tfull_bar + 2;             // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int tiles_m_real = (M + kBM - 1) / kBM;
  const int tiles_m = MC ? ((tiles_m_real + 1) & ~1) : tiles_m_real;   // MC: pad to whole CTA pairs (OOB rows = 0)
  const int tiles_n = (N + BN - 1) / BN;
  const int num_tiles = tiles_m * tiles_n;
  const int num_kb = (K + kBK - 1) / kBK;
  const uint32_t cta_rank = MC ? cluster_ctarank() : 0;
  // persistent schedule: consecutive tile ids run down M, so with MC the pair (2i, 2i+1) shares its column block;
  // blockIdx.x of a cluster is (2c, 2c+1) and gridDim.x is even -> both CTAs walk the same number of tiles.

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], MC ? 2 : 1);   // MC: both CTAs of the pair must have consumed the stage
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 8);  // one arrive per epilogue warp
    }
    fence_mbar_init();
  }
  if (warp == 8) tmem_alloc(tmem_slot, Cfg::kTmemCols);
  tc_fence_before();
  __syncthreads();
  if constexpr (MC) cluster_sync_all();       // peer barriers are initialised before any multicast can land
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();   // predecessor grid complete before any global / TMA access

  if (warp == 10 && lane == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      const int m0 = (t % tiles_m) * kBM;
      const int n0 = (t / tiles_m) * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * Cfg::kStageBytes;
        uint8_t* sb = sa + Cfg::kABytes;
        mbar_arrive_expect_tx(&full_bar[stage], Cfg::kStageBytes);
        const int k0 = kb * kBK;
        if constexpr (!A_MN) {
          tma_load_2d(sa, &map_a, &full_bar[stage], k0, m0);  // box {64 k, 128 rows}
        } else {
#pragma unroll
          for (int c = 0; c < kBM / 64; ++c)                  // box {64 m, 64 k rows} per 64-wide chunk
            tma_load_2d(sa + c * (kBK * 128), &map_a, &full_bar[stage], m0 + c * 64, k0);
        }
        if constexpr (!MC) {
          if constexpr (!B_MN) {
            tma_load_2d(sb, &map_b, &full_bar[stage], k0, n0);  // box {64 k, BN rows}
          } else {
#pragma unroll
            for (int c = 0; c < BN / 64; ++c)
              tma_load_2d(sb + c * (kBK * 128), &map_b, &full_bar[stage], n0 + c * 64, k0);
          }
        } else {  // this CTA's half of the B tile, multicast into both CTAs of the pair
          if constexpr (!B_MN) {
            tma_load_2d_mcast(sb + cta_rank * (BN / 2) * 128, &map_b, &full_bar[stage], k0,
                              n0 + cta_rank * (BN / 2), 0x3);  // box {64 k, BN/2 rows}
          } else {
#pragma unroll
            for (int c = 0; c < BN / 128; ++c) {
              const int cc = cta_rank * (BN / 128) + c;
              tma_load_2d_mcast(sb + cc * (kBK * 128), &map_b, &full_bar[stage], n0 + cc * 64, k0, 0x3);
            }
          }
        }
        if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 11 && lane == 0) {
    // ===================== MMA issuer (single thread) =====================
    constexpr uint32_t idesc = make_idesc_bf16(kBM, BN, A_MN, B_MN);
    constexpr uint32_t a_lbo = A_MN ? kBK * 128 : 16, a_sbo = 1024, a_kstep = A_MN ? 2048 : 32;
    constexpr uint32_t b_lbo = B_MN ? kBK * 128 : 16, b_sbo = 1024, b_kstep = B_MN ? 2048 : 32;
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);  // epilogue has drained this accumulator
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + stage * Cfg::kStageBytes);
        const uint32_t sb = sa + Cfg::kABytes;
        const uint64_t da = make_smem_desc(sa, a_lbo, a_sbo);
        const uint64_t db = make_smem_desc(sb, b_lbo, b_sbo);
#pragma unroll
        for (int k = 0; k < kBK / 16; ++k) {
          umma_bf16(d_tmem, da + ((k * a_kstep) >> 4), db + ((k * b_kstep) >> 4), idesc, (kb | k) != 0);
        }
        if constexpr (MC) umma_commit_mcast(&empty_bar[stage], 0x3);   // release the slot in BOTH CTAs
        else umma_commit(&empty_bar[stage]);  // frees this smem slot once the MMAs above retire
        if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
      }
      umma_commit(&tfull_bar[acc]);      // accumulator complete -> epilogue
    }
  } else if (warp < 8) {
    // ===================== epilogue warps (8): warp w -> TMEM lane quarter w%4, column half w/4 =========
    const int q = warp & 3;
    const int half = warp >> 2;
    float scale = ep.alpha;
    if (ep.scale_ptr != nullptr) {
      const float s = __ldg(ep.scale_ptr);
      scale *= ep.scale_tanh ? tanhf(s) : s;
    }
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int m0 = (t % tiles_m) * kBM;
      const int n0 = (t / tiles_m) * BN;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN;
      if constexpr (TS)
        epilogue_dispatch_tma<BN>(ep, scale, taddr, m0, n0, M, N, q, half, lane, epi_stage + warp * kEpiWarpStage, &map_d);
      else
        epilogue_tile<BN>(ep, scale, taddr, m0, n0, M, N, q, half, lane);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
    }
    if (TS && lane == 0) tma_store_wait_read<0>();   // the stage must outlive the last bulk store's reads
  }

  tc_fence_before();
  __syncthreads();
  if constexpr (MC) cluster_sync_all();       // no CTA leaves while its peer may still signal / write into it
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int BN, bool A_MN, bool B_MN, bool MC, bool TS>
static int launch_gemm(const void* A, long long lda, const void* B, long long ldb, int M, int N, int K,
                       const GemmEpi& ep, cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  CUtensorMap ma, mb;
  int rc;
  if (!A_MN) rc = make_tmap_bf16_2d(&ma, A, M, K, lda, kBM, 64);   // [M][K], box 128 rows x 64 k
  else       rc = make_tmap_bf16_2d(&ma, A, K, M, lda, kBK, 64);   // [K][M], box 64 k-rows x 64 m
  if (rc) return rc;
  if (!B_MN) rc = make_tmap_bf16_2d(&mb, B, N, K, ldb, MC ? BN / 2 : BN, 64);
  else       rc = make_tmap_bf16_2d(&mb, B, K, N, ldb, kBK, 64);
  if (rc) return rc;
  CUtensorMap md = ma;                                               // placeholder when the direct epilogue is used
  if (TS) {                                                          // [M][N] output, box 32 rows x 128 B
    rc = ep.out_fp32 ? make_tmap_f32_2d(&md, ep.out, M, N, ep.ld_out, 32, 32)
                     : make_tmap_bf16_2d(&md, ep.out, M, N, ep.ld_out, 32, 64);
    if (rc) return rc;
  }
  auto kern = gemm_bf16_kernel<BN, A_MN, B_MN, MC, TS>;
  constexpr int smem_bytes = Cfg::kSmemBytes + (TS ? kEpiStageBytes : 0);
  OTB_CHECK_CUDA(ensure_dyn_smem(kern, smem_bytes));   // per (instantiation, device)
  const int tiles_m = (M + kBM - 1) / kBM, tiles_n = (N + BN - 1) / BN;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[2];
  int nattr = 0;
  if (pdl_enabled()) {
    attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[nattr].val.programmaticStreamSerializationAllowed = 1;
    ++nattr;
  }
  if (MC) {
    const int pairs = ((tiles_m + 1) / 2) * tiles_n;
    const int max_pairs = sm_count() / 2;
    cfg.gridDim = dim3(2 * (pairs < max_pairs ? pairs : max_pairs));
    attr[nattr].id = cudaLaunchAttributeClusterDimension;
    attr[nattr].val.clusterDim.x = 2; attr[nattr].val.clusterDim.y = 1; attr[nattr].val.clusterDim.z = 1;
    ++nattr;
  } else {
    const int tiles = tiles_m * tiles_n;
    cfg.gridDim = dim3(tiles < sm_count() ? tiles : sm_count());
  }
  cfg.attrs = attr;
  cfg.numAttrs = nattr;
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  OTB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, ma, mb, md, M, N, K, ep));
  count_launch();
  return OTB_OK;
}


// ================================================================================================
// cta_group::2 variant: a CTA pair (two SMs) computes one 256 x 256 output tile with a single tcgen05.mma stream
// issued by the leader.  Each CTA stages its own 128 rows of A and HALF of the B tile (128 of the 256 columns), so a
// k-block costs 32 KB of smem traffic per SM instead of 48 KB — the 128 x 256 single-CTA kernel saturates the SM's
// shared-memory bandwidth (TMA writes + tensor-core reads = 192 B/clk > 128 B/clk) at ~66 % tensor-pipe activity —
// and the ring deepens to 6 stages.  Barrier protocol: TMA of both CTAs completes on the leader's `full`;
// tcgen05.commit multicasts `empty` / `tmem_full` to both CTAs; both epilogues arrive on the leader's `tmem_empty`.
// ================================================================================================
constexpr int k2Stages = 6;
constexpr int k2StageBytes = 2 * 128 * kBK * 2;   // A 16 KB + B-half 16 KB
constexpr int k2SmemBytes = k2Stages * k2StageBytes + 1024 + 256;

template <bool A_MN, bool B_MN, bool TS>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm2_bf16_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                  const __grid_constant__ CUtensorMap map_d, int M, int N, int K, GemmEpi ep) {
  constexpr int BN = 256;
  pdl_launch_dependents();
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* epi_stage = smem + k2Stages * k2StageBytes;              // 8 x 4 KB (1024-aligned), TMA-store epilogue only
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_stage + (TS ? kEpiStageBytes : 0));
  uint64_t* full_bar = bars;                    // [k2Stages]  (leader's copy is the live one)
  uint64_t* empty_bar = bars + k2Stages;        // [k2Stages]  (both CTAs)
  uint64_t* tfull_bar = bars + 2 * k2Stages;    // [2]         (both CTAs)
  uint64_t* tempty_bar = tfull_bar + 2;         // [2]         (leader's copy is the live one)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int tiles_mp = (M + 255) / 256;          // 256-row pair tiles
  const int tiles_n = (N + BN - 1) / BN;
  const int num_pt = tiles_mp * tiles_n;
  const int num_kb = (K + kBK - 1) / kBK;
  const int cluster_id = blockIdx.x >> 1, num_clusters = gridDim.x >> 1;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    for (int s = 0; s < k2Stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tfull_bar[s], 1); mbar_init(&tempty_bar[s], 16); }   // 8 warps x 2 CTAs
    fence_mbar_init();
  }
  if (warp == 8) tmem_alloc_2cta(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  if (warp == 10 && lane == 0) {
    // ===================== TMA producer (both CTAs) =====================
    int stage = 0;
    uint32_t phase = 0;
    for (int pt = cluster_id; pt < num_pt; pt += num_clusters) {
      const int m0 = (pt % tiles_mp) * 256 + static_cast<int>(rank) * 128;
      const int n0 = (pt / tiles_mp) * BN + static_cast<int>(rank) * 128;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* sa = smem + stage * k2StageBytes;
        uint8_t* sb = sa + 128 * kBK * 2;
        if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * k2StageBytes);   // bytes of BOTH CTAs
        const int k0 = kb * kBK;
        if constexpr (!A_MN) {
          tma_load_2d_2cta(sa, &map_a, &full_bar[stage], k0, m0);
        } else {
#pragma unroll
          for (int c = 0; c < 2; ++c) tma_load_2d_2cta(sa + c * (kBK * 128), &map_a, &full_bar[stage], m0 + c * 64, k0);
        }
        if constexpr (!B_MN) {
          tma_load_2d_2cta(sb, &map_b, &full_bar[stage], k0, n0);
        } else {
#pragma unroll
          for (int c = 0; c < 2; ++c) tma_load_2d_2cta(sb + c * (kBK * 128), &map_b, &full_bar[stage], n0 + c * 64, k0);
        }
        if (++stage == k2Stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 11 && lane == 0 && rank == 0) {
    // ===================== MMA issuer (leader CTA, single thread) =====================
    constexpr uint32_t idesc = make_idesc_bf16(256, BN, A_MN, B_MN);
    constexpr uint32_t a_lbo = A_MN ? kBK * 128 : 16, a_kstep = A_MN ? 2048 : 32;
    constexpr uint32_t b_lbo = B_MN ? kBK * 128 : 16, b_kstep = B_MN ? 2048 : 32;
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int pt = cluster_id; pt < num_pt; pt += num_clusters, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        const uint32_t sa = smem_u32(smem + stage * k2StageBytes);
        const uint32_t sb = sa + 128 * kBK * 2;
        const uint64_t da = make_smem_desc(sa, a_lbo, 1024);
        const uint64_t db = make_smem_desc(sb, b_lbo, 1024);
#pragma unroll
        for (int k = 0; k < kBK / 16; ++k)
          umma_bf16_2cta(d_tmem, da + ((k * a_kstep) >> 4), db + ((k * b_kstep) >> 4), idesc, (kb | k) != 0);
        umma_commit_2cta_mcast(&empty_bar[stage], 0x3);
        if (++stage == k2Stages) { stage = 0; phase ^= 1; }
      }
      umma_commit_2cta_mcast(&tfull_bar[acc], 0x3);
    }
  } else if (warp < 8) {
    // ===================== epilogue warps (both CTAs; each CTA owns its 128 rows) =====================
    const int q = warp & 3, half = warp >> 2;
    float scale = ep.alpha;
    if (ep.scale_ptr != nullptr) {
      const float s = __ldg(ep.scale_ptr);
      scale *= ep.scale_tanh ? tanhf(s) : s;
    }
    int it = 0;
    for (int pt = cluster_id; pt < num_pt; pt += num_clusters, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int m0 = (pt % tiles_mp) * 256 + static_cast<int>(rank) * 128;
      const int n0 = (pt / tiles_mp) * BN;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BN;
      if constexpr (TS)
        epilogue_dispatch_tma<BN>(ep, scale, taddr, m0, n0, M, N, q, half, lane, epi_stage + warp * kEpiWarpStage, &map_d);
      else
        epilogue_tile<BN>(ep, scale, taddr, m0, n0, M, N, q, half, lane);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(&tempty_bar[acc], 0);      // leader's barrier
    }
    if (TS && lane == 0) tma_store_wait_read<0>();   // the stage must outlive the last bulk store's reads
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc_2cta(tmem_base, 512);
  }
}

template <bool A_MN, bool B_MN, bool TS>
static int launch_gemm2(const void* A, long long lda, const void* B, long long ldb, int M, int N, int K,
                        const GemmEpi& ep, cudaStream_t stream) {
  CUtensorMap ma, mb;
  int rc;
  if (!A_MN) rc = make_tmap_bf16_2d(&ma, A, M, K, lda, 128, 64);
  else       rc = make_tmap_bf16_2d(&ma, A, K, M, lda, kBK, 64);
  if (rc) return rc;
  if (!B_MN) rc = make_tmap_bf16_2d(&mb, B, N, K, ldb, 128, 64);
  else       rc = make_tmap_bf16_2d(&mb, B, K, N, ldb, kBK, 64);
  if (rc) return rc;
  CUtensorMap md = ma;
  if (TS) {
    rc = ep.out_fp32 ? make_tmap_f32_2d(&md, ep.out, M, N, ep.ld_out, 32, 32)
                     : make_tmap_bf16_2d(&md, ep.out, M, N, ep.ld_out, 32, 64);
    if (rc) return rc;
  }
  auto kern = gemm2_bf16_kernel<A_MN, B_MN, TS>;
  constexpr int smem_bytes = k2SmemBytes + (TS ? kEpiStageBytes : 0);
  OTB_CHECK_CUDA(ensure_dyn_smem(kern, smem_bytes));
  const int num_pt = ((M + 255) / 256) * ((N + 255) / 256);
  const int max_clusters = sm_count() / 2;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[2];
  int nattr = 0;
  if (pdl_enabled()) {
    attr[nattr].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[nattr].val.programmaticStreamSerializationAllowed = 1;
    ++nattr;
  }
  attr[nattr].id = cudaLaunchAttributeClusterDimension;
  attr[nattr].val.clusterDim.x = 2; attr[nattr].val.clusterDim.y = 1; attr[nattr].val.clusterDim.z = 1;
  ++nattr;
  cfg.gridDim = dim3(2 * (num_pt < max_clusters ? num_pt : max_clusters));
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cfg.attrs = attr;
  cfg.numAttrs = nattr;
  OTB_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, ma, mb, md, M, N, K, ep));
  count_launch();
  return OTB_OK;
}

}  // namespace otb

extern "C" int otb_gemm_bf16(const void* A, int a_mn_major, int64_t lda, const void* B, int b_mn_major, int64_t ldb,
                             int M, int N, int K, const otb_gemm_epilogue* e, void* stream) {
  using namespace otb;
  OTB_CHECK_ARG(A && B && e && e->out, "otb_gemm_bf16: null pointer");
  // Operands go through TMA and the epilogue reads / writes 16 B vectors (uint4 / float4): every matrix and the bias
  // must start on a 16-byte boundary.  A misaligned pointer is an argument error, not a fault inside the kernel.
  {
    const void* ptrs[7] = {A, B, e->out, e->bias, e->residual, e->aux_in, e->aux_out};
    const char* names[7] = {"A", "B", "out", "bias", "residual", "aux_in", "aux_out"};
    for (int i = 0; i < 7; ++i)
      OTB_CHECK_ARG((reinterpret_cast<uintptr_t>(ptrs[i]) & 15) == 0, "otb_gemm_bf16: %s is not 16-byte aligned",
                    names[i]);
  }
  OTB_CHECK_ARG(M > 0 && N > 0 && K > 0, "otb_gemm_bf16: bad shape %d %d %d", M, N, K);
  OTB_CHECK_ARG(N % 8 == 0, "otb_gemm_bf16: N=%d must be a multiple of 8", N);
  OTB_CHECK_ARG(e->ld_out % 8 == 0 && e->ld_out >= N, "otb_gemm_bf16: bad ld_out");
  OTB_CHECK_ARG(!e->accumulate || e->out_fp32, "otb_gemm_bf16: accumulate requires fp32 output");
  OTB_CHECK_ARG(e->aux_in == nullptr || (e->ld_aux_in % 8 == 0 && e->ld_aux_in >= N), "otb_gemm_bf16: bad ld_aux_in");
  OTB_CHECK_ARG(e->aux_out == nullptr || (e->ld_aux_out % 8 == 0 && e->ld_aux_out >= N),
                "otb_gemm_bf16: bad ld_aux_out");
  OTB_CHECK_ARG(e->residual == nullptr || (e->ld_res % 8 == 0 && e->ld_res >= N), "otb_gemm_bf16: bad ld_res");
  OTB_CHECK_ARG(e->act >= 0 && e->act <= 3, "otb_gemm_bf16: bad act");
  if (a_mn_major) OTB_CHECK_ARG(M % 8 == 0 && lda >= M, "otb_gemm_bf16: MN-major A needs M%%8==0, lda>=M");
  else OTB_CHECK_ARG(lda >= K, "otb_gemm_bf16: lda < K");
  if (b_mn_major) OTB_CHECK_ARG(ldb >= N, "otb_gemm_bf16: ldb < N");
  else OTB_CHECK_ARG(ldb >= K, "otb_gemm_bf16: ldb < K");

  GemmEpi ep;
  ep.bias = e->bias;
  ep.aux_in = static_cast<const bf16*>(e->aux_in);
  ep.aux_out = static_cast<bf16*>(e->aux_out);
  ep.scale_ptr = e->scale_ptr;
  ep.residual = static_cast<const bf16*>(e->residual);
  ep.out = e->out;
  ep.ld_out = e->ld_out; ep.ld_aux_in = e->ld_aux_in; ep.ld_aux_out = e->ld_aux_out; ep.ld_res = e->ld_res;
  ep.act = e->act; ep.scale_tanh = e->scale_tanh; ep.out_fp32 = e->out_fp32; ep.accumulate = e->accumulate;
  ep.alpha = e->alpha;
  ep.res_fp32 = e->res_fp32;
  OTB_CHECK_ARG(!e->res_fp32 || e->out_fp32, "otb_gemm_bf16: fp32 residual requires fp32 output");
  // Outputs leave through the smem-staged TMA-store / reduce-add epilogue (r02: FFN up GELU+aux 194 -> 164 us, fp32
  // wgrad 206 -> 171 us, step +3 %; profiles/r02_gemm_selftest_bench.md).  OTB_GEMM_EPI_TMA=0 selects direct stores.
  static const bool epi_tma = [] { const char* v = getenv("OTB_GEMM_EPI_TMA"); return !(v && v[0] == '0'); }();
  ep.tma_out = (epi_tma && !e->res_fp32 && (!e->out_fp32 || e->ld_out % 4 == 0)) ? 1 : 0;
  ep.cls = -1;
  if (ep.tma_out && e->res_fp32 == 0) {
    const bool scaled = (e->scale_ptr != nullptr) || e->alpha != 1.0f;
    for (int c = 0; c < kNumEpiCls; ++c) {
      const EpiCls& k = kEpiCls[c];
      if (k.bias == (e->bias != nullptr) && k.aux_out == (e->aux_out != nullptr) && k.aux_in == (e->aux_in != nullptr) &&
          k.act == (e->aux_in ? 0 : e->act) && (e->aux_in == nullptr || e->act != 3) && k.scale == scaled &&
          k.res == (e->residual != nullptr) && k.out_f32 == (e->out_fp32 != 0) && k.acc == (e->accumulate != 0)) {
        ep.cls = c;
        break;
      }
    }
  }
  static const bool cls_off = [] { const char* v = getenv("OTB_GEMM_EPI_CLS"); return v && v[0] == '0'; }();
  if (cls_off) ep.cls = -1;
  cudaStream_t st = static_cast<cudaStream_t>(stream);

  // Tile-N choice: 256-wide tiles unless that leaves most SMs idle.  CTA-pair multicast (MC) when there are at
  // least two row tiles and enough pairs to fill the chip (otherwise single CTAs spread wider).
  const int tiles_m = (M + kBM - 1) / kBM;
  const int tiles256 = tiles_m * ((N + 255) / 256);
  const bool bn128 = (N <= 128) || (tiles256 < sm_count() && N > 128);
  const int tiles = bn128 ? tiles_m * ((N + 127) / 128) : tiles256;
  static const bool mc_off = (getenv("OTB_GEMM_NO_MCAST") != nullptr);
  // OTB_GEMM_MC_MIN_TILES: smallest tile count that uses the 2-CTA multicast variant (default: one tile per SM).  CLIP
  // out_proj / fc2 (136 tiles of 128x128, K up to 4096) are L2-bandwidth bound at 64 FLOP/B; sharing the B tile in a
  // pair cuts their L2 traffic by a quarter.
  static const int mc_min_tiles = [] { const char* v = getenv("OTB_GEMM_MC_MIN_TILES"); return v ? atoi(v) : 0; }();
  const bool mc = !mc_off && tiles_m >= 2 && (tiles_m % 2 == 0 || tiles_m >= 9) &&
                  tiles >= (mc_min_tiles > 0 ? mc_min_tiles : sm_count());
  const int sel = (a_mn_major ? 2 : 0) | (b_mn_major ? 1 : 0);
  // cta_group::2 pair kernel for the large problems (>= one 256x256 pair tile per SM pair)
  static const int two_cta = [] { const char* e = getenv("OTB_GEMM_2CTA"); return e ? atoi(e) : 1; }();
  // (sending the 36-pair-tile CLIP out_proj / fc2 problems to the pair kernel was measured slower: profiles/r02_call1_knob_ab.md)
  const int pair_tiles = ((M + 255) / 256) * ((N + 255) / 256);
  const bool pair_ok = !bn128 && pair_tiles >= sm_count() / 2;
  if (two_cta && pair_ok) {
#define OTB_GEMM2_CASE(A_, B_)                                                        \
  return ep.tma_out ? launch_gemm2<A_, B_, true>(A, lda, B, ldb, M, N, K, ep, st)     \
                    : launch_gemm2<A_, B_, false>(A, lda, B, ldb, M, N, K, ep, st)
    switch (sel) {
      case 0: OTB_GEMM2_CASE(false, false);
      case 1: OTB_GEMM2_CASE(false, true);
      case 3: OTB_GEMM2_CASE(true, true);
      default: break;
    }
#undef OTB_GEMM2_CASE
  }
#define OTB_GEMM_CASE(BN_, A_, B_)                                                                   \
  if (ep.tma_out)                                                                                     \
    return mc ? launch_gemm<BN_, A_, B_, true, true>(A, lda, B, ldb, M, N, K, ep, st)                 \
              : launch_gemm<BN_, A_, B_, false, true>(A, lda, B, ldb, M, N, K, ep, st);               \
  return mc ? launch_gemm<BN_, A_, B_, true, false>(A, lda, B, ldb, M, N, K, ep, st)                  \
            : launch_gemm<BN_, A_, B_, false, false>(A, lda, B, ldb, M, N, K, ep, st)
  if (bn128) {
    switch (sel) {
      case 0: OTB_GEMM_CASE(128, false, false);
      case 1: OTB_GEMM_CASE(128, false, true);
      case 3: OTB_GEMM_CASE(128, true, true);
      default: break;
    }
  } else {
    switch (sel) {
      case 0: OTB_GEMM_CASE(256, false, false);
      case 1: OTB_GEMM_CASE(256, false, true);
      case 3: OTB_GEMM_CASE(256, true, true);
      default: break;
    }
  }
#undef OTB_GEMM_CASE
  return set_error(OTB_ERR_UNSUPPORTED, "otb_gemm_bf16: layout (A MN-major, B K-major) not instantiated");
}
