// prisma_b200 -- the tcgen05 "shifted-row GEMM" core (sm_100a).
//
//   D[m, n] = sum_{t < taps} sum_{c < Cin} A[m + tap_off[t], c] * W[n, t * kchunks*64 + c]        (fp16 x fp16 -> fp32)
//
// taps == 1, tap_off = {0}  : a plain GEMM (ViT linears, 1x1 convs, transposed convs with k == s, RAFT correlation)
// taps == kh*kw             : an implicit-GEMM convolution over a zero-bordered NHWC activation whose pixels are
//                             flattened to rows; tap (ky,kx) is the same 2-D TMA box shifted by (ky-ph)*Wp + (kx-pw)
//                             rows.  Border rows are computed and discarded (waste 2/(W+2)); no im2col buffer, no 4-D
//                             tensor map; TMA zero-fills out-of-range rows (either sign).
//
// Kernel anatomy (persistent, warp-specialised, one CTA per SM):
//   warp 0   : TMA producer  (A 128x64 and W BNx64 fp16 tiles, 128B swizzle, STAGES-deep mbarrier ring)
//   warp 1   : MMA issuer    (one lane: tcgen05.mma cta_group::1 kind::f16, M=128, N=BN, K=16; fp32 accum in TMEM,
//                             two accumulator stages so the epilogue of tile i overlaps the mainloop of tile i+1)
//   warps 2-9: epilogue      (tcgen05.ld 32x32b -> registers -> smem transpose -> bias / GELU / ReLU / LayerScale /
//                             residuals -> coalesced fp32 and/or fp16 stores with the row mapping of the consumer's
//                             layout; two warps per TMEM lane quarter take alternate 32-column chunks; every
//                             global access of a chunk is issued as a batch of 8 independent requests per lane)
#pragma once
#include "common.cuh"

namespace prisma {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_EPI_WARPS = 8;                          // two per TMEM lane quarter (EW template parameter: 8 or 16)
constexpr int GEMM_THREADS = 64 + 32 * GEMM_EPI_WARPS;      // + TMA producer warp + MMA warp
constexpr int GEMM_SMEM_MAX = 232448;                       // 227 KB of dynamic shared memory per CTA
constexpr int GEMM_MAX_TAPS = 49;
constexpr int GEMM_TF32_ACC_GROUP = 4;  // 3xTF32: K blocks per TMEM chain before the external fp32 add (see the MMA issuer)

enum RowMap : int {
  ROW_LINEAR = 0,   // dst row = m                                   (valid: m < M)
  ROW_PADDED = 1,   // m indexes a zero-bordered [Hp][Wp] image; only interior pixels are stored (borders stay zero)
  ROW_TOK2PAD = 2,  // m = y*W + x (dense tokens)  -> dst row (y+1)*out_wp + x+1
  ROW_PAD2TOK = 5,  // m indexes a zero-bordered image; interior pixel (y,x) -> dense dst row img*H*W + y*W + x
  ROW_TOKSKIP = 4,  // m = b*P + p (patch tokens of image b) -> dst row b*(P+1) + 1 + p  (skips the cls rows; in_w = P)
  ROW_SHUFFLE = 3,  // ConvTranspose k == s: m = y*W + x, n = (dy*s+dx)*cout + co -> dst row (y*s+dy+1)*out_wp + x*s+dx+1
};

struct GemmEpilogue {
  float alpha = 1.0f;            // accumulator scale (e.g. 1/sqrt(C) of the RAFT correlation), applied first
  const float* bias = nullptr;   // [N]
  const float* gamma = nullptr;  // [N]  LayerScale
  int act = 0;                   // 0 none, 1 exact-erf GELU, 2 ReLU, 3 sigmoid, 4 tanh (fast, ~4e-7), 5 softplus, 6 sigmoid (expf + IEEE div)
  const float* pre_f32 = nullptr;  // + a per-element fp32 term BEFORE the activation, indexed by dst row (e.g. the part of a
  int pre_f32_ld = 0;              //   conv over concatenated inputs that does not change between iterations)
  const float* res_f32 = nullptr;  // + residual (fp32), indexed by dst row
  int res_f32_ld = 0;
  const __half* res_a = nullptr;  // + residual (fp16), indexed by dst row
  int res_a_ld = 0;
  const __half* res_b = nullptr;
  int res_b_ld = 0;
  float* out_f32 = nullptr;
  int out_f32_ld = 0;
  __half* out_f16 = nullptr;
  int out_f16_ld = 0;
  __half* out_f16_relu = nullptr;  // relu(result) copy, for consumers that take relu(x) as operand and x as skip
  int out_f16_relu_ld = 0;
  int row_map = ROW_LINEAR;
  int img_rows = 0;  // ROW_PADDED: rows per image (Hp*Wp); 0 = single image
  int in_w = 0;      // ROW_PADDED: Wp ; ROW_TOK2PAD / ROW_SHUFFLE: W
  int in_h = 0;      // ROW_PADDED: Hp ; ROW_TOK2PAD / ROW_SHUFFLE: H (rows per image = H*W)
  int out_wp = 0;    // destination padded width
  int out_img_rows = 0;  // destination rows per image
  int sub = 1;       // ROW_PADDED: keep every sub-th pixel (stride-2 conv evaluated at stride 1)
  int pad = 1;       // ROW_PADDED / ROW_PAD2TOK: border width of the input geometry; out_pad: of the destination
  int out_pad = 1;
  // Border placement.  lead < 0 (default): symmetric border, `pad` pixels on every side (in_h = H + 2 pad).
  // lead == 0: "shared border" layout -- `pad` zero columns only at the END of every row and `pad` zero rows only at the END
  // of every image (in_h = H + pad, in_w = W + pad).  A negative tap shift then lands in the previous row's / previous
  // image's trailing zeros (or before row 0, where TMA zero-fills), so the halo is still all zeros but the GEMM walks
  // (H + pad)(W + pad) rows instead of (H + 2 pad)(W + 2 pad).  out_lead: the same for the destination map.
  int lead = -1;
  int out_lead = -1;
  int shuf_s = 1;
  int shuf_cout = 0;
  // fused DPT output head (dpt.py:96-100): depth = relu(head_b + sum_j head_w[j] * relu(acc[j] + bias[j])), N == 32,
  // written dense fp32 [H][W] (ROW_PADDED input geometry)
  const float* head_w = nullptr;
  float head_b = 0.f;
  float* head_out = nullptr;
  // Column statistics of the stored values, for a normalisation that follows the conv (RAFT's InstanceNorm2d): every
  // 32-row slab of the output space (slab = m / 32; image row counts are multiples of 32, so a slab lies in one image)
  // writes sum and sum of squares over its VALID rows: stat_part[(slab * 2 + {0,1}) * N + n], fp32, deterministic
  // (fixed shuffle tree; a second kernel adds the slabs in double precision in a fixed order).
  float* stat_part = nullptr;
  // Row count known only on the device (SOLOv2: the number of candidates of this frame): when set, only the first
  // round_up(*m_dev, 128) rows of the output space are computed (the launch is sized for the capacity M).
  const int* m_dev = nullptr;
  // dense output (row_map LINEAR; out_f32: scale only; out_f16: scale, bias, GELU / ReLU) stored by TMA: tcgen05.ld ->
  // registers (row per lane) -> swizzled smem box -> cp.async.bulk.tensor
  bool tma_store = false;
  // set by gemm_prepare when tma_store is asked for an in-place fp32 residual update (res_f32 == out_f32: the ViT proj / fc2
  // linears, x += gamma (acc + bias)): the staged box leaves through cp.reduce.async.bulk.tensor ... .add.f32 -- the add is
  // done by the L2 (one round-to-nearest fp32 add per element, as the register path does); the epilogue reads nothing
  bool tma_reduce = false;
  // ConvGRU gate arithmetic in the epilogue of the gate convs (raft/update.py:54-58), all fp32, indexed by dst row:
  //  gru == 1 (the z | r conv, N = 256, act sigmoid): columns [0,128) = z -> out_f32 as usual; columns [128,256) = r are not
  //            stored: r * h (gru_h: fp32 [rows][128]) goes to gru_rh (fp16, pitch gru_rh_ld) -- the q conv's operand;
  //  gru == 2 (the q conv, N = 128, act tanh): h' = (1 - z) h + z q with z = gru_z (fp32, pitch 256) and h = gru_h; h' then
  //            takes the normal output path (out_f32 = the fp32 master of h, in place; out_f16 = the conv operand copy).
  int gru = 0;
  const float* gru_h = nullptr;
  const float* gru_z = nullptr;
  __half* gru_rh = nullptr;
  int gru_rh_ld = 0;
};

struct GemmArgs {
  int M;  // rows of the output space
  int N;  // output columns
  int taps;
  int kchunks;  // 64-wide K blocks per tap
  int tap_off[GEMM_MAX_TAPS];
  int tap_acol[GEMM_MAX_TAPS];  // first A column (elements) of each tap's K slab: 0 for plain convs; the 3xTF32 path walks
                                // [hi | lo] activation halves: (hi, W_hi), (lo, W_hi), (hi, W_lo)
  int n_main;      // work items [0, n_main) are full BN-wide tiles; the remaining tiles are each cut into `tail_split`
  int tail_split;  // narrower tiles (BN / tail_split wide) so the last partial wave costs a fraction of a full one; 1 = off
  int raster_n;  // 1: consecutive tiles walk N first (the CTAs of a wave share few A row panels and all of W: A is read
                 // from HBM once when M >> N); 0: M first
  GemmEpilogue ep;
};

// SWAP ("swap A/B", BN == 128, CG == 1): the tensor core spends >= 128 cycles on every M = 128 instruction whatever its N
// (measured: N = 128 tiles reach half the rate of N = 256 ones with no loads and no epilogue), so a
// GEMM with <= 128 output columns runs transposed: the WEIGHT tile (128 output channels) is the M operand, 256 pixel rows
// are the N operand of one instruction, the accumulator holds channels in its lanes and pixels in its columns, and the
// epilogue transposes through its staging buffer (which it does anyway).  Half the instructions, barriers and TMA boxes
// per FLOP; the operand bytes per FLOP drop by a quarter.
// EW: epilogue warps (EW / 4 per TMEM lane quarter, taking every (EW / 4)-th 32-column chunk).  The epilogue is latency-bound
// (ncu on fc1: issue slots 25 % busy, long-scoreboard / wait stalls) and paces the kernel (DESIGN 4.1), so the fp16 kernels can
// run 16 of them: half the chunks per warp; one operand stage is given up for the staging buffers and the register cap
// drops: 18 warps put 5 on one scheduler's 16 K registers = 96 per thread (spills 100-280 bytes).
template <int BN, int CG = 1, bool TMAST = false, bool SWAP = false, int EW = GEMM_EPI_WARPS>  // CG = CTAs per MMA (cta_group): 2 = a CTA pair computes a 256 x BN tile, each loading half of W
struct GemmCfg {                                   // TMAST: TMA-store epilogue (double-buffered staging, one operand stage fewer)
  static constexpr int A_ROWS = SWAP ? 256 : GEMM_BM;   // activation rows per tile and CTA
  static constexpr int ACC_COLS = SWAP ? 256 : BN;      // TMEM columns of one accumulator stage
  static constexpr int A_BYTES = A_ROWS * GEMM_BK * 2;
  static constexpr int B_BYTES = (BN / CG) * GEMM_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STG_BYTES = EW * 32 * 32 * 4 * (TMAST ? 2 : 1);  // epilogue staging: 32x32 fp32 per warp (x2 buffers)
  static constexpr int FIT = (GEMM_SMEM_MAX - STG_BYTES - 1280) / STAGE_BYTES;  // operand stages that fit beside the staging
  static constexpr int STAGES = FIT > 7 ? 7 : FIT;
  static constexpr int THREADS = 64 + 32 * EW;
  static constexpr int TMEM_COLS = (2 * ACC_COLS <= 32) ? 32 : (2 * ACC_COLS <= 64 ? 64 : (2 * ACC_COLS <= 128 ? 128 : (2 * ACC_COLS <= 256 ? 256 : 512)));
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STG_BYTES + 1024 /*align slack*/ + 256 /*barriers*/;
  static_assert(STAGES >= 3, "too few operand stages");
};

#ifdef __CUDACC__
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752f)); }
// sigmoid / tanh of the fused epilogues: ex2.approx + rcp.approx (relative error ~4e-7, absolute error of tanh ~2e-7) instead
// of expf + IEEE division / tanhf.  Measured on the RAFT gate conv (37 888 x 256 outputs): the exact versions cost 18 us per
// launch on top of an 18.8 us kernel; their accuracy is irrelevant next to the fp16 operand rounding (5e-4).
__device__ __forceinline__ float sigmoid_f(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float tanh_f(float x) { return 1.0f - __fdividef(2.0f, __expf(2.0f * x) + 1.0f); }
__device__ __forceinline__ float softplus_f(float x) { return x > 20.f ? x : log1pf(expf(x)); }  // nn.Softplus(beta 1, threshold 20)

__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void add_h4(float4& v, const uint2& r) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
  v.x += a.x; v.y += a.y; v.z += b.x; v.w += b.y;
}

// Coalesced phase of the epilogue for one 32-column chunk: this lane owns 4 consecutive columns (col..col+3) of the
// 8 rows dr[0..7] (8 lanes cover a row's 32 columns, so a warp instruction touches 4 rows x 128 B fp32 / 64 B fp16).
// All loads of a kind are issued before any is consumed (8 independent requests in flight per lane).
template <bool GRU>  // GRU: compile the ConvGRU gate paths (fp16-operand instantiations only; keeps the 3xTF32 kernels lean)
__device__ __forceinline__ void epilogue_rows8(const GemmEpilogue& ep, float4 (&v)[8], const int (&dr)[8], uint32_t okm,
                                               const float4& bias, const float4& gamma, int col) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    v[i].x = fmaf(v[i].x, ep.alpha, bias.x); v[i].y = fmaf(v[i].y, ep.alpha, bias.y);
    v[i].z = fmaf(v[i].z, ep.alpha, bias.z); v[i].w = fmaf(v[i].w, ep.alpha, bias.w);
  }
  if (ep.pre_f32) {
    float4 t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      t[i] = (okm >> i) & 1 ? *reinterpret_cast<const float4*>(ep.pre_f32 + (size_t)dr[i] * ep.pre_f32_ld + col)
                            : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i].x += t[i].x; v[i].y += t[i].y; v[i].z += t[i].z; v[i].w += t[i].w; }
  }
  if (ep.act == 1) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i].x = gelu_erf(v[i].x); v[i].y = gelu_erf(v[i].y); v[i].z = gelu_erf(v[i].z); v[i].w = gelu_erf(v[i].w); }
  } else if (ep.act == 2) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i].x = fmaxf(v[i].x, 0.f); v[i].y = fmaxf(v[i].y, 0.f); v[i].z = fmaxf(v[i].z, 0.f); v[i].w = fmaxf(v[i].w, 0.f); }
  } else if (ep.act == 3) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i].x = sigmoid_f(v[i].x); v[i].y = sigmoid_f(v[i].y); v[i].z = sigmoid_f(v[i].z); v[i].w = sigmoid_f(v[i].w); }
  } else if (ep.act == 4) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i].x = tanh_f(v[i].x); v[i].y = tanh_f(v[i].y); v[i].z = tanh_f(v[i].z); v[i].w = tanh_f(v[i].w); }
  } else if (ep.act == 6) {  // sigmoid with expf and an IEEE division: the mask predictions of the fp32-class SOLOv2 head
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      v[i].x = 1.0f / (1.0f + expf(-v[i].x)); v[i].y = 1.0f / (1.0f + expf(-v[i].y));
      v[i].z = 1.0f / (1.0f + expf(-v[i].z)); v[i].w = 1.0f / (1.0f + expf(-v[i].w));
    }
  } else if (ep.act == 5) {
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i].x = softplus_f(v[i].x); v[i].y = softplus_f(v[i].y); v[i].z = softplus_f(v[i].z); v[i].w = softplus_f(v[i].w); }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) { v[i].x *= gamma.x; v[i].y *= gamma.y; v[i].z *= gamma.z; v[i].w *= gamma.w; }
  if (GRU && ep.gru == 1) {
    if (col >= 128) {  // warp-uniform: a 32-column chunk lies in one half
      float4 h[8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
        h[i] = (okm >> i) & 1 ? *reinterpret_cast<const float4*>(ep.gru_h + (size_t)dr[i] * 128 + (col - 128))
                              : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if ((okm >> i) & 1)
          *reinterpret_cast<uint2*>(ep.gru_rh + (size_t)dr[i] * ep.gru_rh_ld + (col - 128)) =
              make_uint2(pack_half2(v[i].x * h[i].x, v[i].y * h[i].y), pack_half2(v[i].z * h[i].z, v[i].w * h[i].w));
      return;
    }
  } else if (GRU && ep.gru == 2) {
    float4 z[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      z[i] = (okm >> i) & 1 ? *reinterpret_cast<const float4*>(ep.gru_z + (size_t)dr[i] * 256 + col) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i].x *= z[i].x; v[i].y *= z[i].y; v[i].z *= z[i].z; v[i].w *= z[i].w; }   // z q
#pragma unroll
    for (int i = 0; i < 8; ++i) { z[i].x = 1.f - z[i].x; z[i].y = 1.f - z[i].y; z[i].z = 1.f - z[i].z; z[i].w = 1.f - z[i].w; }
    float4 h[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      h[i] = (okm >> i) & 1 ? *reinterpret_cast<const float4*>(ep.gru_h + (size_t)dr[i] * 128 + col) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {  // (1 - z) * h + z * q, the products rounded separately like the reference's two multiplies
      v[i].x = __fadd_rn(__fmul_rn(z[i].x, h[i].x), v[i].x); v[i].y = __fadd_rn(__fmul_rn(z[i].y, h[i].y), v[i].y);
      v[i].z = __fadd_rn(__fmul_rn(z[i].z, h[i].z), v[i].z); v[i].w = __fadd_rn(__fmul_rn(z[i].w, h[i].w), v[i].w);
    }
  }
  if (ep.res_f32) {
    float4 t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      t[i] = (okm >> i) & 1 ? *reinterpret_cast<const float4*>(ep.res_f32 + (size_t)dr[i] * ep.res_f32_ld + col)
                            : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) { v[i].x += t[i].x; v[i].y += t[i].y; v[i].z += t[i].z; v[i].w += t[i].w; }
  }
  if (ep.res_a) {
    uint2 t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      t[i] = (okm >> i) & 1 ? *reinterpret_cast<const uint2*>(ep.res_a + (size_t)dr[i] * ep.res_a_ld + col) : make_uint2(0u, 0u);
#pragma unroll
    for (int i = 0; i < 8; ++i) add_h4(v[i], t[i]);
  }
  if (ep.res_b) {
    uint2 t[8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
      t[i] = (okm >> i) & 1 ? *reinterpret_cast<const uint2*>(ep.res_b + (size_t)dr[i] * ep.res_b_ld + col) : make_uint2(0u, 0u);
#pragma unroll
    for (int i = 0; i < 8; ++i) add_h4(v[i], t[i]);
  }
  if (ep.out_f32) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((okm >> i) & 1) *reinterpret_cast<float4*>(ep.out_f32 + (size_t)dr[i] * ep.out_f32_ld + col) = v[i];
  }
  if (ep.out_f16) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((okm >> i) & 1)
        *reinterpret_cast<uint2*>(ep.out_f16 + (size_t)dr[i] * ep.out_f16_ld + col) =
            make_uint2(pack_half2(v[i].x, v[i].y), pack_half2(v[i].z, v[i].w));
  }
  if (ep.out_f16_relu) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if ((okm >> i) & 1)
        *reinterpret_cast<uint2*>(ep.out_f16_relu + (size_t)dr[i] * ep.out_f16_relu_ld + col) =
            make_uint2(pack_half2(fmaxf(v[i].x, 0.f), fmaxf(v[i].y, 0.f)), pack_half2(fmaxf(v[i].z, 0.f), fmaxf(v[i].w, 0.f)));
  }
}

template <int BN, int CG, bool TMAST, bool TF32, bool SWAP = false, int EW = GEMM_EPI_WARPS>
__global__ void __launch_bounds__(64 + 32 * EW, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
               const __grid_constant__ CUtensorMap tmBt, const __grid_constant__ CUtensorMap tmD,
               const __grid_constant__ GemmArgs args) {
  static_assert(!SWAP || (BN == 128 && CG == 1 && !TMAST && !TF32), "SWAP: 128 output channels x 256 pixel rows, fp16, one CTA");
  static_assert(!TF32 || (BN <= 128 && CG == 1 && !TMAST), "TF32 (external accumulation): BN <= 128, one CTA, register epilogue");
  static_assert(EW == 8 || (EW == 16 && !TMAST && !TF32), "16 epilogue warps: the plain fp16 kernels only");
  using Cfg = GemmCfg<BN, CG, TMAST, SWAP, EW>;
  constexpr int ACC = Cfg::ACC_COLS;
  constexpr int CSTEP = 32 * (EW / 4);  // column distance between the chunks one warp takes
  constexpr int STAGES = Cfg::STAGES;
  constexpr int BKE = TF32 ? 32 : 64;  // elements per 128-byte K block (fp32 containers for kind::tf32, fp16 otherwise)
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) {
    if (threadIdx.x == 0) printf("prisma: gemm smem base not 1024-aligned\n");
    __trap();
  }
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * Cfg::A_BYTES;
  float* stg_all = reinterpret_cast<float*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES + Cfg::STG_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tfull = bars + 2 * STAGES;
  uint64_t* tempty = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = CG == 2 ? (int)cluster_ctarank() : 0;  // position inside the CTA pair
  const int group = blockIdx.x / CG, num_groups = gridDim.x / CG;
  constexpr int TILE_M = SWAP ? 256 : GEMM_BM * CG;
  const int M_run = args.ep.m_dev ? min(args.M, (*args.ep.m_dev + TILE_M - 1) / TILE_M * TILE_M) : args.M;  // see GemmEpilogue::m_dev
  const int tiles_m = (M_run + TILE_M - 1) / TILE_M;
  const int tiles_n = (args.N + BN - 1) / BN;
  const int num_tiles = tiles_m * tiles_n;
  const int num_kb = args.taps * args.kchunks;
  // work items: full tiles first, then the tail tiles cut into `split` narrow ones (see GemmArgs::n_main)
  const int split = args.tail_split, n_main = split > 1 ? args.n_main : num_tiles;
  const int num_items = n_main + (num_tiles - n_main) * split;
  const int bw_tail = BN / split;  // width of a tail tile
  auto item_tile = [&](int item, int* tm, int* tn, int* nsub, int* bw) {
    int big = item;
    *nsub = 0; *bw = BN;
    if (item >= n_main) { const int u = item - n_main; big = n_main + u / split; *nsub = (u % split) * bw_tail; *bw = bw_tail; }
    *tm = args.raster_n ? big / tiles_n : big % tiles_m;
    *tn = args.raster_n ? big % tiles_n : big / tiles_m;
  };

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    for (int s = 0; s < STAGES; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&tfull[s], 1); mbar_init(&tempty[s], EW * CG); }
    fence_mbar_init();
  }
  if (warp == 1) { if (CG == 2) tmem_alloc_pair(tmem_slot, Cfg::TMEM_COLS); else tmem_alloc(tmem_slot, Cfg::TMEM_COLS); }
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();  // the peer's barriers must exist before anything targets them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int tile = group; tile < num_items; tile += num_groups) {
        int tm, tn, nsub, bw;
        item_tile(tile, &tm, &tn, &nsub, &bw);
        const int m0 = tm * TILE_M + rank * GEMM_BM;
        const int n0 = tn * BN + nsub + rank * (bw / CG);
        const CUtensorMap* tb = bw == BN ? &tmB : &tmBt;               // the tail map has a (bw / CG)-row box
        const uint32_t stage_bytes = Cfg::A_BYTES + (bw / CG) * GEMM_BK * 2;
        int tap = 0, chunk = 0;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          if (CG == 2) {
            // both CTAs' bytes land on the leader's barrier; only the leader arrives (count 1) and posts the total
            if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * stage_bytes);
            tma_load_2d_pair(sA + stage * Cfg::A_BYTES, &tmA, &full[stage], args.tap_acol[tap] + chunk * BKE, m0 + args.tap_off[tap]);
            tma_load_2d_pair(sB + stage * Cfg::B_BYTES, tb, &full[stage], kb * BKE, n0);
          } else {
            mbar_arrive_expect_tx(&full[stage], stage_bytes);
            tma_load_2d(sA + stage * Cfg::A_BYTES, &tmA, &full[stage], args.tap_acol[tap] + chunk * BKE, m0 + args.tap_off[tap]);
            tma_load_2d(sB + stage * Cfg::B_BYTES, tb, &full[stage], kb * BKE, n0);
          }
          if (++chunk == args.kchunks) { chunk = 0; ++tap; }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer (leader CTA of the pair only)
    if (lane == 0 && rank == 0) {
      constexpr uint32_t idesc_full = SWAP ? make_idesc_f16(128, 256) : (TF32 ? make_idesc_tf32(TILE_M, BN) : make_idesc_f16(TILE_M, BN));
      const uint32_t idesc_tail = make_idesc_f16(TILE_M, bw_tail);
      int stage = 0; uint32_t phase = 0;
      int it = 0;
      if (TF32) {
        // External accumulation: the tensor core adds into its fp32 accumulator by TRUNCATING the aligned addend, a bias
        // that grows with the length of the chain (measured: 5e-6 of sum |a||w| after ~900 MMAs).  Here a chain is only
        // GEMM_TF32_ACC_GROUP K blocks long; every finished partial sum is handed to the epilogue warps (tfull), which add it
        // to register-resident running sums with round-to-nearest FADDs, and the TMEM stage is reused (tempty).
        constexpr int G = GEMM_TF32_ACC_GROUP;
        int gi = 0;  // partial sums issued so far (TMEM stage = gi & 1)
        for (int tile = group; tile < num_items; tile += num_groups) {
          for (int kb = 0; kb < num_kb; ++kb) {
            const int kg = kb % G;
            if (kg == 0) { mbar_wait(&tempty[gi & 1], ((gi >> 1) & 1) ^ 1); tc_fence_after(); }
            const uint32_t tmem_d = tmem_base + (gi & 1) * BN;
            mbar_wait(&full[stage], phase);
            tc_fence_after();
            const uint64_t adesc = make_sdesc_sw128(smem_u32(sA + stage * Cfg::A_BYTES));
            const uint64_t bdesc = make_sdesc_sw128(smem_u32(sB + stage * Cfg::B_BYTES));
#pragma unroll
            for (int k = 0; k < GEMM_BK / 16; ++k)  // K = 8 fp32 = 32 B: +2 in the (addr >> 4) field
              umma_tf32(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc_full, (kg | k) != 0 ? 1u : 0u);
            umma_commit(&empty[stage]);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
            if (kg == G - 1 || kb == num_kb - 1) { umma_commit(&tfull[gi & 1]); ++gi; }
          }
        }
      } else
      for (int tile = group; tile < num_items; tile += num_groups, ++it) {
        const uint32_t idesc = tile < n_main ? idesc_full : idesc_tail;
        const int as = it & 1;
        const uint32_t aphase = (it >> 1) & 1;
        mbar_wait(&tempty[as], aphase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + as * ACC;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          // SWAP: the weight tile is the M operand, the 256 activation rows the N operand
          const uint64_t adesc = make_sdesc_sw128(smem_u32(SWAP ? sB + stage * Cfg::B_BYTES : sA + stage * Cfg::A_BYTES));
          const uint64_t bdesc = make_sdesc_sw128(smem_u32(SWAP ? sA + stage * Cfg::A_BYTES : sB + stage * Cfg::B_BYTES));
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k) {
            // advance 16 fp16 = 32 B along K inside the 128 B swizzled row: +2 in the (addr >> 4) field
            if (CG == 2) umma_f16_pair(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            else umma_f16(tmem_d, adesc + 2 * k, bdesc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          if (CG == 2) umma_commit_pair(&empty[stage]); else umma_commit(&empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        if (CG == 2) umma_commit_pair(&tfull[as]); else umma_commit(&tfull[as]);
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue warps (2..9)
    const int quarter = warp & 3;           // TMEM lane quarter this warp may access
    const int chunk_par = (warp - 2) >> 2;  // the EW / 4 warps of a quarter take every (EW / 4)-th 32-column chunk
    const GemmEpilogue& ep = args.ep;
    const uint32_t stg = smem_u32(stg_all) + (warp - 2) * (TMAST ? 8192 : 4096);
    uint32_t st_cnt = 0;  // TMAST: chunks stored so far by this warp (staging buffer parity)
    const int cg = lane & 7;     // coalesced phase: which 4-column group of the 32-column chunk
    const int rsub = lane >> 3;  // coalesced phase: row offset inside a 4-row step
    int it = 0;
    int xgi = 0;  // TF32: partial sums consumed so far
    for (int tile = group; tile < num_items; tile += num_groups, ++it) {
      const int as = it & 1;
      const uint32_t aphase = (it >> 1) & 1;
      int tm, tn, nsub, bw;
      item_tile(tile, &tm, &tn, &nsub, &bw);
      const int m0 = tm * TILE_M + rank * GEMM_BM;
      const int n0 = tn * BN + nsub;
      // ---- row mapping of the 32 output rows a chunk covers (lane == row inside the slab): once per tile (the warp's 32
      // accumulator rows), or -- SWAP, where the accumulator's COLUMNS are the output rows -- once per 32-pixel chunk
      int m = 0, valid = 0, drow = 0;
      int ty = 0, tx = 0, img_base = 0;  // token coordinates / image base row for ROW_SHUFFLE
      const int out_ld = ep.out_lead < 0 ? ep.out_pad : ep.out_lead;  // leading border of the destination map
      int dr8[8], ty8[8], tx8[8], ib8[8];
      uint32_t okrows = 0;
      auto map_rows = [&](const int mbase) {
        m = mbase + lane;
        valid = m < args.M;
        drow = m;
        ty = 0; tx = 0; img_base = 0;
        if (ep.row_map == ROW_PADDED || ep.row_map == ROW_PAD2TOK) {
          int img = 0, r = m;
          if (ep.img_rows > 0) { img = m / ep.img_rows; r = m - img * ep.img_rows; }
          const int y = r / ep.in_w, x = r - y * ep.in_w;
          const int pd = ep.pad, ld = ep.lead < 0 ? ep.pad : ep.lead;
          valid = valid && y >= ld && y < ep.in_h - pd && x >= ld && x < ep.in_w - pd;
          if (ep.row_map == ROW_PAD2TOK) {
            const int ho = (ep.in_h - pd - ld + ep.sub - 1) / ep.sub, wo = (ep.in_w - pd - ld + ep.sub - 1) / ep.sub;
            valid = valid && ((y - ld) % ep.sub == 0) && ((x - ld) % ep.sub == 0);
            drow = img * (ep.out_img_rows > 0 ? ep.out_img_rows : ho * wo) + ((y - ld) / ep.sub) * wo + (x - ld) / ep.sub;
          } else if (ep.sub > 1 || ep.out_wp > 0) {
            // destination geometry differs from the source one (stride-2 sub-sampling and / or another border width)
            valid = valid && ((y - ld) % ep.sub == 0) && ((x - ld) % ep.sub == 0);
            drow = img * ep.out_img_rows + ((y - ld) / ep.sub + out_ld) * ep.out_wp + (x - ld) / ep.sub + out_ld;
          }
        } else if (ep.row_map == ROW_TOKSKIP) {
          drow = m + m / ep.in_w + 1;
        } else if (ep.row_map == ROW_TOK2PAD || ep.row_map == ROW_SHUFFLE) {
          const int per = ep.in_w * ep.in_h;
          const int img = m / per, r = m - img * per;
          ty = r / ep.in_w; tx = r - ty * ep.in_w;
          img_base = img * ep.out_img_rows;
          drow = img_base + (ty + out_ld) * ep.out_wp + tx + out_ld;
        }
        // row mapping of the 8 rows this lane stores in the coalesced phase
        okrows = 0;
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          const int row = rr * 4 + rsub;
          okrows |= (__shfl_sync(0xffffffffu, valid, row) ? 1u : 0u) << rr;
          dr8[rr] = __shfl_sync(0xffffffffu, drow, row);
          if (ep.row_map == ROW_SHUFFLE) {
            ty8[rr] = __shfl_sync(0xffffffffu, ty, row);
            tx8[rr] = __shfl_sync(0xffffffffu, tx, row);
            ib8[rr] = __shfl_sync(0xffffffffu, img_base, row);
          }
        }
      };
      if (!SWAP) map_rows(m0 + quarter * 32);
      // one 32-column chunk of this warp's 32 accumulator rows: r[j] = row `lane`, column c0 + j
      // bias / LayerScale vectors of a chunk: issued BEFORE the TMEM read is waited for, so the global-load latency hides
      // behind it (they used to sit between the shared-memory phases, on the critical path of every chunk)
      auto load_bias_gamma = [&](const int c0, float4& bias4, float4& gamma4) {
        const int n = SWAP ? n0 + quarter * 32 + cg * 4 : n0 + c0 + cg * 4;
        bias4 = make_float4(0.f, 0.f, 0.f, 0.f);
        gamma4 = make_float4(1.f, 1.f, 1.f, 1.f);
        if (n < args.N && ep.bias) bias4 = *reinterpret_cast<const float4*>(ep.bias + n);
        if (n < args.N && ep.gamma) gamma4 = *reinterpret_cast<const float4*>(ep.gamma + n);
      };
      auto process_chunk = [&](uint32_t (&r)[32], const int c0, const float4& bias4, const float4& gamma4) {
        if (TMAST) {
          // ---- TMA-store path: registers -> swizzled 32 x 128 B box (the XOR of the 16-byte slot with row & 7 IS the
          // 128-byte TMA swizzle of a 1024-aligned buffer) -> one cp.async.bulk.tensor store by lane 0; two boxes per warp
          // so the store of chunk i reads shared memory while chunk i + 1 is being staged
          const uint32_t buf = stg + (st_cnt & 1) * 4096;
          if (st_cnt >= 2) { if (lane == 0) tma_store_wait_read<1>(); __syncwarp(); }
          if (ep.bias == nullptr && ep.gamma == nullptr) {
            // scale only (the correlation volume): keep this path minimal -- it is store-bound and every extra instruction
            // per element showed (0.75 -> 0.86 ms per pair when the bias / LayerScale code ran unconditionally)
#pragma unroll
            for (int j = 0; j < 8; ++j)
              sts128(buf + lane * 128 + ((j ^ (lane & 7)) << 4), __uint_as_float(r[4 * j]) * ep.alpha, __uint_as_float(r[4 * j + 1]) * ep.alpha,
                     __uint_as_float(r[4 * j + 2]) * ep.alpha, __uint_as_float(r[4 * j + 3]) * ep.alpha);
          } else {
            const int ncol = n0 + c0;  // column of r[0]; bias / LayerScale: the same addresses in every lane (broadcast loads)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f), g4 = make_float4(1.f, 1.f, 1.f, 1.f);
              if (ncol + 4 * j + 4 <= args.N) {
                if (ep.bias != nullptr) b4 = __ldg(reinterpret_cast<const float4*>(ep.bias + ncol + 4 * j));
                if (ep.gamma != nullptr) g4 = __ldg(reinterpret_cast<const float4*>(ep.gamma + ncol + 4 * j));
              }
              sts128(buf + lane * 128 + ((j ^ (lane & 7)) << 4), fmaf(__uint_as_float(r[4 * j]), ep.alpha, b4.x) * g4.x,
                     fmaf(__uint_as_float(r[4 * j + 1]), ep.alpha, b4.y) * g4.y, fmaf(__uint_as_float(r[4 * j + 2]), ep.alpha, b4.z) * g4.z,
                     fmaf(__uint_as_float(r[4 * j + 3]), ep.alpha, b4.w) * g4.w);
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            if (ep.tma_reduce)
              asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmD)),
                           "r"(buf), "r"(n0 + c0), "r"(m0 + quarter * 32)
                           : "memory");
            else
              asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                               reinterpret_cast<uint64_t>(&tmD)),
                           "r"(buf), "r"(n0 + c0), "r"(m0 + quarter * 32)
                           : "memory");
            tma_store_commit();
          }
          ++st_cnt;
          return;
        }
        if (ep.head_w != nullptr) {
          if (valid) {
            float acc = ep.head_b;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              acc = fmaf(fmaxf(__uint_as_float(r[j]) + __ldg(ep.bias + j), 0.f), __ldg(ep.head_w + j), acc);
            int img = 0, rpix = m;
            if (ep.img_rows > 0) { img = m / ep.img_rows; rpix = m - img * ep.img_rows; }
            const int y = rpix / ep.in_w, x = rpix - y * ep.in_w, pd = ep.pad;
            const size_t pix = ((size_t)img * (ep.in_h - 2 * pd) + (y - pd)) * (ep.in_w - 2 * pd) + (x - pd);
            ep.head_out[pix] = fmaxf(acc, 0.f);
            if (ep.out_f16) {  // also keep the 32 ReLU'd activations (the out_conv hook of the metric head), dense rows
              uint32_t pk[16];
#pragma unroll
              for (int j = 0; j < 16; ++j)
                pk[j] = pack_half2(fmaxf(__uint_as_float(r[2 * j]) + __ldg(ep.bias + 2 * j), 0.f),
                                   fmaxf(__uint_as_float(r[2 * j + 1]) + __ldg(ep.bias + 2 * j + 1), 0.f));
              uint4* dst = reinterpret_cast<uint4*>(ep.out_f16 + pix * ep.out_f16_ld);
#pragma unroll
              for (int j = 0; j < 4; ++j) dst[j] = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
            }
          }
          return;
        }
        // ---- phase 1: row-per-lane registers -> swizzled smem (conflict-free 16 B slots)
        if (SWAP) {
          // the lane holds output column (channel) `lane` of the 32 output rows (pixels) c0 .. c0 + 31: element (row j, column
          // lane) goes to the same swizzled slot the row-per-lane layout uses (32 consecutive words per instruction)
#pragma unroll
          for (int j = 0; j < 32; ++j)
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(stg + j * 128 + ((((lane >> 2) ^ (j & 7))) << 4) + ((lane & 3) << 2)), "r"(r[j]) : "memory");
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j)
            sts128(stg + lane * 128 + ((j ^ (lane & 7)) << 4), __uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]),
                   __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
        }
        __syncwarp();
        // ---- phase 2: 8 lanes x 4 columns cover one row's 32 columns; 4 rows per step -> coalesced global access
        const int n = SWAP ? n0 + quarter * 32 + cg * 4 : n0 + c0 + cg * 4;
        const bool ncol_ok = n < args.N;
        float4 v[8];
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          const int row = rr * 4 + rsub;
          v[rr] = lds128(stg + row * 128 + ((cg ^ (row & 7)) << 4));
        }
        __syncwarp();  // staging may be overwritten by the next chunk from here on
        int col = n;
        if (ep.row_map == ROW_SHUFFLE) {
          const int q = n / ep.shuf_cout;
          col = n - q * ep.shuf_cout;
          const int sdy = q / ep.shuf_s, sdx = q - sdy * ep.shuf_s;
          int drs[8];
#pragma unroll
          for (int rr = 0; rr < 8; ++rr)
            drs[rr] = ib8[rr] + (ty8[rr] * ep.shuf_s + sdy + out_ld) * ep.out_wp + tx8[rr] * ep.shuf_s + sdx + out_ld;
          epilogue_rows8<!TF32 && !TMAST>(ep, v, drs, ncol_ok ? okrows : 0u, bias4, gamma4, col);
        } else {
          epilogue_rows8<!TF32 && !TMAST>(ep, v, dr8, ncol_ok ? okrows : 0u, bias4, gamma4, col);
        }
        if (ep.stat_part != nullptr) {
          float4 sm = make_float4(0.f, 0.f, 0.f, 0.f), sq = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int rr = 0; rr < 8; ++rr)
            if ((okrows >> rr) & 1) {
              sm.x += v[rr].x; sm.y += v[rr].y; sm.z += v[rr].z; sm.w += v[rr].w;
              sq.x = fmaf(v[rr].x, v[rr].x, sq.x); sq.y = fmaf(v[rr].y, v[rr].y, sq.y);
              sq.z = fmaf(v[rr].z, v[rr].z, sq.z); sq.w = fmaf(v[rr].w, v[rr].w, sq.w);
            }
#pragma unroll
          for (int o = 8; o <= 16; o <<= 1) {  // the 4 lanes that hold the same 4 columns (rows rsub, rsub + 4, ...)
            sm.x += __shfl_xor_sync(0xffffffffu, sm.x, o); sm.y += __shfl_xor_sync(0xffffffffu, sm.y, o);
            sm.z += __shfl_xor_sync(0xffffffffu, sm.z, o); sm.w += __shfl_xor_sync(0xffffffffu, sm.w, o);
            sq.x += __shfl_xor_sync(0xffffffffu, sq.x, o); sq.y += __shfl_xor_sync(0xffffffffu, sq.y, o);
            sq.z += __shfl_xor_sync(0xffffffffu, sq.z, o); sq.w += __shfl_xor_sync(0xffffffffu, sq.w, o);
          }
          if (rsub == 0 && ncol_ok) {
            const size_t slab = (size_t)(SWAP ? m0 + c0 : m0 + quarter * 32) >> 5;
            *reinterpret_cast<float4*>(ep.stat_part + (slab * 2) * args.N + n) = sm;
            *reinterpret_cast<float4*>(ep.stat_part + (slab * 2 + 1) * args.N + n) = sq;
          }
        }
      
      };
      if (TF32) {
        // running sums of this warp's chunks live in registers; partial sums arrive every GEMM_TF32_ACC_GROUP K blocks
        constexpr int NCH = (BN + 63) / 64;
        float acc[NCH][32];
#pragma unroll
        for (int i = 0; i < NCH; ++i)
#pragma unroll
          for (int j = 0; j < 32; ++j) acc[i][j] = 0.f;
        const int ngroups = (num_kb + GEMM_TF32_ACC_GROUP - 1) / GEMM_TF32_ACC_GROUP;
        for (int g = 0; g < ngroups; ++g, ++xgi) {
          const int xs = xgi & 1;
          mbar_wait(&tfull[xs], (xgi >> 1) & 1);
          tc_fence_after();
          const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + xs * BN;
#pragma unroll
          for (int i = 0; i < NCH; ++i) {
            const int c0 = chunk_par * 32 + 64 * i;
            if (c0 < bw && n0 + c0 < args.N) {  // warp-uniform
              uint32_t r[32];
              tmem_ld32(taddr + c0, r);
              tmem_ld_wait();
#pragma unroll
              for (int j = 0; j < 32; ++j) acc[i][j] += __uint_as_float(r[j]);
            }
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[xs]);
        }
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int c0 = chunk_par * 32 + 64 * i;
          if (c0 < bw && n0 + c0 < args.N) {
            float4 bias4, gamma4;
            load_bias_gamma(c0, bias4, gamma4);
            uint32_t r[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) r[j] = __float_as_uint(acc[i][j]);
            process_chunk(r, c0, bias4, gamma4);
          }
        }
        continue;  // the TMEM stages were released group by group
      }
      mbar_wait(&tfull[as], aphase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + as * ACC;
      if (SWAP) {
        // this warp: output columns n0 + quarter * 32 .. + 31 (TMEM lanes), alternate 32-pixel chunks (TMEM columns)
#pragma unroll 1
        for (int c0 = chunk_par * 32; c0 < 256; c0 += CSTEP) {
          if (m0 + c0 >= args.M || n0 + quarter * 32 >= args.N) break;  // warp-uniform
          uint32_t r[32];
          tmem_ld32(taddr + c0, r);
          map_rows(m0 + c0);
          float4 bias4, gamma4;
          load_bias_gamma(c0, bias4, gamma4);
          tmem_ld_wait();
          process_chunk(r, c0, bias4, gamma4);
        }
      } else if (TMAST && ep.out_f16 != nullptr) {
        // fp16 destination: a warp takes 64-column blocks (two TMEM chunks) so that every bulk store still moves a
        // 32 x 128-byte box, the same staging layout and swizzle as the fp32 path
#pragma unroll 1
        for (int cb = chunk_par * 64; cb < bw; cb += 128) {
          if (n0 + cb >= args.N) break;  // warp-uniform
          const uint32_t buf = stg + (st_cnt & 1) * 4096;
          if (st_cnt >= 2) { if (lane == 0) tma_store_wait_read<1>(); __syncwarp(); }
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            const int c0 = cb + hf * 32;
            if (c0 < bw && n0 + c0 < args.N) {  // warp-uniform; a missing right half lies beyond N and is clipped by the store
              uint32_t r[32];
              tmem_ld32(taddr + c0, r);
              tmem_ld_wait();
              const int ncol = n0 + c0;  // column of r[0]; every lane holds the same 32 columns of its own row
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                // bias (the same addresses in every lane: one broadcast transaction) + GELU / ReLU in the row-per-lane layout
                float4 ba = make_float4(0.f, 0.f, 0.f, 0.f), bb = ba;
                if (ep.bias != nullptr && ncol + 8 * j + 8 <= args.N) {
                  ba = __ldg(reinterpret_cast<const float4*>(ep.bias + ncol + 8 * j));
                  bb = __ldg(reinterpret_cast<const float4*>(ep.bias + ncol + 8 * j + 4));
                }
                float x[8] = {fmaf(__uint_as_float(r[8 * j]), ep.alpha, ba.x),     fmaf(__uint_as_float(r[8 * j + 1]), ep.alpha, ba.y),
                              fmaf(__uint_as_float(r[8 * j + 2]), ep.alpha, ba.z), fmaf(__uint_as_float(r[8 * j + 3]), ep.alpha, ba.w),
                              fmaf(__uint_as_float(r[8 * j + 4]), ep.alpha, bb.x), fmaf(__uint_as_float(r[8 * j + 5]), ep.alpha, bb.y),
                              fmaf(__uint_as_float(r[8 * j + 6]), ep.alpha, bb.z), fmaf(__uint_as_float(r[8 * j + 7]), ep.alpha, bb.w)};
                if (ep.act == 1) {
#pragma unroll
                  for (int q = 0; q < 8; ++q) x[q] = gelu_erf(x[q]);
                } else if (ep.act == 2) {
#pragma unroll
                  for (int q = 0; q < 8; ++q) x[q] = fmaxf(x[q], 0.f);
                }
                const uint32_t h0 = pack_half2(x[0], x[1]), h1 = pack_half2(x[2], x[3]), h2 = pack_half2(x[4], x[5]), h3 = pack_half2(x[6], x[7]);
                sts128(buf + lane * 128 + (((hf * 4 + j) ^ (lane & 7)) << 4), __uint_as_float(h0), __uint_as_float(h1),
                       __uint_as_float(h2), __uint_as_float(h3));
              }
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                             reinterpret_cast<uint64_t>(&tmD)),
                         "r"(buf), "r"(n0 + cb), "r"(m0 + quarter * 32)
                         : "memory");
            tma_store_commit();
          }
          ++st_cnt;
        }
      } else
#pragma unroll 1
      for (int c0 = chunk_par * 32; c0 < bw; c0 += CSTEP) {
        if (n0 + c0 >= args.N) break;  // warp-uniform
        uint32_t r[32];
        tmem_ld32(taddr + c0, r);
        float4 bias4, gamma4;
        load_bias_gamma(c0, bias4, gamma4);
        tmem_ld_wait();
        process_chunk(r, c0, bias4, gamma4);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { if (CG == 2) mbar_arrive_leader(&tempty[as]); else mbar_arrive(&tempty[as]); }
    }
    if (TMAST && lane == 0) tma_store_wait_all();  // shared memory must outlive the last bulk stores
  }
  __syncwarp();
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();  // no CTA of a pair may exit while the other can still signal it
  if (warp == 1) {
    tc_fence_after();
    if (CG == 2) tmem_dealloc_pair(tmem_base, Cfg::TMEM_COLS); else tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}
#endif  // __CUDACC__

// Host-side prepared launch: tensor maps encoded once, replayed every frame (also inside CUDA graphs).
struct GemmLaunch {
  CUtensorMap tmA, tmB, tmBt;  // tmBt: W with the narrow box of the tail tiles (== tmB when there is no tail)
  CUtensorMap tmD;             // dense output, 32 x 32 boxes (TMA-store epilogue only)
  bool tma_store = false;
  bool tf32 = false;           // kind::tf32 operands (fp32 containers): the 3xTF32 "fp32-class" path of the mask band, with
                               // external fp32 accumulation (GEMM_TF32_ACC_GROUP)
  bool swap = false;           // transposed tiles for N <= 128: 128 output columns x 256 rows per instruction (GemmCfg SWAP)
  GemmArgs args;
  int bn = 128;
  int cg = 1;  // 2 = CTA pairs (cta_group::2), 256 x bn tiles
  int grid = 1;
  double flops = 0;  // algorithmic 2*M*N*K (excluding border/padding waste)
};

// A: fp16 [a_rows][a_cols] with pitch a_pitch (elements);  W: fp16 [w_rows >= round_up(N, bn)][taps*kchunks*64]
int gemm_prepare(GemmLaunch* out, const __half* A, long long a_rows, int a_cols, int a_pitch, const __half* W,
                 int w_rows, int M, int N, int taps, const int* tap_off, const GemmEpilogue& ep, int num_sms,
                 int force_bn = 0);
// 3xTF32: A = fp32 [a_rows][2 * C_half] holding [hi | lo] halves (hi = the top 19 bits of the value, lo = value - hi) of
// which the first C channels enter the product, W = fp32 [w_rows][taps * 3 * C] holding per tap [W_hi | W_hi | W_lo];
// D = sum_t (hi . W_hi + lo . W_hi + hi . W_lo): fp32-class products (the dropped lo . W_lo term is 2^-22 relative), fp32
// accumulate.  Same epilogues.  C, C_half multiples of 32.
int gemm_prepare_tf32x3(GemmLaunch* out, const float* A_split, long long a_rows, int C, int C_half, const float* W3, int w_rows,
                        int M, int N, int taps, const int* tap_off, const GemmEpilogue& ep, int num_sms, int force_bn = 0);
int gemm_run(const GemmLaunch& g, cudaStream_t stream);
int gemm_pick_bn(int M, int N, int num_sms);

}  // namespace prisma
