// prisma_b200 -- RAFT band kernels that are HBM / gather bound (SURVEY.md K11, K13-K15, K20).
#include "flow.cuh"

#include <algorithm>
#include <functional>

#include "pointwise.cuh"

namespace prisma {

// ------------------------------------------------------------------------------------------------
// K11: cv2.resize(frame_u8, None, fx=scale, fy=scale, INTER_CUBIC) -> load_image -> InputPadder('sintel') replicate pad ->
// 2*(x/255)-1 (bands/flow_raft.py:100-101, common/flow.py:13-16,46-56, raft/raft.py:90-91).
// With dsize empty cv::resize keeps inv_scale = fx on BOTH axes (sampling step 1/fx, dsize = cvRound(src*fx)); it does
// not re-derive the step from the rounded output size.  The 8-bit INTER_CUBIC of the reference's OpenCV build (4.13 with
// IPP, which is what `pip install opencv-python` ships and what runs by default) is IPP's float pipeline: the a = -0.75
// cubic evaluated in float32 and rounded half-to-even -- NOT OpenCV's own fixed-point path (2048-scaled short weights),
// which round 1 emulated.  Measured against cv2 on random-noise frames: this kernel differs on ~1e-5 of the bytes, all of
// them exact .5 ties of the real-valued result, where IPP's (closed, CPU-dispatched) operation order decides the
// rounding; tests/test_flow_gpu.py asserts exactly that (every differing byte is a tie, by 1 LSB).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void cv_cubic_coeffs_f(float x, float* f) {  // cv::interpolateCubic, A = -0.75, float32
  const float A = -0.75f;
  const float x1 = __fadd_rn(x, 1.f);
  f[0] = __fsub_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(A, x1), __fmul_rn(5.f, A)), x1), __fmul_rn(8.f, A)), x1), __fmul_rn(4.f, A));
  f[1] = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(A, 2.f), x), __fadd_rn(A, 3.f)), x), x), 1.f);
  const float y = __fsub_rn(1.f, x);
  f[2] = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(__fadd_rn(A, 2.f), y), __fadd_rn(A, 3.f)), y), y), 1.f);
  f[3] = __fsub_rn(__fsub_rn(__fsub_rn(1.f, f[0]), f[1]), f[2]);
}

// one thread per output pixel (3 channels); the 4x4x3 source taps come through L1/L2 (each source byte is reused by
// ~(4/step)^2 = 9 outputs), the output row is written coalesced
__global__ void k_raft_resize(const uint8_t* __restrict__ img, int H, int W, uint8_t* __restrict__ out, int h, int w,
                              double step) {
  const int ox = blockIdx.x * blockDim.x + threadIdx.x;
  const int oy = blockIdx.y;
  if (ox >= w) return;
  const double px = __dsub_rn(__dmul_rn((double)ox + 0.5, step), 0.5), py = __dsub_rn(__dmul_rn((double)oy + 0.5, step), 0.5);
  const int sx = (int)floor(px), sy = (int)floor(py);
  float cx[4], cy[4];
  cv_cubic_coeffs_f((float)(px - (double)sx), cx);
  cv_cubic_coeffs_f((float)(py - (double)sy), cy);
  int xi[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) xi[k] = min(max(sx - 1 + k, 0), W - 1) * 3;
  float hrow[4][3];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint8_t* row = img + (size_t)min(max(sy - 1 + j, 0), H - 1) * W * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      hrow[j][c] = __fadd_rn(__fadd_rn(__fmul_rn((float)row[xi[0] + c], cx[0]), __fmul_rn((float)row[xi[1] + c], cx[1])),
                             __fadd_rn(__fmul_rn((float)row[xi[2] + c], cx[2]), __fmul_rn((float)row[xi[3] + c], cx[3])));
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v = __fadd_rn(__fadd_rn(__fmul_rn(hrow[0][c], cy[0]), __fmul_rn(hrow[1][c], cy[1])),
                              __fadd_rn(__fmul_rn(hrow[2][c], cy[2]), __fmul_rn(hrow[3][c], cy[3])));
    out[((size_t)oy * w + ox) * 3 + c] = (uint8_t)min(max(__float2int_rn(v), 0), 255);
  }
}

__global__ void k_raft_pad_norm(const uint8_t* __restrict__ rs, int h, int w, float* __restrict__ chw, int hp, int wp,
                                int pad_l, int pad_t) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= wp) return;
  const int sx = min(max(x - pad_l, 0), w - 1), sy = min(max(y - pad_t, 0), h - 1);  // replicate
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float v = (float)rs[((size_t)sy * w + sx) * 3 + c];
    chw[((size_t)c * hp + y) * wp + x] = __fsub_rn(__fmul_rn(2.f, __fdiv_rn(v, 255.f)), 1.f);
  }
}

int raft_preprocess(const uint8_t* img, int H, int W, int h, int w, double fx, const int pad[4], uint8_t* resized, float* chw,
                    cudaStream_t s) {
  const double step = 1.0 / fx;  // cv::resize with dsize empty: inv_scale_x = inv_scale_y = fx, sampling step 1 / fx
  dim3 block(128), grid(ceil_div(w, 128), h);
  k_raft_resize<<<grid, block, 0, s>>>(img, H, W, resized, h, w, step);
  const int hp = h + pad[2] + pad[3], wp = w + pad[0] + pad[1];
  dim3 grid2(ceil_div(wp, 128), hp);
  k_raft_pad_norm<<<grid2, block, 0, s>>>(resized, h, w, chw, hp, wp, pad[0], pad[2]);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// K20: process_flow (common/encode.py:113-126): max |flow|, polar HSV encode, truncating u8 cast.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t f2ord_pos(float f) { return __float_as_uint(f); }  // distances are >= 0

__global__ void k_flow_max(const float2* __restrict__ flow, long long n, uint32_t* __restrict__ mx) {
  float hi = 0.f;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float2 f = flow[i];
    hi = fmaxf(hi, __fsqrt_rn(__fadd_rn(__fmul_rn(f.x, f.x), __fmul_rn(f.y, f.y))));
  }
  hi = warp_max(hi);
  if ((threadIdx.x & 31) == 0) atomicMax(mx, f2ord_pos(hi));
}
__global__ void k_zero_u32(uint32_t* p) {
  *p = 0u; }

__device__ __forceinline__ uint8_t polar_channel_u8(float h6f, double off, double rad, double one_minus_rad) {
  double v = fmod(__dadd_rn((double)h6f, off) , 6.0);
  // note: the reference adds the channel offset in f32 (hue*6.0 + 4.0 on an f32 array) before the f64 mod
  v = __dsub_rn(fabs(__dsub_rn(v, 3.0)), 1.0);
  v = fmin(fmax(v, 0.0), 1.0);
  v = __dadd_rn(__dmul_rn(v, rad), one_minus_rad);
  return (uint8_t)(int)__dmul_rn(v, 255.0);
}

__global__ void k_flow_encode(const float2* __restrict__ flow, long long n, const uint32_t* __restrict__ mx,
                              uint8_t* __restrict__ rgb, float* __restrict__ max_out) {
  const float maxd = __uint_as_float(*mx);
  if (blockIdx.x == 0 && threadIdx.x == 0 && max_out) *max_out = maxd;
  const float PI_F = 3.14159274101257324f;  // float32(np.pi)
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    uint8_t* o = rgb + i * 3;
    if (!(maxd > 0.f)) { o[0] = o[1] = o[2] = 0; continue; }  // reference: 0/0 -> NaN -> astype(u8) == 0 on x86
    const float2 f = flow[i];
    const float dX = __fdiv_rn(f.x, maxd), dY = __fdiv_rn(f.y, maxd);
    const float rad = __fsqrt_rn(__fadd_rn(__fmul_rn(dX, dX), __fmul_rn(dY, dY)));
    const float ang = (float)atan2((double)dY, (double)dX);  // correctly rounded f32 arctan2
    const float a = __fmul_rn(__fadd_rn(__fdiv_rn(ang, PI_F), 1.0f), 0.5f);
    const float h6 = __fmul_rn(a, 6.0f);
    const float h6g = __fadd_rn(h6, 4.0f), h6b = __fadd_rn(h6, 2.0f);  // f32 adds, as numpy does on the f32 array
    const double radd = (double)rad, omr = (double)__fsub_rn(1.0f, rad);
    o[0] = polar_channel_u8(h6, 0.0, radd, omr);
    o[1] = polar_channel_u8(h6g, 0.0, radd, omr);
    o[2] = polar_channel_u8(h6b, 0.0, radd, omr);
  }
}

int flow_encode(const float* flow, int H, int W, uint8_t* rgb, uint32_t* mm_scratch, float* max_out, int num_sms,
                cudaStream_t s) {
  const long long n = (long long)H * W;
  k_zero_u32<<<1, 1, 0, s>>>(mm_scratch);
  k_flow_max<<<num_sms * 4, 256, 0, s>>>(reinterpret_cast<const float2*>(flow), n, mm_scratch);
  k_flow_encode<<<num_sms * 8, 256, 0, s>>>(reinterpret_cast<const float2*>(flow), n, mm_scratch, rgb, max_out);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Forward/backward consistency mask (common/flow.py:19-40) and the 16-bit flow PNG packing (common/encode.py:105-110).
// warp_flow = cv2.remap(INTER_LINEAR, BORDER_CONSTANT 0) of a 2-channel f32 image: OpenCV quantises the sampling position
// to 1/32 pixel (cvRound(x*32)), takes the four taps with weights from its float bilinear table ((1-fy/32)(1-fx/32), ...)
// and sums them left to right in f32; reproduced here so the boolean mask is bit-faithful.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 remap_bilinear_c2(const float2* __restrict__ img, int H, int W, float mx, float my) {
  const int sx = __float2int_rn(__fmul_rn(mx, 32.f)), sy = __float2int_rn(__fmul_rn(my, 32.f));
  const int ix = sx >> 5, iy = sy >> 5;
  const float fx = (float)(sx & 31) * (1.f / 32.f), fy = (float)(sy & 31) * (1.f / 32.f);
  const float vx0 = __fsub_rn(1.f, fx), vy0 = __fsub_rn(1.f, fy);
  const float w00 = __fmul_rn(vy0, vx0), w01 = __fmul_rn(vy0, fx), w10 = __fmul_rn(fy, vx0), w11 = __fmul_rn(fy, fx);
  auto at = [&](int y, int x) { return (x >= 0 && x < W && y >= 0 && y < H) ? img[(size_t)y * W + x] : make_float2(0.f, 0.f); };
  const float2 a = at(iy, ix), b = at(iy, ix + 1), c = at(iy + 1, ix), d = at(iy + 1, ix + 1);
  float2 r;
  r.x = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a.x, w00), __fmul_rn(b.x, w01)), __fmul_rn(c.x, w10)), __fmul_rn(d.x, w11));
  r.y = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a.y, w00), __fmul_rn(b.y, w01)), __fmul_rn(c.y, w10)), __fmul_rn(d.y, w11));
  return r;
}
__device__ __forceinline__ float norm2_f32(float x, float y) { return __fsqrt_rn(__fadd_rn(__fmul_rn(x, x), __fmul_rn(y, y))); }

// mask[i] = |f + warp(g, f)| < a1 * (|f| + |warp(g, f)|) + a2     (f = this direction's flow, g = the other one's)
__global__ void k_consistency_mask(const float2* __restrict__ f, const float2* __restrict__ g, int H, int W, float a1,
                                   float a2, uint8_t* __restrict__ mask) {
  const long long total = (long long)H * W;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int y = (int)(i / W), x = (int)(i - (long long)y * W);
    const float2 fl = f[i];
    const float2 w = remap_bilinear_c2(g, H, W, __fadd_rn(fl.x, (float)x), __fadd_rn(fl.y, (float)y));
    const float err = norm2_f32(__fadd_rn(fl.x, w.x), __fadd_rn(fl.y, w.y));
    const float thr = __fadd_rn(__fmul_rn(a1, __fadd_rn(norm2_f32(fl.x, fl.y), norm2_f32(w.x, w.y))), a2);
    mask[i] = err < thr ? 1 : 0;
  }
}
int flow_consistency_masks(const float* fwd, const float* bwd, int H, int W, uint8_t* fwd_mask, uint8_t* bwd_mask,
                           int num_sms, cudaStream_t s) {
  k_consistency_mask<<<num_sms * 8, 256, 0, s>>>(reinterpret_cast<const float2*>(fwd), reinterpret_cast<const float2*>(bwd),
                                                 H, W, 0.05f, 0.5f, fwd_mask);
  k_consistency_mask<<<num_sms * 8, 256, 0, s>>>(reinterpret_cast<const float2*>(bwd), reinterpret_cast<const float2*>(fwd),
                                                 H, W, 0.05f, 0.5f, bwd_mask);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}
// encode_flow: u16 (2^15 + 256 f) per component + validity channel
__global__ void k_flow_u16(const float2* __restrict__ f, const uint8_t* __restrict__ mask, long long n,
                           uint16_t* __restrict__ out) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float fx = __fadd_rn(32768.f, __fmul_rn(f[i].x, 256.f)), fy = __fadd_rn(32768.f, __fmul_rn(f[i].y, 256.f));
    const bool ok = mask[i] && fmaxf(fx, fy) < 65535.f && 0.f < fminf(fx, fy);
    out[i * 3 + 0] = (uint16_t)(int)fx;
    out[i * 3 + 1] = (uint16_t)(int)fy;
    out[i * 3 + 2] = ok ? 65535 : 0;
  }
}
int flow_encode_u16(const float* flow, const uint8_t* mask, int H, int W, uint16_t* out, int num_sms, cudaStream_t s) {
  k_flow_u16<<<num_sms * 8, 256, 0, s>>>(reinterpret_cast<const float2*>(flow), mask, (long long)H * W, out);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// K14 (by linearity): avg_pool2d of the correlation volume over its last two dims == correlation with the
// average-pooled fmap2.  Pool fmap2 (fp16 [P][C]) into the three coarser levels (floor sizes, corr.py:24-27).
// ------------------------------------------------------------------------------------------------
// The pooled features are fp16 like the features themselves (one K-slab).  An fp16 hi/lo pair of the means (two K-slabs: no
// rounding of the means at all) was measured against it: the oracle study (fp16 features, means rounded or not, 12 iterations)
// put the difference at 5e-6 of the largest displacement against a 1e-3 budget, while the second slab made the coarse GEMM
// operand-bound (K = 512 for 128 KB of output).
// One launch pools `frames` feature maps to all three coarse levels: grid.x = cells of level 3, then 2, then 1 (the 8 x 8
// windows, the longest blocks, start first), grid.y = frame.  A thread owns two channels (half2 loads); the sum runs in
// fp32 in raster order of the window.  Level l lands at row coff[l] of the frame's [n123][C] operand.
__global__ void k_pool_fmap(const __half* __restrict__ feat, size_t frame_stride, int W8, int C, __half* __restrict__ out,
                            size_t out_frame_stride, PoolGeom g) {
  int cell = blockIdx.x, lvl = 3;
  if (cell >= g.ln[3]) { cell -= g.ln[3]; lvl = 2; if (cell >= g.ln[2]) { cell -= g.ln[2]; lvl = 1; } }
  const int lw = g.lw[lvl], win = 1 << lvl;
  const int y = cell / lw, x = cell - y * lw;
  const float inv = 1.0f / (float)(win * win);
  const __half* f = feat + blockIdx.y * frame_stride;
  __half* o = out + blockIdx.y * out_frame_stride + (size_t)(g.coff[lvl] + cell) * C;
  for (int c = 2 * threadIdx.x; c < C; c += 2 * blockDim.x) {
    float a0 = 0.f, a1 = 0.f;
    for (int dy = 0; dy < win; ++dy) {
      const __half* row = f + ((size_t)(y * win + dy) * W8 + x * win) * C + c;
#pragma unroll 8
      for (int dx = 0; dx < win; ++dx) {
        const float2 v = __half22float2(*reinterpret_cast<const __half2*>(row + (size_t)dx * C));
        a0 += v.x; a1 += v.y;
      }
    }
    *reinterpret_cast<__half2*>(o + c) = __halves2half2(__float2half_rn(a0 * inv), __float2half_rn(a1 * inv));
  }
}

// ------------------------------------------------------------------------------------------------
// K15: CorrBlock.__call__ (raft/corr.py:29-50) + bilinear_sampler (raft/utils/utils.py:58-72).
// One warp per (image, position).  For pyramid level l the 9x9 window of integer offsets around coords/2^l shares
// one fractional part, so a 10x10 neighbourhood is fetched once: lanes 10g..10g+9 (g = level group) hold one column
// each (10 rows in registers), the right-hand column comes from lane+1 by shuffle.  Channel = l*81 + i*9 + j with
// i moving x and j moving y (the reference's meshgrid quirk), zero outside the volume.
// ------------------------------------------------------------------------------------------------
__global__ void k_corr_lookup(const float* __restrict__ v0, const float* __restrict__ v1, const float* __restrict__ v2,
                              const float* __restrict__ v3, int B, int P, int H8, int W8, int lh0, int lw0, int lp0,
                              int lh1, int lw1, int lp1, int lh2, int lw2, int lp2, int lh3, int lw3, int lp3,
                              const float* __restrict__ coords, __half* __restrict__ out, int out_ld, int out_wp,
                              int out_pad, int out_img_rows) {
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (wid >= B * P) return;
  const int b = wid / P, i = wid - b * P;
  // destination row: dense (b*P + i) or a zero-bordered image (the A operand layout of the motion encoder)
  const size_t orow = out_wp > 0 ? (size_t)b * out_img_rows + (size_t)(i / W8 + out_pad) * out_wp + (i % W8) + out_pad
                                 : (size_t)wid;
  const float cx = coords[((size_t)b * 2 + 0) * P + i], cy = coords[((size_t)b * 2 + 1) * P + i];
  const int grp = lane / 10, col = lane - grp * 10;  // lanes 30,31 idle
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const int lvl = pass == 0 ? grp : 3;
    const bool active = pass == 0 ? (grp < 3) : (grp == 0);
    const float* vol = lvl == 0 ? v0 : (lvl == 1 ? v1 : (lvl == 2 ? v2 : v3));
    const int lh = lvl == 0 ? lh0 : (lvl == 1 ? lh1 : (lvl == 2 ? lh2 : lh3));
    const int lw = lvl == 0 ? lw0 : (lvl == 1 ? lw1 : (lvl == 2 ? lw2 : lw3));
    const int lp = lvl == 0 ? lp0 : (lvl == 1 ? lp1 : (lvl == 2 ? lp2 : lp3));
    const float inv = lvl == 0 ? 1.f : (lvl == 1 ? 0.5f : (lvl == 2 ? 0.25f : 0.125f));
    const float x = cx * inv, y = cy * inv;  // division by 2^l is exact
    const float xf = floorf(x), yf = floorf(y);
    const float wx1 = x - xf, wy1 = y - yf, wx0 = 1.f - wx1, wy0 = 1.f - wy1;
    const int x0 = (int)xf - 4 + col, y0 = (int)yf - 4;
    const float* row = vol + (size_t)wid * lp;
    float v[10];
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const int yy = y0 + r;
      v[r] = (active && x0 >= 0 && x0 < lw && yy >= 0 && yy < lh) ? __ldg(row + (size_t)yy * lw + x0) : 0.f;
    }
    float vn[10];
#pragma unroll
    for (int r = 0; r < 10; ++r) vn[r] = __shfl_down_sync(0xffffffffu, v[r], 1);
    if (active && col < 9) {
      __half* o = out + orow * out_ld + lvl * 81 + col * 9;
#pragma unroll
      for (int j = 0; j < 9; ++j) {
        const float s = wy0 * (wx0 * v[j] + wx1 * vn[j]) + wy1 * (wx0 * v[j + 1] + wx1 * vn[j + 1]);
        o[j] = __float2half_rn(s);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------ FlowCorr
template <typename T>
static int fc_alloc(std::vector<void*>& pool, T** out, size_t n) {
  void* p = nullptr;
  PRISMA_CUDA_OK(cudaMalloc(&p, std::max<size_t>(n * sizeof(T), 256)));
  PRISMA_CUDA_OK(cudaMemset(p, 0, std::max<size_t>(n * sizeof(T), 256)));
  pool.push_back(p);
  *out = reinterpret_cast<T*>(p);
  return 0;
}

FlowCorr::~FlowCorr() {
  cudaSetDevice(device);
  for (void* p : allocs) cudaFree(p);
  if (stream) cudaStreamDestroy(stream);
}

int FlowCorr::init(int dev, int batch, int h8, int w8, int n_frames, const int* f1_idx, const int* f2_idx) {
  device = dev; B = batch; H8 = h8; W8 = w8; P = h8 * w8;
  PRISMA_CHECK(batch >= 1 && batch <= 8 && h8 >= 8 && w8 >= 8, "flowcorr: bad geometry");
  NF = n_frames > 0 ? n_frames : 2 * batch;
  for (int b = 0; b < B; ++b) {
    f1[b] = f1_idx ? f1_idx[b] : b;
    f2[b] = f2_idx ? f2_idx[b] : B + b;
    PRISMA_CHECK(f1[b] >= 0 && f1[b] < NF && f2[b] >= 0 && f2[b] < NF, "flowcorr: frame index out of range");
  }
  PRISMA_CUDA_OK(cudaSetDevice(dev));
  cudaDeviceProp prop;
  PRISMA_CUDA_OK(cudaGetDeviceProperties(&prop, dev));
  PRISMA_CHECK(prop.major == 10, "prisma_b200 kernels are sm_100a only; there is no fallback path");
  num_sms = prop.multiProcessorCount;
  PRISMA_CUDA_OK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  rows_pad = round_up(P, 256);
  PRISMA_TRY(fc_alloc(allocs, &feat, (size_t)NF * rows_pad * C));
  // Levels 1..3 share one operand buffer and one volume: the pooled features of a frame are the rows [coff[l], coff[l] + ln[l])
  // of a [n123][C] matrix, so ONE GEMM per direction writes the three coarse levels side by side into rows of pitch
  // pitch123 (level l = columns coff[l]...).  Two launches per direction instead of four: the coarse levels used to run
  // at 2.8-3.7 TB/s against level 0's 5.1 (short launches, 8-wave ramp each).
  coff[0] = 0;
  for (int l = 0; l < 4; ++l) {
    lh[l] = H8 >> l; lw[l] = W8 >> l; ln[l] = lh[l] * lw[l];
    if (l >= 1) coff[l] = l == 1 ? 0 : coff[l - 1] + round_up(ln[l - 1], 4);
  }
  n123 = coff[3] + ln[3];
  pitch123 = round_up(n123, 4);
  rows123_pad = round_up(pitch123, 256);
  lpitch[0] = round_up(ln[0], 4);
  lrows_pad[0] = rows_pad;
  PRISMA_TRY(fc_alloc(allocs, &pool123, (size_t)NF * rows123_pad * C));
  PRISMA_TRY(fc_alloc(allocs, &vol[0], (size_t)B * P * lpitch[0]));
  PRISMA_TRY(fc_alloc(allocs, &vol123, (size_t)B * P * pitch123));
  for (int l = 1; l < 4; ++l) {
    lpitch[l] = pitch123;
    lrows_pad[l] = rows123_pad;
    pool[l] = pool123 + (size_t)coff[l] * C;
    vol[l] = vol123 + coff[l];
  }
  PRISMA_TRY(fc_alloc(allocs, &coords, (size_t)B * 2 * P));
  PRISMA_TRY(fc_alloc(allocs, &lookup_out, (size_t)B * P * 384));
  // one GEMM per (direction, level): vol_l[b] = feat[f1[b]] . pooled_l(feat[f2[b]])^T / sqrt(C)      (corr.py:53-60)
  const int off[2] = {0, 0};
  bytes_build = flops_build = 0;
  for (int b = 0; b < B; ++b)
    for (int part = 0; part < 2; ++part) {  // part 0: level 0 against the features; part 1: levels 1..3 against the pooled rows
      const int ncols = part == 0 ? lpitch[0] : pitch123;
      GemmEpilogue ep;
      ep.alpha = 1.0f / sqrtf((float)C);
      ep.out_f32 = part == 0 ? vol[0] + (size_t)b * P * lpitch[0] : vol123 + (size_t)b * P * pitch123;
      ep.out_f32_ld = ncols;
      // the volume is store-bound (131 KB per 128 x 256 tile against 4 K-blocks of MMA): leave through TMA bulk stores
      GemmLaunch g;
      ep.tma_store = gemm_pick_bn(P, ncols, num_sms) >= 128;
      const __half* w2 = part == 0 ? feat + (size_t)f2[b] * rows_pad * C : pool123 + (size_t)f2[b] * rows123_pad * C;
      PRISMA_TRY(gemm_prepare(&g, feat + (size_t)f1[b] * rows_pad * C, P, C, C, w2, part == 0 ? rows_pad : rows123_pad, P, ncols, 1,
                              off, ep, num_sms));
      gemms.push_back(g);
    }
  for (int l = 0; l < 4; ++l) {
    flops_build += (double)B * 2.0 * P * (double)ln[l] * C;
    bytes_build += (double)B * 4.0 * P * (double)ln[l];
  }
  bytes_build += 2.0 * B * P * (double)C * 2.0;  // the two fp16 feature maps of every direction, read once
  return 0;
}

int FlowCorr::set_fmaps(const float* fm1, const float* fm2) {
  PRISMA_CHECK(NF == 2 * B, "flowcorr: set_fmaps needs the default frame layout");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  std::vector<__half> h((size_t)B * rows_pad * C, __float2half_rn(0.f));
  for (int which = 0; which < 2; ++which) {
    const float* src = which == 0 ? fm1 : fm2;
    std::fill(h.begin(), h.end(), __float2half_rn(0.f));
    for (int b = 0; b < B; ++b)
      for (int c = 0; c < C; ++c)
        for (int p = 0; p < P; ++p)
          h[((size_t)b * rows_pad + p) * C + c] = __float2half_rn(src[((size_t)b * C + c) * P + p]);
    PRISMA_CUDA_OK(cudaMemcpy(feat + (size_t)which * B * rows_pad * C, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
  }
  return 0;
}

int FlowCorr::pool_frames(int first, int count, cudaStream_t s) {
  PoolGeom g;
  for (int l = 0; l < 4; ++l) { g.lh[l] = lh[l]; g.lw[l] = lw[l]; g.ln[l] = ln[l]; g.coff[l] = coff[l]; }
  k_pool_fmap<<<dim3(ln[1] + ln[2] + ln[3], count), 128, 0, s>>>((const __half*)(feat + (size_t)first * rows_pad * C),
                                                                 (size_t)rows_pad * C, W8, C, pool123 + (size_t)first * rows123_pad * C,
                                                                 (size_t)rows123_pad * C, g);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

int FlowCorr::build_gemms(cudaStream_t s) {
  for (auto& g : gemms) PRISMA_TRY(gemm_run(g, s));
  return 0;
}

int FlowCorr::build(cudaStream_t s) {
  PRISMA_TRY(pool_frames(0, NF, s));
  return build_gemms(s);
}

int FlowCorr::lookup(const float* d_coords, cudaStream_t s) {
  return lookup_to(d_coords, lookup_out, 384, 0, 0, 0, s);
}

int FlowCorr::lookup_to(const float* d_coords, __half* dst, int dst_ld, int dst_wp, int dst_pad, int dst_img_rows,
                        cudaStream_t s) {
  const int warps = B * P;
  k_corr_lookup<<<ceil_div(warps * 32, 256), 256, 0, s>>>(vol[0], vol[1], vol[2], vol[3], B, P, H8, W8, lh[0], lw[0],
                                                          lpitch[0], lh[1], lw[1], lpitch[1], lh[2], lw[2], lpitch[2],
                                                          lh[3], lw[3], lpitch[3], d_coords, dst, dst_ld, dst_wp,
                                                          dst_pad, dst_img_rows);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

static int timed_loop(cudaStream_t s, int iters, float* ms, const std::function<int()>& fn) {
  cudaEvent_t a, b;
  PRISMA_CUDA_OK(cudaEventCreate(&a));
  PRISMA_CUDA_OK(cudaEventCreate(&b));
  PRISMA_TRY(fn());
  PRISMA_CUDA_OK(cudaEventRecord(a, s));
  for (int i = 0; i < iters; ++i) PRISMA_TRY(fn());
  PRISMA_CUDA_OK(cudaEventRecord(b, s));
  PRISMA_CUDA_OK(cudaStreamSynchronize(s));
  float t = 0;
  PRISMA_CUDA_OK(cudaEventElapsedTime(&t, a, b));
  if (ms) *ms = t / std::max(iters, 1);
  cudaEventDestroy(a);
  cudaEventDestroy(b);
  return 0;
}

int FlowCorr::time_build(int iters, float* ms) {
  PRISMA_CUDA_OK(cudaSetDevice(device));
  return timed_loop(stream, iters, ms, [&]() { return build(stream); });
}

int FlowCorr::lookup_host(const float* c, float* out_nchw, int iters, float* ms) {
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_CUDA_OK(cudaMemcpy(coords, c, (size_t)B * 2 * P * 4, cudaMemcpyHostToDevice));
  PRISMA_TRY(timed_loop(stream, iters, ms, [&]() { return lookup(coords, stream); }));
  if (out_nchw) {
    std::vector<__half> h((size_t)B * P * 384);
    PRISMA_CUDA_OK(cudaMemcpy(h.data(), lookup_out, h.size() * 2, cudaMemcpyDeviceToHost));
    for (int b = 0; b < B; ++b)
      for (int k = 0; k < 324; ++k)
        for (int p = 0; p < P; ++p)
          out_nchw[((size_t)b * 324 + k) * P + p] = __half2float(h[((size_t)b * P + p) * 384 + k]);
  }
  return 0;
}

int FlowCorr::read_level(int level, int b, int row0, int nrows, float* out) {
  PRISMA_CHECK(level >= 0 && level < 4 && b >= 0 && b < B && row0 >= 0 && row0 + nrows <= P, "flowcorr: bad range");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_CUDA_OK(cudaMemcpy2D(out, (size_t)ln[level] * 4, vol[level] + ((size_t)b * P + row0) * lpitch[level],
                              (size_t)lpitch[level] * 4, (size_t)ln[level] * 4, nrows, cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace prisma
