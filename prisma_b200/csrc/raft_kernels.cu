// prisma_b200 -- RAFT band: the pointwise / gather kernels around the tcgen05 conv core
// (instance norm, im2col of the 7x7 stem, cnet split, GRU gate algebra, coords update, convex up-sampling).
// Reference: bands/raft/{extractor,update,raft}.py.  All feature maps are NHWC fp16 in the "shared border" layout: `pad`
// zero columns after every row and `pad` zero rows after every image (gemm_tc.cuh GemmEpilogue::lead), so pixel (y, x) of
// image b sits at row (b (H + pad) + y)(W + pad) + x.
#include "raft_kernels.cuh"

namespace prisma {

// ------------------------------------------------------------------------------------------------
// stem im2col: conv1 = Conv2d(3, 64, 7, stride 2, padding 3) (extractor.py:133) on the normalised CHW fp32 image
// -> fp16 [B*Ho*Wo][192], k = (c*7 + ky)*8 + kx (kx = 7 and k >= 168: zero; the engine packs the weights in the same order).
// Stride 2 is applied here, no wasted rows.
// ------------------------------------------------------------------------------------------------
__global__ void k_im2col_stem(const float* __restrict__ x, int B, int H, int W, __half* __restrict__ out) {
  // one thread = one (c, ky) row of one output pixel: 7 consecutive input floats -> a 16-byte store; consecutive threads =
  // consecutive groups, so a warp writes 512 contiguous bytes and its gathers walk the same few image rows
  const int Ho = H / 2, Wo = W / 2;
  const long long total = (long long)B * Ho * Wo * 24;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i % 24);
    const long long pix = i / 24;  // b*Ho*Wo + oy*Wo + ox
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (g < 21) {
      const int b = (int)(pix / ((long long)Ho * Wo));
      const int r = (int)(pix - (long long)b * Ho * Wo);
      const int oy = r / Wo, ox = r - oy * Wo;
      const int c = g / 7, ky = g - c * 7;
      const int iy = oy * 2 - 3 + ky, ix0 = ox * 2 - 3;
      if (iy >= 0 && iy < H) {
        const float* row = x + (((size_t)b * 3 + c) * H + iy) * W;
        if (ix0 >= 0 && ix0 + 6 < W) {
#pragma unroll
          for (int j = 0; j < 7; ++j) v[j] = __ldg(row + ix0 + j);
        } else {
#pragma unroll
          for (int j = 0; j < 7; ++j) if (ix0 + j >= 0 && ix0 + j < W) v[j] = __ldg(row + ix0 + j);
        }
      }
    }
    *reinterpret_cast<uint4*>(out + (size_t)pix * 192 + g * 8) =
        make_uint4(pack_half2(v[0], v[1]), pack_half2(v[2], v[3]), pack_half2(v[4], v[5]), pack_half2(v[6], v[7]));
  }
}
int raft_im2col_stem(const float* x, int B, int H, int W, __half* out, cudaStream_t s) {
  k_im2col_stem<<<148 * 16, 256, 0, s>>>(x, B, H, W, out);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// InstanceNorm2d (no affine, biased variance, eps 1e-5, per image & channel; extractor.py:28-32,129-130):
// deterministic two-stage statistics over a dense fp32 [B][HW][C] conv output, then normalise + ReLU (+ skip) into
// a zero-bordered NHWC fp16 map.
// ------------------------------------------------------------------------------------------------
__global__ void k_in_partial(const float* __restrict__ x, int HW, int C, int rows_per_block, float* __restrict__ part) {
  extern __shared__ float sh[];  // [groups][C][2]
  const int b = blockIdx.y, blk = blockIdx.x;
  const int groups = blockDim.x / C;
  const int g = threadIdx.x / C, c = threadIdx.x - g * C;
  const int r0 = blk * rows_per_block, r1 = min(HW, r0 + rows_per_block);
  float s = 0.f, q = 0.f;
  if (g < groups) {
    const float* p = x + ((size_t)b * HW) * C + c;
    for (int r = r0 + g; r < r1; r += groups) {
      const float v = p[(size_t)r * C];
      s += v;
      q = fmaf(v, v, q);
    }
    sh[(g * C + c) * 2] = s;
    sh[(g * C + c) * 2 + 1] = q;
  }
  __syncthreads();
  if (threadIdx.x < C) {
    float ss = 0.f, qq = 0.f;
    for (int gg = 0; gg < groups; ++gg) { ss += sh[(gg * C + threadIdx.x) * 2]; qq += sh[(gg * C + threadIdx.x) * 2 + 1]; }
    float* o = part + (((size_t)b * gridDim.x + blk) * C + threadIdx.x) * 2;
    o[0] = ss;
    o[1] = qq;
  }
}
__global__ void k_in_final(const float* __restrict__ part, int nblk, int C, int HW, float eps, float* __restrict__ stats) {
  // blockDim.x / C groups of C threads add interleaved stripes of the partial blocks in double, then group 0 adds the groups
  // (fixed order: deterministic)
  __shared__ double shd[512 * 2];
  const int b = blockIdx.x;
  const int groups = blockDim.x / C;
  const int g = threadIdx.x / C, c = threadIdx.x - g * C;
  double s = 0.0, q = 0.0;
  if (g < groups) {
    for (int k = g; k < nblk; k += groups) {
      const float* p = part + (((size_t)b * nblk + k) * C + c) * 2;
      s += p[0];
      q += p[1];
    }
    shd[(g * C + c) * 2] = s;
    shd[(g * C + c) * 2 + 1] = q;
  }
  __syncthreads();
  if (threadIdx.x >= C) return;
  s = 0.0; q = 0.0;
  for (int gg = 0; gg < groups; ++gg) { s += shd[(gg * C + c) * 2]; q += shd[(gg * C + c) * 2 + 1]; }
  const double mean = s / HW;
  const double var = fmax(q / HW - mean * mean, 0.0);
  stats[((size_t)b * C + c) * 2] = (float)mean;
  stats[((size_t)b * C + c) * 2 + 1] = (float)(1.0 / sqrt(var + (double)eps));
}
int instnorm_stats(const float* x, int B, int HW, int C, float* part, float* stats, cudaStream_t s) {
  const int threads = C <= 64 ? 4 * C : 2 * C;
  const int rows_per_block = 512;
  const int nblk = ceil_div(HW, rows_per_block);
  k_in_partial<<<dim3(nblk, B), threads, threads * 2 * sizeof(float), s>>>(x, HW, C, rows_per_block, part);
  k_in_final<<<B, 512, 0, s>>>(part, nblk, C, HW, 1e-5f, stats);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}
// Statistics from the slab partials the conv epilogue wrote (GemmEpilogue::stat_part): image b owns the slabs
// [b * spi, (b + 1) * spi).  Stage 1: nblk blocks per image add stripes of slabs in double (fixed order); stage 2: one
// block per image adds the nblk partial sums and writes (mean, 1 / sqrt(var + eps)).  HW = number of pixels normalised.
__global__ void k_in_slab_stage1(const float* __restrict__ part, int spi, int C, double* __restrict__ part2) {
  extern __shared__ double shd[];  // [groups][C][2]
  const int b = blockIdx.y, blk = blockIdx.x, nblk = gridDim.x;
  const int groups = blockDim.x / C;
  const int g = threadIdx.x / C, c = threadIdx.x - g * C;
  const int s0 = (int)((long long)spi * blk / nblk), s1 = (int)((long long)spi * (blk + 1) / nblk);
  double s = 0.0, q = 0.0;
  if (g < groups) {
    for (int k = s0 + g; k < s1; k += groups) {
      const float* p = part + ((size_t)b * spi + k) * 2 * C;
      s += (double)p[c];
      q += (double)p[C + c];
    }
    shd[(g * C + c) * 2] = s;
    shd[(g * C + c) * 2 + 1] = q;
  }
  __syncthreads();
  if (threadIdx.x < C) {
    double ss = 0.0, qq = 0.0;
    for (int gg = 0; gg < groups; ++gg) { ss += shd[(gg * C + threadIdx.x) * 2]; qq += shd[(gg * C + threadIdx.x) * 2 + 1]; }
    double* o = part2 + (((size_t)b * nblk + blk) * C + threadIdx.x) * 2;
    o[0] = ss;
    o[1] = qq;
  }
}
__global__ void k_in_slab_stage2(const double* __restrict__ part2, int nblk, int C, int HW, float eps, float* __restrict__ stats) {
  const int b = blockIdx.x, c = threadIdx.x;
  if (c >= C) return;
  double s = 0.0, q = 0.0;
  for (int k = 0; k < nblk; ++k) {
    const double* p = part2 + (((size_t)b * nblk + k) * C + c) * 2;
    s += p[0];
    q += p[1];
  }
  const double mean = s / HW;
  const double var = fmax(q / HW - mean * mean, 0.0);
  stats[((size_t)b * C + c) * 2] = (float)mean;
  stats[((size_t)b * C + c) * 2 + 1] = (float)(1.0 / sqrt(var + (double)eps));
}
int instnorm_stats_from_slabs(const float* slab_part, int B, int slabs_per_image, int C, int HW, double* part2, float* stats,
                              cudaStream_t s) {
  const int threads = C <= 64 ? 4 * C : 2 * C, nblk = INSTNORM_STAGE1_BLOCKS;
  k_in_slab_stage1<<<dim3(nblk, B), threads, threads * 2 * sizeof(double), s>>>(slab_part, slabs_per_image, C, part2);
  k_in_slab_stage2<<<B, 128, 0, s>>>(part2, nblk, C, HW, 1e-5f, stats);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}
int instnorm_partial_floats(int B, int HW, int C) { return B * ceil_div(HW, 512) * C * 2; }

// out = relu( skip + relu(norm(x)) )   [skip optional: an fp16 padded map, or a raw fp32 dense map with its own stats]
__global__ void k_in_apply(const float* __restrict__ x, const float* __restrict__ stats, int H, int W, int C,
                           const __half* __restrict__ skip_map, const float* __restrict__ skip_raw,
                           const float* __restrict__ skip_stats, __half* __restrict__ out, int pad, long long img_rows) {
  const int c4 = C >> 2;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_img = (long long)H * W * c4;
  const int b = blockIdx.y;
  if (idx >= per_img) return;
  const int c = (int)(idx % c4) * 4;
  const int px = (int)((idx / c4) % W), py = (int)(idx / ((long long)c4 * W));
  const size_t dense = (((size_t)b * H + py) * W + px) * C + c;
  const int Wp = W + pad;  // shared-border layout: zeros only after each row / image
  const size_t padded = ((size_t)b * img_rows + (size_t)py * Wp + px) * C + c;
  const float4 v = *reinterpret_cast<const float4*>(x + dense);
  const float* st = stats + ((size_t)b * C + c) * 2;
  float y[4] = {fmaxf((v.x - st[0]) * st[1], 0.f), fmaxf((v.y - st[2]) * st[3], 0.f), fmaxf((v.z - st[4]) * st[5], 0.f),
                fmaxf((v.w - st[6]) * st[7], 0.f)};
  if (skip_map) {
    const uint2 r = *reinterpret_cast<const uint2*>(skip_map + padded);
    const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&r.x));
    const float2 bb = __half22float2(*reinterpret_cast<const __half2*>(&r.y));
    y[0] = fmaxf(y[0] + a.x, 0.f); y[1] = fmaxf(y[1] + a.y, 0.f); y[2] = fmaxf(y[2] + bb.x, 0.f); y[3] = fmaxf(y[3] + bb.y, 0.f);
  } else if (skip_raw) {
    const float4 r = *reinterpret_cast<const float4*>(skip_raw + dense);
    const float* s2 = skip_stats + ((size_t)b * C + c) * 2;
    y[0] = fmaxf(y[0] + (r.x - s2[0]) * s2[1], 0.f); y[1] = fmaxf(y[1] + (r.y - s2[2]) * s2[3], 0.f);
    y[2] = fmaxf(y[2] + (r.z - s2[4]) * s2[5], 0.f); y[3] = fmaxf(y[3] + (r.w - s2[6]) * s2[7], 0.f);
  }
  *reinterpret_cast<uint2*>(out + padded) = make_uint2(pack_half2(y[0], y[1]), pack_half2(y[2], y[3]));
}
int instnorm_apply(const float* x, const float* stats, int B, int H, int W, int C, const __half* skip_map,
                   const float* skip_raw, const float* skip_stats, __half* out, int pad, long long img_rows, cudaStream_t s) {
  const long long per_img = (long long)H * W * (C / 4);
  k_in_apply<<<dim3((unsigned)((per_img + 255) / 256), B), 256, 0, s>>>(x, stats, H, W, C, skip_map, skip_raw, skip_stats,
                                                                        out, pad, img_rows);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// cnet output split (raft.py:113-116): net = tanh(cnet[:, :128]) -> h (fp32 master + fp16 operand), inp = relu(rest).
// Destination: the GRU operand maps hx = [h | inp | motion] and rhx = [r*h | inp | motion], 384 channels, pad 2.
// ------------------------------------------------------------------------------------------------
// cn holds the context features per FRAME; direction b reads those of frame df.f[b] (its image1).
__global__ void k_cnet_split(const float* __restrict__ cn, int B, int H, int W, int pad, long long img_rows, DirFrames df,
                             float* __restrict__ h_master, __half* __restrict__ hx, __half* __restrict__ rhx) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // over B*H*W*256
  const long long total = (long long)B * H * W * 256;
  if (idx >= total) return;
  const int c = (int)(idx & 255);
  const long long p = idx >> 8;
  const int b = (int)(p / ((long long)H * W));
  const int r = (int)(p - (long long)b * H * W);
  const int y = r / W, x = r - y * W;
  const int Wp = W + pad;  // shared-border layout: zeros only after each row / image
  const size_t prow = (size_t)b * img_rows + (size_t)y * Wp + x;
  const float v = cn[((size_t)df.f[b] * H * W + r) * 256 + c];
  if (c < 128) {
    const float t = tanhf(v);
    h_master[prow * 128 + c] = t;
    hx[prow * 384 + c] = __float2half_rn(t);
  } else {
    const __half i = __float2half_rn(fmaxf(v, 0.f));
    hx[prow * 384 + c] = i;
    rhx[prow * 384 + c] = i;
  }
}
int raft_cnet_split(const float* cn, int B, int H, int W, int pad, long long img_rows, DirFrames df, float* h_master, __half* hx,
                    __half* rhx, cudaStream_t s) {
  const long long total = (long long)B * H * W * 256;
  k_cnet_split<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(cn, B, H, W, pad, img_rows, df, h_master, hx, rhx);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// convf1 (7x7, 2 -> 128, update.py:84) as a GEMM: im2col of the flow with every fp32 value split into an fp16 pair
// (hi = fp16(v), lo = fp16(v - hi)) so the tensor-core product keeps ~22 bits of the flow (values reach tens of pixels;
// a single fp16 would cost 8e-4 of the 1e-3 budget).  Row = pixel, K = [98 hi | 30 zero | 98 lo | 30 zero].
__global__ void k_flow_im2col(const float* __restrict__ coords0, const float* __restrict__ coords1, int B, int H, int W,
                              __half* __restrict__ out) {
  // one thread = 8 consecutive k of one pixel: two 16-byte stores (hi and lo halves); a warp covers two whole rows
  const int P = H * W;
  const long long total = (long long)B * P * 16;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int g = (int)(i & 15);
    const long long row = i >> 4;
    const int b = (int)(row / P), r = (int)(row - (long long)b * P);
    const int y = r / W, x = r - y * W;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = g * 8 + j;
      v[j] = 0.f;
      if (k < 98) {
        const int ch = k / 49, t = k - ch * 49, ky = t / 7, kx = t - ky * 7;
        const int yy = y + ky - 3, xx = x + kx - 3;
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
          const size_t o = ((size_t)b * 2 + ch) * P + (size_t)yy * W + xx;
          v[j] = coords1[o] - coords0[o];
        }
      }
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const __half h0 = __float2half_rn(v[2 * j]), h1 = __float2half_rn(v[2 * j + 1]);
      hi[j] = pack_half2(__half2float(h0), __half2float(h1));
      lo[j] = pack_half2(v[2 * j] - __half2float(h0), v[2 * j + 1] - __half2float(h1));
    }
    *reinterpret_cast<uint4*>(out + row * 256 + g * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(out + row * 256 + 128 + g * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}
int raft_flow_im2col(const float* coords0, const float* coords1, int B, int H, int W, __half* out, cudaStream_t s) {
  k_flow_im2col<<<148 * 8, 256, 0, s>>>(coords0, coords1, B, H, W, out);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// motion features = cat([conv_out(126), flow(2)]) (update.py:97): the two flow channels of the GRU operand maps
__global__ void k_flow_cols(const float* __restrict__ c0, const float* __restrict__ c1, int B, int H, int W, int pad,
                            long long img_rows, __half* __restrict__ hx, __half* __restrict__ rhx) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P = H * W;
  if (idx >= (long long)B * P) return;
  const int b = (int)(idx / P), r = (int)(idx - (long long)b * P);
  const int y = r / W, x = r - y * W;
  const int Wp = W + pad;  // shared-border layout: zeros only after each row / image
  const size_t prow = (size_t)b * img_rows + (size_t)y * Wp + x;
  const float* a0 = c0 + (size_t)b * 2 * P;
  const float* a1 = c1 + (size_t)b * 2 * P;
  const uint32_t fl = pack_half2(a1[r] - a0[r], a1[(size_t)P + r] - a0[(size_t)P + r]);
  *reinterpret_cast<uint32_t*>(hx + prow * 384 + 382) = fl;
  *reinterpret_cast<uint32_t*>(rhx + prow * 384 + 382) = fl;
}
int raft_flow_cols(const float* c0, const float* c1, int B, int H, int W, int pad, long long img_rows, __half* hx, __half* rhx,
                   cudaStream_t s) {
  k_flow_cols<<<(unsigned)(((long long)B * H * W + 255) / 256), 256, 0, s>>>(c0, c1, B, H, W, pad, img_rows, hx, rhx);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// coords1 += delta_flow (raft.py:133); delta: fp32 padded rows [rows][4] (cols 0,1 used)
__global__ void k_coords_update(const float* __restrict__ delta, int B, int H, int W, int pad, long long img_rows,
                                float* __restrict__ coords1) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P = H * W;
  if (idx >= (long long)B * P) return;
  const int b = (int)(idx / P), r = (int)(idx - (long long)b * P);
  const int y = r / W, x = r - y * W;
  const int Wp = W + pad;  // shared-border layout: zeros only after each row / image
  const size_t prow = (size_t)b * img_rows + (size_t)y * Wp + x;
  coords1[(size_t)b * 2 * P + r] += delta[prow * 4];
  coords1[(size_t)b * 2 * P + P + r] += delta[prow * 4 + 1];
}
int raft_coords_update(const float* delta, int B, int H, int W, int pad, long long img_rows, float* coords1, cudaStream_t s) {
  k_coords_update<<<(unsigned)(((long long)B * H * W + 255) / 256), 256, 0, s>>>(delta, B, H, W, pad, img_rows, coords1);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}
// ------------------------------------------------------------------------------------------------
// FlowHead.conv2 (3x3, 256 -> 2, update.py:19-22) + coords1 += delta_flow (raft.py:133).
// A 3x3 conv with two output channels is no tensor-core shape as such (the narrowest tile wastes 94 % of its columns and
// re-reads the 256-channel map nine times).  It is evaluated as  delta(p) = b + sum_t u_t(p + t),  u_t = W2[t] . x :
// the 18 per-tap, per-output partial products u are ONE 1x1 GEMM (N = 18 -> 32, K = 256 read once, hi/lo fp16 weights =
// exact fp32 weights), and this kernel adds the nine shifted taps per pixel and moves the coordinates.
// u: fp32 [rows][32] in the shared-border row layout (pad rows are zero = the conv's zero padding), column t*2 + o.
// ------------------------------------------------------------------------------------------------
__global__ void k_flow_head2_gather(const float* __restrict__ u, int B, int H, int W, int pad, long long img_rows, float b0,
                                    float b1, float* __restrict__ coords1) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P = H * W, Wp = W + pad;
  if (idx >= (long long)B * P) return;
  const int b = (int)(idx / P), r = (int)(idx - (long long)b * P);
  const int y = r / W, x = r - y * W;
  const long long row0 = (long long)b * img_rows + (long long)y * Wp + x;
  float a0 = b0, a1 = b1;
#pragma unroll
  for (int t = 0; t < 9; ++t) {
    const long long row = row0 + (t / 3 - 1) * Wp + (t % 3 - 1);
    if (row < 0) continue;  // above the first image; every other out-of-image tap reads stored zeros
    const float2 v = *reinterpret_cast<const float2*>(u + row * 32 + t * 2);
    a0 += v.x; a1 += v.y;
  }
  coords1[(size_t)b * 2 * P + r] += a0;
  coords1[(size_t)b * 2 * P + P + r] += a1;
}
int raft_flow_head2_gather(const float* u, int B, int H, int W, int pad, long long img_rows, float b0, float b1, float* coords1,
                           cudaStream_t s) {
  k_flow_head2_gather<<<(unsigned)(((long long)B * H * W + 255) / 256), 256, 0, s>>>(u, B, H, W, pad, img_rows, b0, b1, coords1);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

__global__ void k_coords_init(float* __restrict__ c0, float* __restrict__ c1, int B, int H, int W) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int P = H * W;
  if (idx >= (long long)B * P) return;
  const int b = (int)(idx / P), r = (int)(idx - (long long)b * P);
  const float x = (float)(r % W), y = (float)(r / W);
  c0[(size_t)b * 2 * P + r] = x; c0[(size_t)b * 2 * P + P + r] = y;
  c1[(size_t)b * 2 * P + r] = x; c1[(size_t)b * 2 * P + P + r] = y;
}
int raft_coords_init(float* c0, float* c1, int B, int H, int W, cudaStream_t s) {
  k_coords_init<<<(unsigned)(((long long)B * H * W + 255) / 256), 256, 0, s>>>(c0, c1, B, H, W);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Convex up-sampling (raft.py:73-84) fused with InputPadder.unpad and the HWC permute of flow_raft.py:58-61:
// out[b][Y][X][ch] for the un-padded Hs x Ws image; Y = 8y+a - pad_top, X = 8x+b - pad_left.
// mask: fp32 padded rows [rows][576] (already scaled by 0.25), channel k*64 + a*8 + b, softmax over k = 0..8;
// neighbourhood = unfold(8*flow, 3x3, padding 1) (zero outside).
// ------------------------------------------------------------------------------------------------
__global__ void k_convex_upsample(const float* __restrict__ mask, const float* __restrict__ c0,
                                  const float* __restrict__ c1, int B, int H, int W, int pad, long long img_rows, int Hs,
                                  int Ws, int pad_top, int pad_left, float* __restrict__ out) {
  const int b = blockIdx.y;
  const int r = blockIdx.x;  // coarse pixel
  const int y = r / W, x = r - y * W;
  const int sub = threadIdx.x;  // 0..63: a*8 + bcol
  const int P = H * W;
  const int Wp = W + pad;  // shared-border layout: zeros only after each row / image
  const float* m = mask + ((size_t)b * img_rows + (size_t)y * Wp + x) * 576;
  float w[9];
  float mx = -INFINITY;
#pragma unroll
  for (int k = 0; k < 9; ++k) { w[k] = m[k * 64 + sub]; mx = fmaxf(mx, w[k]); }
  float den = 0.f;
#pragma unroll
  for (int k = 0; k < 9; ++k) { w[k] = expf(w[k] - mx); den += w[k]; }
  float fx = 0.f, fy = 0.f;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const int yy = y + k / 3 - 1, xx = x + k % 3 - 1;
    if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
      const int rr = yy * W + xx;
      const float wk = w[k] / den;
      fx += wk * 8.f * (c1[(size_t)b * 2 * P + rr] - c0[(size_t)b * 2 * P + rr]);
      fy += wk * 8.f * (c1[(size_t)b * 2 * P + P + rr] - c0[(size_t)b * 2 * P + P + rr]);
    }
  }
  const int Y = 8 * y + (sub >> 3) - pad_top, X = 8 * x + (sub & 7) - pad_left;
  if (Y >= 0 && Y < Hs && X >= 0 && X < Ws) {
    float* o = out + (((size_t)b * Hs + Y) * Ws + X) * 2;
    o[0] = fx;
    o[1] = fy;
  }
}
int raft_convex_upsample(const float* mask, const float* c0, const float* c1, int B, int H, int W, int pad, long long img_rows,
                         int Hs, int Ws, int pad_top, int pad_left, float* out, cudaStream_t s) {
  k_convex_upsample<<<dim3(H * W, B), 64, 0, s>>>(mask, c0, c1, B, H, W, pad, img_rows, Hs, Ws, pad_top, pad_left, out);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace prisma
