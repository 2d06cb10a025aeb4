// prisma_b200 -- ViT self-attention on tcgen05 (sm_100a): softmax(q k^T) v, non-causal, head_dim 64
// (dinov2/layers/attention.py:49-62; the 1/sqrt(64) scale is folded into the q rows of the qkv weights, exactly).
//
// One CTA per (128-query tile, head, image); 2 CTAs co-reside per SM so one CTA's softmax overlaps the other's MMAs.
//   warp 0   : TMA producer  (Q once; K/V 128x64 fp16 tiles in a 2-stage ring, 128B swizzle, straight out of the
//                             [tokens][3*D] qkv matrix -- no head split/transposes ever materialise)
//   warp 1   : MMA issuer    (S = Q K^T  -> TMEM cols [0,128);  O += P V -> TMEM cols [128,192): A = P read from TMEM
//                             cols [192,256) (fp16 pairs written there by the softmax warps with tcgen05.st), B = V
//                             from smem as an MN-major operand.  P never goes through shared memory.)
//   warps 2-5: softmax       (thread = ONE query row = one TMEM lane: the 128 scores of the tile sit in 128 registers, so
//                             nothing is exchanged between threads and there is no barrier inside a tile).
// The exp pipe (MUFU, 16 ex2 / clk / SM) bounds this kernel; a softmax warp is in-order and only two of them share a
// scheduler, so the tile loop is written for instruction-level parallelism inside one warp:
//   * row max by four FMNMX3 chains over the 128 registers (no exchange, no barrier); O and l are rescaled lazily, only when a
//     row's max grew by more than 2^8 since the value they are scaled by (p stays <= 256 in fp16);
//   * the exps of a 32-key chunk are computed IN PLACE, all 32 FFMA + MUFU.EX2 issued before the first sum / pack consumes
//     a result, so the warp does not stall on the MUFU latency;
//   * warps whose 32 query rows all lie beyond the last token (last q tile) take no part, and the columns of the last KV tile
//     beyond the last key are zero-filled in 32-column chunks without touching the exp pipe.
#include "attention.cuh"

namespace prisma {

constexpr int ATT_BQ = 128, ATT_BKV = 128, ATT_HD = 64;
constexpr int ATT_THREADS = 192;  // TMA warp + MMA warp + 4 softmax warps (one per TMEM lane quarter)
constexpr int ATT_SOFTMAX_WARPS = 4;
constexpr int ATT_TILE_BYTES = 128 * 64 * 2;  // 16 KB
// Q + 2 x (K, V) + barriers = 82,048 B: two CTAs (+1 KB reserved each) fit the 228 KB of an SM; no alignment slack, the
// dynamic smem base is declared 1024-aligned (128B-swizzle atoms are 1 KB) and checked at kernel entry.
constexpr int ATT_SMEM = ATT_TILE_BYTES * (1 + 2 + 2) + 128 /*barriers*/;

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// Every exp2 of the softmax runs on the MUFU pipe.  Measured against moving a fraction of the elements to the FMA / ALU pipes
// (Cody-Waite split x = n + f, 2^f by a degree-3 minimax polynomial, 2^n by adding n to the exponent field; B200, 2443 tokens,
// 192 heads): none 643 TFLOP/s, every 4th element 636, every 3rd 619, every 2nd 550 -- with two in-order softmax warps per
// scheduler the kernel is bound by issue slots and dependency latency, not by the exp pipe's 16 / clk, so nine instructions
// instead of two per element lose.

// 32 scores -> 32 probabilities, in place; fp16 pairs to pk[16], their sum to four partial sums.  nvalid < 32: the rest are 0.
template <bool PARTIAL>
__device__ __forceinline__ void att_exp_chunk(uint32_t* v, float mscaled, int nvalid, uint32_t* pk, float& s0, float& s1, float& s2,
                                              float& s3) {
  const float LOG2E = 1.4426950408889634f;
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(fmaf(__uint_as_float(v[i]), LOG2E, -mscaled));
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(ex2_approx(__uint_as_float(v[i])));
  if (PARTIAL) {
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = (i < nvalid) ? v[i] : 0u;
  }
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const uint32_t* e = v + c * 8;
    s0 += __uint_as_float(e[0]) + __uint_as_float(e[4]); s1 += __uint_as_float(e[1]) + __uint_as_float(e[5]);
    s2 += __uint_as_float(e[2]) + __uint_as_float(e[6]); s3 += __uint_as_float(e[3]) + __uint_as_float(e[7]);
    pk[c * 4 + 0] = pack_half2(__uint_as_float(e[0]), __uint_as_float(e[1])); pk[c * 4 + 1] = pack_half2(__uint_as_float(e[2]), __uint_as_float(e[3]));
    pk[c * 4 + 2] = pack_half2(__uint_as_float(e[4]), __uint_as_float(e[5])); pk[c * 4 + 3] = pack_half2(__uint_as_float(e[6]), __uint_as_float(e[7]));
  }
}

// A full tile (128 valid keys): the same arithmetic as four att_exp_chunk<false> calls, software-pipelined across the chunks --
// the MUFU.EX2 of chunk c + 1 are issued interleaved with the sums / packs of chunk c, so an in-order warp never waits on the
// exp it has just issued (only two softmax warps share a scheduler: there is nobody else to hide that latency).
__device__ __forceinline__ void att_exp_tile(uint32_t* v, float mscaled, uint32_t tmem_p_row, float& s0, float& s1, float& s2,
                                             float& s3) {
  const float LOG2E = 1.4426950408889634f;
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(ex2_approx(fmaf(__uint_as_float(v[i]), LOG2E, -mscaled)));
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    uint32_t* e = v + c * 32;
    uint32_t* nx = v + (c + 1) * 32;
    if (c + 1 < 4) {
#pragma unroll
      for (int i = 0; i < 32; ++i) nx[i] = __float_as_uint(fmaf(__uint_as_float(nx[i]), LOG2E, -mscaled));
    }
    uint32_t pk[16];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      if (c + 1 < 4) {
#pragma unroll
        for (int i = 0; i < 8; ++i) nx[g * 8 + i] = __float_as_uint(ex2_approx(__uint_as_float(nx[g * 8 + i])));
      }
      const uint32_t* q = e + g * 8;
      s0 += __uint_as_float(q[0]) + __uint_as_float(q[4]); s1 += __uint_as_float(q[1]) + __uint_as_float(q[5]);
      s2 += __uint_as_float(q[2]) + __uint_as_float(q[6]); s3 += __uint_as_float(q[3]) + __uint_as_float(q[7]);
      pk[g * 4 + 0] = pack_half2(__uint_as_float(q[0]), __uint_as_float(q[1])); pk[g * 4 + 1] = pack_half2(__uint_as_float(q[2]), __uint_as_float(q[3]));
      pk[g * 4 + 2] = pack_half2(__uint_as_float(q[4]), __uint_as_float(q[5])); pk[g * 4 + 3] = pack_half2(__uint_as_float(q[6]), __uint_as_float(q[7]));
    }
    tmem_st16(tmem_p_row + c * 16, pk);
  }
}

__global__ void __launch_bounds__(ATT_THREADS, 2)
attention_kernel(const __grid_constant__ CUtensorMap tmQKV, const __grid_constant__ AttnArgs args) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) {
    if (threadIdx.x == 0) printf("prisma: attention smem base not 1024-aligned\n");
    __trap();
  }
  uint8_t* sQ = smem;
  uint8_t* sK = smem + ATT_TILE_BYTES;      // 2 stages
  uint8_t* sV = smem + 3 * ATT_TILE_BYTES;  // 2 stages
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 5 * ATT_TILE_BYTES);
  uint64_t* q_full = bars + 0;
  uint64_t* kv_full = bars + 1;   // [2]
  uint64_t* kv_empty = bars + 3;  // [2]
  uint64_t* s_full = bars + 5;
  uint64_t* p_full = bars + 6;
  uint64_t* pv_done = bars + 7;
  uint64_t* s_free = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int T = args.tokens, D = args.D;
  const int q0 = blockIdx.x * ATT_BQ;
  const int head = blockIdx.y;
  const int row_base = blockIdx.z * T;  // first row of this image in the qkv matrix
  const int n_kv = (T + ATT_BKV - 1) / ATT_BKV;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmQKV);
    mbar_init(q_full, 1);
    for (int s = 0; s < 2; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1); }
    mbar_init(s_full, 1);
    // softmax warps whose 32 rows all lie beyond the last token take no part (last q tile of an image)
    const int n_live = min(ATT_SOFTMAX_WARPS, (args.tokens - blockIdx.x * ATT_BQ + 31) / 32);
    mbar_init(p_full, n_live);
    mbar_init(pv_done, 1);
    mbar_init(s_free, n_live);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmem_S = tmem_base;
  const uint32_t tmem_O = tmem_base + 128;
  const uint32_t tmem_P = tmem_base + 192;  // P as packed fp16 pairs: 64 columns = 128 keys

  if (warp == 0) {
    if (lane == 0) {
      mbar_arrive_expect_tx(q_full, ATT_TILE_BYTES);
      tma_load_2d(sQ, &tmQKV, q_full, head * ATT_HD, row_base + q0);
      for (int j = 0; j < n_kv; ++j) {
        const int st = j & 1;
        mbar_wait(&kv_empty[st], ((j >> 1) & 1) ^ 1);
        mbar_arrive_expect_tx(&kv_full[st], 2 * ATT_TILE_BYTES);
        tma_load_2d(sK + st * ATT_TILE_BYTES, &tmQKV, &kv_full[st], D + head * ATT_HD, row_base + j * ATT_BKV);
        tma_load_2d(sV + st * ATT_TILE_BYTES, &tmQKV, &kv_full[st], 2 * D + head * ATT_HD, row_base + j * ATT_BKV);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      constexpr uint32_t idesc_s = make_idesc_f16(128, 128, 0, 0);
      constexpr uint32_t idesc_o = make_idesc_f16(128, 64, 0, 1);  // B (= V) is MN-major
      const uint64_t qdesc = make_sdesc_sw128(smem_u32(sQ));
      mbar_wait(q_full, 0);
      mbar_wait(&kv_full[0], 0);
      tc_fence_after();
      {
        const uint64_t kdesc = make_sdesc_sw128(smem_u32(sK));
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16(tmem_S, qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
        umma_commit(s_full);
      }
      for (int j = 0; j < n_kv; ++j) {
        const int st = j & 1;
        if (j + 1 < n_kv) {
          // S(j+1) as soon as the softmax warps hold S(j) in registers: it overlaps the whole softmax of tile j
          const int st1 = (j + 1) & 1;
          mbar_wait(s_free, j & 1);
          mbar_wait(&kv_full[st1], ((j + 1) >> 1) & 1);
          tc_fence_after();
          const uint64_t kdesc = make_sdesc_sw128(smem_u32(sK + st1 * ATT_TILE_BYTES));
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16(tmem_S, qdesc + 2 * k, kdesc + 2 * k, idesc_s, k != 0);
          umma_commit(s_full);
        }
        mbar_wait(p_full, j & 1);  // P(j) in TMEM, any rescale of O done
        tc_fence_after();
        const uint32_t vbase = smem_u32(sV + st * ATT_TILE_BYTES);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const uint64_t vdesc = make_sdesc_sw128(vbase + k * 2048);
          umma_f16_ts(tmem_O, tmem_P + k * 8, vdesc, idesc_o, (j | k) != 0);  // A = P from TMEM; O accumulates over all tiles
        }
        umma_commit(pv_done);
        umma_commit(&kv_empty[st]);
      }
    }
  } else {
    const int quarter = warp & 3;         // TMEM lane quarter this warp may access
    const int r = quarter * 32 + lane;    // query row inside the tile == TMEM lane
    const uint32_t lane_sel = static_cast<uint32_t>(quarter * 32) << 16;
    const bool warp_live = q0 + quarter * 32 < T;  // warp-uniform: at least one of my 32 rows is a real query
    const float LOG2E = 1.4426950408889634f;
    float m_used = -INFINITY, l_sum = 0.f;  // m_used: the max P / O are currently scaled by
#ifdef PRISMA_ATTN_PROFILE
    long long t_wait = 0, t_ld = 0, t_max = 0, t_exp = 0, t_st = 0, t_slow = 0, n_slow = 0, t_tot = clock64();
    const bool prof = args.dbg != nullptr && threadIdx.x == 64 && blockIdx.x == 1 && blockIdx.y == 1;
#define ATT_CLK(x) long long x = clock64()
#else
#define ATT_CLK(x)
#endif

    for (int j = 0; warp_live && j < n_kv; ++j) {  // dead warps (rows beyond the last token) are not counted by the barriers
      ATT_CLK(c0_);
      mbar_wait(s_full, j & 1);
      tc_fence_after();
      ATT_CLK(c1_);
      const int valid = min(ATT_BKV, T - j * ATT_BKV);  // valid key columns of this tile (1..128)
      // ---- the whole S row (128 fp32) into registers with one wait; then the TMEM buffer is free for S(j+1)
      uint32_t v[128];
      tmem_ld32(tmem_S + lane_sel, v);
      tmem_ld32(tmem_S + lane_sel + 32, v + 32);
      tmem_ld32(tmem_S + lane_sel + 64, v + 64);
      tmem_ld32(tmem_S + lane_sel + 96, v + 96);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(s_free);
      ATT_CLK(c2_);

      // ---- row max (thread-local), lazy rescale of O and l
      float mx;
      if (valid == ATT_BKV) {  // eight FMNMX3 chains of 8 (short dependent chains: the warp is in-order)
        float m[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) m[c] = fmax3(__uint_as_float(v[c * 16]), __uint_as_float(v[c * 16 + 1]), __uint_as_float(v[c * 16 + 2]));
#pragma unroll
        for (int k = 3; k < 15; k += 2)
#pragma unroll
          for (int c = 0; c < 8; ++c) m[c] = fmax3(m[c], __uint_as_float(v[c * 16 + k]), __uint_as_float(v[c * 16 + k + 1]));
#pragma unroll
        for (int c = 0; c < 8; ++c) m[c] = fmaxf(m[c], __uint_as_float(v[c * 16 + 15]));
        mx = fmaxf(fmax3(m[0], m[1], m[2]), fmax3(m[3], m[4], fmax3(m[5], m[6], m[7])));
      } else {
        mx = -INFINITY;
#pragma unroll
        for (int i = 0; i < 128; ++i) if (i < valid) mx = fmaxf(mx, __uint_as_float(v[i]));
      }
      mx = fmaxf(mx, -60000.f);  // a row of -inf scores must not produce inf - inf
      bool pv_waited = (j == 0);
      if (j == 0) {
        m_used = mx;
      } else {
        const bool need = (mx - m_used) * LOG2E > 8.0f;
        if (__any_sync(0xffffffffu, need)) {
          ATT_CLK(cs0_);
          const float m_new = need ? mx : m_used;
          const float alpha = ex2_approx((m_used - m_new) * LOG2E);  // 1 for rows that keep their max
          mbar_wait(pv_done, (j - 1) & 1);                            // no PV may be in flight on O
          tc_fence_after();
          pv_waited = true;
#pragma unroll 1
          for (int hh = 0; hh < 4; ++hh) {  // 16 columns at a time: the S row stays in registers
            uint32_t o[16];
            tmem_ld16(tmem_O + lane_sel + hh * 16, o);
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; ++i) o[i] = __float_as_uint(__uint_as_float(o[i]) * alpha);
            tmem_st16(tmem_O + lane_sel + hh * 16, o);
          }
          tmem_st_wait();
          l_sum *= alpha;
          m_used = m_new;
#ifdef PRISMA_ATTN_PROFILE
          t_slow += clock64() - cs0_; ++n_slow;
#endif
        }
      }
      ATT_CLK(c2b_);
      // ---- p = exp(s - m_used) in four chunks of 32 keys -> 16 packed fp16 pairs -> 16 TMEM columns each
      const float mscaled = m_used * LOG2E;
      float sum0 = 0.f, sum1 = 0.f, sum2 = 0.f, sum3 = 0.f;
      // P(j-1) must have been consumed by PV(j-1) before the buffer is rewritten (issued a whole softmax ago: no wait in practice)
      if (!pv_waited) { mbar_wait(pv_done, (j - 1) & 1); tc_fence_after(); }
      if (valid == ATT_BKV) {
        att_exp_tile(v, mscaled, tmem_P + lane_sel, sum0, sum1, sum2, sum3);
      } else {
#pragma unroll
        for (int hh = 0; hh < 4; ++hh) {
          const int nv = valid - hh * 32;  // valid columns of this chunk (warp-uniform)
          if (nv >= 32) {
            uint32_t pk[16];
            att_exp_chunk<false>(v + hh * 32, mscaled, 32, pk, sum0, sum1, sum2, sum3);
            tmem_st16(tmem_P + lane_sel + hh * 16, pk);
          } else if (nv > 0) {
            uint32_t pk[16];
            att_exp_chunk<true>(v + hh * 32, mscaled, nv, pk, sum0, sum1, sum2, sum3);
            tmem_st16(tmem_P + lane_sel + hh * 16, pk);
          } else {
            uint32_t pk[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) pk[i] = 0u;
            tmem_st16(tmem_P + lane_sel + hh * 16, pk);
          }
        }
      }
      const float tsum = (sum0 + sum1) + (sum2 + sum3);
      l_sum += tsum;
      ATT_CLK(c3_);
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
#ifdef PRISMA_ATTN_PROFILE
      long long c4_ = clock64();
      t_wait += c1_ - c0_; t_ld += c2_ - c1_; t_max += c2b_ - c2_; t_exp += c3_ - c2b_; t_st += c4_ - c3_;
#endif
    }
#ifdef PRISMA_ATTN_PROFILE
    if (prof) { args.dbg[0] = t_wait; args.dbg[1] = t_ld; args.dbg[2] = t_exp; args.dbg[3] = clock64() - t_tot; args.dbg[4] = n_kv;
                args.dbg[5] = t_st; args.dbg[6] = t_slow; args.dbg[7] = n_slow; args.dbg[8] = t_max; }
#endif
    if (warp_live) {
      // ---- O is complete once the last PV retires: normalise and store my row, out[row][head*64 + d]
      mbar_wait(pv_done, (n_kv - 1) & 1);
      tc_fence_after();
      const float inv = 1.0f / l_sum;
      const int q = q0 + r;
#pragma unroll 1
      for (int hh = 0; hh < 2; ++hh) {
        uint32_t ov[32];
        tmem_ld32(tmem_O + lane_sel + hh * 32, ov);
        tmem_ld_wait();
        if (q < T) {
          __half* dst = args.out + (size_t)(row_base + q) * args.out_ld + head * ATT_HD + hh * 32;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint4 o;
            o.x = pack_half2(__uint_as_float(ov[g * 8 + 0]) * inv, __uint_as_float(ov[g * 8 + 1]) * inv);
            o.y = pack_half2(__uint_as_float(ov[g * 8 + 2]) * inv, __uint_as_float(ov[g * 8 + 3]) * inv);
            o.z = pack_half2(__uint_as_float(ov[g * 8 + 4]) * inv, __uint_as_float(ov[g * 8 + 5]) * inv);
            o.w = pack_half2(__uint_as_float(ov[g * 8 + 6]) * inv, __uint_as_float(ov[g * 8 + 7]) * inv);
            *reinterpret_cast<uint4*>(dst + g * 8) = o;
          }
        }
      }
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
}

int attention_prepare(AttnLaunch* out, const __half* qkv, __half* o, int batch, int tokens, int heads, int D) {
  PRISMA_CHECK(D == heads * ATT_HD, "attention: head_dim must be 64");
  out->args.tokens = tokens;
  out->args.heads = heads;
  out->args.D = D;
  out->args.batch = batch;
  out->args.out = o;
  out->args.out_ld = D;
  out->args.dbg = nullptr;
  PRISMA_TRY(make_tmap_2d_f16(&out->tm, qkv, (uint64_t)3 * D, (uint64_t)batch * tokens, (uint64_t)3 * D, 64, 128));
  out->grid = dim3(ceil_div(tokens, ATT_BQ), heads, batch);
  out->flops = 4.0 * batch * heads * (double)tokens * tokens * ATT_HD;
  return 0;
}

int attention_run(const AttnLaunch& a, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    PRISMA_CUDA_OK(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
    attr_set = true;
  }
  attention_kernel<<<a.grid, ATT_THREADS, ATT_SMEM, s>>>(a.tm, a.args);
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace prisma
