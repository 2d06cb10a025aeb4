// prisma_b200 -- host side of the tcgen05 shifted-row GEMM: TMA descriptor encode, tile-shape choice, launch.
#include "gemm_tc.cuh"

#include <mutex>

#include <nvtx3/nvToolsExt.h>

namespace prisma {

NvtxRange::NvtxRange(const char* name) { nvtxRangePushA(name); }
NvtxRange::~NvtxRange() { nvtxRangePop(); }

static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }
const char* get_last_error() { return g_last_error.c_str(); }

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
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

int make_tmap_2d_f16(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t pitch_elems,
                     uint32_t box_cols, uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  PRISMA_CHECK(fn != nullptr, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  PRISMA_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA base must be 16-byte aligned");
  PRISMA_CHECK((pitch_elems * 2) % 16 == 0, "TMA row pitch must be a multiple of 16 bytes");
  PRISMA_CHECK(box_cols * 2 == 128 && box_rows >= 1 && box_rows <= 256, "TMA box must be 64 fp16 wide, <=256 rows");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {pitch_elems * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PRISMA_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (code " + std::to_string((int)r) + ")");
  return 0;
}

int make_tmap_2d_f32(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t pitch_elems,
                     uint32_t box_cols, uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  PRISMA_CHECK(fn != nullptr, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  PRISMA_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA base must be 16-byte aligned");
  PRISMA_CHECK((pitch_elems * 4) % 16 == 0, "TMA row pitch must be a multiple of 16 bytes");
  PRISMA_CHECK(box_cols * 4 == 128 && box_rows >= 1 && box_rows <= 256, "TMA box must be 32 fp32 wide, <=256 rows");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {pitch_elems * 4};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PRISMA_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (fp32) failed (code " + std::to_string((int)r) + ")");
  return 0;
}

// fp16 destination of the TMA-store epilogue: boxes of 32 rows x 64 columns (128-byte rows), 128-byte swizzle
static int make_tmap_2d_f16_store(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t pitch_elems) {
  EncodeTiledFn fn = get_encode_fn();
  PRISMA_CHECK(fn != nullptr, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  PRISMA_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "TMA base must be 16-byte aligned");
  PRISMA_CHECK((pitch_elems * 2) % 16 == 0, "TMA row pitch must be a multiple of 16 bytes");
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {pitch_elems * 2};
  cuuint32_t box[2] = {64, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  PRISMA_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (fp16 store) failed (code " + std::to_string((int)r) + ")");
  return 0;
}

// Tile-N choice: minimise waves x per-tile time.  Per-tile costs are MEASURED on B200 (8192^3 sweep, relative units
// per 64-wide K block): the 128x256 tile runs at 1351 TF/s, 128x128 at 919 TF/s (L2->SM operand traffic per MMA is
// 1.5x higher), narrower tiles are smem-read bound; plus a per-tile constant for the drain / epilogue hand-off.
int gemm_pick_bn(int M, int N, int num_sms) {
  const int cands[4] = {256, 128, 64, 32};
  const double tile_cost[4] = {128.0, 94.0, 62.0, 45.0};
  int best = 128;
  double best_cost = 1e30;
  const int tiles_m = ceil_div(M, GEMM_BM);
  for (int i = 0; i < 4; ++i) {
    const int bn = cands[i];
    if (bn > 32 && bn >= 2 * round_up(N, 32)) continue;  // mostly padding
    const int tiles = tiles_m * ceil_div(N, bn);
    const int waves = ceil_div(tiles, num_sms);
    const double cost = waves * (tile_cost[i] + 6.0);
    if (cost < best_cost) { best_cost = cost; best = bn; }
  }
  return best;
}

static int gemm_prepare_impl(GemmLaunch* out, const void* A, long long a_rows, int a_cols, int a_pitch, const void* W,
                             int w_rows, int M, int N, int taps, const int* tap_off, const int* tap_acol, const GemmEpilogue& ep,
                             int num_sms, int force_bn, bool tf32);

int gemm_prepare(GemmLaunch* out, const __half* A, long long a_rows, int a_cols, int a_pitch, const __half* W,
                 int w_rows, int M, int N, int taps, const int* tap_off, const GemmEpilogue& ep, int num_sms,
                 int force_bn) {
  return gemm_prepare_impl(out, A, a_rows, a_cols, a_pitch, W, w_rows, M, N, taps, tap_off, nullptr, ep, num_sms, force_bn, false);
}

int gemm_prepare_tf32x3(GemmLaunch* out, const float* A_split, long long a_rows, int C, int C_half, const float* W3, int w_rows,
                        int M, int N, int taps, const int* tap_off, const GemmEpilogue& ep, int num_sms, int force_bn) {
  PRISMA_CHECK(taps * 3 <= GEMM_MAX_TAPS, "gemm(tf32x3): too many taps");
  PRISMA_CHECK(C % 32 == 0 && C_half % 32 == 0 && C <= C_half, "gemm(tf32x3): channel counts must be multiples of 32");
  int off[GEMM_MAX_TAPS], acol[GEMM_MAX_TAPS];
  for (int t = 0; t < taps; ++t)
    for (int p = 0; p < 3; ++p) { off[t * 3 + p] = tap_off[t]; acol[t * 3 + p] = p == 1 ? C_half : 0; }
  // external accumulation (GEMM_TF32_ACC_GROUP): 128-wide tiles at most (the running sums are 64 registers per thread), no
  // narrow tail tiles
  PRISMA_CHECK(force_bn <= 128, "gemm(tf32x3): BLOCK_N is at most 128");
  if (force_bn == 0) force_bn = N > 64 ? 128 : (N > 32 ? 64 : 32);
  return gemm_prepare_impl(out, A_split, a_rows, C, 2 * C_half, W3, w_rows, M, N, taps * 3, off, acol, ep, num_sms, force_bn, true);
}

static int gemm_prepare_impl(GemmLaunch* out, const void* A, long long a_rows, int a_cols, int a_pitch, const void* W,
                             int w_rows, int M, int N, int taps, const int* tap_off, const int* tap_acol, const GemmEpilogue& ep_in,
                             int num_sms, int force_bn, bool tf32) {
  PRISMA_CHECK(taps >= 1 && taps <= GEMM_MAX_TAPS, "gemm: bad tap count");
  PRISMA_CHECK(N % 4 == 0, "gemm: N must be a multiple of 4");
  PRISMA_CHECK(M >= 1 && a_cols >= 1, "gemm: empty problem");
  // force_bn == 512 requests the CTA-pair kernel (256 x 256 tiles); otherwise it is chosen for large problems
  int bn = force_bn ? force_bn : gemm_pick_bn(M, N, num_sms);
  // the TMA-store epilogue exists for 128- and 256-wide tiles; a problem the tile choice gives narrower tiles keeps the
  // register epilogue (same results: the TMA path is an optimisation of the same arithmetic)
  GemmEpilogue ep = ep_in;
  if (ep.tma_store && (bn == 32 || bn == 64) && !tf32) ep.tma_store = false;
  int cg = 1;
  if (bn == 512) { bn = 256; cg = 2; }
  else if (!force_bn && !tf32 && bn == 256 && M >= 1024 && N >= 256) cg = 2;
  PRISMA_CHECK(!(tf32 && cg == 2), "gemm: the tf32 path has no CTA-pair instantiation");
  // Transposed tiles (GemmCfg SWAP) when one 128-wide tile covers all output columns: an M = 128 instruction costs the tensor
  // core >= 128 cycles whatever its N, so 128 x 256 (weights x rows) runs at twice the rate of 128 x 128 (rows x weights).
  // force_bn == 640 requests it.
  bool swap = false;
  if (bn == 640) { bn = 128; cg = 1; swap = true; }
  else if (!force_bn && !tf32 && cg == 1 && bn == 128 && N <= 128 && M >= 4096 && !ep.tma_store && !ep.head_w && !ep.m_dev) swap = true;
  // 64 output columns: the same transposed tile with the upper 64 weight rows zero (they must exist: w_rows >= 128) -- twice
  // the MMA work of a 128 x 64 tile, but half the instructions, barriers and TMA boxes per output row (RAFT pass 6.73 -> 6.57 ms per pair)
  else if (!force_bn && !tf32 && cg == 1 && bn == 64 && N > 32 && N <= 64 && w_rows >= 128 && M >= 4096 && !ep.tma_store &&
           !ep.head_w && !ep.m_dev) { bn = 128; swap = true; }
  PRISMA_CHECK(!swap || (N <= 128 && !tf32 && !ep.tma_store && !ep.head_w), "gemm: transposed tiles need N <= 128, fp16 operands, the plain epilogue");
  out->swap = swap;
  out->tf32 = tf32;
  const int bke = tf32 ? 32 : 64;  // elements per 128-byte K block
  PRISMA_CHECK(bn == 32 || bn == 64 || bn == 128 || bn == 256, "gemm: unsupported BLOCK_N");
  PRISMA_CHECK(!swap || a_rows >= 1, "gemm: empty operand");
  out->cg = cg;
  PRISMA_CHECK(w_rows >= round_up(N, bn), "gemm: weight rows must be padded to a multiple of BLOCK_N");
  const int kchunks = ceil_div(a_cols, bke);
  out->bn = bn;
  out->args.M = M;
  out->args.N = N;
  out->args.taps = taps;
  out->args.kchunks = kchunks;
  out->args.raster_n = M >= N;
  for (int t = 0; t < GEMM_MAX_TAPS; ++t) {
    out->args.tap_off[t] = t < taps ? tap_off[t] : 0;
    out->args.tap_acol[t] = (t < taps && tap_acol) ? tap_acol[t] : 0;
  }
  out->args.ep = ep;
  if (tf32) {
    // the A map spans the [hi | lo] halves (2 * a_cols columns); out-of-range columns of a ragged last K block read as zero
    PRISMA_TRY(make_tmap_2d_f32(&out->tmA, A, (uint64_t)a_pitch, (uint64_t)a_rows, (uint64_t)a_pitch, 32, GEMM_BM));
    PRISMA_TRY(make_tmap_2d_f32(&out->tmB, W, (uint64_t)taps * kchunks * 32, (uint64_t)w_rows, (uint64_t)taps * kchunks * 32, 32, bn));
  } else {
    PRISMA_TRY(make_tmap_2d_f16(&out->tmA, A, (uint64_t)a_cols, (uint64_t)a_rows, (uint64_t)a_pitch, 64, swap ? 256 : GEMM_BM));
    PRISMA_TRY(make_tmap_2d_f16(&out->tmB, W, (uint64_t)taps * kchunks * 64, (uint64_t)w_rows,
                                (uint64_t)taps * kchunks * 64, 64, bn / cg));
  }
  const int tiles = ceil_div(M, swap ? 256 : GEMM_BM * cg) * ceil_div(N, bn);
  const int groups = num_sms / cg;
  out->grid = (tiles < groups ? tiles : groups) * cg;
  // Tail tiles: when the last wave is partial, cut its tiles into narrower ones so that it costs a fraction of a full
  // wave (same measured per-tile costs as gemm_pick_bn).  Only when the narrow tiles still fit one wave.
  out->args.n_main = tiles;
  out->args.tail_split = 1;
  out->tmBt = out->tmB;
  {
    const int full = tiles / groups, rem = tiles % groups;
    auto cost = [](int w) { return w >= 256 ? 134.0 : (w >= 128 ? 100.0 : (w >= 64 ? 68.0 : 51.0)); };
    if (!force_bn && !swap && full >= 1 && rem > 0) {  // fp16 only: the 3xTF32 path always forces its tile width
      int best_split = 1;
      double best = cost(bn);
      for (int split = 2; split <= 4; split *= 2) {
        const int bw = bn / split;
        if (bw < 32 * cg || rem * split > groups) continue;
        if (ep.tma_store && ep.out_f16 && bw < 64) continue;  // the fp16 TMA-store epilogue writes 64-column boxes
        if (cost(bw) < best) { best = cost(bw); best_split = split; }
      }
      if (best_split > 1) {
        out->args.n_main = full * groups;
        out->args.tail_split = best_split;
        PRISMA_TRY(make_tmap_2d_f16(&out->tmBt, W, (uint64_t)taps * kchunks * 64, (uint64_t)w_rows,
                                    (uint64_t)taps * kchunks * 64, 64, bn / best_split / cg));
      }
    }
  }
  if (ep.m_dev) {  // the tile count is decided on the device: no host-side tail cutting
    out->args.n_main = tiles;
    out->args.tail_split = 1;
    out->tmBt = out->tmB;
  }
  out->flops = 2.0 * M * (double)N * taps * a_cols;
  // TMA-store epilogue: a plain dense fp32 output (scale only) leaves through swizzled shared-memory boxes and
  // cp.async.bulk.tensor stores instead of per-lane st.global (the store-bound RAFT correlation volume)
  out->tma_store = false;
  out->tmD = out->tmA;
  if (ep.tma_store) {
    PRISMA_CHECK((ep.out_f32 != nullptr) != (ep.out_f16 != nullptr) && !ep.out_f16_relu && !ep.pre_f32 && !ep.gru &&
                     !ep.res_a && !ep.res_b && ep.row_map == ROW_LINEAR && !ep.head_w && !ep.stat_part,
                 "gemm: the TMA-store epilogue handles one scaled dense output (fp32 or fp16) only");
    PRISMA_CHECK(ep.out_f16 ? (ep.act >= 0 && ep.act <= 2 && !ep.gamma && !ep.res_f32) : ep.act == 0,
                 "gemm: the TMA-store epilogue applies bias + GELU / ReLU (fp16 destinations) or bias + LayerScale (fp32) only");
    // an fp32 residual must be the destination itself (x += ...): it becomes a TMA reduce-add
    PRISMA_CHECK(!ep.res_f32 || (ep.res_f32 == ep.out_f32 && ep.res_f32_ld == ep.out_f32_ld),
                 "gemm: the TMA-store epilogue adds a residual only in place");
    out->args.ep.tma_reduce = ep.res_f32 != nullptr;
    PRISMA_CHECK(!ep.out_f16 || N % 8 == 0, "gemm: the fp16 TMA-store epilogue needs N % 8 == 0");
    PRISMA_CHECK(bn >= 128, "gemm: the TMA-store epilogue is built for BLOCK_N 128 / 256");
    if (ep.out_f16) PRISMA_TRY(make_tmap_2d_f16_store(&out->tmD, ep.out_f16, (uint64_t)N, (uint64_t)M, (uint64_t)ep.out_f16_ld));
    else PRISMA_TRY(make_tmap_2d_f32(&out->tmD, ep.out_f32, (uint64_t)N, (uint64_t)M, (uint64_t)ep.out_f32_ld, 32, 32));
    out->tma_store = true;
  }
  return 0;
}

template <int BN, int CG, bool TMAST = false, bool TF32 = false, bool SWAP = false, int EW = GEMM_EPI_WARPS>
static int launch_bn(const GemmLaunch& g, cudaStream_t stream) {
  static bool attr_set = false;  // per-process, per-instantiation
  using Cfg = GemmCfg<BN, CG, TMAST, SWAP, EW>;
  if (!attr_set) {
    PRISMA_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel<BN, CG, TMAST, TF32, SWAP, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set = true;
  }
  {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(g.grid);
    cfg.blockDim = dim3(Cfg::THREADS);
    cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CG; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = CG == 2 ? 1 : 0;
    PRISMA_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, CG, TMAST, TF32, SWAP, EW>, g.tmA, g.tmB, g.tmBt, g.tmD, g.args));
  }
  PRISMA_CUDA_OK(cudaGetLastError());
  return 0;
}

int gemm_run(const GemmLaunch& g, cudaStream_t stream) {
  if (g.tf32) {  // external accumulation: BLOCK_N <= 128 (gemm_prepare_tf32x3)
    switch (g.bn) {
      case 128: return launch_bn<128, 1, false, true>(g, stream);
      case 64: return launch_bn<64, 1, false, true>(g, stream);
      case 32: return launch_bn<32, 1, false, true>(g, stream);
    }
    set_last_error("gemm_run: unsupported BLOCK_N (tf32)");
    return -1;
  }
  if (g.tma_store) {
    if (g.cg == 2 && g.bn == 256) return launch_bn<256, 2, true>(g, stream);
    if (g.cg == 1 && g.bn == 256) return launch_bn<256, 1, true>(g, stream);
    if (g.cg == 1 && g.bn == 128) return launch_bn<128, 1, true>(g, stream);
    set_last_error("gemm_run: no TMA-store instantiation for this tile shape");
    return -1;
  }
  // 16 epilogue warps (GemmCfg EW) for the transposed and the 128- / 64-wide single-CTA tiles, 8 for the 256-wide and the
  // 32-wide ones.  Measured (same box, whole bench step): 16 warps everywhere: RAFT convs 4.53 -> 4.34 ms per pair but DA
  // linears 16.7 -> 17.4 ms per pass and head convs 7.05 -> 7.38 (the 256-wide tiles lose an operand stage and spill 270 bytes
  // per thread at the 96 registers ptxas then allocates).
  if (g.swap) return launch_bn<128, 1, false, false, true, 16>(g, stream);
  if (g.cg == 2) {
    if (g.bn == 256) return launch_bn<256, 2>(g, stream);
    set_last_error("gemm_run: CTA pairs need BLOCK_N 256");
    return -1;
  }
  switch (g.bn) {
    case 256: return launch_bn<256, 1>(g, stream);
    case 128: return launch_bn<128, 1, false, false, false, 16>(g, stream);
    case 64: return launch_bn<64, 1, false, false, false, 16>(g, stream);
    case 32: return launch_bn<32, 1>(g, stream);
  }
  set_last_error("gemm_run: unsupported BLOCK_N");
  return -1;
}

}  // namespace prisma
