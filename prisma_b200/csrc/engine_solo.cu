// prisma_b200 -- SOLOv2 engine: inference_detector(model, img) of the mask_mmdet band (bands/mask_mmdet.py:133,
// bands/mmdet/apis/inference.py:99-162) for one frame, plus the band's union frame (mask_mmdet.py:43-61,134-146).
//
// Graph of one pass (all paths relative to bands/mmdet/; config values from the un-vendored
// models/solov2_r101_fpn_3x_coco.py, SURVEY.md section 8c):
//   test pipeline (datasets/pipelines/transforms.py Resize/Normalize/Pad)          -> k_solo_preprocess
//   ResNet-101, style "pytorch", frozen BatchNorm (models/backbones/resnet.py)     -> stem im2col GEMM, max-pool, 33 bottlenecks
//       = 100 tcgen05 shifted-row GEMMs on zero-bordered NHWC fp16 maps, BN folded into weights / bias, ReLU and the
//       residual add in the epilogue, stride-2 convs evaluated at stride 1 and sub-sampled by the row map
//   FPN (models/necks/fpn.py:151-204)                                               -> 1x1 / 3x3 GEMMs, nearest-add, [::2]
//   MaskFeatModule + SOLOV2Head towers (models/dense_heads/solov2_head.py)          -> GEMM -> dense fp32 -> GroupNorm+ReLU
//   get_results (solov2_head.py:582-766) + mask_matrix_nms (core/post_processing)   -> candidate list, dynamic conv as ONE GEMM
//       (kernels [n][256] x mask features [HW][256]^T, sigmoid epilogue), mask statistics, rank, binary-mask GEMM for the
//       pairwise intersections, Matrix NMS, two nested bilinear resizes + threshold + the band's union, all on the device
//       with fixed capacities (4096 candidates, nms_pre 500, 100 kept) -- no host round trip inside the pass.
#include "engine_solo.cuh"

#include <math.h>

#include <algorithm>

#include "raft_kernels.cuh"

namespace prisma {

constexpr int SOLO_CAP = 4096, SOLO_NMS_PRE = 500, SOLO_NMS_PAD = 512, SOLO_MAX = 100, SOLO_NC = 80;

template <typename T>
static int s_alloc(std::vector<void*>& pool, T** out, size_t n) {
  void* p = nullptr;
  PRISMA_CUDA_OK(cudaMalloc(&p, std::max<size_t>(n * sizeof(T), 256)));
  PRISMA_CUDA_OK(cudaMemset(p, 0, std::max<size_t>(n * sizeof(T), 256)));
  pool.push_back(p);
  *out = reinterpret_cast<T*>(p);
  return 0;
}

SoloEngine::~SoloEngine() {
  cudaSetDevice(device);
  for (void* p : allocs) cudaFree(p);
  for (void* p : plan_allocs) cudaFree(p);
  if (graph_exec) cudaGraphExecDestroy(graph_exec);
  if (ev0) cudaEventDestroy(ev0);
  if (ev1) cudaEventDestroy(ev1);
  if (stream) cudaStreamDestroy(stream);
}

int SoloEngine::init(const std::string& vin, int dev) {
  std::string v = vin;
  exact_head = true;  // "<variant>-fast": the single-pass fp16 head of round 1 (not mask-id faithful, ~40 % faster per frame)
  if (v.size() > 5 && v.substr(v.size() - 5) == "-fast") { exact_head = false; v = v.substr(0, v.size() - 5); }
  if (v.size() > 6 && v.substr(v.size() - 6) == "-exact") { exact_backbone = true; v = v.substr(0, v.size() - 6); }
  if (!exact_head) exact_backbone = false;  // the fp32-class backbone feeds the fp32-class head
  variant = v;
  if (v == "r101") { const int l[4] = {3, 4, 23, 3}; std::copy(l, l + 4, layers); scale_long = 1333; scale_short = 800; }
  else if (v == "tiny") { const int l[4] = {1, 1, 1, 1}; std::copy(l, l + 4, layers); scale_long = 448; scale_short = 256; }
  else { set_last_error("unknown SOLOv2 variant '" + v + "' (r101)"); return -1; }
  device = dev;
  int n = 0;
  PRISMA_CUDA_OK(cudaGetDeviceCount(&n));
  PRISMA_CHECK(dev >= 0 && dev < n, "bad device ordinal");
  PRISMA_CUDA_OK(cudaSetDevice(dev));
  cudaDeviceProp prop;
  PRISMA_CUDA_OK(cudaGetDeviceProperties(&prop, dev));
  PRISMA_CHECK(prop.major == 10, "prisma_b200 kernels are sm_100a only; there is no fallback path");
  num_sms = prop.multiProcessorCount;
  PRISMA_CUDA_OK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  PRISMA_CUDA_OK(cudaEventCreate(&ev0));
  PRISMA_CUDA_OK(cudaEventCreate(&ev1));
  const char* ng = getenv("PRISMA_NO_GRAPH");
  use_graph = !(ng && ng[0] == '1');
  return 0;
}

int SoloEngine::load_tensor(const std::string& name, const float* data, const int64_t* shape, int ndim) {
  PRISMA_CHECK(!finalized, "load_tensor after finalize");
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
  t.data.assign(data, data + n);
  host[name] = std::move(t);
  return 0;
}

const HostTensor* SoloEngine::get(const std::string& name) {
  auto it = host.find(name);
  if (it == host.end()) { set_last_error("missing SOLOv2 weight tensor '" + name + "'"); return nullptr; }
  return &it->second;
}

// conv weight [Cout][Cin][k][k] -> fp16 [round_up(Cout,256)][k*k*ceil(Cin/64)*64]; eval BatchNorm folded (eps 1e-5);
// GroupNorm affine kept separately (applied by the GN kernel on the fp32 conv output).
int SoloEngine::up_conv(const std::string& name, const std::string& bn, const std::string& gn, int Cout, int Cin, int k,
                        bool bias, SoloConvW* out) {
  const HostTensor* w = get(name + ".weight");
  if (!w) return -1;
  PRISMA_CHECK((long long)w->data.size() == (long long)Cout * Cin * k * k, "SOLOv2 weight '" + name + "' has an unexpected size");
  std::vector<float> sc(Cout, 1.f), sh(Cout, 0.f);
  if (bias) {
    const HostTensor* b = get(name + ".bias");
    if (!b) return -1;
    for (int n = 0; n < Cout; ++n) sh[n] = b->data[n];
  }
  if (!bn.empty()) {
    const HostTensor *g = get(bn + ".weight"), *be = get(bn + ".bias"), *mu = get(bn + ".running_mean"), *var = get(bn + ".running_var");
    if (!g || !be || !mu || !var) return -1;
    for (int n = 0; n < Cout; ++n) {
      const float s = g->data[n] / sqrtf(var->data[n] + 1e-5f);
      sc[n] = s;
      sh[n] = (sh[n] - mu->data[n]) * s + be->data[n];
    }
  }
  const int taps = k * k, kc = ceil_div(Cin, 64), K = taps * kc * 64, rows = round_up(Cout, 256);
  std::vector<__half> h((size_t)rows * K, __float2half_rn(0.f));
  for (int n = 0; n < Cout; ++n)
    for (int t = 0; t < taps; ++t)
      for (int c = 0; c < Cin; ++c)
        h[(size_t)n * K + (size_t)t * kc * 64 + c] = __float2half_rn(w->data[((size_t)n * Cin + c) * taps + t] * sc[n]);
  PRISMA_TRY(s_alloc(allocs, &out->w, h.size()));
  PRISMA_CUDA_OK(cudaMemcpy(out->w, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
  std::vector<float> bv(round_up(Cout, 8), 0.f);
  for (int n = 0; n < Cout; ++n) bv[n] = sh[n];
  PRISMA_TRY(s_alloc(allocs, &out->b, bv.size()));
  PRISMA_CUDA_OK(cudaMemcpy(out->b, bv.data(), bv.size() * 4, cudaMemcpyHostToDevice));
  if (!gn.empty()) {
    const HostTensor *g = get(gn + ".weight"), *be = get(gn + ".bias");
    if (!g || !be) return -1;
    PRISMA_TRY(s_alloc(allocs, &out->gn_w, (size_t)Cout));
    PRISMA_TRY(s_alloc(allocs, &out->gn_b, (size_t)Cout));
    PRISMA_CUDA_OK(cudaMemcpy(out->gn_w, g->data.data(), Cout * 4, cudaMemcpyHostToDevice));
    PRISMA_CUDA_OK(cudaMemcpy(out->gn_b, be->data.data(), Cout * 4, cudaMemcpyHostToDevice));
  }
  out->cout = Cout; out->cin = Cin; out->k = k;
  return 0;
}

// head conv weight [Cout][Cin][k][k] -> fp32 [round_up(Cout,256)][k*k * 3 * cin32], per tap [W_hi | W_hi | W_lo] with
// W_hi = the weight with its low 13 mantissa bits cleared (a TF32 number), W_lo = W - W_hi: the B operand of
// gemm_prepare_tf32x3.  GroupNorm affine kept separately, bias fp32.
// bn (backbone convs): eval BatchNorm folded in fp32 -- weight * gamma / sqrt(var + eps), bias (0 - mean) * that + beta.
int SoloEngine::up_conv3(const std::string& name, const std::string& gn, int Cout, int Cin, int k, bool bias, SoloConvW3* out,
                         const std::string& bn) {
  const HostTensor* w = get(name + ".weight");
  if (!w) return -1;
  PRISMA_CHECK((long long)w->data.size() == (long long)Cout * Cin * k * k, "SOLOv2 weight '" + name + "' has an unexpected size");
  const int taps = k * k, c32 = round_up(Cin, 32), K = taps * 3 * c32, rows = round_up(Cout, 256);
  std::vector<float> h((size_t)rows * K, 0.f);
  auto hi_of = [](float v) { uint32_t u; memcpy(&u, &v, 4); u &= 0xFFFFE000u; float r; memcpy(&r, &u, 4); return r; };
  std::vector<float> sc(Cout, 1.f), sh(Cout, 0.f);
  if (!bn.empty()) {
    const HostTensor *g = get(bn + ".weight"), *be = get(bn + ".bias"), *mu = get(bn + ".running_mean"), *var = get(bn + ".running_var");
    if (!g || !be || !mu || !var) return -1;
    for (int n = 0; n < Cout; ++n) {
      sc[n] = g->data[n] / sqrtf(var->data[n] + 1e-5f);
      sh[n] = (0.f - mu->data[n]) * sc[n] + be->data[n];
    }
  }
  for (int n = 0; n < Cout; ++n)
    for (int t = 0; t < taps; ++t)
      for (int c = 0; c < Cin; ++c) {
        const float v = w->data[((size_t)n * Cin + c) * taps + t] * sc[n], hi = hi_of(v);
        float* base = h.data() + (size_t)n * K + (size_t)t * 3 * c32;
        base[c] = hi; base[c32 + c] = hi; base[2 * c32 + c] = v - hi;
      }
  PRISMA_TRY(s_alloc(allocs, &out->w, h.size()));
  PRISMA_CUDA_OK(cudaMemcpy(out->w, h.data(), h.size() * 4, cudaMemcpyHostToDevice));
  std::vector<float> bv(round_up(Cout, 8), 0.f);
  for (int n = 0; n < Cout; ++n) bv[n] = sh[n];
  if (bias) {
    const HostTensor* b = get(name + ".bias");
    if (!b) return -1;
    PRISMA_CHECK(bn.empty(), "up_conv3: bias and BatchNorm together are not used by this model");
    for (int n = 0; n < Cout; ++n) bv[n] = b->data[n];
  }
  PRISMA_TRY(s_alloc(allocs, &out->b, bv.size()));
  PRISMA_CUDA_OK(cudaMemcpy(out->b, bv.data(), bv.size() * 4, cudaMemcpyHostToDevice));
  if (!gn.empty()) {
    const HostTensor *g = get(gn + ".weight"), *be = get(gn + ".bias");
    if (!g || !be) return -1;
    PRISMA_TRY(s_alloc(allocs, &out->gn_w, (size_t)Cout));
    PRISMA_TRY(s_alloc(allocs, &out->gn_b, (size_t)Cout));
    PRISMA_CUDA_OK(cudaMemcpy(out->gn_w, g->data.data(), Cout * 4, cudaMemcpyHostToDevice));
    PRISMA_CUDA_OK(cudaMemcpy(out->gn_b, be->data.data(), Cout * 4, cudaMemcpyHostToDevice));
  }
  out->cout = Cout; out->cin = Cin; out->cin32 = c32; out->k = k;
  return 0;
}

int SoloEngine::finalize() {
  PRISMA_CHECK(!finalized, "finalize called twice");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  {  // stem 7x7/2: im2col K = 168, k = (c*7 + ky)*8 + kx with kx = 7 zero (the layout raft_im2col_stem writes: one 16-byte group
     // = one 7-pixel input row segment) -> a "1x1 conv" with Cin 168
    const HostTensor* w = get("backbone.conv1.weight");
    if (!w) return -1;
    PRISMA_CHECK(w->data.size() == (size_t)64 * 147, "backbone.conv1 has an unexpected size");
    HostTensor flat;
    flat.shape = {64, 168, 1, 1};
    flat.data.assign((size_t)64 * 168, 0.f);
    for (int o = 0; o < 64; ++o)
      for (int cy = 0; cy < 21; ++cy)
        for (int kx = 0; kx < 7; ++kx) flat.data[(size_t)o * 168 + cy * 8 + kx] = w->data[(size_t)o * 147 + cy * 7 + kx];
    host["backbone.conv1_flat.weight"] = flat;
    PRISMA_TRY(up_conv("backbone.conv1_flat", "backbone.bn1", "", 64, 168, 1, false, &stem));
  }
  int inplanes = 64;
  const int planes_of[4] = {64, 128, 256, 512};
  for (int li = 0; li < 4; ++li) {
    blocks[li].resize(layers[li]);
    for (int b = 0; b < layers[li]; ++b) {
      const std::string p = "backbone.layer" + std::to_string(li + 1) + "." + std::to_string(b) + ".";
      Block& k = blocks[li][b];
      const int pl = planes_of[li];
      k.stride = (b == 0 && li > 0) ? 2 : 1;
      PRISMA_TRY(up_conv(p + "conv1", p + "bn1", "", pl, inplanes, 1, false, &k.c1));
      PRISMA_TRY(up_conv(p + "conv2", p + "bn2", "", pl, pl, 3, false, &k.c2));
      PRISMA_TRY(up_conv(p + "conv3", p + "bn3", "", pl * 4, pl, 1, false, &k.c3));
      k.has_ds = b == 0;
      if (k.has_ds) PRISMA_TRY(up_conv(p + "downsample.0", p + "downsample.1", "", pl * 4, inplanes, 1, false, &k.ds));
      inplanes = pl * 4;
    }
  }
  const int cins[4] = {256, 512, 1024, 2048};
  for (int i = 0; i < 4; ++i) {
    PRISMA_TRY(up_conv("neck.lateral_convs." + std::to_string(i) + ".conv", "", "", 256, cins[i], 1, true, &lateral[i]));
    PRISMA_TRY(up_conv("neck.fpn_convs." + std::to_string(i) + ".conv", "", "", 256, 256, 3, true, &fpnc[i]));
  }
  const std::string m = "mask_head.mask_feature_head.";
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < std::max(i, 1); ++j) {
      const std::string n = m + "convs_all_levels." + std::to_string(i) + ".conv" + std::to_string(j);
      const int cin = j == 0 ? (i == 3 ? 258 : 256) : 128;
      PRISMA_TRY(up_conv(n + ".conv", "", n + ".gn", 128, cin, 3, false, &mf[i][j]));
    }
  PRISMA_TRY(up_conv(m + "conv_pred.conv", "", m + "conv_pred.gn", 256, 128, 1, false, &mf_pred));
  for (int i = 0; i < 4; ++i) {
    const std::string kn = "mask_head.kernel_convs." + std::to_string(i), cn = "mask_head.cls_convs." + std::to_string(i);
    PRISMA_TRY(up_conv(kn + ".conv", "", kn + ".gn", 512, i == 0 ? 258 : 512, 3, false, &kconv[i]));
    PRISMA_TRY(up_conv(cn + ".conv", "", cn + ".gn", 512, i == 0 ? 256 : 512, 3, false, &cconv[i]));
  }
  PRISMA_TRY(up_conv("mask_head.conv_cls", "", "", SOLO_NC, 512, 3, true, &conv_cls));
  PRISMA_TRY(up_conv("mask_head.conv_kernel", "", "", 256, 512, 3, true, &conv_kernel));
  if (exact_head) {  // the same head in fp32 [hi | hi | lo] for the 3xTF32 path
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < std::max(i, 1); ++j) {
        const std::string n = m + "convs_all_levels." + std::to_string(i) + ".conv" + std::to_string(j);
        PRISMA_TRY(up_conv3(n + ".conv", n + ".gn", 128, j == 0 ? (i == 3 ? 258 : 256) : 128, 3, false, &mf3[i][j]));
      }
    PRISMA_TRY(up_conv3(m + "conv_pred.conv", m + "conv_pred.gn", 256, 128, 1, false, &mf_pred3));
    for (int i = 0; i < 4; ++i) {
      const std::string kn = "mask_head.kernel_convs." + std::to_string(i), cn = "mask_head.cls_convs." + std::to_string(i);
      PRISMA_TRY(up_conv3(kn + ".conv", kn + ".gn", 512, i == 0 ? 258 : 512, 3, false, &kconv3[i]));
      PRISMA_TRY(up_conv3(cn + ".conv", cn + ".gn", 512, i == 0 ? 256 : 512, 3, false, &cconv3[i]));
    }
    PRISMA_TRY(up_conv3("mask_head.conv_cls", "", SOLO_NC, 512, 3, true, &conv_cls3));
    PRISMA_TRY(up_conv3("mask_head.conv_kernel", "", 256, 512, 3, true, &conv_kernel3));
  }
  if (exact_backbone) {  // ResNet + FPN in [hi | hi | lo] fp32, BatchNorm folded in fp32
    PRISMA_TRY(up_conv3("backbone.conv1_flat", "", 64, 168, 1, false, &stem3, "backbone.bn1"));
    int inp = 64;
    for (int li = 0; li < 4; ++li) {
      blocks3[li].resize(layers[li]);
      for (int b = 0; b < layers[li]; ++b) {
        const std::string p = "backbone.layer" + std::to_string(li + 1) + "." + std::to_string(b) + ".";
        Block3& k = blocks3[li][b];
        const int pl = planes_of[li];
        PRISMA_TRY(up_conv3(p + "conv1", "", pl, inp, 1, false, &k.c1, p + "bn1"));
        PRISMA_TRY(up_conv3(p + "conv2", "", pl, pl, 3, false, &k.c2, p + "bn2"));
        PRISMA_TRY(up_conv3(p + "conv3", "", pl * 4, pl, 1, false, &k.c3, p + "bn3"));
        if (b == 0) PRISMA_TRY(up_conv3(p + "downsample.0", "", pl * 4, inp, 1, false, &k.ds, p + "downsample.1"));
        inp = pl * 4;
      }
    }
    for (int i = 0; i < 4; ++i) {
      PRISMA_TRY(up_conv3("neck.lateral_convs." + std::to_string(i) + ".conv", "", 256, cins[i], 1, true, &lateral3[i]));
      PRISMA_TRY(up_conv3("neck.fpn_convs." + std::to_string(i) + ".conv", "", 256, 256, 3, true, &fpnc3[i]));
    }
  }
  host.clear();
  finalized = true;
  return 0;
}

// mmcv.imrescale((1333, 800), keep_ratio) + Pad(size_divisor=32) sizes
int SoloEngine::net_shape(int H, int W, int* nh_, int* nw_, int* hp_, int* wp_) const {
  const double s = std::min((double)scale_long / std::max(H, W), (double)scale_short / std::min(H, W));
  *nw_ = (int)(W * s + 0.5);
  *nh_ = (int)(H * s + 0.5);
  *hp_ = round_up(*nh_, 32);
  *wp_ = round_up(*nw_, 32);
  return 0;
}

int SoloEngine::build_plan(int H, int W) {
  PRISMA_CHECK(finalized, "weights not finalized");
  if (plan_H == H && plan_W == W) return 0;
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  for (void* q : plan_allocs) cudaFree(q);
  plan_allocs.clear();
  steps.clear();
  taps.clear();
  flops = 0;
  plan_H = plan_W = 0;
  d_inst = nullptr;
  net_shape(H, W, &nh, &nw, &hp, &wp);
  const int zero_off[1] = {0};
  const char* cur_tag = "pre";
  step_tag.clear();
  auto push_step = [&](std::function<int(cudaStream_t)> fn) { steps.push_back(std::move(fn)); step_tag.push_back(cur_tag); };

  auto new_map = [&](SMap* mm, int h, int w, int c) -> int {
    mm->H = h; mm->W = w; mm->C = c;
    return s_alloc(plan_allocs, &mm->p, (size_t)mm->rows() * c);
  };
  // conv on a zero-bordered map.  dst_map: zero-bordered fp16 output (stride `sub`); dst_dense: dense fp32 [H*W][Cout]
  auto conv = [&](const SMap& in, int cin_cols, const SoloConvW& w, int sub, GemmEpilogue ep, const SMap* dst_map,
                  float* dst_dense) -> int {
    int off[9], taps_n = w.k * w.k;
    if (w.k == 3) { for (int ky = 0; ky < 3; ++ky) for (int kx = 0; kx < 3; ++kx) off[ky * 3 + kx] = (ky - 1) * in.Wp() + (kx - 1); }
    else off[0] = 0;
    ep.in_w = in.Wp(); ep.in_h = in.Hp(); ep.img_rows = 0; ep.sub = sub; ep.pad = 1;
    if (dst_map) {
      ep.row_map = ROW_PADDED;
      if (sub > 1) { ep.out_wp = dst_map->Wp(); ep.out_img_rows = (int)dst_map->rows(); ep.out_pad = 1; }
    } else {
      ep.row_map = ROW_PAD2TOK;
      ep.out_f32 = dst_dense; ep.out_f32_ld = w.cout;
    }
    GemmLaunch g;
    PRISMA_TRY(gemm_prepare(&g, in.p, in.rows(), cin_cols, in.C, w.w, round_up(w.cout, 256), (int)in.rows(), w.cout, taps_n, off,
                            ep, num_sms));
    flops += 2.0 * (in.H / sub) * (double)(in.W / sub) * taps_n * w.cin * w.cout;
    push_step([g](cudaStream_t s) { return gemm_run(g, s); });
    return 0;
  };
  float* gn_part = nullptr; float* gn_stats = nullptr; float* gn_raw = nullptr;
  const size_t raw_max = (size_t)(hp / 4) * (wp / 4) * 256;
  PRISMA_TRY(s_alloc(plan_allocs, &gn_raw, raw_max));
  PRISMA_TRY(s_alloc(plan_allocs, &gn_part, (size_t)gn_partial_floats((hp / 4) * (wp / 4), 512)));
  PRISMA_TRY(s_alloc(plan_allocs, &gn_stats, 1024));
  // ConvModule(norm GN-32): conv (no bias) -> dense fp32 -> GroupNorm + ReLU -> fp16 map (and / or dense fp16)
  auto gnconv = [&](const SMap& in, int cin_cols, const SoloConvW& w, const SMap* dst_map, __half* dst_dense) -> int {
    GemmEpilogue ep;
    PRISMA_TRY(conv(in, cin_cols, w, 1, ep, nullptr, gn_raw));
    const int h = in.H, ww = in.W, c = w.cout; const float* gw = w.gn_w; const float* gb = w.gn_b;
    __half* dm = dst_map ? dst_map->p : nullptr;
    push_step([=](cudaStream_t s) { return groupnorm_relu_f16(gn_raw, h, ww, c, 32, gw, gb, gn_part, gn_stats, dm, dst_dense, s); });
    return 0;
  };

  // ---- test pipeline
  PRISMA_TRY(s_alloc(plan_allocs, &d_img, (size_t)H * W * 3));
  PRISMA_TRY(s_alloc(plan_allocs, &d_resized, (size_t)nh * nw * 3));
  PRISMA_TRY(s_alloc(plan_allocs, &d_net, (size_t)3 * hp * wp));
  {
    const uint8_t* img = d_img; uint8_t* rs = d_resized; float* net = d_net;
    const int nh_ = nh, nw_ = nw, hp_ = hp, wp_ = wp;
    push_step([=](cudaStream_t s) { return solo_preprocess(img, H, W, nh_, nw_, hp_, wp_, net, rs, s); });
  }
  cur_tag = "backbone";
  SMap P[5];
  float* P_dense[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // exact backbone: FPN levels as dense fp32 [H*W][256]
  if (exact_backbone) {
    // ================================================================ fp32-class ResNet + FPN ("-exact" variants)
    // conv = 3xTF32 GEMM (external fp32 accumulation) from a split map to a dense fp32 [Ho*Wo][Cout] map; bias (folded
    // BatchNorm), the residual sum (pre_f32) and ReLU in the epilogue; solo_dense_to_split builds the next conv's operand.
    auto new_xm = [&](XMap* mm, int h, int w, int c) -> int {
      mm->H = h; mm->W = w; mm->C = c;
      return s_alloc(plan_allocs, &mm->p, (size_t)mm->rows() * 2 * c);
    };
    auto conv_b = [&](const XMap& in, const SoloConvW3& w, int sub, GemmEpilogue ep, float* dst_dense) -> int {
      PRISMA_CHECK(in.C == w.cin32, "solo(exact backbone): operand channels do not match the packed weights");
      int off[9], taps_n = w.k * w.k;
      if (w.k == 3) { for (int ky = 0; ky < 3; ++ky) for (int kx = 0; kx < 3; ++kx) off[ky * 3 + kx] = (ky - 1) * in.Wp() + (kx - 1); }
      else off[0] = 0;
      ep.in_w = in.Wp(); ep.in_h = in.Hp(); ep.img_rows = 0; ep.sub = sub; ep.pad = 1;
      ep.row_map = ROW_PAD2TOK; ep.out_f32 = dst_dense; ep.out_f32_ld = w.cout; ep.bias = w.b;
      GemmLaunch g;
      PRISMA_TRY(gemm_prepare_tf32x3(&g, in.p, in.rows(), in.C, in.C, w.w, round_up(w.cout, 256), (int)in.rows(), w.cout, taps_n, off,
                                     ep, num_sms));
      flops += 2.0 * ceil_div(in.H, sub) * (double)ceil_div(in.W, sub) * taps_n * w.cin * w.cout;
      push_step([g](cudaStream_t s) { return gemm_run(g, s); });
      return 0;
    };
    auto to_split = [&](const float* dense, const XMap& o) {
      push_step([=](cudaStream_t s) { return solo_dense_to_split(dense, o.H, o.W, o.C, o.p, o.C, s); });
    };
    // stem: im2col split -> GEMM (+ folded BN, ReLU) -> dense [H/2 * W/2][64] -> max-pool -> dense + split
    const int h2 = hp / 2, w2 = wp / 2, h4 = hp / 4, w4 = wp / 4;
    float *cols = nullptr, *s1d = nullptr, *xd = nullptr;
    PRISMA_TRY(s_alloc(plan_allocs, &cols, (size_t)h2 * w2 * 384));
    PRISMA_TRY(s_alloc(plan_allocs, &s1d, (size_t)h2 * w2 * 64));
    PRISMA_TRY(s_alloc(plan_allocs, &xd, (size_t)h4 * w4 * 64));
    { const float* net = d_net; const int hp_ = hp, wp_ = wp;
      push_step([=](cudaStream_t s) { return solo_im2col_stem_split(net, hp_, wp_, cols, s); }); }
    { GemmEpilogue ep; ep.bias = stem3.b; ep.act = 2; ep.out_f32 = s1d; ep.out_f32_ld = 64;
      GemmLaunch g;
      const int M = h2 * w2;
      PRISMA_TRY(gemm_prepare_tf32x3(&g, cols, M, 192, 192, stem3.w, 256, M, 64, 1, zero_off, ep, num_sms));
      flops += 2.0 * M * 147.0 * 64;
      push_step([g](cudaStream_t s) { return gemm_run(g, s); }); }
    XMap xs;
    PRISMA_TRY(new_xm(&xs, h4, w4, 64));
    { const XMap o = xs; push_step([=](cudaStream_t s) { return maxpool3s2_dense(s1d, h2, w2, 64, xd, o.p, o.H, o.W, s); }); }
    // bottlenecks (resnet.py:255-300)
    XMap CX[4];
    for (int li = 0; li < 4; ++li) {
      for (size_t b = 0; b < blocks3[li].size(); ++b) {
        const Block3& k = blocks3[li][b];
        const int stride = blocks[li][b].stride;
        const int ho = xs.H / stride, wo = xs.W / stride;
        XMap as, ms, os;
        float *ad = nullptr, *md = nullptr, *od = nullptr, *idn = xd;
        PRISMA_TRY(new_xm(&as, xs.H, xs.W, k.c1.cout));
        PRISMA_TRY(new_xm(&ms, ho, wo, k.c2.cout));
        PRISMA_TRY(new_xm(&os, ho, wo, k.c3.cout));
        PRISMA_TRY(s_alloc(plan_allocs, &ad, (size_t)xs.H * xs.W * k.c1.cout));
        PRISMA_TRY(s_alloc(plan_allocs, &md, (size_t)ho * wo * k.c2.cout));
        PRISMA_TRY(s_alloc(plan_allocs, &od, (size_t)ho * wo * k.c3.cout));
        { GemmEpilogue ep; ep.act = 2; PRISMA_TRY(conv_b(xs, k.c1, 1, ep, ad)); }
        to_split(ad, as);
        { GemmEpilogue ep; ep.act = 2; PRISMA_TRY(conv_b(as, k.c2, stride, ep, md)); }
        to_split(md, ms);
        if (b == 0) {
          PRISMA_TRY(s_alloc(plan_allocs, &idn, (size_t)ho * wo * k.ds.cout));
          GemmEpilogue ep; PRISMA_TRY(conv_b(xs, k.ds, stride, ep, idn));
        }
        { GemmEpilogue ep; ep.act = 2; ep.pre_f32 = idn; ep.pre_f32_ld = k.c3.cout; PRISMA_TRY(conv_b(ms, k.c3, 1, ep, od)); }
        to_split(od, os);
        xs = os; xd = od;
      }
      CX[li] = xs;
    }
    cur_tag = "fpn";
    float* Ld[4];
    XMap LX[4];
    for (int i = 0; i < 4; ++i) {
      PRISMA_TRY(s_alloc(plan_allocs, &Ld[i], (size_t)CX[i].H * CX[i].W * 256));
      GemmEpilogue ep; PRISMA_TRY(conv_b(CX[i], lateral3[i], 1, ep, Ld[i]));
    }
    for (int i = 3; i > 0; --i) {
      float* f = Ld[i - 1]; const float* c = Ld[i];
      const int hf = CX[i - 1].H, wf = CX[i - 1].W, hc = CX[i].H, wc = CX[i].W;
      push_step([=](cudaStream_t s) { return nearest_add_dense(f, hf, wf, c, hc, wc, 256, s); });
    }
    for (int i = 0; i < 4; ++i) {
      PRISMA_TRY(new_xm(&LX[i], CX[i].H, CX[i].W, 256));
      to_split(Ld[i], LX[i]);
      P[i].H = CX[i].H; P[i].W = CX[i].W; P[i].C = 256; P[i].p = nullptr;
      PRISMA_TRY(s_alloc(plan_allocs, &P_dense[i], (size_t)P[i].H * P[i].W * 256));
      GemmEpilogue ep; PRISMA_TRY(conv_b(LX[i], fpnc3[i], 1, ep, P_dense[i]));
    }
    P[4].H = (P[3].H - 1) / 2 + 1; P[4].W = (P[3].W - 1) / 2 + 1; P[4].C = 256; P[4].p = nullptr;
    PRISMA_TRY(s_alloc(plan_allocs, &P_dense[4], (size_t)P[4].H * P[4].W * 256));
    { const float* a = P_dense[3]; float* o = P_dense[4]; const int h3 = P[3].H, w3 = P[3].W, h4_ = P[4].H, w4_ = P[4].W;
      push_step([=](cudaStream_t s) { return subsample2_dense(a, h3, w3, 256, o, h4_, w4_, s); }); }
    for (int i = 0; i < 5; ++i) taps["fpn" + std::to_string(i)] = {P_dense[i], 0, P[i].H * P[i].W, 256, 0};
  } else {
    // ---- ResNet stem: 7x7/2 conv + BN + ReLU (im2col GEMM), 3x3/2 max-pool
    SMap s1, x;
    PRISMA_TRY(new_map(&s1, hp / 2, wp / 2, 64));
    {
      __half* cols = nullptr;
      PRISMA_TRY(s_alloc(plan_allocs, &cols, (size_t)(hp / 2) * (wp / 2) * 192));
      const float* net = d_net; const int hp_ = hp, wp_ = wp;
      push_step([=](cudaStream_t s) { return raft_im2col_stem(net, 1, hp_, wp_, cols, s); });
      GemmEpilogue ep; ep.bias = stem.b; ep.act = 2; ep.out_f16 = s1.p; ep.out_f16_ld = 64;
      ep.row_map = ROW_TOK2PAD; ep.in_w = wp / 2; ep.in_h = hp / 2; ep.out_wp = s1.Wp(); ep.out_img_rows = (int)s1.rows(); ep.out_pad = 1;
      GemmLaunch g;
      const int M = (hp / 2) * (wp / 2);
      PRISMA_TRY(gemm_prepare(&g, cols, M, 192, 192, stem.w, 256, M, 64, 1, zero_off, ep, num_sms));
      flops += 2.0 * M * 147.0 * 64;
      push_step([g](cudaStream_t s) { return gemm_run(g, s); });
    }
    PRISMA_TRY(new_map(&x, hp / 4, wp / 4, 64));
    { const SMap a = s1, o = x; push_step([=](cudaStream_t s) { return maxpool3s2_f16(a.p, a.H, a.W, 64, o.p, o.H, o.W, s); }); }
    // ---- bottlenecks (resnet.py:255-300): 1x1 -> 3x3 (stride) -> 1x1, + identity / downsample, ReLU
    SMap C[4];
    for (int li = 0; li < 4; ++li) {
      for (size_t b = 0; b < blocks[li].size(); ++b) {
        const Block& k = blocks[li][b];
        const int ho = x.H / k.stride, wo = x.W / k.stride;
        SMap a, m2, o, idn = x;
        PRISMA_TRY(new_map(&a, x.H, x.W, k.c1.cout));
        PRISMA_TRY(new_map(&m2, ho, wo, k.c2.cout));
        PRISMA_TRY(new_map(&o, ho, wo, k.c3.cout));
        { GemmEpilogue ep; ep.bias = k.c1.b; ep.act = 2; ep.out_f16 = a.p; ep.out_f16_ld = a.C;
          PRISMA_TRY(conv(x, x.C, k.c1, 1, ep, &a, nullptr)); }
        { GemmEpilogue ep; ep.bias = k.c2.b; ep.act = 2; ep.out_f16 = m2.p; ep.out_f16_ld = m2.C;
          PRISMA_TRY(conv(a, a.C, k.c2, k.stride, ep, &m2, nullptr)); }
        if (k.has_ds) {
          PRISMA_TRY(new_map(&idn, ho, wo, k.ds.cout));
          GemmEpilogue ep; ep.bias = k.ds.b; ep.out_f16 = idn.p; ep.out_f16_ld = idn.C;
          PRISMA_TRY(conv(x, x.C, k.ds, k.stride, ep, &idn, nullptr));
        }
        { GemmEpilogue ep; ep.bias = k.c3.b; ep.res_a = idn.p; ep.res_a_ld = idn.C; ep.out_f16_relu = o.p; ep.out_f16_relu_ld = o.C;
          PRISMA_TRY(conv(m2, m2.C, k.c3, 1, ep, &o, nullptr)); }
        x = o;
      }
      C[li] = x;
    }
    cur_tag = "fpn";
    // ---- FPN
    SMap L[4];
    for (int i = 0; i < 4; ++i) {
      PRISMA_TRY(new_map(&L[i], C[i].H, C[i].W, 256));
      GemmEpilogue ep; ep.bias = lateral[i].b; ep.out_f16 = L[i].p; ep.out_f16_ld = 256;
      PRISMA_TRY(conv(C[i], C[i].C, lateral[i], 1, ep, &L[i], nullptr));
    }
    for (int i = 3; i > 0; --i) {
      const SMap f = L[i - 1], c = L[i];
      push_step([=](cudaStream_t s) { return nearest_add_f16(f.p, f.H, f.W, c.p, c.H, c.W, 256, s); });
    }
    for (int i = 0; i < 4; ++i) {
      PRISMA_TRY(new_map(&P[i], L[i].H, L[i].W, 256));
      GemmEpilogue ep; ep.bias = fpnc[i].b; ep.out_f16 = P[i].p; ep.out_f16_ld = 256;
      PRISMA_TRY(conv(L[i], 256, fpnc[i], 1, ep, &P[i], nullptr));
    }
    PRISMA_TRY(new_map(&P[4], (P[3].H - 1) / 2 + 1, (P[3].W - 1) / 2 + 1, 256));
    { const SMap a = P[3], o = P[4]; push_step([=](cudaStream_t s) { return subsample2_f16(a.p, a.H, a.W, 256, o.p, o.H, o.W, s); }); }
    for (int i = 0; i < 5; ++i) taps["fpn" + std::to_string(i)] = {P[i].p, 1, P[i].H, P[i].W, 256};
  }

  head_step0 = steps.size();
  fh = P[0].H; fw = P[0].W;
  const int HW = fh * fw;
  const int F = *std::max_element(num_grids, num_grids + 5), FP = (F + 2) * (F + 2);
  GridSizes gs;
  for (int l = 0; l < 8; ++l) gs.s[l] = l < 5 ? num_grids[l] : 0;
  int cell0[5], cells = 0;
  for (int l = 0; l < 5; ++l) { cell0[l] = cells; cells += num_grids[l] * num_grids[l]; }
  float *ker_all = nullptr, *cls_all = nullptr;  // dense fp32 [5][F*F][256] / [5][F*F][80]
  PRISMA_TRY(s_alloc(plan_allocs, &ker_all, (size_t)5 * F * F * 256));
  PRISMA_TRY(s_alloc(plan_allocs, &cls_all, (size_t)5 * F * F * SOLO_NC));
  float* tower_raw = nullptr;  // dense fp32 conv output [5][F*F][512]
  PRISMA_TRY(s_alloc(plan_allocs, &tower_raw, (size_t)5 * F * F * 512));
  __half* mfeat = nullptr;   // fast head: dense [HW][256] fp16, the "weight" of the dynamic-conv GEMM
  float* mfeat3 = nullptr;   // exact head: dense [HW][3 * 256] fp32 = [hi | hi | lo]
  if (!exact_head) {
  cur_tag = "mask_feature_head";
  // ---- mask feature head (solov2_head.py:133-150)
  SMap acc;
  PRISMA_TRY(new_map(&acc, fh, fw, 128));
  PRISMA_TRY(gnconv(P[0], 256, mf[0][0], &acc, nullptr));
  for (int i = 1; i < 4; ++i) {
    SMap cur = P[i];
    int cin_cols = 256;
    if (i == 3) {  // + generate_coordinate channels: 258 -> 320-channel operand
      SMap cc;
      PRISMA_TRY(new_map(&cc, P[3].H, P[3].W, 320));
      const SMap a = P[3];
      push_step([=](cudaStream_t s) { return resize_bilinear_f16(a.p, a.H, a.W, 256, cc.p, cc.H, cc.W, 320, 1, 0, s); });
      cur = cc; cin_cols = 320;
    }
    for (int j = 0; j < i; ++j) {
      SMap t, u;
      PRISMA_TRY(new_map(&t, cur.H, cur.W, 128));
      PRISMA_TRY(gnconv(cur, cin_cols, mf[i][j], &t, nullptr));
      const bool last = j == i - 1;
      if (last) u = acc; else PRISMA_TRY(new_map(&u, 2 * t.H, 2 * t.W, 128));
      PRISMA_CHECK(u.H == 2 * t.H && u.W == 2 * t.W, "solo: FPN levels are not exact halvings (pad to a multiple of 32)");
      push_step([=](cudaStream_t s) { return resize_bilinear_f16(t.p, t.H, t.W, 128, u.p, u.H, u.W, 128, 0, last ? 1 : 0, s); });
      cur = u; cin_cols = 128;
    }
  }
  PRISMA_TRY(s_alloc(plan_allocs, &mfeat, (size_t)round_up(HW, 256) * 256));
  PRISMA_TRY(gnconv(acc, 128, mf_pred, nullptr, mfeat));
  taps["mask_feats"] = {mfeat, 2, HW, 256, 0};

  cur_tag = "towers";
  // ---- head towers (solov2_head.py:253-292, resize_feats solo_head.py:133-153)
  SMap R0, R4;
  PRISMA_TRY(new_map(&R0, P[1].H, P[1].W, 256));
  PRISMA_TRY(new_map(&R4, P[3].H, P[3].W, 256));
  { const SMap a = P[0], o = R0; push_step([=](cudaStream_t s) { return resize_bilinear_f16(a.p, a.H, a.W, 256, o.p, o.H, o.W, 256, 0, 0, s); }); }
  { const SMap a = P[4], o = R4; push_step([=](cudaStream_t s) { return resize_bilinear_f16(a.p, a.H, a.W, 256, o.p, o.H, o.W, 256, 0, 0, s); }); }
  const SMap lvl_in[5] = {R0, P[1], P[2], P[3], R4};
  // The five levels share the tower weights: they run as one stack of F x F frames (F = largest grid), level l in the
  // top-left S_l x S_l of frame l; pixels outside stay zero = the convs' zero padding.  10 GEMMs + 8 GroupNorms in total.
  struct TMap { __half* p; int C; };
  auto new_tmap = [&](TMap* t, int c) -> int { t->C = c; return s_alloc(plan_allocs, &t->p, (size_t)5 * FP * c); };
  auto conv_t = [&](const TMap& in, int cin_cols, const SoloConvW& w, GemmEpilogue ep, float* dst_dense) -> int {
    int off[9];
    for (int ky = 0; ky < 3; ++ky) for (int kx = 0; kx < 3; ++kx) off[ky * 3 + kx] = (ky - 1) * (F + 2) + (kx - 1);
    ep.in_w = F + 2; ep.in_h = F + 2; ep.img_rows = FP; ep.sub = 1; ep.pad = 1;
    ep.row_map = ROW_PAD2TOK; ep.out_f32 = dst_dense; ep.out_f32_ld = w.cout;
    GemmLaunch g;
    PRISMA_TRY(gemm_prepare(&g, in.p, 5LL * FP, cin_cols, in.C, w.w, round_up(w.cout, 256), 5 * FP, w.cout, 9, off, ep, num_sms));
    double px = 0; for (int l = 0; l < 5; ++l) px += (double)num_grids[l] * num_grids[l];
    flops += 2.0 * px * 9 * w.cin * w.cout;
    push_step([g](cudaStream_t s) { return gemm_run(g, s); });
    return 0;
  };
  auto gnconv_t = [&](const TMap& in, int cin_cols, const SoloConvW& w, const TMap& out) -> int {
    GemmEpilogue ep;
    PRISMA_TRY(conv_t(in, cin_cols, w, ep, tower_raw));
    const float* gw = w.gn_w; const float* gb = w.gn_b; __half* o = out.p; const int c = w.cout;
    push_step([=](cudaStream_t s) { return groupnorm_relu_grid_f16(tower_raw, 5, F, gs, c, 32, gw, gb, o, s); });
    return 0;
  };
  TMap g0, ka, kb, ca, cb;
  PRISMA_TRY(new_tmap(&g0, 320));
  PRISMA_TRY(new_tmap(&ka, 512)); PRISMA_TRY(new_tmap(&kb, 512));
  PRISMA_TRY(new_tmap(&ca, 512)); PRISMA_TRY(new_tmap(&cb, 512));
  for (int l = 0; l < 5; ++l) {
    const int S = num_grids[l];
    const SMap a = lvl_in[l];
    __half* dst = g0.p + (size_t)l * FP * 320;
    push_step([=](cudaStream_t s) { return resize_bilinear_f16(a.p, a.H, a.W, 256, dst, S, S, 320, 1, 0, s, F); });
  }
  PRISMA_TRY(gnconv_t(g0, 320, kconv[0], ka));
  PRISMA_TRY(gnconv_t(ka, 512, kconv[1], kb));
  PRISMA_TRY(gnconv_t(kb, 512, kconv[2], ka));
  PRISMA_TRY(gnconv_t(ka, 512, kconv[3], kb));
  { GemmEpilogue ep; ep.bias = conv_kernel.b; PRISMA_TRY(conv_t(kb, 512, conv_kernel, ep, ker_all)); }
  PRISMA_TRY(gnconv_t(g0, 256, cconv[0], ca));
  PRISMA_TRY(gnconv_t(ca, 512, cconv[1], cb));
  PRISMA_TRY(gnconv_t(cb, 512, cconv[2], ca));
  PRISMA_TRY(gnconv_t(ca, 512, cconv[3], cb));
  { GemmEpilogue ep; ep.bias = conv_cls.b; PRISMA_TRY(conv_t(cb, 512, conv_cls, ep, cls_all)); }
  } else {
  // ================================================================ fp32-class head (solo_exact.cu, gemm_prepare_tf32x3)
  cur_tag = "mask_feature_head";
  auto new_xmap = [&](XMap* mm, int h, int w, int c) -> int {
    mm->H = h; mm->W = w; mm->C = c;
    return s_alloc(plan_allocs, &mm->p, (size_t)mm->rows() * 2 * c);
  };
  // conv on a split map -> dense fp32 [H*W][Cout]; c_used = channels of the map that enter the product (multiple of 32)
  auto conv_x = [&](const XMap& in, int c_used, const SoloConvW3& w, GemmEpilogue ep, float* dst_dense) -> int {
    PRISMA_CHECK(c_used == w.cin32 && c_used <= in.C, "solo(exact): operand channels do not match the packed weights");
    int off[9], taps_n = w.k * w.k;
    if (w.k == 3) { for (int ky = 0; ky < 3; ++ky) for (int kx = 0; kx < 3; ++kx) off[ky * 3 + kx] = (ky - 1) * in.Wp() + (kx - 1); }
    else off[0] = 0;
    ep.in_w = in.Wp(); ep.in_h = in.Hp(); ep.img_rows = 0; ep.sub = 1; ep.pad = 1;
    ep.row_map = ROW_PAD2TOK; ep.out_f32 = dst_dense; ep.out_f32_ld = w.cout;
    GemmLaunch g;
    PRISMA_TRY(gemm_prepare_tf32x3(&g, in.p, in.rows(), c_used, in.C, w.w, round_up(w.cout, 256), (int)in.rows(), w.cout, taps_n, off,
                                   ep, num_sms));
    flops += 2.0 * in.H * (double)in.W * taps_n * w.cin * w.cout;
    push_step([g](cudaStream_t s) { return gemm_run(g, s); });
    return 0;
  };
  auto gnconv_x = [&](const XMap& in, int c_used, const SoloConvW3& w, const XMap* dst_map, float* dst_w3) -> int {
    GemmEpilogue ep;
    PRISMA_TRY(conv_x(in, c_used, w, ep, gn_raw));
    const int h = in.H, ww = in.W, c = w.cout; const float* gw = w.gn_w; const float* gb = w.gn_b;
    float* dm = dst_map ? dst_map->p : nullptr;
    push_step([=](cudaStream_t s) { return groupnorm_relu_split(gn_raw, h, ww, c, 32, gw, gb, gn_part, gn_stats, dm, dst_w3, s); });
    return 0;
  };
  // FPN levels as split maps: from the fp16 maps of the backbone (lo = 0), or -- tests -- from injected fp32 levels
  XMap PX[5];
  for (int i = 0; i < 5; ++i) {
    PRISMA_TRY(new_xmap(&PX[i], P[i].H, P[i].W, 256));
    PRISMA_TRY(s_alloc(plan_allocs, &d_feat_in[i], (size_t)P[i].H * P[i].W * 256));
    feat_h[i] = P[i].H; feat_w[i] = P[i].W;
    const SMap a = P[i]; const XMap o = PX[i]; const float* inj = d_feat_in[i]; const bool* flag = &inject;
    const float* dense = P_dense[i];  // exact backbone: the level is already fp32
    push_step([=](cudaStream_t s) {
      if (*flag) return solo_dense_to_split(inj, a.H, a.W, 256, o.p, 256, s);
      return dense ? solo_dense_to_split(dense, a.H, a.W, 256, o.p, 256, s) : solo_f16map_to_split(a.p, a.H, a.W, 256, o.p, 256, s);
    });
  }
  XMap accx;
  PRISMA_TRY(new_xmap(&accx, fh, fw, 128));
  PRISMA_TRY(gnconv_x(PX[0], 256, mf3[0][0], &accx, nullptr));
  for (int i = 1; i < 4; ++i) {
    XMap cur = PX[i];
    int c_used = 256;
    if (i == 3) {  // + generate_coordinate channels: 258 -> a 288-channel split map (zeros above 258)
      XMap cc;
      PRISMA_TRY(new_xmap(&cc, PX[3].H, PX[3].W, 288));
      const XMap a = PX[3];
      push_step([=](cudaStream_t s) { return resize_bilinear_split(a.p, a.H, a.W, 256, 256, cc.p, cc.H, cc.W, 288, 1, 0, s); });
      cur = cc; c_used = 288;
    }
    for (int j = 0; j < i; ++j) {
      XMap t, u;
      PRISMA_TRY(new_xmap(&t, cur.H, cur.W, 128));
      PRISMA_TRY(gnconv_x(cur, c_used, mf3[i][j], &t, nullptr));
      const bool last = j == i - 1;
      if (last) u = accx; else PRISMA_TRY(new_xmap(&u, 2 * t.H, 2 * t.W, 128));
      PRISMA_CHECK(u.H == 2 * t.H && u.W == 2 * t.W, "solo: FPN levels are not exact halvings (pad to a multiple of 32)");
      push_step([=](cudaStream_t s) { return resize_bilinear_split(t.p, t.H, t.W, 128, 128, u.p, u.H, u.W, 128, 0, last ? 1 : 0, s); });
      cur = u; c_used = 128;
    }
  }
  PRISMA_TRY(s_alloc(plan_allocs, &mfeat3, (size_t)round_up(HW, 256) * 3 * 256));
  PRISMA_TRY(gnconv_x(accx, 128, mf_pred3, nullptr, mfeat3));
  taps["mask_feats"] = {mfeat3, 6, HW, 256, 0};

  cur_tag = "towers";
  XMap R0x, R4x;
  PRISMA_TRY(new_xmap(&R0x, P[1].H, P[1].W, 256));
  PRISMA_TRY(new_xmap(&R4x, P[3].H, P[3].W, 256));
  { const XMap a = PX[0], o = R0x; push_step([=](cudaStream_t s) { return resize_bilinear_split(a.p, a.H, a.W, 256, 256, o.p, o.H, o.W, 256, 0, 0, s); }); }
  { const XMap a = PX[4], o = R4x; push_step([=](cudaStream_t s) { return resize_bilinear_split(a.p, a.H, a.W, 256, 256, o.p, o.H, o.W, 256, 0, 0, s); }); }
  const XMap lvl_inx[5] = {R0x, PX[1], PX[2], PX[3], R4x};
  struct TXMap { float* p; int C; };
  auto new_txmap = [&](TXMap* t, int c) -> int { t->C = c; return s_alloc(plan_allocs, &t->p, (size_t)5 * FP * 2 * c); };
  auto conv_tx = [&](const TXMap& in, int c_used, const SoloConvW3& w, GemmEpilogue ep, float* dst_dense) -> int {
    PRISMA_CHECK(c_used == w.cin32 && c_used <= in.C, "solo(exact): tower operand channels do not match the packed weights");
    int off[9];
    for (int ky = 0; ky < 3; ++ky) for (int kx = 0; kx < 3; ++kx) off[ky * 3 + kx] = (ky - 1) * (F + 2) + (kx - 1);
    ep.in_w = F + 2; ep.in_h = F + 2; ep.img_rows = FP; ep.sub = 1; ep.pad = 1;
    ep.row_map = ROW_PAD2TOK; ep.out_f32 = dst_dense; ep.out_f32_ld = w.cout;
    GemmLaunch g;
    PRISMA_TRY(gemm_prepare_tf32x3(&g, in.p, 5LL * FP, c_used, in.C, w.w, round_up(w.cout, 256), 5 * FP, w.cout, 9, off, ep, num_sms));
    double px = 0; for (int l = 0; l < 5; ++l) px += (double)num_grids[l] * num_grids[l];
    flops += 2.0 * px * 9 * w.cin * w.cout;
    push_step([g](cudaStream_t s) { return gemm_run(g, s); });
    return 0;
  };
  auto gnconv_tx = [&](const TXMap& in, int c_used, const SoloConvW3& w, const TXMap& out) -> int {
    GemmEpilogue ep;
    PRISMA_TRY(conv_tx(in, c_used, w, ep, tower_raw));
    const float* gw = w.gn_w; const float* gb = w.gn_b; float* o = out.p; const int c = w.cout;
    push_step([=](cudaStream_t s) { return groupnorm_relu_grid_split(tower_raw, 5, F, gs, c, 32, gw, gb, o, s); });
    return 0;
  };
  TXMap g0x, kax, kbx, cax, cbx;
  PRISMA_TRY(new_txmap(&g0x, 288));
  PRISMA_TRY(new_txmap(&kax, 512)); PRISMA_TRY(new_txmap(&kbx, 512));
  PRISMA_TRY(new_txmap(&cax, 512)); PRISMA_TRY(new_txmap(&cbx, 512));
  for (int l = 0; l < 5; ++l) {
    const int S = num_grids[l];
    const XMap a = lvl_inx[l];
    float* dst = g0x.p + (size_t)l * FP * 2 * 288;
    push_step([=](cudaStream_t s) { return resize_bilinear_split(a.p, a.H, a.W, 256, 256, dst, S, S, 288, 1, 0, s, F); });
  }
  PRISMA_TRY(gnconv_tx(g0x, 288, kconv3[0], kax));
  PRISMA_TRY(gnconv_tx(kax, 512, kconv3[1], kbx));
  PRISMA_TRY(gnconv_tx(kbx, 512, kconv3[2], kax));
  PRISMA_TRY(gnconv_tx(kax, 512, kconv3[3], kbx));
  { GemmEpilogue ep; ep.bias = conv_kernel3.b; PRISMA_TRY(conv_tx(kbx, 512, conv_kernel3, ep, ker_all)); }
  PRISMA_TRY(gnconv_tx(g0x, 256, cconv3[0], cax));
  PRISMA_TRY(gnconv_tx(cax, 512, cconv3[1], cbx));
  PRISMA_TRY(gnconv_tx(cbx, 512, cconv3[2], cax));
  PRISMA_TRY(gnconv_tx(cax, 512, cconv3[3], cbx));
  { GemmEpilogue ep; ep.bias = conv_cls3.b; PRISMA_TRY(conv_tx(cbx, 512, conv_cls3, ep, cls_all)); }
  }
  float* cls_out[5]; float* ker_out[5];
  for (int l = 0; l < 5; ++l) {
    cls_out[l] = cls_all + (size_t)l * F * F * SOLO_NC;
    ker_out[l] = ker_all + (size_t)l * F * F * 256;
    taps["cls" + std::to_string(l)] = {cls_out[l], 5, num_grids[l], SOLO_NC, F};
    taps["kernel" + std::to_string(l)] = {ker_out[l], 5, num_grids[l], 256, F};
  }

  cur_tag = "decode";
  // ---- decode (solov2_head.py:582-766)
  SoloCand *cand_raw = nullptr, *cand = nullptr;
  PRISMA_TRY(s_alloc(plan_allocs, &cand_raw, (size_t)SOLO_CAP));
  PRISMA_TRY(s_alloc(plan_allocs, &cand, (size_t)SOLO_CAP));
  PRISMA_TRY(s_alloc(plan_allocs, &d_count, 4));
  PRISMA_TRY(s_alloc(plan_allocs, &d_ntop, 4));
  PRISMA_TRY(s_alloc(plan_allocs, &d_nkeep, 4));
  PRISMA_TRY(s_alloc(plan_allocs, &d_top, (size_t)SOLO_NMS_PAD));
  PRISMA_TRY(s_alloc(plan_allocs, &d_keep, (size_t)SOLO_MAX));
  PRISMA_TRY(s_alloc(plan_allocs, &d_keep_label, (size_t)SOLO_MAX));
  PRISMA_TRY(s_alloc(plan_allocs, &d_keep_score, (size_t)SOLO_MAX));
  { int* cnt = d_count; push_step([=](cudaStream_t s) { PRISMA_CUDA_OK(cudaMemsetAsync(cnt, 0, 4, s)); return 0; }); }
  for (int l = 0; l < 5; ++l) {
    const float* lg = cls_out[l]; const int S = num_grids[l], c0 = cell0[l]; const float st = strides[l]; int* cnt = d_count;
    push_step([=](cudaStream_t s) { return solo_candidates(lg, S, c0, SOLO_NC, 0.1f, st, cand_raw, cnt, SOLO_CAP, s, F); });
  }
  { int* cnt = d_count; push_step([=](cudaStream_t s) { return solo_sort_candidates(cand_raw, cnt, SOLO_CAP, cand, s); }); }
  const float** d_lvl_ptr = nullptr; int* d_cell0 = nullptr;
  PRISMA_TRY(s_alloc(plan_allocs, &d_lvl_ptr, 8));
  PRISMA_TRY(s_alloc(plan_allocs, &d_cell0, 8));
  PRISMA_CUDA_OK(cudaMemcpy(d_lvl_ptr, ker_out, 5 * sizeof(float*), cudaMemcpyHostToDevice));
  PRISMA_CUDA_OK(cudaMemcpy(d_cell0, cell0, 5 * sizeof(int), cudaMemcpyHostToDevice));
  int* d_lvl_S = nullptr;
  PRISMA_TRY(s_alloc(plan_allocs, &d_lvl_S, 8));
  PRISMA_CUDA_OK(cudaMemcpy(d_lvl_S, num_grids, 5 * sizeof(int), cudaMemcpyHostToDevice));
  __half* bin = nullptr; float* inter = nullptr;
  PRISMA_TRY(s_alloc(plan_allocs, &bin, (size_t)SOLO_NMS_PAD * HW));
  PRISMA_TRY(s_alloc(plan_allocs, &inter, (size_t)SOLO_NMS_PAD * SOLO_NMS_PAD));
  d_masks = nullptr; d_masks_f = nullptr;
  if (!exact_head) {
    __half* kmat = nullptr;
    PRISMA_TRY(s_alloc(plan_allocs, &kmat, (size_t)SOLO_CAP * 256));
    { const int* cnt = d_count;
      push_step([=](cudaStream_t s) { return solo_gather_kernels(cand, cnt, SOLO_CAP, d_lvl_ptr, d_cell0, 5, SOLO_NC, 256, kmat, s, d_lvl_S, F); }); }
    // dynamic conv: mask_preds = sigmoid(kernels [n][256] . mask_feats [HW][256]^T) as one GEMM (solov2_head.py:717-722)
    __half* masks = nullptr;
    PRISMA_TRY(s_alloc(plan_allocs, &masks, (size_t)SOLO_CAP * HW));
    d_masks = masks;
    {
      GemmEpilogue ep; ep.act = 3; ep.out_f16 = masks; ep.out_f16_ld = HW; ep.m_dev = d_count;  // only the rows of real candidates
      GemmLaunch g;
      PRISMA_TRY(gemm_prepare(&g, kmat, SOLO_CAP, 256, 256, mfeat, round_up(HW, 256), SOLO_CAP, HW, 1, zero_off, ep, num_sms));
      flops += 2.0 * SOLO_CAP * (double)HW * 256;
      push_step([g](cudaStream_t s) { return gemm_run(g, s); });
    }
    { const int* cnt = d_count; const int hw = HW;
      push_step([=](cudaStream_t s) { return solo_mask_stats(masks, hw, 0.5f, cand, cnt, SOLO_CAP, s); });
      int* top = d_top; int* ntop = d_ntop;
      push_step([=](cudaStream_t s) { return solo_rank(cand, cnt, SOLO_CAP, SOLO_NMS_PRE, top, ntop, s); }); }
    { const int* top = d_top; const int* ntop = d_ntop; const int hw = HW;
      push_step([=](cudaStream_t s) { return solo_binarize(masks, hw, 0.5f, top, ntop, SOLO_NMS_PAD, bin, s); }); }
  } else {
    float* kmatx = nullptr;  // candidate kernels as split rows [cap][2 * 256]
    PRISMA_TRY(s_alloc(plan_allocs, &kmatx, (size_t)SOLO_CAP * 512));
    { const int* cnt = d_count;
      push_step([=](cudaStream_t s) { return solo_gather_kernels_split(cand, cnt, SOLO_CAP, d_lvl_ptr, d_cell0, 5, SOLO_NC, 256, kmatx, s, d_lvl_S, F); }); }
    float* masksf = nullptr;  // fp32 sigmoid mask predictions [cap][HW]
    PRISMA_TRY(s_alloc(plan_allocs, &masksf, (size_t)SOLO_CAP * HW));
    d_masks_f = masksf;
    {
      GemmEpilogue ep; ep.act = 6; ep.out_f32 = masksf; ep.out_f32_ld = HW; ep.m_dev = d_count;  // only the rows of real candidates
      GemmLaunch g;
      PRISMA_TRY(gemm_prepare_tf32x3(&g, kmatx, SOLO_CAP, 256, 256, mfeat3, round_up(HW, 256), SOLO_CAP, HW, 1, zero_off, ep, num_sms));
      flops += 2.0 * SOLO_CAP * (double)HW * 256;
      push_step([g](cudaStream_t s) { return gemm_run(g, s); });
    }
    { const int* cnt = d_count; const int hw = HW;
      push_step([=](cudaStream_t s) { return solo_mask_stats(masksf, hw, 0.5f, cand, cnt, SOLO_CAP, s); });
      int* top = d_top; int* ntop = d_ntop;
      push_step([=](cudaStream_t s) { return solo_rank(cand, cnt, SOLO_CAP, SOLO_NMS_PRE, top, ntop, s); }); }
    { const int* top = d_top; const int* ntop = d_ntop; const int hw = HW;
      push_step([=](cudaStream_t s) { return solo_binarize(masksf, hw, 0.5f, top, ntop, SOLO_NMS_PAD, bin, s); }); }
  }
  {  // inter_matrix = M M^T over binary masks (matrix_nms.py:70-71): exact in fp32 (counts < 2^24)
    GemmEpilogue ep; ep.out_f32 = inter; ep.out_f32_ld = SOLO_NMS_PAD;
    GemmLaunch g;
    PRISMA_TRY(gemm_prepare(&g, bin, SOLO_NMS_PAD, HW, HW, bin, SOLO_NMS_PAD, SOLO_NMS_PAD, SOLO_NMS_PAD, 1, zero_off, ep, num_sms));
    flops += 2.0 * SOLO_NMS_PAD * (double)SOLO_NMS_PAD * HW;
    push_step([g](cudaStream_t s) { return gemm_run(g, s); });
  }
  { const int* top = d_top; const int* ntop = d_ntop; int* keep = d_keep; float* ks = d_keep_score; int* kl = d_keep_label; int* nk = d_nkeep;
    push_step([=](cudaStream_t s) {
      return solo_matrix_nms(inter, SOLO_NMS_PAD, cand, top, ntop, SOLO_NC, 2.0f, 0.05f, SOLO_MAX, keep, ks, kl, nk, s); }); }
  PRISMA_TRY(s_alloc(plan_allocs, &d_union, (size_t)H * W));
  taps["resized"] = {d_resized, 3, nh * nw, 3, 0};
  taps["net_input"] = {d_net, 0, 3 * hp, wp, 0};
  taps["cand_count"] = {d_count, 4, 1, 1, 0};
  taps["n_top"] = {d_ntop, 4, 1, 1, 0};
  launches = (int)steps.size();
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  plan_H = H; plan_W = W;
  if (graph_exec) { cudaGraphExecDestroy(graph_exec); graph_exec = nullptr; }
  if (use_graph) {
    PRISMA_TRY(run(stream));  // warm: per-kernel attributes are set outside the capture
    PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
    cudaGraph_t graph = nullptr;
    PRISMA_CUDA_OK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    int r = 0;
    for (auto& st : steps) { r = st(stream); if (r != 0) break; }
    cudaError_t e = cudaStreamEndCapture(stream, &graph);
    if (r != 0) { if (graph) cudaGraphDestroy(graph); return r; }
    PRISMA_CUDA_OK(e);
    PRISMA_CUDA_OK(cudaGraphInstantiate(&graph_exec, graph, 0));
    cudaGraphDestroy(graph);
  }
  return 0;
}

int SoloEngine::run(cudaStream_t s) {
  if (graph_exec) { PRISMA_CUDA_OK(cudaGraphLaunch(graph_exec, s)); return 0; }
  for (auto& st : steps) PRISMA_TRY(st(s));
  return 0;
}

int SoloEngine::infer(const uint8_t* rgb, int H, int W, float confidence, uint8_t* union_out, int* n_out, float* scores_out,
                      int* labels_out, uint8_t* inst_masks_out, float* ms_out) {
  PRISMA_CHECK(rgb != nullptr && H > 0 && W > 0, "bad frame");
  NvtxRange nvtx_pass("prisma.mask_mmdet.infer");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_TRY(build_plan(H, W));
  if (inst_masks_out && !d_inst) PRISMA_TRY(s_alloc(plan_allocs, &d_inst, (size_t)SOLO_MAX * H * W));
  PRISMA_CUDA_OK(cudaMemcpyAsync(d_img, rgb, (size_t)H * W * 3, cudaMemcpyHostToDevice, stream));
  if (getenv("PRISMA_SOLO_PROFILE")) {  // per-stage device times of one ungraphed pass (stderr)
    std::map<std::string, float> acc;
    cudaEvent_t a, b2;
    cudaEventCreate(&a); cudaEventCreate(&b2);
    for (size_t i = 0; i < steps.size(); ++i) {
      cudaEventRecord(a, stream);
      PRISMA_TRY(steps[i](stream));
      cudaEventRecord(b2, stream);
      cudaEventSynchronize(b2);
      float ms = 0; cudaEventElapsedTime(&ms, a, b2);
      acc[step_tag[i]] += ms;
    }
    cudaEventDestroy(a); cudaEventDestroy(b2);
    for (auto& kv : acc) fprintf(stderr, "[solo-profile] %-20s %8.3f ms\n", kv.first.c_str(), kv.second);
  }
  PRISMA_CUDA_OK(cudaEventRecord(ev0, stream));
  PRISMA_TRY(run(stream));
  if (exact_head)
    PRISMA_TRY(solo_final_masks(d_masks_f, fh, fw, nh, nw, H, W, 0.5f, d_keep, d_keep_score, d_keep_label, d_nkeep, SOLO_MAX,
                                confidence, inst_masks_out ? d_inst : nullptr, d_union, stream));
  else
    PRISMA_TRY(solo_final_masks(d_masks, fh, fw, nh, nw, H, W, 0.5f, d_keep, d_keep_score, d_keep_label, d_nkeep, SOLO_MAX,
                                confidence, inst_masks_out ? d_inst : nullptr, d_union, stream));
  PRISMA_CUDA_OK(cudaEventRecord(ev1, stream));
  int n = 0, cnt = 0;
  PRISMA_CUDA_OK(cudaMemcpyAsync(&n, d_nkeep, 4, cudaMemcpyDeviceToHost, stream));
  PRISMA_CUDA_OK(cudaMemcpyAsync(&cnt, d_count, 4, cudaMemcpyDeviceToHost, stream));
  if (union_out) PRISMA_CUDA_OK(cudaMemcpyAsync(union_out, d_union, (size_t)H * W, cudaMemcpyDeviceToHost, stream));
  if (scores_out) PRISMA_CUDA_OK(cudaMemcpyAsync(scores_out, d_keep_score, SOLO_MAX * 4, cudaMemcpyDeviceToHost, stream));
  if (labels_out) PRISMA_CUDA_OK(cudaMemcpyAsync(labels_out, d_keep_label, SOLO_MAX * 4, cudaMemcpyDeviceToHost, stream));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  PRISMA_CHECK(cnt <= SOLO_CAP, "solo: more than 4096 grid cells passed score_thr (candidate capacity exceeded)");
  if (inst_masks_out && n > 0) PRISMA_CUDA_OK(cudaMemcpy(inst_masks_out, d_inst, (size_t)n * H * W, cudaMemcpyDeviceToHost));
  if (n_out) *n_out = n;
  if (ms_out) { float ms = 0; PRISMA_CUDA_OK(cudaEventElapsedTime(&ms, ev0, ev1)); *ms_out = ms; }
  return 0;
}

// ---- tests: head + decode replayed from given FPN levels (the reference's own levels, tests/golden/solo_tiny_head.npz)
int SoloEngine::inject_feat(int level, const float* nchw, int h, int w) {
  PRISMA_CHECK(exact_head, "feature injection exists for the fp32-class head only");
  PRISMA_CHECK(level >= 0 && level < 5 && d_feat_in[level] != nullptr, "no plan yet: call infer once at the frame size");
  PRISMA_CHECK(h == feat_h[level] && w == feat_w[level], "injected level has the wrong size for the planned frame");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  std::vector<float> nhwc((size_t)h * w * 256);
  for (int c = 0; c < 256; ++c)
    for (int p = 0; p < h * w; ++p) nhwc[(size_t)p * 256 + c] = nchw[(size_t)c * h * w + p];
  PRISMA_CUDA_OK(cudaMemcpy(d_feat_in[level], nhwc.data(), nhwc.size() * 4, cudaMemcpyHostToDevice));
  return 0;
}

int SoloEngine::infer_from_feats(int H, int W, int img_h, int img_w, float confidence, uint8_t* union_out, int* n_out,
                                 float* scores_out, int* labels_out, uint8_t* inst_masks_out) {
  PRISMA_CHECK(exact_head && plan_H == H && plan_W == W, "infer_from_feats: call infer once at this frame size first");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  if (inst_masks_out && !d_inst) PRISMA_TRY(s_alloc(plan_allocs, &d_inst, (size_t)SOLO_MAX * H * W));
  inject = true;  // the level-conversion steps read this flag when they run (here: directly, not through the graph)
  int r = 0;
  for (size_t i = head_step0; i < steps.size() && r == 0; ++i) r = steps[i](stream);
  inject = false;
  if (r != 0) return r;
  PRISMA_TRY(solo_final_masks(d_masks_f, fh, fw, img_h > 0 ? img_h : nh, img_w > 0 ? img_w : nw, H, W, 0.5f, d_keep, d_keep_score,
                              d_keep_label, d_nkeep, SOLO_MAX, confidence, inst_masks_out ? d_inst : nullptr, d_union, stream));
  int n = 0, cnt = 0;
  PRISMA_CUDA_OK(cudaMemcpyAsync(&n, d_nkeep, 4, cudaMemcpyDeviceToHost, stream));
  PRISMA_CUDA_OK(cudaMemcpyAsync(&cnt, d_count, 4, cudaMemcpyDeviceToHost, stream));
  if (union_out) PRISMA_CUDA_OK(cudaMemcpyAsync(union_out, d_union, (size_t)H * W, cudaMemcpyDeviceToHost, stream));
  if (scores_out) PRISMA_CUDA_OK(cudaMemcpyAsync(scores_out, d_keep_score, SOLO_MAX * 4, cudaMemcpyDeviceToHost, stream));
  if (labels_out) PRISMA_CUDA_OK(cudaMemcpyAsync(labels_out, d_keep_label, SOLO_MAX * 4, cudaMemcpyDeviceToHost, stream));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  PRISMA_CHECK(cnt <= SOLO_CAP, "solo: more than 4096 grid cells passed score_thr (candidate capacity exceeded)");
  if (inst_masks_out && n > 0) PRISMA_CUDA_OK(cudaMemcpy(inst_masks_out, d_inst, (size_t)n * H * W, cudaMemcpyDeviceToHost));
  if (n_out) *n_out = n;
  return 0;
}

long long SoloEngine::read_tap(const std::string& name, float* out, long long capacity) {
  auto it = taps.find(name);
  if (it == taps.end()) { set_last_error("unknown tap '" + name + "'"); return -1; }
  const SoloTap& t = it->second;
  cudaSetDevice(device);
  cudaStreamSynchronize(stream);
  if (t.kind == 0) {
    const long long n = (long long)t.a * t.b;
    if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
    if (cudaMemcpy(out, t.p, n * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    return n;
  }
  if (t.kind == 2) {
    const long long n = (long long)t.a * t.b;
    if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
    std::vector<__half> h(n);
    if (cudaMemcpy(h.data(), t.p, n * 2, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    for (long long i = 0; i < n; ++i) out[i] = __half2float(h[i]);
    return n;
  }
  if (t.kind == 6) {  // fp32 [a][3 b] rows = [hi | hi | lo] -> dense [a][b] values
    const long long n = (long long)t.a * t.b;
    if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
    std::vector<float> h((size_t)t.a * 3 * t.b);
    if (cudaMemcpy(h.data(), t.p, h.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    for (long long r = 0; r < t.a; ++r)
      for (int c = 0; c < t.b; ++c) out[r * t.b + c] = h[(size_t)r * 3 * t.b + c] + h[(size_t)r * 3 * t.b + 2 * t.b + c];
    return n;
  }
  if (t.kind == 3) {
    const long long n = (long long)t.a * t.b;
    if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
    std::vector<uint8_t> h(n);
    if (cudaMemcpy(h.data(), t.p, n, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    for (long long i = 0; i < n; ++i) out[i] = (float)h[i];
    return n;
  }
  if (t.kind == 5) {  // S x S grid of an F-wide dense fp32 frame: a = S, b = channels, c = F
    const long long n = (long long)t.a * t.a * t.b;
    if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
    std::vector<float> h((size_t)t.c * t.c * t.b);
    if (cudaMemcpy(h.data(), t.p, h.size() * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    for (int y = 0; y < t.a; ++y)
      for (int x = 0; x < t.a; ++x)
        for (int c = 0; c < t.b; ++c) out[((long long)y * t.a + x) * t.b + c] = h[((size_t)y * t.c + x) * t.b + c];
    return n;
  }
  if (t.kind == 4) {
    int v = 0;
    if (capacity < 1 || cudaMemcpy(&v, t.p, 4, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    out[0] = (float)v;
    return 1;
  }
  // padded fp16 map -> dense [H][W][C]
  const long long n = (long long)t.a * t.b * t.c;
  if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
  const long long tot = (long long)(t.a + 2) * (t.b + 2) * t.c;
  std::vector<__half> h(tot);
  if (cudaMemcpy(h.data(), t.p, tot * 2, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
  for (int y = 0; y < t.a; ++y)
    for (int x = 0; x < t.b; ++x)
      for (int c = 0; c < t.c; ++c)
        out[((long long)y * t.b + x) * t.c + c] = __half2float(h[((long long)(y + 1) * (t.b + 2) + x + 1) * t.c + c]);
  return n;
}

}  // namespace prisma
