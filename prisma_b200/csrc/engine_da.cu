// prisma_b200 -- Depth-Anything engine: weights -> kernel layouts, per-resolution launch plan, per-frame run.
//
// Replaces DPT_DINOv2.forward (bands/d_anything/dpt.py:155-166) and the pre/post-processing around it in
// bands/depth_anything.py:100-143,215-221 with the sm_100a kernels of this directory.  Data layout in HBM:
//   * residual stream x            fp32 [T][D]            (T = 1 + ph*pw tokens)
//   * every GEMM operand           fp16, K contiguous     (LayerNorm output, qkv, attention output, MLP hidden)
//   * DPT feature maps             fp16 NHWC with a one-pixel zero border, pixels flattened to rows, so a 3x3
//                                  conv is nine row-shifted GEMM slabs of the same 2-D TMA descriptor
//   * weights                      fp16 [N_pad][taps * ceil64(Cin)], biases / LayerScale / LayerNorm fp32
#include "engine_da.cuh"

#include <math.h>

#include <algorithm>
#include <cstring>

namespace prisma {

// ------------------------------------------------------------------------------------------------ helpers
struct DaCfg { int D, depth, heads, F, oc[4]; int family = FAMILY_DA; int hooks[4] = {0, 0, 0, 0}; bool metric = false; };
static bool da_cfg(const std::string& enc, DaCfg* c) {
  // MiDaS v3 DPT (hubconf DPT_Large -> DPTDepthModel(backbone="vitl16_384"): hooks [5,11,17,23], features 256,
  // reassemble channels [256,512,1024,1024]); "dpt_tiny" is a test-size twin of the same graph
  if (enc == "dpt_large") { *c = {1024, 24, 16, 256, {256, 512, 1024, 1024}, FAMILY_MIDAS, {5, 11, 17, 23}}; return true; }
  if (enc == "dpt_tiny") { *c = {384, 8, 6, 64, {48, 96, 192, 384}, FAMILY_MIDAS, {1, 3, 5, 7}}; return true; }
  if (enc == "zoe_vits") { *c = {384, 12, 6, 64, {48, 96, 192, 384}}; c->metric = true; return true; }
  if (enc == "zoe_vitl") { *c = {1024, 24, 16, 256, {256, 512, 1024, 1024}}; c->metric = true; return true; }
  if (enc == "vits") { *c = {384, 12, 6, 64, {48, 96, 192, 384}}; return true; }
  if (enc == "vitb") { *c = {768, 12, 12, 128, {96, 192, 384, 768}}; return true; }
  if (enc == "vitl") { *c = {1024, 24, 16, 256, {256, 512, 1024, 1024}}; return true; }
  return false;
}

// Resize.get_size, lower_bound / keep_aspect_ratio / multiple of 14 (d_anything/util/transform.py:111-166).
// np.round is round-half-even == nearbyint in the default rounding mode.
void da_net_size(int W, int H, int* wn, int* hn) {
  double sh = 518.0 / H, sw = 518.0 / W;
  if (sw > sh) sh = sw; else sw = sh;
  auto constrain = [](double x) {
    int y = (int)(nearbyint(x / 14.0) * 14.0);
    if (y < 518) y = (int)(ceil(x / 14.0) * 14.0);
    return y;
  };
  *hn = constrain(sh * H);
  *wn = constrain(sw * W);
}

// MiDaS transform = hubconf default_transform, which bands/depth_midas.py:37-40 selects for DPT_Large: the Resize class
// vendored in d_anything/util/transform.py (get_size :111-166, constrain_to_multiple_of :98-109) with
// resize_method="upper_bound", keep_aspect_ratio, multiple of 32, target 384 x 384: the frame is scaled to FIT 384 x 384.
void midas_net_size(int W, int H, int* wn, int* hn) {
  double sh = 384.0 / H, sw = 384.0 / W;
  if (sw < sh) sh = sw; else sw = sh;
  auto constrain = [](double x) {
    int y = (int)(nearbyint(x / 32.0) * 32.0);   // np.round: half to even, as nearbyint
    if (y > 384) y = (int)(floor(x / 32.0) * 32.0);
    return y;
  };
  *hn = constrain(sh * H);
  *wn = constrain(sw * W);
}

DepthEngine::~DepthEngine() {
  cudaSetDevice(device);
  for (void* p : allocs) cudaFree(p);
  for (void* p : plan_allocs) cudaFree(p);
  if (graph_exec) cudaGraphExecDestroy(graph_exec);
  if (ev0) cudaEventDestroy(ev0);
  if (ev1) cudaEventDestroy(ev1);
  for (auto& sl : slot) {
    cudaFree(sl.in); cudaFree(sl.rgb); cudaFree(sl.pred); cudaFree(sl.mm);
    for (cudaEvent_t e : {sl.loaded, sl.consumed, sl.done, sl.drained}) if (e) cudaEventDestroy(e);
  }
  if (mm_host) cudaFreeHost(mm_host);
  if (s_in) cudaStreamDestroy(s_in);
  if (s_out) cudaStreamDestroy(s_out);
  if (stream) cudaStreamDestroy(stream);
}

template <typename T>
static int dev_alloc(std::vector<void*>& pool, T** out, size_t n, bool zero = true) {
  void* p = nullptr;
  PRISMA_CUDA_OK(cudaMalloc(&p, std::max<size_t>(n * sizeof(T), 256)));
  if (zero) PRISMA_CUDA_OK(cudaMemset(p, 0, std::max<size_t>(n * sizeof(T), 256)));
  pool.push_back(p);
  *out = reinterpret_cast<T*>(p);
  return 0;
}

int DepthEngine::init(const std::string& enc, int dev) {
  DaCfg c;
  PRISMA_CHECK(da_cfg(enc, &c), "unknown encoder '" + enc + "' (vits|vitb|vitl|dpt_large)");
  encoder = enc;
  D = c.D; depth = c.depth; heads = c.heads; F = c.F;
  for (int i = 0; i < 4; ++i) { oc[i] = c.oc[i]; hooks[i] = c.hooks[i]; }
  family = c.family;
  metric = c.metric;
  if (family == FAMILY_MIDAS) { patch = 16; pos_grid = 24; }
  device = dev;
  int n = 0;
  PRISMA_CUDA_OK(cudaGetDeviceCount(&n));
  PRISMA_CHECK(dev >= 0 && dev < n, "bad device ordinal");
  PRISMA_CUDA_OK(cudaSetDevice(dev));
  cudaDeviceProp prop;
  PRISMA_CUDA_OK(cudaGetDeviceProperties(&prop, dev));
  PRISMA_CHECK(prop.major == 10, "prisma_b200 kernels are sm_100a only (found sm_" + std::to_string(prop.major) +
                                     std::to_string(prop.minor) + "); there is no fallback path");
  num_sms = prop.multiProcessorCount;
  PRISMA_CUDA_OK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  PRISMA_CUDA_OK(cudaEventCreate(&ev0));
  PRISMA_CUDA_OK(cudaEventCreate(&ev1));
  const char* ng = getenv("PRISMA_NO_GRAPH");
  use_graph = !(ng && ng[0] == '1');
  return 0;
}

int DepthEngine::load_tensor(const std::string& name, const float* data, const int64_t* shape, int ndim) {
  PRISMA_CHECK(!finalized, "load_tensor after finalize");
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
  t.data.assign(data, data + n);
  host[name] = std::move(t);
  return 0;
}

const HostTensor* DepthEngine::get(const std::string& name, std::initializer_list<int64_t> shape) {
  auto it = host.find(name);
  if (it == host.end()) { set_last_error("missing weight tensor '" + name + "'"); return nullptr; }
  if (shape.size()) {
    std::vector<int64_t> s(shape);
    if (s != it->second.shape) { set_last_error("weight tensor '" + name + "' has an unexpected shape"); return nullptr; }
  }
  return &it->second;
}

int DepthEngine::up_f32(const std::string& name, std::initializer_list<int64_t> shape, float** out, float scale_first_rows,
                        int n_scaled) {
  const HostTensor* t = get(name, shape);
  if (!t) return -1;
  std::vector<float> tmp(t->data);
  for (int i = 0; i < n_scaled && i < (int)tmp.size(); ++i) tmp[i] *= scale_first_rows;
  // pad to a multiple of 8 floats so vectorised epilogue loads never run off the end
  tmp.resize(round_up((int)tmp.size(), 8), 0.f);
  PRISMA_TRY(dev_alloc(allocs, out, tmp.size(), false));
  PRISMA_CUDA_OK(cudaMemcpy(*out, tmp.data(), tmp.size() * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

// fp16 [round_up(N,256)][Kpad] from a host fp32 functor w(n, k)
template <typename Fn>
static int up_matrix(std::vector<void*>& pool, __half** out, int N, int Kpad, Fn fn) {
  const int rows = round_up(N, 256);
  std::vector<__half> h((size_t)rows * Kpad, __float2half_rn(0.f));
  for (int n = 0; n < N; ++n) fn(n, h.data() + (size_t)n * Kpad);
  PRISMA_TRY(dev_alloc(pool, out, h.size(), false));
  PRISMA_CUDA_OK(cudaMemcpy(*out, h.data(), h.size() * sizeof(__half), cudaMemcpyHostToDevice));
  return 0;
}

int DepthEngine::up_linear(const std::string& name, int N, int K, __half** out, float scale, int n_scaled) {
  const HostTensor* t = get(name, {N, K});
  if (!t) return -1;
  const int Kpad = round_up(K, 64);
  return up_matrix(allocs, out, N, Kpad, [&](int n, __half* row) {
    const float s = n < n_scaled ? scale : 1.f;
    for (int k = 0; k < K; ++k) row[k] = __float2half_rn(t->data[(size_t)n * K + k] * s);
  });
}

int DepthEngine::up_conv(const std::string& name, int Cout, int Cin, int kh, int kw, __half** out) {
  const HostTensor* t = get(name, {Cout, Cin, kh, kw});
  if (!t) return -1;
  const int kc = ceil_div(Cin, 64), taps = kh * kw;
  return up_matrix(allocs, out, Cout, taps * kc * 64, [&](int n, __half* row) {
    for (int tp = 0; tp < taps; ++tp)
      for (int c = 0; c < Cin; ++c)
        row[(size_t)tp * kc * 64 + c] = __float2half_rn(t->data[((size_t)n * Cin + c) * taps + tp]);
  });
}

// ConvTranspose2d weight [Cin][Cout][s][s], kernel == stride: B[(dy*s+dx)*Cout + co][ci]
int DepthEngine::up_convT(const std::string& name, int Cin, int Cout, int s, __half** out, float** bias_out) {
  const HostTensor* t = get(name + ".weight", {Cin, Cout, s, s});
  const HostTensor* b = get(name + ".bias", {Cout});
  if (!t || !b) return -1;
  const int N = s * s * Cout, Kpad = round_up(Cin, 64);
  PRISMA_TRY(up_matrix(allocs, out, N, Kpad, [&](int n, __half* row) {
    const int q = n / Cout, co = n % Cout, dy = q / s, dx = q % s;
    for (int ci = 0; ci < Cin; ++ci)
      row[ci] = __float2half_rn(t->data[(((size_t)ci * Cout + co) * s + dy) * s + dx]);
  }));
  std::vector<float> be(round_up(N, 8), 0.f);
  for (int n = 0; n < N; ++n) be[n] = b->data[n % Cout];
  PRISMA_TRY(dev_alloc(allocs, bias_out, be.size(), false));
  PRISMA_CUDA_OK(cudaMemcpy(*bias_out, be.data(), be.size() * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

int DepthEngine::finalize() {
  PRISMA_CHECK(!finalized, "finalize called twice");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  const bool midas = family == FAMILY_MIDAS;
  const std::string core = metric ? "core.core." : "";  // ZoeDepth wraps the relative model (zoedepth_v1.py:68, DepthAnythingCore.core)
  const std::string p = midas ? "pretrained.model." : core + "pretrained.";
  const int n_pos = pos_grid * pos_grid + 1, pk = 3 * patch * patch, pkpad = round_up(pk, 64);
  PRISMA_TRY(up_f32(p + "cls_token", {1, 1, D}, &w.cls));
  PRISMA_TRY(up_f32(p + "pos_embed", {1, n_pos, D}, &w.pos));
  if (midas) {
    host_pos = get(p + "pos_embed", {1, n_pos, D})->data;
    host_cls = get(p + "cls_token", {1, 1, D})->data;
  }
  {
    const HostTensor* t = get(p + "patch_embed.proj.weight", {D, 3, patch, patch});
    if (!t) return -1;
    PRISMA_TRY(up_matrix(allocs, &w.patch_w, D, pkpad, [&](int n, __half* row) {
      for (int k = 0; k < pk; ++k) row[k] = __float2half_rn(t->data[(size_t)n * pk + k]);
    }));
    PRISMA_TRY(up_f32(p + "patch_embed.proj.bias", {D}, &w.patch_b));
  }
  w.blk.resize(depth);
  const float qscale = 0.125f;  // head_dim^-0.5, head_dim == 64 for every DINOv2 variant (attention.py:41-42)
  for (int i = 0; i < depth; ++i) {
    const std::string b = p + "blocks." + std::to_string(i) + ".";
    BlockW& k = w.blk[i];
    PRISMA_TRY(up_f32(b + "norm1.weight", {D}, &k.n1w));
    PRISMA_TRY(up_f32(b + "norm1.bias", {D}, &k.n1b));
    PRISMA_TRY(up_linear(b + "attn.qkv.weight", 3 * D, D, &k.qkv_w, qscale, D));
    PRISMA_TRY(up_f32(b + "attn.qkv.bias", {3 * D}, &k.qkv_b, qscale, D));
    PRISMA_TRY(up_linear(b + "attn.proj.weight", D, D, &k.proj_w));
    PRISMA_TRY(up_f32(b + "attn.proj.bias", {D}, &k.proj_b));
    k.g1 = k.g2 = nullptr;  // timm ViT blocks of MiDaS have no LayerScale
    if (!midas) PRISMA_TRY(up_f32(b + "ls1.gamma", {D}, &k.g1));
    PRISMA_TRY(up_f32(b + "norm2.weight", {D}, &k.n2w));
    PRISMA_TRY(up_f32(b + "norm2.bias", {D}, &k.n2b));
    PRISMA_TRY(up_linear(b + "mlp.fc1.weight", 4 * D, D, &k.fc1_w));
    PRISMA_TRY(up_f32(b + "mlp.fc1.bias", {4 * D}, &k.fc1_b));
    PRISMA_TRY(up_linear(b + "mlp.fc2.weight", D, 4 * D, &k.fc2_w));
    PRISMA_TRY(up_f32(b + "mlp.fc2.bias", {D}, &k.fc2_b));
    if (!midas) PRISMA_TRY(up_f32(b + "ls2.gamma", {D}, &k.g2));
  }
  w.nw = w.nb = nullptr;  // MiDaS hooks the raw block outputs; the final norm only feeds the unused `glob`
  if (!midas) {
    PRISMA_TRY(up_f32(p + "norm.weight", {D}, &w.nw));
    PRISMA_TRY(up_f32(p + "norm.bias", {D}, &w.nb));
  }

  // head tensor names: Depth-Anything DPTHead (d_anything/dpt.py:39-100) / MiDaS DPT (midas/backbones/vit.py
  // act_postprocessN = [readout, Transpose, Unflatten, Conv1x1, resize], midas/dpt_depth.py scratch.*)
  const std::string h = core + "depth_head.";
  auto pp = [&](int i) { return "pretrained.act_postprocess" + std::to_string(i + 1) + "."; };
  if (midas)
    for (int i = 0; i < 4; ++i) {
      PRISMA_TRY(up_linear(pp(i) + "0.project.0.weight", D, 2 * D, &w.ro_w[i]));
      PRISMA_TRY(up_f32(pp(i) + "0.project.0.bias", {D}, &w.ro_b[i]));
    }
  for (int i = 0; i < 4; ++i) {
    const std::string n = midas ? pp(i) + "3" : h + "projects." + std::to_string(i);
    const HostTensor* t = get(n + ".weight", {oc[i], D, 1, 1});
    if (!t) return -1;
    const int K = D, N = oc[i];
    PRISMA_TRY(up_matrix(allocs, &w.proj_w[i], N, round_up(K, 64), [&](int r, __half* row) {
      for (int k = 0; k < K; ++k) row[k] = __float2half_rn(t->data[(size_t)r * K + k]);
    }));
    PRISMA_TRY(up_f32(n + ".bias", {oc[i]}, &w.proj_b[i]));
  }
  PRISMA_TRY(up_convT(midas ? pp(0) + "4" : h + "resize_layers.0", oc[0], oc[0], 4, &w.rs0_w, &w.rs0_b));
  PRISMA_TRY(up_convT(midas ? pp(1) + "4" : h + "resize_layers.1", oc[1], oc[1], 2, &w.rs1_w, &w.rs1_b));
  PRISMA_TRY(up_conv((midas ? pp(3) + "4" : h + "resize_layers.3") + ".weight", oc[3], oc[3], 3, 3, &w.rs3_w));
  PRISMA_TRY(up_f32((midas ? pp(3) + "4" : h + "resize_layers.3") + ".bias", {oc[3]}, &w.rs3_b));
  const std::string s = midas ? "scratch." : h + "scratch.";
  const std::string o1 = s + (midas ? "output_conv.0" : "output_conv1"), o2 = s + (midas ? "output_conv.2" : "output_conv2.0"),
                    o3 = s + (midas ? "output_conv.4" : "output_conv2.2");
  for (int i = 0; i < 4; ++i)
    PRISMA_TRY(up_conv(s + "layer" + std::to_string(i + 1) + "_rn.weight", F, oc[i], 3, 3, &w.rn_w[i]));
  for (int i = 0; i < 4; ++i) {
    const std::string r = s + "refinenet" + std::to_string(i + 1) + ".";
    RefineW& k = w.ref[i];
    {
      const HostTensor* t = get(r + "out_conv.weight", {F, F, 1, 1});
      if (!t) return -1;
      PRISMA_TRY(up_matrix(allocs, &k.out_w, F, round_up(F, 64), [&](int n, __half* row) {
        for (int c = 0; c < F; ++c) row[c] = __float2half_rn(t->data[(size_t)n * F + c]);
      }));
      PRISMA_TRY(up_f32(r + "out_conv.bias", {F}, &k.out_b));
    }
    for (int u = 0; u < 2; ++u) {
      if (i == 3 && u == 0) continue;  // refinenet4.resConfUnit1 exists but is never used (dpt.py:127)
      const std::string ru = r + "resConfUnit" + std::to_string(u + 1) + ".";
      PRISMA_TRY(up_conv(ru + "conv1.weight", F, F, 3, 3, &k.c1_w[u]));
      PRISMA_TRY(up_f32(ru + "conv1.bias", {F}, &k.c1_b[u]));
      PRISMA_TRY(up_conv(ru + "conv2.weight", F, F, 3, 3, &k.c2_w[u]));
      PRISMA_TRY(up_f32(ru + "conv2.bias", {F}, &k.c2_b[u]));
    }
  }
  PRISMA_TRY(up_conv(o1 + ".weight", F / 2, F, 3, 3, &w.oc1_w));
  PRISMA_TRY(up_f32(o1 + ".bias", {F / 2}, &w.oc1_b));
  PRISMA_TRY(up_conv(o2 + ".weight", 32, F / 2, 3, 3, &w.oc2_w));
  PRISMA_TRY(up_f32(o2 + ".bias", {32}, &w.oc2_b));
  PRISMA_TRY(up_f32(o3 + ".weight", {1, 32, 1, 1}, &w.oc3_w));
  {
    const HostTensor* t = get(o3 + ".bias", {1});
    if (!t) return -1;
    w.oc3_b = t->data[0];
  }
  if (metric) {
    PRISMA_TRY(up_lin1x1("conv2", F, F, &w.z_conv2));
    PRISMA_TRY(up_lin1x1("seed_bin_regressor._net.0", 256, F, &w.z_seed0));
    PRISMA_TRY(up_lin1x1("seed_bin_regressor._net.2", 64, 256, &w.z_seed2));
    PRISMA_TRY(up_lin1x1("seed_projector._net.0", 128, F, &w.z_sproj0));
    PRISMA_TRY(up_lin1x1("seed_projector._net.2", 128, 128, &w.z_sproj2));
    const int n_attr[4] = {16, 8, 4, 1};
    for (int i = 0; i < 4; ++i) {
      const std::string si = std::to_string(i);
      PRISMA_TRY(up_lin1x1("projectors." + si + "._net.0", 128, F, &w.z_proj0[i]));
      PRISMA_TRY(up_lin1x1("projectors." + si + "._net.2", 128, 128, &w.z_proj2[i]));
      PRISMA_TRY(up_lin1x1("attractors." + si + "._net.0", 128, 128, &w.z_att0[i]));
      PRISMA_TRY(up_lin1x1("attractors." + si + "._net.2", n_attr[i], 128, &w.z_att2[i]));
    }
    PRISMA_TRY(up_lin1x1("conditional_log_binomial.mlp.0", 80, 161, &w.z_clb0));
    PRISMA_TRY(up_lin1x1("conditional_log_binomial.mlp.2", 4, 80, &w.z_clb2));
  }
  host.clear();
  finalized = true;
  return 0;
}

// 1x1 conv weight [N][K][1][1] + bias -> fp16 [round_up(N,256)][round_up(K,64)], fp32 bias padded to a multiple of 8
int DepthEngine::up_lin1x1(const std::string& name, int N, int K, DaWeights::Lin* out) {
  const HostTensor* t = get(name + ".weight", {N, K, 1, 1});
  if (!t) return -1;
  PRISMA_TRY(up_matrix(allocs, &out->w, N, round_up(K, 64), [&](int n, __half* row) {
    for (int k = 0; k < K; ++k) row[k] = __float2half_rn(t->data[(size_t)n * K + k]);
  }));
  PRISMA_TRY(up_f32(name + ".bias", {N}, &out->b));
  out->n = N; out->k = K;
  return 0;
}

// ------------------------------------------------------------------------------------------------ plan
struct PMap {  // B zero-bordered NHWC fp16 feature maps, stacked image-major
  __half* p = nullptr;
  int B = 1, H = 0, W = 0, C = 0;
  int Hp() const { return H + 2; }
  int Wp() const { return W + 2; }
  long long img_rows() const { return (long long)Hp() * Wp(); }
  long long rows() const { return B * img_rows(); }
};

int DepthEngine::new_map(PMap* m, int H, int W, int C) {  // `batch` images
  m->B = batch; m->H = H; m->W = W; m->C = C;
  // +GEMM_BM rows of slack: TMA boxes never need it (OOB reads are zero-filled) but debug reads may
  return dev_alloc(plan_allocs, &m->p, (size_t)m->rows() * C, true);
}

void DepthEngine::add(int group, const char* name, std::function<int(cudaStream_t)> fn) {
  steps.push_back({group, name, std::move(fn)});
}

int DepthEngine::add_gemm(int group, const char* name, const __half* A, long long a_rows, int a_cols, int a_pitch,
                          const __half* W, int M, int N, int taps, const int* tap_off, const GemmEpilogue& ep,
                          double flops) {
  GemmLaunch g;
  PRISMA_TRY(gemm_prepare(&g, A, a_rows, a_cols, a_pitch, W, round_up(N, 256), M, N, taps, tap_off, ep, num_sms));
  if (group == G_LINEAR) work_linear += flops; else work_head += flops;
  add(group, name, [g](cudaStream_t s) { return gemm_run(g, s); });
  return 0;
}

// 3x3 stride-1 'same' conv on a padded map, output in the same padded geometry (or subsampled by `sub`)
int DepthEngine::add_conv3x3(const char* name, const PMap& in, const __half* W, int Cout, GemmEpilogue ep, int sub,
                             const PMap* out_geom) {
  int off[9];
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) off[ky * 3 + kx] = (ky - 1) * in.Wp() + (kx - 1);
  ep.row_map = ROW_PADDED;
  ep.in_w = in.Wp();
  ep.in_h = in.Hp();
  ep.img_rows = (int)in.img_rows();
  ep.sub = sub;
  if (sub > 1) { ep.out_wp = out_geom->Wp(); ep.out_img_rows = (int)out_geom->img_rows(); }
  const double flops = 2.0 * in.B * (double)(in.H / sub + (in.H % sub ? 1 : 0)) * (in.W / sub + (in.W % sub ? 1 : 0)) * 9.0 * in.C * Cout;
  return add_gemm(G_HEAD, name, in.p, in.rows(), in.C, in.C, W, (int)in.rows(), Cout, 9, off, ep, flops);
}

int DepthEngine::build_plan(int H, int W, int Bt) {
  PRISMA_CHECK(finalized, "weights not finalized");
  PRISMA_CHECK(Bt >= 1 && Bt <= 64, "batch must be in [1,64]");
  if (plan_H == H && plan_W == W && batch == Bt) return 0;
  plan_W_req = W;
  batch = Bt;
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  for (void* q : plan_allocs) cudaFree(q);
  plan_allocs.clear();
  steps.clear();
  taps.clear();
  work_linear = work_attn = work_head = 0;
  plan_H = plan_W = 0;

  const bool midas = family == FAMILY_MIDAS;
  if (midas) midas_net_size(W, H, &wn, &hn);
  else if (metric) { hn = 392; wn = 518; }  // config_zoedepth.json img_size, keep_aspect_ratio False (PrepForMidas)
  else da_net_size(W, H, &wn, &hn);
  PRISMA_CHECK(hn >= patch * 2 && wn >= patch * 2, "frame too small for the network input");
  ph = hn / patch; pw = wn / patch;
  const int pkpad = round_up(3 * patch * patch, 64);
  const int P = ph * pw;
  T = P + 1;
  const int BP = Bt * P, BT = Bt * T;
  const int zero_off[1] = {0};

  // ---- frame-level buffers
  PRISMA_TRY(dev_alloc(plan_allocs, &b.img, (size_t)Bt * H * W * 3));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.net_in, (size_t)Bt * 3 * hn * wn));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.patches, (size_t)BP * pkpad));
  if (midas) PRISMA_TRY(dev_alloc(plan_allocs, &ro_cat, (size_t)BP * 2 * D));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.pos, (size_t)BT * D));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.x, (size_t)BT * D));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.tokens_tap, (size_t)BT * D));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.ln, (size_t)BT * D));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.qkv, (size_t)BT * 3 * D));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.attn, (size_t)BT * D));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.hid, (size_t)BT * 4 * D));
  for (int i = 0; i < 4; ++i) PRISMA_TRY(dev_alloc(plan_allocs, &b.feat[i], (size_t)BP * D));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.depth, (size_t)Bt * hn * wn));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.pred, (size_t)Bt * H * W));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.rgb, (size_t)Bt * H * W * 3));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.mm, 2 * Bt));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.minmax, 2 * Bt));
  PRISMA_TRY(dev_alloc(plan_allocs, &b.mag, 2));

  // pos-embed for this resolution (constant per resolution): computed once, here
  if (!midas) {
    PRISMA_TRY(da_pos_embed(w.pos, w.cls, 37, D, ph, pw, b.pos, stream));
  } else {
    // _resize_pos_embed (midas/backbones/vit.py): F.interpolate(grid, size=(ph, pw), mode="bilinear"), align_corners
    // False: src = (dst + 0.5) * in/out - 0.5 clamped at 0, fp32; row 0 = cls + pos[0]
    std::vector<float> pe((size_t)T * D);
    const int S = pos_grid;
    for (int d = 0; d < D; ++d) pe[d] = host_cls[d] + host_pos[d];
    const float scy = (float)S / (float)ph, scx = (float)S / (float)pw;
    for (int oy = 0; oy < ph; ++oy) {
      const float ry = std::max(scy * (oy + 0.5f) - 0.5f, 0.f);
      const int y0 = (int)ry, y1 = y0 + (y0 < S - 1 ? 1 : 0);
      const float ly = ry - y0, hy = 1.f - ly;
      for (int ox = 0; ox < pw; ++ox) {
        const float rx = std::max(scx * (ox + 0.5f) - 0.5f, 0.f);
        const int x0 = (int)rx, x1 = x0 + (x0 < S - 1 ? 1 : 0);
        const float lx = rx - x0, hx = 1.f - lx;
        const float* g = host_pos.data() + D;  // grid part
        float* o = pe.data() + (size_t)(1 + oy * pw + ox) * D;
        for (int d = 0; d < D; ++d)
          o[d] = hy * (hx * g[(size_t)(y0 * S + x0) * D + d] + lx * g[(size_t)(y0 * S + x1) * D + d]) +
                 ly * (hx * g[(size_t)(y1 * S + x0) * D + d] + lx * g[(size_t)(y1 * S + x1) * D + d]);
      }
    }
    PRISMA_CUDA_OK(cudaMemcpyAsync(b.pos, pe.data(), pe.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
    PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  }
  for (int i = 1; i < Bt; ++i)  // one copy per image so that residual rows and destination rows coincide
    PRISMA_CUDA_OK(cudaMemcpyAsync(b.pos + (size_t)i * T * D, b.pos, (size_t)T * D * sizeof(float), cudaMemcpyDeviceToDevice, stream));

  // ---- pre-process + patch embed
  {
    const uint8_t* img = b.img; float* net = b.net_in; __half* pat = b.patches;
    const int hn_ = hn, wn_ = wn;
    const bool metric_ = metric;
    add(G_PRE, "da_preprocess", [=](cudaStream_t s) {
      for (int i = 0; i < Bt; ++i) {
        if (metric_) PRISMA_TRY(zoe_preprocess(img + (size_t)i * H * W * 3, H, W, net + (size_t)i * 3 * hn_ * wn_, hn_, wn_, s));
        else PRISMA_TRY(da_preprocess(img + (size_t)i * H * W * 3, H, W, net + (size_t)i * 3 * hn_ * wn_, hn_, wn_, s, midas));
      }
      return 0;
    });
    const int patch_ = patch;
    add(G_PRE, "patchify", [=](cudaStream_t s) { return da_patchify(net, Bt, hn_, wn_, pat, pkpad, s, patch_); });
    GemmEpilogue ep;
    ep.bias = w.patch_b;
    ep.row_map = ROW_TOKSKIP; ep.in_w = P;       // patch rows b*P+p -> token rows b*T+1+p
    ep.res_f32 = b.pos; ep.res_f32_ld = D;       // + pos-embed of the same token row
    ep.out_f32 = b.x; ep.out_f32_ld = D;
    PRISMA_TRY(add_gemm(G_LINEAR, "patch_embed", b.patches, BP, pkpad, pkpad, w.patch_w, BP, D, 1, zero_off, ep,
                        2.0 * BP * D * 3.0 * patch * patch));
    float* x = b.x; const float* pos = b.pos; const int D_ = D, T_ = T;
    add(G_PRE, "cls_rows", [=](cudaStream_t s) {  // token 0 of every image = cls + pos[0]
      PRISMA_CUDA_OK(cudaMemcpy2DAsync(x, (size_t)T_ * D_ * sizeof(float), pos, (size_t)T_ * D_ * sizeof(float),
                                       D_ * sizeof(float), Bt, cudaMemcpyDeviceToDevice, s));
      return 0;
    });
    if (debug_taps) {
      float* tap = b.tokens_tap; const size_t n = (size_t)BT * D;
      add(G_PRE, "tap_tokens", [=](cudaStream_t s) {
        PRISMA_CUDA_OK(cudaMemcpyAsync(tap, x, n * sizeof(float), cudaMemcpyDeviceToDevice, s));
        return 0;
      });
    }
  }
  // ---- transformer blocks
  AttnLaunch att;
  PRISMA_TRY(attention_prepare(&att, b.qkv, b.attn, Bt, T, heads, D));
  for (int i = 0; i < depth; ++i) {
    const BlockW& k = w.blk[i];
    const float* x = b.x; __half* ln = b.ln; const int T_ = BT, D_ = D;
    add(G_LN, "ln1", [=](cudaStream_t s) { return layernorm_f16(x, k.n1w, k.n1b, ln, T_, D_, 1e-6f, s); });
    // qkv and fc1 write dense fp16 rows: bias (+ GELU) in the row-per-lane registers, then TMA bulk stores -- no staging
    // read-back, no per-lane global stores (the epilogue, not the MMA, paces these launches: DESIGN 4.1)
    { GemmEpilogue ep; ep.bias = k.qkv_b; ep.out_f16 = b.qkv; ep.out_f16_ld = 3 * D; ep.tma_store = BT >= 1024;
      PRISMA_TRY(add_gemm(G_LINEAR, "qkv", b.ln, BT, D, D, k.qkv_w, BT, 3 * D, 1, zero_off, ep, 2.0 * BT * 3.0 * D * D)); }
    work_attn += att.flops;
    add(G_ATTN, "attention", [att](cudaStream_t s) { return attention_run(att, s); });
    // proj / fc2 update the fp32 token stream in place: gamma (acc + bias) is staged and added by TMA reduce-add stores
    // (the add happens in the L2; the epilogue reads nothing)
    { GemmEpilogue ep; ep.bias = k.proj_b; ep.gamma = k.g1; ep.res_f32 = b.x; ep.res_f32_ld = D; ep.out_f32 = b.x; ep.out_f32_ld = D;
      ep.tma_store = BT >= 1024;
      PRISMA_TRY(add_gemm(G_LINEAR, "proj", b.attn, BT, D, D, k.proj_w, BT, D, 1, zero_off, ep, 2.0 * BT * (double)D * D)); }
    add(G_LN, "ln2", [=](cudaStream_t s) { return layernorm_f16(x, k.n2w, k.n2b, ln, T_, D_, 1e-6f, s); });
    { GemmEpilogue ep; ep.bias = k.fc1_b; ep.act = 1; ep.out_f16 = b.hid; ep.out_f16_ld = 4 * D; ep.tma_store = BT >= 1024;
      PRISMA_TRY(add_gemm(G_LINEAR, "fc1", b.ln, BT, D, D, k.fc1_w, BT, 4 * D, 1, zero_off, ep, 2.0 * BT * 4.0 * D * D)); }
    { GemmEpilogue ep; ep.bias = k.fc2_b; ep.gamma = k.g2; ep.res_f32 = b.x; ep.res_f32_ld = D; ep.out_f32 = b.x; ep.out_f32_ld = D;
      ep.tma_store = BT >= 1024;
      PRISMA_TRY(add_gemm(G_LINEAR, "fc2", b.hid, BT, 4 * D, 4 * D, k.fc2_w, BT, D, 1, zero_off, ep, 2.0 * BT * 4.0 * D * D)); }
    if (!midas && i >= depth - 4) {
      __half* f = b.feat[i - (depth - 4)];
      const float* nw = w.nw; const float* nb = w.nb;
      // final norm of the tapped block, patch tokens only (use_clstoken=False, dpt.py:110-111): dense [B*P][D]
      add(G_LN, "ln_out", [=](cudaStream_t s) { return layernorm_f16(x, nw, nb, f, BP, D_, 1e-6f, s, P); });
    }
    if (midas)
      for (int hk = 0; hk < 4; ++hk)
        if (hooks[hk] == i) {
          // forward hook on blocks[i] (raw block output) -> ProjectReadout: GELU(Linear([token | cls]))
          __half* cat = ro_cat; const int Tt = T;
          add(G_LN, "readout_concat", [=](cudaStream_t s) { return readout_concat_f16(x, Bt, Tt, D_, cat, s); });
          GemmEpilogue ep; ep.bias = w.ro_b[hk]; ep.act = 1; ep.out_f16 = b.feat[hk]; ep.out_f16_ld = D;
          PRISMA_TRY(add_gemm(G_HEAD, "readout_project", ro_cat, BP, 2 * D, 2 * D, w.ro_w[hk], BP, D, 1, zero_off, ep,
                              2.0 * BP * 2.0 * D * D));
        }
  }

  // ---- DPT head (dpt.py:103-136), all maps zero-bordered NHWC fp16
  PMap L[4], R[4], Rr[4];
  const int h4 = (ph - 1) / 2 + 1, w4 = (pw - 1) / 2 + 1;
  PRISMA_CHECK(!midas || (ph % 2 == 0 && pw % 2 == 0), "MiDaS input sides are multiples of 32");
  PRISMA_TRY(new_map(&L[0], 4 * ph, 4 * pw, oc[0]));
  PRISMA_TRY(new_map(&L[1], 2 * ph, 2 * pw, oc[1]));
  PRISMA_TRY(new_map(&L[2], ph, pw, oc[2]));
  PRISMA_TRY(new_map(&L[3], h4, w4, oc[3]));
  PMap L3pre;
  PRISMA_TRY(new_map(&L3pre, ph, pw, oc[3]));
  for (int i = 0; i < 4; ++i) {
    PRISMA_TRY(new_map(&R[i], L[i].H, L[i].W, F));
    PRISMA_TRY(new_map(&Rr[i], L[i].H, L[i].W, F));
  }
  // projects (1x1 conv on tokens = GEMM over the patch tokens, cls dropped) + resize layers
  for (int i = 0; i < 4; ++i) {
    const __half* A = b.feat[i];  // patch tokens of all images, cls rows already dropped
    if (i < 2) {
      __half* dense = nullptr;
      PRISMA_TRY(dev_alloc(plan_allocs, &dense, (size_t)BP * oc[i]));
      { GemmEpilogue ep; ep.bias = w.proj_b[i]; ep.out_f16 = dense; ep.out_f16_ld = oc[i];
        PRISMA_TRY(add_gemm(G_HEAD, "project", A, BP, D, D, w.proj_w[i], BP, oc[i], 1, zero_off, ep, 2.0 * BP * (double)D * oc[i])); }
      const int s = i == 0 ? 4 : 2;
      GemmEpilogue ep;
      ep.bias = i == 0 ? w.rs0_b : w.rs1_b;
      ep.out_f16 = L[i].p; ep.out_f16_ld = oc[i];
      ep.row_map = ROW_SHUFFLE; ep.in_w = pw; ep.in_h = ph; ep.out_wp = L[i].Wp(); ep.out_img_rows = (int)L[i].img_rows();
      ep.shuf_s = s; ep.shuf_cout = oc[i];
      PRISMA_TRY(add_gemm(G_HEAD, "resize_convT", dense, BP, oc[i], oc[i], i == 0 ? w.rs0_w : w.rs1_w, BP, s * s * oc[i], 1,
                          zero_off, ep, 2.0 * BP * (double)oc[i] * s * s * oc[i]));
    } else {
      const PMap& dst = i == 2 ? L[2] : L3pre;
      GemmEpilogue ep; ep.bias = w.proj_b[i]; ep.out_f16 = dst.p; ep.out_f16_ld = oc[i];
      ep.row_map = ROW_TOK2PAD; ep.in_w = pw; ep.in_h = ph; ep.out_wp = dst.Wp(); ep.out_img_rows = (int)dst.img_rows();
      PRISMA_TRY(add_gemm(G_HEAD, "project", A, BP, D, D, w.proj_w[i], BP, oc[i], 1, zero_off, ep, 2.0 * BP * (double)D * oc[i]));
    }
  }
  { GemmEpilogue ep; ep.bias = w.rs3_b; ep.out_f16 = L[3].p; ep.out_f16_ld = oc[3];
    PRISMA_TRY(add_conv3x3("resize_conv_s2", L3pre, w.rs3_w, oc[3], ep, 2, &L[3])); }
  // layerN_rn: 3x3, no bias; write x and relu(x) (the RCUs take relu(x) as operand and x as skip)
  for (int i = 0; i < 4; ++i) {
    GemmEpilogue ep; ep.out_f16 = R[i].p; ep.out_f16_ld = F; ep.out_f16_relu = Rr[i].p; ep.out_f16_relu_ld = F;
    PRISMA_TRY(add_conv3x3("layer_rn", L[i], w.rn_w[i], F, ep, 1, nullptr));
  }
  // refinenet4..1 (blocks.py:126-153).  The 1x1 out_conv commutes with the bilinear resize (both linear, the
  // interpolation weights sum to 1), so it runs before the resize on 4x fewer pixels.
  PMap path;  // output of the previous fusion block (already resized to this level)
  PMap r_maps[4];  // refinenet4..1 outputs (the r4..r1 hooks of the metric head)
  for (int lvl = 3; lvl >= 0; --lvl) {
    const RefineW& k = w.ref[lvl];
    PMap t1, S, Sr, U, V;
    PRISMA_TRY(new_map(&t1, R[lvl].H, R[lvl].W, F));
    PRISMA_TRY(new_map(&U, R[lvl].H, R[lvl].W, F));
    PRISMA_TRY(new_map(&V, R[lvl].H, R[lvl].W, F));
    const PMap* in = &R[lvl];
    const PMap* in_relu = &Rr[lvl];
    if (lvl != 3) {
      // output = path + RCU1(R) ; RCU1(R) = conv2(relu(conv1(relu(R)))) + R
      PRISMA_TRY(new_map(&S, R[lvl].H, R[lvl].W, F));
      PRISMA_TRY(new_map(&Sr, R[lvl].H, R[lvl].W, F));
      { GemmEpilogue ep; ep.bias = k.c1_b[0]; ep.act = 2; ep.out_f16 = t1.p; ep.out_f16_ld = F;
        PRISMA_TRY(add_conv3x3("rcu1_conv1", Rr[lvl], k.c1_w[0], F, ep, 1, nullptr)); }
      { GemmEpilogue ep; ep.bias = k.c2_b[0]; ep.res_a = R[lvl].p; ep.res_a_ld = F; ep.res_b = path.p; ep.res_b_ld = F;
        ep.out_f16 = S.p; ep.out_f16_ld = F; ep.out_f16_relu = Sr.p; ep.out_f16_relu_ld = F;
        PRISMA_TRY(add_conv3x3("rcu1_conv2", t1, k.c2_w[0], F, ep, 1, nullptr)); }
      in = &S; in_relu = &Sr;
    }
    { GemmEpilogue ep; ep.bias = k.c1_b[1]; ep.act = 2; ep.out_f16 = t1.p; ep.out_f16_ld = F;
      PRISMA_TRY(add_conv3x3("rcu2_conv1", *in_relu, k.c1_w[1], F, ep, 1, nullptr)); }
    { GemmEpilogue ep; ep.bias = k.c2_b[1]; ep.res_a = in->p; ep.res_a_ld = F; ep.out_f16 = U.p; ep.out_f16_ld = F;
      PRISMA_TRY(add_conv3x3("rcu2_conv2", t1, k.c2_w[1], F, ep, 1, nullptr)); }
    { GemmEpilogue ep; ep.bias = k.out_b; ep.out_f16 = V.p; ep.out_f16_ld = F;
      ep.row_map = ROW_PADDED; ep.in_w = U.Wp(); ep.in_h = U.Hp(); ep.img_rows = (int)U.img_rows();
      PRISMA_TRY(add_gemm(G_HEAD, "out_conv1x1", U.p, U.rows(), F, F, k.out_w, (int)U.rows(), F, 1, zero_off, ep,
                          2.0 * Bt * U.H * (double)U.W * F * F)); }
    const int oh = lvl > 0 ? R[lvl - 1].H : 2 * R[0].H, ow = lvl > 0 ? R[lvl - 1].W : 2 * R[0].W;
    PMap nxt;
    PRISMA_TRY(new_map(&nxt, oh, ow, F));
    { const __half* src = V.p; __half* dst = nxt.p; const int ih = V.H, iw = V.W, C = F;
      add(G_RESAMPLE, "upsample_ac", [=](cudaStream_t s) { return upsample_ac_f16(src, Bt, ih, iw, C, dst, oh, ow, nullptr, s); }); }
    path = nxt;
    r_maps[3 - lvl] = nxt;
    if (lvl == 0) taps["path1"] = {path.p, path.H, path.W, path.C, 1};
  }
  // output_conv1 (3x3 F -> F/2) ; bilinear(align_corners=True) to (14ph,14pw) ; output_conv2 (3x3 -> 32, ReLU, 1x1 -> 1, ReLU)
  PMap O1, O1u;
  PRISMA_TRY(new_map(&O1, path.H, path.W, F / 2));
  PRISMA_TRY(new_map(&O1u, hn, wn, F / 2));
  { GemmEpilogue ep; ep.bias = w.oc1_b; ep.out_f16 = O1.p; ep.out_f16_ld = F / 2;
    PRISMA_TRY(add_conv3x3("output_conv1", path, w.oc1_w, F / 2, ep, 1, nullptr)); }
  { const __half* src = O1.p; __half* dst = O1u.p; const int ih = O1.H, iw = O1.W, C = F / 2, oh = hn, ow = wn;
    add(G_RESAMPLE, "upsample_ac", [=](cudaStream_t s) { return upsample_ac_f16(src, Bt, ih, iw, C, dst, oh, ow, nullptr, s); }); }
  __half* act32 = nullptr;
  if (metric) PRISMA_TRY(dev_alloc(plan_allocs, &act32, (size_t)Bt * hn * wn * 32));
  { GemmEpilogue ep; ep.bias = w.oc2_b; ep.act = 2; ep.head_w = w.oc3_w; ep.head_b = w.oc3_b; ep.head_out = b.depth;
    if (metric) { ep.out_f16 = act32; ep.out_f16_ld = 32; }
    PRISMA_TRY(add_conv3x3("output_conv2_fused", O1u, w.oc2_w, 32, ep, 1, nullptr)); }
  if (metric) PRISMA_TRY(build_metric_head(R[3], r_maps, act32, Bt));
  // (dpt.py:163-164: the final F.interpolate to (h,w) is the identity at equal size and the ReLU is idempotent)

  // ---- post-process (K10)
  {
    const float* d = b.depth; float* pred = b.pred; uint8_t* rgb = b.rgb; uint32_t* mm = b.mm; float* mmo = b.minmax;
    const int hn_ = hn, wn_ = wn, sms = num_sms;
    if (metric) {
      // bands/depth_anything.py:113-119: PIL resize (mode "F", BICUBIC) of the metric depth to the frame, then the video
      // loop's encode with flip = False (:188,215-220)
      const float* md = zoe_metric; float* tmp = zoe_tmp;
      add(G_POST, "depth_postprocess", [=](cudaStream_t s) {
        for (int i = 0; i < Bt; ++i) {
          PRISMA_TRY(pil_bicubic_resize_f32(md + (size_t)i * hn_ * wn_, hn_, wn_, tmp, pred + (size_t)i * H * W, H, W, s));
          PRISMA_TRY(depth_encode_only(pred + (size_t)i * H * W, H, W, 0, rgb + (size_t)i * H * W * 3, mm + 2 * i, mmo + 2 * i, sms, s));
        }
        return 0;
      });
    } else if (!midas)
      add(G_POST, "depth_postprocess", [=](cudaStream_t s) {
        for (int i = 0; i < Bt; ++i)
          PRISMA_TRY(depth_postprocess(d + (size_t)i * hn_ * wn_, hn_, wn_, H, W, 1, pred + (size_t)i * H * W,
                                       rgb + (size_t)i * H * W * 3, mm + 2 * i, mmo + 2 * i, sms, s));
        return 0;
      });
    else  // depth_midas.py:58-63 bicubic(align_corners=True) to the frame size, then the video loop's encode (:141-146)
      add(G_POST, "depth_postprocess", [=](cudaStream_t s) {
        for (int i = 0; i < Bt; ++i) {
          PRISMA_TRY(upsample_bicubic_ac_f32(d + (size_t)i * hn_ * wn_, hn_, wn_, pred + (size_t)i * H * W, H, W, sms, s));
          PRISMA_TRY(depth_encode_only(pred + (size_t)i * H * W, H, W, 1 | 2, rgb + (size_t)i * H * W * 3, mm + 2 * i,
                                       mmo + 2 * i, sms, s));
        }
        return 0;
      });
  }
  if (metric) taps["metric_net"] = {zoe_metric, Bt * hn, wn, 1, 0};
  taps["net_input"] = {b.net_in, Bt * 3, hn * wn, 1, 0};
  taps["tokens"] = {b.tokens_tap, BT, D, 1, 0};
  for (int i = 0; i < 4; ++i) taps["feat" + std::to_string(i)] = {b.feat[i], BP, D, 1, 2};  // patch tokens only
  taps["net_depth"] = {b.depth, Bt * hn, wn, 1, 0};
  taps["x_final"] = {b.x, BT, D, 1, 0};
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  plan_H = H; plan_W = W;
  // ---- one CUDA graph per resolution: ~200 launches per frame replayed with a single cudaGraphLaunch
  if (graph_exec) { cudaGraphExecDestroy(graph_exec); graph_exec = nullptr; }
  if (use_graph) {
    PRISMA_TRY(run_steps_direct(stream));  // warm: sets per-kernel attributes outside the capture
    PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
    cudaGraph_t graph = nullptr;
    PRISMA_CUDA_OK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
    int r = run_steps_direct(stream);
    cudaError_t e = cudaStreamEndCapture(stream, &graph);
    if (r != 0) { if (graph) cudaGraphDestroy(graph); return r; }
    PRISMA_CUDA_OK(e);
    PRISMA_CUDA_OK(cudaGraphInstantiate(&graph_exec, graph, 0));
    cudaGraphDestroy(graph);
  }
  return 0;
}

// ZoeDepth.forward after the core (zoedepth_v1.py:150-199): every 1x1 conv is a GEMM over dense pixel rows (the first one
// of each level reads the zero-bordered map and writes dense rows), the interpolations / attractors / log-binomial are the
// zoe_kernels.  Embeddings and bin centres stay fp32 between levels; GEMM operands are fp16.
int DepthEngine::build_metric_head(const PMap& btlnck, const PMap* r_maps, const __half* act32, int Bt) {
  const int zero_off[1] = {0};
  // 1x1 conv over the pixel rows of all Bt frames; the first conv of a level reads the stacked zero-bordered maps
  auto lin = [&](const char* name, const __half* A, long long a_rows, int a_pitch, const DaWeights::Lin& L, int M, int act,
                 __half* out16, float* out32, int out_ld, const PMap* padded_src) -> int {
    GemmEpilogue ep; ep.bias = L.b; ep.act = act;
    if (out16) { ep.out_f16 = out16; ep.out_f16_ld = out_ld; } else { ep.out_f32 = out32; ep.out_f32_ld = out_ld; }
    if (padded_src) {
      ep.row_map = ROW_PAD2TOK; ep.in_w = padded_src->Wp(); ep.in_h = padded_src->Hp(); ep.img_rows = (int)padded_src->img_rows(); ep.pad = 1;
    }
    const int n_pad = round_up(L.n, 4);  // N % 4: the single attractor of the last level is padded with zero rows
    return add_gemm(G_HEAD, name, A, a_rows, round_up(L.k, 64), a_pitch, L.w, M, n_pad, 1, zero_off, ep, 2.0 * M * (double)L.k * L.n);
  };
  // ---- bottleneck level: x_d0 = conv2(layer4_rn) ; seed bins ; seed embedding
  const int P0 = btlnck.H * btlnck.W, Fp = round_up(F, 64);
  __half *x0 = nullptr, *s1 = nullptr, *e1 = nullptr;
  float *b_prev = nullptr, *emb_prev = nullptr;
  PRISMA_TRY(dev_alloc(plan_allocs, &x0, (size_t)Bt * P0 * Fp));
  PRISMA_TRY(dev_alloc(plan_allocs, &s1, (size_t)Bt * P0 * 256));
  PRISMA_TRY(dev_alloc(plan_allocs, &e1, (size_t)Bt * P0 * 128));
  PRISMA_TRY(dev_alloc(plan_allocs, &b_prev, (size_t)Bt * P0 * 64));
  PRISMA_TRY(dev_alloc(plan_allocs, &emb_prev, (size_t)Bt * P0 * 128));
  PRISMA_TRY(lin("zoe_conv2", btlnck.p, btlnck.rows(), F, w.z_conv2, (int)btlnck.rows(), 0, x0, nullptr, Fp, &btlnck));
  PRISMA_TRY(lin("zoe_seed0", x0, (long long)Bt * P0, Fp, w.z_seed0, Bt * P0, 2, s1, nullptr, 256, nullptr));
  PRISMA_TRY(lin("zoe_seed2", s1, (long long)Bt * P0, 256, w.z_seed2, Bt * P0, 5, nullptr, b_prev, 64, nullptr));
  PRISMA_TRY(lin("zoe_sproj0", x0, (long long)Bt * P0, Fp, w.z_sproj0, Bt * P0, 2, e1, nullptr, 128, nullptr));
  PRISMA_TRY(lin("zoe_sproj2", e1, (long long)Bt * P0, 128, w.z_sproj2, Bt * P0, 0, nullptr, emb_prev, 128, nullptr));
  int Hp_ = btlnck.H, Wp_ = btlnck.W;
  const int n_attr[4] = {16, 8, 4, 1};
  for (int i = 0; i < 4; ++i) {
    const PMap& xb = r_maps[i];
    const int Hi = xb.H, Wi = xb.W, Pi = Hi * Wi;
    __half *t1 = nullptr, *xa = nullptr, *t2 = nullptr;
    float *emb = nullptr, *Aout = nullptr, *bnew = nullptr;
    PRISMA_TRY(dev_alloc(plan_allocs, &t1, (size_t)Bt * Pi * 128));
    PRISMA_TRY(dev_alloc(plan_allocs, &xa, (size_t)Bt * Pi * 128));
    PRISMA_TRY(dev_alloc(plan_allocs, &t2, (size_t)Bt * Pi * 128));
    PRISMA_TRY(dev_alloc(plan_allocs, &emb, (size_t)Bt * Pi * 128));
    PRISMA_TRY(dev_alloc(plan_allocs, &Aout, (size_t)Bt * Pi * 16));
    PRISMA_TRY(dev_alloc(plan_allocs, &bnew, (size_t)Bt * Pi * 64));
    PRISMA_TRY(lin("zoe_proj0", xb.p, xb.rows(), xb.C, w.z_proj0[i], (int)xb.rows(), 2, t1, nullptr, 128, &xb));
    PRISMA_TRY(lin("zoe_proj2", t1, (long long)Bt * Pi, 128, w.z_proj2[i], Bt * Pi, 0, nullptr, emb, 128, nullptr));
    { const float* ep_ = emb_prev; const int hp = Hp_, wp = Wp_;
      add(G_RESAMPLE, "zoe_embed_add", [=](cudaStream_t s) {
        for (int f = 0; f < Bt; ++f)
          PRISMA_TRY(zoe_embed_add(emb + (size_t)f * Pi * 128, Hi, Wi, 128, ep_ + (size_t)f * hp * wp * 128, hp, wp, xa + (size_t)f * Pi * 128, s));
        return 0;
      }); }
    PRISMA_TRY(lin("zoe_att0", xa, (long long)Bt * Pi, 128, w.z_att0[i], Bt * Pi, 2, t2, nullptr, 128, nullptr));
    const int lda = round_up(n_attr[i], 4);
    PRISMA_TRY(lin("zoe_att2", t2, (long long)Bt * Pi, 128, w.z_att2[i], Bt * Pi, 5, nullptr, Aout, lda, nullptr));
    { const float* bp = b_prev; const int hp = Hp_, wp = Wp_, na = n_attr[i];
      add(G_RESAMPLE, "zoe_attractor", [=](cudaStream_t s) {
        for (int f = 0; f < Bt; ++f)
          PRISMA_TRY(zoe_attractor(Aout + (size_t)f * Pi * lda, lda, na, bp + (size_t)f * hp * wp * 64, hp, wp, Hi, Wi, 64,
                                   bnew + (size_t)f * Pi * 64, s));
        return 0;
      }); }
    b_prev = bnew; emb_prev = emb; Hp_ = Hi; Wp_ = Wi;
  }
  // ---- conditional log-binomial at the network resolution
  const int Pf = hn * wn;
  __half *cat = nullptr, *hid = nullptr;
  float* pt = nullptr;
  PRISMA_TRY(dev_alloc(plan_allocs, &cat, (size_t)Bt * Pf * 192));
  PRISMA_TRY(dev_alloc(plan_allocs, &hid, (size_t)Bt * Pf * 128));
  PRISMA_TRY(dev_alloc(plan_allocs, &pt, (size_t)Bt * Pf * 4));
  PRISMA_TRY(dev_alloc(plan_allocs, &zoe_metric, (size_t)Bt * Pf));
  PRISMA_TRY(dev_alloc(plan_allocs, &zoe_tmp, (size_t)hn * std::max(plan_W_req, wn)));
  { const float* rel = b.depth; const float* ep_ = emb_prev; const int he = Hp_, we = Wp_, h_ = hn, w_ = wn;
    add(G_RESAMPLE, "zoe_concat", [=](cudaStream_t s) {
      for (int f = 0; f < Bt; ++f)
        PRISMA_TRY(zoe_concat(act32 + (size_t)f * Pf * 32, rel + (size_t)f * Pf, ep_ + (size_t)f * he * we * 128, he, we, h_, w_,
                              cat + (size_t)f * Pf * 192, s));
      return 0;
    }); }
  PRISMA_TRY(lin("zoe_clb0", cat, (long long)Bt * Pf, 192, w.z_clb0, Bt * Pf, 1, hid, nullptr, 128, nullptr));
  PRISMA_TRY(lin("zoe_clb2", hid, (long long)Bt * Pf, 128, w.z_clb2, Bt * Pf, 5, nullptr, pt, 4, nullptr));
  { const float* bc = b_prev; const int hc = Hp_, wc = Wp_, h_ = hn, w_ = wn; float* out = zoe_metric;
    add(G_POST, "zoe_final", [=](cudaStream_t s) {
      for (int f = 0; f < Bt; ++f)
        PRISMA_TRY(zoe_final(pt + (size_t)f * Pf * 4, bc + (size_t)f * hc * wc * 64, hc, wc, h_, w_, 64, 0.0212f, 50.0f,
                             out + (size_t)f * Pf, s));
      return 0;
    }); }
  return 0;
}

int DepthEngine::run_steps_direct(cudaStream_t s) {
  for (auto& st : steps) { NvtxRange r(st.name); PRISMA_TRY(st.fn(s)); }
  return 0;
}

int DepthEngine::run_steps(cudaStream_t s) {
  if (graph_exec) {
    PRISMA_CUDA_OK(cudaGraphLaunch(graph_exec, s));
    return 0;
  }
  return run_steps_direct(s);
}

int DepthEngine::infer(const uint8_t* rgb, int n, int H, int W, float* depth_out, uint8_t* rgb_out, float* min_out,
                       float* max_out) {
  PRISMA_CHECK(rgb != nullptr && H > 0 && W > 0 && n >= 1, "bad frame batch");
  NvtxRange nvtx_pass("prisma.depth.infer");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_TRY(build_plan(H, W, n));
  PRISMA_CUDA_OK(cudaMemcpyAsync(b.img, rgb, (size_t)n * H * W * 3, cudaMemcpyHostToDevice, stream));
  PRISMA_TRY(run_steps(stream));
  std::vector<float> mm(2 * n);
  if (depth_out) PRISMA_CUDA_OK(cudaMemcpyAsync(depth_out, b.pred, (size_t)n * H * W * 4, cudaMemcpyDeviceToHost, stream));
  if (rgb_out) PRISMA_CUDA_OK(cudaMemcpyAsync(rgb_out, b.rgb, (size_t)n * H * W * 3, cudaMemcpyDeviceToHost, stream));
  PRISMA_CUDA_OK(cudaMemcpyAsync(mm.data(), b.minmax, 8 * n, cudaMemcpyDeviceToHost, stream));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  for (int i = 0; i < n; ++i) {
    if (min_out) min_out[i] = mm[2 * i];
    if (max_out) max_out[i] = mm[2 * i + 1];
  }
  return 0;
}

int DepthEngine::ensure_stream_slots(int H, int W, int Bt, bool want_pred) {
  if (!s_in) {
    PRISMA_CUDA_OK(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
    PRISMA_CUDA_OK(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
    for (auto& sl : slot)
      for (cudaEvent_t* e : {&sl.loaded, &sl.consumed, &sl.done, &sl.drained})
        PRISMA_CUDA_OK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  const size_t px = (size_t)H * W;
  if (slot_frames == (size_t)Bt && slot_bytes_frame == px && (slot_has_pred || !want_pred)) return 0;
  PRISMA_CUDA_OK(cudaDeviceSynchronize());
  for (auto& sl : slot) {
    cudaFree(sl.in); cudaFree(sl.rgb); cudaFree(sl.pred); cudaFree(sl.mm);
    sl.in = sl.rgb = nullptr; sl.pred = sl.mm = nullptr;
    PRISMA_CUDA_OK(cudaMalloc(&sl.in, Bt * px * 3));
    PRISMA_CUDA_OK(cudaMalloc(&sl.rgb, Bt * px * 3));
    if (want_pred) PRISMA_CUDA_OK(cudaMalloc(&sl.pred, Bt * px * 4));
    PRISMA_CUDA_OK(cudaMalloc(&sl.mm, Bt * 8));
  }
  slot_frames = Bt; slot_bytes_frame = px; slot_has_pred = want_pred;
  return 0;
}

// The video loop of the band (bands/depth_anything.py:203-221) over a chunk of n frames.  Three streams: s_in uploads
// pass i+1 into a staging slot while `stream` runs the graph of pass i and s_out drains the results of pass i-1; the
// graph keeps its fixed buffers, staging is two device-to-device copies per pass (~25 MB, microseconds).
// A ragged last pass runs the full-batch graph (frames are independent) and only its valid frames are copied out.
int DepthEngine::infer_stream(const uint8_t* rgb, int n, int H, int W, int pass_frames, float* depth_out, uint8_t* rgb_out,
                              float* min_out, float* max_out) {
  PRISMA_CHECK(rgb != nullptr && H > 0 && W > 0 && n >= 1, "bad frame batch");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  const int Bt = pass_frames > 0 ? std::min(pass_frames, 64) : 4;
  NvtxRange nvtx_pass("prisma.depth.infer_stream");
  PRISMA_TRY(build_plan(H, W, Bt));
  PRISMA_TRY(ensure_stream_slots(H, W, Bt, depth_out != nullptr));
  if (mm_host_frames < (size_t)n) {
    if (mm_host) cudaFreeHost(mm_host);
    mm_host = nullptr; mm_host_frames = 0;
    PRISMA_CUDA_OK(cudaMallocHost(&mm_host, (size_t)n * 8));
    mm_host_frames = n;
  }
  const size_t px = (size_t)H * W;
  const int passes = (n + Bt - 1) / Bt;
  auto frames_of = [&](int i) { return std::min(Bt, n - i * Bt); };
  auto drain = [&](int i) -> int {   // results of pass i -> host
    StreamSlot& sl = slot[i & 1];
    const int f = frames_of(i);
    const size_t o = (size_t)i * Bt;
    PRISMA_CUDA_OK(cudaStreamWaitEvent(s_out, sl.done, 0));
    if (rgb_out) PRISMA_CUDA_OK(cudaMemcpyAsync(rgb_out + o * px * 3, sl.rgb, f * px * 3, cudaMemcpyDeviceToHost, s_out));
    if (depth_out) PRISMA_CUDA_OK(cudaMemcpyAsync(depth_out + o * px, sl.pred, f * px * 4, cudaMemcpyDeviceToHost, s_out));
    PRISMA_CUDA_OK(cudaMemcpyAsync(mm_host + o * 2, sl.mm, f * 8, cudaMemcpyDeviceToHost, s_out));
    PRISMA_CUDA_OK(cudaEventRecord(sl.drained, s_out));
    return 0;
  };
  for (int i = 0; i < passes; ++i) {
    StreamSlot& sl = slot[i & 1];
    const int f = frames_of(i);
    if (i >= 2) PRISMA_CUDA_OK(cudaStreamWaitEvent(s_in, sl.consumed, 0));
    PRISMA_CUDA_OK(cudaMemcpyAsync(sl.in, rgb + (size_t)i * Bt * px * 3, f * px * 3, cudaMemcpyHostToDevice, s_in));
    PRISMA_CUDA_OK(cudaEventRecord(sl.loaded, s_in));
    PRISMA_CUDA_OK(cudaStreamWaitEvent(stream, sl.loaded, 0));
    PRISMA_CUDA_OK(cudaMemcpyAsync(b.img, sl.in, f * px * 3, cudaMemcpyDeviceToDevice, stream));
    PRISMA_CUDA_OK(cudaEventRecord(sl.consumed, stream));
    PRISMA_TRY(run_steps(stream));
    if (i >= 2) PRISMA_CUDA_OK(cudaStreamWaitEvent(stream, sl.drained, 0));
    if (rgb_out) PRISMA_CUDA_OK(cudaMemcpyAsync(sl.rgb, b.rgb, f * px * 3, cudaMemcpyDeviceToDevice, stream));
    if (depth_out) PRISMA_CUDA_OK(cudaMemcpyAsync(sl.pred, b.pred, f * px * 4, cudaMemcpyDeviceToDevice, stream));
    PRISMA_CUDA_OK(cudaMemcpyAsync(sl.mm, b.minmax, f * 8, cudaMemcpyDeviceToDevice, stream));
    PRISMA_CUDA_OK(cudaEventRecord(sl.done, stream));
    if (i >= 1) PRISMA_TRY(drain(i - 1));
  }
  PRISMA_TRY(drain(passes - 1));
  PRISMA_CUDA_OK(cudaStreamSynchronize(s_out));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  for (int i = 0; i < n; ++i) {
    if (min_out) min_out[i] = mm_host[2 * i];
    if (max_out) max_out[i] = mm_host[2 * i + 1];
  }
  return 0;
}

// process_image path (bands/depth_anything.py:146-174): one frame, write_depth's PNG encoding of the prediction
int DepthEngine::infer_image(const uint8_t* rgb, int H, int W, float* depth_out, uint8_t* png_rgb_out, float* min_out,
                             float* max_out) {
  PRISMA_CHECK(rgb != nullptr && png_rgb_out != nullptr, "null argument");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_TRY(build_plan(H, W, 1));
  PRISMA_CUDA_OK(cudaMemcpyAsync(b.img, rgb, (size_t)H * W * 3, cudaMemcpyHostToDevice, stream));
  PRISMA_TRY(run_steps(stream));
  int r = depth_encode_png(b.pred, H, W, metric ? 0 : 1, b.rgb, b.mm, b.mag, b.minmax, num_sms, stream);  // flip = (metric == none)
  float mm[2] = {0, 0};
  if (r == 0) {
    if (depth_out) cudaMemcpyAsync(depth_out, b.pred, (size_t)H * W * 4, cudaMemcpyDeviceToHost, stream);
    cudaMemcpyAsync(png_rgb_out, b.rgb, (size_t)H * W * 3, cudaMemcpyDeviceToHost, stream);
    cudaMemcpyAsync(mm, b.minmax, 8, cudaMemcpyDeviceToHost, stream);
    cudaError_t e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) { set_last_error(std::string("infer_image: ") + cudaGetErrorString(e)); r = -2; }
  }
  if (min_out) *min_out = mm[0];
  if (max_out) *max_out = mm[1];
  return r;
}

int DepthEngine::infer_resident(int H, int W, int n, int iters, float* ms_per_iter) {
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_TRY(build_plan(H, W, n));
  PRISMA_CUDA_OK(cudaEventRecord(ev0, stream));
  for (int i = 0; i < iters; ++i) PRISMA_TRY(run_steps(stream));
  PRISMA_CUDA_OK(cudaEventRecord(ev1, stream));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  float ms = 0;
  PRISMA_CUDA_OK(cudaEventElapsedTime(&ms, ev0, ev1));
  if (ms_per_iter) *ms_per_iter = ms / std::max(iters, 1);
  return 0;
}

int DepthEngine::encode(const float* pred, int H, int W, int flip, uint8_t* rgb_out, float* min_out, float* max_out,
                        int png_variant) {
  PRISMA_CUDA_OK(cudaSetDevice(device));
  float* d_pred = nullptr; uint8_t* d_rgb = nullptr; uint32_t* d_mm = nullptr; float* d_out = nullptr;
  unsigned long long* d_mag = nullptr;
  std::vector<void*> tmp;
  auto cleanup = [&]() { for (void* q : tmp) cudaFree(q); };
  int r = 0;
  if ((r = dev_alloc(tmp, &d_pred, (size_t)H * W, false)) || (r = dev_alloc(tmp, &d_rgb, (size_t)H * W * 3, false)) ||
      (r = dev_alloc(tmp, &d_mm, 2)) || (r = dev_alloc(tmp, &d_out, 2)) || (r = dev_alloc(tmp, &d_mag, 2))) { cleanup(); return r; }
  cudaMemcpyAsync(d_pred, pred, (size_t)H * W * 4, cudaMemcpyHostToDevice, stream);
  r = png_variant ? depth_encode_png(d_pred, H, W, flip, d_rgb, d_mm, d_mag, d_out, num_sms, stream)
                  : depth_encode_only(d_pred, H, W, flip, d_rgb, d_mm, d_out, num_sms, stream);
  float mm[2] = {0, 0};
  if (r == 0) {
    cudaMemcpyAsync(rgb_out, d_rgb, (size_t)H * W * 3, cudaMemcpyDeviceToHost, stream);
    cudaMemcpyAsync(mm, d_out, 8, cudaMemcpyDeviceToHost, stream);
    cudaError_t e = cudaStreamSynchronize(stream);
    if (e != cudaSuccess) { set_last_error(std::string("encode: ") + cudaGetErrorString(e)); r = -2; }
  }
  cleanup();
  if (min_out) *min_out = mm[0];
  if (max_out) *max_out = mm[1];
  return r;
}

long long DepthEngine::read_tap(const std::string& name, float* out, long long capacity) {
  auto it = taps.find(name);
  if (it == taps.end()) { set_last_error("unknown tap '" + name + "'"); return -1; }
  cudaSetDevice(device);
  const Tap& t = it->second;
  if (t.kind == 0 || t.kind == 2) {  // dense f32 / f16 [a][b]
    const long long n = (long long)t.a * t.b;
    if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
    if (t.kind == 0) {
      if (cudaMemcpy(out, t.p, n * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    } else {
      std::vector<__half> h(n);
      if (cudaMemcpy(h.data(), t.p, n * 2, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
      for (long long i = 0; i < n; ++i) out[i] = __half2float(h[i]);
    }
    return n;
  }
  // kind 1: zero-bordered NHWC fp16 map (a=H, b=W, c=C) -> dense [H][W][C] f32
  const long long n = (long long)t.a * t.b * t.c;
  if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
  const size_t tot = (size_t)(t.a + 2) * (t.b + 2) * t.c;
  std::vector<__half> h(tot);
  if (cudaMemcpy(h.data(), t.p, tot * 2, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
  for (int y = 0; y < t.a; ++y)
    for (int x = 0; x < t.b; ++x)
      for (int c = 0; c < t.c; ++c)
        out[((size_t)y * t.b + x) * t.c + c] = __half2float(h[((size_t)(y + 1) * (t.b + 2) + x + 1) * t.c + c]);
  return n;
}

int DepthEngine::profile(int H, int W, int n, float* out8) {
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_TRY(build_plan(H, W, n));
  PRISMA_TRY(run_steps_direct(stream));  // warm
  std::vector<cudaEvent_t> ev(steps.size() + 1);
  for (auto& e : ev) PRISMA_CUDA_OK(cudaEventCreate(&e));
  PRISMA_CUDA_OK(cudaEventRecord(ev[0], stream));
  for (size_t i = 0; i < steps.size(); ++i) {
    PRISMA_TRY(steps[i].fn(stream));
    PRISMA_CUDA_OK(cudaEventRecord(ev[i + 1], stream));
  }
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  for (int i = 0; i < 8; ++i) out8[i] = 0.f;
  const bool verbose = getenv("PRISMA_DA_PROFILE") != nullptr;
  std::vector<std::pair<std::string, std::pair<double, int>>> by_name;  // first-seen order
  for (size_t i = 0; i < steps.size(); ++i) {
    float ms = 0;
    PRISMA_CUDA_OK(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
    out8[steps[i].group] += ms;
    out8[7] += ms;
    if (verbose) {
      // strip digits so the 24 blocks fold into one row per op
      std::string key;
      for (const char* c = steps[i].name; *c; ++c) if (*c < '0' || *c > '9') key.push_back(*c);
      auto it = std::find_if(by_name.begin(), by_name.end(), [&](const auto& kv) { return kv.first == key; });
      if (it == by_name.end()) by_name.push_back({key, {ms, 1}});
      else { it->second.first += ms; it->second.second += 1; }
    }
  }
  if (verbose)
    for (auto& kv : by_name)
      fprintf(stderr, "[da-profile] %-28s x%-3d %8.3f ms  (%.1f us each)\n", kv.first.c_str(), kv.second.second,
              kv.second.first, 1e3 * kv.second.first / kv.second.second);
  for (auto& e : ev) cudaEventDestroy(e);
  return 0;
}

}  // namespace prisma
