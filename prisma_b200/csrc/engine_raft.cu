// prisma_b200 -- RAFT optical-flow engine: flow_raft.infer (bands/flow_raft.py:51-66) for one frame pair, forward
// and backward flow in one pass (batch 2 = [prev,curr] / [curr,prev], flow_raft.py:105-106).
//
// Reference model: bands/raft/raft.py:87-146 (test_mode), extractor.py (BasicEncoder), corr.py (CorrBlock),
// update.py (BasicUpdateBlock).  What differs structurally from the reference, with identical results:
//   * fnet runs on the two distinct frames once (the reference runs it on the 4-image concatenation of two identical
//     pairs; InstanceNorm statistics are per image so the outputs are the same) and cnet likewise;
//   * only the last iteration's up-sampling mask / convex up-sampling is computed (test_mode consumes only that one);
//   * BatchNorm (eval) of cnet is folded into the conv weights; InstanceNorm of fnet is a two-stage reduction +
//     normalise kernel between convs; every conv is the tcgen05 shifted-row GEMM on zero-bordered NHWC fp16 maps.
#include "engine_raft.cuh"

#include <math.h>

#include <algorithm>

namespace prisma {

struct RMap {  // B NHWC fp16 maps in the shared-border layout: `pad` zero columns after every row, `pad` zero rows after every
               // image (see GemmEpilogue::lead); a 1/8-resolution 1080p pair is 2 x 104 x 182 = 37 856 rows = 296 row tiles =
               // exactly two waves of 148 CTAs (the symmetric border made it 305 tiles = 2.06 waves)
  __half* p = nullptr;
  int B = 0, H = 0, W = 0, C = 0, pad = 1;
  int Hp() const { return H + pad; }
  int Wp() const { return W + pad; }
  long long img_rows() const { return ((long long)Hp() * Wp() + 31) / 32 * 32; }  // a 32-row epilogue slab never straddles two images
  long long rows() const { return B * img_rows(); }
};

template <typename T>
static int r_alloc(std::vector<void*>& pool, T** out, size_t n) {
  void* p = nullptr;
  PRISMA_CUDA_OK(cudaMalloc(&p, std::max<size_t>(n * sizeof(T), 256)));
  PRISMA_CUDA_OK(cudaMemset(p, 0, std::max<size_t>(n * sizeof(T), 256)));
  pool.push_back(p);
  *out = reinterpret_cast<T*>(p);
  return 0;
}

RaftEngine::~RaftEngine() {
  cudaSetDevice(device);
  for (void* p : allocs) cudaFree(p);
  for (void* p : plan_allocs) cudaFree(p);
  delete corr;
  if (graph_exec) cudaGraphExecDestroy(graph_exec);
  if (graph_cached) cudaGraphExecDestroy(graph_cached);
  for (auto& sl : slot) {
    cudaFree(sl.in); cudaFree(sl.flow); cudaFree(sl.rgb); cudaFree(sl.mx);
    for (cudaEvent_t e : {sl.loaded, sl.consumed, sl.done, sl.drained}) if (e) cudaEventDestroy(e);
  }
  if (mx_host) cudaFreeHost(mx_host);
  if (s_in) cudaStreamDestroy(s_in);
  if (s_out) cudaStreamDestroy(s_out);
  if (stream) cudaStreamDestroy(stream);
}

int RaftEngine::init(int dev) {
  device = dev;
  int n = 0;
  PRISMA_CUDA_OK(cudaGetDeviceCount(&n));
  PRISMA_CHECK(dev >= 0 && dev < n, "bad device ordinal");
  PRISMA_CUDA_OK(cudaSetDevice(dev));
  cudaDeviceProp prop;
  PRISMA_CUDA_OK(cudaGetDeviceProperties(&prop, dev));
  PRISMA_CHECK(prop.major == 10, "prisma_b200 kernels are sm_100a only; there is no fallback path");
  num_sms = prop.multiProcessorCount;
  device_mem = prop.totalGlobalMem;
  PRISMA_CUDA_OK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  const char* ng = getenv("PRISMA_NO_GRAPH");
  use_graph = !(ng && ng[0] == '1');
  if (const char* np = getenv("PRISMA_RAFT_PAIRS")) stream_pairs = std::min(std::max(atoi(np), 1), 4);
  return 0;
}

int RaftEngine::load_tensor(const std::string& name, const float* data, const int64_t* shape, int ndim) {
  PRISMA_CHECK(!finalized, "load_tensor after finalize");
  HostTensor t;
  size_t n = 1;
  for (int i = 0; i < ndim; ++i) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
  t.data.assign(data, data + n);
  std::string key = name;
  if (key.rfind("module.", 0) == 0) key = key.substr(7);  // DataParallel checkpoints (flow_raft.py:42-44)
  host[key] = std::move(t);
  return 0;
}

const HostTensor* RaftEngine::get(const std::string& name) {
  auto it = host.find(name);
  if (it == host.end()) { set_last_error("missing RAFT weight tensor '" + name + "'"); return nullptr; }
  return &it->second;
}

// conv weight [Cout][Cin][kh][kw] (+bias) -> fp16 [round_up(Npad,256)][taps*kc*64], fp32 bias [Npad]; optional eval-mode
// BatchNorm folding (y = (conv(x) - mean) * gamma / sqrt(var + eps) + beta, eps = 1e-5) and output scale.
// chans: use only these input channels, in this order (the packed conv then has cin = chans->size()); with_bias = false drops
// the bias (when one conv is evaluated as the sum of two convs over disjoint channel sets, only one of them carries it).
int RaftEngine::up_conv(const std::string& name, const std::string& bn, int Cout, int CinSrc, int kh, int kw, int Npad,
                        float out_scale, ConvW* out, int wsplit, const std::vector<int>* chans, bool with_bias) {
  const HostTensor* w = get(name + ".weight");
  const HostTensor* b = get(name + ".bias");
  if (!w || !b) return -1;
  PRISMA_CHECK((long long)w->data.size() == (long long)Cout * CinSrc * kh * kw, "RAFT weight '" + name + "' has an unexpected size");
  const int Cin = chans ? (int)chans->size() : CinSrc;
  std::vector<float> sc(Cout, out_scale), sh(Cout, 0.f);
  for (int n = 0; n < Cout; ++n) sh[n] = with_bias ? b->data[n] * out_scale : 0.f;
  if (!bn.empty()) {
    const HostTensor *g = get(bn + ".weight"), *be = get(bn + ".bias"), *mu = get(bn + ".running_mean"), *var = get(bn + ".running_var");
    if (!g || !be || !mu || !var) return -1;
    for (int n = 0; n < Cout; ++n) {
      const float k = g->data[n] / sqrtf(var->data[n] + 1e-5f);
      sc[n] = k;
      sh[n] = ((with_bias ? b->data[n] : 0.f) - mu->data[n]) * k + be->data[n];
    }
  }
  // wsplit == 2: the weights keep ~22 bits as an fp16 pair.  Weight rounding is a SYSTEMATIC error (the same perturbed
  // filter at every pixel and iteration) and dominates the flow error of the update block; activations' rounding is random
  // and 7x smaller (oracle/tools/raft_precision_study.py).  Tap t occupies the K slabs 2t (hi) and 2t + 1 (lo).
  const int taps = kh * kw, kc = ceil_div(Cin, 64), K = taps * wsplit * kc * 64, rows = round_up(Npad, 256);
  std::vector<__half> h((size_t)rows * K, __float2half_rn(0.f));
  for (int n = 0; n < Cout; ++n)
    for (int t = 0; t < taps; ++t)
      for (int c = 0; c < Cin; ++c) {
        const float v = w->data[((size_t)n * CinSrc + (chans ? (*chans)[c] : c)) * taps + t] * sc[n];
        const __half hi = __float2half_rn(v);
        h[(size_t)n * K + (size_t)t * wsplit * kc * 64 + c] = hi;
        if (wsplit == 2) h[(size_t)n * K + (size_t)(t * 2 + 1) * kc * 64 + c] = __float2half_rn(v - __half2float(hi));
      }
  PRISMA_TRY(r_alloc(allocs, &out->w, h.size()));
  PRISMA_CUDA_OK(cudaMemcpy(out->w, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
  std::vector<float> bias(round_up(Npad, 8), 0.f);
  for (int n = 0; n < Cout; ++n) bias[n] = sh[n];
  PRISMA_TRY(r_alloc(allocs, &out->b, bias.size()));
  PRISMA_CUDA_OK(cudaMemcpy(out->b, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice));
  out->cout = Npad; out->cin = Cin; out->kh = kh; out->kw = kw; out->wsplit = wsplit;
  return 0;
}

int RaftEngine::up_encoder(const std::string& p, bool bn, EncW* e) {
  auto B = [&](const std::string& n) { return bn ? p + n : std::string(); };
  {  // stem: im2col K = 168 -> 192; weight [64][3][7][7] flattens to k = (c*7 + ky)*8 + kx (kx = 7: zero), i.e. a "1x1 conv"
     // with Cin 168 -- one 16-byte im2col group is one 7-pixel input row segment (raft_kernels.cu:k_im2col_stem)
    const HostTensor* w = get(p + "conv1.weight");
    if (!w) return -1;
    PRISMA_CHECK(w->data.size() == (size_t)64 * 147, "RAFT conv1 has an unexpected size");
    HostTensor flat;
    flat.shape = {64, 168, 1, 1};
    flat.data.assign((size_t)64 * 168, 0.f);
    for (int o = 0; o < 64; ++o)
      for (int cy = 0; cy < 21; ++cy)
        for (int kx = 0; kx < 7; ++kx) flat.data[(size_t)o * 168 + cy * 8 + kx] = w->data[(size_t)o * 147 + cy * 7 + kx];
    host[p + "conv1_flat.weight"] = flat;
    host[p + "conv1_flat.bias"] = *get(p + "conv1.bias");
    PRISMA_TRY(up_conv(p + "conv1_flat", B("norm1"), 64, 168, 1, 1, 64, 1.f, &e->stem));
  }
  const int dims[3] = {64, 96, 128};
  int cin = 64;
  for (int li = 0; li < 3; ++li) {
    for (int bi = 0; bi < 2; ++bi) {
      const std::string q = p + "layer" + std::to_string(li + 1) + "." + std::to_string(bi) + ".";
      ResW& r = e->blk[li][bi];
      PRISMA_TRY(up_conv(q + "conv1", B(("layer" + std::to_string(li + 1) + "." + std::to_string(bi) + ".norm1")), dims[li], bi == 0 ? cin : dims[li], 3, 3, dims[li], 1.f, &r.c1));
      PRISMA_TRY(up_conv(q + "conv2", B(("layer" + std::to_string(li + 1) + "." + std::to_string(bi) + ".norm2")), dims[li], dims[li], 3, 3, dims[li], 1.f, &r.c2));
      r.has_ds = (bi == 0 && li > 0);
      if (r.has_ds)
        PRISMA_TRY(up_conv(q + "downsample.0", B(("layer" + std::to_string(li + 1) + "." + std::to_string(bi) + ".downsample.1")), dims[li], cin, 1, 1, dims[li], 1.f, &r.ds));
    }
    cin = dims[li];
  }
  PRISMA_TRY(up_conv(p + "conv2", "", 256, 128, 1, 1, 256, 1.f, &e->out));
  return 0;
}

int RaftEngine::finalize() {
  PRISMA_CHECK(!finalized, "finalize called twice");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_TRY(up_encoder("fnet.", false, &w.fnet));
  PRISMA_TRY(up_encoder("cnet.", true, &w.cnet));
  const std::string u = "update_block.";
  PRISMA_TRY(up_conv(u + "encoder.convc1", "", 256, 324, 1, 1, 256, 1.f, &w.convc1));
  PRISMA_TRY(up_conv(u + "encoder.convc2", "", 192, 256, 3, 3, 192, 1.f, &w.convc2));
  PRISMA_TRY(up_conv(u + "encoder.convf2", "", 64, 128, 3, 3, 64, 1.f, &w.convf2));
  PRISMA_TRY(up_conv(u + "encoder.conv", "", 126, 256, 3, 3, 128, 1.f, &w.conv));  // 126 -> 128 (two zero channels)
  {  // convf1 7x7 on the 2-channel flow: im2col GEMM (K = hi/lo split of 98 taps), fp32 bias
    const HostTensor* wt = get(u + "encoder.convf1.weight");
    const HostTensor* bs = get(u + "encoder.convf1.bias");
    if (!wt || !bs) return -1;
    PRISMA_TRY(r_alloc(allocs, &w.convf1_w, wt->data.size()));
    PRISMA_TRY(r_alloc(allocs, &w.convf1_b, bs->data.size()));
    PRISMA_CUDA_OK(cudaMemcpy(w.convf1_w, wt->data.data(), wt->data.size() * 4, cudaMemcpyHostToDevice));
    PRISMA_CUDA_OK(cudaMemcpy(w.convf1_b, bs->data.data(), bs->data.size() * 4, cudaMemcpyHostToDevice));
    PRISMA_CHECK(wt->data.size() == (size_t)128 * 98, "RAFT convf1 weight has an unexpected size");
    std::vector<__half> hw((size_t)256 * 256, __float2half_rn(0.f));
    for (int co = 0; co < 128; ++co)
      for (int k = 0; k < 98; ++k) {  // [co][ch][ky][kx] flattens to k = ch*49 + ky*7 + kx, the im2col order
        hw[(size_t)co * 256 + k] = __float2half_rn(wt->data[(size_t)co * 98 + k]);
        hw[(size_t)co * 256 + 128 + k] = hw[(size_t)co * 256 + k];
      }
    PRISMA_TRY(r_alloc(allocs, &w.convf1_gemm_w, hw.size()));
    PRISMA_CUDA_OK(cudaMemcpy(w.convf1_gemm_w, hw.data(), hw.size() * 2, cudaMemcpyHostToDevice));
  }
  for (int pass = 0; pass < 2; ++pass) {  // SepConvGRU: (1,5) then (5,1); z and r stacked into one N = 256 conv
    const std::string s = std::to_string(pass + 1);
    const int kh = pass == 0 ? 1 : 5, kw = pass == 0 ? 5 : 1;
    const HostTensor *wz = get(u + "gru.convz" + s + ".weight"), *wr = get(u + "gru.convr" + s + ".weight");
    const HostTensor *bz = get(u + "gru.convz" + s + ".bias"), *br = get(u + "gru.convr" + s + ".bias");
    if (!wz || !wr || !bz || !br) return -1;
    HostTensor wzr, bzr;
    wzr.data = wz->data; wzr.data.insert(wzr.data.end(), wr->data.begin(), wr->data.end());
    bzr.data = bz->data; bzr.data.insert(bzr.data.end(), br->data.begin(), br->data.end());
    host[u + "gru.zr" + s + ".weight"] = wzr;
    host[u + "gru.zr" + s + ".bias"] = bzr;
    PRISMA_TRY(up_conv(u + "gru.zr" + s, "", 256, 384, kh, kw, 256, 1.f, &w.zr[pass]));
    PRISMA_TRY(up_conv(u + "gru.convq" + s, "", 128, 384, kh, kw, 128, 1.f, &w.q[pass]));
  }
  PRISMA_TRY(up_conv(u + "flow_head.conv1", "", 256, 128, 3, 3, 256, 1.f, &w.fh1, 2));  // hi/lo weights: the largest error term
  {  // FlowHead.conv2 (3x3, 256 -> 2) as a 1x1 conv to 18 partial products u[tap*2 + out] (see k_flow_head2_gather)
    const HostTensor* wt = get(u + "flow_head.conv2.weight");
    const HostTensor* bs = get(u + "flow_head.conv2.bias");
    if (!wt || !bs) return -1;
    PRISMA_CHECK(wt->data.size() == (size_t)2 * 256 * 9 && bs->data.size() == 2, "RAFT flow_head.conv2 has an unexpected size");
    HostTensor wu, bu;
    wu.data.assign((size_t)18 * 256, 0.f);
    for (int t = 0; t < 9; ++t)
      for (int o = 0; o < 2; ++o)
        for (int c = 0; c < 256; ++c) wu.data[((size_t)(t * 2 + o)) * 256 + c] = wt->data[((size_t)o * 256 + c) * 9 + t];
    bu.data.assign(18, 0.f);
    host[u + "flow_head.conv2_u.weight"] = wu;
    host[u + "flow_head.conv2_u.bias"] = bu;
    PRISMA_TRY(up_conv(u + "flow_head.conv2_u", "", 18, 256, 1, 1, 32, 1.f, &w.fh2u, 2));  // hi/lo weights: exact to ~22 bits
    w.fh2_b[0] = bs->data[0]; w.fh2_b[1] = bs->data[1];
  }
  PRISMA_TRY(up_conv(u + "mask.0", "", 256, 128, 3, 3, 256, 1.f, &w.mk1));
  PRISMA_TRY(up_conv(u + "mask.2", "", 576, 256, 1, 1, 576, 0.25f, &w.mk2));  // mask = .25 * conv (update.py:135)
  host.clear();
  finalized = true;
  return 0;
}

// ------------------------------------------------------------------------------------------------ plan helpers
int RaftEngine::new_map(RMap* m, int B, int H, int W, int C, int pad) {
  m->B = B; m->H = H; m->W = W; m->C = C; m->pad = pad;
  return r_alloc(plan_allocs, &m->p, (size_t)m->rows() * C);
}

void RaftEngine::add(const char* name, std::function<int(cudaStream_t)> fn) { steps.push_back({cur_mask, name, std::move(fn)}); }

// conv (kh x kw, 'same') on channels [c0, c0+cin) of a padded map; epilogue filled in by the caller
int RaftEngine::add_conv(const char* name, const RMap& in, int c0, const ConvW& cw, GemmEpilogue ep, int sub) {
  PRISMA_CHECK(cw.kh / 2 <= in.pad && cw.kw / 2 <= in.pad, "conv halo exceeds the map border");
  int off[GEMM_MAX_TAPS];
  PRISMA_CHECK(cw.kh * cw.kw * cw.wsplit <= GEMM_MAX_TAPS, "conv: too many taps");
  for (int ky = 0; ky < cw.kh; ++ky)
    for (int kx = 0; kx < cw.kw; ++kx)
      for (int sp = 0; sp < cw.wsplit; ++sp)  // hi / lo weight slabs re-read the same shifted rows
        off[(ky * cw.kw + kx) * cw.wsplit + sp] = (ky - cw.kh / 2) * in.Wp() + (kx - cw.kw / 2);
  if (ep.row_map == ROW_LINEAR) ep.row_map = ROW_PADDED;
  ep.in_w = in.Wp(); ep.in_h = in.Hp(); ep.img_rows = (int)in.img_rows(); ep.pad = in.pad; ep.sub = sub;
  ep.lead = 0; ep.out_lead = 0;  // shared-border maps on both sides
  if (!ep.bias) ep.bias = cw.b;
  GemmLaunch g;
  PRISMA_TRY(gemm_prepare(&g, in.p + c0, in.rows(), cw.cin, in.C, cw.w, round_up(cw.cout, 256), (int)in.rows(), cw.cout,
                          cw.kh * cw.kw * cw.wsplit, off, ep, num_sms));
  { const double f = 2.0 * in.B * (double)(in.H / sub) * (in.W / sub) * cw.kh * cw.kw * cw.cin * cw.cout;
    if (cur_mask & 1) { flops += f; flops_conv += f; }
    if (cur_mask & 2) flops_conv_video += f; }
  add(name, [g](cudaStream_t s) { return gemm_run(g, s); });
  return 0;
}

// destination = interior of another padded map (possibly different border / stride-2 sub-sampled geometry)
static void to_map(GemmEpilogue& ep, const RMap& dst, int col0, bool relu_copy = false) {
  ep.row_map = ROW_PADDED;
  ep.out_wp = dst.Wp(); ep.out_img_rows = (int)dst.img_rows(); ep.out_pad = dst.pad;
  if (relu_copy) { ep.out_f16_relu = dst.p + col0; ep.out_f16_relu_ld = dst.C; }
  else { ep.out_f16 = dst.p + col0; ep.out_f16_ld = dst.C; }
}

// fnet: conv -> dense fp32 -> InstanceNorm statistics; returns the dense buffer slot used
int RaftEngine::add_conv_in(const char* name, const RMap& in, const ConvW& cw, int sub, float* dense, float* stats) {
  GemmEpilogue ep;
  ep.row_map = ROW_PAD2TOK;
  ep.out_f32 = dense; ep.out_f32_ld = cw.cout;
  ep.stat_part = slab_part;  // sum / sum of squares per 32-row slab, written by the conv epilogue itself
  PRISMA_TRY(add_conv(name, in, 0, cw, ep, sub));
  const int Ho = in.H / sub, Wo = in.W / sub, C = cw.cout, B = in.B;
  const int spi = (int)(in.img_rows() / 32);
  PRISMA_CHECK((size_t)round_up((int)in.rows(), 256) / 32 * 2 * C <= slab_part_floats, "instnorm slab partials exceed their buffer");
  float* sp = slab_part; double* p2 = slab_part2;
  add("instnorm_stats", [=](cudaStream_t s) { return instnorm_stats_from_slabs(sp, B, spi, C, Ho * Wo, p2, stats, s); });
  return 0;
}

int RaftEngine::build_encoder(const EncW& e, bool inorm, const __half* stem_cols, RMap* out_map128, int B) {
  const int H2 = Hp_ / 2, W2 = Wp_ / 2;
  RMap x;
  PRISMA_TRY(new_map(&x, B, H2, W2, 64, 1));
  const int zero_off[1] = {0};
  {  // stem GEMM over the im2col matrix
    GemmEpilogue ep;
    ep.bias = e.stem.b;
    GemmLaunch g;
    if (inorm) {
      ep.out_f32 = dense_a; ep.out_f32_ld = 64;
      PRISMA_TRY(gemm_prepare(&g, stem_cols, (long long)B * H2 * W2, 192, 192, e.stem.w, 256, B * H2 * W2, 64, 1, zero_off, ep, num_sms));
      add("stem_gemm", [g](cudaStream_t s) { return gemm_run(g, s); });
      float* d = dense_a; float* st = stats_a; float* part = in_part; __half* o = x.p;
      add("instnorm_stats", [=](cudaStream_t s) { return instnorm_stats(d, B, H2 * W2, 64, part, st, s); });
      const long long ir = x.img_rows();
      add("instnorm_apply", [=](cudaStream_t s) { return instnorm_apply(d, st, B, H2, W2, 64, nullptr, nullptr, nullptr, o, 1, ir, s); });
    } else {
      ep.act = 2;
      ep.row_map = ROW_TOK2PAD; ep.in_w = W2; ep.in_h = H2; ep.out_wp = x.Wp(); ep.out_img_rows = (int)x.img_rows(); ep.out_pad = 1; ep.out_lead = 0;
      ep.out_f16 = x.p; ep.out_f16_ld = 64;
      PRISMA_TRY(gemm_prepare(&g, stem_cols, (long long)B * H2 * W2, 192, 192, e.stem.w, 256, B * H2 * W2, 64, 1, zero_off, ep, num_sms));
      add("stem_gemm", [g](cudaStream_t s) { return gemm_run(g, s); });
    }
    { const double f = 2.0 * B * H2 * (double)W2 * 147 * 64;
      if (cur_mask & 1) { flops += f; flops_conv += f; }
      if (cur_mask & 2) flops_conv_video += f; }
  }
  const int dims[3] = {64, 96, 128};
  for (int li = 0; li < 3; ++li)
    for (int bi = 0; bi < 2; ++bi) {
      const ResW& r = e.blk[li][bi];
      const int sub = r.has_ds ? 2 : 1;
      const int Ho = x.H / sub, Wo = x.W / sub, C = dims[li];
      RMap y, o;
      PRISMA_TRY(new_map(&y, B, Ho, Wo, C, 1));
      PRISMA_TRY(new_map(&o, B, Ho, Wo, C, 1));
      if (inorm) {
        // y = relu(IN(conv1(x))) ; z = conv2(y) ; out = relu(skip + relu(IN(z))), skip = x or IN(downsample(x))
        PRISMA_TRY(add_conv_in("res_conv1", x, r.c1, sub, dense_a, stats_a));
        { float* d = dense_a; float* st = stats_a; __half* yo = y.p;
          const long long ir = y.img_rows();
          add("instnorm_apply", [=](cudaStream_t s) { return instnorm_apply(d, st, B, Ho, Wo, C, nullptr, nullptr, nullptr, yo, 1, ir, s); }); }
        PRISMA_TRY(add_conv_in("res_conv2", y, r.c2, 1, dense_a, stats_a));
        if (r.has_ds) {
          PRISMA_TRY(add_conv_in("res_downsample", x, r.ds, 2, dense_b, stats_b));
          float* d = dense_a; float* st = stats_a; float* d2 = dense_b; float* st2 = stats_b; __half* oo = o.p;
          const long long ir = o.img_rows();
          add("instnorm_apply", [=](cudaStream_t s) { return instnorm_apply(d, st, B, Ho, Wo, C, nullptr, d2, st2, oo, 1, ir, s); });
        } else {
          float* d = dense_a; float* st = stats_a; const __half* sk = x.p; __half* oo = o.p;
          const long long ir = o.img_rows();
          add("instnorm_apply", [=](cudaStream_t s) { return instnorm_apply(d, st, B, Ho, Wo, C, sk, nullptr, nullptr, oo, 1, ir, s); });
        }
      } else {
        // BatchNorm folded: y = relu(conv1'(x)) ; out = relu(skip + relu(conv2'(y)))
        { GemmEpilogue ep; ep.act = 2;
          if (sub > 1) to_map(ep, y, 0); else { ep.out_f16 = y.p; ep.out_f16_ld = C; }
          PRISMA_TRY(add_conv("res_conv1", x, 0, r.c1, ep, sub)); }
        const __half* skip = x.p;
        if (r.has_ds) {
          RMap d;
          PRISMA_TRY(new_map(&d, B, Ho, Wo, C, 1));
          GemmEpilogue ep; to_map(ep, d, 0);
          PRISMA_TRY(add_conv("res_downsample", x, 0, r.ds, ep, 2));
          skip = d.p;
        }
        { GemmEpilogue ep; ep.act = 2; ep.res_a = skip; ep.res_a_ld = C; ep.out_f16_relu = o.p; ep.out_f16_relu_ld = C;
          PRISMA_TRY(add_conv("res_conv2", y, 0, r.c2, ep, 1)); }
      }
      x = o;
    }
  *out_map128 = x;
  return 0;
}

int RaftEngine::set_pairs_per_pass(int np) {
  PRISMA_CHECK(np >= 1 && np <= 4, "pairs per pass must be in [1, 4]");
  stream_pairs = np;
  return 0;
}

// Pairs per pass the clip path uses for frames of this size: the setting, lowered until the fp32 correlation pyramids of
// one pass (2 np directions x P^2 x 4 bytes x 4/3) fit in a third of the device memory (4K frames: one pair per pass).
int RaftEngine::clip_pairs(int H, int W, double scale) const {
  const int hs = (int)nearbyint((double)H * scale), ws = (int)nearbyint((double)W * scale);
  const double P = (double)((hs + 7) / 8) * ((ws + 7) / 8);
  const double per_pair = 2.0 * P * P * 4.0 * (4.0 / 3.0);
  int np = stream_pairs;
  while (np > 1 && per_pair * np > (double)device_mem / 3.0) --np;
  return np;
}

int RaftEngine::use_pairs(int np) {
  if (np != npairs) { npairs = np; cache_valid = false; }  // build_plan sees plan_B != 2 * npairs and rebuilds
  return 0;
}

int RaftEngine::build_plan(int H, int W, double scale, int iters_) {
  PRISMA_CHECK(finalized, "weights not finalized");
  PRISMA_CHECK(iters_ >= 1 && iters_ <= 64, "iterations must be in [1,64]");
  if (plan_H == H && plan_W == W && plan_scale == scale && iters == iters_ && plan_B == 2 * npairs) return 0;
  PRISMA_CUDA_OK(cudaSetDevice(device));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  for (void* q : plan_allocs) cudaFree(q);
  plan_allocs.clear();
  steps.clear();
  taps.clear();
  delete corr; corr = nullptr;
  if (graph_exec) { cudaGraphExecDestroy(graph_exec); graph_exec = nullptr; }
  if (graph_cached) { cudaGraphExecDestroy(graph_cached); graph_cached = nullptr; }
  cache_valid = false; cur_mask = 3;
  plan_H = plan_W = 0; flops = flops_conv = flops_conv_video = 0; iters = iters_;

  Hs = (int)nearbyint((double)H * scale); Ws = (int)nearbyint((double)W * scale);  // cv::resize: dsize = cvRound(src * fx)
  const int pad_h = (((Hs / 8) + 1) * 8 - Hs) % 8, pad_w = (((Ws / 8) + 1) * 8 - Ws) % 8;  // common/flow.py:46-53
  pads[0] = pad_w / 2; pads[1] = pad_w - pad_w / 2; pads[2] = pad_h / 2; pads[3] = pad_h - pad_h / 2;
  Hp_ = Hs + pad_h; Wp_ = Ws + pad_w;
  H8 = Hp_ / 8; W8 = Wp_ / 8;
  // One pass = NP consecutive frame pairs of a clip = NF = NP + 1 frames and B = 2 NP (image1, image2) directions: direction
  // 2p is the forward flow of pair p (frame p -> p + 1), 2p + 1 the backward flow (flow_raft.py:105-106).  NP = 2 doubles the
  // rows of every update-block launch (four waves of tiles instead of two), halving the per-pair share of each launch's
  // fixed cost (DESIGN.md section 4.1).
  const int NP = npairs, NF = NP + 1, B = 2 * NP, P = H8 * W8;
  int fr1[8], fr2[8];
  for (int pp = 0; pp < NP; ++pp) { fr1[2 * pp] = pp; fr2[2 * pp] = pp + 1; fr1[2 * pp + 1] = pp + 1; fr2[2 * pp + 1] = pp; }
  plan_B = B;

  PRISMA_TRY(r_alloc(plan_allocs, &b.img, (size_t)NF * H * W * 3));
  PRISMA_TRY(r_alloc(plan_allocs, &b.resized, (size_t)NF * Hs * Ws * 3));
  PRISMA_TRY(r_alloc(plan_allocs, &b.chw, (size_t)NF * 3 * Hp_ * Wp_));
  PRISMA_TRY(r_alloc(plan_allocs, &b.stem_cols, (size_t)NF * (Hp_ / 2) * (Wp_ / 2) * 192));
  const size_t dense_max = (size_t)NF * (Hp_ / 2) * (Wp_ / 2) * 64;  // largest conv output of the encoders (floats)
  PRISMA_TRY(r_alloc(plan_allocs, &dense_a, dense_max));
  PRISMA_TRY(r_alloc(plan_allocs, &dense_b, dense_max / 2));
  PRISMA_TRY(r_alloc(plan_allocs, &stats_a, NF * 256 * 2));
  PRISMA_TRY(r_alloc(plan_allocs, &stats_b, NF * 256 * 2));
  PRISMA_TRY(r_alloc(plan_allocs, &in_part, (size_t)instnorm_partial_floats(NF, (Hp_ / 2) * (Wp_ / 2), 128)));
  {  // per-slab (32 rows) column sums of the conv epilogues: the largest conv input is a pad-1 half-resolution map
    const long long ir = (((long long)(Hp_ / 2 + 1) * (Wp_ / 2 + 1) + 31) / 32) * 32;
    slab_part_floats = (size_t)(round_up((int)(NF * ir), 256) / 32) * 2 * 128;  // CTA-pair tiles cover 256 rows
    PRISMA_TRY(r_alloc(plan_allocs, &slab_part, slab_part_floats));
    PRISMA_TRY(r_alloc(plan_allocs, &slab_part2, (size_t)NF * INSTNORM_STAGE1_BLOCKS * 128 * 2));
  }
  PRISMA_TRY(r_alloc(plan_allocs, &b.coords0, (size_t)B * 2 * P));
  PRISMA_TRY(r_alloc(plan_allocs, &b.coords1, (size_t)B * 2 * P));
  PRISMA_TRY(r_alloc(plan_allocs, &b.cnet_out, (size_t)NF * P * 256));   // per FRAME (slot 0 = the cached previous frame)
  PRISMA_TRY(r_alloc(plan_allocs, &b.flow_up, (size_t)B * Hs * Ws * 2));
  PRISMA_TRY(r_alloc(plan_allocs, &b.rgb, (size_t)B * Hs * Ws * 3));
  PRISMA_TRY(r_alloc(plan_allocs, &b.mm, 8));
  PRISMA_TRY(r_alloc(plan_allocs, &b.maxd, 8));

  corr = new FlowCorr();
  PRISMA_TRY(corr->init(device, B, H8, W8, NF, fr1, fr2));

  // ---- K11 pre-process of both frames, stem im2col (shared by fnet and cnet)
  {
    const uint8_t* img = b.img; uint8_t* rs = b.resized; float* chw = b.chw; __half* cols = b.stem_cols;
    const int Hs_ = Hs, Ws_ = Ws, Hpp = Hp_, Wpp = Wp_;
    const double fx = scale;
    int pd[4] = {pads[0], pads[1], pads[2], pads[3]};
    int pdc[4] = {pads[0], pads[1], pads[2], pads[3]};
    cur_mask = 1;
    add("raft_preprocess", [=](cudaStream_t s) {
      for (int i = 0; i < NF; ++i)
        PRISMA_TRY(raft_preprocess(img + (size_t)i * H * W * 3, H, W, Hs_, Ws_, fx, pd, rs + (size_t)i * Hs_ * Ws_ * 3,
                                   chw + (size_t)i * 3 * Hpp * Wpp, s));
      return 0;
    });
    add("stem_im2col", [=](cudaStream_t s) { return raft_im2col_stem(chw, NF, Hpp, Wpp, cols, s); });
    // video pass: slot 0 (prev) <- slot NP (the last frame of the previous pass) for everything the encoders produced;
    // only the NP new frames are pre-processed and encoded
    cur_mask = 2;
    {
      FlowCorr* c = corr; float* cn = b.cnet_out; uint8_t* rsz = rs; const size_t rbytes = (size_t)Hs_ * Ws_ * 3;
      const size_t cn_n = (size_t)P * 256 * sizeof(float);
      add("reuse_prev", [=](cudaStream_t s) {
        const size_t n = (size_t)c->rows_pad * c->C * sizeof(__half);
        PRISMA_CUDA_OK(cudaMemcpyAsync(c->feat, c->feat + (size_t)NP * c->rows_pad * c->C, n, cudaMemcpyDeviceToDevice, s));
        const size_t pn = (size_t)c->rows123_pad * c->C * sizeof(__half);
        PRISMA_CUDA_OK(cudaMemcpyAsync(c->pool123, c->pool123 + (size_t)NP * c->rows123_pad * c->C, pn, cudaMemcpyDeviceToDevice, s));
        PRISMA_CUDA_OK(cudaMemcpyAsync(cn, reinterpret_cast<const char*>(cn) + NP * cn_n, cn_n, cudaMemcpyDeviceToDevice, s));
        PRISMA_CUDA_OK(cudaMemcpyAsync(rsz, rsz + NP * rbytes, rbytes, cudaMemcpyDeviceToDevice, s));
        return 0;
      });
    }
    add("raft_preprocess", [=](cudaStream_t s) {
      for (int i = 1; i < NF; ++i)
        PRISMA_TRY(raft_preprocess(img + (size_t)i * H * W * 3, H, W, Hs_, Ws_, fx, pdc, rs + (size_t)i * Hs_ * Ws_ * 3,
                                   chw + (size_t)i * 3 * Hpp * Wpp, s));
      return 0;
    });
    add("stem_im2col", [=](cudaStream_t s) {
      return raft_im2col_stem(chw + (size_t)3 * Hpp * Wpp, NP, Hpp, Wpp, cols + (size_t)(Hpp / 2) * (Wpp / 2) * 192, s);
    });
    cur_mask = 3;
  }
  // ---- fnet (instance norm) -> feature maps straight into the correlation operand buffers
  RMap f128, c128, f128c, c128c;
  const __half* cols1 = b.stem_cols + (size_t)(Hp_ / 2) * (Wp_ / 2) * 192;  // im2col rows of frame 1 (the first new frame)
  cur_mask = 1;
  PRISMA_TRY(build_encoder(w.fnet, true, b.stem_cols, &f128, NF));
  { GemmEpilogue ep; ep.row_map = ROW_PAD2TOK; ep.out_img_rows = corr->rows_pad;
    ep.out_f16 = corr->feat; ep.out_f16_ld = 256;
    PRISMA_TRY(add_conv("fnet_out", f128, 0, w.fnet.out, ep, 1)); }
  { FlowCorr* c = corr; add("corr_pool", [=](cudaStream_t s) { return c->pool_frames(0, NF, s); }); }
  cur_mask = 2;  // video pass: encode the NP new frames alone, into slots 1..NP
  PRISMA_TRY(build_encoder(w.fnet, true, cols1, &f128c, NP));
  { GemmEpilogue ep; ep.row_map = ROW_PAD2TOK; ep.out_img_rows = corr->rows_pad;
    ep.out_f16 = corr->feat + (size_t)corr->rows_pad * 256; ep.out_f16_ld = 256;
    PRISMA_TRY(add_conv("fnet_out", f128c, 0, w.fnet.out, ep, 1)); }
  { FlowCorr* c = corr; add("corr_pool", [=](cudaStream_t s) { return c->pool_frames(1, NP, s); }); }
  cur_mask = 3;
  {  // direction b correlates frame fr1[b] against frame fr2[b] (flow_raft.py:105-106): the GEMMs read the per-frame features
    FlowCorr* c = corr;
    add("corr_build", [c](cudaStream_t s) { return c->build_gemms(s); });
    flops += c->flops_build;
  }
  // ---- cnet (batch norm folded) -> tanh / relu split into the GRU operand maps
  cur_mask = 1;
  PRISMA_TRY(build_encoder(w.cnet, false, b.stem_cols, &c128, NF));
  cur_mask = 2;
  PRISMA_TRY(build_encoder(w.cnet, false, cols1, &c128c, NP));
  cur_mask = 3;
  RMap hx, rhx, corrf, c1, c2, f1, fh, mk;
  PRISMA_TRY(new_map(&hx, B, H8, W8, 384, 2));
  PRISMA_TRY(new_map(&rhx, B, H8, W8, 384, 2));
  PRISMA_TRY(r_alloc(plan_allocs, &b.h_master, (size_t)hx.rows() * 128));
  cur_mask = 1;
  { GemmEpilogue ep; ep.row_map = ROW_PAD2TOK; ep.out_f32 = b.cnet_out; ep.out_f32_ld = 256;
    PRISMA_TRY(add_conv("cnet_out", c128, 0, w.cnet.out, ep, 1)); }
  cur_mask = 2;
  { GemmEpilogue ep; ep.row_map = ROW_PAD2TOK; ep.out_f32 = b.cnet_out + (size_t)P * 256; ep.out_f32_ld = 256;
    PRISMA_TRY(add_conv("cnet_out", c128c, 0, w.cnet.out, ep, 1)); }
  cur_mask = 3;
  {
    const float* cn = b.cnet_out; float* hm = b.h_master; __half* hxp = hx.p; __half* rhp = rhx.p; const int h8 = H8, w8 = W8;
    float* c0 = b.coords0; float* c1p = b.coords1; const long long ir8 = hx.img_rows();
    DirFrames df;  // the context features of direction b are those of its image1 frame
    for (int d = 0; d < 8; ++d) df.f[d] = d < B ? fr1[d] : 0;
    add("cnet_split", [=](cudaStream_t s) { return raft_cnet_split(cn, B, h8, w8, 2, ir8, df, hm, hxp, rhp, s); });
    add("coords_init", [=](cudaStream_t s) { return raft_coords_init(c0, c1p, B, h8, w8, s); });
  }
  // ---- update block, `iters` times (raft.py:123-141)
  PRISMA_TRY(new_map(&corrf, B, H8, W8, 384, 2));
  PRISMA_TRY(new_map(&c1, B, H8, W8, 256, 2));
  PRISMA_TRY(new_map(&c2, B, H8, W8, 256, 2));   // [convc2 out (192) | convf2 out (64)]
  PRISMA_TRY(new_map(&f1, B, H8, W8, 128, 2));
  __half* f1_cols = nullptr;
  PRISMA_TRY(r_alloc(plan_allocs, &f1_cols, (size_t)B * H8 * W8 * 256));
  float* zr_f = nullptr;  // gates in fp32, padded-row layout of the pad-2 maps
  PRISMA_TRY(r_alloc(plan_allocs, &zr_f, (size_t)hx.rows() * 256));
  PRISMA_TRY(new_map(&fh, B, H8, W8, 256, 2));
  float* fh2_u = nullptr;
  PRISMA_TRY(r_alloc(plan_allocs, &fh2_u, (size_t)hx.rows() * 32));
  PRISMA_TRY(new_map(&mk, B, H8, W8, 256, 2));
  PRISMA_TRY(r_alloc(plan_allocs, &b.mask, (size_t)hx.rows() * 576));
  for (int it = 0; it < iters; ++it) {
    {
      FlowCorr* c = corr; const float* c1p = b.coords1; __half* dst = corrf.p; const int wp = corrf.Wp(), ir = (int)corrf.img_rows();
      add("corr_lookup", [=](cudaStream_t s) { return c->lookup_to(c1p, dst, 384, wp, 0, ir, s); });  // shared-border map: no leading border
    }
    { GemmEpilogue ep; ep.act = 2; ep.out_f16 = c1.p; ep.out_f16_ld = 256;            // convc1 1x1 324 -> 256
      ConvW cw = w.convc1; cw.cin = 384;  // the lookup map is zero padded to 384 channels, so are the weights' K
      PRISMA_TRY(add_conv("convc1", corrf, 0, cw, ep, 1)); }
    { GemmEpilogue ep; ep.act = 2; ep.out_f16 = c2.p; ep.out_f16_ld = 256;            // convc2 3x3 256 -> 192
      PRISMA_TRY(add_conv("convc2", c1, 0, w.convc2, ep, 1)); }
    {
      // convf1 7x7 on the flow: im2col with an fp16 hi/lo split of every value (K = 256) + one GEMM, ReLU, -> padded map
      const float* c0 = b.coords0; const float* c1p = b.coords1; __half* cols = f1_cols; const int h8 = H8, w8 = W8;
      add("convf1_im2col", [=](cudaStream_t s) { return raft_flow_im2col(c0, c1p, B, h8, w8, cols, s); });
      GemmEpilogue ep; ep.bias = w.convf1_b; ep.act = 2; ep.out_f16 = f1.p; ep.out_f16_ld = 128;
      ep.row_map = ROW_TOK2PAD; ep.in_w = W8; ep.in_h = H8; ep.out_wp = f1.Wp(); ep.out_img_rows = (int)f1.img_rows(); ep.out_pad = 2; ep.out_lead = 0;
      GemmLaunch g;
      const int zoff[1] = {0};
      PRISMA_TRY(gemm_prepare(&g, f1_cols, (long long)B * H8 * W8, 256, 256, w.convf1_gemm_w, 256, B * H8 * W8, 128, 1, zoff, ep, num_sms));
      { const double f = 2.0 * B * H8 * (double)W8 * 98.0 * 128; flops += f; flops_conv += f; flops_conv_video += f; }
      add("convf1_gemm", [g](cudaStream_t s) { return gemm_run(g, s); });
    }
    { GemmEpilogue ep; ep.act = 2; ep.out_f16 = c2.p + 192; ep.out_f16_ld = 256;      // convf2 3x3 128 -> 64
      PRISMA_TRY(add_conv("convf2", f1, 0, w.convf2, ep, 1)); }
    { // conv 3x3 256 -> 126 (+2 zero channels); the 126 motion channels go to cols 256..381 of hx and rhx; the two
      // trailing columns are rewritten with the flow by flow_cols every iteration -- so restore them here
      GemmEpilogue ep; ep.act = 2; ep.out_f16 = hx.p + 256; ep.out_f16_ld = 384; ep.out_f16_relu = rhx.p + 256; ep.out_f16_relu_ld = 384;
      PRISMA_TRY(add_conv("motion_conv", c2, 0, w.conv, ep, 1));
      const float* c0 = b.coords0; const float* c1p = b.coords1; __half* hxp = hx.p; __half* rhp = rhx.p; const int h8 = H8, w8 = W8;
      const long long ir8 = hx.img_rows();
      add("flow_cols", [=](cudaStream_t s) { return raft_flow_cols(c0, c1p, B, h8, w8, 2, ir8, hxp, rhp, s); });
    }
    for (int pass = 0; pass < 2; ++pass) {  // SepConvGRU horizontal then vertical (update.py:45-60)
      // gate arithmetic in the conv epilogues: r * h -> the q conv's operand; h' = (1 - z) h + z q -> fp32 master + operand copy
      { GemmEpilogue ep; ep.act = 3; ep.out_f32 = zr_f; ep.out_f32_ld = 256;
        ep.gru = 1; ep.gru_h = b.h_master; ep.gru_rh = rhx.p; ep.gru_rh_ld = 384;
        PRISMA_TRY(add_conv("gru_zr", hx, 0, w.zr[pass], ep, 1)); }
      { GemmEpilogue ep; ep.act = 4; ep.out_f32 = b.h_master; ep.out_f32_ld = 128; ep.out_f16 = hx.p; ep.out_f16_ld = 384;
        ep.gru = 2; ep.gru_h = b.h_master; ep.gru_z = zr_f;
        PRISMA_TRY(add_conv("gru_q", rhx, 0, w.q[pass], ep, 1)); }
    }
    { GemmEpilogue ep; ep.act = 2; ep.out_f16 = fh.p; ep.out_f16_ld = 256;            // flow head
      ConvW cw = w.fh1;
      PRISMA_TRY(add_conv("flow_head1", hx, 0, cw, ep, 1)); }
    { // flow_head.conv2: 1x1 GEMM to the 18 per-tap partial products, then the nine-tap gather + coords1 += delta (raft.py:133)
      GemmEpilogue ep; ep.out_f32 = fh2_u; ep.out_f32_ld = 32;
      PRISMA_TRY(add_conv("flow_head2", fh, 0, w.fh2u, ep, 1));
      const float* up = fh2_u; const float b0 = w.fh2_b[0], b1 = w.fh2_b[1]; float* c1p = b.coords1;
      const int h8 = H8, w8 = W8; const long long ir8 = fh.img_rows();
      add("coords_update", [=](cudaStream_t s) { return raft_flow_head2_gather(up, B, h8, w8, 2, ir8, b0, b1, c1p, s); }); }
    if (debug_taps && it == 0) {
      PRISMA_TRY(r_alloc(plan_allocs, &b.h_tap, (size_t)hx.rows() * 128));
      PRISMA_TRY(r_alloc(plan_allocs, &b.coords_tap, (size_t)B * 2 * P));
      float* ht = b.h_tap; const float* hm = b.h_master; float* ct = b.coords_tap; const float* c1p = b.coords1;
      const size_t n1 = (size_t)hx.rows() * 128 * 4, n2 = (size_t)B * 2 * P * 4;
      add("tap_iter0", [=](cudaStream_t s) {
        PRISMA_CUDA_OK(cudaMemcpyAsync(ht, hm, n1, cudaMemcpyDeviceToDevice, s));
        PRISMA_CUDA_OK(cudaMemcpyAsync(ct, c1p, n2, cudaMemcpyDeviceToDevice, s));
        return 0;
      });
    }
  }
  // ---- up-sampling mask (last iteration only) + convex up-sampling + unpad + HWC
  { GemmEpilogue ep; ep.act = 2; ep.out_f16 = mk.p; ep.out_f16_ld = 256;
    PRISMA_TRY(add_conv("mask_head1", hx, 0, w.mk1, ep, 1)); }
  { GemmEpilogue ep; ep.out_f32 = b.mask; ep.out_f32_ld = 576;  // the 0.25 is folded (exactly) into the fp16 weights and the bias
    PRISMA_TRY(add_conv("mask_head2", mk, 0, w.mk2, ep, 1)); }
  {
    const float* m = b.mask; const float* c0 = b.coords0; const float* c1p = b.coords1; float* up = b.flow_up;
    const int h8 = H8, w8 = W8, Hs_ = Hs, Ws_ = Ws, pt = pads[2], pl = pads[0];
    const long long ir8 = hx.img_rows();
    add("convex_upsample", [=](cudaStream_t s) { return raft_convex_upsample(m, c0, c1p, B, h8, w8, 2, ir8, Hs_, Ws_, pt, pl, up, s); });
    uint8_t* rgb = b.rgb; uint32_t* mm = b.mm; float* mx = b.maxd; const int sms = num_sms;
    add("flow_encode", [=](cudaStream_t s) {
      for (int i = 0; i < B; ++i)
        PRISMA_TRY(flow_encode(up + (size_t)i * Hs_ * Ws_ * 2, Hs_, Ws_, rgb + (size_t)i * Hs_ * Ws_ * 3, mm + i, mx + i, sms, s));
      return 0;
    });
  }
  taps["resized"] = {b.resized, NF * Hs, Ws * 3, 1, 3};
  taps["fmap"] = {corr->feat, 0, 0, 0, 4};
  taps["cnet_out"] = {b.cnet_out, NF * P, 256, 1, 0};
  taps["coords1_iter0"] = {b.coords_tap, B * 2, P, 1, 0};
  taps["h_iter0"] = {b.h_tap, (int)hx.rows(), 128, 1, 0};
  taps["coords1"] = {b.coords1, B * 2, P, 1, 0};
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  plan_H = H; plan_W = W; plan_scale = scale;
  if (use_graph) {
    for (int which = 1; which <= 2; ++which) {
      PRISMA_TRY(run_direct(stream, which));  // warm: per-kernel attributes are set outside the capture
      PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
      cudaGraph_t graph = nullptr;
      PRISMA_CUDA_OK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
      int r = run_direct(stream, which);
      cudaError_t e = cudaStreamEndCapture(stream, &graph);
      if (r != 0) { if (graph) cudaGraphDestroy(graph); return r; }
      PRISMA_CUDA_OK(e);
      PRISMA_CUDA_OK(cudaGraphInstantiate(which == 1 ? &graph_exec : &graph_cached, graph, 0));
      cudaGraphDestroy(graph);
    }
  }
  return 0;
}

int RaftEngine::run_direct(cudaStream_t s, int which) {
  for (auto& st : steps)
    if (st.group & which) { NvtxRange r(st.name); PRISMA_TRY(st.fn(s)); }
  return 0;
}

int RaftEngine::infer(const uint8_t* prev, const uint8_t* curr, int H, int W, double scale, int iters_, float* fwd, float* bwd,
                      uint8_t* fwd_rgb, uint8_t* bwd_rgb, float* max_fwd, float* max_bwd, float* ms_out, int reuse_prev) {
  PRISMA_CHECK(curr && (prev || reuse_prev) && H > 0 && W > 0, "bad frame pair");
  NvtxRange nvtx_pass("prisma.flow_raft.infer");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  use_pairs(1);
  PRISMA_TRY(build_plan(H, W, scale, iters_));
  const int which = (reuse_prev && cache_valid) ? 2 : 1;
  PRISMA_CHECK(which == 2 || prev != nullptr, "no cached features for the previous frame: pass it");
  cache_valid = false;
  const size_t fb = (size_t)H * W * 3;
  if (which == 1) PRISMA_CUDA_OK(cudaMemcpyAsync(b.img, prev, fb, cudaMemcpyHostToDevice, stream));
  PRISMA_CUDA_OK(cudaMemcpyAsync(b.img + fb, curr, fb, cudaMemcpyHostToDevice, stream));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (ms_out) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, stream); }
  if (getenv("PRISMA_RAFT_PROFILE")) {  // per-step CUDA-event times, aggregated by step name (diagnostics)
    std::vector<cudaEvent_t> ev(steps.size() + 1);
    for (auto& e : ev) cudaEventCreate(&e);
    cudaEventRecord(ev[0], stream);
    for (size_t i = 0; i < steps.size(); ++i) { if (steps[i].group & which) PRISMA_TRY(steps[i].fn(stream)); cudaEventRecord(ev[i + 1], stream); }
    PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
    std::map<std::string, std::pair<int, float>> agg;
    float tot = 0;
    for (size_t i = 0; i < steps.size(); ++i) {
      float t = 0;
      cudaEventElapsedTime(&t, ev[i], ev[i + 1]);
      agg[steps[i].name].first++; agg[steps[i].name].second += t; tot += t;
    }
    for (auto& e : ev) cudaEventDestroy(e);
    std::vector<std::pair<float, std::string>> v;
    for (auto& kv : agg) v.push_back({kv.second.second, kv.first + " x" + std::to_string(kv.second.first)});
    std::sort(v.rbegin(), v.rend());
    printf("RAFT step profile (%.3f ms total, ungraphed):\n", tot);
    for (auto& x : v) printf("  %8.3f ms  %5.1f %%  %s\n", x.first, 100.f * x.first / tot, x.second.c_str());
  } else if (graph_exec) PRISMA_CUDA_OK(cudaGraphLaunch(which == 1 ? graph_exec : graph_cached, stream));
  else PRISMA_TRY(run_direct(stream, which));
  if (ms_out) cudaEventRecord(e1, stream);
  const size_t n = (size_t)Hs * Ws;
  float mx[2] = {0, 0};
  if (fwd) PRISMA_CUDA_OK(cudaMemcpyAsync(fwd, b.flow_up, n * 8, cudaMemcpyDeviceToHost, stream));
  if (bwd) PRISMA_CUDA_OK(cudaMemcpyAsync(bwd, b.flow_up + n * 2, n * 8, cudaMemcpyDeviceToHost, stream));
  if (fwd_rgb) PRISMA_CUDA_OK(cudaMemcpyAsync(fwd_rgb, b.rgb, n * 3, cudaMemcpyDeviceToHost, stream));
  if (bwd_rgb) PRISMA_CUDA_OK(cudaMemcpyAsync(bwd_rgb, b.rgb + n * 3, n * 3, cudaMemcpyDeviceToHost, stream));
  PRISMA_CUDA_OK(cudaMemcpyAsync(mx, b.maxd, 8, cudaMemcpyDeviceToHost, stream));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  if (ms_out) { cudaEventElapsedTime(ms_out, e0, e1); cudaEventDestroy(e0); cudaEventDestroy(e1); }
  if (max_fwd) *max_fwd = mx[0];
  if (max_bwd) *max_bwd = mx[1];
  cache_valid = true;  // slot 1 now holds the features of `curr`
  return 0;
}


// ------------------------------------------------------------------------------------------------ streamed clip path
int RaftEngine::ensure_stream_slots(int H, int W) {
  if (!s_in) {
    PRISMA_CUDA_OK(cudaStreamCreateWithFlags(&s_in, cudaStreamNonBlocking));
    PRISMA_CUDA_OK(cudaStreamCreateWithFlags(&s_out, cudaStreamNonBlocking));
    for (auto& sl : slot)
      for (cudaEvent_t* e : {&sl.loaded, &sl.consumed, &sl.done, &sl.drained})
        PRISMA_CUDA_OK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
  }
  const size_t in_bytes = (size_t)npairs * H * W * 3, out_px = (size_t)npairs * Hs * Ws;  // per pass: NP frames in, NP pairs out
  if (slot_in_bytes == in_bytes && slot_out_px == out_px) return 0;
  PRISMA_CUDA_OK(cudaDeviceSynchronize());
  for (auto& sl : slot) {
    cudaFree(sl.in); cudaFree(sl.flow); cudaFree(sl.rgb); cudaFree(sl.mx);
    sl.in = sl.rgb = nullptr; sl.flow = sl.mx = nullptr;
    PRISMA_CUDA_OK(cudaMalloc(&sl.in, in_bytes));
    PRISMA_CUDA_OK(cudaMalloc(&sl.flow, 2 * out_px * 2 * sizeof(float)));
    PRISMA_CUDA_OK(cudaMalloc(&sl.rgb, 2 * out_px * 3));
    PRISMA_CUDA_OK(cudaMalloc(&sl.mx, 8 * sizeof(float)));
  }
  slot_in_bytes = in_bytes; slot_out_px = out_px;
  return 0;
}

// process_video's loop (bands/flow_raft.py:97-115) over a chunk: every frame is uploaded once and encoded once (video
// pass); s_in uploads frame j+1 into a staging slot while `stream` replays the graph of pair j and s_out drains pair j-1.
int RaftEngine::infer_stream(const uint8_t* frames, int n, int H, int W, double scale, int iters_, int continue_clip,
                             float* fwd, float* bwd, uint8_t* fwd_rgb, uint8_t* bwd_rgb, float* max_fwd, float* max_bwd,
                             int* pairs_out) {
  PRISMA_CHECK(frames != nullptr && H > 0 && W > 0 && n >= 1, "bad frame chunk");
  NvtxRange nvtx_pass("prisma.flow_raft.infer_stream");
  PRISMA_CUDA_OK(cudaSetDevice(device));
  use_pairs(clip_pairs(H, W, scale));
  const bool same_plan = (plan_H == H && plan_W == W && plan_scale == scale && iters == iters_ && plan_B == 2 * npairs);
  PRISMA_TRY(build_plan(H, W, scale, iters_));
  PRISMA_TRY(ensure_stream_slots(H, W));
  const bool cont = continue_clip && cache_valid && same_plan;
  const int pairs = cont ? n : n - 1;
  if (pairs_out) *pairs_out = pairs;
  if (pairs <= 0) {  // a single frame without history: nothing to pair it with; keep it as the next chunk's `prev`?  No:
    cache_valid = false;  // its features are not computed by any pass, so the next chunk must start a new clip
    return 0;
  }
  const int NP = npairs, B = 2 * NP;
  const int passes = (pairs + NP - 1) / NP;
  if (mx_host_pairs < (size_t)passes * NP) {
    if (mx_host) cudaFreeHost(mx_host);
    mx_host = nullptr; mx_host_pairs = 0;
    PRISMA_CUDA_OK(cudaMallocHost(&mx_host, (size_t)passes * NP * 8));
    mx_host_pairs = (size_t)passes * NP;
  }
  const size_t fb = (size_t)H * W * 3, px = (size_t)Hs * Ws;
  const int first_curr = cont ? 0 : 1;  // index of the `curr` frame of pair 0
  cache_valid = false;
  if (!cont) PRISMA_CUDA_OK(cudaMemcpyAsync(b.img, frames, fb, cudaMemcpyHostToDevice, stream));  // `prev` of pair 0
  // pass g covers pairs [g NP, g NP + NP): its new frames are first_curr + g NP + p.  A last pass with fewer pairs than NP
  // repeats the final frame (the extra pair is computed and dropped; the cached slot still ends up holding the last frame).
  auto drain = [&](int g) -> int {
    StreamSlot& sl = slot[g & 1];
    PRISMA_CUDA_OK(cudaStreamWaitEvent(s_out, sl.done, 0));
    for (int p = 0; p < NP; ++p) {
      const int j = g * NP + p;
      if (j >= pairs) break;
      if (fwd) PRISMA_CUDA_OK(cudaMemcpyAsync(fwd + (size_t)j * px * 2, sl.flow + (size_t)(2 * p) * px * 2, px * 8, cudaMemcpyDeviceToHost, s_out));
      if (bwd) PRISMA_CUDA_OK(cudaMemcpyAsync(bwd + (size_t)j * px * 2, sl.flow + (size_t)(2 * p + 1) * px * 2, px * 8, cudaMemcpyDeviceToHost, s_out));
      if (fwd_rgb) PRISMA_CUDA_OK(cudaMemcpyAsync(fwd_rgb + (size_t)j * px * 3, sl.rgb + (size_t)(2 * p) * px * 3, px * 3, cudaMemcpyDeviceToHost, s_out));
      if (bwd_rgb) PRISMA_CUDA_OK(cudaMemcpyAsync(bwd_rgb + (size_t)j * px * 3, sl.rgb + (size_t)(2 * p + 1) * px * 3, px * 3, cudaMemcpyDeviceToHost, s_out));
    }
    PRISMA_CUDA_OK(cudaMemcpyAsync(mx_host + (size_t)g * B, sl.mx, B * sizeof(float), cudaMemcpyDeviceToHost, s_out));
    PRISMA_CUDA_OK(cudaEventRecord(sl.drained, s_out));
    return 0;
  };
  for (int g = 0; g < passes; ++g) {
    StreamSlot& sl = slot[g & 1];
    const int which = (g == 0 && !cont) ? 1 : 2;
    if (g >= 2) PRISMA_CUDA_OK(cudaStreamWaitEvent(s_in, sl.consumed, 0));
    for (int p = 0; p < NP; ++p) {
      const int fi = std::min(first_curr + g * NP + p, n - 1);
      PRISMA_CUDA_OK(cudaMemcpyAsync(sl.in + (size_t)p * fb, frames + (size_t)fi * fb, fb, cudaMemcpyHostToDevice, s_in));
    }
    PRISMA_CUDA_OK(cudaEventRecord(sl.loaded, s_in));
    PRISMA_CUDA_OK(cudaStreamWaitEvent(stream, sl.loaded, 0));
    PRISMA_CUDA_OK(cudaMemcpyAsync(b.img + fb, sl.in, NP * fb, cudaMemcpyDeviceToDevice, stream));
    PRISMA_CUDA_OK(cudaEventRecord(sl.consumed, stream));
    if (graph_exec) PRISMA_CUDA_OK(cudaGraphLaunch(which == 1 ? graph_exec : graph_cached, stream));
    else PRISMA_TRY(run_direct(stream, which));
    if (g >= 2) PRISMA_CUDA_OK(cudaStreamWaitEvent(stream, sl.drained, 0));
    if (fwd || bwd) PRISMA_CUDA_OK(cudaMemcpyAsync(sl.flow, b.flow_up, B * px * 8, cudaMemcpyDeviceToDevice, stream));
    if (fwd_rgb || bwd_rgb) PRISMA_CUDA_OK(cudaMemcpyAsync(sl.rgb, b.rgb, B * px * 3, cudaMemcpyDeviceToDevice, stream));
    PRISMA_CUDA_OK(cudaMemcpyAsync(sl.mx, b.maxd, B * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    PRISMA_CUDA_OK(cudaEventRecord(sl.done, stream));
    if (g >= 1) PRISMA_TRY(drain(g - 1));
  }
  PRISMA_TRY(drain(passes - 1));
  PRISMA_CUDA_OK(cudaStreamSynchronize(s_out));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  for (int j = 0; j < pairs; ++j) {
    if (max_fwd) max_fwd[j] = mx_host[2 * j];
    if (max_bwd) max_bwd[j] = mx_host[2 * j + 1];
  }
  cache_valid = true;  // slot NP of the feature buffers holds the last frame of the chunk
  return 0;
}

int RaftEngine::time_resident(int H, int W, double scale, int iters_, int reps, float* ms_per_pass) {
  PRISMA_CUDA_OK(cudaSetDevice(device));
  use_pairs(clip_pairs(H, W, scale));
  PRISMA_TRY(build_plan(H, W, scale, iters_));
  const int which = cache_valid ? 2 : 1;
  auto once = [&]() -> int {
    if (graph_exec) PRISMA_CUDA_OK(cudaGraphLaunch(which == 1 ? graph_exec : graph_cached, stream));
    else PRISMA_TRY(run_direct(stream, which));
    return 0;
  };
  cudaEvent_t e0, e1;
  PRISMA_CUDA_OK(cudaEventCreate(&e0));
  PRISMA_CUDA_OK(cudaEventCreate(&e1));
  PRISMA_TRY(once());
  PRISMA_CUDA_OK(cudaEventRecord(e0, stream));
  for (int i = 0; i < std::max(reps, 1); ++i) PRISMA_TRY(once());
  PRISMA_CUDA_OK(cudaEventRecord(e1, stream));
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  float t = 0;
  PRISMA_CUDA_OK(cudaEventElapsedTime(&t, e0, e1));
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (ms_per_pass) *ms_per_pass = t / std::max(reps, 1);
  return 0;
}

// Per-group CUDA-event times of one ungraphed pass (video pass when the previous frame's features are cached):
// out[0] pre-process + stem im2col, [1] conv GEMMs (encoders + update block + heads), [2] correlation build,
// [3] correlation lookup, [4] InstanceNorm, [5] other pointwise (GRU gates, coords, flow im2col, ...), [6] convex
// up-sampling + HSV encode, [7] total.
int RaftEngine::profile(int H, int W, double scale, int iters_, float* out8) {
  PRISMA_CUDA_OK(cudaSetDevice(device));
  use_pairs(clip_pairs(H, W, scale));
  PRISMA_TRY(build_plan(H, W, scale, iters_));
  const int which = cache_valid ? 2 : 1;
  for (int i = 0; i < 8; ++i) out8[i] = 0.f;
  std::vector<cudaEvent_t> ev(steps.size() + 1);
  for (auto& e : ev) PRISMA_CUDA_OK(cudaEventCreate(&e));
  PRISMA_TRY(run_direct(stream, which));  // warm
  PRISMA_CUDA_OK(cudaEventRecord(ev[0], stream));
  for (size_t i = 0; i < steps.size(); ++i) {
    if (steps[i].group & which) PRISMA_TRY(steps[i].fn(stream));
    PRISMA_CUDA_OK(cudaEventRecord(ev[i + 1], stream));
  }
  PRISMA_CUDA_OK(cudaStreamSynchronize(stream));
  for (size_t i = 0; i < steps.size(); ++i) {
    if (!(steps[i].group & which)) continue;
    float t = 0;
    cudaEventElapsedTime(&t, ev[i], ev[i + 1]);
    const std::string n = steps[i].name;
    int g = 5;
    if (n == "raft_preprocess" || n == "stem_im2col" || n == "reuse_prev" || n == "fmap_swap") g = 0;
    else if (n == "corr_build") g = 2;
    else if (n == "corr_lookup") g = 3;
    else if (n.rfind("instnorm", 0) == 0) g = 4;
    else if (n == "convex_upsample" || n == "flow_encode") g = 6;
    else if (n == "convf1_im2col") g = 5;
    else if (n == "stem_gemm" || n == "convf1_gemm" || n.rfind("res_", 0) == 0 || n.rfind("conv", 0) == 0 || n == "fnet_out" ||
             n == "cnet_out" || n == "motion_conv" || n.rfind("gru_zr", 0) == 0 || n == "gru_q" || n == "gru_inp" || n.rfind("flow_head", 0) == 0 ||
             n.rfind("mask_head", 0) == 0) g = 1;
    out8[g] += t; out8[7] += t;
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return 0;
}

long long RaftEngine::read_tap(const std::string& name, float* out, long long capacity) {
  auto it = taps.find(name);
  if (it == taps.end()) { set_last_error("unknown tap '" + name + "'"); return -1; }
  cudaSetDevice(device);
  const Tap& t = it->second;
  if (t.kind == 4) {  // fnet feature maps: fp16 [2][rows_pad][256] -> dense f32 [2][P][256]
    const long long P = (long long)H8 * W8, n = 2 * P * 256;
    if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
    std::vector<__half> h((size_t)2 * corr->rows_pad * 256);
    if (cudaMemcpy(h.data(), t.p, h.size() * 2, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    for (int b2 = 0; b2 < 2; ++b2)
      for (long long i = 0; i < P * 256; ++i) out[b2 * P * 256 + i] = __half2float(h[(size_t)b2 * corr->rows_pad * 256 + i]);
    return n;
  }
  const long long n = (long long)t.a * t.b;
  if (n > capacity) { set_last_error("tap buffer too small"); return -1; }
  if (t.kind == 0) {
    if (cudaMemcpy(out, t.p, n * 4, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
  } else {  // u8
    std::vector<uint8_t> h(n);
    if (cudaMemcpy(h.data(), t.p, n, cudaMemcpyDeviceToHost) != cudaSuccess) { set_last_error("tap copy failed"); return -2; }
    for (long long i = 0; i < n; ++i) out[i] = h[i];
  }
  return n;
}

}  // namespace prisma
