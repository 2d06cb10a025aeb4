/* prisma_b200 -- C ABI of the B200-native per-frame inference engine for PRISMA's band pipeline.
 *
 * The reference (patriciogonzalezvivo/prisma @ e00192dd) is pure Python and has no FFI; each entry point
 * below replaces the body of one reference function, cited as file:line relative to the reference root.
 * Conventions (SURVEY.md section 8b): 0 = OK, negative = error (text via prisma_last_error(), thread-local);
 * nothing throws or exits across the ABI; the caller owns every host buffer, the engine owns device memory,
 * streams and weights; one engine handle is not re-entrant, different handles are independent.
 * All pointers are plain host pointers (pinned or pageable); no torch / numpy types appear here.
 */
#ifndef PRISMA_B200_H
#define PRISMA_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct prisma_engine prisma_engine;

/* ---- library ------------------------------------------------------------------------------------------- */
const char* prisma_last_error(void);
int prisma_device_count(void);          /* number of visible CUDA devices, or negative on error            */
const char* prisma_version(void);

/* ---- Depth-Anything band: replaces bands/depth_anything.py:init_model (:48-76) + infer (:100-143)
 *      + the per-frame encode of process_video (:215-221)                                                  */
/* encoder: "vits" | "vitb" | "vitl" (bands/depth_anything.py:263)                                          */
int prisma_depth_create(const char* encoder, int device, prisma_engine** out);
/* Weight converter input: one call per tensor of the reference state_dict of DPT_DINOv2
 * (bands/d_anything/dpt.py:139-153; names as in SURVEY.md Appendix B), fp32, row-major, host memory.       */
int prisma_depth_load_tensor(prisma_engine* e, const char* name, const float* data, const int64_t* shape, int ndim);
/* Packs the tensors into kernel layouts (fp16 operands, padded K, folded q-scale) and uploads them.        */
int prisma_depth_finalize(prisma_engine* e);
/* One frame.  rgb: h*w*3 u8 RGB.  depth_out (h*w f32, may be NULL) = infer(img) of the reference;
 * rgb_out (h*w*3 u8, may be NULL) = (heat_to_rgb(1 - normalised depth) * 255).astype(u8) (:215-220);
 * min_out / max_out = the per-frame scalars written to <band>_min.csv / _max.csv (:221,231-238).
 * Includes the H2D copy of the frame and the D2H copies of the requested outputs.                          */
int prisma_depth_infer(prisma_engine* e, const uint8_t* rgb, int h, int w, float* depth_out, uint8_t* rgb_out,
                       float* min_out, float* max_out);
/* n frames of one size in one pass (rgb: n*h*w*3; outputs n-major; min_out/max_out: n floats each).  Frames are
 * independent (bands/depth_anything.py:203-221 carries no state across iterations); batching only raises the
 * tile count of every launch.  Results are identical to n calls of prisma_depth_infer.                     */
int prisma_depth_infer_batch(prisma_engine* e, const uint8_t* rgb, int n, int h, int w, float* depth_out,
                             uint8_t* rgb_out, float* min_out, float* max_out);
/* A chunk of the video loop (bands/depth_anything.py:203-221): n frames processed in passes of `pass_frames` (<=0: 4)
 * with the upload of pass i+1 and the download of pass i-1 overlapping the compute of pass i (three streams, two staging
 * slots in HBM).  Same results as n prisma_depth_infer calls.  Host buffers from prisma_host_alloc (pinned) make the
 * copies true asynchronous DMA; pageable buffers work too (the driver stages them).                                  */
int prisma_depth_infer_stream(prisma_engine* e, const uint8_t* rgb, int n, int h, int w, int pass_frames, float* depth_out,
                              uint8_t* rgb_out, float* min_out, float* max_out);
/* Page-locked host memory for frame buffers ("frame in pinned host memory", SURVEY section 8d timed region). */
int prisma_host_alloc(size_t bytes, void** out);
int prisma_host_free(void* p);
/* Same computation with the n frames already resident in device memory and outputs left on the device
 * (bench.py's kernel-only leg): ms per pass (CUDA events on the engine stream) over `iters` passes.       */
int prisma_depth_infer_resident(prisma_engine* e, int h, int w, int n, int iters, float* ms_per_iter);
/* Encoder-only entry used by the parity tests: encode a given h*w f32 prediction (:215-220).               */
int prisma_depth_encode(prisma_engine* e, const float* prediction, int h, int w, int flip, uint8_t* rgb_out,
                        float* min_out, float* max_out);
/* Still-image path = process_image (bands/depth_anything.py:146-174): the prediction is encoded by write_depth
 * (bands/common/io.py:138-166: heat map, Sobel edges in the saturation, (min,max) packed into pixels (0,0),(0,1));
 * png_rgb_out is the h*w*3 RGB array the reference hands to cv2.imwrite.  prisma_depth_encode_png is that encoder
 * alone on a given prediction (parity tests).                                                               */
int prisma_depth_infer_image(prisma_engine* e, const uint8_t* rgb, int h, int w, float* depth_out, uint8_t* png_rgb_out,
                             float* min_out, float* max_out);
int prisma_depth_encode_png(prisma_engine* e, const float* prediction, int h, int w, int flip, uint8_t* rgb_out,
                            float* min_out, float* max_out);
/* Intermediate tensors of the last prisma_depth_infer call as dense fp32 (tests only):
 * "net_input" [3][hn][wn], "tokens" [T][D], "feat0".."feat3" [T][D], "net_depth" [hn][wn], ...
 * returns the number of floats written, or negative.                                                       */
long long prisma_depth_read_tap(prisma_engine* e, const char* name, float* out, long long capacity);
/* Per-kernel-group CUDA-event timings of one pass over n frames (ms), for bench.py's roofline block:
 * out[0]=pre, out[1]=encoder linear GEMMs, out[2]=attention, out[3]=layernorm, out[4]=head convs,
 * out[5]=resamplers, out[6]=post, out[7]=total.                                                             */
int prisma_depth_profile(prisma_engine* e, int h, int w, int n, float* out8);
/* Algorithmic work of one pass over n frames at (h,w): out[0]=encoder-linear FLOP, out[1]=attention FLOP,
 * out[2]=head FLOP, out[3]=kernel launches per pass.                                                       */
int prisma_depth_work(prisma_engine* e, int h, int w, int n, double* out4);

int prisma_engine_destroy(prisma_engine* e);

/* ---- RAFT band, HBM-bound stages (replaces parts of bands/flow_raft.py + bands/raft/corr.py; the conv encoders and
 *      the ConvGRU update block are the next rows of SURVEY.md section 8)                                        */
/* K11: cv2.resize(frame, fx=fy=scale, INTER_CUBIC) + load_image + InputPadder('sintel').pad + 2*(x/255)-1
 * (flow_raft.py:100-101, common/flow.py:13-16,46-56, raft/raft.py:90-91).  rgb u8 h*w*3 -> resized u8 hs*ws*3
 * (may be NULL) and chw_padded f32 [3][hp][wp]; hs = cvRound(h*scale) (half to even, as cv::resize derives dsize from fx),
 * hp/wp = hs/ws rounded up to a multiple of 8.  `scale` is a double on purpose: the sampling step is 1/fx on both axes and
 * host and engine must agree on cvRound(h*scale) (argparse hands the band a Python float = double).                        */
int prisma_flow_preprocess(int device, const uint8_t* rgb, int h, int w, double scale, uint8_t* resized,
                           float* chw_padded);
/* K20: process_flow (common/encode.py:113-126): flow f32 h*w*2 -> rgb u8 h*w*3 + max displacement.            */
int prisma_flow_encode(int device, const float* flow, int h, int w, uint8_t* rgb_out, float* max_disp_out);
/* compute_fwdbwd_mask (common/flow.py:28-40, incl. warp_flow = cv2.remap bilinear :19-26) and encode_flow
 * (common/encode.py:105-110): fwd / bwd f32 h*w*2 -> masks u8 h*w (0/1) and, optionally, the 16-bit PNG payload
 * u16 h*w*3 written by --subpath_mask.                                                                          */
int prisma_flow_masks(int device, const float* fwd, const float* bwd, int h, int w, uint8_t* fwd_mask, uint8_t* bwd_mask,
                      uint16_t* fwd_u16, uint16_t* bwd_u16);
/* K13-K15: CorrBlock (raft/corr.py:12-60) for `batch` image pairs at 1/8 resolution, 256 channels.             */
int prisma_flowcorr_create(int device, int batch, int h8, int w8, prisma_engine** out);
/* fmap1/fmap2: host f32 [batch][256][h8][w8] (NCHW, as BasicEncoder returns them)                              */
int prisma_flowcorr_set_fmaps(prisma_engine* e, const float* fmap1, const float* fmap2);
/* builds the 4-level fp32 correlation pyramid; ms_out = CUDA-event time per build over `iters` builds          */
int prisma_flowcorr_build(prisma_engine* e, int iters, float* ms_out);
/* CorrBlock.__call__: coords host f32 [batch][2][h8][w8] -> out f32 [batch][324][h8][w8] (may be NULL)          */
int prisma_flowcorr_lookup(prisma_engine* e, const float* coords, float* out, int iters, float* ms_out);
/* rows [row0,row0+nrows) of pyramid level `level` of image `b`: out f32 [nrows][(h8>>level)*(w8>>level)]        */
int prisma_flowcorr_read_level(prisma_engine* e, int level, int b, int row0, int nrows, float* out);
/* algorithmic work of one build: out[0] = FLOP, out[1] = bytes (fp32 pyramid written + fp16 features read)      */
int prisma_flowcorr_work(prisma_engine* e, double* out2);

/* ---- RAFT band, whole model: replaces init_model (bands/flow_raft.py:38-48) + infer (:51-66) + the resize of
 *      process_video (:100-101) + process_flow (common/encode.py:113-126) for one frame pair, forward and backward   */
int prisma_flow_create(int device, prisma_engine** out);
/* one call per tensor of the RAFT state_dict (bands/raft/raft.py:24-57; a leading "module." is stripped)           */
int prisma_flow_load_tensor(prisma_engine* e, const char* name, const float* data, const int64_t* shape, int ndim);
int prisma_flow_finalize(prisma_engine* e);
/* prev / curr: h*w*3 u8 RGB frames.  scale = args.scale (0.75), iters = args.iterations.  Outputs (each may be NULL):
 * fwd / bwd: hs*ws*2 f32 flows (hs = round(h*scale)), fwd_rgb / bwd_rgb: hs*ws*3 u8 HSV encodings, max_*: the
 * per-frame max displacement written to <band>.csv.  ms_out: device time of the pass (CUDA events), may be NULL.    */
int prisma_flow_infer(prisma_engine* e, const uint8_t* prev, const uint8_t* curr, int h, int w, double scale, int iters,
                      float* fwd, float* bwd, uint8_t* fwd_rgb, uint8_t* bwd_rgb, float* max_fwd, float* max_bwd,
                      float* ms_out);
/* The loop body of process_video in a video loop (bands/flow_raft.py:97-115): with reuse_prev != 0, `prev` is the `curr` of the
 * previous call -- the engine keeps that frame's fnet / cnet features, so only `curr` is uploaded and encoded (each frame is
 * encoded once per clip instead of twice; results are identical).  prev may be NULL then.  Falls back to the full pass when
 * no valid cache exists (first call, or after a change of resolution / scale / iterations).                              */
int prisma_flow_infer_video(prisma_engine* e, const uint8_t* prev, const uint8_t* curr, int h, int w, double scale, int iters,
                            int reuse_prev, float* fwd, float* bwd, uint8_t* fwd_rgb, uint8_t* bwd_rgb, float* max_fwd,
                            float* max_bwd, float* ms_out);
/* A chunk of process_video's loop (bands/flow_raft.py:97-115): frames = n*h*w*3 u8 RGB, consecutive frames of one clip.
 * continue_clip == 0: a new clip -- pair j = (frame j, frame j+1), n-1 pairs.  continue_clip != 0: the chunk continues the
 * clip of the previous call (the engine still holds the features of the frame before frames[0]) -- pair j = (frame j-1,
 * frame j), n pairs.  Every frame is uploaded and encoded once; the upload of the next frame and the download of the
 * previous pair overlap the compute (three streams, two staging slots; pinned host buffers from prisma_host_alloc make
 * the copies asynchronous DMA).  Outputs are pair-major (fwd / bwd: pairs*hs*ws*2 f32, *_rgb: pairs*hs*ws*3 u8, max_*:
 * pairs floats), each may be NULL; *pairs_out = number of pairs.  Same results as prisma_flow_infer per pair.            */
int prisma_flow_infer_stream(prisma_engine* e, const uint8_t* frames, int n, int h, int w, double scale, int iters,
                             int continue_clip, float* fwd, float* bwd, uint8_t* fwd_rgb, uint8_t* bwd_rgb, float* max_fwd,
                             float* max_bwd, int* pairs_out);
/* Frame pairs per pass of the clip path (prisma_flow_infer_stream / _infer_resident / _work_detail / _profile): 1..4
 * (default 4; PRISMA_RAFT_PAIRS in the environment overrides; lowered per frame size until the correlation pyramids of one
 * pass fit in a third of the device memory -- 4K frames run one pair per pass).  With n, one pass takes n + 1 consecutive frames and
 * produces both directions of the n pairs: every update-block launch covers n times the rows, so the per-launch fixed
 * cost is shared by n pairs.  Results per pair are the same.  The pair calls prisma_flow_infer / _infer_video always use 1.   */
int prisma_flow_set_pairs_per_pass(prisma_engine* e, int pairs);
int prisma_flow_pairs_per_pass(prisma_engine* e);   /* current setting, < 0 on error */
int prisma_flow_plan_pairs(prisma_engine* e);       /* pairs per pass of the plan the last call built, < 0 on error */
/* `reps` passes over the frames already resident on the device (video pass when a previous call left its features,
 * else the full pass), outputs left on the device: ms per PASS (= pairs_per_pass pairs) by CUDA events on the engine
 * stream (bench.py).                                                                                                  */
int prisma_flow_infer_resident(prisma_engine* e, int h, int w, double scale, int iters, int reps, float* ms_per_pass);
/* intermediate tensors of the last pass (tests): "fmap" [2][P][256], "cnet_out" [2P][256], "coords1_iter0",
 * "h_iter0", "coords1"; returns the number of floats written                                                       */
long long prisma_flow_read_tap(prisma_engine* e, const char* name, float* out, long long capacity);
/* out[0] = algorithmic FLOP of one pass, out[1] = kernel launches per pass, out[2] = hs, out[3] = ws               */
int prisma_flow_work(prisma_engine* e, int h, int w, double scale, int iters, double* out4);
/* out[0] / out[1] = algorithmic FLOP of the tcgen05 conv GEMMs of the full / the video pass (encoders, update block, heads;
 * without the correlation build), out[2] / out[3] = FLOP / algorithmic bytes of one correlation-pyramid build (all 2 * pairs_per_pass
 * directions of a pass; bytes = fp32 pyramid written once + fp16 features read once, raft/corr.py:13-27), out[4] / out[5] = kernel
 * steps of the full / video pass, out[6], out[7] = hs, ws                                                              */
int prisma_flow_work_detail(prisma_engine* e, int h, int w, double scale, int iters, double* out8);
/* CUDA-event times (ms) of one pass by kernel group, for bench.py's roofline block (video pass when the previous call left
 * its features): out[0] pre-process, [1] conv GEMMs, [2] correlation build, [3] correlation lookup, [4] InstanceNorm,
 * [5] other pointwise kernels, [6] convex up-sampling + HSV encode, [7] total                                            */
int prisma_flow_profile(prisma_engine* e, int h, int w, double scale, int iters, float* out8);

/* ---- mask_mmdet band: SOLOv2 (bands/mask_mmdet.py; bands/mmdet/apis/inference.py:99-162 inference_detector) ----
 * prisma_mask_create("r101") + load_tensor x N + finalize replace init_detector(CONFIG, MODEL) (mask_mmdet.py:38-41,
 * apis/inference.py:19-61); tensors by the mmdet checkpoint's state_dict names (backbone.*, neck.*, mask_head.*), fp32.
 * prisma_mask_infer replaces inference_detector(model, img) AND the band's union loop (mask_mmdet.py:43-61,134-146):
 *   rgb          h*w*3 u8 RGB frame (the band converts to BGR and the pipeline back, to_rgb=True)
 *   confidence   args.confidence (the band additionally applies its fixed 0.5, getTotalMasks)
 *   union_mask   h*w u8: (255 * number of overlapping instances of the 11 band classes above the thresholds) mod 256
 *   n_inst, scores[100], labels[100]: the kept instances of InstanceData (all 80 classes), sorted by score
 *   inst_masks   optional n_inst*h*w u8 0/1 (results.masks)                                                          */
/* variant: "r101" (the band's SOLOv2 R-101) or "tiny" (test-size twin); a "-fast" suffix selects the single-pass fp16 head.
 * Default = the fp32-class head: every contraction from the FPN levels to the mask predictions runs as three kind::tf32
 * tensor-core passes over [hi | lo] splits of both operands with fp32 activations in between, so that the integer / boolean
 * decode (score_thr, points NMS, mask_thr, Matrix NMS, the final masks) sees the reference's fp32 values to ~1e-6.        */
int prisma_mask_create(const char* variant, int device, prisma_engine** out);
int prisma_mask_load_tensor(prisma_engine* e, const char* name, const float* data, const int64_t* shape, int ndim);
int prisma_mask_finalize(prisma_engine* e);
int prisma_mask_infer(prisma_engine* e, const uint8_t* rgb, int h, int w, float confidence, uint8_t* union_mask, int* n_inst,
                      float* scores, int32_t* labels, uint8_t* inst_masks, float* ms_out);
/* Tests: replay SOLOV2Head.forward + get_results (models/dense_heads/solov2_head.py:253-292,582-766) from GIVEN FPN levels
 * (fp32 NCHW [256][h][w], e.g. the reference's own, tests/golden/solo_tiny_head.npz) for the frame geometry of the last
 * prisma_mask_infer call: inject the five levels, then run head + decode.  img_h / img_w > 0 override the resized-image size
 * (meta img_shape) of the final mask crop.  fp32-class head only.                                                       */
int prisma_mask_inject_feat(prisma_engine* e, int level, const float* nchw, int h, int w);
int prisma_mask_infer_from_feats(prisma_engine* e, int h, int w, int img_h, int img_w, float confidence, uint8_t* union_mask,
                                 int* n_inst, float* scores, int32_t* labels, uint8_t* inst_masks);
/* --sdf (bands/mask_mmdet.py:64-69,150-152): green channel = 255 * (1 - clip(((sdf + 127)/255 - 0.25) * 2, 0, 1)) with sdf the
 * exact Euclidean signed distance of the union mask (what snowy.generate_sdf computes); union_mask / green_out: h*w u8    */
int prisma_mask_sdf(int device, const uint8_t* union_mask, int h, int w, uint8_t* green_out);
/* intermediate tensors of the last pass (tests): "resized", "net_input", "fpn0..4", "mask_feats", "cls0..4", "kernel0..4",
 * "cand_count", "n_top"; returns the number of floats written                                                        */
long long prisma_mask_read_tap(prisma_engine* e, const char* name, float* out, long long capacity);
/* out[0] = algorithmic FLOP of the last planned pass, out[1] = launches, out[2..5] = resized h, w, padded h, w        */
int prisma_mask_work(prisma_engine* e, int h, int w, double* out8);

/* Size of the resized (un-padded) network input each band's transform produces for a w x h frame: depth_anything
 * (d_anything/util/transform.py:111-166 lower_bound x14), depth_midas (upper_bound x32: fits 384 x 384), depth_anything_metric (392 x 518),
 * mask_mmdet (mmcv.imrescale (1333, 800)).  Pure host arithmetic, usable without a GPU.                              */
int prisma_net_size(const char* band, int w, int h, int* wn, int* hn);

/* ---- kernel-level entry points (parity tests and micro-benchmarks call the kernels through the C ABI) ---- */
/* D = A[M,K] * W[N,K]^T (+bias) with fp16 operands / fp32 accumulate on the tcgen05 core; A, W, D host fp32.
 * act: 0 none, 1 gelu, 2 relu; -4 = the TMA-store epilogue (no bias, accumulator scaled by 1/16: the RAFT correlation path).
 * force_bn: 0 = auto, else 32/64/128/256, 512 = CTA pairs.  ms_out (may be NULL): kernel time.                               */
int prisma_debug_gemm(int device, const float* A, const float* W, const float* bias, float* D, int M, int N, int K,
                      int act, int force_bn, int iters, float* ms_out);
/* The same product through the 3xTF32 path of the mask band (kind::tf32 tensor-core MMAs on [hi | lo] splits of both
 * operands: fp32-class products, ~1e-6 relative): D = A W^T + bias, all fp32.  force_bn: 0 = auto, else 32/64/128.    */
int prisma_debug_gemm_tf32x3(int device, const float* A, const float* W, const float* bias, float* D, int M, int N, int K,
                             int force_bn, int iters, float* ms_out);
/* 3x3 (kh x kw) stride-1 'same' convolution, NHWC fp32 host in/out, through the shifted-row GEMM.           */
int prisma_debug_conv(int device, const float* x_nhwc, const float* w_oihw, const float* bias, float* y_nhwc, int H,
                      int W, int Cin, int Cout, int kh, int kw, int relu, float* ms_out);
/* softmax(q k^T) v per head (head_dim 64); qkv host fp32 [T][3*D] (q NOT pre-scaled; scaled inside), out [T][D] */
int prisma_debug_attention(int device, const float* qkv, float* out, int T, int heads, int iters, float* ms_out);
int prisma_debug_layernorm(int device, const float* x, const float* g, const float* b, float* y, int rows, int D);
/* OpenCV-exact cubic resize + normalise (K1): rgb u8 h*w*3 -> f32 [3][hn][wn]                                */
int prisma_debug_da_preprocess(int device, const uint8_t* rgb, int h, int w, float* out, int hn, int wn);

#ifdef __cplusplus
}
#endif
#endif /* PRISMA_B200_H */
