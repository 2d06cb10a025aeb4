// prisma_b200 -- RAFT band, HBM-bound part: pre-process (K11), all-pairs correlation pyramid (K13+K14, on the tcgen05
// GEMM core), correlation lookup (K15) and HSV flow encode (K20).  See flow.cu.
#pragma once
#include <vector>

#include "gemm_tc.cuh"

namespace prisma {

int raft_preprocess(const uint8_t* img, int H, int W, int h, int w, double fx, const int pad[4], uint8_t* resized, float* chw,
                    cudaStream_t s);
int flow_encode(const float* flow, int H, int W, uint8_t* rgb, uint32_t* mm_scratch, float* max_out, int num_sms,
                cudaStream_t s);

int flow_consistency_masks(const float* fwd, const float* bwd, int H, int W, uint8_t* fwd_mask, uint8_t* bwd_mask,
                           int num_sms, cudaStream_t s);
int flow_encode_u16(const float* flow, const uint8_t* mask, int H, int W, uint16_t* out, int num_sms, cudaStream_t s);

// All-pairs correlation pyramid + lookup for `batch` image pairs at 1/8 resolution (h8 x w8, C = 256 channels).
struct PoolGeom { int lh[4], lw[4], ln[4], coff[4]; };

class FlowCorr {
 public:
  ~FlowCorr();
  // batch = number of (image1, image2) directions.  Features are stored per FRAME: direction b correlates frame f1_idx[b]
  // against frame f2_idx[b] (the engine: consecutive frames of a clip, each used by up to four directions; default / tests:
  // 2 * batch frames, direction b = frame b against frame batch + b, which is what set_fmaps fills).
  int init(int device, int batch, int h8, int w8, int n_frames = 0, const int* f1_idx = nullptr, const int* f2_idx = nullptr);
  int set_fmaps(const float* fmap1_nchw, const float* fmap2_nchw);  // host fp32 [B][256][h8][w8]
  int build(cudaStream_t s);                                        // K13 + K14
  int lookup(const float* d_coords, cudaStream_t s);                // K15: coords device fp32 [B][2][h8][w8]
  int lookup_to(const float* d_coords, __half* dst, int dst_ld, int dst_wp, int dst_pad, int dst_img_rows,
                cudaStream_t s);                                    // same, into a zero-bordered fp16 map
  int set_fmaps_device(const __half* f1, const __half* f2, cudaStream_t s);  // device fp16 [B][P][C] (engine path)
  int lookup_host(const float* coords, float* out_nchw, int iters, float* ms);
  int time_build(int iters, float* ms);
  int read_level(int level, int b, int row0, int nrows, float* out);

  int device = 0, B = 0, H8 = 0, W8 = 0, P = 0, C = 256, num_sms = 148;
  int lh[4], lw[4], ln[4], lpitch[4];  // level sizes, element counts, row pitch (multiple of 4) of the fp32 volumes
  int NF = 0;                          // frames held
  int f1[8] = {0}, f2[8] = {0};        // frame of image1 / image2 per direction
  __half* feat = nullptr;              // [NF][rows_pad][C] fp16 features (rows padded to the next multiple of 256)
  // levels 1..3 of a frame: rows [coff[l], coff[l] + ln[l]) of pool123 [NF][rows123_pad][C] = the 2^l x 2^l mean (fp16);
  // pool[l] / vol[l] point at level l inside the shared buffers (rows123_pad * C per frame / pitch123 per position)
  __half* pool123 = nullptr;
  float* vol123 = nullptr;
  int coff[4] = {0, 0, 0, 0}, n123 = 0, pitch123 = 0, rows123_pad = 0;
  __half* pool[4] = {nullptr, nullptr, nullptr, nullptr};
  int pool_frames(int first, int count, cudaStream_t s);   // K14 operands of frames [first, first + count)
  int build_gemms(cudaStream_t s);                          // the 2 * B correlation GEMMs (level 0; levels 1..3)
  float* vol[4] = {nullptr, nullptr, nullptr, nullptr};     // per level fp32 [B*P][lpitch] (levels 1..3: columns of vol123)
  float* coords = nullptr;
  __half* lookup_out = nullptr;  // [B*P][384] fp16 (324 used), the A operand of the motion encoder's convc1
  int rows_pad = 0, lrows_pad[4];
  std::vector<GemmLaunch> gemms;
  std::vector<void*> allocs;
  cudaStream_t stream = nullptr;
  double bytes_build = 0, flops_build = 0;
};

}  // namespace prisma
