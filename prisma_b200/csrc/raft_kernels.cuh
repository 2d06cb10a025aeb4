// prisma_b200 -- RAFT band pointwise / gather kernels (see raft_kernels.cu).
#pragma once
#include "common.cuh"

namespace prisma {

int raft_im2col_stem(const float* x, int B, int H, int W, __half* out, cudaStream_t s);
int instnorm_stats(const float* x, int B, int HW, int C, float* part, float* stats, cudaStream_t s);
int instnorm_partial_floats(int B, int HW, int C);
constexpr int INSTNORM_STAGE1_BLOCKS = 72;
// statistics from the per-slab partials written by the conv epilogue (GemmEpilogue::stat_part); part2: B * 72 * C * 2 doubles
int instnorm_stats_from_slabs(const float* slab_part, int B, int slabs_per_image, int C, int HW, double* part2, float* stats,
                              cudaStream_t s);
int instnorm_apply(const float* x, const float* stats, int B, int H, int W, int C, const __half* skip_map,
                   const float* skip_raw, const float* skip_stats, __half* out, int pad, long long img_rows, cudaStream_t s);
struct DirFrames { int f[8]; };  // frame whose context features direction b uses
int raft_cnet_split(const float* cn, int B, int H, int W, int pad, long long img_rows, DirFrames df, float* h_master, __half* hx,
                    __half* rhx, cudaStream_t s);
int raft_flow_im2col(const float* c0, const float* c1, int B, int H, int W, __half* out, cudaStream_t s);
int raft_flow_cols(const float* c0, const float* c1, int B, int H, int W, int pad, long long img_rows, __half* hx, __half* rhx,
                   cudaStream_t s);
int raft_coords_update(const float* delta, int B, int H, int W, int pad, long long img_rows, float* coords1, cudaStream_t s);
// FlowHead.conv2 as 1x1 GEMM partial products u [rows][32] (column tap*2 + out) + this nine-tap gather; coords1 += delta
int raft_flow_head2_gather(const float* u, int B, int H, int W, int pad, long long img_rows, float b0, float b1, float* coords1,
                           cudaStream_t s);
int raft_coords_init(float* c0, float* c1, int B, int H, int W, cudaStream_t s);
int raft_convex_upsample(const float* mask, const float* c0, const float* c1, int B, int H, int W, int pad, long long img_rows,
                         int Hs, int Ws, int pad_top, int pad_left, float* out, cudaStream_t s);

}  // namespace prisma
