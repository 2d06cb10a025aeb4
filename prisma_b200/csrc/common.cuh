// prisma_b200 -- common device/host helpers for sm_100a (B200).
// Hand-written PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA/TMEM).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <string>

namespace prisma {

// ----------------------------------------------------------------------------------------------
// host-side error plumbing: nothing throws across the C ABI; errors become codes + thread-local text
// ----------------------------------------------------------------------------------------------
void set_last_error(const std::string& msg);

#define PRISMA_CUDA_OK(expr)                                                                     \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      ::prisma::set_last_error(std::string(#expr) + " failed: " + cudaGetErrorString(_e) +       \
                               " (" __FILE__ ":" + std::to_string(__LINE__) + ")");              \
      return -2;                                                                                 \
    }                                                                                            \
  } while (0)

#define PRISMA_CHECK(cond, msg)                                                                  \
  do {                                                                                           \
    if (!(cond)) {                                                                               \
      ::prisma::set_last_error(std::string(msg) + " [" #cond "] (" __FILE__ ":" +                \
                               std::to_string(__LINE__) + ")");                                  \
      return -1;                                                                                 \
    }                                                                                            \
  } while (0)

#define PRISMA_TRY(expr)                                                                         \
  do {                                                                                           \
    int _r = (expr);                                                                             \
    if (_r != 0) return _r;                                                                      \
  } while (0)

// NVTX ranges (header-only nvtx3: a no-op unless a profiler injects its library) around every engine pass and, in the
// un-graphed direct runs, around every named step -- so an Nsight Systems / ncu --nvtx timeline reads in the reference's
// vocabulary (SURVEY.md section 5: the reference has no tracing hooks at all).
struct NvtxRange {
  explicit NvtxRange(const char* name);
  ~NvtxRange();
};

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static inline int round_up(int a, int b) { return ceil_div(a, b) * b; }

#ifdef __CUDACC__
// ----------------------------------------------------------------------------------------------
// device helpers
// ----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug becomes a trap (-> CUDA error on the host), never a hung GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {  // ~2 s
      printf("prisma: mbarrier timeout block=(%d,%d) thread=%d bar=%p parity=%u\n", blockIdx.x, blockIdx.y,
             threadIdx.x, (void*)bar, parity);
      __trap();
    }
  }
}

__device__ __forceinline__ float fmax3(float a, float b, float c) {  // FMNMX3 (sm_100)
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// ---- TMA ----------------------------------------------------------------------------------------
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}

// TMA store: a swizzled shared-memory box -> global (bulk async group of the issuing thread); out-of-range rows / columns
// of the box are clipped by the tensor map
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {  // at most N groups of this thread still READING shared memory
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- CTA pairs (cta_group::2): cluster rank / sync, TMA and commits that target the pair ------------------------
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;  // clears the CTA-rank bit of a shared::cluster address -> CTA 0 of the pair
// TMA load issued by either CTA of a pair; the transaction bytes are accounted on the LEADER CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
      : "memory");
}
// arrive on the leader CTA's copy of a barrier (used by both CTAs' epilogue warps)
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {  // one full warp in EACH CTA
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A * B over the CTA pair: M = 256 (128 rows per CTA), B tile split across the two CTAs
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit -> arrive(1) on the barrier at this smem offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"((uint16_t)3)
               : "memory");
}

// ---- tcgen05 / TMEM -----------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // same warp as alloc
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc], fp16/bf16 inputs, fp32 accumulate; one thread issues.
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::tf32: fp32 containers in shared memory (the tensor core uses sign, 8 exponent and the top 10 mantissa bits), fp32
// accumulate; K = 8 per instruction (32 bytes of a 128-byte swizzled row, like K = 16 of fp16)
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// same with the A operand read from TMEM (lanes = rows, 32-bit columns = fp16 pairs along K) instead of shared memory
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// commit all previously issued tcgen05.mma of this thread -> arrive(1) on an mbarrier when they retire
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// Shared-memory matrix descriptor, 128B-swizzled tiles whose rows are 128 bytes (64 fp16):
//   K-major  : rows = M/N index, 8-row groups 1024 B apart (SBO); K advances inside the 128 B row.
//   MN-major : rows = K index, 128 B = 64 MN elements; 8-row K groups 1024 B apart (SBO).
// Fields (cute/arch/mma_sm100_desc.hpp SmemDescriptor): addr>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout_type [61,64) (2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t make_sdesc_sw128(uint32_t smem_addr, uint32_t sbo_bytes = 1024,
                                                     uint32_t lbo_bytes = 16) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor, kind::f16: D=f32 (c_format=1 @4), A/B = f16 (0) or bf16 (1) @7/@10,
// a_major @15, b_major @16 (0 = K-major, 1 = MN-major), N>>3 @17, M>>4 @24.
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N, int a_mn_major = 0, int b_mn_major = 0) {
  return (1u << 4) | (0u << 7) | (0u << 10) | (static_cast<uint32_t>(a_mn_major) << 15) |
         (static_cast<uint32_t>(b_mn_major) << 16) | (static_cast<uint32_t>(N >> 3) << 17) |
         (static_cast<uint32_t>(M >> 4) << 24);
}

// kind::tf32 instruction descriptor: a_format = b_format = 2 (TF32), D = f32
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (static_cast<uint32_t>(N >> 3) << 17) | (static_cast<uint32_t>(M >> 4) << 24);
}

// TMEM -> registers: this warp's 32 lanes (lane = accumulator row), 32 consecutive fp32 columns.
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM: this warp's 32 lanes, 32 consecutive fp32 columns
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- misc math ------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}
#endif  // __CUDACC__

// ----------------------------------------------------------------------------------------------
// host: TMA descriptor encode through the runtime's driver entry point (no -lcuda link dependency)
// ----------------------------------------------------------------------------------------------
// 2-D fp16 tensor [rows][cols] with row pitch `pitch_elems`; box = box_cols x box_rows, 128B swizzle
// (box_cols must be 64 -> 128-byte inner box).  Out-of-bounds elements (either sign) read as zero.
int make_tmap_2d_f16(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t pitch_elems,
                     uint32_t box_cols, uint32_t box_rows);
// the same for an fp32 tensor (box_cols must be 32 -> 128-byte inner box): the destination of the TMA-store epilogue
int make_tmap_2d_f32(CUtensorMap* out, const void* base, uint64_t cols, uint64_t rows, uint64_t pitch_elems,
                     uint32_t box_cols, uint32_t box_rows);

}  // namespace prisma
