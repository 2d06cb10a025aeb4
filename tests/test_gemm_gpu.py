"""GPU: the tcgen05 shifted-row GEMM core through the C ABI vs a plain fp32 reference on fp16-rounded operands."""
import ctypes as C

import numpy as np
import pytest
import torch

from prisma_b200._lib import PrismaError, check, fptr, lib

pytestmark = pytest.mark.gpu


def _h(a):  # fp16 operand rounding (the kernels' operand type); accumulation is fp32
    return a.astype(np.float16).astype(np.float32)


def _gemm(A, W, bias, act, bn):
    M, K = A.shape
    N = W.shape[0]
    D = np.empty((M, N), np.float32)
    ms = C.c_float()
    check(lib().prisma_debug_gemm(0, fptr(A), fptr(W), fptr(bias) if bias is not None else None, fptr(D), M, N, K, act, bn, 1, C.byref(ms)))
    return D


@pytest.mark.parametrize("M,N,K,act,bn", [
    (128, 128, 64, 0, 128),      # one tile, one k-block
    (256, 256, 256, 0, 128),     # accumulate over k-blocks, several tiles
    (300, 384, 200, 0, 0),       # ragged M, K tail (zero-filled by TMA), auto tile
    (2443, 1152, 384, 0, 0),     # ViT-S qkv
    (2443, 1024, 1024, 2, 256),  # BN=256, relu
    (1813, 1536, 384, 1, 64),    # BN=64, gelu
    (500, 48, 384, 0, 0),        # narrow N (ViT-S head), BN=32/64
    (333, 32, 1152, 2, 32),      # BN=32
    (40000, 256, 128, 0, 0),     # many tiles per CTA (persistent loop, TMEM double buffering)
    (64, 64, 64, 0, 0),          # smaller than a tile
    (512, 256, 128, 0, 512),     # CTA pairs (cta_group::2, 256x256 tiles): one pair tile per pair
    (2443, 3072, 1024, 0, 512),  # CTA pairs, ViT-L qkv: ragged M, many tiles per pair
    (9772, 1024, 4096, 1, 512),  # CTA pairs, 4-frame fc2 shape with gelu
    (300, 256, 200, 2, 512),     # CTA pairs: second CTA's rows partly / fully out of range, K tail
    # auto tile choice with a partial last wave -> mixed-width tail tiles (GemmArgs::tail_split)
    (29316, 1024, 192, 0, 0),    # CTA pairs: 460 pair tiles = 6 waves + 16 -> the 16 cut into 4 x 64-wide tiles
    (26624, 256, 128, 2, 0),     # CTA pairs: 104 pair tiles = 1 wave + 30 -> cut into 2 x 128-wide tiles
    (39008, 128, 384, 1, 0),     # single CTAs, 128-wide: 305 tiles = 2 waves + 9 -> 2 x 64-wide tiles, gelu
    (20000, 64, 128, 0, 0),      # 64-wide: 157 tiles = 1 wave + 9 -> 2 x 32-wide tiles
    # transposed tiles (GemmCfg SWAP, force 640): 128 output columns x 256 rows per instruction, epilogue transposed
    (256, 128, 64, 0, 640),      # one tile, one k-block
    (37000, 128, 1920, 0, 640),  # the RAFT GRU q conv shape: ragged M (the last tile has 136 valid rows), many tiles per CTA
    (5000, 96, 576, 2, 640),     # N = 96 (RAFT encoder layer 2): the fourth column quarter is beyond N; relu
    (777, 128, 200, 1, 640),     # K tail, gelu, M not a multiple of 32
    (151552, 128, 256, 0, 0),    # auto choice picks the transposed tiles (N <= 128, M >= 4096): 8 whole waves
    (4100, 68, 128, 0, 640),     # N % 32 = 4: one 4-column group of the third quarter valid
])
def test_gemm_matches_fp32_reference(M, N, K, act, bn):
    rng = np.random.default_rng(M * 7 + N * 3 + K)
    A = rng.standard_normal((M, K), dtype=np.float32)
    W = (rng.standard_normal((N, K), dtype=np.float32) / np.sqrt(K)).astype(np.float32)
    bias = rng.standard_normal(N, dtype=np.float32)
    got = _gemm(A, W, bias, act, bn)
    ref = torch.from_numpy(_h(A)) @ torch.from_numpy(_h(W)).T + torch.from_numpy(bias)
    if act == 1:
        ref = torch.nn.functional.gelu(ref)
    elif act == 2:
        ref = torch.relu(ref)
    ref = ref.numpy()
    err = np.abs(got - ref).max()
    assert err <= 2e-4 * max(1.0, np.abs(ref).max()), f"max abs err {err}"


@pytest.mark.parametrize("M,N,K,bn", [
    (18360, 18360, 256, 0),   # RAFT correlation level 0 at 1080p x 0.75: CTA pairs, ragged M and N (N % 32 = 24)
    (18360, 4592, 512, 0),    # coarse-level size class with a longer K, N % 32 = 16
    (1000, 264, 256, 128),    # level 3 size class, single CTAs, 128-wide tiles
    (300, 520, 64, 256),      # single CTAs, 256-wide, rows of the last tile out of range
])
def test_gemm_tma_store_epilogue(M, N, K, bn):
    """The TMA-store epilogue (tcgen05.ld -> swizzled smem box -> cp.async.bulk.tensor store): dense fp32 output scaled by
    1/16, boxes clipped at ragged M / N edges, nothing written outside [M][N]."""
    rng = np.random.default_rng(M + N + K)
    A = rng.standard_normal((M, K), dtype=np.float32)
    W = rng.standard_normal((N, K), dtype=np.float32)
    got = _gemm(A, W, None, -4, bn)
    rows = np.unique(np.concatenate([np.arange(0, min(M, 300)), np.arange(max(0, M - 300), M), rng.integers(0, M, 200)]))
    ref = (torch.from_numpy(_h(A[rows])) @ torch.from_numpy(_h(W)).T).numpy() * 0.0625
    err = np.abs(got[rows] - ref).max()
    assert err <= 2e-4 * max(1.0, np.abs(ref).max()), f"max abs err {err}"
    assert np.isfinite(got).all()


@pytest.mark.parametrize("M,N,K,bn", [
    (18360, 18360, 256, 0),   # RAFT correlation level 0 at 1080p x 0.75: CTA pairs, ragged M and N (N % 32 = 24)
    (18360, 4592, 512, 0),    # coarse-level size class with a longer K, N % 32 = 16
    (1000, 264, 256, 128),    # level 3 size class, single CTAs, 128-wide tiles
    (300, 520, 64, 256),      # single CTAs, 256-wide, rows of the last tile out of range
])
def test_gemm_tma_store_epilogue_fp16(M, N, K, bn):
    """The same epilogue with an fp16 destination (32 x 64-byte boxes, 64-byte swizzle): fp32 accumulate, scaled by 1/16,
    rounded once; every element of [M][N] written (the buffer starts as NaN), boxes clipped at the ragged edges."""
    rng = np.random.default_rng(M + N + K + 1)
    A = rng.standard_normal((M, K), dtype=np.float32)
    W = rng.standard_normal((N, K), dtype=np.float32)
    got = _gemm(A, W, None, -5, bn)
    assert np.isfinite(got).all()
    rows = np.unique(np.concatenate([np.arange(0, min(M, 300)), np.arange(max(0, M - 300), M), rng.integers(0, M, 200)]))
    ref = (torch.from_numpy(_h(A[rows])) @ torch.from_numpy(_h(W)).T).numpy() * 0.0625
    err = np.abs(got[rows] - ref).max()
    assert err <= 6e-4 * max(1.0, np.abs(ref).max()), f"max abs err {err}"   # one fp16 rounding: 2^-11 relative


@pytest.mark.parametrize("M,N,K,act,bn", [
    (29316, 4096, 1024, -6, 0),   # ViT-L fc1 at 12 frames: CTA pairs, ragged M, tail tiles, bias + GELU
    (2443, 3072, 1024, -7, 0),    # qkv-like, bias + ReLU
    (700, 328, 200, -6, 128),     # single CTAs, N % 64 = 8: the last 64-column box is clipped to 8 columns, K tail
])
def test_gemm_tma_store_epilogue_fp16_bias_activation(M, N, K, act, bn):
    """The fp16 TMA-store epilogue of the ViT qkv / fc1 linears: bias and GELU / ReLU applied in the row-per-lane registers,
    then 32 x 64-column bulk stores; every element of [M][N] written, boxes clipped at the ragged edges."""
    rng = np.random.default_rng(M + N + K + 2)
    A = rng.standard_normal((M, K), dtype=np.float32)
    W = (rng.standard_normal((N, K), dtype=np.float32) / np.sqrt(K)).astype(np.float32)
    bias = rng.standard_normal(N, dtype=np.float32)
    got = _gemm(A, W, bias, act, bn)
    assert np.isfinite(got).all()
    rows = np.unique(np.concatenate([np.arange(0, min(M, 300)), np.arange(max(0, M - 300), M), rng.integers(0, M, 200)]))
    ref = torch.from_numpy(_h(A[rows])) @ torch.from_numpy(_h(W)).T + torch.from_numpy(bias)
    ref = (torch.nn.functional.gelu(ref) if act == -6 else torch.relu(ref)).numpy()
    err = np.abs(got[rows] - ref).max()
    assert err <= 6e-4 * max(1.0, np.abs(ref).max()), f"max abs err {err}"   # one fp16 rounding: 2^-11 relative


@pytest.mark.parametrize("M,N,K,bn", [
    (29316, 1024, 4096, 0),   # ViT-L fc2 at 12 frames: CTA pairs, ragged M
    (2443, 384, 384, 0),      # ViT-S proj: single CTAs, 128-wide tiles
    (300, 264, 200, 128),     # ragged N (N % 32 = 8), K tail
])
def test_gemm_tma_reduce_epilogue_in_place_residual(M, N, K, bn):
    """x += acc + bias through cp.reduce.async.bulk.tensor .add.f32 (the ViT proj / fc2 epilogue): the debug entry starts from
    zeros and launches twice (warm-up + 1), so D = 2 (A W^T + bias) exactly in fp32; nothing outside [M][N] is touched."""
    rng = np.random.default_rng(M + N + K + 3)
    A = rng.standard_normal((M, K), dtype=np.float32)
    W = (rng.standard_normal((N, K), dtype=np.float32) / np.sqrt(K)).astype(np.float32)
    bias = rng.standard_normal(N, dtype=np.float32)
    got = _gemm(A, W, bias, -8, bn) * 0.5
    assert np.isfinite(got).all()
    rows = np.unique(np.concatenate([np.arange(0, min(M, 300)), np.arange(max(0, M - 300), M), rng.integers(0, M, 200)]))
    ref = (torch.from_numpy(_h(A[rows])) @ torch.from_numpy(_h(W)).T + torch.from_numpy(bias)).numpy()
    err = np.abs(got[rows] - ref).max()
    assert err <= 2e-4 * max(1.0, np.abs(ref).max()), f"max abs err {err}"


@pytest.mark.parametrize("H,W,Cin,Cout,k,relu", [
    (37, 66, 64, 64, 3, 1),
    (19, 33, 384, 64, 3, 0),
    (40, 50, 48, 64, 3, 0),      # Cin < 64: TMA box wider than the tensor
    (24, 31, 128, 32, 1, 0),
    (30, 44, 64, 128, 5, 0),
])
def test_conv_matches_torch(H, W, Cin, Cout, k, relu):
    rng = np.random.default_rng(H * W + Cin)
    x = rng.standard_normal((H, W, Cin), dtype=np.float32)
    w = (rng.standard_normal((Cout, Cin, k, k), dtype=np.float32) / np.sqrt(Cin * k * k)).astype(np.float32)
    b = rng.standard_normal(Cout, dtype=np.float32)
    y = np.empty((H, W, Cout), np.float32)
    ms = C.c_float()
    check(lib().prisma_debug_conv(0, fptr(x), fptr(w), fptr(b), fptr(y), H, W, Cin, Cout, k, k, relu, C.byref(ms)))
    xt = torch.from_numpy(_h(x)).permute(2, 0, 1)[None]
    ref = torch.nn.functional.conv2d(xt, torch.from_numpy(_h(w)), torch.from_numpy(b), padding=k // 2)
    if relu:
        ref = torch.relu(ref)
    ref = ref[0].permute(1, 2, 0).numpy()
    err = np.abs(y - ref).max()
    assert err <= 2e-4 * max(1.0, np.abs(ref).max()), f"max abs err {err}"


@pytest.mark.parametrize("M,N,K,bn", [(300, 256, 512, 0), (4096, 512, 2304, 0), (1600, 80, 4608, 0), (5000, 128, 320, 128), (64, 32, 100, 32)])
def test_gemm_tf32x3_is_fp32_class(M, N, K, bn):
    """The 3xTF32 path (kind::tf32 MMAs on [hi | lo] splits of both operands) against the exact product (float64).  The
    products are fp32-class (the dropped lo x lo term is 2^-22).  The tensor core's own fp32 ACCUMULATION truncates the aligned
    addends instead of rounding them -- with the whole K in one TMEM chain that bias measured 3e-6 .. 6e-6 of sum |a||w| on
    B200 (growing with K), i.e. only 1e-4-class results for K ~ 4600.  The kernel therefore keeps a TMEM chain 4 K-blocks
    (16 MMAs) long and adds the partial sums in registers with round-to-nearest FADDs (GEMM_TF32_ACC_GROUP): the error is
    then that of a CUDA-core fp32 GEMM."""
    rng = np.random.default_rng(M + N + K)
    A = (rng.standard_normal((M, K), dtype=np.float32) * rng.uniform(0.01, 30.0, (M, 1)).astype(np.float32))
    W = (rng.standard_normal((N, K), dtype=np.float32) / np.sqrt(K)).astype(np.float32)
    bias = rng.standard_normal(N, dtype=np.float32)
    D = np.empty((M, N), np.float32)
    ms = C.c_float()
    check(lib().prisma_debug_gemm_tf32x3(0, fptr(A), fptr(W), fptr(bias), fptr(D), M, N, K, bn, 1, C.byref(ms)))
    ref = A.astype(np.float64) @ W.astype(np.float64).T + bias
    scale = np.abs(A).astype(np.float64) @ np.abs(W).astype(np.float64).T + np.abs(bias)
    err = float((np.abs(D - ref) / scale).max())
    print(f"tf32x3 {M}x{N}x{K}: max |err| / sum|a||w| = {err:.2e}, {ms.value * 1e3:.1f} us")
    assert err <= 6e-7, err


def test_gemm_rejects_tile_widths_without_a_kernel():
    """A requested tile width no kernel is built for is an error, never a silent substitute: 256 x 128 CTA-pair tiles
    (force 384) on the fp16 path, and 3xTF32 tiles wider than the 128 columns its register-held running sums allow."""
    A = np.ones((256, 64), np.float32)
    W = np.ones((256, 64), np.float32)
    D = np.empty((256, 256), np.float32)
    with pytest.raises(PrismaError, match="BLOCK_N"):
        check(lib().prisma_debug_gemm(0, fptr(A), fptr(W), None, fptr(D), 256, 256, 64, 0, 384, 1, None))
    with pytest.raises(PrismaError, match="BLOCK_N"):
        check(lib().prisma_debug_gemm_tf32x3(0, fptr(A), fptr(W), None, fptr(D), 256, 256, 64, 256, 1, None))
