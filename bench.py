"""bench.py -- the BASELINE metric: frames/sec at 1080p with depth_anything (ViT-L) AND flow_raft (12 GRU iterations,
forward + backward flow) computed for every frame of a synthetic clip, at N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one chunk of FRAMES_PER_STEP consecutive 1080p frames per GPU pushed through both bands, the way
process.py runs them over a clip (reference process.py:225-256,290: the depth band, then the flow band, over the same
frames): depth_anything in passes of BATCH frames, then flow_raft pair by pair (video pass: every frame is encoded
once).  Frames shard across ranks with no data-path collective (SURVEY.md section 8e) -> weak scaling; NCCL carries only
the barrier and the max-over-ranks of the timings.

  value      : frames/s with the chunk resident in HBM: CUDA events on each engine's stream around its passes, summed
               (the two bands run back to back), max over ranks
  e2e        : frames/s through the public Python API (DepthAnythingEngine.infer_clip + RaftFlowEngine.infer_clip =
               the bands' video loops) from pinned host frames to pinned host results: every step uploads the chunk to
               each band and downloads the heat-encoded depth frame + (min,max) and the HSV-encoded forward and backward
               flow frames + max displacements of every frame
  roofline   : gemm_tc_kernel, the tcgen05 implicit-GEMM core that carries >70 % of the step (ViT linears, DPT head
               convs, RAFT encoder / update-block convs): algorithmic FLOP of all its launches / their CUDA-event time,
               vs the measured sustained bf16 peak; `groups` breaks it down and adds the attention kernel and the
               HBM-bound RAFT correlation build (vs the measured copy bandwidth)
  cpu_baseline / --impl reference : the oracle port of the reference's CPU fp32 path (oracle/da.py + oracle/raft.py) on
               the host cores: one frame for cpu_baseline, one frame per --steps step for --impl reference
  --dump-outputs DIR : what the last timed e2e step handed back to the caller, as .npy files (see dump_outputs)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W = 1080, 1920
ENCODER = os.environ.get("PRISMA_BENCH_ENCODER", "vitl")
RAFT_ITERS, RAFT_SCALE = 12, 0.75
# depth frames per engine pass (frames are independent): 12 frames land the attention grid and the GEMM tile counts just
# under whole waves (DESIGN.md section 5)
BATCH = int(os.environ.get("PRISMA_BENCH_BATCH", "12"))
FRAMES_PER_STEP = int(os.environ.get("PRISMA_BENCH_FRAMES", str(2 * BATCH)))
WORKLOAD = ("synthetic 1080p clip, depth_anything ViT-L + flow_raft (12 GRU iterations, fwd+bwd) on every frame, frames "
            "sharded per GPU (BASELINE metric: frames/sec at 1080p (depth_anything+flow_raft))")


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(hbm=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"], src="measured")
    except Exception:
        return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i] == "Active" for r in self.rows)]
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=reasons, samples=len(sm))


def make_frames(n, h, w, start):
    """Frames [start, start + n) of the synthetic clip (this rank's shard, prisma_b200.shard.frame_range)."""
    from prisma_b200.synthetic import synthetic_frame  # seeded synthetic clip shared with the tests
    base = [synthetic_frame(h, w, (start + t) % 256) for t in range(min(n, 4))]
    # 4 distinct generated frames (the generator is pure numpy and slow), then cheap deterministic variants
    frames = []
    for i in range(n):
        f = base[i % len(base)]
        frames.append(np.ascontiguousarray(np.roll(f, 7 * (i // len(base)), axis=1)))
    return frames


DUMP_SAMPLE = 1 << 21   # elements kept of an output larger than this: 3 frame stacks x 8 MB of float32, under 64 MB in all


def dump_outputs(directory, arrays):
    """Write each array as <directory>/<name>.npy in float32.  An array larger than DUMP_SAMPLE elements is replaced by a
    fixed sample of its flattened elements (sorted indices drawn from a generator seeded with 0), so two builds run with
    the same arguments can be compared output for output."""
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.size > DUMP_SAMPLE:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).integers(0, a.size, DUMP_SAMPLE))]
        np.save(os.path.join(directory, name + ".npy"), a.astype(np.float32))


def cpu_threads():
    """torch CPU scales to ~32 threads on the GPU box's host (measured with tools/cpu_threads.py: 8 thr 7.4 s/frame,
    16: 6.3, 32: 6.0, 64: 7.7, 128: 41 s/frame) -- use the optimum, and say so."""
    return min(32, os.cpu_count() or 1)


def cpu_reference_step(n_frames, threads):
    """The reference's CPU fp32 path for one frame of the workload -- depth_anything.infer + the heat encode, and
    flow_raft.infer (12 iterations, forward+backward) + process_flow of both directions -- as restated by the oracle
    (bit-equal to the imported reference modules, oracle/tools/make_golden.py), timed on the host cores.  frames/s."""
    import torch
    from oracle import da as oda
    from oracle import raft as oraft
    from prisma_b200.seeded_weights import make_da_weights, make_raft_weights
    torch.set_num_threads(threads)
    sd, rsd = make_da_weights(ENCODER, 0), make_raft_weights(0)
    frames = make_frames(n_frames + 1, H, W, 0)

    def one(prev, curr):
        oda.da_encode(oda.da_infer(sd, curr, ENCODER))
        a, b = oraft.raft_preprocess(prev, RAFT_SCALE)[None], oraft.raft_preprocess(curr, RAFT_SCALE)[None]
        fwd, bwd = oraft.raft_infer(rsd, torch.cat([a, b]), torch.cat([b, a]), iters=RAFT_ITERS)
        oraft.process_flow(fwd)
        oraft.process_flow(bwd)
    t0 = time.perf_counter()
    for i in range(n_frames):
        one(frames[i], frames[i + 1])
    dt = time.perf_counter() - t0
    return n_frames / dt, dt


def run_reference(args, rank, world):
    if rank != 0:
        return
    cores = cpu_threads()
    steps = args.steps  # one 1080p frame per step: ~15-40 s of CPU work each (ViT-L + RAFT)
    fps, dt = cpu_reference_step(steps, cores)
    out = {
        "impl": "reference", "metric": "frames/sec at 1080p (depth_anything+flow_raft)", "value": fps, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": 0, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "frame": [H, W], "encoder": ENCODER, "raft_iterations": RAFT_ITERS,
                   "raft_scale": RAFT_SCALE, "frames_per_step": 1},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{steps} frames of the 1080p clip, each through oracle/da.py (ViT-L + encode) and oracle/raft.py "
                                   f"(12 iterations, fwd+bwd, + process_flow), torch CPU fp32, {cores} threads (the measured optimum) "
                                   f"of {os.cpu_count()} host cores; no warm-up step (one frame costs tens of seconds)"},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(out), flush=True)


def measured_traffic():
    """DRAM bytes per launch of the profiled kernels from the committed ncu --set full captures (profiles/)."""
    for name in ("r02c_traffic.json", "r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                t = json.load(f)
            return t.get("traffic_bytes_per_launch"), t
        except Exception:
            continue
    return None, None


def corr_build_block(device, peaks):
    """The HBM-bound RAFT correlation-pyramid build alone (K13+K14, raft/corr.py:13-27), fwd+bwd, P = 102 x 180."""
    import ctypes as C
    from prisma_b200._lib import check, fptr, lib
    l = lib()
    h = C.c_void_p()
    rng = np.random.default_rng(0)
    fm = rng.standard_normal((2, 256, 102, 180), dtype=np.float32)
    check(l.prisma_flowcorr_create(device, 2, 102, 180, C.byref(h)))
    check(l.prisma_flowcorr_set_fmaps(h, fptr(fm), fptr(np.ascontiguousarray(fm[::-1]))))
    ms = C.c_float()
    check(l.prisma_flowcorr_build(h, 3, C.byref(ms)))
    check(l.prisma_flowcorr_build(h, 20, C.byref(ms)))
    work = (C.c_double * 2)()
    check(l.prisma_flowcorr_work(h, work))
    l.prisma_engine_destroy(h)
    gbs = work[1] / (ms.value * 1e-3) / 1e9
    tr = (measured_traffic()[1] or {}).get("corr_level0", {})
    return {"bound": "hbm", "kernel": "gemm_tc_kernel (RAFT all-pairs correlation pyramid: 2 GEMMs per direction (level 0; levels 1-3 side by side), K = 256 / 512, fp32 output)",
            "achieved": gbs, "peak": peaks["hbm"], "unit": "GB/s", "frac": gbs / peaks["hbm"], "ms_per_build": ms.value,
            "algorithmic_bytes": work[1], "traffic": tr.get("traffic_bytes_per_launch"), "traffic_detail": tr or None,
            "peak_source": peaks["src"],
            "note": "4-level fp32 pyramid written once (levels 1-3 by linearity: GEMMs against pooled features), timed alone, back to back"}


def midas_extras(device):
    """depth_midas (MiDaS v3 DPT_Large, BASELINE north_star band) on synthetic 720p frames, 12-frame passes, resident."""
    from prisma_b200.depth import MidasEngine
    from prisma_b200.seeded_weights import make_midas_weights
    eng = MidasEngine(make_midas_weights("dpt_large", 0), device=device)
    eng.time_resident(720, 1280, 2, BATCH)
    ms = eng.time_resident(720, 1280, 4, BATCH)
    w = eng.work(720, 1280, BATCH)
    eng.close()
    flop = w["linear_flop"] + w["attention_flop"] + w["head_flop"]
    return {"workload": "synthetic 720p frames, depth_midas DPT_Large, frames resident",
            "frames_per_s_device": BATCH / (ms * 1e-3), "ms_per_pass": ms, "frames_per_pass": BATCH,
            "tflops": flop / (ms * 1e-3) / 1e12, "launches_per_pass": w["launches"]}


def zoe_extras(device):
    """depth_anything --metric outdoor (what the reference's process.py passes by default): ZoeDepth metric head on ViT-L,
    392x518 network input, 12-frame passes, frames resident."""
    from prisma_b200.depth import ZoeDepthEngine
    from prisma_b200.seeded_weights import make_zoe_weights
    eng = ZoeDepthEngine(make_zoe_weights("vitl", 0), device=device, encoder="vitl")
    eng.time_resident(1080, 1920, 3, BATCH)
    ms = eng.time_resident(1080, 1920, 8, BATCH)
    w = eng.work(1080, 1920, BATCH)
    eng.close()
    return {"workload": "synthetic 1080p frames, depth_anything --metric (ZoeDepth head, 392x518 net input), frames resident",
            "frames_per_s_device": BATCH / (ms * 1e-3), "ms_per_pass": ms, "frames_per_pass": BATCH, "launches_per_pass": w["launches"]}


def mask_extras(device):
    """The mask band (SOLOv2 R-101) on synthetic 1080p frames: host frame in, union mask + instance list out (H2D / D2H
    inside the wall time; `ms` is the device time of the pass).  Three arithmetic variants of the same engine: "exact" (the
    band's default: the whole network in fp32-class 3xTF32, reproduces the oracle's instance list), "mixed" (fp16 backbone,
    fp32-class head + decode), "fast" (fp16 everywhere)."""
    from prisma_b200.mask import SoloV2Engine
    from prisma_b200.seeded_weights import make_solo_weights
    from prisma_b200.synthetic import synthetic_frame
    sd = make_solo_weights("r101", 0)
    f = [synthetic_frame(1080, 1920, t) for t in range(2)]
    out = {"workload": "synthetic 1080p frames, mask_mmdet SOLOv2 R-101 (768x1344 net input), one frame per pass, one lane"}
    for name, variant in (("exact", "r101-exact"), ("mixed", "r101"), ("fast", "r101-fast")):
        eng = SoloV2Engine(sd, device=device, variant=variant)
        for i in range(3):
            eng.infer(f[i % 2])
        n, dev_ms = 8, 0.0
        t0 = time.perf_counter()
        for i in range(n):
            dev_ms += eng.infer(f[i % 2])["ms"]
        e2e_s = time.perf_counter() - t0
        w = eng.work(1080, 1920)
        eng.close()
        out[name] = {"frames_per_s_device": n / (dev_ms * 1e-3), "frames_per_s_e2e": n / e2e_s, "ms_per_pass_device": dev_ms / n,
                     "algorithmic_gflop_per_pass": w["flop"] / 1e9, "tflops": w["flop"] / (dev_ms / n * 1e-3) / 1e12,
                     "launches_per_pass": w["launches"]}
    out.update({k: out["exact"][k] for k in ("frames_per_s_device", "frames_per_s_e2e", "ms_per_pass_device")})
    return out


def depth_720p_extras(eng):
    """BASELINE configs[1] (round 1's headline): depth_anything ViT-L on 720p frames, 12-frame passes, resident."""
    eng.time_resident(720, 1280, 2, BATCH)
    ms = eng.time_resident(720, 1280, 6, BATCH)
    return {"workload": "synthetic 720p frames, depth_anything ViT-L, frames resident (BASELINE configs[1])",
            "frames_per_s_device": BATCH / (ms * 1e-3), "ms_per_pass": ms, "frames_per_pass": BATCH}


def raft_extra_kernels(pairs):
    """Kernels launched by one RAFT video pass of `pairs` frame pairs beyond its step count: raft_preprocess = 2 kernels per
    new frame (1 step), corr_pool = 1 for all new frames (1 step), corr_build = 2 GEMMs per direction (level 0; levels 1-3
    side by side) (1 step), flow_encode = 3 per direction (1 step); reuse_prev is device-to-device copies, not a kernel."""
    return (2 * pairs - 1) + 0 + (4 * pairs - 1) + (6 * pairs - 1) - 1


def run_b200(args, rank, local_rank, world):
    import torch
    from prisma_b200.depth import DepthAnythingEngine, pinned_empty
    from prisma_b200.flow import RaftFlowEngine
    from prisma_b200.seeded_weights import make_da_weights, make_raft_weights   # the B200 arm never touches oracle/

    dist = None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(local_rank)

    from prisma_b200.shard import frame_range, max_over_ranks as _max_over_ranks

    def max_over_ranks(x):
        return _max_over_ranks(x, dist, f"cuda:{local_rank}")

    warm = max(args.warmup, 3)
    da = DepthAnythingEngine(ENCODER, make_da_weights(ENCODER, 0), device=local_rank)
    raft = RaftFlowEngine(make_raft_weights(0), device=local_rank, iterations=RAFT_ITERS, scale=RAFT_SCALE)
    shard_start, shard_stop, _ = frame_range(rank, world, FRAMES_PER_STEP * world)  # weak scaling: one chunk per GPU
    frames = make_frames(shard_stop - shard_start, H, W, shard_start)
    assert FRAMES_PER_STEP % BATCH == 0
    passes = FRAMES_PER_STEP // BATCH
    hs, ws = raft.out_size(H, W)
    # the step's frames and results in pinned host memory (SURVEY 8d: "frame in pinned host memory" -> "encoded u8 frame
    # + scalars in pinned host memory")
    clip = pinned_empty((FRAMES_PER_STEP, H, W, 3), np.uint8)
    clip[...] = np.stack(frames)
    out_depth_rgb = pinned_empty((FRAMES_PER_STEP, H, W, 3), np.uint8)
    out_flow = {"fwd_rgb": pinned_empty((FRAMES_PER_STEP, hs, ws, 3), np.uint8),
                "bwd_rgb": pinned_empty((FRAMES_PER_STEP, hs, ws, 3), np.uint8)}

    last = {}   # what the caller received from the most recent e2e step (for --dump-outputs)

    def e2e_step(cont):
        rgb, mins, maxs, _ = da.infer_clip(clip, pass_frames=BATCH, out_rgb=out_depth_rgb)
        r = raft.infer_clip(clip, continue_clip=cont, want_flow=False, want_rgb=True, out=out_flow)
        last.update(depth_rgb=rgb, depth_min=mins, depth_max=maxs, flow_fwd_rgb=r["fwd_rgb"], flow_bwd_rgb=r["bwd_rgb"],
                    flow_max_fwd=r["max_fwd"], flow_max_bwd=r["max_bwd"])
        return r["pairs"]

    # ---------------- e2e: public API, H2D + D2H inside the timed region.  The clip continues from step to step (every
    # frame is the `curr` of exactly one pair), so each step yields FRAMES_PER_STEP depth frames and FRAMES_PER_STEP pairs.
    e2e_step(False)
    for i in range(warm):
        assert e2e_step(True) == FRAMES_PER_STEP
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    t0 = time.perf_counter()
    for s in range(args.steps):
        e2e_step(True)
    torch.cuda.synchronize(local_rank)
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()

    # ---------------- value: the chunk resident in HBM, CUDA events on each engine's stream (inside the C ABI)
    da.time_resident(H, W, warm, BATCH)
    raft.time_resident(H, W, warm)
    barrier()
    res_ms = 0.0
    for s in range(args.steps):
        res_ms += da.time_resident(H, W, passes, BATCH) * passes         # ms per pass of BATCH frames
        res_ms += raft.time_resident(H, W, FRAMES_PER_STEP // raft.plan_pairs) * FRAMES_PER_STEP   # ms per pair (video passes)
    res_s = max_over_ranks(res_ms * 1e-3)
    clocks = sampler.stop()
    barrier()

    da_prof = da.profile(H, W, BATCH)     # per kernel-group CUDA-event times of one pass of BATCH frames (ms)
    da_work = da.work(H, W, BATCH)
    rf_prof = raft.profile(H, W)          # ... of one video pass, per frame pair
    rf_work = raft.work_detail(H, W)
    if rank == 0:
        peaks = measured_peaks()
        total_frames = args.steps * FRAMES_PER_STEP * world
        value = total_frames / res_s
        tf = lambda flop, ms: flop / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
        # all launches of gemm_tc_kernel in one step: DA linears + head convs (per pass) and RAFT convs (per pair)
        gemm_flop = (da_work["linear_flop"] + da_work["head_flop"]) * passes + rf_work["conv_flop_video"] * FRAMES_PER_STEP
        gemm_ms = (da_prof["linear"] + da_prof["head"]) * passes + rf_prof["conv_gemm"] * FRAMES_PER_STEP
        step_ms_prof = da_prof["total"] * passes + rf_prof["total"] * FRAMES_PER_STEP
        gemm_tf = tf(gemm_flop, gemm_ms)
        corr_gbs = rf_work["corr_bytes"] / (rf_prof["corr_build"] * 1e-3) / 1e9 if rf_prof["corr_build"] > 0 else 0.0
        rf_np = rf_work["pairs_per_pass"]
        launches_step = da_work["launches"] * passes + (rf_work["launches_video"] + raft_extra_kernels(rf_np)) * (FRAMES_PER_STEP // rf_np)
        out = {
            "metric": "frames/sec at 1080p (depth_anything+flow_raft)", "value": value, "unit": "frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": 1e3 * res_s / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16 operands, f32 accumulate", "data": "synthetic",
            "config": {"workload": WORKLOAD, "frame": [H, W], "encoder": ENCODER, "raft_iterations": RAFT_ITERS,
                       "raft_scale": RAFT_SCALE, "frames_per_step": FRAMES_PER_STEP, "depth_frames_per_pass": BATCH,
                       "flow_pairs_per_pass": rf_np, "parallelism": f"frame-sharded x{world}",
                       "l2": "working set per step (0.6 GB fp16 ViT-L weights, 3.6 GB correlation pyramids per pair, activations) "
                             "exceeds the 126 MB L2; no flush needed"},
            "e2e": {"value": total_frames / e2e_s, "unit": "frames/s",
                    "h2d_bytes_per_step": 2 * FRAMES_PER_STEP * H * W * 3,   # each band uploads the chunk
                    "d2h_bytes_per_step": FRAMES_PER_STEP * (H * W * 3 + 8 + 2 * hs * ws * 3 + 8)},
            "gpu_launches": launches_step * args.steps,
            "clocks": clocks,
            "roofline": {"bound": "tensor",
                         "kernel": "gemm_tc_kernel (every tcgen05 contraction of the step: ViT-L linears, DPT head convs, RAFT "
                                   "encoder / motion / ConvGRU / head convs)",
                         "achieved": gemm_tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": gemm_tf / peaks["tf_sustained"],
                         "traffic": measured_traffic()[0], "traffic_detail": measured_traffic()[1], "peak_source": peaks["src"],
                         "share_of_step": gemm_ms / step_ms_prof if step_ms_prof > 0 else None,
                         "groups": {
                             "da_encoder_linears": {"tflops": tf(da_work["linear_flop"], da_prof["linear"]), "ms_per_pass": da_prof["linear"],
                                                    "frac": tf(da_work["linear_flop"], da_prof["linear"]) / peaks["tf_sustained"]},
                             "da_attention": {"tflops": tf(da_work["attention_flop"], da_prof["attention"]), "ms_per_pass": da_prof["attention"]},
                             "da_head_convs": {"tflops": tf(da_work["head_flop"], da_prof["head"]), "ms_per_pass": da_prof["head"]},
                             "raft_convs": {"tflops": tf(rf_work["conv_flop_video"], rf_prof["conv_gemm"]), "ms_per_pair": rf_prof["conv_gemm"]},
                             "raft_corr_build_in_pass": {"bound": "hbm", "achieved": corr_gbs, "peak": peaks["hbm"], "unit": "GB/s",
                                                         "frac": corr_gbs / peaks["hbm"], "ms_per_pair": rf_prof["corr_build"],
                                                         "algorithmic_bytes": rf_work["corr_bytes"]},
                             "da_ms_per_pass": da_prof, "raft_ms_per_pair": rf_prof},
                         "frame_flop": {"depth_anything": (da_work["linear_flop"] + da_work["attention_flop"] + da_work["head_flop"]) / BATCH,
                                        "flow_raft_video_pass": rf_work["conv_flop_video"] + rf_work["corr_flop"]}},
        }
        if world == 1:
            # secondary workloads: a failure there is reported in place and never costs the headline line
            out["extra"] = {}

            def extra(name, fn):
                try:
                    out["extra"][name] = fn()
                except Exception as ex:  # noqa: BLE001
                    out["extra"][name] = {"error": f"{type(ex).__name__}: {ex}"}

            extra("raft_corr_build", lambda: corr_build_block(local_rank, peaks))
            extra("depth_anything_720p", lambda: depth_720p_extras(da))
            if not args.no_extras:
                raft.close()
                extra("depth_midas_720p", lambda: midas_extras(local_rank))
                extra("mask_mmdet_1080p", lambda: mask_extras(local_rank))
                extra("depth_anything_metric_1080p", lambda: zoe_extras(local_rank))
        if world == 1 and not args.no_cpu:
            cores = cpu_threads()
            fps, dt = cpu_reference_step(1, cores)
            out["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port",
                                   "sample": f"1 frame of the 1080p clip through oracle/da.py (ViT-L + encode) and oracle/raft.py (12 "
                                             f"iterations, fwd+bwd, + process_flow), torch CPU fp32, {cores} threads of "
                                             f"{os.cpu_count()} host cores (the measured optimum), {dt:.1f} s"}
        print(json.dumps(out), flush=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    da.close()
    raft.close()
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=6)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary workloads (other bands)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last end-to-end step returned (depth and flow frames, "
                         "per-frame scalars) as DIR/<name>.npy in float32; frame stacks are a fixed seeded sample; "
                         "rank 0's frames when --gpus > 1")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_b200(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
