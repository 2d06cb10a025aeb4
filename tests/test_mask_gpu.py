"""mask_mmdet band (SURVEY.md section 8 rows a15-a19): SOLOv2 CUDA path vs oracle/solo.py, stage by stage.

The oracle restates the vendored mmdet sources and is pinned bit-equal to them (loaded by path with mmcv's primitives
stubbed, see oracle/solo.py and tests/golden/solo_tiny_head.npz).
"tiny" is a test-size twin of the same graph (one bottleneck per ResNet stage, test scale (448, 256)); "r101" is the
real configuration.  Float stages: 1e-3-class tolerances (fp16 operands, fp32 accumulate, fp16 feature maps); the decode
is integer / boolean work downstream of those floats, so it is compared as sets: same instances (label, score within
2e-3, mask IoU >= 0.97) wherever the oracle's own decisions are not within rounding of a threshold.
"""
import numpy as np
import pytest
import torch

from oracle import solo as osolo
from prisma_b200.synthetic import synthetic_frame
from prisma_b200.seeded_weights import SOLO_CONFIGS, make_solo_weights


def rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max()), float(np.linalg.norm(a - b) / np.linalg.norm(b))


def test_solo_oracle_pipeline_shapes():
    # 1080p and 720p both land on 750x1333 -> padded 768x1344 (SURVEY.md section 8 sizes)
    for hw in ((1080, 1920), (720, 1280)):
        x, meta = osolo.solo_preprocess(np.zeros(hw + (3,), np.uint8))
        assert meta["img_shape"] == (750, 1333) and tuple(x.shape) == (1, 3, 768, 1344)
    c = SOLO_CONFIGS["r101"]
    assert sum(g * g for g in c["num_grids"]) == 3872


@pytest.fixture(scope="module")
def tiny():
    from prisma_b200.mask import SoloV2Engine
    sd = make_solo_weights("tiny", 0)
    eng = SoloV2Engine(sd, variant="tiny")
    yield eng, sd
    eng.close()


def check_instances(res, scores, labels, masks, min_match=0.9, tag=""):
    """GPU instances vs oracle instances: greedy match on (label, IoU).  Prints the residual: how many oracle instances were
    reproduced (same label, IoU >= 0.97, score within 2 %), how many at the same rank, and for every miss its rank / score and
    the best same-label IoU found -- the misses sit at the tail of the list, where consecutive scores differ by less than the
    backbone's fp16 rounding moves them (the max_per_img = 100 cut and the 0.05 filter threshold then pick other members)."""
    n_ref = len(scores)
    assert abs(len(res["scores"]) - n_ref) <= max(2, n_ref // 10), (len(res["scores"]), n_ref)
    ref_m = masks.numpy().reshape(n_ref, -1)
    got_m = res["masks"].reshape(len(res["scores"]), -1)
    used, matched, same_rank, misses, score_err = set(), 0, 0, [], []
    for i in range(n_ref):
        best, bj = 0.0, -1
        for j in range(len(res["scores"])):
            if j in used or res["labels"][j] != int(labels[i]):
                continue
            inter = np.logical_and(ref_m[i], got_m[j]).sum()
            union = np.logical_or(ref_m[i], got_m[j]).sum()
            iou = inter / union if union else 1.0
            if iou > best:
                best, bj = iou, j
        if bj >= 0 and best >= 0.97 and abs(float(scores[i]) - float(res["scores"][bj])) <= 2e-3 + 2e-2 * float(scores[i]):
            used.add(bj)
            matched += 1
            same_rank += int(bj == i)
            score_err.append(abs(float(scores[i]) - float(res["scores"][bj])) / max(float(scores[i]), 1e-6))
        else:
            misses.append((i, round(float(scores[i]), 5), int(labels[i]), round(float(best), 3)))
    gaps = np.diff(-np.asarray(scores, dtype=np.float64)) if n_ref > 1 else np.array([0.0])
    print(f"{tag} instances: {matched}/{n_ref} reproduced ({same_rank} at the same rank), median score rel err "
          f"{np.median(score_err) if score_err else float('nan'):.2e}, max {max(score_err) if score_err else float('nan'):.2e}; "
          f"median gap between consecutive oracle scores {np.median(gaps):.2e}; misses (rank, score, label, best IoU): {misses[:12]}")
    assert matched >= min_match * n_ref, (matched, n_ref)
    return matched, misses


@pytest.mark.gpu
def test_solo_tiny_stages_and_results(tiny):
    eng, sd = tiny
    img = synthetic_frame(240, 320, 0)
    res = eng.infer(img, confidence=0.5, want_instances=True)
    taps = {}
    scores, labels, masks = osolo.solo_infer(sd, img, "tiny", taps)
    meta = taps["meta"]
    nh, nw = meta["img_shape"]
    hp, wp = meta["pad_shape"]
    # test pipeline: cv2 8-bit bilinear (fixed point, emulated exactly) + normalise + pad: byte-equal / float-equal
    rs = eng.read_tap("resized", (nh, nw, 3)).astype(np.uint8)
    assert np.array_equal(rs, meta["resized_u8"])
    net = eng.read_tap("net_input", (3, hp, wp))
    assert np.abs(net - taps["net_input"][0].numpy()).max() <= 1e-6
    # FPN levels (ResNet + FPN)
    for i, f in enumerate(taps["fpn"]):
        got = eng.read_tap(f"fpn{i}", (f.shape[2], f.shape[3], 256)).transpose(2, 0, 1)
        m, l2 = rel(got, f[0].numpy())
        assert m < 4e-3 and l2 < 2e-3, (f"fpn{i}", m, l2)
    mf = taps["mask_feats"][0]
    got = eng.read_tap("mask_feats", (mf.shape[1] * mf.shape[2], 256)).T.reshape(mf.shape)
    m, l2 = rel(got, mf.numpy())
    assert m < 6e-3 and l2 < 3e-3, ("mask_feats", m, l2)
    for l, (k, c) in enumerate(zip(taps["kernels"], taps["cls"])):
        S = k.shape[-1]
        gk = eng.read_tap(f"kernel{l}", (S * S, 256)).T.reshape(k.shape[1:])
        gc = eng.read_tap(f"cls{l}", (S * S, 80)).T.reshape(c.shape[1:])
        m, l2 = rel(gk, k[0].numpy())
        assert m < 8e-3 and l2 < 4e-3, (f"kernel{l}", m, l2)
        assert np.abs(gc - c[0].numpy()).max() < 2e-2, (f"cls{l}", np.abs(gc - c[0].numpy()).max())   # logits around -8
    n_cand = int((taps["cls_scores"] > 0.1).sum())
    got_cand = int(eng.read_tap("cand_count", (1,))[0])
    assert abs(got_cand - n_cand) <= max(3, n_cand // 50), (got_cand, n_cand)
    check_instances(res, scores, labels, masks, tag="tiny 240x320")
    ref_union = osolo.band_union(scores, labels, masks, 0.5)[..., 0]
    assert (res["union"] != ref_union).mean() < 5e-3
    bbox, mres = eng.inference_detector(img)
    assert len(bbox) == 80 and len(mres) == 80 and sum(len(m) for m in mres) == len(res["scores"])


@pytest.mark.gpu
def test_solo_head_and_decode_from_the_reference_levels_reproduce_the_reference_instances(tiny, golden_dir):
    """north_star: mask ids bit-exact.  tests/golden/solo_tiny_head.npz holds the VENDORED mmdet SOLOV2Head's own FPN
    levels and its final scores / labels / masks (oracle/tools/make_golden.py).  Replaying head + decode from those levels
    on the fp32-class path (three kind::tf32 tensor-core passes per contraction, fp32 activations) must give the same
    instance list: the same labels in the same order, scores to 5e-5 relative, masks bit-equal except razor-margin boundary
    pixels (|p - 0.5| ~ 1e-6), at most 1e-6 of the bits.  Measured on B200: labels equal, scores 6.4e-6, 3 of 7.68 M mask
    bits (an exact-arithmetic emulation of 3xTF32 in the oracle: 1.5e-6 and 1 bit; two fp32 implementations that sum in a
    different order -- cuDNN vs MKL-DNN -- differ the same way).  Getting there needed the external fp32 accumulation of
    gemm_prepare_tf32x3: with whole-K TMEM chains the tensor core's truncating accumulate left 4.6e-4 on the class logits,
    swapped two ranks and moved scores by 2e-3.  The single-pass fp16 head of round 1 changes a third of the list on the
    same input (labels differ, scores off by 2e-3, 4 % of the mask bits)."""
    import os
    eng, sd = tiny
    g = np.load(os.path.join(golden_dir, "solo_tiny_head.npz"))
    frame = synthetic_frame(240, 320, 0)
    eng.infer(frame, confidence=0.5)                       # plans the 240x320 geometry (250x333 -> padded 256x352)
    feats = [g[f"feat{i}"].astype(np.float32) for i in range(5)]
    res = eng.infer_from_feats(feats, (240, 320), confidence=0.5, img_shape=(250, 333))   # the fixture's meta (make_golden.py)
    n = int(g["n"])
    ref_masks = np.unpackbits(g["masks"], axis=-1)[..., :320].astype(bool)
    # intermediate tensors against the reference's own
    cls0 = eng.read_tap("cls0", (40 * 40, 80)).T.reshape(80, 40, 40)
    k4 = eng.read_tap("kernel4", (12 * 12, 256)).T.reshape(256, 12, 12)
    mf = eng.read_tap("mask_feats", (64 * 88, 256)).T.reshape(256, 64, 88)
    e_cls = float(np.abs(cls0 - g["cls0"][0]).max())
    e_k = float(np.abs(k4 - g["kernel4"][0]).max() / np.abs(g["kernel4"]).max())
    e_mf = float(np.abs(mf[::8] - g["mask_feats_sub"][0]).max() / np.abs(g["mask_feats_sub"]).max())
    print(f"exact head vs reference: cls logits max abs {e_cls:.2e}, kernel preds rel {e_k:.2e}, mask feats rel {e_mf:.2e}")
    same_n = len(res["scores"]) == n
    lab_eq = same_n and np.array_equal(res["labels"], g["labels"][:n].astype(np.int32))
    rel = np.abs(res["scores"] - g["scores"][:n]) / np.maximum(g["scores"][:n], 1e-6) if same_n else np.array([np.inf])
    diff_bits = int((res["masks"] != ref_masks[:n]).sum()) if same_n else -1
    print(f"instances {len(res['scores'])} (reference {n}): labels equal {lab_eq}, max score rel err {rel.max():.2e}, "
          f"mask bits differing {diff_bits} of {ref_masks[:n].size}")
    if same_n and not lab_eq:
        bad = np.nonzero(res["labels"] != g["labels"][:n])[0]
        print("  first label mismatches (rank, got, ref, score got, score ref):",
              [(int(i), int(res["labels"][i]), int(g["labels"][i]), float(res["scores"][i]), float(g["scores"][i])) for i in bad[:6]])
    assert e_cls <= 5e-5 and e_k <= 1e-5 and e_mf <= 5e-6, (e_cls, e_k, e_mf)
    assert same_n and lab_eq
    assert rel.max() <= 5e-5, rel.max()
    assert diff_bits <= 1e-6 * ref_masks[:n].size, diff_bits


@pytest.mark.gpu
@pytest.mark.parametrize("H,W", [(160, 208), (480, 640), (720, 1280), (1080, 1920), (333, 517)])
def test_solo_test_pipeline_resize_is_byte_equal_to_cv2(tiny, H, W):
    """mmcv.imrescale = cv2.resize(INTER_LINEAR) on u8, up- and down-scaling, noise frames (the hardest case for a
    fixed-point emulation): the resized image is byte-equal to cv2's (oracle/solo.py calls cv2 itself)."""
    eng, sd = tiny
    img = np.random.default_rng(H * W).integers(0, 256, (H, W, 3), dtype=np.uint8)
    eng.infer(img, confidence=0.5)
    x, meta = osolo.solo_preprocess(img, SOLO_CONFIGS["tiny"]["img_scale"])
    nh, nw = meta["img_shape"]
    rs = eng.read_tap("resized", (nh, nw, 3)).astype(np.uint8)
    assert np.array_equal(rs, meta["resized_u8"])


@pytest.fixture(scope="module")
def r101_oracle():
    """The CPU oracle on the R-101 config (one 720p frame): shared by the fp16-backbone and the fp32-class-backbone tests."""
    sd = make_solo_weights("r101", 0)
    img = synthetic_frame(720, 1280, 0)
    taps = {}
    scores, labels, masks = osolo.solo_infer(sd, img, "r101", taps)
    return sd, img, taps, scores, labels, masks


@pytest.mark.gpu
def test_solo_r101_720p_matches_oracle(r101_oracle):
    from prisma_b200.mask import SoloV2Engine
    sd, img, taps, scores, labels, masks = r101_oracle
    eng = SoloV2Engine(sd, variant="r101")
    res = eng.infer(img, confidence=0.3, want_instances=True)
    for i in (0, 3):
        f = taps["fpn"][i]
        got = eng.read_tap(f"fpn{i}", (f.shape[2], f.shape[3], 256)).transpose(2, 0, 1)
        m, l2 = rel(got, f[0].numpy())
        assert m < 1e-2 and l2 < 4e-3, (f"fpn{i}", m, l2)   # 33 bottlenecks of fp16 maps
    eng.close()
    check_instances(res, scores, labels, masks, min_match=0.8, tag="r101 720p")


def check_instances_exact(res, scores, labels, masks, tag="", score_tol=5e-5):
    """north_star: mask ids bit-exact.  The fp32-class engine ("-exact": backbone, FPN, head and decode all in 3xTF32 with
    fp32 accumulation) must reproduce the oracle's instance list itself: same count, same labels in the same order, scores to
    fp32 summation-order accuracy, and masks that differ in at most a 1e-5 fraction of their bits (two fp32 implementations
    that add in a different order differ the same way at pixels whose mask logit sits within 1e-6 of the threshold)."""
    n_ref = len(scores)
    assert len(res["scores"]) == n_ref, (len(res["scores"]), n_ref)
    assert np.array_equal(res["labels"], np.asarray(labels, dtype=res["labels"].dtype)), "labels / order differ"
    serr = np.abs(res["scores"] - np.asarray(scores, np.float32)) / np.maximum(np.asarray(scores, np.float32), 1e-6)
    ref_m = masks.numpy().reshape(n_ref, -1).astype(bool)
    got_m = res["masks"].reshape(n_ref, -1)
    bits = int((ref_m != got_m).sum())
    print(f"{tag} exact: {n_ref} instances, labels equal in order, score rel err max {serr.max() if n_ref else 0:.2e}, "
          f"{bits} of {ref_m.size} mask bits differ")
    assert (serr.max() if n_ref else 0.0) <= score_tol
    assert bits <= max(8, int(1e-5 * ref_m.size)), (bits, ref_m.size)
    return bits


@pytest.mark.gpu
def test_solo_tiny_exact_backbone_reproduces_the_oracle_instances():
    """End to end (frame -> instances) on the test-size twin with the fp32-class backbone: FPN levels to 1e-5, instances exact."""
    from prisma_b200.mask import SoloV2Engine
    sd = make_solo_weights("tiny", 0)
    eng = SoloV2Engine(sd, variant="tiny-exact")
    img = synthetic_frame(240, 320, 0)
    res = eng.infer(img, confidence=0.5, want_instances=True)
    taps = {}
    scores, labels, masks = osolo.solo_infer(sd, img, "tiny", taps)
    for i, f in enumerate(taps["fpn"]):
        got = eng.read_tap(f"fpn{i}", (f.shape[2], f.shape[3], 256)).transpose(2, 0, 1)
        m, l2 = rel(got, f[0].numpy())
        print(f"tiny-exact fpn{i}: max rel {m:.2e} l2 rel {l2:.2e}")
        assert m < 2e-5 and l2 < 5e-6, (f"fpn{i}", m, l2)
    eng.close()
    check_instances_exact(res, scores, labels, masks, tag="tiny-exact 240x320")
    ref_union = osolo.band_union(scores, labels, masks, 0.5)[..., 0]
    assert (res["union"] != ref_union).mean() <= 1e-5


@pytest.mark.gpu
def test_solo_r101_exact_backbone_720p_reproduces_the_oracle_instances(r101_oracle):
    """The real config (ResNet-101, 33 bottlenecks) with the fp32-class backbone: the instance list of the oracle itself."""
    from prisma_b200.mask import SoloV2Engine
    sd, img, taps, scores, labels, masks = r101_oracle
    eng = SoloV2Engine(sd, variant="r101-exact")
    res = eng.infer(img, confidence=0.3, want_instances=True)
    for i in (0, 3):
        f = taps["fpn"][i]
        got = eng.read_tap(f"fpn{i}", (f.shape[2], f.shape[3], 256)).transpose(2, 0, 1)
        m, l2 = rel(got, f[0].numpy())
        print(f"r101-exact fpn{i}: max rel {m:.2e} l2 rel {l2:.2e}  ({res['ms']:.2f} ms per frame)")
        assert m < 1e-4 and l2 < 5e-5, (f"fpn{i}", m, l2)   # 100 convs deep: the summation-order differences add up
    eng.close()
    # 100 convs deep the tensor core's truncating fp32 accumulate (chains of 16 MMAs between the round-to-nearest external
    # sums) shows as a uniform 1.5e-5 shrink of the FPN levels; the scores follow (measured 1.07e-4 relative, 5.5e-5 with
    # chains of 4 MMAs); the instance list and all but 53 of 18.4 M mask bits are the oracle's
    check_instances_exact(res, scores, labels, masks, tag="r101-exact 720p", score_tol=2e-4)


@pytest.mark.gpu
def test_sdf_green_channel_bit_exact():
    """--sdf: exact Euclidean signed distance of the union -> green channel, vs scipy's exact EDT (integer squared
    distances, correctly rounded sqrt: bit-exact)."""
    from prisma_b200.mask import sdf_green
    rng = np.random.default_rng(0)
    H, W = 270, 480
    yy, xx = np.mgrid[0:H, 0:W]
    m = np.zeros((H, W), np.uint8)
    for _ in range(7):  # a few discs and boxes, some overlapping (254 = two instances)
        cy, cx, r = rng.integers(0, H), rng.integers(0, W), rng.integers(8, 60)
        m[(yy - cy) ** 2 + (xx - cx) ** 2 < r * r] += 255
    m[100:140, 200:330] = 255
    assert np.array_equal(sdf_green(m), osolo.sdf_green(m))
    for special in (np.zeros((64, 96), np.uint8), np.full((64, 96), 255, np.uint8)):
        assert np.array_equal(sdf_green(special), osolo.sdf_green(special))


@pytest.mark.gpu
def test_solo_lanes_equal_sequential_calls():
    """SoloV2Lanes.map (three engines taking consecutive frames from worker threads, the band's video loop) returns the same
    unions / scores / labels, in frame order, as one engine called frame by frame."""
    from prisma_b200.mask import SoloV2Engine, SoloV2Lanes
    from prisma_b200.seeded_weights import make_solo_weights
    from prisma_b200.synthetic import synthetic_frame
    sd = make_solo_weights("tiny", 0)
    frames = [synthetic_frame(240, 320, t) for t in range(7)]
    one = SoloV2Engine(sd, variant="tiny")
    ref = [one.infer(f, confidence=0.3) for f in frames]
    one.close()
    lanes = SoloV2Lanes(sd, variant="tiny", lanes=3)
    got = list(lanes.map(iter(frames), confidence=0.3))
    lanes.close()
    assert len(got) == len(ref)
    for a, b in zip(got, ref):
        assert np.array_equal(a["union"], b["union"]) and np.array_equal(a["scores"], b["scores"]) and np.array_equal(a["labels"], b["labels"])
