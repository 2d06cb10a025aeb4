"""Host-side logic on CPU: transform size arithmetic of every band through the C ABI vs the oracle (hypothesis), the
metadata helpers, the .flo writer."""
import ctypes as C
import json
import os

import numpy as np
from hypothesis import given, settings, strategies as st

from oracle import da as oda
from oracle import midas as omidas
from prisma_b200._lib import check, lib


def net_size(band, w, h):
    wn, hn = C.c_int(), C.c_int()
    check(lib().prisma_net_size(band.encode(), w, h, C.byref(wn), C.byref(hn)))
    return wn.value, hn.value


@settings(max_examples=300, deadline=None)
@given(st.integers(32, 4096), st.integers(32, 2304))
def test_transform_sizes_match_the_oracle(w, h):
    assert net_size("depth_anything", w, h) == oda.da_get_size(w, h)
    assert net_size("depth_midas", w, h) == omidas.midas_get_size(w, h)
    assert net_size("depth_anything_metric", w, h) == (518, 392)
    s = min(1333 / max(h, w), 800 / min(h, w))
    assert net_size("mask_mmdet", w, h) == (int(w * s + 0.5), int(h * s + 0.5))


def test_survey_sizes():
    # SURVEY.md section 8: both 720p and 1080p give a 518x924 Depth-Anything input and a 750x1333 SOLOv2 input
    for w, h in ((1280, 720), (1920, 1080)):
        assert net_size("depth_anything", w, h) == (924, 518)
        assert net_size("mask_mmdet", w, h) == (1333, 750)
    assert net_size("depth_anything", 640, 480) == (686, 518) and net_size("depth_midas", 640, 480) == (384, 288)


def test_flo_writer_and_metadata_roundtrip(tmp_path):
    from prisma_b200.flow import write_flo
    from bands.common import meta
    flow = np.random.default_rng(0).standard_normal((5, 7, 2)).astype(np.float32)
    p = tmp_path / "f.flo"
    write_flo(str(p), flow)
    raw = np.fromfile(p, np.float32)
    assert raw[0] == np.float32(202021.25) and tuple(raw[1:3].view(np.int32)) == (7, 5)   # Middlebury header: w, h
    assert np.array_equal(raw[3:].reshape(5, 7, 2), flow)
    folder = tmp_path / "clip"
    data = meta.create_metadata(str(folder))
    meta.add_band(data, "rgba", url="rgba.mp4")
    meta.write_metadata(str(folder), data)
    meta.set_default_band(str(folder), "depth", "rgba")
    back = meta.load_metadata(str(folder))
    assert back["bands"]["rgba"]["url"] == "rgba.mp4" and back["bands"]["depth"] == back["bands"]["rgba"]
    assert meta.get_url(str(folder), back, "rgba") == os.path.join(str(folder), "rgba.mp4")
    assert json.load(open(folder / "metadata.json")) == back


def test_shard_flag_stripping_and_frame_ranges():
    """`<band>.py --gpus N` hands its workers the same command line minus the sharding flags; every worker owns a contiguous
    frame range (flow bands read one halo frame)."""
    from bands.common.sharded import strip_flags
    from prisma_b200.shard import frame_range
    argv = ["-i", "clip", "--gpus", "4", "--encoder", "vits", "--device-list=0,1,2,3", "-o", "x.mp4", "--seeded-weights", "--device", "3", "-n"]
    assert strip_flags(argv) == ["-i", "clip", "--encoder", "vits", "-o", "x.mp4", "--seeded-weights", "-n"]
    got = [frame_range(r, 3, 100, 1) for r in range(3)]
    assert [g[0] for g in got] == [0] + [g[1] for g in got[:-1]] and got[-1][1] == 100   # contiguous cover of [0, 100)
    assert got[0][2] == 0 and all(g[2] == g[0] - 1 for g in got[1:])                      # halo frame

def test_mask_band_precision_flag_selects_the_engine_variant():
    """bands/mask_mmdet.py --precision: exact (default, the whole network fp32-class) / mixed / fast -> engine variant names."""
    from bands import mask_mmdet as band
    p = band.build_parser()
    assert p.parse_args(["-i", "x.png"]).precision == "exact"
    for flag, variant in (("exact", "r101-exact"), ("mixed", "r101"), ("fast", "r101-fast")):
        a = p.parse_args(["-i", "x.png", "--precision", flag])
        assert "r101" + {"fast": "-fast", "exact": "-exact"}.get(a.precision, "") == variant


def test_bench_dump_outputs_is_bounded_and_reproducible(tmp_path):
    """bench.py --dump-outputs at the benchmark's own output shapes: float32 .npy files, 64 MB at most in all, the same
    sample from run to run, small arrays kept whole."""
    import bench
    n, hs, ws = bench.FRAMES_PER_STEP, int(np.rint(bench.H * bench.RAFT_SCALE)), int(np.rint(bench.W * bench.RAFT_SCALE))
    rng = np.random.default_rng(1)
    arrays = {"depth_rgb": rng.integers(0, 256, (n, bench.H, bench.W, 3), dtype=np.uint8),
              "flow_fwd_rgb": rng.integers(0, 256, (n, hs, ws, 3), dtype=np.uint8),
              "flow_bwd_rgb": rng.integers(0, 256, (n, hs, ws, 3), dtype=np.uint8),
              "depth_min": rng.standard_normal(n).astype(np.float32), "flow_max_fwd": rng.standard_normal(n).astype(np.float32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(k + ".npy" for k in arrays)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 << 20
    for f in files:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b)
    assert np.array_equal(np.load(tmp_path / "a" / "depth_min.npy"), arrays["depth_min"])
    assert np.load(tmp_path / "a" / "depth_rgb.npy").size == bench.DUMP_SAMPLE
