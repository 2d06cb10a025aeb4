"""oracle/zoe.py replayed against the fixture written by oracle/tools/make_golden.py from the imported reference ZoeDepth
(bit-equal there); runs on CPU."""
import os

import numpy as np

from oracle import da as oda
from oracle import zoe as ozoe
from prisma_b200.seeded_weights import make_zoe_weights


def test_zoe_oracle_matches_reference_fixture(golden_dir, recorded_threads):
    g = np.load(os.path.join(golden_dir, "zoe_vits_240x320.npz"))
    sd = make_zoe_weights("vits", 0)
    taps = {}
    pred = ozoe.zoe_infer(sd, g["image"], "vits", taps)
    assert np.array_equal(taps["metric"].squeeze().numpy(), g["metric_net"])
    assert np.array_equal(pred, g["prediction"])
    rgb, dmin, dmax = oda.da_encode(pred, flip=False)
    assert np.array_equal(rgb, g["rgb"]) and np.float32(dmin) == g["dmin"] and np.float32(dmax) == g["dmax"]
