"""oracle/solo.py replayed against the fixture written by oracle/tools/make_golden.py (golden_solo) from the VENDORED mmdet
sources -- ResNet, FPN, MaskFeatModule, SOLOV2Head.forward, get_results, mask_matrix_nms, generate_coordinate, loaded by
path with the absent mmcv's three primitives (ConvModule, BaseModule, build_*_layer) stubbed -- bit-equal there.  CPU."""
import os

import numpy as np
import torch

from oracle import solo as osolo
from prisma_b200.seeded_weights import SOLO_CONFIGS, make_solo_weights


def test_solo_oracle_matches_vendored_mmdet_fixture(golden_dir, recorded_threads):
    g = np.load(os.path.join(golden_dir, "solo_tiny_head.npz"))
    sd = make_solo_weights("tiny", 0)
    c = SOLO_CONFIGS["tiny"]
    with torch.no_grad():
        fpn = osolo.fpn(sd, osolo.resnet(sd, torch.from_numpy(g["net_x"]), c["layers"]))
        for i, f in enumerate(fpn):
            assert np.array_equal(f.numpy(), g[f"fpn{i}"]), f"fpn{i}"
        feats = [torch.from_numpy(g[f"feat{i}"].astype(np.float32)) for i in range(5)]
        mf = osolo.mask_feat(sd, feats)
        kernels, cls = osolo.head(sd, feats, c["num_grids"])
        assert np.array_equal(mf.numpy()[:, ::8], g["mask_feats_sub"])
        assert np.array_equal(cls[0].numpy(), g["cls0"]) and np.array_equal(kernels[4].numpy(), g["kernel4"])
        scores, labels, masks = osolo.get_results(kernels, cls, mf, dict(img_shape=(250, 333), ori_shape=(240, 320)),
                                                  osolo.TEST_CFG, c["strides"], c["num_grids"])
    n = int(g["n"])
    assert len(scores) == n and np.array_equal(labels.numpy(), g["labels"]) and np.array_equal(scores.numpy(), g["scores"])
    assert np.array_equal(np.packbits(masks.numpy(), axis=-1), g["masks"])
