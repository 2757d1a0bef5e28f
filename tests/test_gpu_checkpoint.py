"""SURVEY.md §8f rank 1 on the GPU: the trained weights of the reference's shipped `bat_kitti_car.ckpt` through the fused CUDA
path in eval mode reproduce what the REFERENCE's own BAT computes with those weights.  tests/golden/bat_kitti_car_q4.npz,
written by tests/golden/make_golden.py, holds the weights as 4-bit codes per output channel with BatchNorm statistics and
biases exact (the float32 originals are 6 MB), and the reference's outputs computed with exactly those weights."""
import os

import numpy as np
import pytest
import torch

from _params import unpack_state_4bit
from open3dsot_b200.config import load_config
from open3dsot_b200.datasets.synthetic import synthetic_siamese_batch
from open3dsot_b200.models import get_model

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "bat_kitti_car_q4.npz")


def rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def test_real_checkpoint_eval_outputs_match_the_reference():
    g = dict(np.load(GOLDEN))
    cfg = load_config(os.path.join(ROOT, "cfgs", "BAT_Car.yaml"))
    net = get_model(cfg.net_model)(cfg)
    net.load_state_dict(unpack_state_4bit({k: v for k, v in g.items() if not k.startswith("out:")}), strict=True)
    net = net.cuda().eval()
    batch = synthetic_siamese_batch(2, 512, 1024, seed=4242, box_aware=True, device="cuda")
    with torch.no_grad():
        ep = net(batch)
    assert np.array_equal(ep["sample_idxs"].cpu().numpy(), g["out:sample_idxs"])
    errs = {k: rel(ep[k], g[f"out:{k}"]) for k in ("estimation_cla", "vote_xyz", "center_xyz", "pred_search_bc", "estimation_boxes")}
    print("\n[bat_kitti_car.ckpt, 4-bit weights, eval] " + ", ".join(f"{k} {v:.1e}" for k, v in errs.items()))
    # seeds / votes / box clouds come before the vote ball-query; the proposals after it (a neighbour on the radius may flip)
    for k in ("estimation_cla", "vote_xyz", "center_xyz", "pred_search_bc"):
        assert errs[k] < 1e-4, (k, errs[k])
    assert errs["estimation_boxes"] < 1e-3
