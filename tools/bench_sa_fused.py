"""The inference set-abstraction layer at the tracker's shapes (BAT_Car, B = 1: search 1024 / template 512 points): the single
kernel (csrc/sa_fused.cu) next to the multi-kernel path, CUDA-event times per layer; run under
`ncu --set full -k regex:sa_fused_kernel` for the digest in profiles/.
usage: python tools/bench_sa_fused.py [--batch 1] [--iters 20]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from open3dsot_b200 import runtime
from open3dsot_b200.pointnet2.utils.pointnet2_modules import PointnetSAModule

SHAPES = [
    # name, N, C, mlp, npoint, radius
    ("sa1_search", 1024, 0, [0, 64, 64, 128], 512, 0.3),
    ("sa2_search", 512, 128, [128, 128, 128, 256], 256, 0.5),
    ("sa3_search", 256, 256, [256, 256, 256, 256], 128, 0.7),
    ("sa1_template", 512, 0, [0, 64, 64, 128], 256, 0.3),
    ("sa2_template", 256, 128, [128, 128, 128, 256], 128, 0.5),
    ("sa3_template", 128, 256, [256, 256, 256, 256], 64, 0.7),
]


def timed(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3  # us


def graph_timed(fn, iters):
    """device time of one call with the host out of the way: `iters` calls captured in one CUDA graph"""
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(iters):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--only-fused", action="store_true")
    ap.add_argument("--eager", action="store_true", help="no CUDA graph (for ncu)")
    a = ap.parse_args()
    torch.manual_seed(0)
    res = {}
    with torch.no_grad(), runtime.static_weights_scope():
        for name, N, C, mlp, npoint, radius in SHAPES:
            sa = PointnetSAModule(mlp=list(mlp), radius=radius, nsample=32, use_fps=False).cuda().eval()
            xyz = torch.rand(a.batch, N, 3, device="cuda") * 2.0
            feats = torch.randn(a.batch, C, N, device="cuda") if C else None
            run = lambda: sa(xyz, feats, npoint, True)
            runtime.set_sa_fused(True)
            res[name + "_fused_us"] = round((timed if a.eager else graph_timed)(run, a.iters), 2)
            if not a.only_fused:
                runtime.set_sa_fused(False)
                res[name + "_multi_us"] = round((timed if a.eager else graph_timed)(run, a.iters), 2)
                runtime.set_sa_fused(True)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
