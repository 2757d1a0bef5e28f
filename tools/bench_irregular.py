"""The irregular (non-GEMM) kernels of the step at the benchmark's own shapes (BAT_Car, B = 48): one launch set per kernel,
timed with CUDA events; run under `ncu --set full -k regex:...` for the digests in profiles/.
usage: python tools/bench_irregular.py [--batch 48] [--iters 10]"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from open3dsot_b200 import ops
from open3dsot_b200.datasets.synthetic import synthetic_siamese_batch


def timed(fn, iters):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=48)
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    B = a.batch
    b = synthetic_siamese_batch(B, 512, 1024, seed=20260924)
    search = b["search_points"].to(dev)
    tmpl = b["template_points"].to(dev)
    res = {}
    # FPS: search 1024 -> 512 (fps_kernel<128,8>), template 512 -> 256 (fps_kernel<128,4>)
    res["fps_search_1024_512"] = timed(lambda: ops.furthest_point_sampling(search, 512), a.iters)
    res["fps_template_512_256"] = timed(lambda: ops.furthest_point_sampling(tmpl, 256), a.iters)
    idx = ops.furthest_point_sampling(search, 512)
    xyz1 = torch.gather(search, 1, idx.long().unsqueeze(-1).expand(-1, -1, 3)).contiguous()      # SA1 output coordinates
    # SA2-search: 256 centres over 512 points, r 0.5, 32 samples, 128 feature channels
    f1 = torch.randn(B, 512, 128, device=dev)
    c2 = xyz1[:, :256].contiguous()
    res["ballquery_group_sa2"] = timed(lambda: ops.ballquery_group(xyz1, c2, f1, 0.5, 32), a.iters)
    g2, i2 = ops.ballquery_group(xyz1, c2, f1, 0.5, 32)
    gg2 = torch.randn_like(g2)
    res["ballquery_group_grad_sa2"] = timed(lambda: ops.ballquery_group_grad(gg2, i2, 512, 0.5, False), a.iters)
    # SA3-search: 128 centres over 256 points, r 0.7, 256 channels
    f2 = torch.randn(B, 256, 256, device=dev)
    c3 = c2[:, :128].contiguous()
    res["ballquery_group_sa3"] = timed(lambda: ops.ballquery_group(c2, c3, f2, 0.7, 32), a.iters)
    g3, i3 = ops.ballquery_group(c2, c3, f2, 0.7, 32)
    gg3 = torch.randn_like(g3)
    res["ballquery_group_grad_sa3"] = timed(lambda: ops.ballquery_group_grad(gg3, i3, 256, 0.7, False), a.iters)
    # SA1-search: 512 centres over 1024 points, r 0.3, no features
    res["ballquery_group_sa1"] = timed(lambda: ops.ballquery_group(search, xyz1, None, 0.3, 32), a.iters)
    # plain ball query (the `_ext` entry point)
    res["ball_query_sa1"] = timed(lambda: ops.ball_query(xyz1, search, 0.3, 32), a.iters)
    # FP module front end: 512 unknown points, 128 known, 256 channels
    kf = torch.randn(B, 128, 256, device=dev)
    res["three_nn_interpolate"] = timed(lambda: ops.three_nn_interpolate(xyz1, c3, kf), a.iters)
    out, ti, tw = ops.three_nn_interpolate(xyz1, c3, kf)
    go = torch.randn_like(out)
    res["three_nn_interpolate_grad"] = timed(lambda: ops.three_nn_interpolate_grad(go, ti, tw, 128), a.iters)
    print(json.dumps({k: round(v, 2) for k, v in res.items()}))


if __name__ == "__main__":
    main()
