"""Micro-benchmark of one MLP stack (forward, backward) on the fused kernels, per GEMM-core level.
usage: python tools/bench_stack.py [--shape sa3|sa2|sa1|bax] [--levels 0,1,3] [--iters 10] [--fwd-only]"""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from open3dsot_b200 import fused, runtime
from open3dsot_b200.pointnet2.utils import pytorch_utils as pt

SHAPES = {  # chans, P, S  (config 2, search branch, B = 48)
    "sa3": ([260, 256, 256, 256], 48 * 128 * 32, 32),
    "sa2": ([132, 128, 128, 256], 48 * 256 * 32, 32),
    "sa1": ([4, 64, 64, 128], 48 * 512 * 32, 32),
    "bax": ([268, 256, 256, 256], 48 * 128 * 4, 4),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shape", default="sa3")
    ap.add_argument("--levels", default="0,1,3")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--fwd-only", action="store_true")
    ap.add_argument("--profile", action="store_true", help="print per-kernel device times of one fwd+bwd (CUPTI)")
    ap.add_argument("--no-dx", action="store_true", help="the stack input needs no gradient (first SA level)")
    ap.add_argument("--force-mt", type=int, default=0)
    a = ap.parse_args()
    chans, P, S = SHAPES[a.shape]
    from open3dsot_b200 import _lib
    torch.manual_seed(0)
    mod = pt.SharedMLP(list(chans), bn=True).cuda().train()
    specs = fused.parse_stack(mod)
    x = torch.randn(P, chans[0], device="cuda")
    flops = sum(2 * P * chans[i] * chans[i + 1] for i in range(len(chans) - 1))
    # activation traffic every kernel of the stack has to move at least once (fp32), see DESIGN.md section 4
    nw = [((c + 3) // 4) * 4 for c in chans]
    fwd_fl = sum(nw[i] + nw[i + 1] for i in range(len(nw) - 1))
    bwd_fl = sum(2 * nw[i + 1] + 2 * nw[i] for i in range(len(nw) - 1)) + sum(2 * nw[i + 1] + nw[i] for i in range(len(nw) - 1))
    gb_f, gb_b = 4e-9 * P * fwd_fl, 4e-9 * P * bwd_fl
    _lib.check(_lib.lib().o3d_debug_set(0, a.force_mt), "o3d_debug_set")
    for lv in [int(v) for v in a.levels.split(",")]:
        runtime.set_tc(lv)
        xin = x.clone().requires_grad_(not a.fwd_only and not a.no_dx)
        for _ in range(2):
            out = fused.mlp_stack(xin, specs, S, True)
            if not a.fwd_only:
                out.sum().backward()
        torch.cuda.synchronize()
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        tf = tb = 0.0
        for _ in range(a.iters):
            e[0].record()
            out = fused.mlp_stack(xin, specs, S, True)
            e[1].record()
            if not a.fwd_only:
                go = torch.ones_like(out)
                out.backward(go)
            e[2].record()
            torch.cuda.synchronize()
            tf += e[0].elapsed_time(e[1])
            tb += e[1].elapsed_time(e[2])
        tf /= a.iters
        tb /= a.iters
        if a.profile:
            from torch.profiler import profile, ProfilerActivity
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(3):
                    out = fused.mlp_stack(xin, specs, S, True)
                    if not a.fwd_only:
                        out.backward(torch.ones_like(out))
                torch.cuda.synchronize()
            evs = [e for e in prof.events() if e.device_type.name == "CUDA"]
            n = len(evs) // 3
            for e in evs[2 * n:]:
                if e.device_time > 8:
                    print(f"    {e.device_time:9.1f} us  {e.name[:110]}")
        print(f"shape {a.shape} P={P} level {lv}: fwd {tf:.3f} ms ({flops / tf / 1e9:.1f} TFLOP/s, {gb_f / tf * 1e3:.0f} GB/s)"
              f"  bwd {tb:.3f} ms ({2 * flops / max(tb, 1e-9) / 1e9:.1f} TFLOP/s, {gb_b / max(tb, 1e-9) * 1e3:.0f} GB/s)", flush=True)


if __name__ == "__main__":
    main()
