"""bench.py — BAT-Car forward+backward(+Adam) template–search pairs/s on synthetic KITTI-Car-shaped pairs.

Contract (see the task brief): `python bench.py --gpus N --steps K --warmup W`; for N>1 the driver launches it under
torchrun, one rank per GPU.  Rank 0 prints ONE JSON line.

  value        whole-job pairs/s with the batch already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e          the same metric through the public engine call `TrainStep.step(batch)` (open3dsot_b200/engine.py: zero-grad,
               `model.training_step`, backward, gradient all-reduce, Adam) fed from PINNED HOST memory: H2D copy of the batch
               + the step + D2H read of the loss inside the timed region
  roofline     the dominant kernel timed alone, live, with CUDA events on its launch stream
  cpu_baseline the oracle (CPU restatement of the reference path) on a bounded sample of the same workload
  --impl reference   times only that CPU path (the reference ships no CPU/native code of its own: SURVEY.md facts 1-3)

A "step" = one optimisation step of BAT_Car.yaml at batch 48 per GPU (BASELINE.json configs[1]); weak scaling.
Timing hygiene: >= 3 warm-up steps, L2 flushed (256 MiB write) between timed steps and excluded from the timing,
clocks sampled with nvidia-smi during the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

CFG_FILE = os.path.join(ROOT, "cfgs", "BAT_Car.yaml")
WORKLOAD = "BAT_Car.yaml train step (fwd+bwd+Adam), synthetic KITTI-Car pairs, template 512 / search 1024 pts, batch 48/GPU"
METRIC = "template-search pairs/sec, BAT-Car fwd+bwd"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=48, help="pairs per GPU (BAT_Car.yaml config 2: 48)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-batch", type=int, default=2, help="pairs per CPU-baseline step (bounded sample)")
    ap.add_argument("--cpu-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--fused", type=int, default=None, help="override O3D_FUSED (1 = fused kernels, 0 = composed)")
    ap.add_argument("--tc", type=int, default=None, help="override O3D_TC (0 = CUDA cores, 1 = tcgen05 fwd+dgrad, 3 = + wgrad)")
    ap.add_argument("--no-graph", action="store_true", help="do not capture the step into a CUDA graph")
    ap.add_argument("--track", action="store_true", help="secondary mode: B=1 tracking frames/s (SURVEY.md 8f rank 2)")
    ap.add_argument("--sampler", action="store_true", help="secondary mode: on-device training-batch construction (8f rank 3)")
    ap.add_argument("--track-points", type=int, default=60000, help="points per synthetic scan in --track mode")
    ap.add_argument("--kernel-table", default=None, metavar="FILE",
                    help="also write the per-kernel device times of 3 steps (CUPTI, no replay, warm caches) to FILE")
    ap.add_argument("--ncu-step", action="store_true", help="run ONE eager step between cudaProfilerStart/Stop and exit (for "
                    "`ncu --profile-from-start off --metrics dram__bytes_read.sum,dram__bytes_write.sum`: DRAM bytes per step)")
    ap.add_argument("--cfg", default=None, help="other config to exercise (P2B_Car.yaml, M2_track_kitti.yaml, ...): a parity / "
                    "plumbing run of BASELINE.json configs[2..4], NOT the headline metric")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last device-timed step computed (loss, gradients, updated "
                         "parameters, BatchNorm running statistics) as DIR/<name>.npy; that step starts from the model's initial "
                         "state, so that two runs or builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.track or args.sampler):
        ap.error("--dump-outputs writes the training step's outputs; it does not apply to --impl reference, --track or --sampler")
    return args


# ----------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.lower() == "active"})
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w_max": max(pw) if pw else None}


# ----------------------------------------------------------------------------------------------- CPU baseline
def cpu_baseline(batch_pairs, steps, seed=20260924):
    """The oracle's BAT training step (forward + backward; no optimizer) on the host cores."""
    from open3dsot_b200.config import load_config
    from open3dsot_b200.datasets.synthetic import synthetic_siamese_batch
    from open3dsot_b200.models import get_model
    from oracle import modules as om
    # torch's CPU kernels stop scaling (and then slow down) on these small per-pair tensors: cap the thread pool
    cores = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    cfg = load_config(CFG_FILE)
    torch.manual_seed(0)
    net = get_model(cfg.net_model)(cfg)
    pnames = [k for k, _ in net.named_parameters()]
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    for k in pnames:
        sd[k].requires_grad_(True)
    batch = synthetic_siamese_batch(batch_pairs, cfg.template_size, cfg.search_size, seed=seed)
    times = []
    for i in range(steps + 1):
        for k in pnames:
            sd[k].grad = None
        t0 = time.perf_counter()
        loss, _, _ = om.bat_training_loss(sd, cfg, {k: v.clone() for k, v in batch.items()})
        loss.backward()
        dt = time.perf_counter() - t0
        if i > 0:  # first iteration = warm-up
            times.append(dt)
    times.sort()
    med = times[len(times) // 2]
    return {"value": batch_pairs / med, "unit": "pairs/s", "cores": cores, "kind": "port",
            "sample": f"oracle BAT fwd+bwd, batch {batch_pairs} pairs of 512/1024 pts, median of {steps} steps after 1 warm-up",
            "ms_per_step": med * 1e3}


def track_cpu_baseline(cfg, seq, frames):
    """The reference's frame as it runs on the host: numpy crop / resample / BoxCloud / box update (oracle/tracking_ref.py)
    around the oracle's eval-mode forward on the CPU (oracle/modules.py)."""
    import numpy as np
    from open3dsot_b200.models import get_model
    from oracle import modules as om
    from oracle import tracking_ref as tr
    cores = min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    net = get_model(cfg.net_model)(cfg).eval()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    if cfg.net_model.lower() not in ("bat", "p2b"):
        return None                                  # the oracle restates the matching models' forward only
    fwd = om.bat_forward if cfg.net_model.lower() == "bat" else om.p2b_forward
    boxes = [tr.Box(seq[0]["3d_bbox"].center, seq[0]["3d_bbox"].wlh, seq[0]["3d_bbox"].rotation_matrix)]
    times = []
    for i in range(1, min(frames, len(seq))):
        t0 = time.perf_counter()
        ref = boxes[-1]
        search = tr.generate_subwindow(seq[i]["pc"].points.astype(np.float64), ref, cfg.search_bb_scale, cfg.search_bb_offset)
        tmpl, canon = tr.get_model([seq[0]["pc"].points.astype(np.float64), seq[i - 1]["pc"].points.astype(np.float64)],
                                   [boxes[0], ref], offset=cfg.model_bb_offset, scale=cfg.model_bb_scale)
        tp, _ = tr.regularize_pc(tmpl.T, cfg.template_size, seed=1)
        sp, _ = tr.regularize_pc(search.T, cfg.search_size, seed=1)
        batch = {"template_points": torch.tensor(tp, dtype=torch.float32)[None], "search_points": torch.tensor(sp, dtype=torch.float32)[None]}
        if cfg.net_model.lower() == "bat":
            batch["points2cc_dist_t"] = torch.tensor(tr.get_point_to_box_distance(tp, canon), dtype=torch.float32)[None]
        with torch.no_grad():
            out = fwd(sd, cfg, batch, False)
        est = out["estimation_boxes"][0].numpy()
        est = est[est[:, 4].argmax(), :4]
        boxes.append(tr.get_offset_bb(ref, est, degrees=cfg.degrees, use_z=cfg.use_z, limit_box=cfg.limit_box))
        if i > 1:
            times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return {"value": 1.0 / med, "unit": "frames/s", "cores": cores, "kind": "port",
            "sample": f"numpy frame geometry + oracle {cfg.net_model} eval forward, B=1, median of {len(times)} frames", "ms_per_frame": med * 1e3}


def run_track(args):
    """Secondary mode (SURVEY.md 8f rank 2): B=1 tracking frames/s on a synthetic tracklet — the reference-shaped host loop,
    the fixed-shape device frame, and the same frame replayed from one CUDA graph; CPU baseline beside it."""
    from open3dsot_b200.config import load_config
    from open3dsot_b200.datasets.synthetic import synthetic_sequence
    from open3dsot_b200.models import get_model
    from open3dsot_b200.tracking.device_tracker import DeviceTracker
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = load_config(CFG_FILE if args.cfg is None else os.path.join(ROOT, "cfgs", args.cfg), {"up_axis": [0, 0, 1]})
    torch.manual_seed(0)
    if os.environ.get("O3D_FORCE_MT"):
        from open3dsot_b200 import _lib
        _lib.lib().o3d_debug_set(0, int(os.environ["O3D_FORCE_MT"]))
    net = get_model(cfg.net_model)(cfg).to(dev).eval()
    frames, npts = max(args.steps + args.warmup + 1, 12), args.track_points
    seq = synthetic_sequence(n_frames=frames, n_points=npts, seed=20260924)
    pts = [torch.tensor(f["pc"].points.T.copy(), device=dev) for f in seq]
    w = max(args.warmup, 3)
    net.evaluate_one_sequence(seq[: w + 1])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    net.evaluate_one_sequence(seq)
    torch.cuda.synchronize()
    res = {"host_loop_fps": (frames - 1) / (time.perf_counter() - t0)}
    sampler = ClockSampler(0)
    sampler.start()
    for name, graph in (("device_eager", False), ("device_graph", True)):
        trk = DeviceTracker(net, max_points=npts, use_graph=graph)
        trk.reset(pts[0], seq[0]["3d_bbox"].to_tensor(dev))
        for i in range(1, w + 1):
            trk.step(pts[i])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for i in range(w + 1, frames):
            trk.step(pts[i])
        e1.record()
        torch.cuda.synchronize()
        n = frames - w - 1
        res[name + "_fps"] = n / max(time.perf_counter() - t0, e0.elapsed_time(e1) * 1e-3)
        res[name + "_ms_device"] = e0.elapsed_time(e1) / n
    clocks = sampler.stop()
    if args.kernel_table:                       # per-kernel device time of eager device frames (CUPTI)
        from torch.profiler import ProfilerActivity, profile
        trk = DeviceTracker(net, max_points=npts, use_graph=False)
        trk.reset(pts[0], seq[0]["3d_bbox"].to_tensor(dev))
        for i in range(1, 4):
            trk.step(pts[i])
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(4, 7):
                trk.step(pts[i])
            torch.cuda.synchronize()
        agg = {}
        for e in prof.events():
            if e.device_type.name == "CUDA":
                a = agg.setdefault(e.name, [0, 0.0])
                a[0] += 1
                a[1] += e.device_time
        tot = sum(v[1] for v in agg.values())
        with open(args.kernel_table, "w") as f:
            f.write(f"# CUPTI kernel activity, 3 eager tracking frames; {sum(v[0] for v in agg.values()) / 3:.0f} launches, {tot / 3:.1f} us of kernel time per frame\n")
            for name, (n, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                f.write(f"{100 * us / tot:7.2f}% {us / 3:9.1f} us {n / 3:7.1f}  {name[:140]}\n")
    cb = None if args.no_cpu_baseline else track_cpu_baseline(cfg, seq, 8)
    print(json.dumps({"metric": f"tracking frames/sec, {cfg.net_model} B=1 (crop + resample + network + box update per frame)",
                      "value": res["device_graph_fps"], "unit": "frames/s", "n_gpus": 1, "steps": frames - w - 1, "warmup": w,
                      "ms_per_step": res["device_graph_ms_device"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                      "dtype": "f32", "data": "synthetic",
                      "config": {"workload": f"{os.path.basename(args.cfg or CFG_FILE)} tracking inference, synthetic tracklet, "
                                             f"{npts} points per scan, template {cfg.template_size} / search {cfg.search_size}",
                                 "l2": "every frame reads a different scan", "cuda_graph": True},
                      "clocks": clocks, **res, "cpu_baseline": cb}))


def sampler_cpu_baseline(cfg, tracklets, n_pairs=24):
    """The reference's per-pair batch construction on one host core: the numpy restatement of siamese_processing."""
    import numpy as np
    from oracle import tracking_ref as tr
    frames = [f for t in tracklets for f in t]
    starts, k = [], 0
    for t in tracklets:
        starts += [k] * len(t)
        k += len(t)
    rng = np.random.default_rng(0)
    deg = 5.0 if cfg.degrees else np.deg2rad(5.0)

    def fr(f):
        b = f["3d_bbox"]
        return f["pc"].points.astype(np.float64), tr.Box(b.center, b.wlh, b.rotation_matrix)
    t0 = time.perf_counter()
    for i in range(n_pairs):
        k = int(rng.integers(len(frames)))
        prev = max(k - 1, starts[k])
        tr.siamese_processing(fr(frames[starts[k]]), fr(frames[prev]), fr(frames[k]), i % cfg.get("num_candidates", 1), cfg,
                              rng.uniform(-0.3, 0.3, 3), rng.normal(size=3) * np.sqrt([1.0, 1.0, deg]))
    dt = time.perf_counter() - t0
    return {"value": n_pairs / dt, "unit": "pairs/s", "cores": 1, "kind": "port",
            "sample": f"numpy siamese_processing, {n_pairs} pairs, scans of {frames[0]['pc'].points.shape[1]} points, one core "
                      f"(the reference runs one such worker per DataLoader process, 10 per GPU)", "ms_per_pair": dt / n_pairs * 1e3}


def run_sampler(args):
    """Secondary mode (SURVEY.md 8f rank 3): training batches built on the device, alone and feeding the training step."""
    from open3dsot_b200.config import load_config
    from open3dsot_b200.datasets.device_sampler import DeviceSiameseSampler
    from open3dsot_b200.datasets.synthetic import synthetic_sequence
    from open3dsot_b200.engine import TrainStep
    from open3dsot_b200.models import get_model
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = load_config(CFG_FILE if args.cfg is None else os.path.join(ROOT, "cfgs", args.cfg), {"batch_size": args.batch})
    tracklets = [synthetic_sequence(n_frames=8, n_points=args.track_points, seed=20260924 + i) for i in range(6)]
    smp = DeviceSiameseSampler(tracklets, cfg, dev, seed=1)
    w, n = max(args.warmup, 3), args.steps
    for _ in range(w):
        batch, valid = smp.next_batch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        batch, valid = smp.next_batch()
    e1.record()
    torch.cuda.synchronize()
    ms_sampler = e0.elapsed_time(e1) / n
    torch.manual_seed(0)
    net = get_model(cfg.net_model)(cfg).to(dev).train()
    eng = TrainStep(net, lr=cfg.lr, weight_decay=cfg.wd, use_graph=True, warmup=2)
    for _ in range(w + 3):
        eng.step(smp.next_batch()[0])
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    e0.record()
    for _ in range(n):
        loss = eng.step(smp.next_batch()[0])
    e1.record()
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / n
    clocks = sampler.stop()
    cb = None if args.no_cpu_baseline else sampler_cpu_baseline(cfg, tracklets)
    print(json.dumps({"metric": f"training pairs/sec with batches constructed on the device, {cfg.net_model}", "value": args.batch / ms_step * 1e3,
                      "unit": "pairs/s", "n_gpus": 1, "steps": n, "warmup": w, "ms_per_step": ms_step, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                      "config": {"workload": f"{os.path.basename(args.cfg or CFG_FILE)} train step fed by DeviceSiameseSampler: "
                                             f"6 synthetic tracklets x 8 scans of {args.track_points} points resident on the device, "
                                             f"batch {args.batch}", "l2": "every step builds a new batch from different frames"},
                      "clocks": clocks, "sampler_ms_per_batch": ms_sampler, "sampler_pairs_per_s": args.batch / ms_sampler * 1e3,
                      "last_loss": float(loss), "cpu_baseline": cb}))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # bounded sample: one "step" = the oracle's BAT forward+backward on `cpu_batch` pairs; at most ~150 s in total
    t0 = time.perf_counter()
    probe = cpu_baseline(1, 1)
    per_pair = probe["ms_per_step"] * 1e-3
    budget = 150.0 - (time.perf_counter() - t0)
    steps = max(1, min(args.steps, int(budget / max(per_pair * args.cpu_batch, 1e-3)) - 1))
    cb = cpu_baseline(args.cpu_batch, steps)
    cb["sample"] += f" ({steps} of the requested {args.steps} steps fit the time box)"
    line = {"metric": METRIC, "value": cb["value"], "unit": "pairs/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": WORKLOAD, "note": "CPU path = oracle port (the reference has no CPU/native code)"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------- our arm
def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def gather_roofline(dev, batch_pairs):
    """The irregular kernels of the lifted set-abstraction layer, SA2-search shape at the benchmark batch (48 clouds, 256 centres x 32
    neighbours over 512 points, 128 channels), each timed alone through the C ABI with CUDA events:
      ball_query+relative coordinates (o3d_ballquery_group, C = 0)   writes idx + (dx, dy, dz, 0) per position
      gather pass (o3d_lift_stats)    row indices + BatchNorm statistics of Y0 = Z[idx] + s.u (Z is L2-resident)
      scatter pass (o3d_lift_scatter) dY0 = a*g + b + c*Y0 accumulated into dZ[idx] (vector REDs), du
    All three are HBM-side kernels: achieved = algorithmic bytes / time against the measured copy bandwidth."""
    import ctypes
    from open3dsot_b200 import _lib, ops
    from open3dsot_b200.datasets.synthetic import synthetic_siamese_batch
    L = _lib.lib()
    B, N, M, S, C0 = max(batch_pairs, 48), 512, 256, 32, 128
    b = synthetic_siamese_batch(min(B, 64), 512, 1024, seed=1)
    xyz = b["search_points"][:, :N].contiguous().repeat((B + 63) // 64, 1, 1)[:B].contiguous().to(dev)
    new_xyz = xyz[:, :M].contiguous()
    P = B * M * S
    st = torch.cuda.current_stream().cuda_stream
    rel, idx = ops.ballquery_group(xyz, new_xyz, None, 0.5, S, False)
    z = torch.randn(B * N, C0, device=dev)
    u = torch.randn(4, C0, device=dev) * 0.3
    g = torch.randn(P, C0, device=dev) * 1e-3
    co = [torch.rand(C0, device=dev) + 0.5, torch.randn(C0, device=dev) * 1e-4, torch.randn(C0, device=dev) * 1e-4]
    gidx = torch.empty(P, dtype=torch.int32, device=dev)
    stat = torch.zeros(2 * C0, dtype=torch.float64, device=dev)
    dz, du = torch.zeros_like(z), torch.zeros_like(u)
    lf = _lib.LiftDesc()
    lf.z, lf.ldz, lf.ridx, lf.ridx_mod, lf.rows_per_cloud, lf.pos_per_cloud, lf.grp = z.data_ptr(), C0, idx.data_ptr(), 0, N, M * S, S
    lf.s, lf.u, lf.d_z, lf.d_s, lf.d_u = rel.data_ptr(), u.data_ptr(), dz.data_ptr(), None, du.data_ptr()
    runs = {
        "ballquery_group_kernel (ball query + relative coordinates)":
            (lambda: ops.ballquery_group(xyz, new_xyz, None, 0.5, S, False), xyz.numel() * 4 + new_xyz.numel() * 4 + P * 4 + P * 16),
        "lift_stats_kernel (gather pass: indices + BN statistics)":
            (lambda: _lib.check(L.o3d_lift_stats(ctypes.byref(lf), P, C0, gidx.data_ptr(), None, stat.data_ptr(), stat.data_ptr() + 8 * C0, st),
                                "o3d_lift_stats"), P * (4 + 4 + 16) + z.numel() * 4),
        "lift_scatter_kernel (scatter pass: dY0 -> dZ, du)":
            (lambda: _lib.check(L.o3d_lift_scatter(ctypes.byref(lf), P, C0, gidx.data_ptr(), None, g.data_ptr(), C0, co[0].data_ptr(),
                                                   co[1].data_ptr(), co[2].data_ptr(), st), "o3d_lift_scatter"),
             g.numel() * 4 + P * (4 + 16) + 2 * z.numel() * 4)}
    peaks, how = measured_peaks()
    traffic = {}
    try:
        with open(os.path.join(ROOT, "profiles", "r2_irregular_traffic.json")) as f:
            traffic = json.load(f)
    except (OSError, ValueError):
        pass
    out = []
    for name, (fn, nbytes) in runs.items():
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        n = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        ach = nbytes / (ms * 1e-3) / 1e9
        out.append({"kernel": name + f", SA2-search shape, B={B}: P={P}, {C0} channels", "bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"],
                    "peak_source": how + " (MEASURED_PEAKS.json hbm_gbs, burst copy)", "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                    "traffic": traffic.get(name.split(" ")[0]), "ms_per_launch": ms, "algorithmic_bytes_per_launch": nbytes})
    return out


def ncu_traffic(P, key="fwd"):
    """DRAM bytes per launch of a roofline kernel as ncu measured them (dram__bytes_read.sum + dram__bytes_write.sum of
    one `--set full` capture of the same kernel and shape, committed under profiles/); None when the shape differs."""
    path = os.path.join(ROOT, "profiles", "r1_roofline_traffic.json")
    try:
        with open(path) as f:
            rec = json.load(f)[key]
        return float(rec["dram_bytes_per_launch"]) if f"P={P}," in rec["shape"] else None
    except (OSError, ValueError, KeyError):
        return None


def roofline_probe(dev, batch_pairs):
    """The dominant kernel family of the step — the point-wise MLP GEMM (pw_tc_kernel, forward, SA3-search layer:
    196608 positions x 256 -> 256 channels) — timed alone with CUDA events on its stream through the C ABI.
    It is bounded by BOTH roofs at this shape (arithmetic intensity 64 FLOP/B of fp32 activations, 3 tensor passes):
      tensor : algorithmic 2*P*K*N FLOP vs measured bf16 peak / 2 (TF32 rate) / 3 (3xTF32 passes)
      hbm    : algorithmic bytes (X read + Y written once, fp32) vs the measured copy bandwidth
    `frac` is reported against the TIGHTER of the two (the larger time bound)."""
    import ctypes
    from open3dsot_b200 import _lib
    L = _lib.lib()
    P, K, N = max(batch_pairs, 48) * 128 * 32, 256, 256
    x = torch.randn(P, K, device=dev)
    w = torch.randn(N, K, device=dev) * 0.05
    y = torch.empty(P, N, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    tiles = torch.empty(int(L.o3d_pw_tc_wtile_bytes(N, K)), dtype=torch.uint8, device=dev)
    _lib.check(L.o3d_pw_tc_pretile(w.data_ptr(), K, N, K, tiles.data_ptr(), st), "pretile")
    stat = torch.zeros(2 * N, dtype=torch.float64, device=dev)

    def launch():
        _lib.check(L.o3d_pw_fwd_tc(x.data_ptr(), K, None, None, 0, tiles.data_ptr(), None, P, K, N, y.data_ptr(), N,
                                   stat.data_ptr(), stat.data_ptr() + 8 * N, 0, None, None, None, N, st), "o3d_pw_fwd_tc")
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    n = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    peaks, how = measured_peaks()
    flops = 2.0 * P * K * N
    alg_bytes = 4.0 * P * (K + N)                      # 403 MB per launch: larger than the 126 MB L2
    tf = flops / (ms * 1e-3) / 1e12
    gbs = alg_bytes / (ms * 1e-3) / 1e9
    tensor_peak = peaks["bf16_tflops"] / 2.0 / 3.0      # TF32 runs at half the bf16 rate; 3 passes per product
    t_tensor, t_hbm = flops / (tensor_peak * 1e12), alg_bytes / (peaks["hbm_gbs"] * 1e9)
    bound = "tensor" if t_tensor >= t_hbm else "hbm"
    return {"kernel": "pw_tc_kernel<2,TcAct,TcFwdEpi> (SA3-search layer: P=%d, K=256, N=256, 3xTF32)" % P,
            "bound": bound, "achieved": tf if bound == "tensor" else gbs,
            "peak": tensor_peak if bound == "tensor" else peaks["hbm_gbs"],
            "unit": "TFLOP/s" if bound == "tensor" else "GB/s",
            "frac": (tf / tensor_peak) if bound == "tensor" else (gbs / peaks["hbm_gbs"]),
            "peak_source": how + " MEASURED_PEAKS.json: bf16_tflops/2/3 (TF32 rate, three passes) and hbm_gbs (burst)",
            "traffic": ncu_traffic(P), "ms_per_launch": ms, "algorithmic_flops_per_launch": flops,
            "algorithmic_bytes_per_launch": alg_bytes, "achieved_tflops_fp32_equiv": tf, "achieved_gbs": gbs,
            "frac_of_tensor_roof": tf / tensor_peak, "frac_of_hbm_roof": gbs / peaks["hbm_gbs"]}


def roofline_backward_probe(dev, batch_pairs):
    """The two backward GEMMs on the SA2-search shape (393216 positions, 128 -> 128 channels, BN + ReLU on both sides),
    each timed alone through the C ABI.  At 128 channels both are HBM-bound: dgrad reads g, y and the previous layer's raw
    output (for the ReLU mask) and writes the input gradient; wgrad reads g, y and the layer input."""
    from open3dsot_b200 import _lib
    L = _lib.lib()
    P, C = max(batch_pairs, 48) * 256 * 32, 128
    g = torch.randn(P, C, device=dev) * 1e-3
    y = torch.randn(P, C, device=dev)
    yprev = torch.randn(P, C, device=dev)
    out = torch.empty(P, C, device=dev)
    w = torch.randn(C, C, device=dev) * 0.05
    a, b, cc = (torch.rand(C, device=dev) + 0.5), torch.randn(C, device=dev) * 1e-4, torch.randn(C, device=dev) * 1e-4
    sc, sh = (torch.rand(C, device=dev) + 0.5), torch.randn(C, device=dev) * 0.1
    stat = torch.zeros(2 * C, dtype=torch.float64, device=dev)
    dw = torch.zeros(C, C, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    wt = w.t().contiguous()
    tiles = torch.empty(int(L.o3d_pw_tc_wtile_bytes(C, C)), dtype=torch.uint8, device=dev)
    _lib.check(L.o3d_pw_tc_pretile(wt.data_ptr(), C, C, C, tiles.data_ptr(), st), "pretile")

    def dgrad():
        _lib.check(L.o3d_pw_dgrad_tc(g.data_ptr(), C, y.data_ptr(), C, a.data_ptr(), b.data_ptr(), cc.data_ptr(), None, None, 0, 0,
                                     tiles.data_ptr(), P, C, C, out.data_ptr(), C, yprev.data_ptr(), C, sc.data_ptr(),
                                     sh.data_ptr(), 1, stat.data_ptr(), stat.data_ptr() + 8 * C, st), "o3d_pw_dgrad_tc")

    part = torch.empty(int(L.o3d_pw_wgrad_tc2_workspace_floats()), device=dev)

    def wgrad():      # the split-K kernel + ordered reduction the step uses for every tensor-core weight gradient (deterministic)
        dw.zero_()
        _lib.check(L.o3d_pw_wgrad_tc2(g.data_ptr(), C, y.data_ptr(), C, a.data_ptr(), b.data_ptr(), cc.data_ptr(), None, None, 0, 0,
                                      yprev.data_ptr(), C, sc.data_ptr(), sh.data_ptr(), 1, P, C, C, dw.data_ptr(), C, part.data_ptr(),
                                      part.numel(), st), "o3d_pw_wgrad_tc2")
    peaks, how = measured_peaks()
    res = []
    for name, fn, nbytes, key in (("pw_tc_kernel<1,TcDy,TcDgradEpi<128>> (dgrad)", dgrad, 4.0 * P * C * 4, "dgrad"),
                                  ("pw_wgrad_tc2_kernel<1,1> + wgrad_reduce_kernel (wgrad, split-K, deterministic)", wgrad, 4.0 * P * C * 3, "wgrad")):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        n = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        gbs = nbytes / (ms * 1e-3) / 1e9
        res.append({"kernel": name + ", SA2-search layer: P=%d, 128 -> 128 channels" % P, "bound": "hbm", "achieved": gbs,
                    "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"], "traffic": ncu_traffic(P, key),
                    "ms_per_launch": ms, "algorithmic_bytes_per_launch": nbytes,
                    "peak_source": how + " (MEASURED_PEAKS.json hbm_gbs, burst copy)"})
    return res


def kernel_table(eng, batches, path, steps=3):
    """Per-kernel device time of `steps` training steps as CUPTI records them (activity tracing: no replay, no
    serialisation beyond the step's own stream order).  Not a bench value: tracing adds a little launch overhead."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(steps):
            eng.step(batches[i % len(batches)])
        torch.cuda.synchronize()
    agg = {}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        a = agg.setdefault(e.name, [0, 0.0])
        a[0] += 1
        a[1] += e.device_time
    total = sum(v[1] for v in agg.values())
    with open(path, "w") as f:
        f.write(f"# CUPTI kernel activity, {steps} steps; total kernel time {total / steps / 1e3:.3f} ms per step\n")
        f.write("#  share   ms/step  launches/step  kernel\n")
        for name, (n, us) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write(f"{100 * us / total:7.2f}% {us / steps / 1e3:9.3f} {n / steps:8.1f}  {name[:150]}\n")


def train_state(eng):
    """What a training step reads besides its batch: parameters, Adam moments and step counter, BatchNorm buffers."""
    return [eng.flat.flat, eng.opt.exp_avg, eng.opt.exp_avg_sq, eng.opt.state, *eng.model.buffers()]


def step_outputs(eng, loss):
    """Device copies of what a training step computes: the loss `TrainStep.step` returns, the gradient of every parameter and
    the parameters after the Adam update (each one flat float32 array in `model.parameters()` order, as the engine keeps
    them), and the BatchNorm running statistics the step leaves in the model.
    The backward scatters with float atomics, so gradients repeat from run to run only to rounding; compare with a tolerance
    scaled to each array (a few gradients are 0 in exact arithmetic, e.g. of a bias feeding BatchNorm, and hold only rounding,
    which Adam's lr * g / (|g| + eps) carries into the parameters as about lr / eps times that rounding).  Two runs of
    BAT_Car.yaml on one B200 (1,000 W): loss and BatchNorm statistics bitwise equal; gradients 6.0e-7 apart normwise (at
    most 2.2e-6 in an element, largest |g| 0.93); parameters 9.0e-7 normwise (at most 3.3e-5 in an element, largest 3.2)."""
    out = {"loss": loss.reshape(1), "gradients": eng.flat.grad, "parameters": eng.flat.flat}
    for k, b in eng.model.named_buffers():
        out["buffer." + k] = b
    return {k: v.detach().clone() for k, v in out.items()}


def write_outputs(outputs, out_dir, limit_bytes=64 << 20):
    """DIR/<name>.npy for every output, float32 (integer counters as float64)."""
    import numpy as np
    arrays = {k: v.cpu().numpy() for k, v in outputs.items()}
    arrays = {k: v.astype(np.float32 if v.dtype.kind == "f" else np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= limit_bytes, f"--dump-outputs: {total} bytes exceed the {limit_bytes}-byte limit"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_ours(args):
    from open3dsot_b200 import ddp, ops, runtime
    from open3dsot_b200.config import load_config
    from open3dsot_b200.datasets.synthetic import synthetic_siamese_batch
    from open3dsot_b200.models import get_model
    import torch.distributed as dist

    if args.fused is not None:
        runtime.set_fused(bool(args.fused))
    if args.tc is not None:
        runtime.set_tc(args.tc)
    rank, world, local = ddp.init_distributed()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback for the product path)"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    numa_cpus = ddp.pin_to_gpu_numa_node(local) if world > 1 else 0     # ranks stay on the socket next to their GPU
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    cfg_file = CFG_FILE if args.cfg is None else os.path.join(ROOT, "cfgs", args.cfg)
    cfg = load_config(cfg_file, {"batch_size": args.batch})
    is_motion = cfg.net_model.lower() == "m2track"
    if args.cfg is not None and "PEDESTRIAN_NUSCENES" in args.cfg:
        cfg.template_size, cfg.search_size = 256, 512          # BASELINE.json configs[4] override (SURVEY.md §8d C5)
    torch.manual_seed(0)
    net = get_model(cfg.net_model)(cfg).to(dev).train()
    from open3dsot_b200.engine import TrainStep
    eng = TrainStep(net, lr=cfg.lr, weight_decay=cfg.wd, use_graph=not args.no_graph, warmup=2)
    # --dump-outputs: the last device-timed step restarts from this initial state (restored outside its timed window).  The
    # kernels' float atomics round differently from run to run and training amplifies that over the ~30 earlier steps, so
    # only a step from a known state can be compared between runs and builds.
    initial_state = [t.clone() for t in train_state(eng)] if args.dump_outputs else None

    # distinct host batches (pinned), one device-resident copy of each
    n_batches = 4
    if is_motion:
        from open3dsot_b200.datasets.synthetic import synthetic_motion_batch
        host = [{k: v.pin_memory() for k, v in synthetic_motion_batch(args.batch, cfg.point_sample_size,
                                                                      seed=20260924 + rank * 100 + i).items()}
                for i in range(n_batches)]
    else:
        host = [synthetic_siamese_batch(args.batch, cfg.template_size, cfg.search_size, seed=20260924 + rank * 100 + i,
                                        box_aware=getattr(cfg, "box_aware", False), pin_memory=True)
                for i in range(n_batches)]
    # every batch is ONE slab (engine.BatchSlab): a step's inputs move with a single copy per hop
    from open3dsot_b200.engine import BatchSlab
    host_slabs = [BatchSlab.like(b, "cpu", pin=True).load(b) for b in host]
    resident = [host_slabs[0].sibling(dev) for _ in host]
    for r, hs in zip(resident, host_slabs):
        r.buf.copy_(hs.buf)
    h2d_bytes = host_slabs[0].nbytes
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ops.LAUNCHES = 0
    eng.step(resident[0])                                       # eager: counts the kernels of one step
    launches_per_step = ops.LAUNCHES
    for i in range(max(args.warmup, 3) + 3):                    # includes graph capture when enabled
        eng.step(resident[i % n_batches])
    barrier()
    if args.ncu_step:
        flush.fill_(1.0)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        eng.step(resident[0])
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return

    # ---- device-resident timing
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        if initial_state is not None and i == args.steps - 1:
            for t, t0 in zip(train_state(eng), initial_state):  # not timed; before the flush, so this step starts cold too
                t.copy_(t0)
        flush.fill_(float(i))                                   # evict L2; not timed
        evs[i][0].record()
        loss = eng.step(resident[i % n_batches])
        evs[i][1].record()
    barrier()
    wall = time.perf_counter() - t_wall0
    outputs = step_outputs(eng, loss) if args.dump_outputs else None
    launches = launches_per_step * args.steps
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([dev_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms = float(t.item())

    # ---- end-to-end timing through the public engine call, fed from PINNED HOST memory: every step copies its batch
    # host->device (on a copy stream, overlapping the previous step) and its loss device->host (async into pinned memory);
    # the host synchronises once at the end, as a training loop that logs asynchronously does
    barrier()
    copy_stream = torch.cuda.Stream()
    staging = [host_slabs[0].sibling(dev) for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    loss_host = torch.zeros(args.steps, dtype=torch.float32).pin_memory()
    main = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()

    def upload(i):
        slot = i % 2
        with torch.cuda.stream(copy_stream):
            if i >= 2:
                copy_stream.wait_event(consumed[slot])
            staging[slot].buf.copy_(host_slabs[i % n_batches].buf, non_blocking=True)   # ONE H2D copy per step
            ready[slot].record(copy_stream)

    upload(0)
    for i in range(args.steps):
        if i + 1 < args.steps:
            upload(i + 1)
        slot = i % 2
        main.wait_event(ready[slot])
        loss = eng.step(staging[slot])
        consumed[slot].record(main)
        loss_host[i:i + 1].copy_(loss.reshape(1), non_blocking=True)      # D2H read of the step's loss (4 bytes)
    e1.record()
    torch.cuda.synchronize()          # this rank's own work only: no collective inside the timed region besides the step's
    e2e_s = max(time.perf_counter() - t0, e0.elapsed_time(e1) * 1e-3)
    last = float(loss_host[-1])
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                          # max over ranks, taken after the timed region
    e2e_s = float(t.item())
    clocks = sampler.stop() if rank == 0 else None

    if rank != 0:
        _shutdown(eng, world)
        return
    if outputs is not None:
        write_outputs(outputs, args.dump_outputs)
    if args.kernel_table:
        kernel_table(eng, resident, args.kernel_table)
    roof = roofline_probe(dev, args.batch)
    roof_gather = gather_roofline(dev, args.batch)
    roof_bwd = roofline_backward_probe(dev, args.batch)
    cb = None
    if world == 1 and not args.no_cpu_baseline:
        cb = cpu_baseline(args.cpu_batch, args.cpu_steps)
    pairs = args.batch * world * args.steps
    workload = WORKLOAD if args.cfg is None else f"{args.cfg} train step, synthetic batch {args.batch}/GPU (not the headline config)"
    line = {"metric": METRIC if args.cfg is None else "samples/sec, " + args.cfg, "value": pairs / (dev_ms * 1e-3), "unit": "pairs/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "global_batch": args.batch * world, "parallelism": f"dp{world}",
                       "mode": "fused" if runtime.fused_enabled() else "composed",
                       "gemm_core": {0: "cuda-core-fp32", 1: "tcgen05-3xTF32 fwd+dgrad, cuda-core wgrad",
                                     3: "tcgen05-3xTF32 fwd+dgrad+wgrad"}.get(runtime.tc_level(), str(runtime.tc_level())),
                       "cuda_graph": not args.no_graph,
                       "l2": "256 MiB flush write between timed steps, excluded from timing",
                       "optimizer": "Adam(0.5,0.999), one kernel over the flat parameter bucket", "last_loss": last,
                       "ddp": None if world == 1 else {"allreduce_in_graph": bool(eng.graph_has_update) if eng.graph is not None else False,
                                                       "numa_cpus_per_rank": numa_cpus},
                       "first_layer": "lifted (no grouped tensor)" if runtime.lift_enabled() else "materialised grouping"},
            "clocks": clocks, "gpu_launches": launches, "wall_s_timed_region": wall,
            "e2e": {"value": pairs / e2e_s, "unit": "pairs/s", "h2d_bytes_per_step": h2d_bytes,
                    "d2h_bytes_per_step": 4, "ms_per_step": e2e_s / args.steps * 1e3},
            "roofline": roof, "roofline_gather": roof_gather, "roofline_backward": roof_bwd, "cpu_baseline": cb}
    print(json.dumps(line), flush=True)
    _shutdown(eng, world)


def _shutdown(eng, world):
    """Leave cleanly under torchrun: drop the captured step graph (it holds NCCL kernels) before the process group goes, and
    never let a stuck communicator teardown keep the job alive — the JSON line is already out, so a watchdog ends the process."""
    if world <= 1:
        return
    import torch.distributed as dist
    sys.stdout.flush()
    torch.cuda.synchronize()
    if getattr(eng, "graph", None) is not None:
        eng.graph.reset()
        eng.graph = None
    t = threading.Timer(20.0, lambda: os._exit(0))
    t.daemon = True
    t.start()
    try:
        dist.destroy_process_group()
    finally:
        t.cancel()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.track:
        run_track(a)
    elif a.sampler:
        run_sampler(a)
    else:
        run_ours(a)
