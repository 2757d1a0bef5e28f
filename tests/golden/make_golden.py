"""Generate the golden fixtures in tests/golden/*.npz by running the REFERENCE's own Python
(/root/reference: pointnet2/utils/*.py, models/backbone/pointnet.py, models/head/*.py, models/bat.py,
models/p2b.py, models/base_model.py — unmodified, imported from where they lie) on CPU.

The reference's native dependency `pointnet2_ops._ext` (absent, see oracle/pointnet2_ops_ref.c) is replaced by the
C oracle through oracle/ext_stub.py; its absent host-side dependencies (pytorch_lightning, easydict, torchmetrics,
nuscenes, shapely, pyquaternion, datasets/*) are replaced by inert stand-ins, and `Tensor.cuda()` is neutralised
because the reference hard-codes it (pointnet2_modules.py:56, base_model.py:151).

So these vectors pin the COMPOSITION (QueryAndGroup, SA / FP modules, backbone, xcorr, RPN, whole-model
forward, losses, gradients) against the reference itself; the nine ops underneath remain "parity unpinned".

Run only inside the authoring container:   python tests/golden/make_golden.py
The GPU box never reads /root/reference; it only sees the committed .npz files.
"""
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import ext_stub  # noqa: E402
from _params import det_state_dict  # noqa: E402
from open3dsot_b200.compat.easydict import EasyDict  # noqa: E402
from open3dsot_b200.compat import lightning as _pl_shim  # noqa: E402
from open3dsot_b200.datasets.synthetic import synthetic_siamese_batch  # noqa: E402
from open3dsot_b200.config import load_yaml  # noqa: E402


def install_stubs():
    ext_stub.install()
    torch.Tensor.cuda = lambda self, *a, **k: self  # reference hard-codes .cuda()

    def mod(name, **attrs):
        m = types.ModuleType(name)
        for k, v in attrs.items():
            setattr(m, k, v)
        sys.modules[name] = m
        return m

    mod("easydict", EasyDict=EasyDict)
    pl = mod("pytorch_lightning", LightningModule=_pl_shim.LightningModule)
    pl.utilities = mod("pytorch_lightning.utilities")
    pl.utilities.distributed = mod("pytorch_lightning.utilities.distributed")

    class _Metric(nn.Module):
        def __init__(self, *a, **k):
            super().__init__()

        def forward(self, *a, **k):          # logging-only metric objects of the reference
            return torch.zeros(2)

    mod("torchmetrics", Metric=_Metric, Accuracy=_Metric)
    nus = mod("nuscenes"); nus.utils = mod("nuscenes.utils")
    nus.utils.geometry_utils = mod("nuscenes.utils.geometry_utils")
    sys.modules["nuscenes.utils"] = nus.utils
    # datasets.points_utils: load the reference's own file (its torch box transforms are used by M2TRACK.forward);
    # its numpy-side imports (pyquaternion, nuscenes, datasets.data_classes) are inert stand-ins
    mod("pyquaternion", Quaternion=object)
    ds = mod("datasets"); ds.__path__ = []
    mod("datasets.data_classes", PointCloud=object, Box=object)
    import importlib.util
    spec = importlib.util.spec_from_file_location("datasets.points_utils", os.path.join(REF, "datasets", "points_utils.py"))
    pu = importlib.util.module_from_spec(spec)
    sys.modules["datasets.points_utils"] = pu
    spec.loader.exec_module(pu)
    ds.points_utils = pu
    ut = mod("utils")
    ut.metrics = mod("utils.metrics", TorchSuccess=_Metric, TorchPrecision=_Metric,
                     estimateOverlap=None, estimateAccuracy=None)
    sys.path.insert(0, REF)  # `pointnet2`, `models` resolve to the reference packages


def np_(t):
    return t.detach().cpu().numpy().copy()


def gen_modules(out):
    from pointnet2.utils import pointnet2_utils as ru, pointnet2_modules as rm
    from models.head.xcorr import P2B_XCorr, BoxAwareXCorr
    from models.head.rpn import P2BVoteNetRPN
    g = torch.Generator().manual_seed(11)
    B, N, C, M = 2, 96, 8, 24
    xyz = torch.rand(B, N, 3, generator=g) * 1.2
    xyz[:, 10:20] = xyz[:, 0:10]                      # exact duplicates -> ties
    feats = torch.randn(B, C, N, generator=g)
    new_xyz = xyz[:, :M].contiguous()
    out["qg_xyz"], out["qg_feats"] = np_(xyz), np_(feats)
    for norm in (False, True):
        qg = ru.QueryAndGroup(0.35, 16, use_xyz=True, return_idx=True, normalize_xyz=norm)
        nf, idx = qg(xyz, new_xyz, feats)
        out[f"qg_out_norm{int(norm)}"], out[f"qg_idx_norm{int(norm)}"] = np_(nf), np_(idx)

    # SA module, train + eval, FPS and arange centres
    for tag, use_fps in (("fps", True), ("arange", False)):
        sa = rm.PointnetSAModule(mlp=[C, 16, 16, 32], radius=0.35, nsample=16, use_fps=use_fps)
        sa.load_state_dict(det_state_dict(sa.state_dict(), seed=1))
        x_in = xyz.clone().requires_grad_(False)
        f_in = feats.clone().requires_grad_(True)
        sa.train()
        nx, nf, sidx = sa(x_in, f_in, M, True)
        nf.square().sum().backward()
        out[f"sa_{tag}_train_out"], out[f"sa_{tag}_idx"], out[f"sa_{tag}_newxyz"] = np_(nf), np_(sidx), np_(nx)
        out[f"sa_{tag}_train_gfeat"] = np_(f_in.grad)
        out[f"sa_{tag}_train_gw0"] = np_(sa.mlps[0].layer0.conv.weight.grad)
        out[f"sa_{tag}_train_gw2"] = np_(sa.mlps[0].layer2.conv.weight.grad)
        out[f"sa_{tag}_train_ggamma1"] = np_(sa.mlps[0].layer1.bn.bn.weight.grad)
        out[f"sa_{tag}_rm2"] = np_(sa.mlps[0].layer2.bn.bn.running_mean)
        out[f"sa_{tag}_rv2"] = np_(sa.mlps[0].layer2.bn.bn.running_var)
        sa.eval()
        sa.load_state_dict(det_state_dict(sa.state_dict(), seed=1))
        _, nf_e, _ = sa(x_in, feats, M, True)
        out[f"sa_{tag}_eval_out"] = np_(nf_e)

    # FP module
    fp = rm.PointnetFPModule(mlp=[C + 4, 16, 12])
    fp.load_state_dict(det_state_dict(fp.state_dict(), seed=2))
    fp.train()
    unknown, known = xyz[:, :48].contiguous(), xyz[:, 40:72].contiguous()
    uf = torch.randn(B, 4, 48, generator=g)
    kf = torch.randn(B, C, 32, generator=g).requires_grad_(True)
    y = fp(unknown, known, uf, kf)
    y.square().sum().backward()
    out["fp_unknown"], out["fp_known"], out["fp_uf"], out["fp_kf"] = np_(unknown), np_(known), np_(uf), np_(kf)
    out["fp_out"], out["fp_gkf"] = np_(y), np_(kf.grad)

    # xcorr heads + rpn (small channel counts)
    f, hid, Mt, Ns = 16, 16, 12, 20
    tf = torch.randn(B, f, Mt, generator=g); sf = torch.randn(B, f, Ns, generator=g)
    txyz = torch.rand(B, Mt, 3, generator=g); sxyz = torch.rand(B, Ns, 3, generator=g)
    tbc = torch.rand(B, Mt, 9, generator=g); sbc = torch.rand(B, Ns, 9, generator=g)
    for k_, v_ in dict(xc_tf=tf, xc_sf=sf, xc_txyz=txyz, xc_sxyz=sxyz, xc_tbc=tbc, xc_sbc=sbc).items():
        out[k_] = np_(v_)
    px = P2B_XCorr(f, hid, f); px.load_state_dict(det_state_dict(px.state_dict(), seed=3)); px.train()
    out["p2bx_out"] = np_(px(tf, sf, txyz))
    bx = BoxAwareXCorr(f, hid, f, k=4, bc_channel=9); bx.load_state_dict(det_state_dict(bx.state_dict(), seed=4))
    bx.train()
    out["bax_out"] = np_(bx(tf, sf, txyz, sxyz, tbc, sbc))
    rp = P2BVoteNetRPN(f, vote_channel=f, num_proposal=8); rp.load_state_dict(det_state_dict(rp.state_dict(), seed=5))
    rp.train()
    boxes, cla, vxyz, cen = rp(sxyz, sf)
    out["rpn_boxes"], out["rpn_cla"], out["rpn_vote_xyz"], out["rpn_centers"] = np_(boxes), np_(cla), np_(vxyz), np_(cen)


def gen_model(name, cfg_file, B, M, N, out, seed):
    from models import get_model
    cfg = EasyDict(load_yaml(os.path.join(ROOT, "cfgs", cfg_file)))
    net = get_model(cfg.net_model)(cfg)
    net.load_state_dict(det_state_dict(net.state_dict(), seed=seed), strict=False)
    net.train()
    net.log = lambda *a, **k: None
    batch = synthetic_siamese_batch(B, M, N, seed=1234 + seed, box_aware=(name == "bat"))
    # Place the regression target so that the objectness terms are exercised (base_model.py:142-157): per sample one
    # proposal centre closer than 0.3 m (label 1, feeds loss_box) and one in the 0.3-0.6 m band (masked out); with the
    # synthetic labels every centre is farther than 0.6 m and neither term would be pinned.
    with torch.no_grad():
        cen = net({k: v.clone() for k, v in batch.items()})["center_xyz"]
    net.load_state_dict(det_state_dict(net.state_dict(), seed=seed), strict=False)
    for b in range(B):
        d = torch.cdist(cen[b], cen[b])
        ok = ((d > 0.56) & (d < 0.84)).nonzero()
        assert len(ok), "no pair of proposal centres 0.56-0.84 m apart"
        i, j = (int(v) for v in ok[0])
        batch["box_label"][b, :3] = cen[b, i] + 0.25 * (cen[b, j] - cen[b, i]) / d[i, j]
    out[f"{name}_box_label"] = np_(batch["box_label"])
    terms = {}
    ref_compute_loss = net.compute_loss

    def spy(data, output):
        ld = ref_compute_loss(data, output)
        terms.update({k: v.detach().clone() for k, v in ld.items()})
        return ld
    net.compute_loss = spy
    b2 = {k: v.clone() for k, v in batch.items()}
    loss = net.training_step(b2, 0)
    loss.backward()
    net.compute_loss = ref_compute_loss
    out[f"{name}_loss"] = np_(loss)
    for k, v in terms.items():
        out[f"{name}_term::{k}"] = np_(v)
    sd = dict(net.named_parameters())
    for k in ("conv_final.bias", "backbone.SA_modules.0.mlps.0.layer0.conv.weight",
              "backbone.SA_modules.2.mlps.0.layer2.bn.bn.weight", "rpn.vote_layer.2.conv.bias",
              "xcorr.mlp.layer0.conv.weight", "rpn.FC_proposal.2.conv.weight"):
        out[f"{name}_grad::{k}"] = np_(sd[k].grad)[:16]   # first rows only: keeps the fixture small
    out[f"{name}_gradnorms"] = np.array([float(p.grad.norm()) for _, p in sorted(sd.items())], dtype=np.float64)
    # forward outputs in train mode (fresh copy so that running stats restart from the same state)
    net.load_state_dict(det_state_dict(net.state_dict(), seed=seed), strict=False)
    with torch.no_grad():
        ep = net(batch)
    for k in ("estimation_boxes", "estimation_cla", "vote_xyz", "center_xyz", "sample_idxs"):
        out[f"{name}_{k}"] = np_(ep[k])
    if "pred_search_bc" in ep:
        out[f"{name}_pred_search_bc"] = np_(ep["pred_search_bc"])
    net.eval()
    net.load_state_dict(det_state_dict(net.state_dict(), seed=seed), strict=False)
    with torch.no_grad():
        ep = net(batch)
    out[f"{name}_eval_boxes"] = np_(ep["estimation_boxes"])
    out[f"{name}_eval_cla"] = np_(ep["estimation_cla"])


def gen_m2track(out):
    """M2_track_kitti.yaml (BASELINE.json configs[2]) at B=4, point_sample_size 256: forward, loss, gradient norms."""
    from models import get_model
    from open3dsot_b200.datasets.synthetic import synthetic_motion_batch
    cfg = EasyDict(load_yaml(os.path.join(ROOT, "cfgs", "M2_track_kitti.yaml")))
    net = get_model(cfg.net_model)(cfg)
    net.load_state_dict(det_state_dict(net.state_dict(), seed=31), strict=False)
    net.train()
    net.log = lambda *a, **k: None
    net.logger.experiment.add_scalars = lambda *a, **k: None
    batch = synthetic_motion_batch(4, 256, seed=77)
    loss = net.training_step({k: v.clone() for k, v in batch.items()}, 0)
    loss.backward()
    out["m2_loss"] = np_(loss)
    sd = dict(net.named_parameters())
    out["m2_gradnorms"] = np.array([float(p.grad.norm()) if p.grad is not None else 0.0 for _, p in sorted(sd.items())],
                                   dtype=np.float64)
    net.load_state_dict(det_state_dict(net.state_dict(), seed=31), strict=False)
    with torch.no_grad():
        ep = net({k: v.clone() for k, v in batch.items()})
    for k in ("estimation_boxes", "seg_logits", "motion_pred", "aux_estimation_boxes", "pred_bc", "motion_cls"):
        out[f"m2_{k}"] = np_(ep[k])
    net.eval()
    net.load_state_dict(det_state_dict(net.state_dict(), seed=31), strict=False)
    with torch.no_grad():
        ep = net({k: v.clone() for k, v in batch.items()})
    out["m2_eval_boxes"] = np_(ep["estimation_boxes"])


def gen_checkpoint_eval():
    """SURVEY.md §8f rank 1: the trained weights of the reference's shipped `pretrained_models/bat_kitti_car.ckpt` (6 MB of
    float32), stored as 4-bit codes per output channel with BatchNorm statistics and biases exact (tests/_params.py
    `pack_state_4bit`), and what the reference's own BAT computes in eval mode with exactly those weights on a fixed
    synthetic pair -> bat_kitti_car_q4.npz (weights under their state-dict keys, outputs under 'out:<name>')."""
    from models import get_model
    from open3dsot_b200.checkpoint import load_lightning_checkpoint
    from _params import pack_state_4bit, unpack_state_4bit
    ck = load_lightning_checkpoint(os.path.join(REF, "pretrained_models", "bat_kitti_car.ckpt"))
    cfg = EasyDict(load_yaml(os.path.join(ROOT, "cfgs", "BAT_Car.yaml")))
    net = get_model(cfg.net_model)(cfg)
    packed = pack_state_4bit({k: v for k, v in ck["state_dict"].items() if k in net.state_dict()})
    net.load_state_dict(unpack_state_4bit(packed), strict=True)
    net.eval()
    batch = synthetic_siamese_batch(2, 512, 1024, seed=4242, box_aware=True)
    with torch.no_grad():
        ep = net({k: v.clone() for k, v in batch.items()})
    for k in ("estimation_boxes", "estimation_cla", "vote_xyz", "center_xyz", "sample_idxs", "pred_search_bc"):
        packed[f"out:{k}"] = np_(ep[k])
    np.savez_compressed(os.path.join(HERE, "bat_kitti_car_q4.npz"), **packed)


def _with_tensors(obj, fn):
    """Apply `fn` to every tensor inside nested dicts / lists / tuples, in place where the container allows."""
    if isinstance(obj, torch.Tensor):
        return fn(obj)
    if isinstance(obj, dict):
        for k in list(obj):
            obj[k] = _with_tensors(obj[k], fn)
    elif isinstance(obj, list):
        obj[:] = [_with_tensors(x, fn) for x in obj]
    elif isinstance(obj, tuple):
        obj = type(obj)(_with_tensors(x, fn) for x in obj)
    return obj


def gen_checkpoint_skeletons():
    """The reference's shipped checkpoints (18-27 MB each) cut down for tests/test_checkpoint_compat.py: every tensor keeps
    its first value, viewed at its full shape with zero strides, so the file has the original's format (legacy pickle or
    zip), top-level keys, state-dict key order, shapes and dtypes, optimizer-state layout, hyper-parameters (pickled as
    `easydict.EasyDict`) and Lightning bookkeeping (the `ModelCheckpoint` class as a callbacks key) in a few KiB."""
    import zipfile
    from open3dsot_b200.checkpoint import load_lightning_checkpoint
    os.makedirs(os.path.join(HERE, "checkpoints"), exist_ok=True)
    for name in ("bat_kitti_car.ckpt", "bat_kitti_pedestrian.ckpt", "mmtrack_kitti_car.ckpt"):
        src = os.path.join(REF, "pretrained_models", name)
        ck = load_lightning_checkpoint(src)
        _with_tensors(ck, lambda t: t.reshape(-1)[:1].clone().reshape([1] * t.dim()).expand(t.shape) if t.numel() else t)
        # globals the restricted unpickler turned into placeholders, and our EasyDict, are written under their original names
        names = {k.__module__: k for k in ck.get("callbacks", {}) if isinstance(k, type)}
        saved = {m: sys.modules.get(m) for m in ["easydict"] + [".".join(p.split(".")[:i + 1]) for p in names
                                                                for i in range(p.count(".") + 1)]}
        for m in saved:
            sys.modules[m] = types.ModuleType(m)
        for m, cls in names.items():
            setattr(sys.modules[m], cls.__name__, cls)
        old = (EasyDict.__module__, EasyDict.__qualname__)
        EasyDict.__module__, EasyDict.__qualname__ = "easydict", "EasyDict"
        sys.modules["easydict"].EasyDict = EasyDict
        try:
            torch.save(ck, os.path.join(HERE, "checkpoints", name), _use_new_zipfile_serialization=zipfile.is_zipfile(src))
        finally:
            EasyDict.__module__, EasyDict.__qualname__ = old
            for m, mod in saved.items():
                if mod is None:
                    sys.modules.pop(m, None)
                else:
                    sys.modules[m] = mod


def main():
    assert os.path.isdir(REF), "golden vectors can only be generated where /root/reference exists"
    install_stubs()
    torch.set_num_threads(8)
    mods = {}
    gen_modules(mods)
    np.savez_compressed(os.path.join(HERE, "ref_modules.npz"), **mods)
    models = {}
    gen_model("bat", "BAT_Car.yaml", 2, 256, 512, models, seed=21)
    gen_model("p2b", "P2B_Car.yaml", 2, 256, 512, models, seed=22)   # BASELINE.json configs[0] shape; B=2 (B=1 is a degenerate BatchNorm case)
    gen_m2track(models)
    np.savez_compressed(os.path.join(HERE, "ref_models.npz"), **models)
    gen_checkpoint_eval()
    gen_checkpoint_skeletons()
    for f in ("ref_modules.npz", "ref_models.npz", "bat_kitti_car_q4.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
