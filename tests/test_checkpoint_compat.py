"""Drop-in check of the checkpoint surface (SURVEY.md §8f rank 1): the reference's shipped BAT / M2-Track checkpoints
load, key for key, into our modules.  The files under tests/golden/checkpoints/ are those checkpoints cut down by
tests/golden/make_golden.py: the original format, keys, shapes, hyper-parameters and Lightning bookkeeping, with every
tensor reduced to its first value (stride-0 views), since the originals are 18-27 MB each."""
import os

import pytest
import torch

from open3dsot_b200.checkpoint import load_lightning_checkpoint, load_reference_weights
from open3dsot_b200.config import load_config
from open3dsot_b200.models import get_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CKPT_DIR = os.path.join(ROOT, "tests", "golden", "checkpoints")


@pytest.mark.parametrize("ckpt,cfg_file", [("bat_kitti_car.ckpt", "BAT_Car.yaml"),
                                           ("bat_kitti_pedestrian.ckpt", "BAT_Pedestrian.yaml"),
                                           ("mmtrack_kitti_car.ckpt", "M2_track_kitti.yaml")])
def test_reference_checkpoint_loads_strictly(ckpt, cfg_file):
    cfg = load_config(os.path.join(ROOT, "cfgs", cfg_file))
    net = get_model(cfg.net_model)(cfg)
    ours = net.state_dict()
    ck = load_reference_weights(net, os.path.join(CKPT_DIR, ckpt), strict=False)
    ref_sd = ck["state_dict"]
    # every parameter / buffer of ours exists in the checkpoint with the same shape; the checkpoint's extra entries are
    # only the reference's metric-module buffers (torchmetrics), which carry no weights
    for k, v in ours.items():
        assert k in ref_sd and tuple(ref_sd[k].shape) == tuple(v.shape), k
    extra = [k for k in ref_sd if k not in ours]
    assert all(k.split(".")[0] in ("prec", "success", "seg_acc", "motion_acc") for k in extra), extra
    assert "hyper_parameters" in ck and ck.get("pytorch-lightning_version", "").startswith("1.3")
    w = net.state_dict()
    some = next(k for k in w if k.endswith("weight") and w[k].dim() >= 2)
    assert torch.equal(w[some], ref_sd[some])


def test_checkpoint_hparams_are_attribute_accessible():
    ck = load_lightning_checkpoint(os.path.join(CKPT_DIR, "bat_kitti_car.ckpt"))
    hp = ck["hyper_parameters"]
    cfg = hp["config"] if "config" in hp else hp
    assert cfg.net_model == "BAT" and cfg.use_fps is True


def test_restricted_unpickler_neutralises_foreign_globals(tmp_path):
    """A crafted pickle that names `builtins.eval` / `os.system` must not reach them: every global outside the exact
    whitelist resolves to an inert placeholder class (open3dsot_b200/checkpoint.py:_SAFE)."""
    import io
    import pickle
    from open3dsot_b200.checkpoint import _RestrictedUnpickler
    marker = tmp_path / "pwned"
    for payload in (b"cbuiltins\neval\n(S'__import__(\"os\").system(\"touch %b\")'\ntR." % str(marker).encode(),
                    b"cos\nsystem\n(S'touch %b'\ntR." % str(marker).encode(),
                    b"cbuiltins\ngetattr\n(cbuiltins\n__import__\nS'os'\ntR."):
        try:
            _RestrictedUnpickler(io.BytesIO(payload)).load()
        except Exception:
            pass                       # an inert placeholder may refuse the call signature; what matters: nothing ran
    assert not marker.exists()
    for mod, name in (("builtins", "eval"), ("builtins", "exec"), ("builtins", "getattr"), ("builtins", "__import__"),
                      ("torch.hub", "load"), ("numpy.testing._private.utils", "runstring"), ("os", "system")):
        cls = _RestrictedUnpickler(io.BytesIO(b"")).find_class(mod, name)
        assert isinstance(cls, type) and cls.__module__ == mod and cls("x") is not None
        import builtins
        assert cls is not getattr(builtins, name, None)
    assert _RestrictedUnpickler(io.BytesIO(b"")).find_class("collections", "OrderedDict").__name__ == "OrderedDict"
    pickle.dumps(1)


def test_save_checkpoint_round_trips_in_the_reference_layout(tmp_path):
    """`save_lightning_checkpoint` writes the §8b layout: the reference's key names, `hyper_parameters.config` pickled as
    `easydict.EasyDict` (no trace of this package in the file), Lightning's bookkeeping keys; reading it back is lossless."""
    from open3dsot_b200.checkpoint import save_lightning_checkpoint
    cfg = load_config(os.path.join(ROOT, "cfgs", "BAT_Car.yaml"))
    net = get_model(cfg.net_model)(cfg)
    load_reference_weights(net, os.path.join(CKPT_DIR, "bat_kitti_car.ckpt"), strict=False)
    path = str(tmp_path / "ours.ckpt")
    save_lightning_checkpoint(net, path, epoch=7, global_step=1234)
    raw = open(path, "rb").read()
    assert b"easydict" in raw and b"open3dsot_b200" not in raw
    ck = load_lightning_checkpoint(path)
    ref = load_lightning_checkpoint(os.path.join(CKPT_DIR, "bat_kitti_car.ckpt"))
    assert set(ref.keys()) - set(ck.keys()) <= {"hparams_name"}
    assert ck["epoch"] == 7 and ck["global_step"] == 1234 and ck["pytorch-lightning_version"] == "1.3.8"
    assert ck["hyper_parameters"]["config"].net_model == "BAT" and ck["hyper_parameters"]["config"].use_fps is True
    assert list(ck["state_dict"].keys()) == [k for k in ref["state_dict"].keys() if k in ck["state_dict"]]   # same names, same order
    for k, v in ck["state_dict"].items():
        assert torch.equal(v, ref["state_dict"][k]), k
    net2 = get_model(cfg.net_model)(cfg)
    load_reference_weights(net2, path, strict=True)
