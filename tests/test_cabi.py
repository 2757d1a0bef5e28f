"""C-ABI boundary checks that need no GPU: the library loads, exports every symbol the header declares,
the Python prototypes cover them, and the product path refuses CPU tensors / a missing library loudly."""
import ctypes
import os
import re

import pytest
import torch

from open3dsot_b200 import _lib, ops

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "o3d_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(o3d_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    syms = _header_symbols()
    assert len(syms) >= 17
    L = ctypes.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(L, s), f"{s} declared in include/o3d_b200.h but not exported"


def test_python_prototypes_match_header():
    assert sorted(_lib.PROTOTYPES) == _header_symbols()


def test_version_and_thread_rule():
    L = _lib.lib()
    assert L.o3d_version() == 100
    assert [L.o3d_opt_threads(n) for n in (1, 100, 512, 1024)] == [1, 64, 512, 512]


def test_cpu_tensors_are_rejected_like_upstream():
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.furthest_point_sampling(torch.zeros(1, 8, 3), 4)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.ball_query(torch.zeros(1, 2, 3), torch.zeros(1, 8, 3), 0.3, 4)


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libo3d_b200.so")
    with pytest.raises(RuntimeError, match="no CPU or PyTorch fallback"):
        _lib.lib()


def test_argument_errors_return_status_not_crash():
    L = _lib.lib()
    assert L.o3d_fps(None, 1, 8, 4, None, None) < 0
    assert b"null" in L.o3d_last_error()
    assert L.o3d_ballquery_group(1, 1, 1, 1, 8, 4, 3, 0.3, 4, 0, None, 1, None) < 0   # C % 4 != 0


def _sa_desc(C, widths):
    d = _lib.StackDesc()
    d.n_layers, d.xyz_first, d.c0, d.K0 = len(widths), 1, C, ((C + 3) & ~3) + 4
    cin = C + 3
    dummy = ctypes.c_void_p(16)                     # never dereferenced by the planning entry points
    for l, w in enumerate(widths):
        d.cin[l], d.cout[l], d.relu[l], d.has_bn[l] = cin, w, 1, 1
        d.weight[l] = d.gamma[l] = d.beta[l] = d.running_mean[l] = d.running_var[l] = dummy
        cin = w
    return d


def test_fused_sa_layer_plan_and_argument_checks():
    """host-side planning of o3d_sa_fused_* (no launch): block sizes follow the tile arithmetic, shapes outside the kernel's range
    and bad arguments come back as a status + message, never as a crash"""
    L = _lib.lib()
    tile = 2 * 128 * 32 * 4                          # one 128-channel x 32-k weight tile: TF32 hi | lo
    # SA3 of the backbone: 256 features -> 256, 256, 256: 3 layers x 2 channel tiles x 8 k-blocks
    n = L.o3d_sa_fused_prepared_bytes(ctypes.byref(_sa_desc(256, [256, 256, 256])))
    assert n >= 48 * tile and n < 48 * tile + 16384 and n % 1024 == 0
    # SA1: coordinates only — the first layer has no tensor-core part
    n1 = L.o3d_sa_fused_prepared_bytes(ctypes.byref(_sa_desc(0, [64, 64, 128])))
    assert 4 * tile <= n1 < 4 * tile + 16384
    assert L.o3d_sa_fused_prepared_bytes(ctypes.byref(_sa_desc(257, [256, 256, 256]))) >= (18 + 32) * tile   # vote clustering: 9 k-blocks in
    assert L.o3d_sa_fused_prepared_bytes(ctypes.byref(_sa_desc(8, [16, 300]))) == -1       # > 256 channels in a layer
    assert L.o3d_sa_fused_prepared_bytes(ctypes.byref(_sa_desc(300, [64, 64]))) == -1      # > 288 input features
    d = _sa_desc(8, [16, 32])
    assert L.o3d_sa_fused_forward(ctypes.byref(d), 16, 16, 16, 16, 8, 1, 64, 32, 0.3, 24, 0, 16, 32, None, None) < 0
    assert b"nsample" in L.o3d_last_error()
    assert L.o3d_sa_fused_forward(ctypes.byref(d), 16, 16, 16, None, 8, 1, 64, 32, 0.3, 16, 0, 16, 32, None, None) < 0
    assert b"features" in L.o3d_last_error()
    assert L.o3d_resample(16, 16, 16, 16, 1, 100, 4096, 16, 16, 16, None, None) < 0        # size > 2048
    assert b"size" in L.o3d_last_error()


def test_stack_plan_rejects_unknown_use_tc_bits():
    """use_tc has two bits (tensor-core forward + dgrad, tensor-core wgrad); a descriptor with any other bit set is refused
    instead of silently running the default kernels"""
    L = _lib.lib()
    d = _sa_desc(64, [128, 128])
    d.P, d.S, d.training = 256, 32, 1
    for use_tc, ok in ((3, True), (7, False), (11, False)):
        d.use_tc = use_tc
        for backward in (0, 1):
            n = L.o3d_stack_workspace_bytes(ctypes.byref(d), backward)
            assert (n > 0) if ok else (n == -1), (use_tc, backward, n)


def test_debug_set_accepts_only_the_force_mt_switch():
    L = _lib.lib()
    assert L.o3d_debug_set(1, 0) < 0
    assert b"o3d_debug_set" in L.o3d_last_error()
    assert L.o3d_debug_set(0, 2) < 0
    assert L.o3d_debug_set(0, 0) == 0
