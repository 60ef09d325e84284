"""The per-thread bodies of the depthwise kernels (sniper_b200/csrc/depthwise_core.cuh) executed on the CPU by
tests/dw_emulate.cu with the launch geometry of depthwise.cu, against torch float64 (grouped conv2d and its autograd):
pins the tap algebra, strides, borders, ragged widths, row strides and the weight-gradient grid decomposition without
a GPU.  (The launches themselves are covered by tests/test_zz_mobilenet_gpu.py.)"""
import ctypes
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "dw_emulate.cu")
OUT = os.path.join(ROOT, "tests", "_build", "libdw_emul.so")
pytestmark = pytest.mark.skipif(shutil.which("nvcc") is None, reason="nvcc not available")


@pytest.fixture(scope="module")
def emu():
    core = os.path.join(ROOT, "sniper_b200", "csrc", "depthwise_core.cuh")
    if not os.path.exists(OUT) or os.path.getmtime(OUT) < max(os.path.getmtime(SRC), os.path.getmtime(core)):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        # compiled under a private name and renamed into place: parallel test workers never load a half-written file
        tmp = "%s.%d" % (OUT, os.getpid())
        subprocess.check_call(["nvcc", "-O2", "-std=c++17", "-Xcompiler", "-fPIC", "-shared", "-o", tmp, SRC],
                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        os.replace(tmp, OUT)
    return ctypes.CDLL(OUT)


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def _case(NB, H, W, C, stride, dtype, ld_extra=0, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(NB, H, W, C + ld_extra, generator=g).to(dtype)
    w = torch.randn(9, C, generator=g) * 0.3
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    dy = torch.randn(NB, Ho, Wo, C + ld_extra, generator=g).to(dtype)
    return x, w, dy, Ho, Wo


def _ref(x, w, dy, C, stride):
    """float64 grouped convolution of the values the kernel reads (bf16 inputs are exact in float64)."""
    xd = x[..., :C].double().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    wd = w.double().t().reshape(C, 1, 3, 3).contiguous().requires_grad_(True)       # [9,C] tap-major -> (C,1,3,3)
    y = F.conv2d(xd, wd, stride=stride, padding=1, groups=C)
    y.backward(dy[..., :C].double().permute(0, 3, 1, 2))
    return (y.detach().permute(0, 2, 3, 1), xd.grad.permute(0, 2, 3, 1), wd.grad.reshape(C, 9).t())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("NB,H,W,C,stride,ld_extra", [
    (2, 8, 8, 64, 1, 0), (2, 8, 8, 64, 2, 0), (1, 7, 9, 8, 1, 0), (1, 7, 9, 8, 2, 4), (3, 5, 6, 132, 1, 0),
    (1, 16, 16, 192, 2, 0), (2, 1, 1, 4, 1, 0), (1, 2, 3, 4, 2, 0)])
def test_depthwise_cores_match_float64(emu, dtype, NB, H, W, C, stride, ld_extra):
    dt = 0 if dtype == torch.float32 else 1
    x, w, dy, Ho, Wo = _case(NB, H, W, C, stride, dtype, ld_extra)
    ld = C + ld_extra
    y_ref, dx_ref, dw_ref = _ref(x, w, dy, C, stride)
    tol = 1e-5 if dtype == torch.float32 else 1e-2           # bf16: only the OUTPUT rounding (inputs are exact)
    # forward
    y = torch.full((NB, Ho, Wo, ld), 7.0).to(dtype)
    emu.emu_dw_fwd(_p(x), ctypes.c_long(ld), _p(w), _p(y), ctypes.c_long(ld), NB, H, W, C, stride, dt)
    assert torch.allclose(y[..., :C].double(), y_ref, rtol=tol, atol=tol * 3)
    if ld_extra:
        assert (y[..., C:].float() == 7.0).all()              # padding columns untouched
    # data gradient
    dx = torch.full((NB, H, W, ld), 7.0).to(dtype)
    emu.emu_dw_dgrad(_p(dy), ctypes.c_long(ld), _p(w), _p(dx), ctypes.c_long(ld), NB, H, W, C, stride, dt)
    assert torch.allclose(dx[..., :C].double(), dx_ref, rtol=tol, atol=tol * 3)
    # weight gradient (accumulates); any grid width gives the same sums
    scale = float(dw_ref.abs().max()) + 1.0
    for gx in (1, 3, 37, 592):
        dw = torch.ones(9, C)
        emu.emu_dw_wgrad(_p(x), ctypes.c_long(ld), _p(dy), ctypes.c_long(ld), _p(dw), NB, H, W, C, stride, dt, gx)
        assert torch.allclose(dw.double() - 1.0, dw_ref, rtol=1e-4, atol=1e-5 * scale), gx


@pytest.mark.parametrize("NB,H,W,C,stride,ld_extra", [(2, 8, 32, 64, 1, 0), (1, 19, 45, 128, 1, 0), (2, 9, 7, 64, 1, 64), (1, 16, 32, 64, 2, 0),
                                                      (2, 11, 37, 192, 2, 0), (1, 1, 1, 64, 1, 0), (1, 40, 70, 64, 2, 0)])
def test_tiled_bf16_kernels_match_float64(emu, NB, H, W, C, stride, ld_extra):
    """The shared-memory tiled forward (and, flipped, the stride-1 data gradient): stage + compute phases per block."""
    x, w, dy, Ho, Wo = _case(NB, H, W, C, stride, torch.bfloat16, ld_extra, seed=4)
    ld = C + ld_extra
    y_ref, dx_ref, _ = _ref(x, w, dy, C, stride)
    y = torch.full((NB, Ho, Wo, ld), 7.0).to(torch.bfloat16)
    emu.emu_dw_tiled(_p(x), ctypes.c_long(ld), _p(w), _p(y), ctypes.c_long(ld), NB, H, W, C, stride, 0)
    assert torch.allclose(y[..., :C].double(), y_ref, rtol=1e-2, atol=3e-2)
    if ld_extra:
        assert (y[..., C:].float() == 7.0).all()
    if stride == 1:
        dx = torch.full((NB, H, W, ld), 7.0).to(torch.bfloat16)
        emu.emu_dw_tiled(_p(dy), ctypes.c_long(ld), _p(w), _p(dx), ctypes.c_long(ld), NB, H, W, C, 1, 1)
        assert torch.allclose(dx[..., :C].double(), dx_ref, rtol=1e-2, atol=3e-2)
        # identical to the register-window kernels (same products, same order within a row)
        dx2 = torch.zeros_like(dx)
        emu.emu_dw_dgrad(_p(dy), ctypes.c_long(ld), _p(w), _p(dx2), ctypes.c_long(ld), NB, H, W, C, 1, 1)
        assert torch.equal(dx[..., :C].float(), dx2[..., :C].float())
    y2 = torch.zeros_like(y)
    emu.emu_dw_fwd(_p(x), ctypes.c_long(ld), _p(w), _p(y2), ctypes.c_long(ld), NB, H, W, C, stride, 1)
    assert torch.equal(y[..., :C].float(), y2[..., :C].float())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_first_layer_im2col_and_add(emu, dtype):
    dt = 0 if dtype == torch.float32 else 1
    g = torch.Generator().manual_seed(3)
    NB, H, W, Kp = 2, 10, 12, 64
    x = torch.randn(NB, 3, H, W, generator=g)
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    col = torch.full((NB * Ho * Wo, Kp), 5.0).to(dtype)
    emu.emu_im2col3x3s2(_p(x), _p(col), NB, H, W, Kp, dt)
    # definition: unfold gives (ci, kh, kw) order -> reorder to (kh, kw, ci)
    u = F.unfold(x, 3, padding=1, stride=2).view(NB, 3, 9, Ho * Wo).permute(0, 3, 2, 1).reshape(NB * Ho * Wo, 27)
    assert torch.equal(col[:, :27].float(), u.to(dtype).float()) and not col[:, 27:].float().any()
    # the GEMM this feeds == the convolution
    wt = torch.randn(8, 3, 3, 3, generator=g)
    rows = wt.permute(0, 2, 3, 1).reshape(8, 27)
    y = col[:, :27].double() @ rows.double().t()
    ref = F.conv2d(x.to(dtype).double(), wt.double(), stride=2, padding=1).permute(0, 2, 3, 1).reshape(-1, 8)
    assert torch.allclose(y, ref, atol=1e-9)
    a = torch.randn(6, 12, generator=g).to(dtype)
    b = torch.randn(6, 12, generator=g).to(dtype)
    o = torch.zeros(6, 12).to(dtype)
    emu.emu_add_rows(_p(a), ctypes.c_long(12), _p(b), ctypes.c_long(12), _p(o), ctypes.c_long(12), ctypes.c_long(6), 12, dt)
    assert torch.equal(o.float(), (a.float() + b.float()).to(dtype).float())
    emu.emu_add_rows(_p(a), ctypes.c_long(12), _p(b), ctypes.c_long(12), _p(a), ctypes.c_long(12), ctypes.c_long(6), 12, dt)
    assert torch.equal(a.float(), o.float())                  # in place


def test_bf16_rounding_helper_is_round_to_nearest_even(emu):
    """store4<bf16> uses a hand-written rounding (usable on the host); it must equal torch's fp32 -> bf16 cast."""
    g = torch.Generator().manual_seed(1)
    a = torch.cat([torch.randn(4096, generator=g) * 10 ** torch.randint(-20, 20, (4096,), generator=g).float(),
                   torch.tensor([0.0, -0.0, 1.0, 1.00390625, 1.01171875, 3.0e38, -3.0e38, 1.0e-38])])    # (no inf: 0 * inf of a neighbouring tap is NaN)
    a = a[: a.numel() // 4 * 4].contiguous()
    # through the depthwise forward with a centre-tap-only kernel: bf16-exact inputs times (1 + 2^-9) land between bf16
    # neighbours, exact ties included
    C = 4
    n = a.numel() // C
    x = a.view(1, n, 1, C).to(torch.bfloat16)
    w = torch.zeros(9, C)
    w[4] = 1.0 + 2.0 ** -9        # x * (1 + 2^-9): results fall between bf16 neighbours, incl. exact ties
    y = torch.zeros(1, n, 1, C, dtype=torch.bfloat16)
    emu.emu_dw_fwd(_p(x), ctypes.c_long(C), _p(w), _p(y), ctypes.c_long(C), 1, n, 1, C, 1, 1)
    want = (x.float() * w[4]).to(torch.bfloat16)
    fin = torch.isfinite(want.float())
    assert torch.equal(y.float()[fin], want.float()[fin])


def test_depthwise_cores_random_shapes(emu):
    """Seeded sweep over odd shapes (maps down to 1x1, widths that leave ragged strips / tiles, channel counts around the
    lane-mapping thresholds, padded rows): every kernel body against float64, tiled == register-window bit for bit."""
    rng = np.random.RandomState(12)
    for it in range(40):
        NB, H, W = int(rng.randint(1, 4)), int(rng.randint(1, 21)), int(rng.randint(1, 41))
        C = int(rng.choice([4, 8, 60, 64, 68, 124, 128, 192]))
        stride = int(rng.randint(1, 3))
        dtype = torch.bfloat16 if rng.rand() < 0.5 else torch.float32
        extra = int(rng.choice([0, 4, 8]))
        dt = 0 if dtype == torch.float32 else 1
        x, w, dy, Ho, Wo = _case(NB, H, W, C, stride, dtype, extra, seed=100 + it)
        ld = C + extra
        y_ref, dx_ref, dw_ref = _ref(x, w, dy, C, stride)
        tol = 1e-5 if dtype == torch.float32 else 1e-2
        tag = (NB, H, W, C, stride, str(dtype), extra)
        y = torch.zeros(NB, Ho, Wo, ld).to(dtype)
        emu.emu_dw_fwd(_p(x), ctypes.c_long(ld), _p(w), _p(y), ctypes.c_long(ld), NB, H, W, C, stride, dt)
        assert torch.allclose(y[..., :C].double(), y_ref, rtol=tol, atol=3 * tol), tag
        dx = torch.zeros(NB, H, W, ld).to(dtype)
        emu.emu_dw_dgrad(_p(dy), ctypes.c_long(ld), _p(w), _p(dx), ctypes.c_long(ld), NB, H, W, C, stride, dt)
        assert torch.allclose(dx[..., :C].double(), dx_ref, rtol=tol, atol=3 * tol), tag
        dw = torch.zeros(9, C)
        emu.emu_dw_wgrad(_p(x), ctypes.c_long(ld), _p(dy), ctypes.c_long(ld), _p(dw), NB, H, W, C, stride, dt,
                         int(rng.randint(1, 50)))
        assert torch.allclose(dw.double(), dw_ref, rtol=1e-4, atol=1e-5 * (float(dw_ref.abs().max()) + 1.0)), tag
        if dt == 1 and C % 64 == 0 and ld % 8 == 0:
            y2 = torch.zeros_like(y)
            emu.emu_dw_tiled(_p(x), ctypes.c_long(ld), _p(w), _p(y2), ctypes.c_long(ld), NB, H, W, C, stride, 0)
            assert torch.equal(y2[..., :C].float(), y[..., :C].float()), tag
            if stride == 1:
                dx2 = torch.zeros_like(dx)
                emu.emu_dw_tiled(_p(dy), ctypes.c_long(ld), _p(w), _p(dx2), ctypes.c_long(ld), NB, H, W, C, 1, 1)
                assert torch.equal(dx2[..., :C].float(), dx[..., :C].float()), tag
