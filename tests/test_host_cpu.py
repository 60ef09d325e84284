"""Host-side ops of the path vs the reference's own compiled code (oracle/_ref) and the CPU oracle.
No GPU, no compute kernels: runs in the CPU test tier."""
import os
import re
import sys

import numpy as np
import pytest

import oracle_lib as O
import ref_golden as G
from sniper_b200 import _lib, host, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_header_matches_library_and_bindings():
    hdr = open(os.path.join(ROOT, "include", "sniper_b200.h")).read()
    protos = re.findall(r"\n(?:int|size_t|const char\*)\s+(sniper_\w+)\s*\(([^;]*)\);", hdr)
    assert len(protos) >= 30
    L = _lib.lib()
    for name, args in protos:
        assert hasattr(L, name), "library does not export " + name
        assert name in _lib.SIGNATURES, "no ctypes signature for " + name
        plist = [] if args.strip() == "void" else [a.strip() for a in args.split(",")]
        codes = ""
        for a in plist:
            if "*" in a:
                codes += "p"
            else:
                ty = a.rsplit(" ", 1)[0].strip()
                codes += {"int": "i", "long": "l", "float": "f", "double": "d", "size_t": "z", "unsigned": "u"}[ty]
        assert codes == _lib.SIGNATURES[name][1], "%s: header %s vs ctypes %s" % (name, codes, _lib.SIGNATURES[name][1])
    for name in _lib.SIGNATURES:
        assert any(n == name for n, _ in protos), name + " missing from the header"
    assert L.sniper_abi_version() == 2


def _config1_boxes(seed, n, W=1333, H=800):
    """SURVEY 8d config 1 generator: sqrt(area) log-uniform in [8,400], aspect in [0.5,2]."""
    rng = np.random.RandomState(seed)
    s = np.exp(rng.uniform(np.log(8), np.log(400), n))
    ar = np.exp(rng.uniform(np.log(0.5), np.log(2.0), n))
    w, h = s * np.sqrt(ar), s / np.sqrt(ar)
    cx, cy = rng.uniform(0, W, n), rng.uniform(0, H, n)
    b = np.stack([np.clip(cx - w / 2, 0, W - 1), np.clip(cy - h / 2, 0, H - 1), np.clip(cx + w / 2, 0, W - 1),
                  np.clip(cy + h / 2, 0, H - 1)], 1)
    return b.astype(np.float32)


def _ref_chips_generate(boxes, W, H, size, stride, seed):
    """The reference's lib/chips/cchips.cpp (oracle/_ref/libref_chips.so), or its stored outputs where it is not built."""
    run = None if O.ref_chips() is None else lambda: O.ref_chips_generate(boxes, W, H, size, stride, seed=seed)
    return G.reference("host_cpu.chips_generate", (boxes, W, H, size, stride, seed), run)


@pytest.mark.parametrize("scale,stride,seed", [(3.0, 58, 1), (1.667, 56, 2), (0.8, 59, 3), (0.384, 57, 4)])
def test_chips_generate_matches_reference_cchips(scale, stride, seed):
    # config 1: one 1333x800 image, 20 GT + proposals, chip 512; reference lib/chips/cchips.cpp compiled as-is
    gt = _config1_boxes(0, 20)
    props = _config1_boxes(1, 400)
    boxes = np.concatenate([gt, props]) * np.float32(scale)
    W, H = int(1333 * scale), int(800 * scale)
    boxes[:, [0, 2]] = np.clip(boxes[:, [0, 2]], 0, W - 1)
    boxes[:, [1, 3]] = np.clip(boxes[:, [1, 3]], 0, H - 1)
    ref = _ref_chips_generate(boxes, W, H, 512, stride, seed)
    host.srand(seed)
    ours = host.chips_generate(boxes, W, H, 512, stride)
    assert ours.shape == ref.shape and ours.tobytes() == ref.tobytes()      # chip indices: bit-exact
    assert len(ours) > 0
    # every box that fits into some candidate chip is covered by a returned chip
    ov = host.ignore_overlaps(ours.astype(np.float64), boxes.astype(np.float64))
    assert (ov.max(0) == 1).sum() > 0


def test_chips_empty_and_tiny_image():
    assert host.chips_generate(np.zeros((0, 4), np.float32), 600, 400, 512, 32).shape == (0, 4)
    b = np.array([[10, 10, 50, 60]], np.float32)
    host.srand(1)
    c = host.chips_generate(b, 300, 200, 512, 32)      # image smaller than a chip: corner chips only
    np.testing.assert_array_equal(c, _ref_chips_generate(b, 300, 200, 512, 32, 1))
    assert len(c) == 1


def test_cpu_nms_and_soft_nms_match_oracle():
    rng = np.random.RandomState(2)
    boxes = _config1_boxes(5, 6000)
    dets = np.concatenate([boxes, rng.rand(6000, 1).astype(np.float32)], 1).astype(np.float32)
    keep = host.cpu_nms(dets, 0.7)
    np.testing.assert_array_equal(np.array(keep, np.int32), O.cpu_nms(dets, 0.7))
    assert 0 < len(keep) < 6000
    d2 = dets[:1500].copy()
    out = host.cpu_soft_nms(d2, sigma=0.55).copy()
    ref = O.cpu_soft_nms(dets[:1500], sigma=0.55)
    assert out.tobytes() == ref.tobytes()
    # ties: default order = stable descending
    dets[:, 4] = np.round(dets[:, 4] * 8) / 8
    k2 = host.cpu_nms(dets, 0.5, order=None)
    assert len(k2) > 0
    assert host.cpu_nms(np.zeros((0, 5), np.float32), 0.5) == []


def test_bbox_overlaps_match_oracle():
    a = _config1_boxes(7, 200).astype(np.float64)
    b = _config1_boxes(8, 50).astype(np.float64)
    assert host.bbox_overlaps(a, b).tobytes() == O.bbox_overlaps(a, b).tobytes()
    assert host.ignore_overlaps(a, b).tobytes() == O.bbox_overlaps(a, b, ignore=True).tobytes()


def test_product_path_fails_loudly_without_library(monkeypatch):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libsniper_b200.so")
    with pytest.raises(RuntimeError):
        _lib.lib()


def test_gemm_launch_plan_host_logic():
    """sniper_gemm_plan (host only): tile width, ring depth, persistent grid and tail split of the tcgen05 kernel for the
    shapes of the training step.  out = {block_n, stages, staging bufs, tiles, grid, tail mode, first tail tile, factor}."""
    import ctypes
    from sniper_b200 import _lib
    L = _lib.lib()

    def plan(M, N, K, dtype=0):
        out = (ctypes.c_int * 8)()
        _lib.check(L.sniper_gemm_plan(M, N, K, dtype, ctypes.cast(out, ctypes.c_void_p)))
        return list(out)
    # conv2 of a stage-3 unit: 160 tiles of 128 x 256 on 148 SMs -> the 12 tail tiles are cut into 4 column pieces
    bn, stages, stg, tiles, grid, mode, first, factor = plan(20480, 256, 2304)
    assert (bn, tiles, grid, mode, first, factor) == (256, 160, 148, 2, 148, 4) and stages == 4 and stg == 1
    # conv3 (K = 256): short K -> two staging buffers, one ring stage less; 640 tiles -> 48 tail tiles x 2 pieces
    bn, stages, stg, tiles, grid, mode, first, factor = plan(20480, 1024, 256)
    assert (bn, stg, stages, tiles, mode, first, factor) == (256, 2, 3, 640, 2, 592, 2)
    # fc_offset: 47 tiles of 128 x 128 < 148 SMs, long K -> K-slices (3 per tile)
    bn, stages, stg, tiles, grid, mode, first, factor = plan(6000, 128, 12544)
    assert (bn, tiles, mode, first, factor) == (128, 47, 1, 0, 3) and grid == 141
    # a multiple of the grid, a single tile, a ragged N (direct epilogue): no tail split
    assert plan(148 * 128, 256, 512)[5] == 0
    assert plan(128, 64, 64)[3:6] == [1, 1, 0]
    assert plan(20480, 72, 4608)[5] == 0
    # K-slices only where the fitted cost model predicts a gain (K = 1024 is too short for 128-wide tiles)
    assert plan(6000, 128, 1024)[5] == 0
    with pytest.raises(_lib.SniperError):
        plan(128, 128, 100)


# ---------------------------------------------------------------------------------------------------------------
# Pinning against the reference's OWN Cython host code (lib/nms/cpu_nms.pyx, lib/bbox/bbox.pyx), compiled from
# the reference tree by oracle/build_ref_cython.py into oracle/_ref (4 dead tokens rewritten on the fly, see that
# file); where they are not built, their stored outputs (tests/ref_golden.py).
# ---------------------------------------------------------------------------------------------------------------
def _ref_cython(module, fn, *args, **kw):
    """module.fn(*args, **kw) of the reference's Cython code built into oracle/_ref, or its stored outputs where it is
    not built."""
    import importlib
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    try:
        mod = importlib.import_module(module)
    except ImportError:
        mod = None

    def run():
        return np.asarray(getattr(mod, fn)(*[np.copy(a) if isinstance(a, np.ndarray) else a for a in args], **kw))
    return G.reference("host_cpu.%s.%s" % (module, fn), (args, kw), None if mod is None else run)


@pytest.mark.parametrize("seed,n,thresh", [(0, 600, 0.7), (1, 2000, 0.5), (2, 50, 0.3)])
def test_cpu_nms_matches_reference_cython(seed, n, thresh):
    rng = np.random.RandomState(seed)
    rois = synth.rois_for_pool(rng, n, 1)
    dets = np.concatenate([rois[:, 1:], rng.permutation(n).reshape(-1, 1) / float(n)], 1).astype(np.float32)   # tie-free
    want = [int(i) for i in _ref_cython("ref_cpu_nms", "cpu_nms", dets, thresh)]
    assert host.cpu_nms(dets, thresh) == want                       # product (libsniper_b200.so, host_ops.cpp)
    assert O.cpu_nms(dets, thresh).tolist() == want                 # oracle (oracle/host.c)
    assert 0 < len(want) < n


@pytest.mark.parametrize("method,sigma,Nt", [(2, 0.55, 0.3), (1, 0.5, 0.3), (0, 0.5, 0.45)])
def test_cpu_soft_nms_matches_reference_cython(method, sigma, Nt):
    """Gaussian (SNIPER's setting sigma 0.55, yml:225), linear and hard variants: same surviving rows in the same
    order; scores bit-identical for linear / hard, within 1 ulp for the Gaussian (the reference calls np.exp on a
    float32 scalar, the restatements double exp)."""
    rng = np.random.RandomState(7 + method)
    n = 400
    rois = synth.rois_for_pool(rng, n, 1)
    boxes = np.concatenate([rois[:, 1:], (rng.permutation(n).reshape(-1, 1) + 1.0) / (n + 1.0)], 1).astype(np.float32)
    want = _ref_cython("ref_cpu_nms", "cpu_soft_nms", boxes, sigma=sigma, Nt=Nt, threshold=0.001, method=method)
    got = host.cpu_soft_nms(boxes.copy(), sigma=sigma, Nt=Nt, threshold=0.001, method=method)
    orc = O.cpu_soft_nms(boxes.copy(), sigma=sigma, Nt=Nt, threshold=0.001, method=method)
    assert got.shape == want.shape and orc.shape == want.shape and 0 < want.shape[0] <= n
    assert np.array_equal(got[:, :4], want[:, :4]) and np.array_equal(orc[:, :4], want[:, :4])
    if method == 2:
        assert np.abs(got[:, 4] - want[:, 4]).max() <= 2e-7 and np.abs(orc[:, 4] - want[:, 4]).max() <= 2e-7
    else:
        assert np.array_equal(got[:, 4], want[:, 4]) and np.array_equal(orc[:, 4], want[:, 4])


def test_bbox_overlaps_match_reference_cython():
    rng = np.random.RandomState(3)
    a = synth.rois_for_pool(rng, 300, 1)[:, 1:].astype(np.float64)
    b = synth.rois_for_pool(rng, 80, 1)[:, 1:].astype(np.float64)
    want = _ref_cython("ref_bbox", "bbox_overlaps_cython", a, b)
    assert np.array_equal(host.bbox_overlaps(a, b), want) and np.array_equal(O.bbox_overlaps(a, b), want)
    want_i = _ref_cython("ref_bbox", "ignore_overlaps_cython", a, b)
    assert np.array_equal(host.ignore_overlaps(a, b), want_i) and np.array_equal(O.bbox_overlaps(a, b, ignore=True), want_i)
    assert (want > 0).sum() > 100
