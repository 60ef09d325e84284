"""Tensor-level wrappers over the C-ABI (torch tensors are only device memory + streams here).

Every function launches on torch's current CUDA stream, allocates outputs with torch, and raises
`SniperError` when the native call fails.  There is no CPU fallback.
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib as _libmod
from ._lib import check, lib

TF32, BF16 = 0, 1
NCHW, NHWC = 0, 1


def reset_launch_count():
    _libmod.launches[0] = 0


def launch_count():
    """GPU kernels launched through the C-ABI since the last reset."""
    return _libmod.launches[0]


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _f32(t):
    assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), "expected contiguous fp32 CUDA tensor"
    return t


def _farr(v):
    a = np.ascontiguousarray(np.asarray(v, dtype=np.float32))
    return a, a.ctypes.data_as(ctypes.c_void_p)


def _iarr(v):
    a = np.ascontiguousarray(np.asarray(v, dtype=np.int32))
    return a, a.ctypes.data_as(ctypes.c_void_p)


def generate_anchors(feat_stride, scales, ratios):
    """multi_proposal_target.cu:75-114 anchor table, [len(ratios)*len(scales), 4] (ratio-major)."""
    s, sp = _farr(scales)
    r, rp = _farr(ratios)
    out = np.zeros((len(r) * len(s), 4), np.float32)
    check(lib().sniper_generate_anchors(int(feat_stride), sp, len(s), rp, len(r), out.ctypes.data_as(ctypes.c_void_p)))
    return out


def multi_proposal(cls_prob, bbox_pred, im_info, *, feat_stride=16, scales=(2, 4, 7, 10, 13, 16, 24),
                   ratios=(0.5, 1, 2), rpn_pre_nms_top_n=12000, rpn_post_nms_top_n=300, threshold=0.7,
                   suppress_anchor_types=False, fast_nms=False, roi_iou_thresh=0.3, layout=NCHW, return_keep=False):
    """MultiProposal forward -- the inference proposal operator (multi_proposal.cc:273-374 semantics: decode, min-size
    filter, the rpn_pre_nms_top_n best anchors, greedy NMS), on device; suppress_anchor_types / fast_nms select the two
    extras of the reference's GPU build (multi_proposal.cu:505-508, 267-387).  Returns rois [B*R,5], scores [B*R]
    (+ keep_idx [B*R] original anchor indices / -1 for filler rows, num_kept [B])."""
    _f32(cls_prob), _f32(bbox_pred), _f32(im_info)
    A = len(scales) * len(ratios)
    if layout == NCHW:
        B, H, W = bbox_pred.shape[0], bbox_pred.shape[2], bbox_pred.shape[3]
        assert bbox_pred.shape[1] == 4 * A and cls_prob.numel() == B * 2 * A * H * W
        sc, dc = 0, 0
    else:
        B, H, W = bbox_pred.shape[0], bbox_pred.shape[1], bbox_pred.shape[2]
        sc, dc = cls_prob.shape[3], bbox_pred.shape[3]
        assert dc >= 4 * A and sc >= 2 * A
    R = int(rpn_post_nms_top_n)
    dev = cls_prob.device
    rois = torch.empty(B * R, 5, device=dev)
    scores = torch.empty(B * R, device=dev)
    keep = torch.empty(B * R, dtype=torch.int32, device=dev) if return_keep else None
    nkept = torch.empty(B, dtype=torch.int32, device=dev) if return_keep else None
    L = lib()
    ws_bytes = L.sniper_multi_proposal_workspace_bytes(B, A, H, W, int(rpn_pre_nms_top_n))
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    s, sp = _farr(scales)
    r, rp = _farr(ratios)
    check(L.sniper_multi_proposal_fwd(
        _ptr(cls_prob), _ptr(bbox_pred), _ptr(im_info), B, A, H, W, int(rpn_pre_nms_top_n), R, int(feat_stride), sp,
        len(s), rp, len(r), float(threshold), (1 if suppress_anchor_types else 0) | (2 if fast_nms else 0),
        float(roi_iou_thresh), layout, sc, dc, _ptr(rois),
        _ptr(scores), _ptr(keep), _ptr(nkept), _ptr(ws), ws_bytes, _stream()))
    if return_keep:
        return rois, scores, keep, nkept
    return rois, scores


def multi_proposal_target(cls_prob, bbox_pred, im_info, gt_boxes, valid_ranges, *, feat_stride=16,
                          scales=(2, 4, 7, 10, 13, 16, 24), ratios=(0.5, 1, 2), rpn_post_nms_top_n=300,
                          threshold=0.7, layout=NCHW, return_keep=False, return_fallback=False):
    """MultiProposalTarget forward (reference GPU-operator semantics, multi_proposal_target.cu:362-589).

    NCHW: cls_prob [B,2A,H,W] (or [B,2,A*H,W]), bbox_pred [B,4A,H,W].  NHWC: [B,H,W,2A] / [B,H,W,4A].
    Returns rois [B*R,5], label [B*R], bbox_target [B*R,4], bbox_weight [B*R,4] (+ keep_idx, num_kept).
    """
    _f32(cls_prob), _f32(bbox_pred), _f32(im_info), _f32(gt_boxes), _f32(valid_ranges)
    A = len(scales) * len(ratios)
    if layout == NCHW:
        B, H, W = bbox_pred.shape[0], bbox_pred.shape[2], bbox_pred.shape[3]
        assert bbox_pred.shape[1] == 4 * A and cls_prob.numel() == B * 2 * A * H * W
        sc, dc = 0, 0
    else:
        B, H, W = bbox_pred.shape[0], bbox_pred.shape[1], bbox_pred.shape[2]
        sc, dc = cls_prob.shape[3], bbox_pred.shape[3]
        assert dc >= 4 * A and sc >= 2 * A
    R = int(rpn_post_nms_top_n)
    max_gt = gt_boxes.shape[1]
    dev = cls_prob.device
    rois = torch.empty(B * R, 5, device=dev)
    label = torch.empty(B * R, device=dev)
    bbox_target = torch.empty(B * R, 4, device=dev)
    bbox_weight = torch.empty(B * R, 4, device=dev)
    keep = torch.empty(B * R, dtype=torch.int32, device=dev) if return_keep else None
    nkept = torch.empty(B, dtype=torch.int32, device=dev) if return_keep else None
    L = lib()
    ws_bytes = L.sniper_multi_proposal_target_workspace_bytes(B, A, H, W)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    s, sp = _farr(scales)
    r, rp = _farr(ratios)
    check(L.sniper_multi_proposal_target_fwd(
        _ptr(cls_prob), _ptr(bbox_pred), _ptr(im_info), _ptr(gt_boxes), _ptr(valid_ranges), B, A, H, W, max_gt, R,
        int(feat_stride), sp, len(s), rp, len(r), float(threshold), layout, sc, dc, _ptr(rois), _ptr(label),
        _ptr(bbox_target), _ptr(bbox_weight), _ptr(keep), _ptr(nkept), _ptr(ws), ws_bytes, _stream()))
    if return_fallback:
        # per-chip flag written by mpt_nms_fast_kernel into the workspace tail (1 = sequential emulation was used)
        off = B * A * H * W * 24 + 64
        fb = ws[off:off + B * 1026 * 4].view(torch.int32)[B * 1025:B * 1026].clone()
        return rois, label, bbox_target, bbox_weight, keep, nkept, fb
    if return_keep:
        return rois, label, bbox_target, bbox_weight, keep, nkept
    return rois, label, bbox_target, bbox_weight


def _ps_dims(data, layout):
    if layout == NCHW:
        B, C, H, W = data.shape
    else:
        B, H, W, C = data.shape
    return B, C, H, W


def deform_psroi_fwd(data, rois, trans, *, spatial_scale, output_dim, group_size, pooled_size, part_size=0,
                     sample_per_part=1, trans_std=0.0, no_trans=False, layout=NCHW, want_count=True,
                     want_sample_idx=False):
    """DeformablePSROIPooling forward (deformable_psroi_pooling.cu:71-161)."""
    _f32(data), _f32(rois)
    B, C, H, W = _ps_dims(data, layout)
    N = rois.shape[0]
    P = pooled_size
    shape = (N, output_dim, P, P) if layout == NCHW else (N, P, P, output_dim)
    out = torch.empty(shape, device=data.device)
    cnt = torch.empty(shape, device=data.device) if want_count else None
    S = sample_per_part
    sidx = torch.empty(N * output_dim * P * P, S * S, 4, dtype=torch.int32, device=data.device) if want_sample_idx else None
    ncls = 1 if no_trans else trans.shape[1] // 2
    if _psroi_tiled(layout, group_size, ncls, C, H, W, S) and not want_sample_idx:
        rc = lib().sniper_deform_psroi_fwd_tiled(_ptr(data), _ptr(rois), _ptr(None if no_trans else _f32(trans)), N, B, C,
                                                 H, W, float(spatial_scale), output_dim, group_size, P, part_size, S,
                                                 float(trans_std), int(no_trans), ncls, _ptr(out), _ptr(cnt), _stream())
        if rc != -2:
            check(rc)
            return out, cnt, sidx
    check(lib().sniper_deform_psroi_fwd(_ptr(data), _ptr(rois), _ptr(None if no_trans else _f32(trans)), N, C, H, W,
                                        float(spatial_scale), output_dim, group_size, P, part_size, S,
                                        float(trans_std), int(no_trans), ncls, layout, _ptr(out), _ptr(cnt),
                                        _ptr(sidx), _stream()))
    return out, cnt, sidx


_psroi_ws = {}


def _psroi_tiled(layout, group_size, ncls, C, H, W, S):
    """True when the chip-tiled PSROI kernels are requested (SNIPER_PSROI_TILED=1) and apply; the library re-checks and
    answers -2 otherwise.  Opt-in: measured 4x SLOWER than the warp-per-bin kernels on B200 (forward 2.0 vs 0.48 ms,
    backward 4.1 vs 0.85 ms per call at 6000 ROIs) -- with one lane per bin the shared-memory accesses of a warp scatter
    over pixels (bank conflicts, CAS-loop float atomics), which costs more than the global gathers / REDs it removes."""
    return (layout == NHWC and group_size == 1 and ncls == 1 and C % 16 == 0 and H * W * 17 * 4 <= 100 * 1024 and S <= 4
            and os.environ.get("SNIPER_PSROI_TILED", "0") == "1" and os.environ.get("SNIPER_PSROI_EXACT") != "1")


def deform_psroi_bwd(top_diff, data, rois, trans, *, spatial_scale, output_dim, group_size, pooled_size,
                     part_size=0, sample_per_part=1, trans_std=0.0, no_trans=False, layout=NCHW,
                     data_diff=None, trans_diff=None):
    """DeformablePSROIPooling backward (deformable_psroi_pooling.cu:203-330); returns (data_diff, trans_diff)."""
    _f32(top_diff), _f32(data), _f32(rois)
    B, C, H, W = _ps_dims(data, layout)
    N = rois.shape[0]
    if data_diff is None:
        data_diff = torch.zeros_like(data)
    if trans_diff is None and not no_trans:
        trans_diff = torch.zeros_like(trans)
    ncls = 1 if no_trans else trans.shape[1] // 2
    if _psroi_tiled(layout, group_size, ncls, C, H, W, sample_per_part):
        need = int(lib().sniper_deform_psroi_bwd_tiled_workspace_bytes(N, C, pooled_size, int(no_trans)))
        ws = None
        if need:      # caller-owned scratch, kept per device and grown on demand (allocated outside any graph capture
            key = (data.device.index, "psroi_bwd")      # by the first eager step; the captured steps reuse it)
            ws = _psroi_ws.get(key)
            if ws is None or ws.numel() < need:
                ws = _psroi_ws[key] = torch.empty(need, dtype=torch.uint8, device=data.device)
        rc = lib().sniper_deform_psroi_bwd_tiled(_ptr(top_diff), _ptr(data), _ptr(rois), _ptr(None if no_trans else trans),
                                                 N, B, C, H, W, float(spatial_scale), output_dim, group_size, pooled_size,
                                                 part_size, sample_per_part, float(trans_std), int(no_trans), ncls,
                                                 _ptr(data_diff), _ptr(trans_diff), _ptr(ws), 0 if ws is None else ws.numel(),
                                                 _stream())
        if rc != -2:
            check(rc)
            if not no_trans:
                _libmod.launches[0] += 1          # + trans_reduce_kernel (the counting proxy adds one per call)
            return data_diff, trans_diff
    check(lib().sniper_deform_psroi_bwd(_ptr(top_diff), _ptr(data), _ptr(rois), _ptr(None if no_trans else trans), N, C,
                                        H, W, float(spatial_scale), output_dim, group_size, pooled_size, part_size,
                                        sample_per_part, float(trans_std), int(no_trans), ncls, layout,
                                        _ptr(data_diff), _ptr(trans_diff), _stream()))
    return data_diff, trans_diff


def psroi_fwd(data, rois, *, spatial_scale, output_dim, group_size, pooled_size, layout=NCHW, want_bins=False):
    """PSROIPooling forward (psroi_pooling.cu:51-118)."""
    _f32(data), _f32(rois)
    B, C, H, W = _ps_dims(data, layout)
    N, P = rois.shape[0], pooled_size
    shape = (N, output_dim, P, P) if layout == NCHW else (N, P, P, output_dim)
    out = torch.empty(shape, device=data.device)
    bins = torch.empty(N * output_dim * P * P, 4, dtype=torch.int32, device=data.device) if want_bins else None
    check(lib().sniper_psroi_fwd(_ptr(data), _ptr(rois), N, C, H, W, float(spatial_scale), output_dim, group_size, P,
                                 layout, _ptr(out), _ptr(bins), _stream()))
    return out, bins


def psroi_bwd(top_diff, rois, data_shape, *, spatial_scale, output_dim, group_size, pooled_size, layout=NCHW):
    """PSROIPooling backward (psroi_pooling.cu:146-210)."""
    _f32(top_diff), _f32(rois)
    data_diff = torch.zeros(data_shape, device=top_diff.device)
    B, C, H, W = _ps_dims(data_diff, layout)
    check(lib().sniper_psroi_bwd(_ptr(top_diff), _ptr(rois), rois.shape[0], C, H, W, float(spatial_scale), output_dim,
                                 group_size, pooled_size, layout, _ptr(data_diff), _stream()))
    return data_diff


def _dt(t):
    return TF32 if t.dtype == torch.float32 else BF16


_gemm_ws = {}


def _ensure_gemm_workspace(device):
    """The tcgen05 kernel's tail-split scratch is caller-owned (the library never allocates): one zero-filled torch
    buffer per device, registered once and kept alive for the life of the process."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if idx not in _gemm_ws:
        L = lib()
        n = L.sniper_gemm_tail_workspace_bytes()
        buf = torch.zeros(n, dtype=torch.uint8, device=torch.device("cuda", idx))
        check(L.sniper_gemm_set_tail_workspace(buf.data_ptr(), n, idx))
        _gemm_ws[idx] = buf


def gemm_nt(a, b, *, out=None, scale=None, bias=None, residual=None, relu=False, accumulate=False, out_dtype=None,
            stats=None):
    """C[M,N] = epi(A[M,K] @ B[N,K]^T) on tcgen05 tensor cores (fp32 storage -> TF32 math, or bf16 operands with fp32
    accumulation).  The output is fp32 or bf16 (default: the operands' dtype); a residual has the output's dtype."""
    assert a.is_cuda and a.dim() == 2 and b.dim() == 2 and a.shape[1] == b.shape[1] and a.dtype == b.dtype
    assert a.stride(1) == 1 and b.stride(1) == 1
    M, K = a.shape
    N = b.shape[0]
    _ensure_gemm_workspace(a.device)
    if out is None:
        out = torch.empty(M, N, device=a.device, dtype=out_dtype or a.dtype)
    out_bf16 = out.dtype == torch.bfloat16
    assert residual is None or residual.dtype == out.dtype, "bf16 output takes a bf16 residual"
    check(lib().sniper_gemm_nt(_ptr(a), a.stride(0), _ptr(b), b.stride(0), _ptr(out), out.stride(0), M, N, K, _dt(a),
                               _ptr(scale), _ptr(bias), _ptr(residual), 0 if residual is None else residual.stride(0),
                               int(relu), int(accumulate), int(out_bf16), _ptr(stats), _stream()))
    return out


def conv_taps(kh, kw, dil, pad):
    """Tap offsets (dh, dw) in input coordinates for a kh x kw kernel, row-major over (kh, kw)."""
    dh = [i * dil - pad for i in range(kh) for _ in range(kw)]
    dw = [j * dil - pad for _ in range(kh) for j in range(kw)]
    return dh, dw


def conv2d_nhwc(x, w, *, kh, kw, stride=1, dil=1, pad=0, out=None, scale=None, bias=None, residual=None, relu=False,
                accumulate=False, taps=None, out_hw=None, out_map=None, stats=None, out_dtype=None):
    """NHWC implicit-GEMM convolution.  x: [N,H,W,Cin]; w: [Cout, kh*kw*Cin] (tap-major, channel-minor).  fp32 tensors
    run as TF32, bf16 tensors as bf16 (fp32 accumulation); the output (and the residual) may be fp32 or bf16."""
    NB, H, W, Cin = x.shape
    Cout = w.shape[0]
    dh, dw = taps if taps is not None else conv_taps(kh, kw, dil, pad)
    ntaps = len(dh)
    assert w.shape[1] == ntaps * Cin and w.is_contiguous() and x.stride(3) == 1
    x_ld = x.stride(2)
    assert x.stride(1) == W * x_ld and x.stride(0) == H * W * x_ld
    if out_hw is None:
        Ho = (H + 2 * pad - dil * (kh - 1) - 1) // stride + 1
        Wo = (W + 2 * pad - dil * (kw - 1) - 1) // stride + 1
    else:
        Ho, Wo = out_hw
    _ensure_gemm_workspace(x.device)
    if out is None:
        out = torch.empty(NB, Ho, Wo, Cout, device=x.device, dtype=out_dtype or x.dtype)
    assert x.dtype == w.dtype and (residual is None or residual.dtype == out.dtype), "bf16 output takes a bf16 residual"
    oH, oW, os_, ooh, oow = (Ho, Wo, 1, 0, 0) if out_map is None else out_map
    _, dhp = _iarr(dh)
    _, dwp = _iarr(dw)
    check(lib().sniper_conv2d_nhwc(_ptr(x), x_ld, NB, H, W, Cin, _ptr(w), Cout, ntaps, dhp, dwp, stride, Ho, Wo,
                                   _ptr(out), _rows(out)[2], oH, oW, os_, ooh, oow, _dt(x), _ptr(scale), _ptr(bias),
                                   _ptr(residual), 0 if residual is None else _rows(residual)[2], int(relu),
                                   int(accumulate), int(out.dtype == torch.bfloat16), _ptr(stats), _stream()))
    return out


def conv2d_wgrad_nhwc(dy, x, *, kh, kw, stride=1, dil=1, pad=0, dw_out=None, splits=8, taps=None):
    """dW[Cout, kh*kw*Cin] += dY^T * im2col(X).  dy: [N,Ho,Wo,Cout], x: [N,H,W,Cin]."""
    NB, H, W, Cin = x.shape
    _, Ho, Wo, Cout = dy.shape
    dh, dw = taps if taps is not None else conv_taps(kh, kw, dil, pad)
    ntaps = len(dh)
    _ensure_gemm_workspace(x.device)
    assert dy.dtype == x.dtype
    if dw_out is None:
        dw_out = torch.zeros(Cout, ntaps * Cin, device=x.device)
    _, dhp = _iarr(dh)
    _, dwp = _iarr(dw)
    check(lib().sniper_conv2d_wgrad_nhwc(_ptr(dy), dy.stride(2), _ptr(x), x.stride(2), NB, H, W, Cin, Cout, ntaps, dhp,
                                         dwp, stride, Ho, Wo,
                                         _ptr(dw_out), _dt(x), splits, _stream()))
    return dw_out


# ---------------------------------------------------------------------------------------------
# HBM-bound layers ([M, C] views of NHWC tensors; `ld` = row stride in elements)
# ---------------------------------------------------------------------------------------------
def _rows(t):
    """(M, C, ld) of a tensor whose last dim is contiguous and whose leading dims collapse to rows."""
    C = t.shape[-1]
    assert t.stride(-1) == 1
    ld = t.stride(-2) if t.dim() >= 2 else C
    M = t.numel() // C
    return M, C, ld


def _sdt(t):
    """storage dtype code of the C-ABI: 0 = fp32, 1 = bf16"""
    if t.dtype == torch.float32:
        return 0
    assert t.dtype == torch.bfloat16, "activations are fp32 or bf16"
    return 1


def affine_act(x, scale, shift, relu=True, out=None):
    M, C, ldx = _rows(x)
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=x.dtype)
    assert out.dtype == x.dtype
    check(lib().sniper_affine_act(_ptr(x), ldx, _ptr(scale), _ptr(shift), _ptr(out), _rows(out)[2], M, C, int(relu),
                                  _sdt(x), _stream()))
    return out


def cast_rows(x, dtype=None, out=None):
    """out[M,C] = cast(x[M,C]) between fp32 and bf16; x / out may be channel slices (row-strided views)."""
    M, C, ldx = _rows(x)
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=dtype)
    check(lib().sniper_cast_rows(_ptr(x), ldx, _sdt(x), _ptr(out), _rows(out)[2], _sdt(out), M, C, _stream()))
    return out


class BNPool:
    """One device allocation for the state of every BatchNorm of a model (filled by ONE H2D copy instead of ~9 fill
    kernels per layer): per layer 6 float vectors [gamma? beta? moving_mean moving_var mean invstd scale shift] and a
    double[2C] statistics scratch."""

    def __init__(self, total_channels, device):
        self.device = device
        self.f = torch.zeros(8 * total_channels)         # host side until finalize()
        self.d_len = 4 * total_channels
        self.fo = 0
        self.do = 0
        self.pending = []

    def take(self, C, ones=False):
        o = self.fo
        self.fo += (C + 3) // 4 * 4          # keep every vector 16-byte aligned
        if ones:
            self.f[o:o + C] = 1.0
        return o

    def take_sums(self, C):
        o = self.do
        self.do += 2 * C
        return o

    def finalize(self):
        self.f = self.f[:max(self.fo, 1)].to(self.device)
        self.d = torch.zeros(max(self.do, 1), dtype=torch.float64, device=self.device)
        for fn in self.pending:
            fn()
        self.pending = []


class BNState:
    """Per-BN device state: parameters, moving statistics and the per-step (mean, invstd, scale, shift)."""

    def __init__(self, C, device, gamma=None, beta=None, dgamma=None, dbeta=None, pool=None):
        self.C = C
        self.dgamma, self.dbeta = dgamma, dbeta
        if pool is None:
            z = lambda: torch.zeros(C, device=device)
            self.gamma = gamma if gamma is not None else torch.ones(C, device=device)
            self.beta = beta if beta is not None else z()
            self.moving_mean, self.moving_var = z(), torch.ones(C, device=device)
            self.mean, self.invstd, self.scale, self.shift = z(), z(), z(), z()
            self.sums = torch.zeros(2 * C, dtype=torch.float64, device=device)
            self.sums_f = torch.zeros(2 * C, dtype=torch.float64, device=device)
            return
        og = pool.take(C, ones=True) if gamma is None else None
        ob = pool.take(C) if beta is None else None
        om, ov = pool.take(C), pool.take(C, ones=True)
        rest = [pool.take(C) for _ in range(4)]
        osum = pool.take_sums(C)
        osum_f = pool.take_sums(C)

        def bind():
            v = lambda o: pool.f[o:o + C]
            self.gamma = gamma if gamma is not None else v(og)
            self.beta = beta if beta is not None else v(ob)
            self.moving_mean, self.moving_var = v(om), v(ov)
            self.mean, self.invstd, self.scale, self.shift = [v(o) for o in rest]
            self.sums = pool.d[osum:osum + 2 * C]
            self.sums_f = pool.d[osum_f:osum_f + 2 * C]       # forward statistics accumulated by the producing conv
        pool.pending.append(bind)


def bn_stats(x, bn, eps=2e-5, momentum=0.9, fix_gamma=False, update_moving=True):
    """Train-mode BatchNorm statistics of x -> bn.(mean, invstd, scale, shift) (+ moving stats)."""
    M, C, ldx = _rows(x)
    check(lib().sniper_bn_stats(_ptr(x), ldx, M, C, _ptr(bn.gamma), _ptr(bn.beta), float(eps), float(momentum),
                                int(fix_gamma), _ptr(bn.moving_mean if update_moving else None),
                                _ptr(bn.moving_var if update_moving else None), _ptr(bn.sums), _ptr(bn.mean),
                                _ptr(bn.invstd), _ptr(bn.scale), _ptr(bn.shift), _sdt(x), _stream()))


def bn_finalize(bn, M, eps=2e-5, momentum=0.9, fix_gamma=False, update_moving=True):
    """Same as bn_stats when bn.sums was already accumulated by the producing conv's epilogue (stats=bn.sums)."""
    check(lib().sniper_bn_finalize(_ptr(bn.sums), M, bn.C, _ptr(bn.gamma), _ptr(bn.beta), float(eps), float(momentum),
                                   int(fix_gamma), _ptr(bn.moving_mean if update_moving else None),
                                   _ptr(bn.moving_var if update_moving else None), _ptr(bn.mean), _ptr(bn.invstd),
                                   _ptr(bn.scale), _ptr(bn.shift), _stream()))


def bn_apply_train(x, bn, eps=2e-5, momentum=0.9, relu=True, fix_gamma=False, update_moving=True, out=None):
    """relu?(bn_train(x)) when the statistics of x already sit in bn.sums_f (accumulated by the producing conv's
    epilogue): finalisation + apply in one launch.  bn.sums_f is left as is -- it is cleared by bn_param_grad_batched."""
    M, C, ldx = _rows(x)
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=x.dtype)
    check(lib().sniper_bn_apply_train(_ptr(x), ldx, _ptr(bn.sums_f), M, C, _ptr(bn.gamma), _ptr(bn.beta), float(eps),
                                      float(momentum), int(fix_gamma), _ptr(bn.moving_mean if update_moving else None),
                                      _ptr(bn.moving_var if update_moving else None), _ptr(bn.mean), _ptr(bn.invstd),
                                      _ptr(bn.scale), _ptr(bn.shift), _ptr(out), _rows(out)[2], int(relu), _sdt(x),
                                      _stream()))
    return out


def bn_frozen(bn, eps=2e-5, fix_gamma=False):
    check(lib().sniper_bn_frozen(bn.C, _ptr(bn.gamma), _ptr(bn.beta), _ptr(bn.moving_mean), _ptr(bn.moving_var),
                                 float(eps), int(fix_gamma), _ptr(bn.scale), _ptr(bn.shift), _stream()))


def bn_relu_bwd(x, dy, bn, add=None, out=None, defer=False):
    """Backward of relu(bn_train(x)); accumulates bn.dgamma / bn.dbeta; returns dx (+ add).
    defer=True leaves (s1, s2) in bn.sums for one bn_param_grad_batched call at the end of the backward pass."""
    M, C, ldx = _rows(x)
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=x.dtype)
    assert dy.dtype == x.dtype and out.dtype == x.dtype and (add is None or add.dtype == x.dtype)
    check(lib().sniper_bn_relu_bwd(_ptr(x), ldx, _ptr(dy), _rows(dy)[2], _ptr(bn.scale), _ptr(bn.shift), _ptr(bn.mean),
                                   _ptr(bn.invstd), _ptr(bn.sums), _ptr(add), 0 if add is None else _rows(add)[2],
                                   _ptr(out), _rows(out)[2], None if defer else _ptr(bn.dgamma),
                                   None if defer else _ptr(bn.dbeta), M, C, _sdt(x), _stream()))
    return out


def bn_act_bwd(x, dy, bn, act, add=None, out=None, defer=False):
    """Backward of act(bn_train(x)), act 1 = ReLU, 2 = clip(y, 0, 6), 3 = none; otherwise as bn_relu_bwd."""
    M, C, ldx = _rows(x)
    if out is None:
        out = torch.empty(x.shape, device=x.device, dtype=x.dtype)
    assert dy.dtype == x.dtype and out.dtype == x.dtype and (add is None or add.dtype == x.dtype)
    check(lib().sniper_bn_act_bwd(_ptr(x), ldx, _ptr(dy), _rows(dy)[2], _ptr(bn.scale), _ptr(bn.shift), _ptr(bn.mean),
                                  _ptr(bn.invstd), _ptr(bn.sums), _ptr(add), 0 if add is None else _rows(add)[2],
                                  _ptr(out), _rows(out)[2], None if defer else _ptr(bn.dgamma),
                                  None if defer else _ptr(bn.dbeta), M, C, int(act), _sdt(x), _stream()))
    return out


def affine_relu_bwd(x, dy, scale, shift, add=None, relu=True, out=None):
    M, C, ldx = _rows(x)
    if out is None:
        out = torch.empty(x.shape, device=x.device)
    check(lib().sniper_affine_relu_bwd(_ptr(x), ldx, _ptr(dy), _rows(dy)[2], _ptr(scale), _ptr(shift), _ptr(add),
                                       0 if add is None else _rows(add)[2], _ptr(out), _rows(out)[2], M, C, int(relu),
                                       _stream()))
    return out


def relu_bwd(y, dy, out=None):
    M, C, ldy = _rows(y)
    if out is None:
        out = torch.empty(y.shape, device=y.device, dtype=y.dtype)
    assert dy.dtype == y.dtype and out.dtype == y.dtype
    check(lib().sniper_relu_bwd(_ptr(y), ldy, _ptr(dy), _rows(dy)[2], _ptr(out), _rows(out)[2], M, C, _sdt(y), _stream()))
    return out


def maxpool3x3s2(x):
    NB, H, W, C = x.shape
    y = torch.empty(NB, (H - 1) // 2 + 1, (W - 1) // 2 + 1, C, device=x.device, dtype=x.dtype)
    check(lib().sniper_maxpool3x3s2_nhwc(_ptr(x), _ptr(y), NB, H, W, C, _sdt(x), _stream()))
    return y


def stem_conv(x_nchw, w, in_scale, in_shift, out_scale, out_shift, out_dtype=torch.float32):
    """bn_data -> conv0 7x7/2 pad 3 -> bn0 -> relu; NCHW fp32 in, NHWC out (fp32 or bf16).  w: [64,7,7,3]."""
    NB, C, H, W = x_nchw.shape
    assert C == 3 and w.shape == (64, 7, 7, 3)
    y = torch.empty(NB, (H - 1) // 2 + 1, (W - 1) // 2 + 1, 64, device=x_nchw.device, dtype=out_dtype)
    check(lib().sniper_stem_conv(_ptr(x_nchw), _ptr(w), _ptr(in_scale), _ptr(in_shift), _ptr(out_scale),
                                 _ptr(out_shift), _ptr(y), NB, H, W, _sdt(y), _stream()))
    return y


def stem_rows(w, dtype=torch.float32):
    """conv0 weights [64,7,7,3] -> the B operand of the tensor-core stem: [64, Kp] rows in (kh, kw, c) order, zero-padded
    to the MMA's K granularity (160 fp32 / 192 bf16)."""
    Kp = 160 if dtype == torch.float32 else 192
    rows = torch.zeros(64, Kp, device=w.device, dtype=torch.float32)
    rows[:, :147] = w.reshape(64, 147)
    return rows.to(dtype)


def stem_conv_tc(x_nchw, rows, in_scale, in_shift, out_scale, out_shift, out_dtype=torch.float32):
    """The stem on the tensor cores: im2col of bn_data(x) (sniper_stem_im2col) + tcgen05 GEMM with bn0 + ReLU in the
    epilogue.  rows = stem_rows(conv0_w, dtype): fp32 rows run as TF32, bf16 rows as bf16 (fp32 accumulation)."""
    NB, C, H, W = x_nchw.shape
    assert C == 3 and rows.shape[0] == 64
    Ho, Wo, Kp = (H - 1) // 2 + 1, (W - 1) // 2 + 1, rows.shape[1]
    col = torch.empty(NB * Ho * Wo, Kp, device=x_nchw.device, dtype=rows.dtype)
    check(lib().sniper_stem_im2col(_ptr(x_nchw), _ptr(in_scale), _ptr(in_shift), _ptr(col), NB, H, W, Kp, _sdt(col),
                                   _stream()))
    y = gemm_nt(col, rows, scale=out_scale, bias=out_shift, relu=True, out_dtype=out_dtype)
    return y.view(NB, Ho, Wo, 64)


def weight_transpose(w, Cout, T, Cin, sel_dev, out=None):
    """w [Cout,T,Cin] -> [Cin, len(sel), Cout] with out[ci,j,co] = w[co, sel[j], ci] (data-gradient operand)."""
    Tsel = sel_dev.numel()
    if out is None:
        out = torch.empty(Cin, Tsel * Cout, device=w.device)
    check(lib().sniper_weight_transpose(_ptr(w), _ptr(out), Cout, T, Cin, Tsel, _ptr(sel_dev), _stream()))
    return out


def weight_transpose_jobs(jobs, device):
    """jobs: list of (w fp32, wt fp32|bf16, sel_dev, Cout, T, Cin).  Returns the device job table for
    weight_transpose_batched."""
    rows, b0 = [], 0
    for w, wt, sel, Cout, T, Cin in jobs:
        Tsel = sel.numel()
        assert w.dtype == torch.float32
        rows.append([w.data_ptr(), wt.data_ptr(), sel.data_ptr(), Cout, T, Cin, Tsel, b0, _sdt(wt)])
        b0 += ((Cin + 31) // 32) * ((Cout + 31) // 32) * Tsel
    return torch.tensor(rows, dtype=torch.int64, device=device), len(rows), b0


def weight_transpose_batched(table):
    t, n, blocks = table
    check(lib().sniper_weight_transpose_batched(_ptr(t), n, blocks, _stream()))


def bn_param_grad_jobs(states, device):
    """states: BNState objects whose backward ran with defer=True."""
    rows = [[b.sums.data_ptr(), 0 if b.dgamma is None else b.dgamma.data_ptr(),
             0 if b.dbeta is None else b.dbeta.data_ptr(), b.C, b.sums_f.data_ptr()] for b in states]
    return torch.tensor(rows, dtype=torch.int64, device=device), len(rows)


def bn_param_grad_batched(table):
    t, n = table
    check(lib().sniper_bn_param_grad_batched(_ptr(t), n, _stream()))


def colsum_accum(x, out):
    M, C, ldx = _rows(x)
    check(lib().sniper_colsum(_ptr(x), ldx, M, C, _ptr(out), _stream()))
    return out


def sgd_mom(w, mom, g, lr, wd, momentum, rescale=1.0):
    check(lib().sniper_sgd_mom(_ptr(w), _ptr(mom), _ptr(g), w.numel(), float(lr), float(wd), float(momentum),
                               float(rescale), _stream()))


def sgd_mom_dev(w, mom, g, hyper, lr_mult, wd_mult, momentum, rescale=1.0, w_bf16=None):
    """SGD-momentum with lr / wd read from the device buffer `hyper` = [lr, wd] (graph-replay safe schedule);
    w_bf16: optional bf16 shadow of the updated weights (multi_precision, optimizer_op-inl.h:377-404)."""
    check(lib().sniper_sgd_mom_dev(_ptr(w), _ptr(mom), _ptr(g), w.numel(), _ptr(hyper), float(lr_mult), float(wd_mult),
                                   float(momentum), float(rescale), _ptr(w_bf16), _stream()))


def count_valid(label, out, ignore=-1):
    check(lib().sniper_count_valid(_ptr(label), label.numel(), int(ignore), _ptr(out), _stream()))


def rpn_softmax_loss(score, label, A, grad_scale, valid_cnt, prob, dscore, loss_sum):
    """score/prob/dscore: NHWC [B,H,W,>=2A]; label [B, A*H*W] in (a,h,w) order."""
    B, H, W, _ = score.shape
    ld = score.stride(2)
    check(lib().sniper_rpn_softmax_loss(_ptr(score), ld, _ptr(label), B, H, W, A, float(grad_scale), _ptr(valid_cnt),
                                        _ptr(prob), prob.stride(2), _ptr(dscore), 0 if dscore is None else dscore.stride(2),
                                        _ptr(loss_sum), _stream()))


def rpn_smooth_l1_loss(pred, target, weight, C4, grad_scale, dpred, loss_sum):
    B, H, W, _ = pred.shape
    check(lib().sniper_rpn_smooth_l1_loss(_ptr(pred), pred.stride(2), _ptr(target), _ptr(weight), B, H, W, C4,
                                          float(grad_scale), _ptr(dpred), dpred.stride(2), _ptr(loss_sum), _stream()))


def softmax_ce(logits, label, K, grad_scale, valid_cnt, prob, grad, loss_sum, ignore=-1):
    N, ld = logits.shape[0], logits.stride(0)
    check(lib().sniper_softmax_ce(_ptr(logits), ld, _ptr(label), N, K, int(ignore), float(grad_scale), _ptr(valid_cnt),
                                  _ptr(prob), 0 if prob is None else prob.stride(0), _ptr(grad),
                                  0 if grad is None else grad.stride(0), _ptr(loss_sum), _stream()))


def smooth_l1_loss(pred, target, weight, C, grad_scale, grad, loss_sum):
    N, ld = pred.shape[0], pred.stride(0)
    check(lib().sniper_smooth_l1_loss(_ptr(pred), ld, _ptr(target), _ptr(weight), N, C, float(grad_scale), _ptr(grad),
                                      grad.stride(0), _ptr(loss_sum), _stream()))


def focus_head(x3, w, b, label, grad_scale, valid_cnt, prob, dx3, dw, db, stats):
    """AutoFocus FocusPixel head, forward + backward in one launch.  x3: conv_new_3_relu [..., 256] fp32 rows (M rows);
    w / b: conv_new_out weight [>=2, 256] / bias [>=2] (rows 0, 1 used); label: scale_label [M] (or [B, H*W]) in
    {-1, 0, 1}; valid_cnt: device int32 count of labels != -1.  Writes prob [M, 2] and dx3 (the gradient of conv_new_3's
    PRE-activation: the ReLU mask is applied); accumulates dw rows 0..1, db[0..1], and stats[0..2] += (sum of -log p,
    correct count, valid count)."""
    C = x3.shape[-1]
    M = x3.numel() // C
    assert x3.is_contiguous() and dx3.is_contiguous() and prob.is_contiguous() and w.is_contiguous()
    assert x3.dtype == w.dtype == dx3.dtype == prob.dtype == torch.float32 and w.shape[-1] == C and label.numel() == M
    assert prob.numel() == 2 * M and dx3.shape == x3.shape
    check(lib().sniper_focus_head(_ptr(x3), M, C, _ptr(w), _ptr(b), _ptr(label), float(grad_scale), _ptr(valid_cnt),
                                  _ptr(prob), _ptr(dx3), _ptr(dw), _ptr(db), _ptr(stats), _stream()))


def focus_label(boxes, offsets, B, *, H=32, W=32, feat_stride=16, dc_low=5, small_thresh=64, dc_high=90, out=None):
    """FocusPixel labels (gen_mask, data_workers.py:165-192): boxes [N,4] fp32 device (every chip's GT after shift /
    scale / round / clip, chip-major, in GT order), offsets int32 [B+1] device -> scale_label [B, H*W] fp32 in {-1, 0, 1}."""
    assert boxes.dtype == torch.float32 and boxes.is_contiguous() and offsets.dtype == torch.int32
    if out is None:
        out = torch.empty(B, H * W, device=offsets.device)
    check(lib().sniper_focus_label(_ptr(boxes), _ptr(offsets), int(B), int(H), int(W), int(feat_stride), float(dc_low),
                                   float(small_thresh), float(dc_high), _ptr(out), _stream()))
    return out


def deform_im2col(x, offset, *, kh=3, kw=3, stride=1, dil=1, pad=1, dgroups=4, out=None):
    """Bilinear-sampled im2col (deformable_im2col.cuh:216-263): x [N,H,W,C], offset [N,Ho,Wo,>=dg*2*kh*kw]
    -> col [N*Ho*Wo, kh*kw*C] (tap-major)."""
    NB, H, W, C = x.shape
    Ho = (H + 2 * pad - dil * (kh - 1) - 1) // stride + 1
    Wo = (W + 2 * pad - dil * (kw - 1) - 1) // stride + 1
    if out is None:
        out = torch.empty(NB * Ho * Wo, kh * kw * C, device=x.device, dtype=x.dtype)
    assert x.is_contiguous() and offset.dtype == torch.float32 and out.dtype == x.dtype
    check(lib().sniper_deform_im2col(_ptr(x), _ptr(offset), NB, H, W, C, kh, kw, stride, dil, pad, dgroups,
                                     offset.stride(2), _ptr(out), _sdt(x), _stream()))
    return out


def deform_col2im(dcol, x, offset, *, kh=3, kw=3, stride=1, dil=1, pad=1, dgroups=4, dx=None, doffset=None):
    """Transposes of deform_im2col: dx (accumulated, always fp32) and doffset (fp32)
    (deformable_im2col.cuh:317-360, 419-480).  dcol / x: fp32 or bf16."""
    NB, H, W, C = x.shape
    if dx is None:
        dx = torch.zeros(x.shape, device=x.device)
    if doffset is None:
        doffset = torch.zeros_like(offset)
    assert dcol.dtype == x.dtype and dx.dtype == torch.float32 and doffset.dtype == torch.float32
    check(lib().sniper_deform_col2im(_ptr(dcol), _ptr(x), _ptr(offset), NB, H, W, C, kh, kw, stride, dil, pad, dgroups,
                                     offset.stride(2), _ptr(dx), _ptr(doffset), _sdt(x), _stream()))
    return dx, doffset


def anchor_target(gt_valid, ngt, gt_invalid, ninv, im_info, *, H=32, W=32, feat_stride=16,
                  scales=(2, 4, 7, 10, 13, 16, 24), ratios=(0.5, 1, 2), pos_thresh=0.5, neg_thresh=0.4, disable=None,
                  want_argmax=False):
    """RPN anchor matching of anchor_worker.worker (data_workers.py:194-363) for a whole chip batch.
    gt_valid [B,G,4] / gt_invalid [B,Gi,4] float32 (first ngt[b] / ninv[b] rows used, int32 counts),
    disable: optional uint8 [B,H*W*A] (the host's npr.choice subsampling).  Returns label [B,A*H*W],
    bbox_target, bbox_weight [B,4A,H,W] (+ argmax [B,H*W*A])."""
    B, G = gt_valid.shape[0], gt_valid.shape[1]
    Gi = gt_invalid.shape[1]
    A = len(scales) * len(ratios)
    dev = gt_valid.device
    label = torch.empty(B, A * H * W, device=dev)
    bt = torch.empty(B, 4 * A, H, W, device=dev)
    bw = torch.empty(B, 4 * A, H, W, device=dev)
    am = torch.empty(B, H * W * A, dtype=torch.int32, device=dev) if want_argmax else None
    scratch = torch.zeros(B * max(G, 1), dtype=torch.int64, device=dev)
    s, sp = _farr(scales)
    r, rp = _farr(ratios)
    check(lib().sniper_anchor_target(_ptr(gt_valid), _ptr(ngt), G, _ptr(gt_invalid), _ptr(ninv), Gi, _ptr(im_info),
                                     _ptr(disable), B, H, W, int(feat_stride), sp, len(s), rp, len(r), float(pos_thresh),
                                     float(neg_thresh), _ptr(scratch), _ptr(label), _ptr(bt), _ptr(bw), _ptr(am),
                                     _stream()))
    return (label, bt, bw, am) if want_argmax else (label, bt, bw)


def soft_nms_batched(dets, offsets, *, sigma=0.55, Nt=0.3, threshold=0.001, method=2):
    """cpu_soft_nms (lib/nms/cpu_nms.pyx:17-110) on every segment dets[offsets[p]:offsets[p+1]] ([.,5] rows x1,y1,x2,y2,score)
    at once.  Returns (dets_out, counts): the first counts[p] rows of segment p are its surviving detections in the
    reference's output order; `dets` itself is not modified."""
    assert dets.is_cuda and dets.dtype == torch.float32 and dets.dim() == 2 and dets.shape[1] == 5 and dets.is_contiguous()
    assert offsets.dtype == torch.int32 and offsets.is_cuda
    P = offsets.numel() - 1
    out = dets.clone()
    counts = torch.zeros(max(P, 1), dtype=torch.int32, device=dets.device)
    scratch = torch.empty_like(dets)
    check(lib().sniper_soft_nms_batched(_ptr(out), _ptr(offsets), P, float(sigma), float(Nt), float(threshold), int(method),
                                        _ptr(counts), _ptr(scratch), _stream()))
    return out, counts[:P]


# ---------------------------------------------------------------------------------------------
# MobileNetV2 layers (symbols/faster/mobilenetv2_e2e.py): depthwise 3x3, first-layer im2col, shortcut add
# ---------------------------------------------------------------------------------------------
def depthwise3x3(x, w, stride=1, out=None):
    """x: [N,H,W,C] (fp32 | bf16), w: [9,C] fp32 tap-major -> [N,Ho,Wo,C]; pad 1."""
    NB, H, W, C = x.shape
    assert w.shape == (9, C) and w.dtype == torch.float32 and w.is_contiguous() and x.stride(3) == 1
    ldx = x.stride(2)
    assert x.stride(1) == W * ldx and x.stride(0) == H * W * ldx
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    if out is None:
        out = torch.empty(NB, Ho, Wo, C, device=x.device, dtype=x.dtype)
    assert out.dtype == x.dtype and out.shape == (NB, Ho, Wo, C)
    check(lib().sniper_depthwise3x3_fwd(_ptr(x), ldx, _ptr(w), _ptr(out), out.stride(2), NB, H, W, C, stride, _sdt(x),
                                        _stream()))
    return out


def depthwise3x3_dgrad(dy, w, in_hw, stride=1, out=None):
    """dx [N,H,W,C] of depthwise3x3 for dy [N,Ho,Wo,C]."""
    NB, Ho, Wo, C = dy.shape
    H, W = in_hw
    assert (H - 1) // stride + 1 == Ho and (W - 1) // stride + 1 == Wo and dy.is_contiguous()
    if out is None:
        out = torch.empty(NB, H, W, C, device=dy.device, dtype=dy.dtype)
    check(lib().sniper_depthwise3x3_dgrad(_ptr(dy), dy.stride(2), _ptr(w), _ptr(out), out.stride(2), NB, H, W, C, stride,
                                          _sdt(dy), _stream()))
    return out


def depthwise3x3_wgrad(x, dy, dw, stride=1):
    """dw[9,C] (fp32) += correlation of dy with the shifted input."""
    NB, H, W, C = x.shape
    assert dw.shape == (9, C) and dw.dtype == torch.float32 and dw.is_contiguous() and x.dtype == dy.dtype
    assert x.is_contiguous() and dy.is_contiguous()
    check(lib().sniper_depthwise3x3_wgrad(_ptr(x), x.stride(2), _ptr(dy), dy.stride(2), _ptr(dw), NB, H, W, C, stride,
                                          _sdt(x), _stream()))
    return dw


def im2col3x3s2(x_nchw, Kp, dtype=torch.float32, out=None):
    """[N,3,H,W] fp32 -> [N,Ho,Wo,Kp] rows of the first layer's 3x3 / stride-2 patches, K order (kh, kw, ci)."""
    NB, Cin, H, W = x_nchw.shape
    assert x_nchw.dtype == torch.float32 and x_nchw.is_contiguous()
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    if out is None:
        out = torch.empty(NB, Ho, Wo, Kp, device=x_nchw.device, dtype=dtype)
    check(lib().sniper_im2col3x3s2_nchw(_ptr(x_nchw), _ptr(out), NB, H, W, Cin, Kp, _sdt(out), _stream()))
    return out


def add_rows(a, b, out=None):
    M, C, lda = _rows(a)
    if out is None:
        out = torch.empty(a.shape, device=a.device, dtype=a.dtype)
    assert a.dtype == b.dtype == out.dtype and a.shape == b.shape
    check(lib().sniper_add_rows(_ptr(a), lda, _ptr(b), _rows(b)[2], _ptr(out), _rows(out)[2], M, C, _sdt(a), _stream()))
    return out
