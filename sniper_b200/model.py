"""ResNet-101 SNIPER Faster-R-CNN / R-FCN training graph on the sm_100a kernels (NHWC, explicit backward).

Mirrors symbols/faster/resnet_mx_101_e2e.py of the reference layer by layer (names are the reference's
parameter names so checkpoints map one to one):
  resnetc4        :394-420   residual_unit :36-69
  resnetc5        :422-448   residual_unit_deform :106-145
  get_rpn         :147-155   get_symbol_rcnn (is_train) :227-345   init_weight_rcnn :450-485
The forward/backward order is fixed at construction (no graph executor, no autograd): every method below
is a sequence of C-ABI launches on the current CUDA stream, so one training step can be captured into a CUDA
graph.  Frozen layers (conv0, bn0, stage1 -- FIXED_PARAMS, sniper_res101_e2e.yml:22-25 -- and bn_data) run
forward only.
"""
import math
import os

import numpy as np
import torch

from . import ops

SCALES = (2, 4, 7, 10, 13, 16, 24)
RATIOS = (0.5, 1, 2)


class Cfg:
    """The slice of configs/faster/sniper_res101_e2e.yml the training graph reads."""
    num_classes = 81
    num_anchors = 21
    feat_stride = 16
    scales = SCALES
    ratios = RATIOS
    rpn_post_nms_top_n = 300          # multi_proposal_target-inl.h:70
    rpn_batch_size = 256              # TRAIN.RPN_BATCH_SIZE
    batch_images = 16                 # TRAIN.BATCH_IMAGES (per GPU)
    bn_eps = 2e-5
    bn_momentum = 0.995               # main_train.py:27
    lr = 0.015                        # TRAIN.lr .. warmup_step: sniper_res101_e2e.yml:104-111
    lr_step = "5.33"
    lr_factor = 0.1
    warmup = True
    warmup_lr = 0.0005
    warmup_step = 1000
    wd = 1e-4
    momentum = 0.9
    units = (3, 4, 23, 3)
    filter_list = (64, 256, 512, 1024, 2048)
    grad_scale = 1.0                  # TRAIN.scale only applies to fp16 (bf16 has fp32's exponent range: no loss scale)
    # Mixed precision (BASELINE config 3; the reference's TRAIN.fp16, sniper_res101_e2e.yml:107): the backbone from the
    # output of conv0 to the concat stores activations, weights and gradients of activations in bf16 (the reference:
    # fp16 between the two Casts, resnet_mx_101_e2e.py:405-406 and :250-252), BatchNorm arithmetic and statistics stay
    # fp32, the RPN / R-FCN heads stay fp32 (TF32 math) exactly where the reference keeps them fp32, and the optimizer
    # keeps fp32 master weights + momentum and rewrites the bf16 copies every step (multi_precision SGD).
    bf16 = os.environ.get("SNIPER_BF16", "0") == "1"
    wgrad_splits = 0                  # 0 = choose per layer (fill one wave of 148 persistent CTAs)
    # BN statistics accumulated by the producing conv's TMA-store epilogue (column sums of the staged chunk + double
    # REDs) instead of a separate colsum pass.  Measured on B200: 39.1 -> 37.8 ms/step, so ON by default
    # (SNIPER_FUSE_BN=0 restores the separate pass for A/B runs).
    fuse_bn_stats = os.environ.get("SNIPER_FUSE_BN", "1") == "1"
    # run weight gradients on a second stream (see WgradScheduler); SNIPER_WGRAD_STREAM=0/1 overrides for A/B runs
    wgrad_stream = os.environ.get("SNIPER_WGRAD_STREAM", "1") == "1"
    # AutoFocus training (TRAIN.AUTO_FOCUS, sniper_res101_e2e_autofocus.yml:106-119): the FocusPixel branch conv_new_2 ->
    # conv_new_3 -> conv_new_out is part of the trained graph, fed by batch["scale_label"] (cls_scale_prob loss)
    autofocus = False


# ------------------------------------------------------------------------------------------------
class WgradScheduler:
    """Weight gradients are off the critical path of the backward pass (nothing but the optimizer reads them), so
    they can run on a second stream next to the HBM-bound BatchNorm / elementwise kernels of the data-gradient
    chain.  fork() makes the side stream wait for everything enqueued so far on the main stream, join() makes the
    main stream wait for the side stream; tensors handed to the side stream are kept alive until join()."""

    def __init__(self, enabled):
        self.enabled = enabled
        self.side = None
        self.keep = []

    def __call__(self, fn, *args):
        if not self.enabled:
            return fn(*args)
        if self.side is None:
            self.side = torch.cuda.Stream()
        main = torch.cuda.current_stream()
        self.side.wait_stream(main)
        self.keep.append(args)
        with torch.cuda.stream(self.side):
            fn(*args)

    def join(self):
        if self.enabled and self.side is not None:
            torch.cuda.current_stream().wait_stream(self.side)
        self.keep = []


# ------------------------------------------------------------------------------------------------
class ParamStore:
    """All trainable parameters in ONE flat fp32 buffer (+ grad, + momentum): one NCCL all-reduce and one
    fused SGD launch per optimizer group per step (replaces ~330 per-key kvstore push/pull pairs,
    SNIPER-mxnet/python/mxnet/model.py:126-136).  Groups = (lr_mult, wd_mult) as MXNet derives them:
    wd_mult 0 for names not ending in _weight/_gamma, lr_mult from the symbol attribute (offset: 0.01)."""

    def __init__(self):
        self.specs = []   # (name, shape, group)
        self.views = {}
        self.grads = {}

    bucket = 0      # set by the model while it registers parameters: gradients of one bucket are complete at the same
                    # point of the backward pass and form one contiguous all-reduce (0 = heads + stage 4, 1 = stage 3, ...)

    def add(self, name, shape, lr_mult=1.0):
        wd_mult = 1.0 if (name.endswith("_weight") or name.endswith("_gamma")) else 0.0
        self.specs.append((name, tuple(shape), (self.bucket, lr_mult, wd_mult)))

    def finalize(self, device, lowp=False):
        """lowp: also keep a bf16 copy of the whole buffer (`w16`, same offsets) for the mixed-precision backbone."""
        groups = sorted(set(g for _, _, g in self.specs))      # bucket-major: each bucket is one contiguous range
        off = 0
        self.segments = []
        self.bucket_ranges = []
        layout = {}
        for g in groups:
            start = off
            for name, shape, gg in self.specs:
                if gg != g:
                    continue
                n = int(np.prod(shape))
                layout[name] = (off, shape)
                off += (n + 3) // 4 * 4          # keep every tensor 16-byte aligned
            self.segments.append((start, off, g[1:]))
            b = g[0]
            while len(self.bucket_ranges) <= b:
                self.bucket_ranges.append([start, start])
            self.bucket_ranges[b][0] = min(self.bucket_ranges[b][0], start) if self.bucket_ranges[b][1] > self.bucket_ranges[b][0] else start
            self.bucket_ranges[b][1] = off
        self.total = off
        self.w = torch.zeros(off, device=device)
        self.g = torch.zeros(off, device=device)
        self.mom = torch.zeros(off, device=device)
        # [lr, wd] on the device: read by sgd_mom_dev_kernel, so a captured update graph follows the LR schedule
        self.hyper = torch.zeros(2, device=device)
        self._hyper_host = (None, None)
        self.w16 = torch.zeros(off, device=device, dtype=torch.bfloat16) if lowp else None
        self.views16 = {}
        for name, (o, shape) in layout.items():
            n = int(np.prod(shape))
            self.views[name] = self.w[o:o + n].view(shape)
            self.grads[name] = self.g[o:o + n].view(shape)
            if lowp:
                self.views16[name] = self.w16[o:o + n].view(shape)
        self.layout = layout

    def sync_lowp(self):
        """bf16 copies := round(fp32 masters); after initialisation / checkpoint loading (the update kernel keeps them
        in step afterwards)."""
        if self.w16 is not None:
            self.w16.copy_(self.w)

    def __getitem__(self, name):
        return self.views[name]

    def grad(self, name):
        return self.grads[name]

    def set_hyper(self, lr, wd):
        """Stream-ordered 8-byte H2D of (lr, wd); call OUTSIDE graph capture (the captured update only reads it)."""
        if (lr, wd) != self._hyper_host:
            self.hyper.copy_(torch.tensor([lr, wd], dtype=torch.float32))
            self._hyper_host = (lr, wd)

    def sgd_step(self, momentum, rescale=1.0):
        """optimizer_op-inl.h:279-300 on every (lr_mult, wd_mult) segment, lr / wd taken from self.hyper."""
        for s, e, (lr_mult, wd_mult) in self.segments:
            ops.sgd_mom_dev(self.w[s:e], self.mom[s:e], self.g[s:e], self.hyper, lr_mult, wd_mult, momentum, rescale,
                            None if self.w16 is None else self.w16[s:e])


# ------------------------------------------------------------------------------------------------
class Conv:
    """NHWC convolution with weights [Cout, kh*kw*Cin] (tap-major), optional bias; data/weight gradients on
    the tcgen05 kernels.  Cout is padded up to `cout_pad` with zero rows where the reference's channel
    count (72, 126, 85, 98) is not a multiple of 32."""

    def __init__(self, P, name, cin, cout, k=1, stride=1, dil=1, pad=0, bias=False, trainable=True, cout_pad=None,
                 lr_mult=1.0, need_dgrad=True, plain_wt=False, lowp=False):
        """lowp: this layer reads bf16 activations -> bf16 weights (the ParamStore's bf16 copy; fp32 master + gradient)."""
        self.lowp = lowp
        self.wdtype = torch.bfloat16 if lowp else torch.float32
        self.name, self.cin, self.cout, self.k = name, cin, cout, k
        self.stride, self.dil, self.pad, self.bias = stride, dil, pad, bias
        self.coutp = cout_pad or cout
        self.trainable, self.need_dgrad, self.plain_wt = trainable, need_dgrad, plain_wt
        self.K = k * k * cin
        self.P = P
        if trainable:
            P.add(name + "_weight", (self.coutp, self.K), lr_mult)
            if bias:
                P.add(name + "_bias", (self.coutp,), lr_mult)
        self.wt = None
        self.frozen_w = None
        self.frozen_b = None

    # ---- parameters
    @property
    def w(self):
        """the operand the kernels read: bf16 copy for a mixed-precision layer, else the fp32 parameter"""
        if not self.trainable:
            return self.frozen_w
        return self.P.views16[self.name + "_weight"] if self.lowp else self.P[self.name + "_weight"]

    @property
    def master(self):
        """the fp32 parameter the optimizer updates (frozen layers: the stored weight itself)"""
        return self.P[self.name + "_weight"] if self.trainable else self.frozen_w

    @property
    def b(self):
        if not self.bias:
            return None
        return self.P[self.name + "_bias"] if self.trainable else self.frozen_b

    def init(self, std=None, device=None, gen=None):
        shape = (self.coutp, self.K)
        if std is None:
            std = math.sqrt(2.0 / self.K)      # He-normal backbone (SURVEY 8d config 2)
        w = torch.zeros(shape, device=device)
        if std > 0:
            w[:self.cout].normal_(0, std, generator=gen)
        if self.trainable:
            self.master.copy_(w)
            if self.lowp:
                self.w.copy_(w)
            if self.bias:
                self.b.zero_()
        else:
            self.frozen_w = w.to(self.wdtype)
            if self.bias:
                self.frozen_b = torch.zeros(self.coutp, device=device)

    # ---- forward
    def fwd(self, x, out=None, scale=None, shift=None, relu=False, residual=None, stats=None, out_dtype=None):
        """y = epi(conv(x)); epilogue order: *scale, +shift (or +bias), +residual, relu; `stats` (a BN's
        double[2C] scratch) receives the column sums of y for the consumer's train-mode statistics."""
        add = shift if shift is not None else self.b
        return ops.conv2d_nhwc(x, self.w, kh=self.k, kw=self.k, stride=self.stride, dil=self.dil, pad=self.pad, out=out,
                               scale=scale, bias=add, residual=residual, relu=relu, stats=stats, out_dtype=out_dtype)

    # ---- backward
    def bwd_jobs(self):
        """Re-layout jobs of the (just updated) weights for the data gradient, [Cin, taps', Cout]: a list of
        (w, wt, sel, Cout, T, Cin) for ops.weight_transpose_jobs (all of them run as ONE launch per step)."""
        if not (self.trainable and self.need_dgrad):
            return []
        dev = self.w.device
        k, T = self.k, self.k * self.k
        if self.plain_wt:
            # plain 2-D transpose [Cout, K] -> [K, Cout] (deformable conv: the GEMM runs on the im2col buffer)
            if getattr(self, "_sel", None) is None:
                self._sel = torch.zeros(1, dtype=torch.int32, device=dev)
                self.wt = torch.empty(self.K, self.coutp, device=dev, dtype=self.wdtype)
            return [(self.master, self.wt, self._sel, self.coutp, 1, self.K)]
        if self.stride == 1 or k == 1:
            sel = list(range(T - 1, -1, -1))
            if getattr(self, "_sel", None) is None:
                self._sel = torch.tensor(sel, dtype=torch.int32, device=dev)
                self.wt = torch.empty(self.cin, T * self.coutp, device=dev, dtype=self.wdtype)
            return [(self.master, self.wt, self._sel, self.coutp, T, self.cin)]
        # stride 2, 3x3, pad 1: four output-parity classes, each a stride-1 conv over dY
        assert k == 3 and self.stride == 2 and self.pad == 1 and self.dil == 1
        if getattr(self, "_sel", None) is None:
            self._sel, self.wt, self._taps = [], [], []
            for ph in (0, 1):
                for pw in (0, 1):
                    khs = [1] if ph == 0 else [0, 2]
                    kws = [1] if pw == 0 else [0, 2]
                    sel = [kh * 3 + kw for kh in khs for kw in kws]
                    dh = [(ph + 1 - kh) // 2 for kh in khs for _ in kws]
                    dw = [(pw + 1 - kw) // 2 for _ in khs for kw in kws]
                    self._sel.append(torch.tensor(sel, dtype=torch.int32, device=dev))
                    self.wt.append(torch.empty(self.cin, len(sel) * self.coutp, device=dev, dtype=self.wdtype))
                    self._taps.append((dh, dw, ph, pw))
        return [(self.master, w, s, self.coutp, 9, self.cin) for s, w in zip(self._sel, self.wt)]

    def prepare_bwd(self):
        """Rebuilds this layer's data-gradient operands from the fp32 master weights (one small batched launch; the
        model does it for all layers at once)."""
        jobs = self.bwd_jobs()
        if jobs:
            ops.weight_transpose_batched(ops.weight_transpose_jobs(jobs, jobs[0][0].device))

    def bwd_data(self, dy, in_hw, out=None, residual=None):
        """dX = conv^T(dY).  dy: [N,Ho,Wo,coutp]; returns [N,H,W,Cin] (+ residual)."""
        NB = dy.shape[0]
        H, W = in_hw
        k = self.k
        if self.stride == 1:
            padb = self.dil * (k - 1) - self.pad
            return ops.conv2d_nhwc(dy, self.wt, kh=k, kw=k, stride=1, dil=self.dil, pad=padb, out=out, residual=residual)
        if out is None:
            out = torch.zeros(NB, H, W, self.cin, device=dy.device, dtype=dy.dtype) if residual is None else residual
        Ho, Wo = dy.shape[1], dy.shape[2]
        if k == 1:
            # dX[2a, 2b] = dY[a,b] * W ; other positions receive nothing
            return ops.conv2d_nhwc(dy, self.wt, kh=1, kw=1, out=out, residual=residual if residual is not None else None,
                                   out_hw=(Ho, Wo), out_map=(H, W, 2, 0, 0))
        for wt, (dh, dw, ph, pw) in zip(self.wt, self._taps):
            ops.conv2d_nhwc(dy, wt, kh=0, kw=0, taps=(dh, dw), out=out, residual=residual if residual is not None else None,
                            out_hw=(H // 2, W // 2), out_map=(H, W, 2, ph, pw))
        return out

    def bwd_weight(self, dy, x, splits=8, dy32=None):
        """dy32: fp32 form of dy for the bias gradient when dy itself is bf16 (the bias-gradient kernel reads fp32)."""
        gw = self.P.grad(self.name + "_weight")
        ops.conv2d_wgrad_nhwc(dy, x, kh=self.k, kw=self.k, stride=self.stride, dil=self.dil, pad=self.pad, dw_out=gw,
                              splits=splits)
        if self.bias:
            ops.colsum_accum(dy if dy32 is None else dy32, self.P.grad(self.name + "_bias"))


class BN:
    """BatchNorm + ReLU.  train: batch statistics over this GPU's chips (README.md:10); frozen: moving stats."""

    def __init__(self, P, name, C, frozen, fix_gamma=False):
        self.name, self.C, self.frozen, self.fix_gamma = name, C, frozen, fix_gamma
        self.P = P
        if not frozen:
            P.add(name + "_gamma", (C,))
            P.add(name + "_beta", (C,))
        self.st = None

    def build(self, device, pool=None):
        """pool: an ops.BNPool shared by all layers of a model (one allocation, one H2D); gamma of a trainable layer is
        then initialised by the caller in the flat parameter buffer."""
        if self.frozen:
            self.st = ops.BNState(self.C, device, pool=pool)
        else:
            self.st = ops.BNState(self.C, device, self.P[self.name + "_gamma"], self.P[self.name + "_beta"],
                                  self.P.grad(self.name + "_gamma"), self.P.grad(self.name + "_beta"), pool=pool)
            if pool is None:
                self.st.gamma.fill_(1.0)

    def fwd(self, x, cfg, relu=True, have_stats=False):
        """have_stats: the producer of x already accumulated sum / sum-of-squares into self.st.sums."""
        if self.frozen:
            return ops.affine_act(x, self.st.scale, self.st.shift, relu=relu)
        if have_stats and self.fused_apply:
            return ops.bn_apply_train(x, self.st, eps=cfg.bn_eps, momentum=cfg.bn_momentum, relu=relu)
        if have_stats:
            ops.bn_finalize(self.st, x.numel() // self.C, eps=cfg.bn_eps, momentum=cfg.bn_momentum)
        else:
            ops.bn_stats(x, self.st, eps=cfg.bn_eps, momentum=cfg.bn_momentum)
        return ops.affine_act(x, self.st.scale, self.st.shift, relu=relu)

    fuse = False   # set from Cfg.fuse_bn_stats by SniperResNet101

    fused_apply = False   # set per instance by SniperResNet101: statistics go to st.sums_f and the finalisation rides in
                          # the apply kernel (sums_f is cleared by the end-of-step bn_param_grad_batched launch)

    def stats_sink(self):
        """The scratch a producer may accumulate this BN's input statistics into (None: compute them here)."""
        if self.frozen or not BN.fuse:
            return None
        return self.st.sums_f if self.fused_apply else self.st.sums

    defer = False   # set per instance by SniperResNet101: dgamma/dbeta of all layers by one bn_param_grad_batched launch

    def bwd(self, x, dy, add=None):
        return ops.bn_relu_bwd(x, dy, self.st, add=add, defer=self.defer)


# ------------------------------------------------------------------------------------------------
class Unit:
    """Pre-activation bottleneck (residual_unit :36-69 / residual_unit_deform :106-145)."""

    def __init__(self, P, name, cin, cout, stride, dim_match, frozen, deform=False, first_trainable=False, lowp=False):
        mid = cout // 4
        self.name, self.cin, self.cout, self.mid = name, cin, cout, mid
        self.stride, self.dim_match, self.frozen, self.deform = stride, dim_match, frozen, deform
        self.lowp = lowp
        t = not frozen
        self.bn1 = BN(P, name + "_bn1", cin, frozen)
        self.conv1 = Conv(P, name + "_conv1", cin, mid, 1, trainable=t, lowp=lowp)
        self.bn2 = BN(P, name + "_bn2", mid, frozen)
        if deform:
            # 72 offset channels, zero-padded to a width the MMA / TMA tiles accept (bf16 weight gradients: x64)
            self.offset = Conv(P, name + "_offset", mid, 72, 3, 1, 2, 2, bias=True, cout_pad=128 if lowp else 96, lowp=lowp)
            self.conv2 = Conv(P, name + "_conv2", mid, mid, 3, 1, 2, 2, trainable=t, plain_wt=True, lowp=lowp)
        else:
            self.conv2 = Conv(P, name + "_conv2", mid, mid, 3, stride, 1, 1, trainable=t, lowp=lowp)
        self.bn3 = BN(P, name + "_bn3", mid, frozen)
        self.conv3 = Conv(P, name + "_conv3", mid, cout, 1, trainable=t, lowp=lowp)
        self.sc = None if dim_match else Conv(P, name + "_sc", cin, cout, 1, stride, trainable=t, lowp=lowp)
        self.first_trainable = first_trainable
        self.saved = None

    def convs(self):
        cs = [self.conv1, self.conv2, self.conv3]
        if self.sc is not None:
            cs.append(self.sc)
        if self.deform:
            cs.append(self.offset)
        return cs

    def bns(self):
        return [self.bn1, self.bn2, self.bn3]

    def fwd(self, x, cfg, out=None, x_has_stats=False, next_bn=None):
        """x_has_stats: the producer of x already accumulated bn1's statistics; next_bn: the BN that consumes
        this unit's output (its statistics are accumulated by conv3's epilogue)."""
        sink = next_bn.stats_sink() if next_bn is not None else None
        if self.frozen:
            a1 = self.bn1.fwd(x, cfg)
            a2 = self.conv1.fwd(a1, scale=self.bn2.st.scale, shift=self.bn2.st.shift, relu=True)
            a3 = self.conv2.fwd(a2, scale=self.bn3.st.scale, shift=self.bn3.st.shift, relu=True)
            res = x if self.dim_match else self.sc.fwd(a1)
            return self.conv3.fwd(a3, out=out, residual=res, stats=sink)
        fused = BN.fuse
        a1 = self.bn1.fwd(x, cfg, have_stats=x_has_stats and fused)
        c1 = self.conv1.fwd(a1, stats=self.bn2.stats_sink())
        a2 = self.bn2.fwd(c1, cfg, have_stats=fused)
        if self.deform:
            off = self.offset.fwd(a2, out_dtype=torch.float32)                 # [N,H,W,96] fp32, 72 used
            col = ops.deform_im2col(a2, off, kh=3, kw=3, stride=1, dil=2, pad=2, dgroups=4)
            c2 = ops.gemm_nt(col, self.conv2.w, stats=self.bn3.stats_sink())
            c2 = c2.view(a2.shape[0], a2.shape[1], a2.shape[2], self.mid)
        else:
            off = col = None
            c2 = self.conv2.fwd(a2, stats=self.bn3.stats_sink())
        a3 = self.bn3.fwd(c2, cfg, have_stats=fused)
        res = x if self.dim_match else self.sc.fwd(a1)
        y = self.conv3.fwd(a3, out=out, residual=res, stats=sink)
        self.saved = (x, a1, c1, a2, c2, a3, off, col)
        return y

    def fwd_infer(self, x, cfg, out=None):
        """Inference forward (is_train=False: every BatchNorm uses its moving statistics, resnet_mx_101_e2e.py:36-69 with
        use_global_stats): BN + ReLU ride in the producing conv's epilogue as per-channel scale/shift."""
        a1 = ops.affine_act(x, self.bn1.st.scale, self.bn1.st.shift, relu=True)
        a2 = self.conv1.fwd(a1, scale=self.bn2.st.scale, shift=self.bn2.st.shift, relu=True)
        if self.deform:
            off = self.offset.fwd(a2, out_dtype=torch.float32)
            col = ops.deform_im2col(a2, off, kh=3, kw=3, stride=1, dil=2, pad=2, dgroups=4)
            a3 = ops.gemm_nt(col, self.conv2.w, scale=self.bn3.st.scale, bias=self.bn3.st.shift, relu=True)
            a3 = a3.view(a2.shape[0], a2.shape[1], a2.shape[2], self.mid)
        else:
            a3 = self.conv2.fwd(a2, scale=self.bn3.st.scale, shift=self.bn3.st.shift, relu=True)
        res = x if self.dim_match else self.sc.fwd(a1)
        return self.conv3.fwd(a3, out=out, residual=res)

    def bwd(self, dout, cfg, extra_add=None):
        """dout: grad of the unit output [N,Ho,Wo,cout] (may be a channel slice).  Returns grad of the input
        (+ extra_add, used to merge the c4 half of the concat gradient into stage4_unit1's input gradient)."""
        x, a1, c1, a2, c2, a3, off, col = self.saved
        sp = cfg.wgrad_splits
        W = cfg.wsched
        hw_in = (x.shape[1], x.shape[2])
        hw_mid = (c2.shape[1], c2.shape[2])
        W(self.conv3.bwd_weight, dout, a3, sp)
        da3 = self.conv3.bwd_data(dout, hw_mid)
        dc2 = self.bn3.bwd(c2, da3)
        if self.deform:
            M = dc2.numel() // self.mid
            gw = self.conv2.P.grad(self.conv2.name + "_weight")
            W(lambda d, c: ops.conv2d_wgrad_nhwc(d, c, kh=1, kw=1, dw_out=gw, splits=sp), dc2,
              col.view(a2.shape[0], a2.shape[1], a2.shape[2], -1))
            dcol = ops.gemm_nt(dc2.view(M, self.mid), self.conv2.wt)         # wt = W^T [9*mid, mid]
            da2, doff = ops.deform_col2im(dcol, a2, off, kh=3, kw=3, stride=1, dil=2, pad=2, dgroups=4)   # fp32 sums
            if self.lowp:
                doff16 = ops.cast_rows(doff, torch.bfloat16)
                da2 = ops.cast_rows(da2, torch.bfloat16)
                W(self.offset.bwd_weight, doff16, a2, sp, doff)
                da2 = self.offset.bwd_data(doff16, (a2.shape[1], a2.shape[2]), out=da2, residual=da2)
            else:
                W(self.offset.bwd_weight, doff, a2, sp)
                da2 = self.offset.bwd_data(doff, (a2.shape[1], a2.shape[2]), out=da2, residual=da2)
        else:
            W(self.conv2.bwd_weight, dc2, a2, sp)
            da2 = self.conv2.bwd_data(dc2, (a2.shape[1], a2.shape[2]))
        dc1 = self.bn2.bwd(c1, da2)
        W(self.conv1.bwd_weight, dc1, a1, sp)
        if self.sc is not None:
            W(self.sc.bwd_weight, dout, a1, sp)
        da1 = self.conv1.bwd_data(dc1, hw_in)
        if self.sc is not None:
            da1 = self.sc.bwd_data(dout, hw_in, out=da1, residual=da1)
        # (for the first trainable unit dx itself is unused -- its input comes from the frozen stage -- but
        #  bn1's gamma/beta gradients are produced by the same pass)
        dx = self.bn1.bwd(x, da1, add=dout if self.dim_match else extra_add)
        self.saved = None
        return None if self.first_trainable else dx


# ------------------------------------------------------------------------------------------------
class SniperResNet101:
    """get_symbol_rcnn(cfg, is_train=True) as an executable object (resnet_mx_101_e2e.py:227-345)."""

    def __init__(self, cfg=None, device="cuda", seed=5, deform_offset_std=0.0):
        self.cfg = cfg or Cfg()
        cfg = self.cfg
        self.device = device
        BN.fuse = bool(cfg.fuse_bn_stats)
        cfg.wsched = WgradScheduler(bool(cfg.wgrad_stream))
        self._wt_table = None
        self._bn_table = None
        P = self.P = ParamStore()
        fl = cfg.filter_list
        # ---- frozen stem: bn_data, conv0, bn0 (resnetc4 :402-408)
        self.bn_data = BN(P, "bn_data", 3, frozen=True, fix_gamma=True)
        self.bn0 = BN(P, "bn0", 64, frozen=True)
        self.conv0_w = None
        # ---- stages
        self.units = []
        cin = fl[0]
        for i, n in enumerate(cfg.units):
            stage = i + 1
            cout = fl[i + 1]
            frozen = (stage == 1)
            # gradient buckets in the order the backward pass completes them: heads + stage 4, stage 3, stage 2
            P.bucket = {4: 0, 3: 1, 2: 2}.get(stage, 2)
            deform = (stage == 4)
            stride = 1 if stage in (1, 4) else 2
            for j in range(n):
                u = Unit(P, "stage%d_unit%d" % (stage, j + 1), cin if j == 0 else cout, cout, stride if j == 0 else 1,
                         dim_match=(j > 0), frozen=frozen, deform=deform, first_trainable=(stage == 2 and j == 0),
                         lowp=bool(cfg.bf16))
                self.units.append(u)
            cin = cout
        A = cfg.num_anchors
        P.bucket = 0
        # ---- heads (get_rpn :147-155, conv_new_1 :256-257, FCs :288-303)
        self.rpn_conv = Conv(P, "rpn_conv_3x3", 3072, 512, 3, 1, 1, 1, bias=True)
        # rpn_bbox_pred (4A) and rpn_cls_score (2A) fused into one 1x1 conv: rows [0,4A) | [4A,6A), padded to 128
        self.rpn_head = Conv(P, "rpn_head", 512, 6 * A, 1, bias=True, cout_pad=128)
        self.conv_new_1 = Conv(P, "conv_new_1", 3072, 256, 1, bias=True)
        self.fc_offset = Conv(P, "offset", 7 * 7 * 256, 98, 1, bias=True, cout_pad=128, lr_mult=0.01)
        self.fc_new_1 = Conv(P, "fc_new_1", 7 * 7 * 256, 1024, 1, bias=True)
        self.fc_new_2 = Conv(P, "fc_new_2", 1024, 1024, 1, bias=True)
        # cls_score (81) and bbox_pred (4) fused: rows [0,81) | [81,85), padded to 96
        self.fc_out = Conv(P, "cls_bbox", 1024, cfg.num_classes + 4, 1, bias=True, cout_pad=96)
        # ---- AutoFocus branch (resnet_mx_101_e2e.py:259-267): trained in bucket 0 after the R-FCN head, fp32 after the
        # Cast in both precisions.  conv_new_out keeps 32 rows (rows 2..31 zero, their gradients too) so that focus_map
        # and forward_inference(autofocus=True) read the trained weights unchanged; sniper_focus_head reads rows 0..1.
        self.af_train = bool(getattr(cfg, "autofocus", False))
        if self.af_train:
            self.conv_new_2 = Conv(P, "conv_new_2", 3072, 256, 3, 1, 1, 1, bias=True)
            self.conv_new_3 = Conv(P, "conv_new_3", 256, 256, 1, bias=True)
            self.conv_new_out = Conv(P, "conv_new_out", 256, 2, 1, bias=True, cout_pad=32, need_dgrad=False)
        P.finalize(device, lowp=bool(cfg.bf16))
        self.act_dtype = torch.bfloat16 if cfg.bf16 else torch.float32
        self._init_weights(seed, deform_offset_std)
        for b in self.train_bns():
            b.fused_apply = bool(cfg.fuse_bn_stats) and os.environ.get("SNIPER_BN_APPLY_FUSED", "1") == "1"
        self.loss_buf = torch.zeros(8, device=device)
        self.cnt_buf = torch.zeros(2, dtype=torch.int32, device=device)
        self.step_count = 0
        self.af = None          # AutoFocus branch (inference): enable_autofocus(), or the trained layers (cfg.autofocus)
        if self.af_train:
            self.af = [self.conv_new_2, self.conv_new_3, self.conv_new_out]
            self.af_cnt = torch.zeros(1, dtype=torch.int32, device=device)

    # ---------------------------------------------------------------- AutoFocus branch (resnet_mx_101_e2e.py:259-267, 385-386)
    def enable_autofocus(self, seed=9, arg=None):
        """conv_new_2 (3x3, 3072 -> 256) + ReLU -> conv_new_3 (1x1) + ReLU -> conv_new_out (1x1 -> 2) on the concat
        feature map; `forward_inference(autofocus=True)` returns its channel softmax, the FocusPixel map of
        `cfg.TEST.AUTO_FOCUS`.  Inference-only here (the AutoFocus training label `scale_label` is not built): the three
        layers live outside the parameter store.  arg: reference-named weights (`conv_new_2_weight` OIHW ...), else
        N(0, 0.01) like init_weight_rcnn (:468-474)."""
        from . import checkpoint as ck
        if self.af_train:
            raise RuntimeError("enable_autofocus(): this network trains the AutoFocus branch (Cfg.autofocus); its weights "
                               "are parameters -- load them with load_reference")
        dev = self.device
        g = torch.Generator()
        g.manual_seed(seed)
        specs = (("conv_new_2", 3072, 256, 3, 1, None), ("conv_new_3", 256, 256, 1, 0, None), ("conv_new_out", 256, 2, 1, 0, 32))
        convs = []
        for name, cin, cout, k, pad, cpad in specs:
            c = Conv(self.P, name, cin, cout, k, pad=pad, bias=True, trainable=False, cout_pad=cpad)
            w = torch.zeros(c.coutp, c.K)
            b = torch.zeros(c.coutp)
            if arg is not None and name + "_weight" in arg:
                w[:cout] = torch.from_numpy(ck.conv_to_rows(np.asarray(arg[name + "_weight"], np.float32)))
                b[:cout] = torch.from_numpy(np.asarray(arg[name + "_bias"], np.float32))
            else:
                w[:cout].normal_(0, 0.01, generator=g)
            c.frozen_w, c.frozen_b = w.to(dev), b.to(dev)
            convs.append(c)
        self.af = convs

    def focus_map(self, cat):
        """scale_prob[:, 1] = softmax over the two channels of conv_new_out: [B, Hf, Wf] probability of 'focus'."""
        c2, c3, co = self.af
        x = c2.fwd(cat, relu=True)
        x = c3.fwd(x, relu=True)
        z = co.fwd(x)[..., :2]
        return torch.softmax(z, dim=-1)[..., 1]

    # ---------------------------------------------------------------- init (init_weight_rcnn :450-485)
    def _init_weights(self, seed, deform_offset_std):
        """Random initialisation generated on the HOST (CPU generator) into one flat image of the parameter buffer and
        moved with a single H2D copy; all BatchNorm state comes from one pooled allocation.  (Per-tensor device fills
        cost ~800 tiny launches at start-up and pushed the real kernels out of the driver's launch window.)"""
        dev = self.device
        g = torch.Generator()
        g.manual_seed(seed)
        cfg = self.cfg
        P = self.P
        host = torch.zeros(P.total)

        def fill(c, std=None):
            if std is None:
                std = math.sqrt(2.0 / c.K)      # He-normal backbone (SURVEY 8d config 2)
            w = torch.zeros(c.coutp, c.K)
            if std > 0:
                w[:c.cout].normal_(0, std, generator=g)
            if c.trainable:
                o, _ = P.layout[c.name + "_weight"]
                host[o:o + w.numel()] = w.view(-1)
            else:
                c.frozen_w = w.to(dev, c.wdtype)
                if c.bias:
                    c.frozen_b = torch.zeros(c.coutp).to(dev)

        self.conv0_w = torch.zeros(64, 7, 7, 3).normal_(0, math.sqrt(2.0 / 147), generator=g).to(dev)
        self._stem_rows = None
        all_bns = [self.bn_data, self.bn0] + [b for u in self.units for b in u.bns()]
        pool = ops.BNPool(sum(b.C for b in all_bns), dev)
        for bn in all_bns:
            bn.build(dev, pool)
            if not bn.frozen:
                o, _ = P.layout[bn.name + "_gamma"]
                host[o:o + bn.C] = 1.0
        for u in self.units:
            for c in u.convs():
                # offset convolutions: zeros in the reference (:451-456)
                fill(c, deform_offset_std if c.name.endswith("_offset") else None)
        for c in (self.rpn_conv, self.rpn_head, self.conv_new_1, self.fc_new_1, self.fc_new_2, self.fc_out):
            fill(c, 0.01)
        fill(self.fc_offset, deform_offset_std and 0.001)                  # zeros in the reference (:476-477)
        if self.af_train:                                                  # N(0, 0.01), zero biases (:468-474)
            for c in (self.conv_new_2, self.conv_new_3, self.conv_new_out):
                fill(c, 0.01)
        P.w.copy_(host)
        P.sync_lowp()
        pool.finalize()
        self.bn_pool = pool
        # bn_data: frozen, fix_gamma; realistic pixel statistics so that conv0 sees O(1) inputs
        self.bn_data.st.moving_var.fill_(60.0 ** 2)
        ops.bn_frozen(self.bn_data.st, cfg.bn_eps, fix_gamma=True)
        for bn in all_bns[1:]:
            if bn.frozen:
                ops.bn_frozen(bn.st, cfg.bn_eps)

    def train_bns(self):
        return [b for u in self.units if not u.frozen for b in u.bns()]

    def trainable_convs(self):
        cs = []
        for u in self.units:
            if not u.frozen:
                cs += u.convs()
        cs += [self.rpn_conv, self.rpn_head, self.conv_new_1, self.fc_offset, self.fc_new_1, self.fc_new_2, self.fc_out]
        if self.af_train:
            cs += [self.conv_new_2, self.conv_new_3, self.conv_new_out]
        return cs

    # ---------------------------------------------------------------- one training step
    def forward_backward(self, batch, on_bucket=None):
        """One forward + backward pass; see fb_phases.  on_bucket(k): called when gradient bucket k (P.bucket_ranges[k])
        is complete -- the eager form of the overlapped all-reduce."""
        out = None
        for k, out in enumerate(self.fb_phases(batch)):
            if on_bucket is not None:
                on_bucket(k)
        return out

    def fb_phases(self, batch):
        """Generator form of the pass, one `yield` per completed gradient bucket (0: forward + heads + stage-4 backward,
        1: stage-3 backward, 2: stage-2 backward), so that the trainer can capture each phase as its own CUDA graph and
        start the bucket's all-reduce while the next phase computes.  Every phase ends with all its kernels (including the
        weight-gradient side stream) joined on the current stream.  Yields the output dict each time.

        batch: dict of device tensors named as MNIteratorE2E provides them (MNIteratorE2E.py:175-219):
        data [B,3,512,512], label [B,A*H*W], bbox_target/bbox_weight [B,4A,H,W], gt_boxes [B,100,5],
        valid_ranges [B,2], im_info [B,3] (+ scale_label [B,H*W] when cfg.autofocus).  Leaves parameter gradients in
        self.P.g and returns the outputs of the reference's Group([rpn_cls_prob, rpn_bbox_loss, cls_prob, bbox_loss, label])
        (:338) as a dict; with cfg.autofocus also cls_scale_prob (Group of :335-336), NHWC [B,H,W,2] like rpn_cls_prob (the
        reference's is (B, 2, H*W)), and loss_buf[4:7] = (focus log-loss sum, correct count, valid count)."""
        cfg = self.cfg
        P = self.P
        A = cfg.num_anchors
        data = batch["data"]
        B = data.shape[0]
        n1, n2, n3, n4 = cfg.units
        P.g.zero_()
        self.loss_buf.zero_()
        self.cnt_buf.zero_()
        if self.af_train:
            self.af_cnt.zero_()
        # weights were updated by the previous step: refresh the data-gradient operands
        if self._wt_table is None:
            jobs = [j for c in self.trainable_convs() for j in c.bwd_jobs()]
            self._wt_table = ops.weight_transpose_jobs(jobs, data.device)
            for b in self.train_bns():
                b.defer = True
            self._bn_tables = []
            for stage_units in (self.units[n1 + n2 + n3:], self.units[n1 + n2:n1 + n2 + n3], self.units[n1:n1 + n2]):
                self._bn_tables.append(ops.bn_param_grad_jobs([b.st for u in stage_units for b in u.bns()], data.device))
        ops.weight_transpose_batched(self._wt_table)

        # ---- backbone forward
        lowp = bool(cfg.bf16)
        x = self.stem(data)                                             # the reference's Cast sits right after conv0
        x = ops.maxpool3x3s2(x)
        Hf = data.shape[2] // cfg.feat_stride
        # Concat(c4, c5): fp32.  fp32 mode: the two producing convs write their channel slices in place.  Mixed
        # precision: c4 / c5 are bf16 tensors and the reference's Cast(relu1, float32) (:250-252) fills the slices.
        cat = torch.empty(B, Hf, Hf, 3072, device=data.device)
        last3 = n1 + n2 + n3 - 1
        has_stats = False
        c4 = None
        for i, u in enumerate(self.units):
            out = None
            if not lowp:
                if i == last3:
                    out = cat[..., :1024]
                elif i == len(self.units) - 1:
                    out = cat[..., 1024:]
            nxt = self.units[i + 1].bn1 if i + 1 < len(self.units) else None
            x = u.fwd(x, cfg, out=out, x_has_stats=has_stats, next_bn=nxt)
            has_stats = nxt is not None and not nxt.frozen
            if i == last3:
                c4 = x
        if lowp:
            ops.cast_rows(c4, out=cat[..., :1024])
            ops.cast_rows(x, out=cat[..., 1024:])

        # ---- RPN (get_rpn) + conv_new_1
        rpn = self.rpn_conv.fwd(cat, relu=True)
        head = self.rpn_head.fwd(rpn)                                      # [B,H,W,128]: 4A deltas | 2A scores
        feat = self.conv_new_1.fwd(cat, relu=True)
        if self.af_train:
            # ---- AutoFocus branch + SoftmaxOutput('cls_scale_prob', multi_output, valid) (:259-267, 313-315): conv_new_out,
            # the loss and its whole backward down to conv_new_3's pre-activation in one launch
            f2 = self.conv_new_2.fwd(cat, relu=True)
            f3 = self.conv_new_3.fwd(f2, relu=True)
            scale_prob = torch.empty(B, Hf, Hf, 2, device=data.device)
            df3 = torch.empty_like(f3)
            ops.count_valid(batch["scale_label"], self.af_cnt)
            ops.focus_head(f3, self.conv_new_out.w, self.conv_new_out.b, batch["scale_label"], cfg.grad_scale, self.af_cnt,
                           scale_prob, df3, P.grad("conv_new_out_weight"), P.grad("conv_new_out_bias"), self.loss_buf[4:7])
        dhead = torch.zeros_like(head)
        prob = torch.empty(B, Hf, Hf, 2 * A, device=data.device)
        ops.count_valid(batch["label"], self.cnt_buf[0:1])
        ops.rpn_softmax_loss(head[..., 4 * A:6 * A], batch["label"], A, cfg.grad_scale, self.cnt_buf[0:1], prob,
                             dhead[..., 4 * A:6 * A], self.loss_buf[0:1])
        ops.rpn_smooth_l1_loss(head, batch["bbox_target"], batch["bbox_weight"], 4 * A,
                               3.0 * cfg.grad_scale / float(cfg.batch_images * cfg.rpn_batch_size), dhead,
                               self.loss_buf[1:2])
        # ---- proposals + targets, all on device
        rois, label, bbox_target, bbox_weight = ops.multi_proposal_target(
            prob, head, batch["im_info"], batch["gt_boxes"], batch["valid_ranges"], feat_stride=cfg.feat_stride,
            scales=cfg.scales, ratios=cfg.ratios, rpn_post_nms_top_n=cfg.rpn_post_nms_top_n, layout=ops.NHWC)
        N = rois.shape[0]
        # ---- R-FCN head
        ps = dict(spatial_scale=1.0 / cfg.feat_stride, output_dim=256, group_size=1, pooled_size=7, part_size=7,
                  sample_per_part=4, layout=ops.NHWC)
        offset_t, _, _ = ops.deform_psroi_fwd(feat, rois, None, no_trans=True, want_count=False, **ps)
        off = ops.gemm_nt(offset_t.view(N, -1), self.fc_offset.w, bias=self.fc_offset.b)          # [N,128], 98 used
        trans = off[:, :98].contiguous().view(N, 2, 7, 7)
        pooled, _, _ = ops.deform_psroi_fwd(feat, rois, trans, no_trans=False, trans_std=0.1, want_count=False, **ps)
        fc1 = ops.gemm_nt(pooled.view(N, -1), self.fc_new_1.w, bias=self.fc_new_1.b, relu=True)
        fc2 = ops.gemm_nt(fc1, self.fc_new_2.w, bias=self.fc_new_2.b, relu=True)
        out = ops.gemm_nt(fc2, self.fc_out.w, bias=self.fc_out.b)                                  # [N,96]
        K = cfg.num_classes
        dout = torch.zeros_like(out)
        cls_prob = torch.empty(N, K, device=data.device)
        ops.count_valid(label, self.cnt_buf[1:2])
        ops.softmax_ce(out, label, K, cfg.grad_scale, self.cnt_buf[1:2], cls_prob, dout, self.loss_buf[2:3])
        ops.smooth_l1_loss(out[:, K:K + 4], bbox_target, bbox_weight, 4, cfg.grad_scale / (188.0 * 16.0),
                           dout[:, K:K + 4], self.loss_buf[3:4])

        # ================= backward =================
        sp = cfg.wgrad_splits
        W = cfg.wsched
        v4 = lambda t: t.view(1, 1, t.shape[0], t.shape[1])
        W(self.fc_out.bwd_weight, v4(dout), v4(fc2), sp)
        dfc2 = ops.relu_bwd(fc2, ops.gemm_nt(dout, self.fc_out.wt))
        W(self.fc_new_2.bwd_weight, v4(dfc2), v4(fc1), sp)
        dfc1 = ops.relu_bwd(fc1, ops.gemm_nt(dfc2, self.fc_new_2.wt))
        W(self.fc_new_1.bwd_weight, v4(dfc1), v4(pooled.view(N, -1)), sp)
        dpooled = ops.gemm_nt(dfc1, self.fc_new_1.wt).view(pooled.shape)
        dfeat, dtrans = ops.deform_psroi_bwd(dpooled, feat, rois, trans, no_trans=False, trans_std=0.1, **ps)
        doff = torch.zeros_like(off)
        doff[:, :98] = dtrans.view(N, 98)
        W(self.fc_offset.bwd_weight, v4(doff), v4(offset_t.view(N, -1)), sp)
        doffset_t = ops.gemm_nt(doff, self.fc_offset.wt).view(offset_t.shape)
        ops.deform_psroi_bwd(doffset_t, feat, rois, None, no_trans=True, data_diff=dfeat, **ps)
        dfeat = ops.relu_bwd(feat, dfeat)
        hw = (Hf, Hf)
        W(self.conv_new_1.bwd_weight, dfeat, cat, sp)
        dcat = self.conv_new_1.bwd_data(dfeat, hw)
        W(self.rpn_head.bwd_weight, dhead, rpn, sp)
        drpn = ops.relu_bwd(rpn, self.rpn_head.bwd_data(dhead, hw))
        W(self.rpn_conv.bwd_weight, drpn, cat, sp)
        dcat = self.rpn_conv.bwd_data(drpn, hw, out=dcat, residual=dcat)
        if self.af_train:
            W(self.conv_new_3.bwd_weight, df3, f2, sp)
            df2 = ops.relu_bwd(f2, self.conv_new_3.bwd_data(df3, hw))
            W(self.conv_new_2.bwd_weight, df2, cat, sp)
            dcat = self.conv_new_2.bwd_data(df2, hw, out=dcat, residual=dcat)
        # ---- backbone backward (stage 4, then stage 3 with the c4 half of dcat added, then stage 2)
        g, g4 = dcat[..., 1024:], dcat[..., :1024]
        if lowp:      # backward of the Cast: the backbone's activation gradients are bf16
            g, g4 = ops.cast_rows(g, torch.bfloat16), ops.cast_rows(g4, torch.bfloat16)
        out = dict(rpn_cls_prob=prob, rpn_bbox_loss=self.loss_buf[1:2], cls_prob=cls_prob, bbox_loss=self.loss_buf[3:4],
                   label=label, rois=rois, losses=self.loss_buf, rpn_head=head, cat=cat, bbox_target=bbox_target,
                   bbox_weight=bbox_weight)
        if self.af_train:
            out["cls_scale_prob"] = scale_prob
        bounds = [len(self.units), n1 + n2 + n3, n1 + n2, n1]          # stage 4 | stage 3 | stage 2
        for k in range(3):
            for i in range(bounds[k] - 1, bounds[k + 1] - 1, -1):
                u = self.units[i]
                g = u.bwd(g, cfg, extra_add=g4 if i == last3 + 1 else None)
            ops.bn_param_grad_batched(self._bn_tables[k])
            W.join()
            if k == 2:
                self.step_count += 1
            yield out

    def forward_inference(self, data, im_info, suppress_anchor_types=False, autofocus=False):
        """get_symbol_rcnn(cfg, is_train=False) (resnet_mx_101_e2e.py:227-345 with the test branch :258-266, 321-326):
        backbone with moving-statistics BN -> RPN -> MultiProposal (device inference proposal op) -> deformable
        R-FCN head -> (rois [B*R,5], rpn scores [B*R], cls_prob [B*R,K], bbox_pred [B*R,4]).  No parameter is touched."""
        cfg = self.cfg
        A = cfg.num_anchors
        B = data.shape[0]
        for b in self.train_bns():
            ops.bn_frozen(b.st, cfg.bn_eps)        # scale/shift from the moving statistics (the next training step
        x = self.stem(data)                                               # recomputes them from batch statistics)
        x = ops.maxpool3x3s2(x)
        n1, n2, n3, n4 = cfg.units
        Hf, Wf = data.shape[2] // cfg.feat_stride, data.shape[3] // cfg.feat_stride
        cat = torch.empty(B, Hf, Wf, 3072, device=data.device)
        last3 = n1 + n2 + n3 - 1
        lowp = bool(cfg.bf16)
        for i, u in enumerate(self.units):
            out = None
            if not lowp:
                out = cat[..., :1024] if i == last3 else (cat[..., 1024:] if i == len(self.units) - 1 else None)
            x = u.fwd_infer(x, cfg, out=out)
            if lowp and i == last3:
                ops.cast_rows(x, out=cat[..., :1024])
        if lowp:
            ops.cast_rows(x, out=cat[..., 1024:])
        rpn = self.rpn_conv.fwd(cat, relu=True)
        head = self.rpn_head.fwd(rpn)
        feat = self.conv_new_1.fwd(cat, relu=True)
        fmap = None
        if autofocus:
            if self.af is None:
                raise RuntimeError("forward_inference(autofocus=True): call enable_autofocus() first")
            fmap = self.focus_map(cat)
        prob = torch.empty(B, Hf, Wf, 2 * A, device=data.device)
        ignore = torch.full((B, A * Hf * Wf), -1.0, device=data.device)
        cnt = torch.ones(1, dtype=torch.int32, device=data.device)
        loss = torch.zeros(1, device=data.device)
        ops.rpn_softmax_loss(head[..., 4 * A:6 * A], ignore, A, 1.0, cnt, prob, None, loss)
        rois, scores = ops.multi_proposal(prob, head, im_info, feat_stride=cfg.feat_stride, scales=cfg.scales,
                                          ratios=cfg.ratios, rpn_post_nms_top_n=cfg.rpn_post_nms_top_n,
                                          suppress_anchor_types=suppress_anchor_types, layout=ops.NHWC)
        N = rois.shape[0]
        ps = dict(spatial_scale=1.0 / cfg.feat_stride, output_dim=256, group_size=1, pooled_size=7, part_size=7,
                  sample_per_part=4, layout=ops.NHWC)
        offset_t, _, _ = ops.deform_psroi_fwd(feat, rois, None, no_trans=True, want_count=False, **ps)
        off = ops.gemm_nt(offset_t.view(N, -1), self.fc_offset.w, bias=self.fc_offset.b)
        trans = off[:, :98].contiguous().view(N, 2, 7, 7)
        pooled, _, _ = ops.deform_psroi_fwd(feat, rois, trans, no_trans=False, trans_std=0.1, want_count=False, **ps)
        fc1 = ops.gemm_nt(pooled.view(N, -1), self.fc_new_1.w, bias=self.fc_new_1.b, relu=True)
        fc2 = ops.gemm_nt(fc1, self.fc_new_2.w, bias=self.fc_new_2.b, relu=True)
        out = ops.gemm_nt(fc2, self.fc_out.w, bias=self.fc_out.b)
        K = cfg.num_classes
        cls_prob = torch.empty(N, K, device=data.device)
        lab = torch.full((N,), -1.0, device=data.device)
        ops.softmax_ce(out, lab, K, 1.0, cnt, cls_prob, None, loss)
        if autofocus:
            return rois, scores, cls_prob, out[:, K:K + 4], fmap
        return rois, scores, cls_prob, out[:, K:K + 4]

    def forward_rpn(self, data, im_info, suppress_anchor_types=False):
        """get_symbol_rpn(cfg, is_train=False) (resnet_mx_101_e2e.py:157-225): backbone with moving-statistics BatchNorm ->
        RPN head -> MultiProposal -> (rois [B*R,5], rpn scores [B*R]); the proposal-extraction half of
        `forward_inference` (same launches up to the proposal operator)."""
        cfg = self.cfg
        A = cfg.num_anchors
        B = data.shape[0]
        for b in self.train_bns():
            ops.bn_frozen(b.st, cfg.bn_eps)
        x = self.stem(data)
        x = ops.maxpool3x3s2(x)
        n1, n2, n3, n4 = cfg.units
        Hf, Wf = data.shape[2] // cfg.feat_stride, data.shape[3] // cfg.feat_stride
        cat = torch.empty(B, Hf, Wf, 3072, device=data.device)
        last3 = n1 + n2 + n3 - 1
        lowp = bool(cfg.bf16)
        for i, u in enumerate(self.units):
            out = None
            if not lowp:
                out = cat[..., :1024] if i == last3 else (cat[..., 1024:] if i == len(self.units) - 1 else None)
            x = u.fwd_infer(x, cfg, out=out)
            if lowp and i == last3:
                ops.cast_rows(x, out=cat[..., :1024])
        if lowp:
            ops.cast_rows(x, out=cat[..., 1024:])
        rpn = self.rpn_conv.fwd(cat, relu=True)
        head = self.rpn_head.fwd(rpn)
        prob = torch.empty(B, Hf, Wf, 2 * A, device=data.device)
        ignore = torch.full((B, A * Hf * Wf), -1.0, device=data.device)
        cnt = torch.ones(1, dtype=torch.int32, device=data.device)
        loss = torch.zeros(1, device=data.device)
        ops.rpn_softmax_loss(head[..., 4 * A:6 * A], ignore, A, 1.0, cnt, prob, None, loss)
        return ops.multi_proposal(prob, head, im_info, feat_stride=cfg.feat_stride, scales=cfg.scales, ratios=cfg.ratios,
                                  rpn_post_nms_top_n=cfg.rpn_post_nms_top_n, suppress_anchor_types=suppress_anchor_types,
                                  layout=ops.NHWC)

    # ---------------------------------------------------------------- reference checkpoints (utils.py:45-100)
    def _named_convs(self):
        cs = [c for u in self.units for c in u.convs()]
        cs += [self.rpn_conv, self.rpn_head, self.conv_new_1, self.fc_offset, self.fc_new_1, self.fc_new_2, self.fc_out]
        if self.af_train:
            cs += [self.conv_new_2, self.conv_new_3, self.conv_new_out]
        return cs

    def _named_bns(self):
        return [self.bn_data, self.bn0] + [b for u in self.units for b in u.bns()]

    def stem(self, data):
        """bn_data -> conv0 -> bn0 -> ReLU (resnetc4 :402-408), NHWC out.  Default: im2col + tcgen05 GEMM (TF32 for the
        fp32 configuration, bf16 operands in the mixed-precision one); SNIPER_STEM_TC=0: the FP32-FMA direct kernel."""
        if os.environ.get("SNIPER_STEM_TC", "1") != "1":
            return ops.stem_conv(data, self.conv0_w, self.bn_data.st.scale, self.bn_data.st.shift, self.bn0.st.scale,
                                 self.bn0.st.shift, out_dtype=self.act_dtype)
        if self._stem_rows is None:            # frozen layer: built once (load_reference resets it)
            self._stem_rows = ops.stem_rows(self.conv0_w, self.act_dtype)
        return ops.stem_conv_tc(data, self._stem_rows, self.bn_data.st.scale, self.bn_data.st.shift, self.bn0.st.scale,
                                self.bn0.st.shift, out_dtype=self.act_dtype)

    def load_reference(self, arg, aux, allow_missing=False):
        """Loads a reference checkpoint (`arg_params`, `aux_params` as numpy dicts, e.g. checkpoint.read_params of a
        released SNIPER `.params` file): OIHW -> tap-major rows, NCHW-flattened FC inputs -> NHWC, fused heads.
        allow_missing=True is the reference's normal training start: an ImageNet ResNet-101 checkpoint holds only the
        backbone, and `init_weight_rcnn` (resnet_mx_101_e2e.py:450-485) initialises the offset layers, the RPN and
        the R-FCN head -- here those layers simply keep the values the constructor gave them (zeros for the offset layers,
        N(0, 0.01) for the heads).  Returns the list of layers that were not in the checkpoint."""
        from . import checkpoint as ck
        cfg = self.cfg
        dev = self.device
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(dev)
        skipped = []
        self._stem_rows = None
        if "conv0_weight" in arg or not allow_missing:
            self.conv0_w.copy_(t(arg["conv0_weight"].transpose(0, 2, 3, 1)))
        else:
            skipped.append("conv0")
        for c in self._named_convs():
            parts = ck.FUSED.get(c.name, (c.name,))
            if allow_missing and any(p + "_weight" not in arg for p in parts):
                skipped.append(c.name)
                continue
            w, b = ck.conv_from_reference(c.name, c.cout, c.coutp, c.cin, c.k, c.bias, arg)
            c.master.copy_(t(w))
            if c.bias:
                c.b.copy_(t(b))
        for bn in self._named_bns():
            if allow_missing and bn.name + "_gamma" not in arg:
                skipped.append(bn.name)
                continue
            bn.st.gamma.copy_(t(arg[bn.name + "_gamma"]))
            bn.st.beta.copy_(t(arg[bn.name + "_beta"]))
            bn.st.moving_mean.copy_(t(aux[bn.name + "_moving_mean"]))
            bn.st.moving_var.copy_(t(aux[bn.name + "_moving_var"]))
            if bn.frozen:
                ops.bn_frozen(bn.st, cfg.bn_eps, fix_gamma=bn.fix_gamma)
        self.P.sync_lowp()
        self._wt_table = None      # data-gradient operands are rebuilt from the new weights on the next step
        return skipped

    def export_reference(self, grads=False):
        """The inverse of load_reference: (arg_params, aux_params) under the reference's names and layouts.
        grads=True: the parameter GRADIENTS of the last forward_backward in the same names / layouts (what
        `executor.grad_dict` holds in the reference; trainable tensors only, aux empty)."""
        from . import checkpoint as ck
        cfg = self.cfg
        A, K = cfg.num_anchors, cfg.num_classes
        n = lambda x: x.detach().cpu().numpy().copy()
        arg, aux = {}, {}
        if not grads:
            arg["conv0_weight"] = np.ascontiguousarray(n(self.conv0_w).transpose(0, 3, 1, 2))
        parts = {"rpn_head": (4 * A, 2 * A), "cls_bbox": (K, 4)}
        for c in self._named_convs():
            if grads and not c.trainable:
                continue
            w = self.P.grad(c.name + "_weight") if grads else (c.master.float() if c.master.dtype == torch.bfloat16 else c.master)
            b = (self.P.grad(c.name + "_bias") if grads else c.b) if c.bias else None
            ck.conv_to_reference(c.name, c.cout, c.cin, c.k, n(w), n(b) if c.bias else None, parts.get(c.name), arg)
        for bn in self._named_bns():
            if grads:
                if not bn.frozen:
                    arg[bn.name + "_gamma"] = n(bn.st.dgamma)
                    arg[bn.name + "_beta"] = n(bn.st.dbeta)
                continue
            arg[bn.name + "_gamma"] = n(bn.st.gamma)
            arg[bn.name + "_beta"] = n(bn.st.beta)
            aux[bn.name + "_moving_mean"] = n(bn.st.moving_mean)
            aux[bn.name + "_moving_var"] = n(bn.st.moving_var)
        return arg, aux

    def set_lr(self, lr=None):
        """Writes (lr, wd) into the device hyper-parameter buffer the update kernels read (outside graph capture)."""
        self.P.set_hyper(float(self.cfg.lr if lr is None else lr), float(self.cfg.wd))

    def update(self, lr=None):
        """SGD-momentum on every trainable tensor.  lr=None: keep whatever set_lr() last wrote (the form that is
        captured into the update graph); a number: set it first (eager use)."""
        if lr is not None or self.P._hyper_host[0] is None:
            self.set_lr(lr)
        self.P.sgd_step(self.cfg.momentum)

    def train_step(self, batch, lr=None, allreduce=None):
        out = self.forward_backward(batch)
        if allreduce is not None:
            allreduce(self.P.g)           # ONE collective per step over the flat gradient bucket
        self.update(lr)
        return out
