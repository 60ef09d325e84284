"""Symbol-class facade: the object `main_train.py` / `main_test.py` get from `symbols/faster/resnet_mx_101_e2e.py`.

Mirrors the reference's `Symbol` base class (symbols/symbol.py:9-61) and `resnet_mx_101_e2e`
(symbols/faster/resnet_mx_101_e2e.py:20-35 constructor, :227-345 get_symbol_rcnn, :450-485 init_weight_rcnn,
:6-17 checkpoint_callback) with the same method names, argument meaning and dictionary keys, so that the driver code
around them reads the same:

    sym_inst = resnet_mx_101_e2e(n_proposals=400, momentum=args.momentum)
    sym = sym_inst.get_symbol_rcnn(config)
    sym_inst.infer_shape({'data': (20, 3, 512, 512), ...})
    arg_params, aux_params = load_param(pretrained, epoch)          # sniper_b200.checkpoint.load_param
    sym_inst.init_weight_rcnn(config, arg_params, aux_params)
    sym_inst.check_parameter_shapes(arg_params, aux_params, data_shape_dict)
    net = sym.bind('cuda:0', batch_images=20)                        # -> sniper_b200.model.SniperResNet101
    net.load_reference(arg_params, aux_params)

What `get_symbol_rcnn` returns is not an MXNet graph: it is a `NetSymbol` that knows the reference's argument / auxiliary /
output names and shapes (pure host code, usable without a GPU) and binds to the one hand-scheduled network this package
implements.  Reference symbol FILES are not executed; the graph they describe is `model.SniperResNet101`.
"""
import numpy as np

from . import checkpoint as ck

UNITS = (3, 4, 23, 3)
FILTER_LIST = (64, 256, 512, 1024, 2048)


class NetSymbol(object):
    """Names and shapes of the SNIPER ResNet-101 R-FCN graph as `mx.sym.Symbol` exposes them."""

    rpn_only = False        # get_symbol_rpn (resnet_mx_101_e2e.py:157-225): backbone + RPN head (+ MultiProposal at test time)

    def __init__(self, cfg, is_train=True, num_classes=81, num_anchors=21, rois_per_chip=300, max_gt=100, rpn_only=False,
                 autofocus=False):
        """autofocus: the AutoFocus TRAINING graph (TRAIN.AUTO_FOCUS, :239-240, 259-267, 313-315, 335-336): scale_label
        data, conv_new_2 / conv_new_3 / conv_new_out parameters, cls_scale_prob output."""
        self.cfg, self.is_train = cfg, is_train
        self.num_classes, self.num_anchors, self.rois, self.max_gt = num_classes, num_anchors, rois_per_chip, max_gt
        self.rpn_only = rpn_only
        self.autofocus = bool(autofocus) and is_train and not rpn_only
        self._args, self._aux = [], []
        self._build()

    # ---- graph description (resnet_mx_101_e2e.py:36-69 residual_unit, :106-145 residual_unit_deform, :394-448, :227-345)
    def _conv(self, n, o, i, k, bias=False):
        self._args.append((n + "_weight", (o, i, k, k)))
        if bias:
            self._args.append((n + "_bias", (o,)))

    def _bn(self, n, c):
        self._args += [(n + "_gamma", (c,)), (n + "_beta", (c,))]
        self._aux += [(n + "_moving_mean", (c,)), (n + "_moving_var", (c,))]

    def _fc(self, n, o, i):
        self._args += [(n + "_weight", (o, i)), (n + "_bias", (o,))]

    def _build(self):
        A, K = self.num_anchors, self.num_classes
        self._bn("bn_data", 3)
        self._conv("conv0", 64, 3, 7)
        self._bn("bn0", 64)
        cin = FILTER_LIST[0]
        for si, n in enumerate(UNITS):
            cout = FILTER_LIST[si + 1]
            mid = cout // 4
            for j in range(n):
                nm = "stage%d_unit%d" % (si + 1, j + 1)
                ci = cin if j == 0 else cout
                self._bn(nm + "_bn1", ci); self._conv(nm + "_conv1", mid, ci, 1)
                self._bn(nm + "_bn2", mid)
                if si == 3:
                    self._conv(nm + "_offset", 72, mid, 3, bias=True)
                self._conv(nm + "_conv2", mid, mid, 3)
                self._bn(nm + "_bn3", mid); self._conv(nm + "_conv3", cout, mid, 1)
                if j == 0:
                    self._conv(nm + "_sc", cout, ci, 1)
            cin = cout
        self._conv("rpn_conv_3x3", 512, 3072, 3, True)
        self._conv("rpn_cls_score", 2 * A, 512, 1, True)
        self._conv("rpn_bbox_pred", 4 * A, 512, 1, True)
        if self.rpn_only:
            return
        self._conv("conv_new_1", 256, 3072, 1, True)
        self._fc("offset", 2 * 7 * 7, 256 * 7 * 7)
        self._fc("fc_new_1", 1024, 256 * 7 * 7)
        self._fc("fc_new_2", 1024, 1024)
        self._fc("cls_score", K, 1024)
        self._fc("bbox_pred", 4, 1024)
        if self.autofocus:
            self._conv("conv_new_2", 256, 3072, 3, True)
            self._conv("conv_new_3", 256, 256, 1, True)
            self._conv("conv_new_out", 2, 256, 1, True)

    # ---- mx.sym.Symbol surface
    def data_names(self):
        if self.rpn_only:
            return ["data", "label", "bbox_target", "bbox_weight"] if self.is_train else ["data", "im_info", "im_ids"]
        if self.is_train:
            names = ["data", "im_info", "gt_boxes", "valid_ranges", "label", "bbox_target", "bbox_weight"]
            return names + ["scale_label"] if self.autofocus else names
        return ["data", "im_info", "im_ids", "chip_ids"]

    def list_arguments(self):
        return self.data_names() + [n for n, _ in self._args]

    def list_auxiliary_states(self):
        return [n for n, _ in self._aux]

    def list_outputs(self):
        if self.rpn_only:      # Group([rpn_cls_prob, rpn_bbox_loss]) / Group([rois, rpn_scores, im_ids]) (:214, :222)
            return ["rpn_cls_prob_output", "rpn_bbox_loss_output"] if self.is_train else ["rois_output", "rois_score", "im_ids"]
        if self.is_train:      # mx.sym.Group order of get_symbol_rcnn (resnet_mx_101_e2e.py:335-338); metric.py reads it by position
            names = ["rpn_cls_prob_output", "rpn_bbox_loss_output", "cls_prob_reshape_output", "bbox_loss_reshape_output",
                     "blockgrad0_output"]
            return names[:2] + ["cls_scale_prob_output"] + names[2:] if self.autofocus else names
        # test-time group (:386-389): rois, cls_prob, bbox_pred and the three pass-through inputs
        return ["rois_output", "cls_prob_reshape_output", "bbox_pred_reshape_output", "im_ids", "im_info", "chip_ids"]

    def infer_shape(self, **data_shapes):
        """(arg_shapes, out_shapes, aux_shapes) in list_arguments / list_outputs / list_auxiliary_states order."""
        B = data_shapes["data"][0]
        H, W = data_shapes["data"][2] // 16, data_shapes["data"][3] // 16
        A, K, R = self.num_anchors, self.num_classes, self.rois
        dflt = {"data": data_shapes["data"], "im_info": (B, 3), "im_ids": (B,), "chip_ids": (B,),
                "gt_boxes": (B, self.max_gt, 5), "valid_ranges": (B, 2),
                "label": (B, A * H * W), "bbox_target": (B, 4 * A, H, W), "bbox_weight": (B, 4 * A, H, W),
                "scale_label": (B, H * W)}
        arg = [tuple(data_shapes.get(n, dflt[n])) for n in self.data_names()] + [s for _, s in self._args]
        if self.rpn_only:
            out = [(B, 2, A * H, W), (B, 4 * A, H, W)] if self.is_train else [(B * R, 5), (B * R,), (B,)]
            return arg, out, [s for _, s in self._aux]
        if self.is_train:
            # the last head is BlockGrad(label_reshape): Reshape(label, (-1,)) (resnet_mx_101_e2e.py:281,334) -> (B*R,)
            out = [(B, 2, A * H, W), (B, 4 * A, H, W), (B, R, K), (B, R, 4), (B * R,)]
            if self.autofocus:          # cls_scale_prob over conv_new_out_reshape (0, 2, -1) (:266, 313-315)
                out.insert(2, (B, 2, H * W))
        else:
            out = [(B * R, 5), (B, R, K), (B, R, 4), (B,), (B, 3), (B,)]
        return arg, out, [s for _, s in self._aux]

    def bind(self, device="cuda:0", batch_images=20, bf16=False, seed=5, **cfg_overrides):
        """The executor: `model.SniperResNet101` on `device` (needs the CUDA library; fails loudly without a GPU)."""
        from . import model
        c = model.Cfg()
        c.batch_images = batch_images
        c.bf16 = bool(bf16)
        c.autofocus = self.autofocus
        for k, v in cfg_overrides.items():
            setattr(c, k, v)
        return model.SniperResNet101(c, device=device, seed=seed)


MNV2_BOTTLENECKS = ((1, 16, 1, 1), (6, 24, 2, 2), (6, 32, 3, 2), (6, 64, 4, 2), (6, 96, 3, 1), (6, 160, 3, 2), (6, 320, 1, 1))


class MobileNetSymbol(NetSymbol):
    """Names and shapes of the MobileNetV2 SNIPER graph (symbols/faster/mobilenetv2_e2e.py:171-305; train graph)."""
    feat_stride = 32

    def __init__(self, cfg, is_train=True, num_classes=81, num_anchors=15, rois_per_chip=300, max_gt=100):
        NetSymbol.__init__(self, cfg, is_train, num_classes, num_anchors, rois_per_chip, max_gt)

    def _unit(self, prefix, o, i, k, groups=1):
        self._args.append((prefix + "-conv2d_weight", (o, i // groups, k, k)))
        self._bn(prefix + "-batchnorm", o)

    def _build(self):
        A, K = self.num_anchors, self.num_classes
        self._unit("first-3x3-conv", 32, 3, 3)
        in_c = 32
        for si, (t, c, n, st) in enumerate(MNV2_BOTTLENECKS):
            for j in range(n):
                ci = in_c if j == 0 else c
                e = int(round(ci * t))
                p = "seq-%d-block%d" % (si, j)
                self._unit(p + "-exp", e, ci, 1)
                self._unit(p + "-depthwise", e, e, 3, groups=e)
                self._unit(p + "-linear", c, e, 1)
            in_c = c
        self._unit("last-1x1-conv", 1280, in_c, 1)
        self._conv("rpn_conv_3x3", 256, 1280, 3, True)
        self._conv("rpn_cls_score", 2 * A, 256, 1, True)
        self._conv("rpn_bbox_pred", 4 * A, 256, 1, True)
        self._conv("conv_new_1", 256, 1280, 1, True)
        self._fc("offset", 2 * 7 * 7, 256 * 7 * 7)
        self._fc("fc_new_1", 512, 256 * 7 * 7)
        self._fc("fc_new_2", 512, 512)
        self._fc("cls_score", K, 512)
        self._fc("bbox_pred", 4, 512)

    def data_names(self):
        if self.is_train:
            return ["data", "im_info", "gt_boxes", "valid_ranges", "crowd_boxes", "label", "bbox_target", "bbox_weight"]
        return ["data", "im_info", "im_ids", "chip_ids"]

    def infer_shape(self, **data_shapes):
        B = data_shapes["data"][0]
        H, W = data_shapes["data"][2] // 32, data_shapes["data"][3] // 32
        A, K, R = self.num_anchors, self.num_classes, self.rois
        dflt = {"data": data_shapes["data"], "im_info": (B, 3), "im_ids": (B,), "chip_ids": (B,),
                "gt_boxes": (B, self.max_gt, 5), "valid_ranges": (B, 2), "crowd_boxes": (B, 10, 5),
                "label": (B, A * H * W), "bbox_target": (B, 4 * A, H, W), "bbox_weight": (B, 4 * A, H, W)}
        arg = [tuple(data_shapes.get(n, dflt[n])) for n in self.data_names()] + [s for _, s in self._args]
        if self.is_train:
            out = [(B, 2, A * H, W), (B, 4 * A, H, W), (B, R, K), (B, R, 4), (B * R,)]
        else:
            out = [(B * R, 5), (B, R, K), (B, R, 4), (B,), (B, 3), (B,)]
        return arg, out, [s for _, s in self._aux]

    def bind(self, device="cuda:0", batch_images=40, bf16=True, seed=5, **cfg_overrides):
        """The executor: `model_mnv2.SniperMobileNetV2` (training graph)."""
        from . import model_mnv2
        c = model_mnv2.MCfg()
        c.batch_images = batch_images
        c.bf16 = bool(bf16)
        for k, v in cfg_overrides.items():
            setattr(c, k, v)
        return model_mnv2.SniperMobileNetV2(c, device=device, seed=seed)


def recognise_graph(sym):
    """Host-only: decides whether a graph built by the reference's own symbol file through `mxnet_compat` (or loaded from
    a `-symbol.json`) is one this package executes, by its parameter set: every non-data argument / auxiliary state must
    be exactly what `NetSymbol` (the hand-written description of model.SniperResNet101) lists, with the same shapes.
    Returns the executor settings read off the graph's own attributes: batch_images (MultiProposalTarget batch_size),
    num_anchors (rpn_cls_score num_filter / 2), num_classes (cls_score num_hidden), bf16 (a Cast to float16 inside the
    backbone = TRAIN.fp16), is_train.  Raises NotImplementedError naming the first differences otherwise."""
    from . import mxnet_compat as MC
    nodes = {n.name: n for n in MC._dfs(sym._heads)}
    is_train = "multi_proposal_target" in nodes
    if "rpn_cls_score" not in nodes:
        raise NotImplementedError("not a SNIPER Faster-R-CNN / R-FCN graph (no rpn_cls_score node)")
    rpn_only = "cls_score" not in nodes                        # get_symbol_rpn: backbone + RPN head (+ MultiProposal)
    if rpn_only:
        is_train = "rois" not in nodes
    A = int(nodes["rpn_cls_score"].attrs["num_filter"]) // 2
    K = 81 if rpn_only else int(nodes["cls_score"].attrs["num_hidden"])
    B = int(nodes["multi_proposal_target"].attrs.get("batch_size", 16)) if "multi_proposal_target" in nodes else \
        int(nodes["rois"].attrs.get("batch_size", 1)) if "rois" in nodes else 1
    fp16 = any(n.op == "Cast" and n.attrs.get("dtype") == "float16" for n in nodes.values())
    mnv2 = "first-3x3-conv-conv2d" in nodes
    stride = 32 if mnv2 else 16
    if rpn_only and mnv2:
        raise NotImplementedError("MobileNetV2: no RPN-only graph in the reference")
    ours = NetSymbol(None, is_train=is_train, num_anchors=A, rpn_only=True) if rpn_only else \
        (MobileNetSymbol if mnv2 else NetSymbol)(None, is_train=is_train, num_classes=K, num_anchors=A)
    data = set(ours.data_names()) | {"scale_label", "crowd_boxes"}
    H = 512
    shapes = {"data": (B, 3, H, H)}
    if is_train:
        Hf = H // stride
        shapes.update({"label": (B, A * Hf * Hf), "bbox_target": (B, 4 * A, Hf, Hf), "bbox_weight": (B, 4 * A, Hf, Hf),
                       "gt_boxes": (B, 100, 5), "valid_ranges": (B, 2), "im_info": (B, 3), "crowd_boxes": (B, 10, 5)})
    else:
        shapes.update({"im_info": (B, 3), "im_ids": (B,), "chip_ids": (B,)})
    if rpn_only:
        shapes = {k: v for k, v in shapes.items() if k in ours.data_names()}
    args, _, auxs = sym.infer_shape_partial(**shapes)
    theirs = {n: tuple(s) for n, s in zip(sym.list_arguments(), args) if n not in data}
    theirs_aux = {n: tuple(s) for n, s in zip(sym.list_auxiliary_states(), auxs)}
    mine = {n: tuple(s) for n, s in ours._args}
    mine_aux = {n: tuple(s) for n, s in ours._aux}
    # the AutoFocus branch (conv_new_2/3/out): trained when the graph is a training graph with the scale_label loss
    # (TRAIN.AUTO_FOCUS), else the inference branch of model.enable_autofocus()
    af = {k for k in theirs if k.startswith(("conv_new_2_", "conv_new_3_", "conv_new_out_"))}
    af_train = bool(af) and is_train and "cls_scale_prob" in nodes
    if af_train:
        ours = NetSymbol(None, is_train=True, num_classes=K, num_anchors=A, autofocus=True)
        mine = {n: tuple(s) for n, s in ours._args}
        af = set()
    diff = sorted((set(theirs) - af) ^ set(mine)) + sorted(set(theirs_aux) ^ set(mine_aux))
    diff += sorted(k for k in mine if k in theirs and theirs[k] != mine[k])
    if diff:
        raise NotImplementedError("this package executes the ResNet-101 and MobileNetV2 SNIPER R-FCN graphs only; the given "
                                  "graph differs in %d parameters, e.g. %s" % (len(diff), ", ".join(diff[:6])))
    if mnv2 and not is_train:
        raise NotImplementedError("MobileNetV2: only the training graph is executable")
    info = dict(batch_images=B, num_anchors=A, num_classes=K, bf16=fp16, is_train=is_train, autofocus=bool(af) or af_train)
    if af_train:                              # the executor trains the FocusPixel branch (Cfg.autofocus)
        info["autofocus_train"] = True
    if mnv2:
        info["network"] = "mobilenetv2"
    if rpn_only:
        if is_train:
            raise NotImplementedError("RPN-only TRAINING (get_symbol_rpn, is_train=True) has no executor here: the end-to-end "
                                      "graph trains the RPN; the RPN-only test graph binds to SniperResNet101.forward_rpn")
        info["rpn_only"] = True
    return info


def bind_graph(sym, device="cuda:0", **overrides):
    """`mxnet_compat.Symbol.bind`: the executor for a recognised graph (model.SniperResNet101; fp16 graphs run the bf16
    mixed-precision configuration).  Needs the CUDA library -- fails loudly without it."""
    info = recognise_graph(sym)
    cls = MobileNetSymbol if info.get("network") == "mobilenetv2" else NetSymbol
    ours = cls(None, is_train=info["is_train"], num_classes=info["num_classes"], num_anchors=info["num_anchors"])
    if info.get("autofocus_train"):               # the FocusPixel branch is trained: Cfg.autofocus (not enable_autofocus)
        ours = NetSymbol(None, is_train=True, num_classes=info["num_classes"], num_anchors=info["num_anchors"],
                         autofocus=True)
    # (an RPN-only test graph binds to the full network object: its executor is `forward_rpn`)
    kw = dict(batch_images=info["batch_images"], bf16=info["bf16"], num_classes=info["num_classes"],
              num_anchors=info["num_anchors"])
    kw.update(overrides)
    net = ours.bind(device, **kw)
    if info["autofocus"] and not info.get("autofocus_train"):
        net.enable_autofocus()
    return net


class Symbol(object):
    """symbols/symbol.py:9-61."""

    def __init__(self):
        self.arg_shape_dict = None
        self.out_shape_dict = None
        self.aux_shape_dict = None
        self.sym = None

    @property
    def symbol(self):
        return self.sym

    def get_bbox_param_names(self):
        raise NotImplementedError()

    def get_symbol(self, cfg, is_train=True):
        raise NotImplementedError()

    def init_weights(self, cfg, arg_params, aux_params):
        raise NotImplementedError()

    def get_msra_std(self, shape):
        fan_in = float(shape[1])
        if len(shape) > 2:
            fan_in *= np.prod(shape[2:])
        return np.sqrt(2 / fan_in)

    def infer_shape(self, data_shape_dict):
        arg_shape, out_shape, aux_shape = self.sym.infer_shape(**data_shape_dict)
        self.arg_shape_dict = dict(zip(self.sym.list_arguments(), arg_shape))
        self.out_shape_dict = dict(zip(self.sym.list_outputs(), out_shape))
        self.aux_shape_dict = dict(zip(self.sym.list_auxiliary_states(), aux_shape))

    def check_parameter_shapes(self, arg_params, aux_params, data_shape_dict, is_train=True):
        for k in self.sym.list_arguments():
            if k in data_shape_dict or (False if is_train else 'label' in k):
                continue
            assert k in arg_params, k + ' not initialized'
            assert tuple(arg_params[k].shape) == tuple(self.arg_shape_dict[k]), \
                'shape inconsistent for ' + k + ' inferred ' + str(self.arg_shape_dict[k]) + ' provided ' + str(
                    arg_params[k].shape)
        for k in self.sym.list_auxiliary_states():
            assert k in aux_params, k + ' not initialized'
            assert tuple(aux_params[k].shape) == tuple(self.aux_shape_dict[k]), \
                'shape inconsistent for ' + k + ' inferred ' + str(self.aux_shape_dict[k]) + ' provided ' + str(
                    aux_params[k].shape)


def checkpoint_callback(bbox_param_names, prefix, means, stds):
    """resnet_mx_101_e2e.py:6-17: epoch-end callback writing `<prefix>-%04d.params` with the `*_test` box-regression
    copies.  `arg` / `aux`: dicts of numpy arrays under the reference's names (model.export_reference())."""
    def _callback(iter_no, sym, arg, aux):
        if bbox_param_names[0] in arg:
            ck.save_checkpoint(prefix, iter_no + 1, arg, aux, bbox_param_names=tuple(bbox_param_names))
    return _callback


class resnet_mx_101_e2e(Symbol):
    """symbols/faster/resnet_mx_101_e2e.py:20-35."""

    def __init__(self, n_proposals=400, momentum=0.95, fix_bn=False, test_nbatch=1):
        Symbol.__init__(self)
        self.momentum = momentum
        self.use_global_stats = True
        self.workspace = 512
        self.units = UNITS
        self.filter_list = list(FILTER_LIST)
        self.fix_bn = fix_bn
        self.test_nbatch = test_nbatch
        self.n_proposals = n_proposals

    def get_bbox_param_names(self):
        return ['bbox_pred_weight', 'bbox_pred_bias']

    def get_symbol_rcnn(self, cfg, is_train=True):
        num_classes = getattr(getattr(cfg, "dataset", None), "NUM_CLASSES", 81)
        net = getattr(cfg, "network", None)
        num_anchors = getattr(net, "NUM_ANCHORS", 21) if net is not None else 21
        autofocus = bool(getattr(getattr(cfg, "TRAIN", None), "AUTO_FOCUS", False))
        self.sym = NetSymbol(cfg, is_train=is_train, num_classes=num_classes, num_anchors=num_anchors, autofocus=autofocus)
        return self.sym

    get_symbol = get_symbol_rcnn

    def get_symbol_rpn(self, cfg, is_train=True):
        """:157-225 -- the RPN-only graph (proposal extraction); its executor is `SniperResNet101.forward_rpn`."""
        net = getattr(cfg, "network", None)
        num_anchors = getattr(net, "NUM_ANCHORS", 21) if net is not None else 21
        self.sym = NetSymbol(cfg, is_train=is_train, num_anchors=num_anchors, rpn_only=True)
        return self.sym

    def init_weight_rpn(self, cfg, arg_params, aux_params, seed=None):
        """:487-500 -- zero offset layers, N(0, 0.01) RPN head."""
        rng = np.random.RandomState(seed) if seed is not None else np.random
        sh = self.arg_shape_dict
        for u in (1, 2, 3):
            for sfx in ('_weight', '_bias'):
                arg_params['stage4_unit%d_offset%s' % (u, sfx)] = np.zeros(sh['stage4_unit%d_offset%s' % (u, sfx)], np.float32)
        for n in ('rpn_conv_3x3', 'rpn_cls_score', 'rpn_bbox_pred'):
            arg_params[n + '_weight'] = (rng.standard_normal(sh[n + '_weight']) * 0.01).astype(np.float32)
            arg_params[n + '_bias'] = np.zeros(sh[n + '_bias'], np.float32)

    def init_weight_rcnn(self, cfg, arg_params, aux_params, seed=None):
        """:450-485 -- zeros for every offset layer, N(0, 0.01) weights + zero biases for the RPN and the R-FCN head.
        Arrays are numpy float32 (the reference's mx.nd arrays); `seed` makes the draw reproducible."""
        rng = np.random.RandomState(seed) if seed is not None else np.random
        sh = self.arg_shape_dict
        zeros = lambda n: np.zeros(sh[n], np.float32)
        normal = lambda n: (rng.standard_normal(sh[n]) * 0.01).astype(np.float32)
        for u in (1, 2, 3):
            arg_params['stage4_unit%d_offset_weight' % u] = zeros('stage4_unit%d_offset_weight' % u)
            arg_params['stage4_unit%d_offset_bias' % u] = zeros('stage4_unit%d_offset_bias' % u)
        for n in ('rpn_conv_3x3', 'rpn_cls_score', 'rpn_bbox_pred', 'conv_new_1'):
            arg_params[n + '_weight'] = normal(n + '_weight')
            arg_params[n + '_bias'] = zeros(n + '_bias')
        if getattr(self.sym, "autofocus", False):              # TRAIN.AUTO_FOCUS (:468-474)
            for n in ('conv_new_2', 'conv_new_3', 'conv_new_out'):
                arg_params[n + '_weight'] = normal(n + '_weight')
                arg_params[n + '_bias'] = zeros(n + '_bias')
        arg_params['offset_weight'] = zeros('offset_weight')
        arg_params['offset_bias'] = zeros('offset_bias')
        for n in ('fc_new_1', 'fc_new_2', 'cls_score', 'bbox_pred'):
            arg_params[n + '_weight'] = normal(n + '_weight')
            arg_params[n + '_bias'] = zeros(n + '_bias')

    init_weights = init_weight_rcnn


class mobilenetv2_e2e(Symbol):
    """symbols/faster/mobilenetv2_e2e.py:152-158 (constructor), :171-305 (get_symbol_rcnn), :364-391 (init_weight_rcnn)."""

    def __init__(self, n_proposals=400, momentum=0.95, fix_bn=False, test_nbatch=1):
        Symbol.__init__(self)
        self.multiplier = 1
        self.test_nbatch = test_nbatch

    def get_bbox_param_names(self):
        return ['bbox_pred_weight', 'bbox_pred_bias']

    def get_symbol_rcnn(self, cfg, is_train=True):
        num_classes = getattr(getattr(cfg, "dataset", None), "NUM_CLASSES", 81)
        net = getattr(cfg, "network", None)
        num_anchors = getattr(net, "NUM_ANCHORS", 15) if net is not None else 15
        self.sym = MobileNetSymbol(cfg, is_train=is_train, num_classes=num_classes, num_anchors=num_anchors)
        return self.sym

    get_symbol = get_symbol_rcnn

    def init_weight_rcnn(self, cfg, arg_params, aux_params, seed=None):
        rng = np.random.RandomState(seed) if seed is not None else np.random
        sh = self.arg_shape_dict
        for n in ('rpn_conv_3x3', 'rpn_cls_score', 'rpn_bbox_pred', 'conv_new_1', 'fc_new_1', 'fc_new_2', 'cls_score',
                  'bbox_pred'):
            arg_params[n + '_weight'] = (rng.standard_normal(sh[n + '_weight']) * 0.01).astype(np.float32)
            arg_params[n + '_bias'] = np.zeros(sh[n + '_bias'], np.float32)
        arg_params['offset_weight'] = np.zeros(sh['offset_weight'], np.float32)
        arg_params['offset_bias'] = np.zeros(sh['offset_bias'], np.float32)

    init_weights = init_weight_rcnn
