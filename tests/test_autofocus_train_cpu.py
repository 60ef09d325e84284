"""AutoFocus training (TRAIN.AUTO_FOCUS) on the host, without a GPU:

* the FocusPixel labels: oracle/focus_label_np.gen_mask equals the reference's OWN anchor_worker.worker run with
  AUTO_FOCUS on (oracle/run_ref_anchor_worker.py; stored outputs under tests/golden/ref_calls/ where the reference is not
  built) on cases that cover every flag band and its boundaries, overlapping boxes in both orders, boxes partly and wholly
  outside the chip, boxes at x / y = 511, a scaled and shifted crop and a chip with more than 100 boxes; and the
  iterator's focus boxes, rasterised by that oracle, equal the reference worker's mask for the same chips;
* the network: `SniperResNet101(Cfg(autofocus=True))` executed through tests/fake_ops.py + tests/fake_ops_autofocus.py
  (float64 restatements of every C-ABI call, sniper_focus_head / sniper_focus_label included) against oracle/torch_graph_autofocus.forward_train
  in exact mode -- rois, the five loss sums, cls_scale_prob and all 303 parameter gradients -- two SGD updates under
  MXNet's rule, the checkpoint round trip, and the parameter layout of the default configuration;
* the symbol: NetSymbol of the AutoFocus training graph against the graph the reference's own symbol file builds
  (tests/golden/ref_symbols_autofocus.json)."""
import hashlib
import json
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
import ref_golden as G  # noqa: E402

HAVE_REF = os.path.isdir("/root/reference/lib") and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_chips.so"))
AF = dict(dc_low=5, small_thresh=64, dc_high=90)          # sniper_res101_e2e_autofocus.yml:106-119


# ------------------------------------------------------------------------------------------------ FocusPixel labels
def _ref_worker_mask(boxes, crop, scale, n_valid=1):
    """anchor_worker.worker of the reference with AUTO_FOCUS on, on image-space GT `boxes` of one chip -> mask_scale."""
    im_info = [512, 512, scale]
    gtids = np.arange(len(boxes))
    nids = np.arange(min(n_valid, len(boxes))).astype(np.int32)
    classes = np.ones((len(boxes), 1))

    def run():
        import run_ref_anchor_worker as RA
        cfg = RA.make_cfg()
        cfg.TRAIN.AUTO_FOCUS = True
        cfg.TRAIN.AUTO_FOCUS_DC_LOW, cfg.TRAIN.AUTO_FOCUS_SMALL_THRESH = AF["dc_low"], AF["small_thresh"]
        cfg.TRAIN.AUTO_FOCUS_DC_HIGH = AF["dc_high"]
        W = RA.load_reference_worker()(cfg, 512)
        np.random.seed(0)
        out = W.worker([im_info, np.array(crop, np.float64), scale, nids.copy(), gtids.copy(), boxes.copy(), boxes.copy(),
                        classes.copy()])
        return np.asarray(out[4], np.float32).ravel()
    return G.reference("autofocus_cpu.gen_mask", (boxes, np.asarray(crop, np.float64), float(scale), n_valid),
                       run if HAVE_REF else None)


def _side_box(x1, y1, side, aspect=1.0):
    """a box whose sqrt(w*h) is exactly `side` (integer w, h with w*h = side^2 when aspect = 1)"""
    w = side * aspect
    h = side * side / w
    return [x1, y1, x1 + w, y1 + h]


def _focus_cases():
    """(name, boxes [n,4] float32 image space, crop origin, scale)"""
    cases = []
    # every band and both edges of each: sides 4, 5, 6 | 63, 64, 65 | 89, 90, 91 (exact integer sides)
    b = [_side_box(10 + 40 * i % 400, 10 + 45 * (i // 10), s) for i, s in enumerate((4, 5, 6, 63, 64, 65, 89, 90, 91))]
    cases.append(("bands", b, (0.0, 0.0), 1.0))
    # the same sides from non-square boxes (w*h = side^2 with w != h): 5 = sqrt(25) = 1x25, 64 = 32x128, 90 = 60x135
    cases.append(("bands_rect", [[20, 20, 21, 45], [100, 30, 132, 158], [250, 200, 310, 335], [400, 400, 402, 432]],
                  (0.0, 0.0), 1.0))
    # overlapping boxes with different flags, both orders (the last writer wins; a >= DC_HIGH box writes nothing)
    cases.append(("overlap_pos_last", [[100, 100, 200, 200], [120, 120, 160, 160]], (0.0, 0.0), 1.0))
    cases.append(("overlap_neg_last", [[120, 120, 160, 160], [100, 100, 200, 200]], (0.0, 0.0), 1.0))
    cases.append(("overlap_big_last", [[120, 120, 160, 160], [50, 50, 400, 400], [300, 300, 303, 303]], (0.0, 0.0), 1.0))
    # partly outside the chip, wholly outside it (clipped onto the border: side 0 -> -1 stripes in row / column 0 or 31)
    cases.append(("outside", [[-30, 200, 20, 230], [490, -20, 540, 30], [600, 100, 700, 180], [100, -90, 160, -40],
                              [-80, -80, -10, -10], [200, 560, 260, 620]], (0.0, 0.0), 1.0))
    # touching x or y = 511 (ceil(511/16) + 1 = 33 > 32: the loop stops at the last cell)
    cases.append(("edge511", [[480, 100, 511, 130], [100, 490, 130, 511], [470, 470, 511, 511]], (0.0, 0.0), 1.0))
    # a scaled, shifted crop (im_scale != 1, crop origin != 0): rounding after the scale decides the side
    rng = np.random.RandomState(3)
    x = rng.uniform(300, 900, 30)
    y = rng.uniform(200, 700, 30)
    s = np.exp(rng.uniform(np.log(2), np.log(120), 30))
    cases.append(("scaled", np.stack([x, y, x + s, y + s * rng.uniform(0.5, 2, 30)], 1), (310.5, 190.25), 1.667))
    cases.append(("downscaled", np.stack([x, y, x + 3 * s, y + 2 * s], 1), (250.0, 150.0), 0.6))
    # more than 100 boxes on one chip (no cap at 100 for the mask).  At most 90 of them survive the worker's 10-px filter:
    # its gt_boxes table holds 100 rows and the reference worker cannot pack more (data_workers.py:365)
    n_big, n_small = 90, 60
    x = rng.uniform(0, 350, n_big)
    y = rng.uniform(0, 350, n_big)
    s = np.exp(rng.uniform(np.log(12), np.log(150), n_big))
    big = np.stack([x, y, x + s, y + s], 1)
    x = rng.uniform(0, 500, n_small)
    y = rng.uniform(0, 500, n_small)
    s = rng.uniform(1, 8, n_small)
    small = np.stack([x, y, x + s, y + s], 1)
    order = rng.permutation(n_big + n_small)
    cases.append(("many", np.concatenate([big, small])[order], (0.0, 0.0), 1.0))
    return [(nm, np.asarray(b, np.float32), c, sc) for nm, b, c, sc in cases]


FOCUS_CASES = _focus_cases()


@pytest.mark.parametrize("case", range(len(FOCUS_CASES)), ids=[c[0] for c in FOCUS_CASES])
def test_gen_mask_oracle_matches_reference_anchor_worker(case):
    """The iterator's focus boxes (chip_focus_boxes: shift, scale, round, clip, no filtering, no cap) rasterised by the
    float64 oracle == mask_scale of the reference's anchor_worker, bit for bit."""
    import focus_label_np as FL
    from sniper_b200 import iterator as IT
    name, boxes, crop, scale = FOCUS_CASES[case]
    ref = _ref_worker_mask(boxes, crop, scale)
    fb = IT.chip_focus_boxes([512, 512, scale], np.array(crop), scale, boxes)
    assert fb.shape == (len(boxes), 4)
    ours = FL.gen_mask(fb, 16, 32, 32, **AF)
    assert ours.dtype == np.float32 and ours.tobytes() == ref.tobytes()
    m = ref.reshape(32, 32)
    if name == "bands":
        assert (m == 1).any() and (m == -1).any() and (m == 0).any()
    if name == "outside":                           # the clipped, zero-area boxes leave -1 stripes on the border
        assert (m[:, 0] == -1).any() and (m[0, :] == -1).any() and (m[:, 31] == -1).any() and (m[31, :] == -1).any()
    if name == "many":
        assert len(boxes) > 100


def test_iterator_carries_focus_boxes():
    """MNIteratorE2E with TRAIN.AUTO_FOCUS: label_name gains scale_label and every raw batch carries, per chip, exactly
    chip_focus_boxes of the chip's GT (all of them, in GT order); without the flag the raw batch has no focus fields."""
    from sniper_b200 import iterator as IT
    cfg = IT.default_config()
    roidb = IT.synthetic_roidb(4, seed=2, n_prop=200)
    np.random.seed(4)
    it0 = IT.MNIteratorE2E(roidb, cfg, batch_size=4)
    assert it0.label_name == ['label', 'bbox_target', 'bbox_weight', 'gt_boxes']
    raw0 = next(iter(it0))
    assert not hasattr(raw0, "focus_boxes") or raw0.focus_boxes is None
    cfg.TRAIN.AUTO_FOCUS = True
    cfg.TRAIN.AUTO_FOCUS_DC_LOW, cfg.TRAIN.AUTO_FOCUS_SMALL_THRESH, cfg.TRAIN.AUTO_FOCUS_DC_HIGH = 5, 64, 90
    np.random.seed(4)
    it = IT.MNIteratorE2E(IT.synthetic_roidb(4, seed=2, n_prop=200), cfg, batch_size=4)
    assert it.label_name[-1] == 'scale_label'
    chips = [(it.roidb[it.inds[i]], it.roidb[it.inds[i]]['chip_order'][0]) for i in range(4)]    # the first batch
    raw = next(iter(it))
    off = raw.focus_off.numpy()
    assert off[0] == 0 and len(off) == 5
    import focus_label_np as FL
    for k, (r, cid) in enumerate(chips):
        crop = r['crops'][cid]
        gtids = np.where(r['max_overlaps'] == 1)[0]
        gt = r['boxes'][gtids, :]
        want = IT.chip_focus_boxes([512, 512, crop[1]], crop[0], crop[1], gt)
        got = raw.focus_boxes[off[k]:off[k + 1]].numpy()
        assert len(got) == len(gtids) and np.array_equal(got, want.astype(np.float32)), k
        # rasterised by the oracle: the reference worker's mask for the same chip
        ref = _ref_worker_mask(gt, np.asarray(crop[0], np.float64), crop[1])
        assert FL.gen_mask(got, 16, 32, 32, **AF).tobytes() == ref.tobytes(), k


# ------------------------------------------------------------------------------------------------ the network
@pytest.fixture
def f64():
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    yield
    torch.set_default_dtype(old)


def _net(monkeypatch, B, seed=5, autofocus=True):
    import fake_ops_autofocus as fake_ops
    from sniper_b200 import model, ops
    fake_ops.install(monkeypatch, ops)
    cfg = model.Cfg()
    cfg.batch_images, cfg.bf16, cfg.wgrad_stream, cfg.autofocus = B, False, False, autofocus
    net = model.SniperResNet101(cfg, device="cpu", seed=seed, deform_offset_std=0.01)
    g = torch.Generator().manual_seed(seed + 1)
    for bn in net._named_bns():
        if bn.name == "bn_data":
            continue
        lo, hi, sd = (0.15, 0.25, 0.02) if bn.name.endswith("_bn3") else (0.8, 1.2, 0.1)
        bn.st.gamma.copy_(torch.empty(bn.C).uniform_(lo, hi, generator=g))
        bn.st.beta.copy_(torch.empty(bn.C).normal_(0, sd, generator=g))
        if bn.frozen:
            bn.st.moving_mean.copy_(torch.empty(bn.C).normal_(0, 0.1, generator=g))
            bn.st.moving_var.copy_(torch.empty(bn.C).uniform_(0.6, 1.6, generator=g))
            ops.bn_frozen(bn.st, cfg.bn_eps)
    if autofocus:        # non-zero biases and a larger conv_new_out so that the focus softmax is not flat
        for c, sd in ((net.conv_new_2, 0.05), (net.conv_new_3, 0.05), (net.conv_new_out, 0.5)):
            c.b[:c.cout].copy_(torch.empty(c.cout).normal_(0, sd, generator=g))
        net.conv_new_out.master[:2].mul_(30.0)
    return cfg, net


def _batch(B, chip, seed=7):
    from sniper_b200 import synth_batch
    b = synth_batch.make_batch(B, seed=seed, device="cpu", chip=chip)
    b = {k: v.double() for k, v in b.items()}
    H = chip // 16
    rng = np.random.RandomState(seed)
    b["scale_label"] = torch.from_numpy(rng.choice([-1.0, 0.0, 1.0], (B, H * H), p=[0.3, 0.5, 0.2]))
    return b


def _rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def _proposals(out, batch, A=21):
    import oracle_lib as O
    prob = out["rpn_cls_prob"].permute(0, 3, 1, 2).contiguous()
    bbox = out["rpn_head"][..., :4 * A].permute(0, 3, 1, 2).contiguous()
    return O.multi_proposal_target(prob.numpy(), bbox.numpy(), batch["im_info"].numpy(), batch["gt_boxes"].numpy(),
                                   batch["valid_ranges"].numpy())


def test_autofocus_training_graph_matches_the_autograd_oracle(monkeypatch, f64):
    import torch_graph as TG
    import torch_graph_autofocus as TGA
    B, chip = 1, 256
    cfg, net = _net(monkeypatch, B)
    batch = _batch(B, chip)
    out = net.forward_backward(batch)
    res = _proposals(out, batch)
    assert out["rois"].numpy().astype(np.float32).tobytes() == res["rois"].tobytes()
    arg, aux = net.export_reference()
    assert arg["conv_new_out_weight"].shape == (2, 256, 1, 1) and arg["conv_new_2_weight"].shape == (256, 3072, 3, 3)
    P, Aux = TG.params_to_torch(arg, aux)
    TG.MODE[0] = "exact"
    obj, ref = TGA.forward_train(P, Aux, batch, lambda *_: res, batch_images=B)
    obj.backward()
    Hf = chip // 16
    sp = out["cls_scale_prob"]
    assert sp.shape == (B, Hf, Hf, 2)
    e_sp = _rel(sp.reshape(B, Hf * Hf, 2).permute(0, 2, 1), ref["cls_scale_prob"])
    assert e_sp < 1e-12, e_sp
    assert ref["cls_scale_prob"].min() < 0.3 and ref["cls_scale_prob"].max() > 0.7      # a non-trivial focus softmax
    assert ref["loss_sums"].shape == (5,)
    assert torch.allclose(out["losses"][:5], ref["loss_sums"], rtol=1e-7), (out["losses"][:5], ref["loss_sums"])
    lab = batch["scale_label"].reshape(-1).long()
    nvalid = int((lab != -1).sum())
    pred = (sp.reshape(-1, 2)[:, 1] > sp.reshape(-1, 2)[:, 0]).long()
    assert float(out["losses"][6]) == nvalid and float(out["losses"][5]) == int((pred == lab)[lab != -1].sum())
    garg, _ = net.export_reference(grads=True)
    rows = []
    for name, p in P.items():
        if not p.requires_grad:
            assert name not in garg, name
            continue
        assert p.grad is not None and garg[name].shape == tuple(p.grad.shape), name
        rows.append((_rel(torch.from_numpy(garg[name]), p.grad), name))
    rows.sort(reverse=True)
    print("worst gradient errors", rows[:5])
    assert len(rows) == 303
    # the bound of the default graph's test (the data-gradient operands are stored in fp32); the branch's own six
    # tensors sit above every fp32 operand store
    assert rows[0][0] < 1e-5, rows[:5]
    af = {n: e for e, n in rows if n.startswith("conv_new_") and n[9] in "23o"}
    print("AutoFocus gradient errors", af)
    assert len(af) == 6 and max(af.values()) < 1e-7, af
    # rows 2..31 of conv_new_out: zero weights, zero gradients
    assert not net.conv_new_out.master[2:].any() and not net.P.grad("conv_new_out_weight")[2:].any()
    assert not net.conv_new_out.b[2:].any() and not net.P.grad("conv_new_out_bias")[2:].any()
    assert net.P.grad("conv_new_out_weight")[:2].abs().sum() > 0


def test_autofocus_two_sgd_steps_match_the_reference_update_rule(monkeypatch, f64):
    """forward_backward + update() twice against the oracle graph + MXNet's SGD-momentum rule: the six new tensors are
    ordinary parameters (lr_mult 1, wd_mult 1 for weights / 0 for biases); the padding rows of conv_new_out stay zero."""
    import torch_graph as TG
    import torch_graph_autofocus as TGA
    B, chip = 1, 256
    cfg, net = _net(monkeypatch, B)
    batches = [_batch(B, chip), _batch(B, chip, seed=9)]
    arg, aux = net.export_reference()
    arg0 = {k: v.copy() for k, v in arg.items()}
    P, Aux = TG.params_to_torch(arg, aux)
    mom = {k: torch.zeros_like(v) for k, v in P.items() if v.requires_grad}
    TG.MODE[0] = "exact"
    for step, lr in enumerate((0.004, 0.011)):
        batch = batches[step]
        out = net.forward_backward(batch)
        res = _proposals(out, batch)
        net.update(lr=lr)
        for v in P.values():
            v.grad = None
        obj, _ = TGA.forward_train(P, Aux, batch, lambda *_: res, batch_images=B)
        obj.backward()
        with torch.no_grad():
            for k, m in mom.items():
                wd = cfg.wd if (k.endswith("_weight") or k.endswith("_gamma")) else 0.0
                lr_k = lr * (0.01 if k in ("offset_weight", "offset_bias") else 1.0)
                m.mul_(cfg.momentum).sub_(lr_k * (P[k].grad + wd * P[k]))
                P[k].add_(m)
    got, _ = net.export_reference()
    worst = sorted(((_rel(torch.from_numpy(got[k]), P[k]), k) for k in P), reverse=True)
    print("worst parameter errors after two updates", worst[:4])
    assert worst[0][0] < 2e-7, worst[:5]
    for k in ("conv_new_2_weight", "conv_new_2_bias", "conv_new_3_weight", "conv_new_3_bias", "conv_new_out_weight",
              "conv_new_out_bias"):
        assert not np.array_equal(got[k], arg0[k]), k
        assert _rel(torch.from_numpy(got[k]), P[k]) < 2e-7, k
    assert not net.conv_new_out.master[2:].any() and not net.conv_new_out.b[2:].any()


def test_autofocus_checkpoint_round_trip(monkeypatch, tmp_path):
    """export_reference -> save_checkpoint -> load_param -> load_reference restores the branch (OIHW, conv_new_out
    unpadded (2, 256, 1, 1)); forward_inference(autofocus=True) reads the trained layers."""
    from sniper_b200 import checkpoint as ck
    _, net = _net(monkeypatch, 1)
    arg, aux = net.export_reference()
    shapes = {"conv_new_2_weight": (256, 3072, 3, 3), "conv_new_2_bias": (256,), "conv_new_3_weight": (256, 256, 1, 1),
              "conv_new_3_bias": (256,), "conv_new_out_weight": (2, 256, 1, 1), "conv_new_out_bias": (2,)}
    for k, s in shapes.items():
        assert arg[k].shape == s, k
    arg = {k: v.astype(np.float32) for k, v in arg.items()}
    aux = {k: v.astype(np.float32) for k, v in aux.items()}
    ck.save_checkpoint(str(tmp_path / "af"), 1, arg, aux)
    a2, x2 = ck.load_param(str(tmp_path / "af"), 1)
    _, net2 = _net(monkeypatch, 1, seed=8)
    assert not np.array_equal(net2.export_reference()[0]["conv_new_2_weight"], arg["conv_new_2_weight"])
    assert net2.load_reference(a2, x2) == []
    back, _ = net2.export_reference()
    for k in shapes:
        assert np.array_equal(back[k].astype(np.float32), arg[k]), k
    assert net2.af == [net2.conv_new_2, net2.conv_new_3, net2.conv_new_out]
    assert not net2.conv_new_out.master[2:].any()
    with pytest.raises(RuntimeError):
        net2.enable_autofocus()


def test_default_configuration_layout_is_unchanged(monkeypatch):
    """Cfg() (autofocus off): 297 trainable tensors, no conv_new_2/3/out, and the parameter store's layout and gradient
    buckets are those of a network built before the AutoFocus layers existed (pinned numbers)."""
    _, net = _net(monkeypatch, 1, autofocus=False)
    P = net.P
    assert not any(n.startswith(("conv_new_2", "conv_new_3", "conv_new_out")) for n in P.layout)
    assert net.af is None and not net.af_train
    _, net_af = _net(monkeypatch, 1)
    extra = {n: s for n, (o, s) in net_af.P.layout.items() if n not in P.layout}
    assert sorted(extra) == ["conv_new_2_bias", "conv_new_2_weight", "conv_new_3_bias", "conv_new_3_weight",
                             "conv_new_out_bias", "conv_new_out_weight"]
    assert extra["conv_new_out_weight"] == (32, 256)
    n_extra = sum((int(np.prod(s)) + 3) // 4 * 4 for s in extra.values())
    assert net_af.P.total == P.total + n_extra
    # bucket 0 grows by exactly the branch; buckets 1 and 2 keep their sizes
    assert net_af.P.bucket_ranges[0][1] - net_af.P.bucket_ranges[0][0] == P.bucket_ranges[0][1] - P.bucket_ranges[0][0] + n_extra
    for k in (1, 2):
        assert net_af.P.bucket_ranges[k][1] - net_af.P.bucket_ranges[k][0] == P.bucket_ranges[k][1] - P.bucket_ranges[k][0]
    # the default layout itself, pinned to what the flat buffer looked like before the AutoFocus layers existed
    digest = hashlib.sha256(repr(sorted(P.layout.items())).encode()).hexdigest()[:16]
    assert (P.total, len(P.layout), digest) == (74199936, 293, "7ebaec71442817f7")
    assert P.bucket_ranges == [[0, 46894464], [46894464, 72981888], [72981888, 74199936]]
    arg, _ = net.export_reference()
    assert "conv_new_2_weight" not in arg


# ------------------------------------------------------------------------------------------------ symbols
def _yml_cfg(fp16=True):
    from types import SimpleNamespace as S
    return S(dataset=S(NUM_CLASSES=81), network=S(NUM_ANCHORS=21),
             TRAIN=S(AUTO_FOCUS=True, fp16=fp16, BATCH_IMAGES=20), TEST=S(AUTO_FOCUS=True))


def test_autofocus_train_symbol_matches_the_reference_graph():
    """NetSymbol(autofocus train) == the graph resnet_mx_101_e2e.py builds under sniper_res101_e2e_autofocus.yml with
    BATCH_IMAGES = 20 (tests/golden/ref_symbols_autofocus.json): argument names / shapes in order, auxiliary states, outputs in the
    reference's Group order [rpn_cls_prob, rpn_bbox_loss, cls_scale_prob, cls_prob, bbox_loss, label]."""
    from sniper_b200 import symbols
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_symbols_autofocus.json")))["resnet101_train_autofocus"]
    inst = symbols.resnet_mx_101_e2e(n_proposals=400, momentum=0.995)
    sym = inst.get_symbol_rcnn(_yml_cfg())
    shapes = {n: tuple(s) for n, s in gold["arguments"] if n in sym.data_names()}
    assert set(shapes) == set(sym.data_names()) and "scale_label" in shapes and shapes["scale_label"] == (20, 1024)
    arg_s, out_s, aux_s = sym.infer_shape(**shapes)
    ours = dict(zip(sym.list_arguments(), arg_s))
    theirs = {n: tuple(s) for n, s in gold["arguments"]}
    assert ours == theirs
    assert [n for n, _ in gold["auxiliary"]] == sym.list_auxiliary_states()
    assert [tuple(s) for _, s in gold["auxiliary"]] == [tuple(s) for s in aux_s]
    assert [n for n, _ in gold["outputs"]] == sym.list_outputs()
    assert [tuple(s) for _, s in gold["outputs"]] == [tuple(s) for s in out_s]
    assert sym.list_outputs()[2] == "cls_scale_prob_output"
    inst.infer_shape(shapes)
    arg = {}
    inst.init_weight_rcnn(_yml_cfg(), arg, {}, seed=1)
    for n in ("conv_new_2", "conv_new_3", "conv_new_out"):
        assert 0.009 < arg[n + "_weight"].std() < 0.011 and not arg[n + "_bias"].any()
    # without TRAIN.AUTO_FOCUS the symbol is the plain training graph
    plain = symbols.resnet_mx_101_e2e().get_symbol_rcnn(_yml_cfg().__class__(
        dataset=_yml_cfg().dataset, network=_yml_cfg().network, TRAIN=type(_yml_cfg().TRAIN)(AUTO_FOCUS=False)))
    assert "scale_label" not in plain.list_arguments() and len(plain.list_outputs()) == 5


def test_recognise_graph_reports_autofocus_train():
    """The reference's own symbol file under the AutoFocus yml, through mxnet_compat: recognised as the AutoFocus training
    graph, bf16 for the yml's fp16; the test graph keeps the inference route (enable_autofocus)."""
    if not os.path.isdir("/root/reference/symbols"):
        pytest.skip("needs the reference's symbol file (the stored description is checked above)")
    import run_ref_symbols as RS
    from sniper_b200 import mxnet_compat as MC
    from sniper_b200 import symbols
    res = MC.load_symbol_file("/root/reference/symbols/faster/resnet_mx_101_e2e.py")
    cfg = RS.load_config("sniper_res101_e2e_autofocus.yml")
    cfg.TRAIN.BATCH_IMAGES = 20
    with MC.NameManager():
        sym = res.resnet_mx_101_e2e(n_proposals=400, momentum=0.995).get_symbol_rcnn(cfg)
    info = symbols.recognise_graph(sym)
    assert info["autofocus_train"] and info["bf16"] and info["is_train"] and info["batch_images"] == 20
    # bound (here on the CPU stand-ins): a network that trains the branch -- not the inference-only enable_autofocus()
    import fake_ops_autofocus as fake_ops
    from sniper_b200 import ops
    mp = pytest.MonkeyPatch()
    try:
        fake_ops.install(mp, ops)
        net = symbols.bind_graph(sym, device="cpu", batch_images=2, wgrad_stream=False)
    finally:
        mp.undo()
    assert net.af_train and net.cfg.autofocus and net.cfg.bf16
    assert net.af == [net.conv_new_2, net.conv_new_3, net.conv_new_out] and all(c.trainable for c in net.af)
    assert "conv_new_2_weight" in net.P.layout
    with MC.NameManager():
        tsym = res.resnet_mx_101_e2e(n_proposals=400, momentum=0.995, test_nbatch=2).get_symbol_rcnn(cfg, is_train=False)
    tinfo = symbols.recognise_graph(tsym)
    assert tinfo["autofocus"] and "autofocus_train" not in tinfo and not tinfo["is_train"]
