"""AutoFocus training on the B200: the two kernels against their float64 restatements, the input stage with
TRAIN.AUTO_FOCUS, one whole training step against oracle/torch_graph_autofocus.forward_train in torch_graph's "tf32" mode,
and the CUDA-graph trainer from the iterator's raw batches."""
import math
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

AF = dict(dc_low=5, small_thresh=64, dc_high=90)


def _rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).norm() / (b.norm() + 1e-30)).item()


def _af_config(on=True):
    from sniper_b200 import iterator as IT
    cfg = IT.default_config()
    if on:
        cfg.TRAIN.AUTO_FOCUS = True
        cfg.TRAIN.AUTO_FOCUS_DC_LOW, cfg.TRAIN.AUTO_FOCUS_SMALL_THRESH = AF["dc_low"], AF["small_thresh"]
        cfg.TRAIN.AUTO_FOCUS_DC_HIGH = AF["dc_high"]
    return cfg


# ------------------------------------------------------------------------------------------------ sniper_focus_label
def _random_chip_boxes(rng, n):
    """integer chip boxes like the iterator produces (rounded, clipped to [0, 511]), including zero-area border boxes,
    sides on the band edges and boxes touching 511"""
    x1 = rng.randint(-60, 540, n).astype(np.float64)
    y1 = rng.randint(-60, 540, n).astype(np.float64)
    side = np.where(rng.rand(n) < 0.3, rng.choice([5, 6, 63, 64, 65, 89, 90, 91], n), rng.randint(0, 200, n))
    asp = rng.choice([1, 1, 1, 2, 4], n)
    b = np.stack([x1, y1, x1 + side * asp, y1 + side], 1)
    return np.clip(b, 0, 511).astype(np.float32)


def test_focus_label_bit_exact():
    """sniper_focus_label == oracle/focus_label_np.gen_mask bit for bit: on the CPU test's fixture cases (the chip
    boxes the iterator derives from them) and on a batch of 20 chips with up to 150 boxes each."""
    import torch
    import focus_label_np as FL
    import test_autofocus_train_cpu as C
    from sniper_b200 import iterator as IT, ops
    chips = [IT.chip_focus_boxes([512, 512, sc], np.array(crop), sc, b).astype(np.float32) for _, b, crop, sc in C.FOCUS_CASES]
    rng = np.random.RandomState(11)
    chips += [_random_chip_boxes(rng, int(rng.randint(0, 151))) for _ in range(20)]
    chips.append(np.zeros((0, 4), np.float32))                       # a chip without GT: all zeros
    off = np.concatenate([[0], np.cumsum([len(c) for c in chips])]).astype(np.int32)
    boxes = torch.from_numpy(np.concatenate(chips)).cuda()
    lab = ops.focus_label(boxes, torch.from_numpy(off).cuda(), len(chips), **AF)
    torch.cuda.synchronize()
    want = np.stack([FL.gen_mask(c, 16, 32, 32, **AF) for c in chips])
    got = lab.cpu().numpy()
    assert got.tobytes() == want.tobytes(), np.argwhere(got != want)[:10]
    assert (want == 1).sum() > 100 and (want == -1).sum() > 100 and max(len(c) for c in chips) > 100


def test_input_stage_with_autofocus():
    """InputStage.run with TRAIN.AUTO_FOCUS: the seven existing tensors are bit-identical to a run without the flag on
    the same raw batch, and scale_label is the oracle's mask of the raw batch's focus boxes."""
    import torch
    import focus_label_np as FL
    from sniper_b200 import iterator as IT
    B = 8
    np.random.seed(5)
    it = IT.MNIteratorE2E(IT.synthetic_roidb(6, seed=3, n_gt=(1, 40), n_prop=200), _af_config(), batch_size=B)
    raw = next(iter(it))
    off = raw.focus_off.numpy().copy()
    plain = IT.InputStage(_af_config(False), "cuda", B).run(raw)
    plain = {k: v.clone() for k, v in plain.items()}
    withaf = IT.InputStage(_af_config(), "cuda", B).run(raw)
    torch.cuda.synchronize()
    assert set(withaf) == set(plain) | {"scale_label"}
    for k, v in plain.items():
        assert torch.equal(v, withaf[k]), k
    fb = raw.focus_boxes.numpy()
    want = np.stack([FL.gen_mask(fb[off[b]:off[b + 1]], 16, 32, 32, **AF) for b in range(B)])
    got = withaf["scale_label"].cpu().numpy()
    assert got.shape == (B, 1024) and got.tobytes() == want.tobytes()


# ------------------------------------------------------------------------------------------------ sniper_focus_head
def test_focus_head_against_float64():
    """sniper_focus_head on M = 20480 rows (20 chips x 32 x 32) against float64 torch, grad_scale 3, with mixed, all-ignored
    and all-valid labels.  Tolerances from the fp32 accumulation depth: a logit is a 256-term fp32 dot product (relative
    error <~ 256 * 2^-24 = 1.5e-5 worst case, ~1e-6 typical), prob inherits it (abs 1e-5); dx3 is two fp32 products
    (rel 1e-6); dW / db sum 20480 rows in fp32 partial sums of ~4 rows per warp, 8 warps per block and a float atomic per
    block (rel. Frobenius 1e-5); the loss sum is ~10^4 fp32 terms (rel 1e-5); the correct count is exact away from ties
    (|z1 - z0| < 1e-4 excluded).  The ReLU mask is exact: dx3 == 0 wherever x3 == 0."""
    import torch
    from sniper_b200 import ops
    torch.manual_seed(0)
    M, C = 20480, 256
    x = torch.relu(torch.randn(M, C, device="cuda") * 0.7 + 0.1)
    w = torch.zeros(32, C, device="cuda")
    w[:2] = torch.randn(2, C, device="cuda") * 0.1
    b = torch.zeros(32, device="cuda")
    b[:2] = torch.tensor([0.3, -0.2])
    gs = 3.0
    labels = dict(mixed=torch.randint(-1, 2, (M,), device="cuda").float(), ignored=torch.full((M,), -1.0, device="cuda"),
                  valid=torch.randint(0, 2, (M,), device="cuda").float())
    for name, lab in labels.items():
        cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
        ops.count_valid(lab, cnt)
        prob = torch.empty(M, 2, device="cuda")
        dx = torch.empty_like(x)
        dw = torch.full((32, C), 0.5, device="cuda")             # accumulated into: starts non-zero
        db = torch.full((32,), 0.25, device="cuda")
        stats = torch.zeros(3, device="cuda")
        ops.focus_head(x, w, b, lab, gs, cnt, prob, dx, dw, db, stats)
        torch.cuda.synchronize()
        xd, wd, bd = x.double(), w[:2].double(), b[:2].double()
        z = xd @ wd.t() + bd
        p = torch.softmax(z, 1)
        li = lab.long()
        valid = li != -1
        nv = int(valid.sum())
        dz = torch.where(valid[:, None], (p - torch.nn.functional.one_hot(li.clamp(min=0), 2).double()) * gs / max(nv, 1),
                         torch.zeros_like(p))
        dx_ref = (dz @ wd) * (xd > 0)
        dw_ref = dz.t() @ xd
        db_ref = dz.sum(0)
        loss_ref = -(torch.log(p.gather(1, li.clamp(min=0)[:, None]).squeeze(1))[valid]).sum().item()
        sure = valid & ((z[:, 1] - z[:, 0]).abs() > 1e-4)
        cor_ref = int(((z[:, 1] > z[:, 0]).long() == li)[sure].sum())
        e = dict(prob=(prob.double() - p).abs().max().item(), dx=_rel(dx, dx_ref) if nv else dx.abs().max().item(),
                 dw=_rel(dw[:2] - 0.5, dw_ref) if nv else (dw[:2] - 0.5).abs().max().item(),
                 db=_rel(db[:2] - 0.25, db_ref) if nv else (db[:2] - 0.25).abs().max().item())
        print(name, "valid", nv, {k: "%.2e" % v for k, v in e.items()}, "loss", stats[0].item(), loss_ref)
        assert e["prob"] < 1e-5 and e["dx"] < 1e-5 and e["dw"] < 1e-5 and e["db"] < 1e-5, (name, e)
        assert bool((dx[x == 0] == 0).all())                                             # ReLU mask exact
        assert bool((dw[2:] == 0.5).all()) and bool((db[2:] == 0.25).all())              # padding rows untouched
        assert abs(stats[0].item() - loss_ref) <= 1e-5 * abs(loss_ref) + 1e-6
        assert stats[2].item() == nv
        n_cor = stats[1].item()
        unsure = int((valid & ~sure).sum())
        assert cor_ref <= n_cor <= cor_ref + unsure
        if name == "ignored":
            assert nv == 0 and stats[0].item() == 0 and stats[1].item() == 0 and not dx.any()


# ------------------------------------------------------------------------------------------------ whole step
# Measured on one B200 (NVIDIA B200, 1000 W power limit; 2 chips, seeds 5 / 7), against the oracle's "tf32" mode:
#   loss sums rel 4.3e-5 / 3.0e-4 / 6.9e-8 / 3.0e-6 and the focus loss sum 2.9e-6;
#   branch gradients conv_new_2 w / b 7.9e-3 / 4.2e-3, conv_new_3 w / b 3.5e-3 / 2.4e-3, conv_new_out w / b 2.7e-4 / 1.2e-4;
#   cls_scale_prob max abs 1.0e-2 (the focus softmax is steep here: conv_new_out scaled x30).
# Bounds: those of tests/test_graph_parity_gpu.py TOL_TF32 -- loss sums 5e-3, head gradients 8e-2, activations 1e-2 rel.
# Frobenius (cls_scale_prob) -- and for the kernel's own output, conv_new_out's gradient, 1e-3.
TOL = dict(loss=5e-3, head=8e-2, act=1e-2, out_grad=1e-3)


def test_autofocus_step_matches_tf32_oracle():
    import torch
    import oracle_lib as O
    import torch_graph as TG
    import torch_graph_autofocus as TGA
    from sniper_b200 import model, ops, synth_batch
    B, seed = 2, 5
    cfg = model.Cfg()
    cfg.batch_images, cfg.autofocus = B, True
    net = model.SniperResNet101(cfg, deform_offset_std=0.01, seed=seed)
    g = torch.Generator(device="cuda")
    g.manual_seed(seed + 1)
    for bn in net._named_bns():
        if bn.name == "bn_data":
            continue
        lo, hi, sd = (0.15, 0.25, 0.02) if bn.name.endswith("_bn3") else (0.8, 1.2, 0.1)
        bn.st.gamma.copy_(torch.empty(bn.C, device="cuda").uniform_(lo, hi, generator=g))
        bn.st.beta.copy_(torch.empty(bn.C, device="cuda").normal_(0, sd, generator=g))
        if bn.frozen:
            bn.st.moving_mean.copy_(torch.empty(bn.C, device="cuda").normal_(0, 0.1, generator=g))
            bn.st.moving_var.copy_(torch.empty(bn.C, device="cuda").uniform_(0.6, 1.6, generator=g))
            ops.bn_frozen(bn.st, cfg.bn_eps)
    net.conv_new_out.master[:2].mul_(30.0)          # a focus softmax away from 1/2
    batch = synth_batch.make_batch(B, seed=7, device="cuda")
    rng = np.random.RandomState(7)
    batch["scale_label"] = torch.from_numpy(rng.choice([-1.0, 0.0, 1.0], (B, 1024), p=[0.3, 0.5, 0.2]).astype(np.float32)).cuda()
    out = net.forward_backward(batch)
    torch.cuda.synchronize()
    A = cfg.num_anchors
    prob = out["rpn_cls_prob"].permute(0, 3, 1, 2).contiguous()
    bbox = out["rpn_head"][..., :4 * A].permute(0, 3, 1, 2).contiguous()
    garg, _ = net.export_reference(grads=True)
    ls = out["losses"][:5].double().cpu()
    arg, aux = net.export_reference()
    res = O.multi_proposal_target(prob.cpu().numpy(), bbox.cpu().numpy(), batch["im_info"].cpu().numpy(),
                                  batch["gt_boxes"].cpu().numpy(), batch["valid_ranges"].cpu().numpy())
    assert out["rois"].cpu().numpy().tobytes() == res["rois"].tobytes()
    assert np.array_equal(out["label"].cpu().numpy(), res["label"].reshape(-1))
    P, Aux = TG.params_to_torch(arg, aux, torch.float64, "cuda")
    b64 = {k: v.double() for k, v in batch.items()}
    TG.MODE[0] = "tf32"
    try:
        obj, ref = TGA.forward_train(P, Aux, b64, lambda *_: res, batch_images=B)
        obj.backward()
    finally:
        TG.MODE[0] = "exact"
        TG.LOWP[0] = False
    lr_ = ref["loss_sums"].cpu()
    e_loss = [abs(ls[i] - lr_[i]).item() / (abs(lr_[i]).item() + 1e-30) for i in range(5)]
    sp = out["cls_scale_prob"].reshape(B, 1024, 2).permute(0, 2, 1)
    e_sp = _rel(sp, ref["cls_scale_prob"])
    rows = {n: _rel(torch.from_numpy(garg[n]).cuda(), P[n].grad) for n in garg if n.startswith(("conv_new_2", "conv_new_3",
                                                                                                  "conv_new_out"))}
    print("loss sums ours", ls.tolist(), "tf32-ref", lr_.tolist(), "rel", ["%.1e" % v for v in e_loss])
    print("cls_scale_prob rel err %.2e max abs %.2e" % (e_sp, (sp.double() - ref["cls_scale_prob"]).abs().max().item()), "branch gradient errors", {k: "%.2e" % v for k, v in rows.items()})
    assert len(rows) == 6
    for i in range(5):
        assert abs(ls[i] - lr_[i]) <= TOL["loss"] * abs(lr_[i]) + 1e-4, (i, ls[i].item(), lr_[i].item())
    assert e_sp < TOL["act"]
    for n, r in rows.items():
        assert r < (TOL["out_grad"] if n.startswith("conv_new_out") else TOL["head"]), (n, r)
    assert not net.conv_new_out.master[2:].any() and not net.P.grad("conv_new_out_weight")[2:].any()


# ------------------------------------------------------------------------------------------------ trainer
@pytest.mark.parametrize("bf16", [False, True])
def test_trainer_step_raw_autofocus(bf16):
    """Iterator (TRAIN.AUTO_FOCUS) -> InputStage -> Trainer.step_raw under CUDA graphs at a fixed lr: the AutoFocus
    metrics are reported, finite, and the focus log-loss falls over the run; the padding rows of conv_new_out stay zero;
    forward_inference(autofocus=True) then reads the trained branch."""
    import torch
    from sniper_b200 import iterator as IT, model, trainer
    B, steps = 4, 24 if not bf16 else 6
    cfg = model.Cfg()
    cfg.batch_images, cfg.autofocus, cfg.bf16 = B, True, bf16
    tr = trainer.Trainer(cfg, use_graph=True, seed=5, scheduler=None)
    np.random.seed(2)
    it = IT.MNIteratorE2E(IT.synthetic_roidb(3, seed=4, n_gt=(5, 30), n_prop=200), _af_config(), batch_size=B)
    stage = IT.InputStage(_af_config(), "cuda", B)
    hist = []
    for k in range(steps):
        if not it.get_batch():
            it.reset()
            it.get_batch()
        r = tr.step_raw(it.batch, stage, lr=0.004)
        assert all(math.isfinite(r[k2]) for k2 in ("rpn_cls_loss", "rpn_bbox_loss", "rcnn_cls_loss", "rcnn_bbox_loss"))
        assert set(r) >= {"autofocus_logloss", "autofocus_acc"}
        assert math.isfinite(r["autofocus_logloss"]) and 0.0 <= r["autofocus_acc"] <= 1.0
        hist.append(r["autofocus_logloss"])
    assert tr.g_fb is not None
    net = tr.net
    assert not net.conv_new_out.master[2:].any() and not net.conv_new_out.b[2:].any()
    assert bool(torch.isfinite(net.P.w).all())
    print("autofocus log-loss", ["%.3f" % v for v in hist])
    if not bf16:
        assert np.mean(hist[-4:]) < np.mean(hist[:4]) - 0.02, hist
    data = tr.static["data"]
    rois, _, _, _, fmap = net.forward_inference(data, tr.static["im_info"], autofocus=True)
    torch.cuda.synchronize()
    assert fmap.shape == (B, 32, 32) and bool(torch.isfinite(fmap).all())
