"""TEST INFRASTRUCTURE: torch-CPU stand-ins for the two AutoFocus-training entry points of `sniper_b200.ops`
(sniper_focus_head, sniper_focus_label), in the style of tests/fake_ops.py (float64 arithmetic, one rounding to the dtype
the product stores).  `install` patches them over `sniper_b200.ops` together with every stand-in of fake_ops, so that
`SniperResNet101(Cfg(autofocus=True))` runs on the CPU against oracle/torch_graph_autofocus.py.  Never imported by the
product path."""
import numpy as np
import torch
import torch.nn.functional as F

import fake_ops


def focus_head(x3, w, b, label, grad_scale, valid_cnt, prob, dx3, dw, db, stats):
    """sniper_focus_head: conv_new_out (exact products, not a tensor-core contraction) + 2-way softmax + SoftmaxOutput's
    'valid' gradient, dx3 through conv_new_3's ReLU, dW / db accumulated, (log-loss sum, correct, valid) accumulated."""
    C = x3.shape[-1]
    x = x3.double().reshape(-1, C)
    w2, b2 = w.double()[:2], b.double()[:2]
    p = torch.softmax(x @ w2.t() + b2, 1)
    lab = label.reshape(-1).long()
    valid = lab != -1
    v = int(valid_cnt.reshape(-1)[0].item())
    norm = grad_scale / max(v, 1)
    onehot = F.one_hot(lab.clamp(min=0), 2).to(p.dtype)
    dz = torch.where(valid.unsqueeze(1), (p - onehot) * norm, torch.zeros_like(p))
    prob.copy_(p.reshape(prob.shape))
    dx3.copy_(((dz @ w2) * (x > 0)).reshape(dx3.shape))
    dw[:2] += (dz.t() @ x).to(dw.dtype)
    db[:2] += dz.sum(0).to(db.dtype)
    pl = p.gather(1, lab.clamp(min=0).unsqueeze(1)).squeeze(1).clamp(min=1e-14)
    stats[0] += -(torch.log(pl)[valid]).sum()
    stats[1] += float(((p[:, 1] > p[:, 0]).long() == lab)[valid].sum())
    stats[2] += float(v)


def focus_label(boxes, offsets, B, *, H=32, W=32, feat_stride=16, dc_low=5, small_thresh=64, dc_high=90, out=None):
    """sniper_focus_label through the float64 restatement of gen_mask (oracle/focus_label_np.py)."""
    import focus_label_np as FL
    bx, off = boxes.detach().cpu().numpy().astype(np.float64), offsets.detach().cpu().numpy()
    res = np.stack([FL.gen_mask(bx[off[b]:off[b + 1]], feat_stride, H, W, dc_low, small_thresh, dc_high)
                    for b in range(B)])
    t = torch.from_numpy(res.astype(np.float32))
    if out is None:
        return t
    out.copy_(t)
    return out


def install(monkeypatch, ops_module):
    fake_ops.install(monkeypatch, ops_module)
    for k in ("focus_head", "focus_label"):
        monkeypatch.setattr(ops_module, k, globals()[k])
