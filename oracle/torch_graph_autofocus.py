"""ORACLE -- test infrastructure only.  The AutoFocus TRAINING graph (`get_symbol_rcnn(is_train=True)` with
TRAIN.AUTO_FOCUS, symbols/faster/resnet_mx_101_e2e.py:239-240, 259-267, 313-315, 335-336) on top of
oracle/torch_graph.forward_train: the FocusPixel branch conv_new_2 (3x3, pad 1) -> ReLU -> conv_new_3 (1x1) -> ReLU ->
conv_new_out (1x1, 2 channels) on relu1, and SoftmaxOutput('cls_scale_prob', multi_output, normalization='valid',
use_ignore, ignore_label=-1) against batch["scale_label"] [B, H*W]: the objective gains grad_scale * sum(nll) /
max(#valid, 1), like the RPN term.  conv_new_2 / conv_new_3 follow torch_graph.MODE like every other head convolution;
conv_new_out is an FP32-FMA contraction in the product (sniper_focus_head), so MODE "tf32" leaves it untruncated."""
import torch
import torch.nn.functional as F

import torch_graph as TG


def forward_train(P, A, batch, proposals, batch_images, grad_scale=1.0, **kw):
    """torch_graph.forward_train + the AutoFocus branch and loss.  Returns (objective, out); out gains cls_scale_prob
    (B, 2, H*W) (the reference's layout) and a fifth loss sum (the focus log-loss sum) in loss_sums."""
    objective, out = TG.forward_train(P, A, batch, proposals, batch_images, grad_scale=grad_scale, **kw)
    relu1 = out["relu1"]
    B = relu1.shape[0]
    f = F.relu(TG.conv2d(relu1, P["conv_new_2_weight"], P["conv_new_2_bias"], 1, 1))
    f = F.relu(TG.conv2d(f, P["conv_new_3_weight"], P["conv_new_3_bias"]))
    z = TG.conv2d(f, P["conv_new_out_weight"], P["conv_new_out_bias"], exact=True).reshape(B, 2, -1)
    label = batch["scale_label"].reshape(B, -1).long()
    logp = F.log_softmax(z, 1)
    valid = label != -1
    loss_sum = -(logp.gather(1, label.clamp(min=0).unsqueeze(1)).squeeze(1))[valid].sum()
    objective = objective + grad_scale * loss_sum / max(int(valid.sum()), 1)
    out["cls_scale_prob"] = logp.exp()
    out["loss_sums"] = torch.cat([out["loss_sums"], loss_sum.detach().reshape(1)])
    return objective, out
