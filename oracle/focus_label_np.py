"""ORACLE -- test infrastructure only.  Float64 numpy restatement of the AutoFocus FocusPixel label `gen_mask`
(anchor_worker.worker, lib/data_utils/data_workers.py:165-192; called at :220-222 on the chip's GT boxes after the shift
into the chip, the scale, np.round and clip_boxes, BEFORE filter_boxes drops the small ones).

    side = sqrt((x2 - x1) * (y2 - y1))                (no +1)
    flag = 1   if DC_LOW < side < SMALL
           -1  if SMALL <= side < DC_HIGH  or  side <= DC_LOW
           none (the box writes nothing) if side >= DC_HIGH
    cells: columns int(x1 / stride) .. min(ceil(x2 / stride) + 1, W) - 1, rows likewise (one past the ceiling)
    boxes in GT order, the last box that writes a cell wins, uncovered cells are 0.

Pinned against the reference's own anchor_worker (oracle/run_ref_anchor_worker.py with AUTO_FOCUS on) by
tests/test_autofocus_train_cpu.py, and the device kernel sniper_focus_label against this by the GPU test."""
import math

import numpy as np


def gen_mask(boxes, feat_stride=16, H=32, W=32, dc_low=5, small_thresh=64, dc_high=90):
    """boxes [n,4] (chip coordinates, rounded and clipped) -> scale_label [H*W] float32 in {-1, 0, 1}."""
    mask = np.zeros((H, W), np.float32)
    for x1, y1, x2, y2 in np.asarray(boxes, np.float64).reshape(-1, 4)[:, :4]:
        side = math.sqrt((x2 - x1) * (y2 - y1))
        if dc_low < side < small_thresh:
            flag = 1.0
        elif small_thresh <= side < dc_high or side <= dc_low:
            flag = -1.0
        else:
            continue
        cx1, cy1 = int(x1 / feat_stride), int(y1 / feat_stride)
        cx2, cy2 = min(int(math.ceil(x2 / feat_stride)) + 1, W), min(int(math.ceil(y2 / feat_stride)) + 1, H)
        if cx2 > cx1 and cy2 > cy1:
            mask[cy1:cy2, cx1:cx2] = flag
    return mask.reshape(H * W)
