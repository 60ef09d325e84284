"""The SNIPER training iterator with a GPU input stage.

Host side (`MNIteratorE2E`): same construction arguments, epoch logic and per-chip bookkeeping as the reference's
lib/iterators/MNIteratorE2E.py -- `reset()` (:41-105: chip extraction, box assignment and negative-chip mining through
`chip_worker`, <= 2 negative chips per image, padding of the chip list to a multiple of the batch, permutation) and
`_get_batch()` (:112-219: chip selection through `chip_order` / `crop_idx`, valid ranges, im_info, the GT bookkeeping in
front of the anchor matching, data_workers.py:194-281) -- but instead of resizing pixels and matching anchors in a
`Pool(64)` of host processes it emits a small pinned **raw batch**: the uint8 source rectangle of every chip, a chip
table, and the (valid GT, invalid GT, gt_boxes) arrays.

Device side (`InputStage`): one H2D copy of that raw batch, then `sniper_chip_input` (flip + cv2-style bilinear resize
+ pad + BGR->RGB + mean subtraction, data_workers.py:80-121), `sniper_anchor_target` (anchor matching, :283-363) and
`sniper_anchor_subsample` (the npr.choice subsampling, :326-338) fill exactly the tensors `MNIteratorE2E.provide_data /
provide_label` name: data, valid_ranges, im_info, label, bbox_target, bbox_weight, gt_boxes (SURVEY appendix B.5).

What stays on the host is what north_star keeps there: lib/chips sampling and the iterator's index logic.
"""
import math

import numpy as np
import torch

from . import host, ops
from ._lib import check, lib
from .chip_worker import chip_worker


def _clip(boxes, im_shape):
    """bbox_transform.clip_boxes (lib/bbox/bbox_transform.py:35-50), in place like the reference."""
    boxes[:, 0::4] = np.maximum(np.minimum(boxes[:, 0::4], im_shape[1] - 1), 0)
    boxes[:, 1::4] = np.maximum(np.minimum(boxes[:, 1::4], im_shape[0] - 1), 0)
    boxes[:, 2::4] = np.maximum(np.minimum(boxes[:, 2::4], im_shape[1] - 1), 0)
    boxes[:, 3::4] = np.maximum(np.minimum(boxes[:, 3::4], im_shape[0] - 1), 0)
    return boxes


def _big_enough(boxes, min_size):
    ws = boxes[:, 2] - boxes[:, 0] + 1
    hs = boxes[:, 3] - boxes[:, 1] + 1
    return np.where((ws >= min_size) & (hs >= min_size))[0]


def _to_chip(b, cur_crop, im_scale, im_info):
    """The first step of anchor_worker.worker on GT boxes (data_workers.py:210-220): shift into the chip (in place, like
    the reference), scale, round, clip to the chip."""
    b[:, 0] -= cur_crop[0]
    b[:, 2] -= cur_crop[0]
    b[:, 1] -= cur_crop[1]
    b[:, 3] -= cur_crop[1]
    return _clip(np.round(b * im_scale), im_info[:2])


def chip_focus_boxes(im_info, cur_crop, im_scale, gt_boxes):
    """The boxes AutoFocus's gen_mask rasterises (data_workers.py:220-222): EVERY GT box of the image in roidb order,
    shifted / scaled / rounded / clipped like chip_ground_truth's, before its 10-px filter and without its cap at
    max_n_gts.  Boxes outside the chip collapse onto its border (zero area)."""
    return _to_chip(np.array(gt_boxes, copy=True), cur_crop, im_scale, im_info)


def chip_ground_truth(im_info, cur_crop, im_scale, nids, gtids, gt_boxes, boxes, classes, max_n_gts=100):
    """The GT bookkeeping of anchor_worker.worker in front of the anchor matching (data_workers.py:194-281):
    shift into the chip, scale, round, clip to the chip, drop boxes under 10 px, then split the chip's GT into
    `valid` (GT this chip is responsible for: it coincides with a box of props_in_chips) and `invalid` (other GT that
    fall into the chip: anchors on them are ignored).  Returns (valid [n,4], invalid [m,4], gt_boxes [max_n_gts,5])."""
    gt_boxes = np.array(gt_boxes, copy=True)
    boxes = np.asarray(boxes)
    vgt = boxes[np.intersect1d(gtids, nids)]          # fancy indexing: a copy
    gt_boxes = _to_chip(gt_boxes, cur_crop, im_scale, im_info)
    vgt = _to_chip(vgt, cur_crop, im_scale, im_info)
    ids = _big_enough(gt_boxes, 10)
    if len(ids) == 0:
        gt_boxes = np.zeros((0, 4))
        classes = np.zeros((0, 1))
    else:
        gt_boxes = gt_boxes[ids]
        classes = classes[ids]
    all_gt = gt_boxes.copy()
    ids = _big_enough(vgt, 10)
    vgt = vgt[ids] if len(ids) > 0 else np.zeros((0, 4))
    if len(vgt) > 0 and len(gt_boxes) > 0:
        mov = host.bbox_overlaps(gt_boxes.astype(float), vgt.astype(float)).max(axis=1)
    else:
        mov = np.zeros((len(gt_boxes)))
    invalid = gt_boxes[np.where(mov < 1)[0], :]
    valid = gt_boxes[np.where(mov == 1)[0], :]
    fgt = -np.ones((max_n_gts, 5))
    if len(all_gt) > 0:
        k = min(len(all_gt), max_n_gts)
        fgt[:k, :] = np.hstack((all_gt, classes))[:k]
    return valid, invalid, fgt


class RawBatch(object):
    """Pinned host buffers of one batch (what crosses PCIe): source pixels + small per-chip arrays."""

    def __init__(self, B, max_gt, pixel_capacity):
        pin = self.pin
        self.pixels = pin(pixel_capacity, dtype=torch.uint8)
        self.table = pin(B, 8, dtype=torch.int64)
        self.valid_ranges = pin(B, 2, dtype=torch.float32)
        self.im_info = pin(B, 3, dtype=torch.float32)
        self.gt_valid = pin(B, max_gt, 4, dtype=torch.float32)
        self.ngt = pin(B, dtype=torch.int32)
        self.gt_invalid = pin(B, max_gt, 4, dtype=torch.float32)
        self.ninv = pin(B, dtype=torch.int32)
        self.gt_boxes = pin(B, max_gt, 5, dtype=torch.float32)
        self.anchor_im_info = pin(B, 3, dtype=torch.float32)
        self.used_pixels = 0
        self.seed = 0
        # TRAIN.AUTO_FOCUS only: every chip's focus boxes (chip_focus_boxes) back to back, chip b owning rows
        # [focus_off[b], focus_off[b+1]); focus_boxes grows with the largest batch seen
        self.focus_boxes = None
        self.focus_off = None

    @staticmethod
    def pin(*s, dtype):
        t = torch.zeros(*s, dtype=dtype)
        return t.pin_memory() if torch.cuda.is_available() else t    # host-only use (no GPU): plain pageable buffers

    def nbytes(self):
        small = (self.table, self.valid_ranges, self.im_info, self.gt_valid, self.ngt, self.gt_invalid, self.ninv,
                 self.gt_boxes, self.anchor_im_info)
        n = int(self.used_pixels + sum(t.numel() * t.element_size() for t in small))
        if self.focus_off is not None:
            n += int(self.focus_off.numel() * 4 + int(self.focus_off[-1]) * 16)
        return n


class MNIteratorE2E(object):
    def __init__(self, roidb, config, batch_size=4, threads=8, nGPUs=1, pad_rois_to=400, crop_size=(512, 512),
                 image_loader=None, n_buffers=3):
        """roidb entries: 'image' (path) or 'image_data' (decoded uint8 HxWx3 BGR), 'width', 'height', 'boxes' [n,4],
        'max_overlaps' (== 1 for GT rows), 'max_classes', 'flipped'.  image_loader(path) -> uint8 BGR array replaces
        cv2.imread (this image has no OpenCV)."""
        assert batch_size % nGPUs == 0, 'batch_size should be divisible by number of GPUs'
        self.roidb = roidb
        self.cfg = config
        self.batch_size = batch_size
        self.crop_size = crop_size
        self.image_loader = image_loader
        self.pixel_mean = config.network.PIXEL_MEANS
        self.chip_worker = chip_worker(chip_size=self.crop_size[0], cfg=config)
        self.max_gt = 100
        self.data_name = ['data', 'valid_ranges', 'im_info']
        self.label_name = ['label', 'bbox_target', 'bbox_weight', 'gt_boxes']
        self.auto_focus = bool(getattr(config.TRAIN, "AUTO_FOCUS", False))
        if self.auto_focus:                   # MNIteratorE2E.py:28-29: the FocusPixel labels of AutoFocus training
            self.label_name.append('scale_label')
        self.epiter = 0
        # the largest source rectangle of a chip: crop_size / (smallest scale factor) on each side, x3 channels
        self._buffers = [None] * n_buffers
        self._next_buffer = 0
        self.batch = None
        self.reset()

    # ---------------------------------------------------------------- epoch (MNIteratorE2E.py:41-105)
    def reset(self):
        self.cur_i = 0
        self.n_neg_per_im = 2
        self.crop_idx = [0] * len(self.roidb)
        self.chip_worker.reset()
        chip_count = 0
        for r in self.roidb:
            r['crops'] = self.chip_worker.chip_extractor(r)
            chip_count += len(r['crops'])
        for r in self.roidb:
            ps = self.chip_worker.box_assigner(r)
            r['props_in_chips'] = ps[0]
            if self.cfg.TRAIN.USE_NEG_CHIPS:
                r['neg_crops'] = ps[1]
                r['neg_props_in_chips'] = ps[2]
        chipindex = []
        for i, r in enumerate(self.roidb):
            if self.cfg.TRAIN.USE_NEG_CHIPS:
                cs = r['neg_crops']
                if len(cs) > 0:
                    sel_inds = np.arange(len(cs))
                    if len(cs) > self.n_neg_per_im:
                        sel_inds = np.random.permutation(sel_inds)[0:self.n_neg_per_im]
                    for ind in sel_inds:
                        chip_count += 1
                        r['crops'].append(r['neg_crops'][ind])
                        r['props_in_chips'].append(r['neg_props_in_chips'][ind].astype(np.int32))
            chipindex += [i] * len(r['crops'])
        self.chip_count = chip_count
        chipindex = np.array(chipindex)
        if chipindex.shape[0] % self.batch_size > 0:
            extra = self.batch_size - (chipindex.shape[0] % self.batch_size)
            chipindex = np.hstack((chipindex, chipindex[0:extra]))
        self.inds = np.array(np.random.permutation(chipindex), dtype=int)
        for r in self.roidb:
            r['chip_order'] = np.random.permutation(np.arange(len(r['crops'])))
        self.epiter += 1
        self.size = len(self.inds)

    def __len__(self):
        return len(self.inds)

    def __iter__(self):
        return self

    def __next__(self):
        if not self.get_batch():
            raise StopIteration
        return self.batch

    next = __next__

    def get_batch(self):
        if self.cur_i >= self.size:
            return False
        self.batch = self._get_batch()
        self.cur_i += self.batch_size
        return True

    # ---------------------------------------------------------------- one batch (MNIteratorE2E.py:112-219)
    def _image(self, r):
        if 'image_data' in r:
            return r['image_data']
        if self.image_loader is None:
            raise RuntimeError("roidb entry has no 'image_data' and no image_loader was given (no OpenCV in this image)")
        return self.image_loader(r['image'])

    def _raw(self, need_pixels):
        i = self._next_buffer
        self._next_buffer = (i + 1) % len(self._buffers)
        buf = self._buffers[i]
        if buf is None or buf.pixels.numel() < need_pixels:
            buf = self._buffers[i] = RawBatch(self.batch_size, self.max_gt, int(need_pixels * 1.25) + 4096)
        return buf

    def _get_batch(self):
        cur_from, cur_to = self.cur_i, self.cur_i + self.batch_size
        entries = [self.roidb[self.inds[i]] for i in range(cur_from, cur_to)]
        cropids = [r['chip_order'][self.crop_idx[self.inds[i]] % len(r['chip_order'])]
                   for r, i in zip(entries, range(cur_from, cur_to))]
        for i in range(cur_from, cur_to):
            self.crop_idx[self.inds[i]] += 1
        # source rectangles (im_worker.worker: flip, then im[int(y1):int(y2), int(x1):int(x2)])
        rects = []
        for r, cid in zip(entries, cropids):
            crop = r['crops'][cid]
            im = self._image(r)
            H, W = im.shape[0], im.shape[1]
            x1, y1, x2, y2 = int(crop[0][0]), int(crop[0][1]), int(crop[0][2]), int(crop[0][3])
            y1c, y2c = min(max(y1, 0), H), min(max(y2, 0), H)
            x1c, x2c = min(max(x1, 0), W), min(max(x2, 0), W)
            if r.get('flipped', False):      # columns [x1, x2) of the flipped image = [W - x2, W - x1) of the stored one
                xa, xb = W - x2c, W - x1c
            else:
                xa, xb = x1c, x2c
            rects.append((im, y1c, y2c, xa, xb))
        need = sum(max(y2 - y1, 0) * max(xb - xa, 0) * 3 for _, y1, y2, xa, xb in rects)
        raw = self._raw(need)
        pix = raw.pixels.numpy()
        off = 0
        S0, S1 = self.crop_size
        focus = []
        for k, (r, cid, (im, y1, y2, xa, xb)) in enumerate(zip(entries, cropids, rects)):
            crop = r['crops'][cid]
            im_scale = crop[1]
            h, w = max(y2 - y1, 0), max(xb - xa, 0)
            n = h * w * 3
            if n:
                pix[off:off + n].reshape(h, w, 3)[...] = im[y1:y2, xa:xb, :3]
            dst_h, dst_w = int(np.rint(h * im_scale)), int(np.rint(w * im_scale))      # cv2.resize dsize = cvRound(...)
            raw.table[k] = torch.tensor([off, h, w, dst_h, dst_w, 1 if r.get('flipped', False) else 0,
                                         int(np.float64(im_scale).view(np.int64)), 0], dtype=torch.int64)
            off += n
            scalei, height, width = crop[4], crop[2], crop[3]
            vr = self.cfg.TRAIN.VALID_RANGES[scalei]
            raw.valid_ranges[k, 0] = 0 if vr[0] < 0 else vr[0] * im_scale
            raw.valid_ranges[k, 1] = S1 if vr[1] < 0 else vr[1] * im_scale
            raw.im_info[k] = torch.tensor([height, width, im_scale], dtype=torch.float32)
            # the anchor matcher sees the chip as a full crop_size x crop_size image (MNIteratorE2E.py:137)
            info = [S0, S1, im_scale]
            raw.anchor_im_info[k] = torch.tensor(info, dtype=torch.float32)
            gtids = np.where(r['max_overlaps'] == 1)[0]
            classes = r['max_classes'][gtids]
            valid, invalid, fgt = chip_ground_truth(info, crop[0], im_scale, r['props_in_chips'][cid], gtids,
                                                    r['boxes'][gtids, :], r['boxes'].copy(),
                                                    classes.reshape(len(classes), 1), self.max_gt)
            nv, ni = min(len(valid), self.max_gt), min(len(invalid), self.max_gt)
            raw.ngt[k], raw.ninv[k] = nv, ni
            if nv:
                raw.gt_valid[k, :nv] = torch.from_numpy(np.ascontiguousarray(valid[:nv], dtype=np.float32))
            if ni:
                raw.gt_invalid[k, :ni] = torch.from_numpy(np.ascontiguousarray(invalid[:ni], dtype=np.float32))
            raw.gt_boxes[k] = torch.from_numpy(fgt.astype(np.float32))
            if self.auto_focus:
                focus.append(chip_focus_boxes(info, crop[0], im_scale, r['boxes'][gtids, :]))
        if self.auto_focus:
            n = sum(len(f) for f in focus)
            if raw.focus_boxes is None or raw.focus_boxes.shape[0] < n:
                raw.focus_boxes = raw.pin(max(int(n * 1.25), 256), 4, dtype=torch.float32)
                raw.focus_off = raw.pin(len(focus) + 1, dtype=torch.int32)
            o = 0
            for k, f in enumerate(focus):
                raw.focus_off[k] = o
                if len(f):
                    raw.focus_boxes[o:o + len(f)] = torch.from_numpy(np.ascontiguousarray(f, dtype=np.float32))
                o += len(f)
            raw.focus_off[len(focus)] = o
        raw.used_pixels = off
        raw.seed = (self.epiter * 1000003 + self.cur_i) & 0x7FFFFFFF
        return raw


class PrefetchingIter(object):
    """Background-thread prefetch of raw batches (the role of mx.io.PrefetchingIter around MNIteratorE2E in
    main_train.py): the host bookkeeping of batch i+1 runs while the GPU computes batch i.  The wrapped iterator must
    own at least depth + 2 raw buffers (n_buffers)."""

    def __init__(self, it, depth=2, epochs=None):
        import queue
        import threading
        self.it = it
        self.q = queue.Queue(maxsize=depth)
        self.epochs = epochs
        self._stop = False
        # Every ctypes call of the training step releases the GIL and has to win it back from the producer thread; with
        # the default 5 ms switch interval each of those hand-overs can stall the step by up to 5 ms (measured: step_raw
        # 56 ms instead of 36 ms next to a busy producer).  0.5 ms keeps the hand-over cost small.
        import sys
        self._switch = sys.getswitchinterval()
        sys.setswitchinterval(5e-4)
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        ep = 0
        while not self._stop:
            for raw in self.it:
                if self._stop:
                    return
                self.q.put(raw)
            ep += 1
            if self.epochs is not None and ep >= self.epochs:
                self.q.put(None)
                return
            self.it.reset()

    def __iter__(self):
        return self

    def __next__(self):
        raw = self.q.get()
        if raw is None:
            raise StopIteration
        return raw

    def close(self):
        """Stops and JOINS the worker (a daemon thread still inside a ctypes call when the interpreter exits aborts the
        process): keep draining the queue so that a worker blocked in put() can see the stop flag."""
        import queue
        self._stop = True
        while self.th.is_alive():
            try:
                while True:
                    self.q.get_nowait()
            except queue.Empty:
                pass
            self.th.join(timeout=0.02)
        import sys
        sys.setswitchinterval(self._switch)


class InputStage(object):
    """Device half of the iterator: raw batch -> the network's input tensors (all on `device`)."""

    def __init__(self, cfg, device, batch_size, crop_size=512, max_gt=100):
        self.cfg = cfg
        self.device = torch.device(device)
        self.B, self.S, self.max_gt = batch_size, crop_size, max_gt
        net = cfg.network
        self.scales, self.ratios, self.stride = tuple(net.ANCHOR_SCALES), tuple(net.ANCHOR_RATIOS), net.RPN_FEAT_STRIDE
        self.rpn_batch = cfg.TRAIN.RPN_BATCH_SIZE
        self.num_fg = int(self.rpn_batch * cfg.TRAIN.RPN_FG_FRACTION)
        self.pos, self.neg = cfg.TRAIN.RPN_POSITIVE_OVERLAP, cfg.TRAIN.RPN_NEGATIVE_OVERLAP
        self.means = torch.tensor(list(net.PIXEL_MEANS), dtype=torch.float32, device=self.device)
        self.pixels = None
        z = lambda *s, dtype=torch.float32: torch.zeros(*s, dtype=dtype, device=self.device)
        B = batch_size
        self.dev = dict(table=z(B, 8, dtype=torch.int64), valid_ranges=z(B, 2), im_info=z(B, 3), gt_valid=z(B, max_gt, 4),
                        ngt=z(B, dtype=torch.int32), gt_invalid=z(B, max_gt, 4), ninv=z(B, dtype=torch.int32),
                        gt_boxes=z(B, max_gt, 5), anchor_im_info=z(B, 3))
        self.data = z(B, 3, crop_size, crop_size)
        # AutoFocus training (TRAIN.AUTO_FOCUS): FocusPixel labels from the raw batch's focus boxes
        self.auto_focus = bool(getattr(cfg.TRAIN, "AUTO_FOCUS", False))
        if self.auto_focus:
            T = cfg.TRAIN
            self.focus_thresh = dict(dc_low=T.AUTO_FOCUS_DC_LOW, small_thresh=T.AUTO_FOCUS_SMALL_THRESH,
                                     dc_high=T.AUTO_FOCUS_DC_HIGH)
            Hf = crop_size // self.stride
            self.focus_boxes = z(256, 4)
            self.focus_off = z(B + 1, dtype=torch.int32)
            self.scale_label = z(B, Hf * Hf)

    def run(self, raw, subsample=True):
        """H2D of the raw batch + the three kernels; returns the batch dict Trainer / SniperResNet101 consume.  Everything
        is enqueued on the current stream; the returned tensors are owned by this object and overwritten by the next
        call."""
        n = raw.used_pixels
        if self.pixels is None or self.pixels.numel() < n:
            self.pixels = torch.empty(int(n * 1.25) + 4096, dtype=torch.uint8, device=self.device)
        self.pixels[:n].copy_(raw.pixels[:n], non_blocking=True)
        for k in self.dev:
            self.dev[k].copy_(getattr(raw, k), non_blocking=True)
        st = torch.cuda.current_stream().cuda_stream
        check(lib().sniper_chip_input(self.pixels.data_ptr(), self.dev["table"].data_ptr(), self.means.data_ptr(),
                                      self.data.data_ptr(), self.B, self.S, st))
        Hf = self.S // self.stride
        label, bt, bw = ops.anchor_target(self.dev["gt_valid"], self.dev["ngt"], self.dev["gt_invalid"], self.dev["ninv"],
                                          self.dev["anchor_im_info"], H=Hf, W=Hf, feat_stride=self.stride,
                                          scales=self.scales, ratios=self.ratios, pos_thresh=self.pos,
                                          neg_thresh=self.neg)
        if subsample:
            A = len(self.scales) * len(self.ratios)
            check(lib().sniper_anchor_subsample(label.data_ptr(), bt.data_ptr(), bw.data_ptr(), self.B, A, Hf, Hf,
                                                self.num_fg, self.rpn_batch, int(raw.seed), st))
        out = dict(data=self.data, label=label, bbox_target=bt, bbox_weight=bw, gt_boxes=self.dev["gt_boxes"],
                   valid_ranges=self.dev["valid_ranges"], im_info=self.dev["im_info"])
        if self.auto_focus:
            if raw.focus_off is None:
                raise ValueError("InputStage(TRAIN.AUTO_FOCUS): the raw batch carries no focus boxes (build the iterator "
                                 "with the same config)")
            nb = int(raw.focus_off[-1])
            if self.focus_boxes.shape[0] < nb:
                self.focus_boxes = torch.zeros(int(nb * 1.25), 4, device=self.device)
            self.focus_boxes[:nb].copy_(raw.focus_boxes[:nb], non_blocking=True)
            self.focus_off.copy_(raw.focus_off, non_blocking=True)
            ops.focus_label(self.focus_boxes, self.focus_off, self.B, H=Hf, W=Hf, feat_stride=self.stride,
                            out=self.scale_label, **self.focus_thresh)
            out["scale_label"] = self.scale_label
        return out


def synthetic_roidb(n_images, seed=0, width=1333, height=800, n_gt=(1, 20), n_prop=300, num_classes=81):
    """COCO-shaped synthetic roidb with decoded images in memory (no dataset, no OpenCV in this image): random uint8
    pixels, GT boxes with sqrt(area) log-uniform in [8, 400] px (SURVEY 8d), a few hundred proposals, random flips."""
    rng = np.random.RandomState(seed)
    out = []
    for i in range(n_images):
        W, H = (width, height) if rng.rand() < 0.7 else (height, width)
        g = int(rng.randint(n_gt[0], n_gt[1] + 1))
        n = g + n_prop
        s = np.exp(rng.uniform(np.log(8), np.log(400), n))
        ar = np.exp(rng.uniform(np.log(0.5), np.log(2.0), n))
        w, h = s * np.sqrt(ar), s / np.sqrt(ar)
        cx, cy = rng.uniform(0, W, n), rng.uniform(0, H, n)
        boxes = np.stack([np.clip(cx - w / 2, 0, W - 1), np.clip(cy - h / 2, 0, H - 1),
                          np.clip(cx + w / 2, 0, W - 1), np.clip(cy + h / 2, 0, H - 1)], 1).astype(np.float32)
        out.append({'image_data': rng.randint(0, 256, (H, W, 3)).astype(np.uint8), 'width': W, 'height': H,
                    'boxes': boxes, 'flipped': bool(rng.rand() < 0.5),
                    'max_overlaps': np.concatenate([np.ones(g), rng.uniform(0, 0.9, n_prop)]).astype(np.float32),
                    'max_classes': np.concatenate([rng.randint(1, num_classes, g), np.zeros(n_prop)]).astype(np.int32)})
    return out


def default_config(neg=True):
    """The slice of configs/faster/sniper_res101_e2e.yml the iterator reads (:21-39, 76-101, 120-140)."""
    import types
    S = types.SimpleNamespace
    return S(network=S(PIXEL_MEANS=[103.06, 115.90, 123.15], ANCHOR_SCALES=[2, 4, 7, 10, 13, 16, 24],
                       ANCHOR_RATIOS=[0.5, 1, 2], RPN_FEAT_STRIDE=16, NUM_ANCHORS=21),
             TRAIN=S(SCALES=[(1400, 2000), (800, 1280), (-1, 512)], VALID_RANGES=[(-1, 80), (32, 150), (120, -1)],
                     CPP_CHIPS=True, USE_NEG_CHIPS=neg, RPN_BATCH_SIZE=256, RPN_FG_FRACTION=0.5,
                     RPN_POSITIVE_OVERLAP=0.5, RPN_NEGATIVE_OVERLAP=0.4, BATCH_IMAGES=16),
             # TEST block of configs/faster/sniper_res101_e2e_autofocus.yml:191-245 (AutoFocus inference, BASELINE config 5)
             TEST=S(SCALES=[(480, 512), (800, 1280), (1400, 2000)], BATCH_IMAGES=[8, 8, 2], MAX_PER_IMAGE=200,
                    VALID_RANGES=[(75, -1), (32, 180), (-1, 75)], AUTO_FOCUS=True, DO_PRUNING=[False, True, True],
                    CHIP_HYPERPARAMS=[(3, 0.02, 16), (3, 0.2, 20)], NMS=0.45, NMS_SIGMA=0.55),
             dataset=S(NUM_CLASSES=81))
