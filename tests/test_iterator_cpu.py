"""Host half of the training iterator (sniper_b200/iterator.py): the GT bookkeeping in front of the anchor matching
against the reference's OWN anchor_worker.worker executed here (oracle/run_ref_anchor_worker.py), and the epoch /
batch index logic of MNIteratorE2E (lib/iterators/MNIteratorE2E.py:41-219)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ref_golden as G  # noqa: E402
from sniper_b200 import iterator as IT  # noqa: E402

HAVE_REF = os.path.isdir("/root/reference/lib") and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_chips.so"))


def _chip_case(seed):
    """One synthetic chip: image-space boxes (GT first), a crop window, a scale, the chip's own box ids."""
    rng = np.random.RandomState(seed)
    n_gt, n_prop = int(rng.randint(2, 16)), 40
    scale = float(rng.choice([3.0, 1.667, 0.75]))
    side = 512.0 / scale
    cx0, cy0 = rng.uniform(0, 900 - side), rng.uniform(0, 600 - side)
    crop = np.array([cx0, cy0, cx0 + side, cy0 + side])
    w = rng.uniform(4, side * 0.8, n_gt + n_prop)
    h = rng.uniform(4, side * 0.8, n_gt + n_prop)
    x1 = rng.uniform(cx0 - 30, cx0 + side - 5, n_gt + n_prop)
    y1 = rng.uniform(cy0 - 30, cy0 + side - 5, n_gt + n_prop)
    boxes = np.stack([x1, y1, x1 + w, y1 + h], 1).astype(np.float32)
    gtids = np.arange(n_gt)
    nids = np.sort(rng.choice(n_gt + n_prop, 12, replace=False)).astype(np.int32)
    classes = rng.randint(1, 81, (n_gt, 1)).astype(np.float64)
    return boxes, gtids, nids, classes, crop, scale


@pytest.mark.parametrize("seed", range(8))
def test_chip_ground_truth_matches_reference_anchor_worker(seed):
    """gt_boxes [100,5] bit for bit; the valid / invalid split through its only observable effect, the labels: with the
    reference's subsampling disabled (RPN_BATCH_SIZE = all anchors) the label map of the reference worker equals the
    oracle's anchor matching run on OUR (valid, invalid) sets."""
    import anchor_target_np as AT
    boxes, gtids, nids, classes, crop, scale = _chip_case(seed)
    im_info = [512, 512, scale]

    def run():
        import run_ref_anchor_worker as RA
        cfg = RA.make_cfg()
        cfg.TRAIN.RPN_BATCH_SIZE = 10 ** 6          # no npr.choice subsampling: deterministic labels
        cfg.TRAIN.RPN_FG_FRACTION = 1.0
        W = RA.load_reference_worker()(cfg, 512)
        out = W.worker([im_info, crop.copy(), scale, nids.copy(), gtids.copy(), boxes[gtids].copy(), boxes.copy(),
                        classes.copy()])
        return np.asarray(out[0], np.float32).ravel(), np.asarray(out[3], np.float64)
    # where the reference is not present: its outputs stored by tests/ref_golden.py
    ref_label, ref_fgt = G.reference("iterator_cpu.anchor_worker", (boxes, gtids, nids, classes, crop, scale),
                                     run if HAVE_REF else None)
    valid, invalid, fgt = IT.chip_ground_truth(im_info, crop.copy(), scale, nids.copy(), gtids.copy(), boxes[gtids].copy(),
                                               boxes.copy(), classes.copy())
    assert fgt.tobytes() == ref_fgt.tobytes()
    res = AT.anchor_target(valid, invalid, im_info)
    lab, _, _ = AT.pack(res["labels"], res["targets"], 32, 32, res["A"])
    assert np.array_equal(lab, ref_label)
    assert (ref_label == 1).sum() > 0 or len(valid) == 0


def test_epoch_and_batch_bookkeeping():
    """Every chip of the epoch is visited, negative chips are capped at 2 per image, the chip list is padded to whole
    batches, and each raw batch carries consistent tables."""
    cfg = IT.default_config()
    np.random.seed(3)
    roidb = IT.synthetic_roidb(6, seed=1, n_prop=400)
    it = IT.MNIteratorE2E(roidb, cfg, batch_size=4)
    assert it.size % 4 == 0 and it.size >= it.chip_count
    for r in roidb:
        n_neg = len(r['crops']) - len([c for c in r['crops'] if not any(c is n for n in r.get('neg_crops', []))])
        assert n_neg <= 2
        assert sorted(r['chip_order'].tolist()) == list(range(len(r['crops'])))
        assert len(r['props_in_chips']) == len(r['crops'])
    seen = 0
    for raw in it:
        seen += 4
        t = raw.table.numpy()
        assert (t[:, 1] >= 0).all() and (t[:, 2] >= 0).all()
        assert raw.used_pixels == int((t[:, 1] * t[:, 2] * 3).sum())
        assert np.array_equal(t[:, 0], np.concatenate([[0], np.cumsum(t[:-1, 1] * t[:-1, 2] * 3)]))
        sc = t[:, 6].view(np.float64) if False else np.array([np.int64(v).view(np.float64) for v in t[:, 6]])
        assert np.array_equal(t[:, 3], np.rint(t[:, 1] * sc).astype(np.int64))
        info = raw.im_info.numpy()
        assert np.allclose(info[:, 2], sc.astype(np.float32))
        vr = raw.valid_ranges.numpy()
        assert (vr[:, 0] >= 0).all() and (vr[:, 1] > vr[:, 0]).all() and (vr[:, 1] <= 512 + 1e-3).all()
        ng = raw.ngt.numpy()
        gb = raw.gt_boxes.numpy()
        assert ((gb[:, :, 4] > 0).sum(1) >= ng).all()          # valid GT are a subset of the chip's gt_boxes rows
    assert seen == it.size
    assert it.get_batch() is False
    it.reset()
    assert it.epiter == 2 and it.cur_i == 0
