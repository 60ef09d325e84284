"""sniper_b200.chip_worker (positive chips per scale, box -> chip assignment, negative-chip mining) against the
reference's OWN chip_worker class executed here (oracle/run_ref_chip_worker.py: data_workers.py:373-594 with the
reference's chip_generator, Cython overlaps and cchips.cpp), same roidb entry, same chip stride, same C rand() seed.
Everything is graded exact: chip coordinates (float64 bits), scale, tagged sizes, scale index, the box ids of every
chip in order, the negative chips and their box ids.  Golden copy: tests/golden/chip_worker_ref.npz."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import run_ref_chip_worker as RR  # noqa: E402
from sniper_b200 import chip_worker as CW  # noqa: E402

HAVE_REF = os.path.isdir("/root/reference/lib") and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libref_chips.so"))
GOLD = os.path.join(ROOT, "tests", "golden", "chip_worker_ref.npz")
CASES = [
    dict(seed=0, cfg={}, roidb=dict()),                                                       # yml scales, 1333x800
    dict(seed=3, cfg={}, roidb=dict(width=640, height=480, n_gt=7, n_prop=600)),
    dict(seed=5, cfg=dict(scales=(3.0, 1.667, 512.0)), roidb=dict(width=500, height=375, n_gt=12, n_prop=900)),  # main_train.py:55
    dict(seed=7, cfg=dict(neg=False), roidb=dict(width=1024, height=1024, n_gt=30, n_prop=0)),
    dict(seed=9, cfg={}, roidb=dict(width=2000, height=300, n_gt=3, n_prop=1500)),
    dict(seed=11, cfg=dict(scales=((512, 512),), valid_ranges=((-1, -1),)), roidb=dict(width=800, height=600, n_gt=10, n_prop=400)),
]


def _flatten(crops, out):
    """(crops, box_assigner output) -> dict of arrays (comparable / storable)."""
    d = {}

    def chips(prefix, lst):
        d[prefix + "_xyxy"] = np.array([c[0] for c in lst], np.float64).reshape(-1, 4)
        d[prefix + "_scale"] = np.array([c[1] for c in lst], np.float64)
        d[prefix + "_hwi"] = np.array([[c[2], c[3], c[4]] for c in lst], np.int64).reshape(-1, 3)

    def lists(prefix, ll):
        d[prefix + "_len"] = np.array([len(x) for x in ll], np.int64)
        d[prefix + "_ids"] = np.concatenate([np.asarray(x, np.int64) for x in ll]) if len(ll) else np.zeros(0, np.int64)
    chips("pos", crops)
    lists("props", out[0])
    if len(out) == 3:
        chips("neg", out[1])
        lists("negprops", out[2])
    return d


def _same(a, b):
    assert a.keys() == b.keys()
    for k in a:
        assert a[k].shape == b[k].shape, (k, a[k].shape, b[k].shape)
        assert a[k].tobytes() == b[k].tobytes(), k


def _ours(case):
    cfg = RR.make_cfg(**case["cfg"])
    return _flatten(*RR.run(CW.chip_worker, cfg, RR.synth_roidb(case["seed"], **case["roidb"]), seed=1 + case["seed"]))


@pytest.mark.parametrize("ci", range(len(CASES)))
def test_matches_reference_class_executed_here(ci):
    """Where the reference tree is not present, against the reference's outputs stored in the golden copy."""
    case = CASES[ci]
    if HAVE_REF:
        W = RR.load_reference_chip_worker()
        cfg = RR.make_cfg(**case["cfg"])
        ref = _flatten(*RR.run(W, cfg, RR.synth_roidb(case["seed"], **case["roidb"]), seed=1 + case["seed"]))
    else:
        gold = np.load(GOLD)
        pre = "c%d_" % ci
        ref = {k[len(pre):]: gold[k] for k in gold.files if k.startswith(pre)}
    ours = _ours(case)
    _same(ours, ref)
    assert ref["pos_xyxy"].shape[0] > 0


def test_matches_committed_golden():
    gold = np.load(GOLD)
    for ci, case in enumerate(CASES):
        ours = _ours(case)
        for k, v in ours.items():
            g = gold["c%d_%s" % (ci, k)]
            assert g.shape == v.shape and g.tobytes() == v.tobytes(), (ci, k)


def test_negative_chips_need_a_crowd():
    """> 25 uncovered boxes (or > 10 off the finest scale) per negative chip (data_workers.py:577-578)."""
    o = _ours(CASES[0])
    lens, scale_idx = o["negprops_len"], o["neg_hwi"][:, 2]
    assert len(lens) > 0 and ((lens > 25) | ((lens > 10) & (scale_idx != 0))).all()


if __name__ == "__main__":      # regenerates the golden from the REFERENCE class
    W = RR.load_reference_chip_worker()
    store = {}
    for ci, case in enumerate(CASES):
        cfg = RR.make_cfg(**case["cfg"])
        ref = _flatten(*RR.run(W, cfg, RR.synth_roidb(case["seed"], **case["roidb"]), seed=1 + case["seed"]))
        for k, v in ref.items():
            store["c%d_%s" % (ci, k)] = v
    np.savez_compressed(GOLD, **store)
    print("wrote", GOLD, os.path.getsize(GOLD), "bytes")
