"""WarmupMultiBatchScheduler (sniper_b200/lr_scheduler.py) against the reference class itself
(lib/train_utils/lr_scheduler.py:10-66), executed here with `mxnet.lr_scheduler.LRScheduler` stubbed by the three lines
of its constructor (python/mxnet/lr_scheduler.py: `self.base_lr = base_lr`), and against committed golden values."""
import json
import os
import sys
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sniper_b200 import lr_scheduler  # noqa: E402

REF = "/root/reference/lib/train_utils/lr_scheduler.py"
GOLD = os.path.join(ROOT, "tests", "golden", "lr_schedule.json")
CASES = [
    dict(step=[3000, 4000], factor=0.1, warmup=True, warmup_lr=0.0005, warmup_step=1000, base_lr=0.015),
    dict(step=[50], factor=0.5, warmup=False, warmup_lr=0.0, warmup_step=0, base_lr=0.01),
    dict(step=[10, 20, 30], factor=0.1, warmup=True, warmup_lr=5e-6, warmup_step=15, base_lr=1.5e-4),
]
QUERY = list(range(1, 60)) + [999, 1000, 1001, 2999, 3000, 3001, 3002, 4000, 4001, 5000]


def _ref_class():
    class LRScheduler(object):
        def __init__(self, base_lr=0.01):
            self.base_lr = base_lr
    mx = types.ModuleType("mxnet")
    mls = types.ModuleType("mxnet.lr_scheduler")
    mls.LRScheduler = LRScheduler
    mx.lr_scheduler = mls
    saved = {k: sys.modules.get(k) for k in ("mxnet", "mxnet.lr_scheduler")}
    sys.modules["mxnet"], sys.modules["mxnet.lr_scheduler"] = mx, mls
    try:
        ns = {}
        exec(compile(open(REF).read(), REF, "exec"), ns)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
    return ns["WarmupMultiBatchScheduler"]


def _run(cls, case):
    kw = dict(case)
    base = kw.pop("base_lr")
    s = cls(kw.pop("step"), **kw)
    s.base_lr = base
    return [s(n) for n in QUERY]


def test_matches_committed_golden():
    gold = json.load(open(GOLD))
    for case, want in zip(CASES, gold):
        got = _run(lr_scheduler.WarmupMultiBatchScheduler, case)
        assert got == want


def test_matches_reference_class_executed_here():
    """Where the reference tree is not present, against the reference class's values stored in the golden file."""
    if os.path.exists(REF):
        want = [_run(_ref_class(), case) for case in CASES]
    else:
        want = json.load(open(GOLD))
    for case, w in zip(CASES, want):
        assert _run(lr_scheduler.WarmupMultiBatchScheduler, case) == w


def test_from_config_is_the_yml_schedule():
    s = lr_scheduler.from_config()                      # sniper_res101_e2e.yml:104-111
    assert s(1) == 0.0005 + 1 * (0.015 - 0.0005) / 1000
    assert s(999) < 0.015 and s(1000) == 0.015
    s2 = lr_scheduler.from_config(roidb_len=1000, batch_size=10)       # 5.33 epochs -> 533 updates (inside warm-up)
    assert s2.step == [533]
    s3 = lr_scheduler.from_config(fp16=True)
    assert abs(s3.base_lr - 0.00015) < 1e-12 and abs(s3.warmup_lr - 5e-6) < 1e-15


if __name__ == "__main__":      # regenerates the golden from the REFERENCE class
    json.dump([_run(_ref_class(), c) for c in CASES], open(GOLD, "w"))
