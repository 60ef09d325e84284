"""TEST INFRASTRUCTURE (oracle/): executes the reference's own symbol file symbols/faster/resnet_mx_101_e2e.py, unchanged,
under its own configs/faster/sniper_res101_e2e_autofocus.yml (TRAIN.AUTO_FOCUS, fp16) with BATCH_IMAGES = 20 against
sniper_b200.mxnet_compat, and writes what the AutoFocus TRAINING graph looks like (argument / auxiliary / output names and
shapes, operator census, MD5 of the `-symbol.json` text) to tests/golden/ref_symbols_autofocus.json, with the helpers of
oracle/run_ref_symbols.py.  The committed fixture lets a machine without the reference tree check
`sniper_b200.symbols.NetSymbol(autofocus=True)`.

    python oracle/run_ref_symbols_autofocus.py            # needs the reference tree (SNIPER_REFERENCE)
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import run_ref_symbols as RS  # noqa: E402


def build():
    from sniper_b200 import mxnet_compat as MC
    res = MC.load_symbol_file(os.path.join(RS.REF, "symbols/faster/resnet_mx_101_e2e.py"))
    cfg = RS.load_config("sniper_res101_e2e_autofocus.yml")
    cfg.TRAIN.BATCH_IMAGES = 20
    with MC.NameManager():
        sym = res.resnet_mx_101_e2e(n_proposals=400, momentum=0.995).get_symbol_rcnn(cfg)
    d = RS.train_shapes(cfg, 20, 16)
    d["scale_label"] = (20, (512 // 16) ** 2)
    out = RS.describe(sym, d)
    out["cfg"] = dict(fp16=bool(cfg.TRAIN.fp16), batch_images=20, num_anchors=int(cfg.network.NUM_ANCHORS),
                      num_classes=int(cfg.dataset.NUM_CLASSES), auto_focus=True)
    return {"resnet101_train_autofocus": out}


if __name__ == "__main__":
    res = build()
    path = os.path.join(ROOT, "tests", "golden", "ref_symbols_autofocus.json")
    with open(path, "w") as f:
        json.dump(res, f, sort_keys=True, separators=(",", ":"))
    for k, v in res.items():
        print(k, len(v["arguments"]), "args", len(v["auxiliary"]), "aux", v["outputs"], v["ops"])
