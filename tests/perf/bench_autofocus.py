"""Cost of AutoFocus training on one GPU, in one command:

  * the training step (forward + backward + update, CUDA graphs, B = 20 chips of 512 x 512) with Cfg.autofocus off and
    on, in the fp32 / TF32 and in the bf16 configuration; the two arms of a precision are built side by side and timed
    in alternating rounds (CUDA events around every step), so that drift of the shared machine hits both alike;
  * the two AutoFocus kernels from CUDA events over many launches: sniper_focus_head on conv_new_3_relu [20*32*32, 256]
    (operands rotated over buffers larger than the 126 MB L2, so every pass reads HBM) and sniper_focus_label on 20 chips
    of 150 boxes, each next to its HBM lower bound (bytes the kernel must move / 7.7 TB/s);
  * the card's name, power limit and maximum SM clock (nvidia-smi), read in the same run.

    python tests/perf/bench_autofocus.py --out profiles/autofocus_train_b200.json [--rounds 6 --steps 8 --warmup 3]

Needs a GPU; there is no CPU fallback."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12          # HGX B200 data sheet, one GPU


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(nvidia_smi=q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unavailable",
                torch_name=torch.cuda.get_device_name(0))


def batch(B, seed=3):
    from sniper_b200 import synth_batch
    b = synth_batch.make_batch(B, seed=seed, device="cpu", pinned=True)
    rng = np.random.RandomState(seed)
    b["scale_label"] = torch.from_numpy(rng.choice([-1.0, 0.0, 1.0], (B, 1024), p=[0.3, 0.5, 0.2]).astype(np.float32))
    b["scale_label"] = b["scale_label"].pin_memory()
    return b


def step_times(bf16, B, rounds, steps, warmup):
    from sniper_b200 import model, trainer
    arms = {}
    for af in (False, True):
        cfg = model.Cfg()
        cfg.batch_images, cfg.bf16, cfg.autofocus = B, bf16, af
        tr = trainer.Trainer(cfg, use_graph=True, seed=5, scheduler=None)
        hb = batch(B)
        if not af:
            hb = {k: v for k, v in hb.items() if k != "scale_label"}
        tr.load(hb)
        tr.capture()
        for _ in range(warmup):
            tr.step_device(lr=0.0)
        torch.cuda.synchronize()
        arms["on" if af else "off"] = tr
    per = {"off": [], "on": []}
    for r in range(rounds):
        order = ("off", "on") if r % 2 == 0 else ("on", "off")
        for k in order:
            tr = arms[k]
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
            for a, b in ev:
                a.record()
                tr.step_device(lr=0.0)
                b.record()
            torch.cuda.synchronize()
            per[k].append([a.elapsed_time(b) for a, b in ev])
    out = {}
    for k, rs in per.items():
        med = [float(np.median(x)) for x in rs]
        allv = [v for x in rs for v in x]
        out[k] = dict(median_ms=float(np.median(allv)), round_medians_ms=med, spread_ms=float(max(med) - min(med)),
                      min_ms=float(min(allv)), max_ms=float(max(allv)), steps=len(allv))
    out["delta_ms"] = out["on"]["median_ms"] - out["off"]["median_ms"]
    out["launches_per_step"] = {k: arms[k].launches_per_step for k in arms}
    del arms
    torch.cuda.empty_cache()
    return out


def kernel_times(B=20, iters=400):
    from sniper_b200 import ops
    M, C = B * 1024, 256
    torch.manual_seed(0)
    nbuf = 4                                 # 4 x (x3 + dx3) = 168 MB > 126 MB L2
    xs = [torch.relu(torch.randn(M, C, device="cuda")) for _ in range(nbuf)]
    dxs = [torch.empty_like(x) for x in xs]
    w = torch.randn(32, C, device="cuda") * 0.05
    bias = torch.zeros(32, device="cuda")
    lab = torch.randint(-1, 2, (M,), device="cuda").float()
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.count_valid(lab, cnt)
    prob = torch.empty(M, 2, device="cuda")
    dw, db, stats = torch.zeros(32, C, device="cuda"), torch.zeros(32, device="cuda"), torch.zeros(3, device="cuda")

    def head(i):
        ops.focus_head(xs[i % nbuf], w, bias, lab, 1.0, cnt, prob, dxs[i % nbuf], dw, db, stats)
    for i in range(20):
        head(i)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        head(i)
    b.record()
    torch.cuda.synchronize()
    t_head = a.elapsed_time(b) / iters * 1e-3
    bytes_head = 2 * M * C * 4 + M * 2 * 4 + M * 4            # x3 read, dx3 written, prob written, labels read
    rng = np.random.RandomState(1)
    nb = 150
    x1 = rng.randint(0, 480, (B * nb, 1))
    y1 = rng.randint(0, 480, (B * nb, 1))
    s = rng.randint(0, 120, (B * nb, 1))
    boxes = torch.from_numpy(np.clip(np.hstack([x1, y1, x1 + s, y1 + s]), 0, 511).astype(np.float32)).cuda()
    off = torch.arange(0, B * nb + 1, nb, dtype=torch.int32, device="cuda")
    out = torch.empty(B, 1024, device="cuda")
    for _ in range(20):
        ops.focus_label(boxes, off, B, out=out)
    torch.cuda.synchronize()
    a.record()
    for _ in range(iters):
        ops.focus_label(boxes, off, B, out=out)
    b.record()
    torch.cuda.synchronize()
    t_lab = a.elapsed_time(b) / iters * 1e-3
    bytes_lab = B * 1024 * 4 + B * nb * 16 + (B + 1) * 4
    return dict(focus_head=dict(rows=M, channels=C, time_us=t_head * 1e6, bytes=bytes_head,
                                hbm_bound_us=bytes_head / HBM_BYTES_PER_S * 1e6,
                                share_of_hbm_bound=bytes_head / HBM_BYTES_PER_S / t_head,
                                note="x3 / dx3 rotated over 4 buffer pairs (168 MB) so that passes read HBM"),
                focus_label=dict(chips=B, boxes_per_chip=nb, time_us=t_lab * 1e6, bytes=bytes_lab,
                                 hbm_bound_us=bytes_lab / HBM_BYTES_PER_S * 1e6,
                                 note="launch / latency bound: the data is ~0.1 MB"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=6)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_autofocus.py needs a GPU"
    res = dict(card=card(), batch=a.batch, rounds=a.rounds, steps_per_round=a.steps)
    res["kernels"] = kernel_times(a.batch)
    for name, bf16 in (("tf32", False), ("bf16", True)):
        res["step_" + name] = step_times(bf16, a.batch, a.rounds, a.steps, a.warmup)
        print(name, json.dumps(res["step_" + name]), flush=True)
    print(json.dumps(res))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
