#!/usr/bin/env python
"""bench.py -- SNIPER 512x512-chip training throughput (chips/sec) on N B200s of one node.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torch.distributed.run)
  python bench.py --impl reference ...                      (CPU reference arm, rank 0 only)

Workload (BASELINE.json configs[1]): ResNet-101 SNIPER Faster-R-CNN/R-FCN, 512x512 chips, 20 chips per
GPU, fp32 storage with TF32 tensor-core math, synthetic COCO-shaped chips + boxes, random-init weights.
A step = forward + backward + (N>1: one NCCL gradient all-reduce) + fused SGD-momentum update.
`value` : chips/sec with the batch already resident in HBM (CUDA-graph replay of the step); every timed step starts
          from the same model state, restored between steps outside the timed window.
`e2e`   : chips/sec through Trainer.step(): pinned host batch -> H2D -> step -> D2H of the loss scalars.
The data batches rotate through a pool larger than L2 (7 x 63 MB of input + >10 GB of activations per step),
so no timed iteration finds its inputs in L2.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FWD_GFLOP_PER_CHIP = 145.54      # BASELINE.md section 2 / SURVEY.md 8d
TRAIN_GFLOP_PER_CHIP = 420.2
CHIPS_PER_GPU = 20


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.stop_flag = False
        self.max_mhz = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:6]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        s = sorted(self.samples)
        med = s[len(s) // 2] if s else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def ncu_traffic():
    """DRAM bytes per tcgen05 launch from the committed ncu capture (profiles/gemm_dram_r01.json); None if absent."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "gemm_dram_r01.json")))
        return d["dram_read_bytes_per_launch"] + d["dram_write_bytes_per_launch"]
    except Exception:
        return None


def gpu_head_start(ms=150.0):
    """Keeps the GPU busy for ~ms milliseconds (a spin kernel on the current stream) so that the host can enqueue a whole
    eager step behind it: the launches then run back to back and a CUDA-event pair around one launch measures that
    kernel only.  Without it the per-launch events also count the host's launch latency wherever the GPU has caught up
    with the host (after the BatchNorm kernels got faster the eager pass became host-bound in places and the summed
    tcgen05 time read 80 ms instead of 25 ms)."""
    import torch
    torch.cuda._sleep(int(ms * 1e-3 * 1.9e9))


def entry_point_breakdown(trainer, path):
    """CUDA-event time per C-ABI entry point over one eager, single-stream training step -> markdown table at `path`
    (a cheap complement to the ncu launch list: SNIPER_BREAKDOWN=<file>)."""
    import torch
    from sniper_b200 import _lib
    L = _lib.lib()
    names = [n for n in _lib.SIGNATURES if _lib.KERNELS_PER_CALL.get(n, 1) > 0]
    rec, orig = [], {}

    def wrap(name, raw):
        def fn(*a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = raw(*a)
            e1.record()
            rec.append((name, e0, e1))
            return r
        return fn
    for n in names:
        orig[n] = getattr(L, n)
        L._cache[n] = wrap(n, orig[n])
    ws = trainer.net.cfg.wsched
    ws_enabled, ws.enabled = ws.enabled, False
    try:
        gpu_head_start()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        trainer.net.forward_backward(trainer.static)
        trainer.net.update()
        t1.record()
        torch.cuda.synchronize()
    finally:
        ws.enabled = ws_enabled
        for n in names:
            L._cache[n] = orig[n]
    agg = {}
    for n, a, b in rec:
        c = agg.setdefault(n, [0, 0.0])
        c[0] += 1
        c[1] += a.elapsed_time(b)
    tot = sum(v[1] for v in agg.values())
    with open(path, "w") as f:
        f.write("| entry point | calls | total ms | share |\n|---|---:|---:|---:|\n")
        for n, (c, ms) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
            f.write("| `%s` | %d | %.3f | %.1f%% |\n" % (n, c, ms, 100 * ms / tot))
        f.write("\nsum of entry points %.2f ms; eager single-stream step (incl. launch gaps) %.2f ms\n" % (tot, t0.elapsed_time(t1)))


def tc_kernel_time(trainer, peak_bf16):
    """CUDA-event time and algorithmic FLOPs of every tcgen05 launch of one (eager, single-stream) training step.
    Returns (ms, flops, launches, ideal_ms): ideal_ms = sum over launches of flops / peak of the launch's operand type
    (bf16: the measured cuBLAS bf16 figure; fp32 operands = kind::tf32, half that issue rate)."""
    import torch
    from sniper_b200 import _lib
    L = _lib.lib()
    names = ["sniper_gemm_nt", "sniper_conv2d_nhwc", "sniper_conv2d_wgrad_nhwc"]
    events, flops, descs = [], [0.0], []
    orig = {}

    def wrap(name, raw):
        def fn(*a):
            if name == "sniper_gemm_nt":
                M, N, K, dt = a[6], a[7], a[8], a[9]
                fl = 2.0 * M * N * K
                descs.append(["gemm", M, N, K, fl, dt])
            elif name == "sniper_conv2d_nhwc":
                NB, Cin, Cout, ntaps, Ho, Wo, dt = a[2], a[5], a[7], a[8], a[12], a[13], a[21]
                fl = 2.0 * NB * Ho * Wo * Cout * ntaps * Cin
                descs.append(["conv", NB * Ho * Wo, Cout, ntaps * Cin, fl, dt])
            else:
                NB, Cin, Cout, ntaps, Ho, Wo, dt = a[4], a[7], a[8], a[9], a[13], a[14], a[16]
                fl = 2.0 * NB * Ho * Wo * Cout * ntaps * Cin
                descs.append(["wgrad", Cout, ntaps * Cin, NB * Ho * Wo, fl, dt])
            flops[0] += fl
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = raw(*a)
            e1.record()
            events.append((e0, e1))
            return r
        return fn
    for n in names:
        orig[n] = getattr(L, n)
        L._cache[n] = wrap(n, orig[n])
    ws = trainer.net.cfg.wsched
    ws_enabled, ws.enabled = ws.enabled, False     # single stream: per-launch events must not overlap other kernels
    try:
        gpu_head_start()
        trainer.net.forward_backward(trainer.static)
        torch.cuda.synchronize()
    finally:
        ws.enabled = ws_enabled
        for n in names:
            L._cache[n] = orig[n]
    times = [a.elapsed_time(b) for a, b in events]
    ms = sum(times)
    ideal_ms = sum(d[4] / ((peak_bf16 if d[5] == 1 else peak_bf16 / 2.0) * 1e12) * 1e3 for d in descs)
    dump = os.environ.get("SNIPER_DUMP_GEMM")
    if dump:
        if getattr(trainer.net.cfg, "bf16", False):
            dump = dump.replace(".md", "") + "_bf16.md"
        agg = {}
        for d, t in zip(descs, times):
            k = (d[0], d[1], d[2], d[3], "bf16" if d[5] == 1 else "tf32")
            e = agg.setdefault(k, [0, 0.0, 0.0])
            e[0] += 1; e[1] += t; e[2] += d[4]
        rows = sorted(agg.items(), key=lambda kv: -kv[1][1])
        with open(dump, "w") as f:
            f.write("| kind | M | N | K | operands | launches | total ms | TFLOP/s |\n|---|---:|---:|---:|---|---:|---:|---:|\n")
            for (kind, M, N, K, dt), (n, t, fl) in rows:
                f.write("| %s | %d | %d | %d | %s | %d | %.3f | %.1f |\n" % (kind, M, N, K, dt, n, t, fl / (t / 1e3) / 1e12))
            f.write("\ntotal %.3f ms, %.1f GFLOP\n" % (ms, flops[0] / 1e9))
    return ms, flops[0], len(events), ideal_ms


DUMP_BYTES = 64 << 20
DUMP_MAX_ELEMS = 1 << 20


def dump_outputs(out_dir, arrays):
    """Writes each tensor of `arrays` as out_dir/<name>.npy, floating types as float32 and integer types as float64.
    A tensor of more than DUMP_MAX_ELEMS elements (or one that would take the dump past DUMP_BYTES) is written as a
    fixed sample of its flattened elements (seeded, sorted indices), the same for every run with the same arguments, so
    that two builds can be compared output for output."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    left = DUMP_BYTES
    for name in sorted(arrays):
        t = arrays[name].detach()
        dt = torch.float32 if t.is_floating_point() else torch.float64
        n = min(t.numel(), DUMP_MAX_ELEMS, left // (4 if dt == torch.float32 else 8))
        if n < t.numel():
            idx = np.unique(np.random.RandomState(0).randint(0, t.numel(), n))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.to(dt).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes


def measure(args, cfg, rank, local_rank, world, pool, dev_pool, sampler=None, dump_dir=None):
    """Device-resident and end-to-end timing of one configuration; returns a dict (identical on every rank).
    Every warm-up and timed device step starts from the model state the trainer was created with (weights, momentum,
    BN moving statistics, restored between steps outside the timed window): the step's backward kernels accumulate
    with float atomics, so a state carried from step to step drifts apart between runs in its last bits, and the
    proposal selection of later steps turns that into different rois.  With the state restored, a step's inputs are the
    same in every run with the same arguments.
    `dump_dir`: rank 0 writes there what the last timed device step produced (its outputs and the updated weights)."""
    import torch
    import torch.distributed as dist
    from sniper_b200.trainer import Trainer
    trainer = Trainer(cfg, device="cuda:%d" % local_rank, world_size=world, use_graph=not args.no_graph)
    trainer.load(pool[0])
    trainer.capture()
    P = trainer.net.P
    snap = trainer._snapshot()
    w16 = None if P.w16 is None else P.w16.clone()

    def restore():
        trainer._restore(snap)
        if w16 is not None:
            P.w16.copy_(w16)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def dev_step(i):
        b = dev_pool[i % len(dev_pool)]
        for k, v in b.items():
            trainer.static[k].copy_(v, non_blocking=True)      # D2D rotate: inputs stay HBM-resident, never L2-hot
        trainer.step_device()

    for i in range(max(args.warmup, 3)):
        restore()
        dev_step(i)
    if sampler is not None and rank == 0:
        sampler.start()
    barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    for i in range(args.steps):
        restore()
        ev[i][0].record()
        dev_step(i)
        ev[i][1].record()
    barrier()
    ms = sum(a.elapsed_time(b) for a, b in ev)
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, dict(trainer.out, weights=trainer.net.P.w))
    # ---- end to end through the public API (host batch in, host losses out)
    for i in range(2):
        trainer.step(pool[i % len(pool)], prefetch=pool[(i + 1) % len(pool)])
    barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    losses = None
    for i in range(args.steps):
        # every step: H2D of the next step's inputs (copy stream, overlapped), D2D into the graph's static buffers,
        # forward+backward, all-reduce, update, D2H of the losses + stream sync
        losses = trainer.step(pool[(i + 2) % len(pool)], prefetch=pool[(i + 3) % len(pool)])
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)
    if sampler is not None and rank == 0:
        sampler.stop_flag = True
    t = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    out = {"ms": ms, "ms_e2e": ms_e2e, "losses": losses, "launches_per_step": trainer.launches_per_step}
    if getattr(args, "iterator_leg", False):
        out["iterator"] = iterator_leg(args, trainer, local_rank, barrier)
    if rank == 0:
        peaks, peak_src = load_peaks()
        peak_bf16 = peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"])
        if os.environ.get("SNIPER_BREAKDOWN"):
            path = os.environ["SNIPER_BREAKDOWN"]
            entry_point_breakdown(trainer, path.replace(".md", "") + "_bf16.md" if cfg.bf16 else path)
        tc_ms, tc_flops, tc_n, ideal_ms = tc_kernel_time(trainer, peak_bf16)
        out.update(tc_ms=tc_ms, tc_flops=tc_flops, tc_n=tc_n, ideal_ms=ideal_ms, peak_bf16=peak_bf16, peak_src=peak_src)
    del trainer
    torch.cuda.empty_cache()
    return out


def iterator_leg(args, trainer, local_rank, barrier):
    """The same step fed by the REAL input path: synthetic COCO-shaped roidb (decoded uint8 images in memory) ->
    chip_worker / MNIteratorE2E on the host (background prefetch thread) -> raw uint8 batch over PCIe -> GPU input stage
    (resize, mean, anchor matching, label subsampling) -> training step -> losses back.  Reported next to `e2e`."""
    import numpy as np
    import torch
    from sniper_b200 import iterator as IT
    np.random.seed(1234 + local_rank)
    cfg = IT.default_config()
    roidb = IT.synthetic_roidb(24, seed=11 + local_rank, n_prop=300)
    it = IT.MNIteratorE2E(roidb, cfg, batch_size=args.chips, n_buffers=6)
    stage = IT.InputStage(cfg, "cuda:%d" % local_rank, args.chips)
    pf = IT.PrefetchingIter(it, depth=3)
    nbytes = []
    for _ in range(8):        # more than n_buffers: every pinned staging buffer is allocated (cudaHostAlloc) before the clock starts
        trainer.step_raw(next(pf), stage)
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    losses = None
    for _ in range(args.steps):
        raw = next(pf)
        nbytes.append(raw.nbytes())
        losses = trainer.step_raw(raw, stage)
    t1.record()
    barrier()
    pf.close()
    ms = t0.elapsed_time(t1)
    return {"ms": ms, "h2d_bytes_per_step": int(sum(nbytes) / max(len(nbytes), 1)), "losses": losses,
            "chips_in_epoch": int(it.chip_count)}


def run_config5(args):
    """BASELINE config 5 (SURVEY 8d): AutoFocus inference over TEST.SCALES (480,512) -> (800,1280) -> (1400,2000) with
    DO_PRUNING [F,T,T] on synthetic 1333x800 images, random-init weights (so the FocusPixel maps and detections are
    noise: the numbers measure the machinery, not accuracy).  One JSON line: imgs/s over the whole pyramid (second pass,
    after a warm-up pass), per-scale seconds, device soft-NMS latency and the host `cpu_soft_nms` time on the same
    problems for comparison."""
    import numpy as np
    import torch
    from sniper_b200 import inference, iterator as IT, model, synth_batch, tester as TS
    n = int(args.config5)
    cfg = IT.default_config()
    rng = np.random.RandomState(5)
    roidb = [dict(width=W, height=H, image_data=rng.randint(0, 256, (H, W, 3)).astype(np.uint8))
             for (W, H) in [((1333, 800) if rng.rand() < 0.7 else (800, 1333)) for _ in range(n)]]
    mc = model.Cfg()
    mc.batch_images = 2
    net = model.SniperResNet101(mc, deform_offset_std=0.01)
    net.train_step(synth_batch.make_batch(2, seed=7, device="cuda"), lr=0.001)
    net.enable_autofocus(seed=3)
    TS.imdb_detection_wrapper(net, cfg, roidb)          # warm-up pass over the same images (allocator, lazy kernel loading)
    torch.cuda.synchronize()
    t0 = time.time()
    boxes, stats = TS.imdb_detection_wrapper(net, cfg, roidb, nms_backend="device")
    torch.cuda.synchronize()
    total = time.time() - t0
    t1 = time.time()
    TS.imdb_detection_wrapper(net, cfg, roidb, nms_backend="host")
    host_total = time.time() - t1
    ndet = int(sum(len(boxes[j][i]) for j in range(1, 81) for i in range(n)))
    print(json.dumps({"metric": "AutoFocus inference images/sec (ResNet-101, 3 scales)", "value": round(n / total, 3),
                      "unit": "images/s", "n_gpus": 1, "images": n, "seconds": round(total, 3),
                      "config": {"workload": "BASELINE.json configs[4]: AutoFocus inference pyramid, synthetic 1333x800 images, "
                                             "random-init weights", "scales": [list(s) for s in cfg.TEST.SCALES],
                                 "batch_images": list(cfg.TEST.BATCH_IMAGES)},
                      "per_scale": [{k: (round(v, 4) if isinstance(v, float) else v) for k, v in st.items()}
                                    for st in stats["scales"]],
                      "soft_nms_device_s": round(stats["nms_s"], 4),
                      "same_pyramid_with_host_soft_nms_s": round(host_total, 3), "detections": ndet,
                      "data": "synthetic"}))


def hbm_kernel_table(B, lowp, peak_gbs):
    """The depthwise / BatchNorm-backward kernels of the MobileNetV2 step alone, at the step's largest shapes: CUDA-event
    time per launch (after warm-up, inputs >> L2) and ALGORITHMIC bytes (each operand once) / time against the measured
    HBM copy bandwidth.  These are the HBM-bound launches of config 4 (depthwise.cu, elementwise.cu)."""
    import torch
    from sniper_b200 import ops
    dt = torch.bfloat16 if lowp else torch.float32
    es = 2 if lowp else 4
    rows = []

    def timed(name, fn, nbytes, reps=5):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / reps
        gbs = nbytes / us / 1e3
        rows.append({"kernel": name, "us": round(us, 1), "algorithmic_mb": round(nbytes / 1e6, 1), "gbs": round(gbs, 1),
                     "frac_of_hbm_peak": round(gbs / peak_gbs, 3)})

    for (H, C, s) in ((256, 64, 1), (256, 128, 2), (128, 192, 1), (32, 384, 1)):
        x = torch.randn(B, H, H, C, device="cuda").to(dt)
        w = torch.randn(9, C, device="cuda")
        Ho = (H - 1) // s + 1
        dy = torch.randn(B, Ho, Ho, C, device="cuda").to(dt)
        y = torch.empty_like(dy)
        dx = torch.empty_like(x)
        dw = torch.zeros(9, C, device="cuda")
        nin, nout = x.numel() * es, dy.numel() * es
        tag = "%dx%dx%d s%d" % (H, H, C, s)
        timed("dw_fwd " + tag, lambda: ops.depthwise3x3(x, w, s, out=y), nin + nout)
        timed("dw_dgrad " + tag, lambda: ops.depthwise3x3_dgrad(dy, w, (H, H), s, out=dx), nin + nout)
        timed("dw_wgrad " + tag, lambda: ops.depthwise3x3_wgrad(x, dy, dw, s), nin + nout)
        if s == 1:
            st = ops.BNState(C, "cuda")
            ops.bn_stats(x, st, eps=1e-5, momentum=0.9)
            # reduction pass reads x, dy; apply pass reads x, dy and writes dx: 5 tensor passes
            timed("bn_act_bwd(clip) " + tag, lambda: ops.bn_act_bwd(x, dy, st, 2, out=dx), 5 * nin)
        del x, dy, y, dx
    return rows


def measure_config4(args, rank, local_rank, world, B, bf16=True, kernel_table=True):
    """One measurement of BASELINE config 4 (MobileNetV2 SNIPER training step) on the already initialised process group:
    device-resident chips/s (`value`) and end to end from pinned host batches (`e2e`), max over ranks.  Returns the block
    on rank 0, None elsewhere."""
    import torch
    import torch.distributed as dist
    from sniper_b200 import model_mnv2 as MM
    from sniper_b200 import synth_batch
    from sniper_b200.trainer import Trainer
    cfg = MM.MCfg()
    cfg.batch_images = B
    cfg.bf16 = bool(bf16)
    npool = 3
    pool = [synth_batch.make_batch(B, seed=300 + 17 * rank + i, device="cpu", pinned=True, A=cfg.num_anchors,
                                   stride=cfg.feat_stride) for i in range(npool)]
    dev_pool = [{k: v.to("cuda:%d" % local_rank) for k, v in b.items()} for b in pool]
    h2d = sum(v.numel() * v.element_size() for v in pool[0].values())
    net = MM.SniperMobileNetV2(cfg, device="cuda:%d" % local_rank)
    trainer = Trainer(cfg, device="cuda:%d" % local_rank, world_size=world, use_graph=not args.no_graph, net=net)
    trainer.load(pool[0])
    trainer.capture()
    sampler = ClockSampler(local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def dev_step(i):
        b = dev_pool[i % npool]
        for k, v in b.items():
            trainer.static[k].copy_(v, non_blocking=True)
        trainer.step_device()

    for i in range(max(args.warmup, 3)):
        dev_step(i)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        dev_step(i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    for i in range(2):
        trainer.step(pool[i % npool], prefetch=pool[(i + 1) % npool])
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    losses = None
    for i in range(args.steps):
        losses = trainer.step(pool[(i + 2) % npool], prefetch=pool[(i + 3) % npool])
    t1.record()
    barrier()
    ms_e2e = t0.elapsed_time(t1)
    sampler.stop_flag = True
    t = torch.tensor([ms, ms_e2e], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    launches = trainer.launches_per_step
    if rank == 0 and os.environ.get("SNIPER_BREAKDOWN"):
        entry_point_breakdown(trainer, os.environ["SNIPER_BREAKDOWN"].replace(".md", "") + "_config4.md")
    del trainer, net, dev_pool
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    peaks, peak_src = load_peaks()
    chips = B * world * args.steps
    block = {
        "metric": "512x512 chips/sec train (MobileNetV2 SNIPER)", "value": round(chips / (ms / 1e3), 2), "unit": "chips/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if cfg.bf16 else "tf32",
        "data": "synthetic",
        "config": {"workload": "BASELINE.json configs[3]: MobileNetV2 SNIPER, 512x512 chips, %d chips/GPU, stride 32, 15 "
                               "anchors, mixed precision (bf16 for the reference's fp16); random-init weights; the step's "
                               "working set (GBs of activations) exceeds L2, inputs rotate over %d HBM-resident batches"
                               % (B, npool), "global_batch": B * world, "parallelism": "dp%d" % world},
        "e2e": {"value": round(chips / (ms_e2e / 1e3), 2), "unit": "chips/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": 32, "ms_per_step": round(ms_e2e / args.steps, 3)},
        "gpu_launches": launches * args.steps, "launches_per_step": launches, "losses": losses,
        "clocks": sampler.summary()}
    # SURVEY 8d: MobileNetV2 forward 9.73 GFLOP / chip (backbone 3.26 incl. 0.216 depthwise, heads 6.47); a training step
    # ~3x that.  At these rates the tensor cores idle: the configuration is HBM bound (BatchNorm, depthwise, PSROI).
    block["algorithmic_gflop_per_chip"] = {"fwd": 9.73, "train_step": 29.2}
    block["tensor_tflops_at_this_rate"] = round(block["value"] * 29.2e9 / 1e12, 1)
    if kernel_table:
        table = hbm_kernel_table(B, bool(cfg.bf16), peaks["hbm_gbs"])
        block["hbm_kernels"] = table
        block["hbm_peak_gbs"] = peaks["hbm_gbs"]
        block["peak_source"] = peak_src
        dom = max((r for r in table if r["kernel"].startswith("bn_act_bwd")), key=lambda r: r["us"])
        block["roofline"] = {"bound": "hbm", "kernel": "sniper_bn_act_bwd (largest per-step share of this configuration; shape "
                             + dom["kernel"].split(") ")[1] + ", timed alone)", "achieved": dom["gbs"], "peak": peaks["hbm_gbs"],
                             "unit": "GB/s", "frac": dom["frac_of_hbm_peak"], "traffic": None,
                             "algorithmic_bytes_per_launch": int(dom["algorithmic_mb"] * 1e6)}
    if kernel_table and not getattr(args, "skip_cpu", False):
        # the same step on the host cores (oracle port, bounded sample; a reported baseline, not a target)
        try:
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import cpu_train_step
            block["cpu_baseline"] = cpu_train_step.run_mnv2(1, steps=3, warmup=1, budget_s=20)
        except Exception as e:
            block["cpu_baseline"] = {"error": "%s: %s" % (type(e).__name__, e)}
    return block


def run_config4(args):
    """`bench.py --config4 B`: BASELINE config 4 alone -- MobileNetV2 SNIPER, 512x512 chips, mixed precision (bf16 in place
    of the reference's fp16; --fp32 for TF32), B chips per GPU (BASELINE: 40 = 320 / 8), synthetic chips + boxes,
    random-init weights.  One JSON line."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    block = measure_config4(args, rank, local_rank, world, int(args.config4), bf16=not args.fp32)
    if rank == 0:
        print(json.dumps(block), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_ours(args):
    import torch
    import torch.distributed as dist
    from sniper_b200 import model, synth_batch
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        raise SystemExit("--gpus %d needs torch.distributed.run (WORLD_SIZE unset)" % args.gpus)
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pool = [synth_batch.make_batch(args.chips, seed=100 + 17 * rank + i, device="cpu", pinned=True) for i in range(args.pool)]
    dev_pool = [{k: v.to("cuda:%d" % local_rank) for k, v in b.items()} for b in pool]
    h2d = sum(v.numel() * v.element_size() for v in pool[0].values())
    sampler = ClockSampler(local_rank)
    # ---- the metric's configuration: BASELINE.json configs[1] (fp32 storage, TF32 tensor-core math)
    cfg = model.Cfg()
    cfg.batch_images = args.chips
    cfg.bf16 = bool(args.bf16)
    m = measure(args, cfg, rank, local_rank, world, pool, dev_pool, sampler, dump_dir=args.dump_outputs)
    # ---- configs[2]'s precision (bf16 backbone + fp32 master weights) on the same N GPUs, reported as an extra block
    m3 = None
    if not args.bf16 and not args.skip_config3:
        cfg3 = model.Cfg()
        cfg3.batch_images = args.chips
        cfg3.bf16 = True
        m3 = measure(args, cfg3, rank, local_rank, world, pool, dev_pool)
    # ---- configs[3]: the MobileNetV2 SNIPER step (40 chips/GPU, mixed precision) as one more extra block
    m4 = None
    # (only at N = 1 unless --config4-multi: its multi-GPU path shares the trainer's bucketed all-reduce but has not been
    # run on more than one GPU, and an exception on one rank would leave the others waiting in a collective and take the
    # metric's own scaling run down with it)
    if not args.bf16 and not args.skip_config4 and (world == 1 or args.config4_multi):
        try:
            m4 = measure_config4(args, rank, local_rank, world, 40, bf16=True, kernel_table=(world == 1))
        except Exception as e:      # an extra block must not take the metric's line down with it
            m4 = {"error": "%s: %s" % (type(e).__name__, e)} if rank == 0 else None
    result = None
    if rank == 0:
        chips = args.chips * world * args.steps

        def block(mm, bf16):
            value = chips / (mm["ms"] / 1e3)
            peak_tf = mm["peak_bf16"] / 2.0
            achieved = mm["tc_flops"] / (mm["tc_ms"] / 1e3) / 1e12
            # mixed launches (bf16 backbone + TF32 heads): peak = the FLOP-weighted peak of the launch mix, i.e.
            # frac = (time the launches would take at their operand type's peak) / (time they took)
            frac = mm["ideal_ms"] / mm["tc_ms"]
            eff_peak = achieved / frac
            step_ideal = mm["ideal_ms"] * (TRAIN_GFLOP_PER_CHIP * args.chips * 1e9 / mm["tc_flops"])
            return value, {
                "bound": "tensor",
                "kernel": "gemm_tc_kernel (all tcgen05 GEMM/conv/wgrad launches of a step; %s)" % (
                    "bf16 backbone launches + TF32 head launches" if bf16 else "kind::tf32"),
                "achieved": round(achieved, 1), "peak": round(eff_peak if bf16 else peak_tf, 1), "unit": "TFLOP/s",
                "frac": round(frac, 4), "traffic": None if bf16 else ncu_traffic(),
                "launches_per_step": mm["tc_n"], "kernel_ms_per_step": round(mm["tc_ms"], 3),
                "algorithmic_gflop_per_step": round(mm["tc_flops"] / 1e9, 1),
                "peak_source": "%s bf16_tflops_sustained (%.0f) for bf16 operands, half of it for fp32 operands "
                               "(kind::tf32 issues at half the bf16 rate)" % (mm["peak_src"], mm["peak_bf16"]),
                "step_frac": round(step_ideal / (mm["ms"] / args.steps), 4)}

        value, roof = block(m, bool(args.bf16))
        e2e = chips / (m["ms_e2e"] / 1e3)
        cpu = None
        if not args.skip_cpu:
            cpu = cpu_baseline(sample_chips=args.cpu_chips, steps=3, warmup=1)
        prec = ("bf16 backbone activations/weights + fp32 master weights, fp32 (TF32 math) heads" if args.bf16
                else "fp32 I/O + TF32 tcgen05 math")
        result = {
            "metric": "512x512 chips/sec train (ResNet-101)", "value": round(value, 2), "unit": "chips/s",
            "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": round(m["ms"] / args.steps, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16 (fp32 master, fp32 heads)" if args.bf16 else "tf32 (fp32 storage)",
            "data": "synthetic",
            "config": {"workload": "ResNet-101 SNIPER Faster-R-CNN/R-FCN, 512x512 chips, batch %d/GPU, %s, "
                                   "fwd+bwd+allreduce+SGD with the reference warm-up LR schedule (BASELINE.json configs[%d])"
                                   % (args.chips, prec, 2 if args.bf16 else 1),
                       "global_batch": args.chips * world, "parallelism": "dp%d" % world,
                       "l2_hygiene": "inputs rotate through %d distinct batches (%.0f MB each); activations >10 GB/step >> 126 MB L2" % (len(pool), h2d / 1e6),
                       "cuda_graph": not args.no_graph},
            "e2e": {"value": round(e2e, 2), "unit": "chips/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 32,
                    "ms_per_step": round(m["ms_e2e"] / args.steps, 3)},
            "gpu_launches": int(m["launches_per_step"] * args.steps),
            "roofline": roof,
            "losses": m["losses"],
            "clocks": sampler.summary(),
        }
        if "iterator" in m:
            itl = m["iterator"]
            result["e2e_iterator"] = {
                "value": round(chips / (itl["ms"] / 1e3), 2), "unit": "chips/s", "ms_per_step": round(itl["ms"] / args.steps, 3),
                "h2d_bytes_per_step": itl["h2d_bytes_per_step"], "d2h_bytes_per_step": 32, "losses": itl["losses"],
                "path": "synthetic roidb -> chip_worker / MNIteratorE2E (host, prefetch thread) -> raw uint8 crops over PCIe "
                        "-> sniper_chip_input + sniper_anchor_target + sniper_anchor_subsample -> Trainer.step_raw"}
        if m3 is not None:
            v3, roof3 = block(m3, True)
            result["config3"] = {
                "workload": "same graph, bf16 backbone activations/weights + fp32 master weights + fp32 (TF32) heads "
                            "(BASELINE.json configs[2] precision) on %d GPU(s), batch %d/GPU" % (world, args.chips),
                "value": round(v3, 2), "unit": "chips/s", "ms_per_step": round(m3["ms"] / args.steps, 3),
                "e2e": {"value": round(chips / (m3["ms_e2e"] / 1e3), 2), "unit": "chips/s",
                        "ms_per_step": round(m3["ms_e2e"] / args.steps, 3)},
                "speedup_vs_tf32": round(v3 / value, 3), "roofline": roof3, "losses": m3["losses"]}
        if m4 is not None:
            result["config4"] = m4
        if cpu is not None:
            result["cpu_baseline"] = cpu
        print(json.dumps(result), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return result


def cpu_baseline(sample_chips=1, steps=2, warmup=1, budget_s=None):
    """Reference-style CPU execution of the same training step on the host cores (kind 'port': the MXNet CPU
    stack cannot be built offline; dense layers run in PyTorch-CPU fp32, SNIPER ops in the C oracle / the reference's
    own CPU MultiProposalTarget binary).  Warm steps only: `warmup` untimed steps precede the `steps` timed ones."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import cpu_train_step
    return cpu_train_step.run(sample_chips, steps=steps, warmup=warmup, budget_s=budget_s)


def run_reference(args):
    """The reference arm: `--steps K --warmup W` training steps of a bounded sample (--cpu-chips chips per step) of the
    same workload on the host cores; stops after ~3 minutes of timed steps and reports the steps really timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cpu = cpu_baseline(sample_chips=args.cpu_chips, steps=args.steps, warmup=min(args.warmup, 3), budget_s=180.0)
    v = cpu["value"]
    print(json.dumps({
        "impl": "reference", "metric": "512x512 chips/sec train (ResNet-101)", "value": v, "unit": "chips/s",
        "n_gpus": args.gpus, "steps": cpu["steps_timed"], "warmup": cpu["warmup_steps"],
        "ms_per_step": round(1e3 * cpu["sec_per_step"], 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": "ResNet-101 SNIPER Faster-R-CNN/R-FCN, 512x512 chips, fp32, CPU host cores; each step = "
                               "%d chip(s) (bounded sample of the 20-chip batch)" % args.cpu_chips},
        "cpu_baseline": cpu,
        "e2e": {"value": v, "unit": "chips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--chips", type=int, default=CHIPS_PER_GPU, help="chips per GPU (BASELINE: 20)")
    ap.add_argument("--pool", type=int, default=7, help="distinct input batches rotated through")
    ap.add_argument("--cpu-chips", type=int, default=1, help="chips in the bounded CPU-baseline sample")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--bf16", action="store_true", help="run the main measurement in mixed precision (configs[2])")
    ap.add_argument("--skip-config3", action="store_true", help="do not append the bf16 block to the JSON line")
    ap.add_argument("--skip-iterator", action="store_true", help="do not measure the e2e_iterator block")
    ap.add_argument("--config5", type=int, default=0, metavar="N_IMAGES",
                    help="instead of the training bench: BASELINE config 5, the AutoFocus inference pyramid on N synthetic "
                         "1333x800 images (imgs/s, per-scale detect / post-processing time, soft-NMS latency)")
    ap.add_argument("--config4", type=int, default=0, metavar="CHIPS_PER_GPU",
                    help="instead of the ResNet-101 bench: BASELINE config 4, the MobileNetV2 SNIPER training step with this "
                         "many chips per GPU (BASELINE: 40), mixed precision unless --fp32")
    ap.add_argument("--fp32", action="store_true", help="--config4 in fp32 storage / TF32 math")
    ap.add_argument("--skip-config4", action="store_true", help="do not append the MobileNetV2 block to the JSON line")
    ap.add_argument("--config4-multi", action="store_true", help="append the MobileNetV2 block at N > 1 too")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (outputs and updated weights, "
                         "a fixed sample of the large ones, <= 64 MB) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.config4 or args.config5 or args.impl == "reference"):
        ap.error("--dump-outputs applies to the ResNet-101 training bench only")
    args.iterator_leg = not args.skip_iterator
    if args.config4:
        run_config4(args)
    elif args.config5:
        run_config5(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
