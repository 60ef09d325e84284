"""Training-step driver: the `Module.forward_backward` / `update` / `update_metric` inner loop of
BaseModule.fit (SNIPER-mxnet/python/mxnet/module/base_module.py:505-535) for the SNIPER graph.

One process per GPU.  Per step: pinned host batch -> H2D (on a copy stream, one step ahead when the caller names the
next batch: `step(batch, prefetch=next_batch)`, as MNIteratorE2E's prefetch threads do), one CUDA-graph replay of
forward+backward, ONE NCCL all-reduce over the flat gradient bucket (replaces the per-key kvstore
push/pull, model.py:126-136 / comm.h:433-553; sum without 1/N as rescale_grad=1.0, utils.py:30,37), one
CUDA-graph replay of the fused SGD-momentum update, D2H of the four loss scalars (what the reference's
metrics read with asnumpy(), lib/train_utils/metric.py:109-125; with AutoFocus training also its two metrics, :50-94).
"""
import torch

from . import lr_scheduler, model, ops


class Trainer:
    def __init__(self, cfg=None, device="cuda:0", world_size=1, use_graph=True, seed=5, deform_offset_std=0.0,
                 scheduler="config", net=None):
        """scheduler: "config" = the reference's WarmupMultiBatchScheduler built from cfg (lr, lr_step, warmup*), None =
        constant cfg.lr, or any callable num_update -> lr.  net: an already constructed network exposing the same
        surface as model.SniperResNet101 (P, fb_phases, forward_backward, train_bns, set_lr, update), e.g.
        model_mnv2.SniperMobileNetV2; default: the ResNet-101 graph built from cfg."""
        self.cfg = cfg or (net.cfg if net is not None else model.Cfg())
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        self.world_size = world_size
        self.overlap_allreduce = True     # False: one all-reduce of the whole buffer after the backward pass (A/B runs)
        self._works = []
        self.net = net if net is not None else model.SniperResNet101(self.cfg, device=self.device, seed=seed,
                                                                     deform_offset_std=deform_offset_std)
        self.use_graph = use_graph
        self.static = None
        self.g_fb = None
        self.g_up = None
        self.out = None
        self.loss_host = torch.zeros(8).pin_memory()
        self.launches_per_step = 0
        # input pipeline: two device staging sets filled by a copy stream while the previous step computes
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self.stage = [None, None]
        self.stage_ready = [None, None]      # event: H2D into stage[i] finished
        self.stage_free = [None, None]       # event: the step that consumed stage[i] has copied it out
        self.stage_owner = [None, None]      # the host batch object sitting in stage[i] (kept alive: identity match)
        self.next_stage = 0
        import os
        self.overlap_allreduce = os.environ.get("SNIPER_AR_OVERLAP", "1") == "1"
        # optimizer state of mxnet.optimizer.SGD that lives on the host: update count and LR schedule
        self.num_update = 0
        if scheduler == "config":
            c = self.cfg
            scheduler = lr_scheduler.from_config(lr=c.lr, lr_step=getattr(c, "lr_step", "5.33"),
                                                 lr_factor=getattr(c, "lr_factor", 0.1), warmup=getattr(c, "warmup", True),
                                                 warmup_lr=getattr(c, "warmup_lr", 0.0005),
                                                 warmup_step=getattr(c, "warmup_step", 1000),
                                                 roidb_len=getattr(c, "roidb_len", None),
                                                 batch_size=getattr(c, "batch_images", 16) * world_size)
        self.scheduler = scheduler
        self.lr = self.cfg.lr

    def next_lr(self, lr=None):
        """mxnet.optimizer: `_update_count` then `_get_lr` -> scheduler(num_update) with the incremented count."""
        self.num_update += 1
        if lr is None:
            lr = self.scheduler(self.num_update) if self.scheduler is not None else self.cfg.lr
        self.lr = float(lr)
        return self.lr

    # ---- device-resident step (inputs already in HBM)
    def _alloc_static(self, batch):
        self.static = {k: torch.empty_like(v, device=self.device) for k, v in batch.items()}

    def load(self, host_batch):
        """H2D of one chip batch (pinned host tensors) into the static device buffers."""
        if self.static is None:
            self._alloc_static(host_batch)
        for k, v in host_batch.items():
            self.static[k].copy_(v, non_blocking=True)

    def prefetch(self, host_batch):
        """Starts the H2D of a FUTURE batch on the copy stream (overlaps the step in flight)."""
        i = self.next_stage
        self.next_stage ^= 1
        if self.stage[i] is None:
            self.stage[i] = {k: torch.empty_like(v, device=self.device) for k, v in host_batch.items()}
        if self.stage_free[i] is not None:
            self.copy_stream.wait_event(self.stage_free[i])
        with torch.cuda.stream(self.copy_stream):
            for k, v in host_batch.items():
                self.stage[i][k].copy_(v, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        self.stage_ready[i] = ev
        self.stage_owner[i] = host_batch

    def _load_or_take(self, host_batch):
        """Brings `host_batch` into the static buffers: from its staging set if it was prefetched, else by H2D now."""
        for i in (0, 1):
            if self.stage_owner[i] is host_batch and self.stage_ready[i] is not None:
                if self.static is None:
                    self._alloc_static(host_batch)
                cur = torch.cuda.current_stream()
                cur.wait_event(self.stage_ready[i])
                for k in self.static:
                    self.static[k].copy_(self.stage[i][k], non_blocking=True)     # D2D, ~25 us
                ev = torch.cuda.Event()
                ev.record(cur)
                self.stage_free[i] = ev
                self.stage_owner[i] = None
                return
        self.load(host_batch)

    def _allreduce(self):
        """The whole gradient buffer in one collective (eager / warm-up path)."""
        if self.world_size > 1:
            torch.distributed.all_reduce(self.net.P.g, op=torch.distributed.ReduceOp.SUM)

    def _allreduce_bucket(self, k):
        """Starts the sum of gradient bucket k over the ranks on NCCL's own stream (it first waits for everything
        enqueued so far on the current stream, i.e. the phase that produced the bucket) and returns at once, so the next
        backward phase overlaps the transfer.  No 1/N: rescale_grad = 1.0 (lib/train_utils/utils.py:30,37)."""
        if self.world_size > 1 and self.overlap_allreduce:
            a, b = self.net.P.bucket_ranges[k]
            self._works.append(torch.distributed.all_reduce(self.net.P.g[a:b], op=torch.distributed.ReduceOp.SUM,
                                                            async_op=True))

    def _allreduce_finish(self):
        if self.world_size > 1:
            if self.overlap_allreduce:
                for w in self._works:
                    w.wait()                      # the current stream waits for the collective
                self._works = []
            else:
                self._allreduce()

    def _snapshot(self):
        P = self.net.P
        bns = self.net.train_bns()
        return (P.w.clone(), P.mom.clone(), [(b.st.moving_mean.clone(), b.st.moving_var.clone()) for b in bns])

    def _restore(self, snap):
        P = self.net.P
        P.w.copy_(snap[0])
        P.mom.copy_(snap[1])
        for b, (m, v) in zip(self.net.train_bns(), snap[2]):
            b.st.moving_mean.copy_(m)
            b.st.moving_var.copy_(v)

    def capture(self):
        """Warm up eagerly, then capture forward+backward and the optimizer update as two CUDA graphs.  The warm-up runs
        complete training steps on whatever sits in the static buffers; weights, momentum and the BN moving statistics
        are snapshotted before and restored afterwards, so capture() leaves the model exactly as it found it (a freshly
        loaded checkpoint is not disturbed and the first step() applies ONE update, like the reference's)."""
        snap = self._snapshot()
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.net.set_lr(0.0)
            for _ in range(2):
                ops.reset_launch_count()
                self.out = self.net.forward_backward(self.static)
                self._allreduce()
                self.net.update()
                self.launches_per_step = ops.launch_count()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self._restore(snap)
        if not self.use_graph:
            return
        # forward + backward as one CUDA graph per gradient bucket (model.fb_phases), sharing one memory pool: between
        # the replays the trainer starts the bucket's all-reduce, which then runs under the next phase's kernels
        pool = torch.cuda.graph_pool_handle()
        self.g_fb = []
        phases = self.net.fb_phases(self.static)
        for _ in range(getattr(self.net, "n_phases", 3)):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, pool=pool):
                self.out = next(phases)
            self.g_fb.append(g)
        self.g_up = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.g_up, pool=pool):
            self.net.update()
        torch.cuda.synchronize()

    def step_device(self, lr=None):
        """One training step on the batch currently in the static buffers.  The learning rate comes from the schedule
        (or `lr`) and reaches the captured update graph through the device hyper-parameter buffer."""
        self.net.set_lr(self.next_lr(lr))
        if self.g_fb is not None:
            for k, g in enumerate(self.g_fb):
                g.replay()
                self._allreduce_bucket(k)
            self._allreduce_finish()
            self.g_up.replay()
        else:
            self.out = self.net.forward_backward(self.static, on_bucket=self._allreduce_bucket)
            self._allreduce_finish()
            self.net.update()
        return self.out

    def _losses(self):
        """The host loss scalars of the step just run.  A network that trains the AutoFocus branch (Cfg.autofocus) adds the
        two AutoFocus metrics of lib/train_utils/metric.py:50-94 for this batch: AutoFocusLogLoss (mean -log p(label)
        over the FocusPixel labels != -1) and AutoFocusAcc (argmax == label over the same); nan without a valid label."""
        h = self.loss_host
        res = {"rpn_cls_loss": float(h[0]), "rpn_bbox_loss": float(h[1]), "rcnn_cls_loss": float(h[2]),
               "rcnn_bbox_loss": float(h[3]), "lr": self.lr}
        if getattr(self.net, "af_train", False):
            n = float(h[6])
            res["autofocus_logloss"] = float(h[4]) / n if n > 0 else float("nan")
            res["autofocus_acc"] = float(h[5]) / n if n > 0 else float("nan")
        return res

    # ---- public end-to-end step from the iterator's raw batch (uint8 source rectangles + chip tables)
    def step_raw(self, raw, input_stage, lr=None):
        """One training step on a `iterator.RawBatch`: H2D of the raw bytes, GPU input stage (resize / mean / flip,
        anchor matching, label subsampling), forward + backward + all-reduce + update, D2H of the losses."""
        batch = input_stage.run(raw)
        if self.static is None:
            self.static = {k: torch.empty_like(v) for k, v in batch.items()}
        for k, v in batch.items():
            self.static[k].copy_(v, non_blocking=True)
        if self.g_fb is None and self.use_graph:
            self.capture()
        out = self.step_device(lr)
        self.loss_host.copy_(out["losses"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._losses()

    # ---- public end-to-end step: host batch in, host losses out
    def step(self, host_batch, prefetch=None, lr=None):
        """One training step on `host_batch` (pinned host tensors) -> host loss scalars.  `prefetch`: the batch of the
        NEXT call; its H2D copy is issued now on the copy stream and overlaps this step's compute.  `lr` overrides the
        schedule for this update."""
        self._load_or_take(host_batch)
        if prefetch is not None:
            self.prefetch(prefetch)
        if self.g_fb is None and self.use_graph:
            self.capture()
        out = self.step_device(lr)
        self.loss_host.copy_(out["losses"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self._losses()
