"""CUDA-graph replay of the hot path.

A training step of the module is ≈280 kernel launches enqueued from Python through ctypes, plus autograd's and the
optimizer's host bookkeeping (≈2 ms of host time against a ≈7 ms step: hidden while the host runs ahead of the GPU,
exposed as soon as it does not — small batches, inference at batch ≤ 8, rank 0 of a multi-GPU job driving NCCL hooks).
Every launch argument of the engine's plans is fixed when the arena is built (engine.py), so the whole step is captured
once per (batch size, input dtype) and replayed with a single cudaGraphLaunch:

  GraphedTrainStep(model, optimizer)(pixel_values, labels) -> loss
      [eager] patchify(pixel_values) → arena, labels → arena
      [graph] forward plan → backward plan (side-stream weight-gradient GEMMs become parallel graph branches;
              programmatic-dependent-launch edges are preserved) → ‖g‖² → clip → AdamW (+ bf16 shadow, + grad clear)
      The AdamW step count lives on the device (vitk_adamw_tick): a replay has fixed kernel arguments.
      ``param.grad`` is not materialised (the gradients are consumed and cleared inside the graph); use the eager
      module path when gradients must be inspected, accumulated over micro-batches or all-reduced.

  GraphedForward(model, example)(pixel_values) -> logits          (eval / predict, Trainer.prediction_step)

Same kernels, same order, same numerics as the eager path (tests/test_gpu_graph.py compares them bit for bit where the
kernels are deterministic).
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch

from . import ops


def _patchify_into(model, ar, pixel_values: torch.Tensor) -> None:
    cfg = model.config
    B = pixel_values.shape[0]
    if pixel_values.dtype == torch.uint8:
        x = pixel_values.reshape(B, cfg.image_size, cfg.image_size)
        ops.patchify_u8(x if x.is_contiguous() else x.contiguous(), cfg.image_mean, cfg.image_std, out=ar.apatch)
    else:
        x = pixel_values if pixel_values.dtype == torch.float32 else pixel_values.to(torch.float32)
        ops.patchify_f32(x if x.is_contiguous() else x.contiguous(), out=ar.apatch)


class GraphedForward:
    """no-grad forward of one batch size as one graph launch.  ``model`` must be on the GPU; weights may change between
    calls (the bf16 shadow is refreshed eagerly before the replay when the masters moved)."""

    def __init__(self, model, example: torch.Tensor):
        self.model = model
        model._check_inputs(example)
        eng = model.engine()
        self.B = example.shape[0]
        self.ar = eng.arena(self.B, False)
        model.shadow()
        stream = torch.cuda.Stream(device=eng.dev)
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):                      # warm-up: lazy per-kernel attributes, tensor-map cache
            _patchify_into(model, self.ar, example.to(eng.dev))
            self.ar.fwd.run(stream.cuda_stream)
        torch.cuda.current_stream().wait_stream(stream)
        n0 = ops.direct_launch_count()
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.ar.fwd.run(torch.cuda.current_stream().cuda_stream)
        self.launches_per_replay = ops.direct_launch_count() - n0
        self.replays = 0

    def __call__(self, pixel_values: torch.Tensor) -> torch.Tensor:
        if pixel_values.shape[0] != self.B:
            raise ValueError(f"GraphedForward was captured for batch {self.B}, got {pixel_values.shape[0]}")
        model = self.model
        model._check_inputs(pixel_values)
        model.shadow()
        if pixel_values.device != self.ar.apatch.device:
            pixel_values = pixel_values.to(self.ar.apatch.device, non_blocking=True)
        _patchify_into(model, self.ar, pixel_values)
        self.graph.replay()
        ops.note_graph_replay(self.launches_per_replay)
        self.replays += 1
        return self.ar.logits.clone()


class GraphedTrainStep:
    """forward + backward + global-norm clip + AdamW of ``model`` under ``optimizer`` (a VitkAdamW) per call."""

    def __init__(self, model, optimizer):
        from .optim import VitkAdamW
        if not isinstance(optimizer, VitkAdamW):
            raise TypeError("GraphedTrainStep needs a VitkAdamW (its kernels carry the step count on the device)")
        if any(not p.requires_grad for p in model.param_list()):
            raise ValueError("GraphedTrainStep: frozen parameters are not supported; use the eager path")
        self.model, self.opt = model, optimizer
        self._graphs: Dict[Tuple[int, torch.dtype], tuple] = {}
        self.replays = 0
        self.kernel_launches = 0            # kernels executed by replays (vitk_launch_count only sees the capture)
        self._step_dev: Optional[torch.Tensor] = None
        self._bc_dev: Optional[torch.Tensor] = None

    def _capture(self, pixel_values: torch.Tensor, labels: torch.Tensor):
        model, opt = self.model, self.opt
        eng = model.engine()
        if eng.grad_sync is not None and getattr(eng.grad_sync, "world", 1) > 1:
            raise NotImplementedError("GraphedTrainStep: the overlapped NCCL gradient all-reduce is not captured; "
                                      "use the eager path for data-parallel training")
        B = pixel_values.shape[0]
        ar = eng.arena(B, True)
        p, g = model.flat_parameters(), model.flat_grads()
        if opt._m is None or opt._m.device != p.device or opt._m.numel() != p.numel():
            opt._init_state()
        if self._step_dev is None:
            self._step_dev = torch.zeros(1, dtype=torch.int64, device=p.device)
            self._bc_dev = torch.zeros(2, dtype=torch.float32, device=p.device)
        for q in model.param_list():
            q.grad = None
        model.shadow()
        lay = model.layout
        segs = opt._segments([True] * len(lay.names))
        stream = torch.cuda.Stream(device=eng.dev)
        stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(stream):
            ar.dloss.fill_(1.0)
            ops.fill_zero(g)
        torch.cuda.current_stream().wait_stream(stream)
        torch.cuda.synchronize()
        n0 = ops.direct_launch_count()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            s = torch.cuda.current_stream().cuda_stream
            ar.fwd_loss.run(s)
            ar.backward_plan(True, False).run(s)
            opt._enqueue(g, p, segs, True, 0, (self._step_dev, self._bc_dev))
        n = ops.direct_launch_count() - n0
        model._grads_clean = True
        return graph, ar, n

    def __call__(self, pixel_values: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        model, opt = self.model, self.opt
        model._check_inputs(pixel_values)
        key = (pixel_values.shape[0], pixel_values.dtype)
        ent = self._graphs.get(key)
        if ent is None:
            # one eager forward + backward first (no optimizer step, gradients dropped): per-kernel attributes and the
            # tensor-map cache are initialised outside the capture
            model(pixel_values=pixel_values, labels=labels).loss.backward()
            ent = self._graphs[key] = self._capture(pixel_values, labels)
        graph, ar, n = ent
        if pixel_values.device != ar.apatch.device:
            pixel_values = pixel_values.to(ar.apatch.device, non_blocking=True)
        model.shadow()
        self._step_dev.fill_(opt._step)                      # the host count is authoritative (eager steps may interleave)
        _patchify_into(model, ar, pixel_values)
        ar.labels.copy_(labels.reshape(ar.labels.shape), non_blocking=True)
        graph.replay()
        opt._step += 1
        model.mark_shadow_fresh()
        model._grads_clean = True
        ops.note_graph_replay(n)
        self.replays += 1
        self.kernel_launches += n
        return ar.loss[0]
