"""Sequencer of the hot path: owns the activation arena for a batch size and replays a
pre-built list of C-ABI kernel launches for forward and backward (SURVEY.md §3.2/§3.3 give the
HF call order this follows: modeling_vit.py:100-128 embeddings, :328-346 per layer, :455 final
LayerNorm, :641-646 head + loss; backward is the reverse autograd order of §3.3).

Data layout in HBM (per-GPU batch B, T tokens, D hidden, F intermediate, M = B·T):
  residual stream ........ fp32 [M, D]   (h before every layer, h1 after attention)
  GEMM operands .......... bf16 [M, D|3D|F] row-major (K contiguous for forward/dgrad; the same
                           buffers are read "MN-major" by the wgrad GEMMs, no transposes)
  fused QKV .............. bf16 [B, T, 3, H, 64] = [M, 3D]   (attention reads it in place)
  weights ................ fp32 masters in one flat buffer + bf16 shadow of the GEMM weights
  gradients .............. one flat fp32 buffer (param.grad are views); wgrad GEMMs accumulate
                           into it with red.global.add, so split-K needs no workspace.
Nothing here allocates per step: every launch argument is fixed when the arena is built, which
is also what makes the whole step capturable in a CUDA graph.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Callable, Dict, List, Optional, Set, Tuple

import torch

from . import _lib, ops
from ._lib import (EPI_ACCUM_F32, EPI_BIAS_BF16, EPI_BIAS_GELUG_BF16, EPI_BIAS_RESID_F32, EPI_MUL_BF16, EPI_PATCH_F32,
                   EPI_STORE_BF16, EPI_UNPATCH_F32)

bf16, f32 = torch.bfloat16, torch.float32


class _Plan:
    """A list of (cfunc, args) launches; ``run`` appends the stream and checks return codes.  Steps marked with
    ``side(True)`` run on ``side_stream`` (on the main stream when it is None)."""

    def __init__(self, side_stream: Optional[torch.cuda.Stream] = None):
        self.steps: List[Tuple[object, tuple, str]] = []
        self.gemm_flops: Dict[int, float] = {}      # step index → 2·M·N·K (bench.py's roofline leg)
        self.side_stream = side_stream
        self.side_steps: Set[int] = set()           # indices of the steps launched on the side stream
        self._segments = {}                         # callbacks? → [(CUDAGraph | None, callback | None)]
        self._warm = set()
        self._keep = []      # keeps GemmArgs structs alive
        self._side = False
        self.sync_points: List[Tuple[torch.cuda.Event, Callable]] = []

    def side(self, on: bool):
        """Steps added while on=True are launched on the side stream (weight-gradient work that only the optimizer
        consumes); fork()/join() order it against the main chain."""
        self._side = on

    def fork(self):
        self.steps.append((None, (), "fork"))  # the side stream waits for everything enqueued on main so far

    def join(self):
        self.steps.append((None, (), "join"))  # the main stream waits for everything enqueued on the side stream so far

    def _launch(self, fn, args: tuple, name: str):
        if self._side:
            self.side_steps.add(len(self.steps))
        self.steps.append((fn, args, name))

    def add(self, name: str, *args):
        self._launch(getattr(_lib.lib(), name), args, name)

    def gemm(self, a, b, M, N, K, d, epilogue, **kw):
        """One vitk_gemm_bf16 launch; keyword arguments as for ops.gemm_args."""
        g = ops.gemm_args(a, b, M, N, K, d, epilogue=epilogue, **kw)
        self._keep.append(g)
        self.gemm_flops[len(self.steps)] = 2.0 * M * N * K
        self._launch(_lib.lib().vitk_gemm_bf16, (C.byref(g),), "vitk_gemm_bf16")

    def call(self, fn: Callable[[], None]):
        self.steps.append((None, (fn,), "python"))

    def sync_point(self, after: Callable[[torch.cuda.Event], None]) -> None:
        """Everything enqueued on the main stream so far is marked by an EXTERNAL event (an event-record node when the
        plan is replayed as a CUDA graph — the graph is not cut), and ``after(event)`` is called on the host once the whole
        plan has been enqueued: the gradient sync then makes its communication stream wait for the event.  The bucket
        boundaries of data-parallel training cost no graph segmentation and no host callback in the middle of backward."""
        ev = torch.cuda.Event(external=True, enable_timing=os.environ.get("VITK_SYNC_TIMING") == "1")   # timing: tools/peer_sync_probe.py
        self.steps.append((None, (ev,), "record"))
        self.sync_points.append((ev, after))

    def _run_range(self, lo: int, hi: int, stream: int, run_py: bool = True):
        side = self.side_stream
        side_handle = side.cuda_stream if side is not None else stream
        for i in range(lo, hi):
            fn, args, name = self.steps[i]
            if fn is None:
                if name == "python":
                    if run_py:
                        args[0]()
                elif name == "record":
                    args[0].record(torch.cuda.current_stream())
                elif side is not None:
                    main = torch.cuda.current_stream()
                    ev = torch.cuda.Event()
                    if name == "fork":
                        ev.record(main)
                        side.wait_event(ev)
                    else:
                        ev.record(side)
                        main.wait_event(ev)
                continue
            rc = fn(*args, side_handle if i in self.side_steps else stream)
            if rc != 0:
                _lib.check(rc, name)

    def run(self, stream: int, callbacks: bool = True):
        """Enqueue the plan on the current stream.  The first call launches kernel by kernel (it also initialises
        per-kernel attributes and the tensor-map cache); the second call captures every run of launches between two
        Python callbacks into a CUDA graph (side-stream forks/joins become parallel branches), and from then on a
        plan costs one cudaGraphLaunch per segment instead of one ctypes call + cudaLaunchKernelEx per kernel
        (≈140 per plan).  ``callbacks=False`` skips the Python callbacks (no gradient sync attached): one segment."""
        self._enqueue(stream, callbacks)
        if callbacks:
            for ev, after in self.sync_points:
                after(ev)

    def _enqueue(self, stream: int, callbacks: bool):
        if torch.cuda.is_current_stream_capturing():
            self._run_range(0, len(self.steps), stream, callbacks)
            return
        segs = self._segments.get(callbacks)
        if segs is None:
            if callbacks not in self._warm:
                self._warm.add(callbacks)
                self._run_range(0, len(self.steps), stream, callbacks)
                return
            segs = self._segments[callbacks] = self._capture(callbacks)
        for g, fn in segs:
            if fn is None:
                g[0].replay()
                ops.note_graph_replay(g[1])
            else:
                fn()

    def _capture(self, callbacks: bool):
        bounds, lo = [], 0
        for i, (fn, args, name) in enumerate(self.steps):
            if fn is None and name == "python" and callbacks:
                if i > lo:
                    bounds.append((lo, i, None))
                bounds.append((i, i + 1, args[0]))
                lo = i + 1
        if lo < len(self.steps):
            bounds.append((lo, len(self.steps), None))
        segs = []
        for lo, hi, cb in bounds:
            if cb is not None:
                segs.append((None, cb))
                continue
            g = torch.cuda.CUDAGraph()
            n0 = ops.direct_launch_count()
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._run_range(lo, hi, torch.cuda.current_stream().cuda_stream, run_py=False)
            segs.append(((g, ops.direct_launch_count() - n0), None))
        return segs


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


class Arena:
    """Activation + scratch buffers and launch plans for one (batch size, training?) pair."""

    def __init__(self, eng: "Engine", B: int, train: bool):
        cfg = eng.cfg
        dev = eng.dev
        D, Fi, H, L, Cn = cfg.hidden_size, cfg.intermediate_size, cfg.num_attention_heads, cfg.num_hidden_layers, cfg.num_labels
        T, P = cfg.seq_len, cfg.num_patches
        M = B * T
        self.B, self.train, self.M = B, train, M
        self.ticket = -1

        def new(shape, dt):
            return torch.empty(shape, dtype=dt, device=dev)

        nl = L if train else 1                     # inference reuses one layer's worth of buffers
        self.apatch = new((B * P, 768), bf16)
        self.h = [new((M, D), f32) for _ in range(L + 1 if train else 1)]
        self.h1 = [new((M, D), f32) for _ in range(nl)] if train else self.h
        self.n1 = [new((M, D), bf16) for _ in range(nl)]
        self.n2 = [new((M, D), bf16) for _ in range(nl)] if train else self.n1
        self.st = [new((4, M), f32) for _ in range(nl)]          # mean1, rstd1, mean2, rstd2
        self.qkv = [new((M, 3 * D), bf16) for _ in range(nl)]
        self.o = [new((M, D), bf16) for _ in range(nl)]
        self.lse = [new((B, H, T), f32) for _ in range(nl)]
        self.gp = [new((M, Fi), bf16) for _ in range(nl)] if train else None     # gelu'(u), saved for backward
        self.a = [new((M, Fi), bf16) for _ in range(nl)]
        self.labels = new((B, Cn), f32)
        self.logits = new((B, Cn), f32)
        self.loss = new((1,), f32)
        self.dlogits = new((B, Cn), f32)
        self.hstat = new((2, B), f32)
        self.fwd = self._build_forward(eng, with_labels=False)
        self.fwd_loss = self._build_forward(eng, with_labels=True)
        self._eng = eng
        self._outputs_plans: Dict[bool, _Plan] = {}
        self.hs: Optional[torch.Tensor] = None         # eval arena, outputs plans: the residual stream of every layer
        self.qkv_all: List[torch.Tensor] = self.qkv if train else []
        self.lse_all: List[torch.Tensor] = self.lse if train else []
        if train:
            self.dh = [new((M, D), bf16) for _ in range(2)]
            self.dn = new((M, D), bf16)
            self.du = new((M, Fi), bf16)
            self.do = new((M, D), bf16)
            self.dqkv = new((M, 3 * D), bf16)
            self.attn_ws = new((ops.attn_bwd_workspace_bytes(B, T, H),), torch.uint8)
            self.dpatch = new((B * P, D), bf16)
            self.dloss = new((1,), f32)
            self.dlogits_in = new((B, Cn), f32)
            self._bwd_plans: Dict[Tuple[bool, bool], _Plan] = {}
            self._data_plans: Dict[bool, _Plan] = {}
            self._sink: Optional[dict] = None
            self.bwd_loss = self.backward_plan(True, False)
            self.bwd_logits = self.backward_plan(False, False)

    def backward_plan(self, from_loss: bool, staged: bool) -> _Plan:
        """Launch plan of the backward pass writing gradients into the flat buffer (staged=False) or into the
        accumulation staging buffer (staged=True, built on first use)."""
        key = (from_loss, staged)
        pl = self._bwd_plans.get(key)
        if pl is None:
            eng = self._eng
            pl = self._bwd_plans[key] = self._build_backward(eng, from_loss, eng.g_stage() if staged else eng.g)
        return pl

    def data_backward_plan(self, from_loss: bool) -> _Plan:
        """Launch plan of the backward pass that computes only the data gradients, down to ``dh[0]`` (the gradient of
        the embeddings output), for a model none of whose parameters requires grad (built on first use).  It is the
        backward plan without the weight-gradient GEMMs, the bias column sums, the embeddings backward, the side stream
        and the gradient-sync points; it never touches a flat gradient buffer.  The parameter gradients the head and
        LayerNorm entry points must still write go to a small scratch buffer, (C + 2)·D + C floats per arena."""
        pl = self._data_plans.get(from_loss)
        if pl is None:
            eng = self._eng
            if self._sink is None:
                cfg = eng.cfg
                D, Cn = cfg.hidden_size, cfg.num_labels
                buf = torch.empty(((Cn + 2) * D + Cn,), dtype=f32, device=eng.dev)
                gf, bf = buf[Cn * D:(Cn + 1) * D], buf[(Cn + 1) * D:(Cn + 2) * D]
                layer = {"g1": gf, "b1": bf, "g2": gf, "b2": bf, "bo": None, "bf2": None}     # None: no bias column sum
                self._sink = {"wc": buf[:Cn * D].view(Cn, D), "gf": gf, "bf": bf, "bc": buf[(Cn + 2) * D:],
                              "layers": [layer] * cfg.num_hidden_layers}
            pl = self._data_plans[from_loss] = self._build_backward(eng, from_loss, self._sink, data_only=True)
        return pl

    def outputs_plan(self, with_labels: bool) -> _Plan:
        """Forward plan that keeps what hidden states and attention maps are read from (built on first use): the top layer
        runs on every token, and every layer's input stream, qkv and lse stay in buffers of their own — in the train arena
        those that backward keeps anyway; the eval arena gets a [L+1, M, D] stream buffer and L qkv / lse buffers here."""
        pl = self._outputs_plans.get(with_labels)
        if pl is None:
            eng = self._eng
            cfg = eng.cfg
            D, H, L, T = cfg.hidden_size, cfg.num_attention_heads, cfg.num_hidden_layers, cfg.seq_len
            if not self.train and self.hs is None:
                self.hs = torch.empty((L + 1, self.M, D), dtype=f32, device=eng.dev)
                self.qkv_all = [torch.empty((self.M, 3 * D), dtype=bf16, device=eng.dev) for _ in range(L)]
                self.lse_all = [torch.empty((self.B, H, T), dtype=f32, device=eng.dev) for _ in range(L)]
            pl = self._outputs_plans[with_labels] = self._build_forward(eng, with_labels, outputs=True)
        return pl

    def hidden_states(self) -> Tuple[torch.Tensor, ...]:
        """Copies of the L+1 residual-stream tensors an outputs plan left behind, each fp32 [B, T, D]."""
        cfg = self._eng.cfg
        L, T, D = cfg.num_hidden_layers, cfg.seq_len, cfg.hidden_size
        hs = torch.stack(self.h) if self.train else self.hs.clone()
        return hs.view(L + 1, self.B, T, D).unbind(0)

    # ------------------------------------------------------------------ forward plan
    def _build_forward(self, eng: "Engine", with_labels: bool, outputs: bool = False) -> _Plan:
        cfg, w = eng.cfg, eng.w
        D, Fi, H, L, Cn = cfg.hidden_size, cfg.intermediate_size, cfg.num_attention_heads, cfg.num_hidden_layers, cfg.num_labels
        T, P, B, M = cfg.seq_len, cfg.num_patches, self.B, self.M
        eps = cfg.layer_norm_eps
        scale = 64 ** -0.5
        pl = _Plan()
        # residual stream before / after each layer, and where each layer's qkv / lse go: the train arena keeps them all;
        # the eval arena updates one buffer in place, except in an outputs plan
        if self.train:
            hs, qkv, lse = self.h, self.qkv, self.lse
        elif outputs:
            hs, qkv, lse = self.hs, self.qkv_all, self.lse_all
        else:
            hs, qkv, lse = [self.h[0]] * (L + 1), [self.qkv[0]] * L, [self.lse[0]] * L
        h0 = hs[0]
        pl.add("vitk_embed_cls", _p(w["cls"]), _p(w["pos"]), B, T, D, _p(h0))
        pl.gemm(self.apatch, w["wp16"], B * P, D, 768, h0, EPI_PATCH_F32, bias=w["bp"], aux=w["pos"], rows_in=P, rows_out=T,
                row_off=1, ldd=D, ld_aux=D)
        def cls_rows(t: torch.Tensor) -> torch.Tensor:      # the B CLS rows of a [B·T, width] buffer, in place (row stride T·width)
            width = t.shape[1]
            return t.view(B, T * width)[:, :width]

        for l in range(L):
            i = l if self.train else 0
            hin, hout = hs[l], hs[l + 1]
            h1 = self.h1[i] if self.train else hout
            lw = w["layers"][l]
            st = self.st[i]
            pl.add("vitk_layernorm_fwd", _p(hin), D, _p(lw["g1"]), _p(lw["b1"]), eps, M, D, _p(self.n1[i]), _p(st[0]), _p(st[1]))
            pl.gemm(self.n1[i], lw["wqkv16"], M, 3 * D, D, qkv[l], EPI_BIAS_BF16, bias=lw["bqkv"])
            if l == L - 1 and eng.cls_only_top and not outputs:
                # ---- top layer: the classifier reads sequence_output[:, 0] only (HF modeling_vit.py:641), so after the keys
                # and values of all tokens exist, everything else of this layer is computed for the B CLS rows alone —
                # attention of one query per head, then out-proj / LN / MLP on strided [B, ·] views that leave the rows
                # where the (CLS-only) backward of this layer expects them.  Dead rows are never read; FLOPs in bench.py
                # stay on the dense convention.  (An outputs plan needs every row, and runs this layer densely: the rows
                # the CLS-only backward reads are among those the dense layer writes.)
                pl.add("vitk_attn_cls_fwd", _p(qkv[l]), B, T, H, scale, _p(self.o[i]), _p(lse[l]))
                o_c, hin_c, h1_c, hout_c = cls_rows(self.o[i]), cls_rows(hin), cls_rows(h1), cls_rows(hout)
                n2_c, a_c = cls_rows(self.n2[i]), cls_rows(self.a[i])
                pl.gemm(o_c, lw["wo16"], B, D, D, h1_c, EPI_BIAS_RESID_F32, bias=lw["bo"], aux=hin_c)
                pl.add("vitk_layernorm_fwd_rows", _p(h1), T * D, _p(lw["g2"]), _p(lw["b2"]), eps, B, D, T, _p(self.n2[i]),
                       _p(st[2]), _p(st[3]))
                pl.gemm(n2_c, lw["w1_16"], B, Fi, D, a_c, EPI_BIAS_GELUG_BF16, d2=cls_rows(self.gp[i]) if self.train else None,
                        bias=lw["bf1"])
                pl.gemm(a_c, lw["w2_16"], B, D, Fi, hout_c, EPI_BIAS_RESID_F32, bias=lw["bf2"], aux=h1_c)
                continue
            pl.add("vitk_attn_fwd", _p(qkv[l]), B, T, H, scale, _p(self.o[i]), _p(lse[l]))
            pl.gemm(self.o[i], lw["wo16"], M, D, D, h1, EPI_BIAS_RESID_F32, bias=lw["bo"], aux=hin)
            pl.add("vitk_layernorm_fwd", _p(h1), D, _p(lw["g2"]), _p(lw["b2"]), eps, M, D, _p(self.n2[i]), _p(st[2]), _p(st[3]))
            pl.gemm(self.n2[i], lw["w1_16"], M, Fi, D, self.a[i], EPI_BIAS_GELUG_BF16, d2=self.gp[i] if self.train else None,
                    bias=lw["bf1"])
            pl.gemm(self.a[i], lw["w2_16"], M, D, Fi, hout, EPI_BIAS_RESID_F32, bias=lw["bf2"], aux=h1)
        hl = hs[L]
        self.h_last = hl
        if with_labels:
            pl.add("vitk_head_fwd", _p(hl), B, T, D, Cn, _p(w["gf"]), _p(w["bf"]), eps, _p(w["wc"]), _p(w["bc"]), _p(self.labels),
                   _p(self.logits), _p(self.loss), _p(self.dlogits), _p(self.hstat[0]), _p(self.hstat[1]))
        else:
            pl.add("vitk_head_fwd", _p(hl), B, T, D, Cn, _p(w["gf"]), _p(w["bf"]), eps, _p(w["wc"]), _p(w["bc"]), None,
                   _p(self.logits), None, None, _p(self.hstat[0]), _p(self.hstat[1]))
        return pl

    # ------------------------------------------------------------------ backward plan
    def _build_backward(self, eng: "Engine", from_loss: bool, g: dict, data_only: bool = False) -> _Plan:
        """data_only: leave out every launch that only produces parameter gradients (see data_backward_plan)."""
        cfg, w = eng.cfg, eng.w
        D, Fi, H, L, Cn = cfg.hidden_size, cfg.intermediate_size, cfg.num_attention_heads, cfg.num_hidden_layers, cfg.num_labels
        T, P, B, M = cfg.seq_len, cfg.num_patches, self.B, self.M
        scale = 64 ** -0.5
        wgrad = not data_only
        pl = _Plan(eng.side_stream if wgrad else None)
        # one external-event sync point per gradient bucket (no host callback, no break in the CUDA graph)
        ends = eng.grad_sync.bucket_end_layers() if eng.grad_sync is not None and wgrad else set()
        done_hi = [L - 1]

        def layer_done(l):
            if l in ends:
                lo, hi = l, done_hi[0]
                done_hi[0] = l - 1
                pl.sync_point(lambda ev, lo=lo, hi=hi: eng._layers_grads_ready(lo, hi, ev))
        dh, dh1 = self.dh
        pl.add("vitk_head_bwd", _p(self.h_last), _p(self.hstat[0]), _p(self.hstat[1]), _p(w["gf"]), _p(w["bf"]), _p(w["wc"]),
               B, T, D, Cn, _p(self.dlogits if from_loss else self.dlogits_in), _p(self.dloss) if from_loss else None,
               _p(dh), _p(g["wc"]), _p(g["bc"]), _p(g["gf"]), _p(g["bf"]))
        # ---- top layer: only the B CLS rows of the residual stream carry gradient (HF modeling_vit.py:641 reads
        # sequence_output[:, 0]), so its MLP and attention-output backward run on strided [B, ·] views of the same
        # buffers (row stride T·width) instead of all M rows.  The zero rows are materialised only where the dense
        # attention backward needs them (dO) and in the residual gradient that flows on (dh1).
        # Algorithmic FLOPs are still counted dense in bench.py; this removes work, it does not approximate.
        def cls_rows(t: torch.Tensor) -> torch.Tensor:
            width = t.shape[1]
            return t.view(B, T * width)[:, :width]

        l = L - 1
        lw, lg, st = w["layers"][l], g["layers"][l], self.st[l]
        dh_c, dh1_c, dn_c, do_c = cls_rows(dh), cls_rows(dh1), cls_rows(self.dn), cls_rows(self.do)
        du_c, a_c, gp_c, n2_c, o_c = cls_rows(self.du), cls_rows(self.a[l]), cls_rows(self.gp[l]), cls_rows(self.n2[l]), cls_rows(self.o[l])
        if wgrad:
            pl.gemm(dh_c, a_c, D, Fi, B, lg["w2"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
            pl.add("vitk_colsum_bf16", _p(dh_c), B, D, T * D, _p(lg["bf2"]))
        pl.gemm(dh_c, lw["w2_16"], B, Fi, D, du_c, EPI_MUL_BF16, b_mn_major=True, aux=gp_c)
        if wgrad:
            pl.gemm(du_c, n2_c, Fi, D, B, lg["w1"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
            pl.add("vitk_colsum_bf16", _p(du_c), B, Fi, T * Fi, _p(lg["bf1"]))
        pl.gemm(du_c, lw["w1_16"], B, D, Fi, dn_c, EPI_STORE_BF16, b_mn_major=True)
        pl.add("vitk_fill_zero", _p(dh1), dh1.numel() * 2)
        pl.add("vitk_layernorm_bwd_rows", _p(self.dn), _p(self.h1[l]), T * D, _p(st[2]), _p(st[3]), _p(lw["g2"]), _p(dh), B, D, T,
               _p(dh1), _p(lg["g2"]), _p(lg["b2"]), _p(lg["bo"]))
        if wgrad:
            pl.gemm(dh1_c, o_c, D, D, B, lg["wo"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
        if eng.cls_only_top:
            pl.gemm(dh1_c, lw["wo16"], B, D, D, do_c, EPI_STORE_BF16, b_mn_major=True)
            pl.add("vitk_attn_cls_bwd", _p(self.qkv[l]), _p(self.o[l]), _p(self.do), _p(self.lse[l]), B, T, H, scale, _p(self.dqkv))
        else:
            pl.add("vitk_fill_zero", _p(self.do), self.do.numel() * 2)
            pl.gemm(dh1_c, lw["wo16"], B, D, D, do_c, EPI_STORE_BF16, b_mn_major=True)
            pl.add("vitk_attn_bwd", _p(self.qkv[l]), _p(self.o[l]), _p(self.do), _p(self.lse[l]), B, T, H, scale,
                   _p(self.dqkv), _p(self.attn_ws))
        if wgrad:
            pl.gemm(self.dqkv, self.n1[l], 3 * D, D, M, lg["wqkv"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
            pl.add("vitk_colsum_bf16", _p(self.dqkv), M, 3 * D, 3 * D, _p(lg["bqkv"]))
        pl.gemm(self.dqkv, lw["wqkv16"], M, D, 3 * D, self.dn, EPI_STORE_BF16, b_mn_major=True)
        pl.add("vitk_layernorm_bwd", _p(self.dn), _p(self.h[l]), D, _p(st[0]), _p(st[1]), _p(lw["g1"]), _p(dh1), M, D,
               _p(dh), _p(lg["g1"]), _p(lg["b1"]), _p(g["layers"][l - 1]["bf2"]) if l > 0 else None)
        layer_done(l)
        # ---- layers L-2 … 0: dense
        # Dense layers.  Weight gradients (and the two wide bias column sums) are consumed only by the optimizer, so
        # they go to a side stream: fork after the tensor they read is produced, join once per layer before the
        # buffers they read are overwritten.  Their CTAs fill the SMs the main chain leaves idle in its partial last
        # waves and kernel tails (every kernel here is a persistent grid sized for the whole GPU).
        for l in reversed(range(L - 1)):
            lw, lg, st = w["layers"][l], g["layers"][l], self.st[l]
            # MLP
            if wgrad:
                pl.fork()
                pl.side(True)
                pl.gemm(dh, self.a[l], D, Fi, M, lg["w2"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
                pl.side(False)
            pl.gemm(dh, lw["w2_16"], M, Fi, D, self.du, EPI_MUL_BF16, b_mn_major=True, aux=self.gp[l])
            if wgrad:
                pl.fork()
                pl.side(True)
                pl.gemm(self.du, self.n2[l], Fi, D, M, lg["w1"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
                pl.add("vitk_colsum_bf16", _p(self.du), M, Fi, Fi, _p(lg["bf1"]))
                pl.side(False)
            pl.gemm(self.du, lw["w1_16"], M, D, Fi, self.dn, EPI_STORE_BF16, b_mn_major=True)
            pl.add("vitk_layernorm_bwd", _p(self.dn), _p(self.h1[l]), D, _p(st[2]), _p(st[3]), _p(lw["g2"]), _p(dh), M, D,
                   _p(dh1), _p(lg["g2"]), _p(lg["b2"]), _p(lg["bo"]))
            # attention
            if wgrad:
                pl.fork()
                pl.side(True)
                pl.gemm(dh1, self.o[l], D, D, M, lg["wo"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
                pl.side(False)
            pl.gemm(dh1, lw["wo16"], M, D, D, self.do, EPI_STORE_BF16, b_mn_major=True)
            pl.add("vitk_attn_bwd", _p(self.qkv[l]), _p(self.o[l]), _p(self.do), _p(self.lse[l]), B, T, H, scale,
                   _p(self.dqkv), _p(self.attn_ws))
            if wgrad:
                pl.fork()
                pl.side(True)
                pl.gemm(self.dqkv, self.n1[l], 3 * D, D, M, lg["wqkv"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
                pl.add("vitk_colsum_bf16", _p(self.dqkv), M, 3 * D, 3 * D, _p(lg["bqkv"]))
                pl.side(False)
            pl.gemm(self.dqkv, lw["wqkv16"], M, D, 3 * D, self.dn, EPI_STORE_BF16, b_mn_major=True)
            if wgrad:
                pl.join()      # side work of this layer read dh / du / dh1 / dqkv, which the next kernels overwrite
            pl.add("vitk_layernorm_bwd", _p(self.dn), _p(self.h[l]), D, _p(st[0]), _p(st[1]), _p(lw["g1"]), _p(dh1), M, D,
                   _p(dh), _p(lg["g1"]), _p(lg["b1"]), _p(g["layers"][l - 1]["bf2"]) if l > 0 else None)
            layer_done(l)
        if wgrad:
            pl.add("vitk_embed_bwd", _p(dh), B, T, D, _p(g["pos"]), _p(g["cls"]), _p(g["bp"]), _p(self.dpatch))
            pl.gemm(self.dpatch, self.apatch, D, 768, B * P, g["wp"], EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True)
            if eng.grad_sync is not None:
                pl.sync_point(lambda ev: eng._rest_grads_ready(ev))
        return pl


class Engine:
    def __init__(self, model):
        self.model = model
        self.cfg = model.config
        self.dev = model.flat_parameters().device
        self.ticket = 0
        self.arenas: Dict[Tuple[int, bool], Arena] = {}
        self.grad_sync = None            # parallel.GradSync, set by the caller for N>1
        self.side_stream = torch.cuda.Stream(device=self.dev)    # weight-gradient work of the backward plans
        # top encoder layer computed for the CLS rows only (forward and backward); VITK_CLS_ONLY_TOP=0 runs it densely
        self.cls_only_top = os.environ.get("VITK_CLS_ONLY_TOP", "1") != "0"
        self.w = self._weight_views(model.flat_parameters(), model.shadow())
        self.g = self._weight_views(model.flat_grads(), None)
        self._g_stage = None
        self._grad_views = {n: model.layout.view(model.flat_grads(), n) for n in model.layout.names}
        self._params = dict(model.named_parameters())
        self._plist = model.param_list()
        # gradient views handed to autograd: one split of the flat buffer (flat order), reshaped per parameter
        lay = model.layout
        by_off = sorted(lay.names, key=lambda n: lay.offset[n])
        ends = [lay.offset[n] for n in by_off[1:]] + [lay.total]
        self._split_sizes = [e - lay.offset[n] for n, e in zip(by_off, ends)]
        pos = {n: i for i, n in enumerate(by_off)}
        self._spans = [(pos[n], math.prod(lay.shapes[n]), lay.shapes[n]) for n in lay.names]     # HF order

    def g_stage(self):
        if self._g_stage is None:
            self._g_stage = self._weight_views(self.model.stage_grads(), None)
        return self._g_stage

    def _weight_views(self, flat: torch.Tensor, shadow: Optional[torch.Tensor]):
        """Kernel-facing views of a flat buffer laid out by FlatLayout.  With ``shadow`` (bf16 copy
        of the GEMM prefix) the matrix weights come from it under keys ending in ``16``."""
        cfg, lay = self.cfg, self.model.layout
        D, Fi = cfg.hidden_size, cfg.intermediate_size
        want16 = shadow is not None

        def v(name):
            return lay.view(flat, name)

        def v16(name, rows, cols):
            o = lay.offset[name]
            src = shadow if want16 else flat
            return src[o:o + rows * cols].view(rows, cols)

        def span(name, n):
            o = lay.offset[name]
            return flat[o:o + n]

        sfx = "16" if want16 else ""
        out = {"cls": v("vit.embeddings.cls_token").view(D), "pos": v("vit.embeddings.position_embeddings").view(-1, D),
               "bp": v("vit.embeddings.patch_embeddings.projection.bias"),
               "wp" + sfx: v16("vit.embeddings.patch_embeddings.projection.weight", D, 768),
               "gf": v("vit.layernorm.weight"), "bf": v("vit.layernorm.bias"),
               "wc": v("classifier.weight"), "bc": v("classifier.bias"), "layers": []}
        for i in range(cfg.num_hidden_layers):
            p = f"vit.encoder.layer.{i}."
            out["layers"].append({
                "wqkv" + sfx: v16(p + "attention.attention.query.weight", 3 * D, D),
                "bqkv": span(p + "attention.attention.query.bias", 3 * D),
                "wo" + sfx: v16(p + "attention.output.dense.weight", D, D), "bo": v(p + "attention.output.dense.bias"),
                ("w1_16" if want16 else "w1"): v16(p + "intermediate.dense.weight", Fi, D), "bf1": v(p + "intermediate.dense.bias"),
                ("w2_16" if want16 else "w2"): v16(p + "output.dense.weight", D, Fi), "bf2": v(p + "output.dense.bias"),
                "g1": v(p + "layernorm_before.weight"), "b1": v(p + "layernorm_before.bias"),
                "g2": v(p + "layernorm_after.weight"), "b2": v(p + "layernorm_after.bias")})
        return out

    def arena(self, B: int, train: bool) -> Arena:
        key = (B, train)
        a = self.arenas.get(key)
        if a is None:
            a = self.arenas[key] = Arena(self, B, train)
        return a

    # ------------------------------------------------------------------ forward
    def forward(self, pixel_values: torch.Tensor, labels: Optional[torch.Tensor], save: bool, output_attentions: bool = False,
                output_hidden_states: bool = False):
        """Runs the forward plan → (loss | None, logits, hidden_states | None, attentions | None), all fresh tensors.
        Either flag selects the arena's outputs plan; the attention maps are then recomputed per layer by
        vitk_attn_probs straight into one [L, B, H, T, T] allocation."""
        cfg = self.cfg
        B = pixel_values.shape[0]
        ar = self.arena(B, save)
        if pixel_values.device != self.dev:
            pixel_values = pixel_values.to(self.dev, non_blocking=True)
        self.model.shadow()                                   # refresh bf16 weights if the masters moved
        if pixel_values.dtype == torch.uint8:
            x = pixel_values.reshape(B, cfg.image_size, cfg.image_size)
            ops.patchify_u8(x if x.is_contiguous() else x.contiguous(), cfg.image_mean, cfg.image_std, out=ar.apatch)
        else:
            x = pixel_values if pixel_values.dtype == f32 else pixel_values.to(f32)     # HF:444-446 casts to the weight dtype
            ops.patchify_f32(x if x.is_contiguous() else x.contiguous(), out=ar.apatch)
        if labels is not None:
            ar.labels.copy_(labels.reshape(B, cfg.num_labels), non_blocking=True)
        if output_attentions or output_hidden_states:
            plan = ar.outputs_plan(labels is not None)
        else:
            plan = ar.fwd_loss if labels is not None else ar.fwd
        plan.run(torch.cuda.current_stream().cuda_stream)
        if save:
            self.ticket += 1
            ar.ticket = self.ticket
        hidden = ar.hidden_states() if output_hidden_states else None
        attn = None
        if output_attentions:
            H, L, T = cfg.num_attention_heads, cfg.num_hidden_layers, cfg.seq_len
            probs = torch.empty((L, B, H, T, T), dtype=f32, device=self.dev)
            for l in range(L):
                ops.attn_probs(ar.qkv_all[l], ar.lse_all[l], B, T, H, 64 ** -0.5, out=probs[l])
            attn = probs.unbind(0)
        loss = ar.loss[0].clone() if labels is not None else None
        return loss, ar.logits.clone(), hidden, attn

    # ------------------------------------------------------------------ backward
    def bind_grads(self) -> None:
        """Fold every ``param.grad`` that lives outside the flat gradient buffer (cloned by autograd, replaced by a
        DDP bucket view, assigned by the user) into it and re-point ``param.grad`` at the flat views, so the flat
        optimizer sees all gradients.  Parameters whose grad is None are left alone."""
        for p, (n, gv) in zip(self._plist, self._grad_views.items()):
            gt = p.grad
            if gt is not None and gt.data_ptr() != gv.data_ptr():
                gv.copy_(gt)
                p.grad = gv

    def backward(self, ticket: int, dloss: Optional[torch.Tensor], dlogits: Optional[torch.Tensor],
                 needs: Optional[Tuple[bool, ...]] = None, input_grad: bool = False) -> Tuple[tuple, Optional[torch.Tensor]]:
        """Runs the backward launch plan and returns (one gradient per parameter (HF order; None where ``needs`` is
        False), the gradient of ``pixel_values`` or None).  The parameter gradients are fresh views of the flat buffer the
        kernels wrote.  If no ``param.grad`` is populated the main flat buffer is used (autograd adopts the views, no
        copy); otherwise — gradient accumulation — the kernels write the staging buffer and autograd adds it onto
        ``param.grad``.  When no parameter needs a gradient and ``input_grad`` is set, the arena's data-only plan runs
        instead: no weight-gradient work, no flat gradient buffer and no gradient sync.  With ``input_grad`` the input
        gradient fp32 [B, 3, S, S] is one UNPATCH_F32 GEMM from the final ``dh`` into a fresh tensor."""
        ar = next((a for a in self.arenas.values() if a.train and a.ticket == ticket), None)
        if ar is None:
            raise RuntimeError("chest_x_ray_vit_b200: the activations of this forward were overwritten by a later "
                               "forward with the same batch size; call backward() before the next forward()")
        n = len(self._plist)
        if dloss is None and dlogits is None:
            return (None,) * n, None
        if needs is None:
            needs = (True,) * n
        data_only = input_grad and not any(needs)
        if data_only:
            plan_for = ar.data_backward_plan
        else:
            model = self.model
            staged = any(p.grad is not None for p in self._plist)
            if staged:
                flat = model.stage_grads()
                ops.fill_zero(flat)
            else:
                flat = model.flat_grads()
                if not model._grads_clean:
                    ops.fill_zero(flat)
                model._grads_clean = False
            if self.grad_sync is not None:
                self.grad_sync.begin(flat)

            def plan_for(from_loss: bool) -> _Plan:
                return ar.backward_plan(from_loss, staged)
        stream = torch.cuda.current_stream().cuda_stream
        callbacks = self.grad_sync is not None and not data_only
        if dloss is not None and dlogits is None:
            ar.dloss.copy_(dloss.reshape(1), non_blocking=True)
            plan_for(True).run(stream, callbacks=callbacks)
        else:
            if dloss is not None:      # both the loss and the logits were used downstream
                torch.add(dlogits.to(f32), ar.dlogits * dloss.to(f32), out=ar.dlogits_in)
            else:
                ar.dlogits_in.copy_(dlogits)
            plan_for(False).run(stream, callbacks=callbacks)
        dx = self._input_grad(ar) if input_grad else None
        ar.ticket = -1
        if data_only:
            return (None,) * n, dx
        chunks = flat.split_with_sizes(self._split_sizes)
        return tuple((chunks[i].view(sh) if chunks[i].numel() == k else chunks[i][:k].view(sh)) if nd else None
                     for (i, k, sh), nd in zip(self._spans, needs)), dx

    def _input_grad(self, ar: Arena) -> torch.Tensor:
        """d loss / d pixel_values = col2im(dh[:, 1:] · Wp): the final ``dh`` (layer 0's LayerNorm backward wrote it) times
        the bf16 patch weight [D, 768], scattered into a fresh fp32 [B, 3, S, S] tensor by the UNPATCH_F32 epilogue.
        vitk_patchify_f32 only reorders and rounds its input, so this is the gradient of the fp32 pixels as passed.
        Fresh because autograd adopts it as ``x.grad`` without a copy."""
        cfg = self.cfg
        S = cfg.image_size
        dx = torch.empty((ar.B, 3, S, S), dtype=f32, device=self.dev)
        ops.gemm(ar.dh[0], self.w["wp16"], ar.M, 768, cfg.hidden_size, dx, epilogue=EPI_UNPATCH_F32, b_mn_major=True,
                 ldd=S, rows_out=cfg.seq_len, row_off=1)
        return dx

    def _layers_grads_ready(self, lo: int, hi: int, ev=None) -> None:
        if self.grad_sync is not None:
            self.grad_sync.layers_ready(lo, hi, after=ev)

    def _rest_grads_ready(self, ev=None) -> None:
        if self.grad_sync is not None:
            self.grad_sync.rest_ready(after=ev)
