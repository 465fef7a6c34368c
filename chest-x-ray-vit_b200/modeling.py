"""Drop-in ``ViTForImageClassification`` for the Chest-X-Ray-ViT fine-tuning path on B200.

Mirrors the surface the reference uses (/root/reference/ViT-Training.py:83-90 constructs it,
:120-132 trains it through HF Trainer, :137 predicts with it) and that HF defines in
transformers/models/vit/modeling_vit.py:605-653 (HF 5.5.0):

    model = ViTForImageClassification(config)            # same parameter names / shapes as HF
    out = model(pixel_values=x, labels=y)                # ImageClassifierOutput(loss, logits)
    out.loss.backward(); optimizer.step()                # fp32 grads land in param.grad
    x.requires_grad_(); model(pixel_values=x).logits[:, c].sum().backward()   # x.grad: saliency / attribution
    out = model(pixel_values=x, output_attentions=True,  # + hidden_states (L+1 × [B,T,D]) and attentions
              output_hidden_states=True)                 #   (L × [B,H,T,T]), as HF's eager attention returns them
    out = model(pixel_values=x512, labels=y,             # another resolution: the position embeddings resized
                interpolate_pos_encoding=True)           #   bicubically to the input's patch grid, as in HF

Every FLOP and byte of forward/backward runs in libvitk's sm_100a kernels through the C ABI
(include/vitk.h); PyTorch provides device memory, streams and the autograd hook only.  There is
no fallback: unsupported configurations raise.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import ops
from .engine import Engine

f32 = torch.float32


@dataclass
class ViTConfig:
    """The HF ViTConfig fields the path depends on (configuration_vit.py:50-65) plus the
    image-processor constants the uint8 fast path needs (image_processing_vit.py:20-27)."""
    hidden_size: int = 768
    num_hidden_layers: int = 12
    num_attention_heads: int = 12
    intermediate_size: int = 3072
    hidden_act: str = "gelu"
    hidden_dropout_prob: float = 0.0
    attention_probs_dropout_prob: float = 0.0
    initializer_range: float = 0.02
    layer_norm_eps: float = 1e-12
    image_size: int = 384
    patch_size: int = 16
    num_channels: int = 3
    qkv_bias: bool = True
    num_labels: int = 14
    problem_type: Optional[str] = "multi_label_classification"
    id2label: Optional[Dict[int, str]] = None
    label2id: Optional[Dict[str, int]] = None
    image_mean: Tuple[float, float, float] = (0.5, 0.5, 0.5)
    image_std: Tuple[float, float, float] = (0.5, 0.5, 0.5)
    output_attentions: bool = False         # defaults of forward()'s keyword arguments, as in HF PretrainedConfig
    output_hidden_states: bool = False

    @classmethod
    def from_hf(cls, hf_config, **overrides) -> "ViTConfig":
        """Build from a ``transformers.ViTConfig`` (or anything with the same attributes)."""
        kw = {}
        for f in cls.__dataclass_fields__:
            if hasattr(hf_config, f):
                kw[f] = getattr(hf_config, f)
        kw.update(overrides)
        return cls(**kw)

    @property
    def num_patches(self) -> int:
        return (self.image_size // self.patch_size) ** 2

    @property
    def seq_len(self) -> int:
        return self.num_patches + 1

    def validate(self) -> None:
        """Hard preconditions of the kernel path (SURVEY §8b): reject, never fall back."""
        def need(cond, msg):
            if not cond:
                raise ValueError(f"chest_x_ray_vit_b200: unsupported config — {msg}")
        need(self.hidden_dropout_prob == 0.0 and self.attention_probs_dropout_prob == 0.0, "dropout must be 0.0")
        need(self.hidden_act == "gelu", "hidden_act must be 'gelu' (exact erf form)")
        need(self.qkv_bias, "qkv_bias must be True")
        need(self.patch_size == 16 and self.num_channels == 3, "patch_size 16 and 3 channels only")
        need(self.image_size % 16 == 0, "image_size must be a multiple of 16")
        need(self.hidden_size == 64 * self.num_attention_heads, "head_dim must be 64")
        need(self.hidden_size in (128, 256, 512, 768, 1024), "hidden_size must be one of 128/256/512/768/1024")
        need(self.intermediate_size % 128 == 0, "intermediate_size must be a multiple of 128")
        need(1 <= self.num_labels <= 64, "num_labels must be in [1, 64]")
        need(self.problem_type in (None, "multi_label_classification"),
             "only the multi-label BCEWithLogits loss of the reference is implemented")


class ImageClassifierOutput:
    """Same access patterns as transformers.modeling_outputs.ImageClassifierOutput
    (modeling_outputs.py:1238-1260): attributes, ``out["loss"]`` and ``out[0]``."""
    __slots__ = ("loss", "logits", "hidden_states", "attentions")

    def __init__(self, loss=None, logits=None, hidden_states=None, attentions=None):
        self.loss, self.logits, self.hidden_states, self.attentions = loss, logits, hidden_states, attentions

    def to_tuple(self):
        return tuple(v for v in (self.loss, self.logits, self.hidden_states, self.attentions) if v is not None)

    def keys(self):
        return [k for k in self.__slots__ if getattr(self, k) is not None]

    def __getitem__(self, k):
        if isinstance(k, str):
            v = getattr(self, k) if k in self.__slots__ else None
            if v is None:
                raise KeyError(k)
            return v
        return self.to_tuple()[k]

    def __contains__(self, k):
        return k in self.__slots__ and getattr(self, k) is not None

    def __iter__(self):
        return iter(self.keys())

    def __len__(self):
        return len(self.to_tuple())


def param_specs(cfg: ViTConfig) -> List[Tuple[str, Tuple[int, ...], str]]:
    """(HF state-dict name, shape, kind) in HF ``named_parameters()`` order (SURVEY App. B.3).
    kind: 'gemm' (bf16 shadow + weight decay), 'decay' (fp32 only, decayed), 'nodecay'
    (biases and LayerNorm affine: excluded from weight decay, HF trainer.py:1280-1290)."""
    D, Fi, P, Cc = cfg.hidden_size, cfg.intermediate_size, cfg.patch_size, cfg.num_channels
    s: List[Tuple[str, Tuple[int, ...], str]] = [
        ("vit.embeddings.cls_token", (1, 1, D), "decay"),
        ("vit.embeddings.position_embeddings", (1, cfg.seq_len, D), "decay"),
        ("vit.embeddings.patch_embeddings.projection.weight", (D, Cc, P, P), "gemm"),
        ("vit.embeddings.patch_embeddings.projection.bias", (D,), "nodecay"),
    ]
    for i in range(cfg.num_hidden_layers):
        p = f"vit.encoder.layer.{i}."
        for n in ("query", "key", "value"):
            s.append((p + f"attention.attention.{n}.weight", (D, D), "gemm"))
            s.append((p + f"attention.attention.{n}.bias", (D,), "nodecay"))
        s += [(p + "attention.output.dense.weight", (D, D), "gemm"), (p + "attention.output.dense.bias", (D,), "nodecay"),
              (p + "intermediate.dense.weight", (Fi, D), "gemm"), (p + "intermediate.dense.bias", (Fi,), "nodecay"),
              (p + "output.dense.weight", (D, Fi), "gemm"), (p + "output.dense.bias", (D,), "nodecay"),
              (p + "layernorm_before.weight", (D,), "nodecay"), (p + "layernorm_before.bias", (D,), "nodecay"),
              (p + "layernorm_after.weight", (D,), "nodecay"), (p + "layernorm_after.bias", (D,), "nodecay")]
    s += [("vit.layernorm.weight", (D,), "nodecay"), ("vit.layernorm.bias", (D,), "nodecay"),
          ("classifier.weight", (cfg.num_labels, D), "decay"), ("classifier.bias", (cfg.num_labels,), "nodecay")]
    return s


class FlatLayout:
    """Where each parameter lives in the flat fp32 buffer.  Order:
         [patch W | layer0 {Wq Wk Wv Wo W1 W2} | ... | layerL-1 {...}]   'gemm'    (bf16 shadow)
         [pos | cls | classifier.W]                                       'decay'
         [every bias and LayerNorm affine, q/k/v biases adjacent]         'nodecay'
    so the fused QKV weight [3D,D] and bias [3D] are single views, each layer's GEMM weights are
    one contiguous all-reduce bucket, and weight decay / bf16 shadow apply to prefixes."""

    def __init__(self, cfg: ViTConfig):
        specs = param_specs(cfg)
        self.shapes = {n: sh for n, sh, _ in specs}
        self.kinds = {n: k for n, _, k in specs}
        order = [n for n, _, k in specs if k == "gemm"] + \
                [n for n, _, k in specs if k == "decay" and "position" in n] + \
                [n for n, _, k in specs if k == "decay" and "position" not in n] + \
                [n for n, _, k in specs if k == "nodecay"]
        self.offset: Dict[str, int] = {}
        off = 0
        self.gemm_end = self.decay_end = 0
        for n in order:
            self.offset[n] = off
            off += (math.prod(self.shapes[n]) + 7) // 8 * 8      # keep every view 32-byte aligned
            if self.kinds[n] == "gemm":
                self.gemm_end = off
            if self.kinds[n] in ("gemm", "decay"):
                self.decay_end = off
        self.total = off
        self.names = [n for n, _, _ in specs]     # HF order
        # all-reduce buckets as (start, end) element ranges, in the order backward finishes them
        D, Fi, L = cfg.hidden_size, cfg.intermediate_size, cfg.num_hidden_layers
        per_layer = 4 * D * D + 2 * D * Fi
        wp = math.prod(self.shapes["vit.embeddings.patch_embeddings.projection.weight"])
        self.layer_range = [(wp + i * per_layer, wp + (i + 1) * per_layer) for i in range(L)]
        self.rest_ranges = [(0, wp), (self.gemm_end, self.total)]

    def view(self, flat: torch.Tensor, name: str) -> torch.Tensor:
        o = self.offset[name]
        return flat[o:o + math.prod(self.shapes[name])].view(self.shapes[name])


class _Holder(nn.Module):
    """Parameter container that only exists to reproduce HF's module/parameter names."""


class ViTForImageClassification(nn.Module):
    main_input_name = "pixel_values"

    def __init__(self, config: ViTConfig):
        super().__init__()
        if not isinstance(config, ViTConfig):
            config = ViTConfig.from_hf(config)
        config.validate()
        self.config = config
        self.num_labels = config.num_labels
        self.layout = FlatLayout(config)
        flat = torch.zeros(self.layout.total, dtype=f32)
        self._flat_params = flat          # plain attribute (not a buffer: DDP would re-broadcast it every forward)
        self._flat_grads: Optional[torch.Tensor] = None
        self._stage_grads: Optional[torch.Tensor] = None     # second gradient buffer, only for accumulation (see backward)
        self._grads_clean = False                            # flat gradient buffer known to be all zero (VitkAdamW step)
        self._flat_shadow: Optional[torch.Tensor] = None     # bf16 copy of the 'gemm' prefix
        self._shadow_version = -1
        self._engine: Optional[Engine] = None
        self._pnames: List[str] = []
        self._plist = None
        for name in self.layout.names:
            self._register(name, nn.Parameter(self.layout.view(flat, name)))
        self.reset_parameters()

    # ------------------------------------------------------------------ HF checkpoint interchange
    @classmethod
    def from_pretrained(cls, source, **kwargs) -> "ViTForImageClassification":
        """``ViTForImageClassification.from_pretrained(dir_or_state_dict, num_labels=14, id2label=…, label2id=…,
        ignore_mismatched_sizes=True, problem_type="multi_label_classification")`` as the reference calls it
        (ViT-Training.py:83-90); see checkpoint.load_pretrained.  ``output_loading_info=True`` also returns the key report."""
        from .checkpoint import load_pretrained
        want_info = kwargs.pop("output_loading_info", False)
        model, info = load_pretrained(cls, source, **kwargs)
        return (model, info) if want_info else model

    def save_pretrained(self, save_directory: str, safe_serialization: bool = True) -> None:
        from .checkpoint import save_pretrained
        save_pretrained(self, save_directory, safe_serialization)

    # ------------------------------------------------------------------ parameters
    def _register(self, name: str, p: nn.Parameter) -> None:
        mod = self
        parts = name.split(".")
        for part in parts[:-1]:
            if not hasattr(mod, part):
                mod.add_module(part, nn.ModuleList() if part == "layer" else _Holder())
            mod = getattr(mod, part)
        mod.register_parameter(parts[-1], p)
        self._pnames.append(name)

    def reset_parameters(self, generator: Optional[torch.Generator] = None) -> None:
        """HF ViTPreTrainedModel._init_weights (modeling_vit.py:385-398): trunc_normal(std) for
        Linear/Conv weights, position embeddings and CLS; zero biases; unit LayerNorm."""
        std = self.config.initializer_range
        with torch.no_grad():
            for name, p in self.named_parameters():
                if "layernorm" in name and name.endswith("weight"):
                    p.fill_(1.0)
                elif name.endswith("bias"):
                    p.zero_()
                else:
                    t = torch.empty(p.shape, dtype=f32)
                    nn.init.trunc_normal_(t, mean=0.0, std=std, a=-2 * std, b=2 * std, generator=generator)
                    p.copy_(t)

    def _apply(self, fn, recurse=True):
        out = super()._apply(fn, recurse)
        self._reflatten()
        return out

    def _reflatten(self) -> None:
        """After .to()/.cuda() every parameter is an independent tensor again: gather them back
        into one flat fp32 buffer (kept as views) and drop device-bound caches."""
        params = dict(self.named_parameters())
        dev = params[self._pnames[0]].device
        flat = torch.zeros(self.layout.total, dtype=f32, device=dev)
        with torch.no_grad():
            for name, p in params.items():
                v = self.layout.view(flat, name)
                v.copy_(p.detach().to(f32))
                p.data = v
                p.grad = None
        self._flat_params = flat
        self._flat_grads = None
        self._stage_grads = None
        self._grads_clean = False
        self._flat_shadow = None
        self._shadow_version = -1
        self._engine = None
        self._plist = None

    def flat_parameters(self) -> torch.Tensor:
        return self._flat_params

    def flat_grads(self) -> torch.Tensor:
        if self._flat_grads is None:
            self._flat_grads = torch.zeros_like(self._flat_params)
            self._grads_clean = True
        return self._flat_grads

    def set_flat_grads(self, buf: torch.Tensor) -> None:
        """Adopt ``buf`` (fp32, ``layout.total`` elements, on the model's device) as the flat gradient buffer — e.g. a
        symmetric-memory allocation other GPUs can read (parallel.PeerGradSync).  Launch plans are rebuilt."""
        if buf.dtype != f32 or buf.numel() != self.layout.total or buf.device != self._flat_params.device or not buf.is_contiguous():
            raise ValueError("set_flat_grads: need a contiguous fp32 tensor of layout.total elements on the model's device")
        buf.zero_()
        for p in self.param_list():
            p.grad = None
        self._flat_grads = buf
        self._grads_clean = True
        self._engine = None

    def stage_grads(self) -> torch.Tensor:
        """Second flat gradient buffer: a backward that finds ``param.grad`` already populated (gradient
        accumulation) writes here and autograd adds it onto ``param.grad``."""
        if self._stage_grads is None:
            self._stage_grads = torch.zeros_like(self._flat_params)
        return self._stage_grads

    def param_list(self) -> List[nn.Parameter]:
        if self._plist is None:
            self._plist = [self.get_parameter(n) for n in self.layout.names]
        return self._plist

    def shadow(self) -> torch.Tensor:
        """bf16 copy of the GEMM weights, refreshed whenever the fp32 masters changed."""
        flat = self._flat_params
        if self._flat_shadow is None:
            self._flat_shadow = torch.empty(self.layout.gemm_end, dtype=torch.bfloat16, device=flat.device)
            self._shadow_version = -1
        key = self._param_version()
        if self._shadow_version != key:
            ops.cast_f32_bf16(flat[: self.layout.gemm_end], self._flat_shadow)
            self._shadow_version = key
        return self._flat_shadow

    def _param_version(self) -> int:
        # in-place updates (optimizer.step, load_state_dict, init) bump each parameter's counter; writes through the
        # flat buffer itself (broadcast_parameters, flat.copy_()) bump the buffer's
        return sum(p._version for p in self.param_list()) + self._flat_params._version

    def mark_shadow_fresh(self) -> None:
        """Called by VitkAdamW, whose kernel rewrites the shadow together with the masters."""
        self._shadow_version = self._param_version()

    def invalidate_shadow(self) -> None:
        """Force the bf16 GEMM weights to be re-derived from the fp32 masters at the next forward.  Call it after
        writing to parameter memory by a route PyTorch's version counters do not see (raw pointers, NCCL on an alias)."""
        self._shadow_version = -1

    def engine(self) -> Engine:
        if self._engine is None:
            if self._flat_params.device.type != "cuda":
                raise RuntimeError("chest_x_ray_vit_b200 runs on CUDA (sm_100a) only: move the model with .cuda() first "
                                   "— there is no CPU path")
            ops.check_device(self._flat_params.device.index or 0)
            self._engine = Engine(self)
        return self._engine

    # ------------------------------------------------------------------ forward
    def _check_inputs(self, pixel_values: torch.Tensor, interpolate_pos_encoding: bool = False) -> None:
        cfg = self.config
        if pixel_values.dtype == torch.uint8:
            if pixel_values.dim() == 4 and pixel_values.shape[1] == 1:
                pass
            elif pixel_values.dim() != 3:
                raise ValueError("uint8 pixel_values must be grayscale [B,H,W] or [B,1,H,W]")
            h, w = pixel_values.shape[-2:]
        else:
            if pixel_values.dim() != 4:
                raise ValueError("pixel_values must be [batch, channels, height, width]")
            if pixel_values.shape[1] != cfg.num_channels:
                raise ValueError(
                    "Make sure that the channel dimension of the pixel values match with the one set in the configuration."
                    f" Expected {cfg.num_channels} but got {pixel_values.shape[1]}.")       # HF:155-160
            h, w = pixel_values.shape[-2:]
        if interpolate_pos_encoding:
            # HF floors H and W to whole patches (HF:166, 81-82) and drops the remainder pixels; this path does not
            if h % cfg.patch_size or w % cfg.patch_size or h < cfg.patch_size or w < cfg.patch_size:
                raise ValueError(f"interpolate_pos_encoding=True needs a height and width that are positive multiples of "
                                 f"{cfg.patch_size}, got {h}*{w}: crop or pad the image to whole patches")
        elif h != cfg.image_size or w != cfg.image_size:
            raise ValueError(f"Input image size ({h}*{w}) doesn't match model ({cfg.image_size}*{cfg.image_size}).")  # HF:161-165

    def forward(self, pixel_values: Optional[torch.Tensor] = None, labels: Optional[torch.Tensor] = None,
                interpolate_pos_encoding: Optional[bool] = None, output_attentions: Optional[bool] = None,
                output_hidden_states: Optional[bool] = None, **kwargs) -> ImageClassifierOutput:
        """HF ViTForImageClassification.forward (modeling_vit.py:620-653).  ``pixel_values``:
        fp32 [B,3,H,W] (the collate_fn contract) or uint8 grayscale [B,H,W] (normalised on the
        GPU with config.image_mean/std).  Unknown kwargs (``num_items_in_batch``) are ignored.

        ``output_hidden_states`` (default ``config.output_hidden_states``): ``hidden_states`` is a tuple of L+1 fp32
        [B,T,D] tensors — the embeddings output, then the output of each encoder layer; the last one is taken before
        the final LayerNorm, as in HF.  ``output_attentions`` (default ``config.output_attentions``): ``attentions`` is
        a tuple of L fp32 [B,H,T,T] softmax probabilities per layer, what HF's ``eager`` attention returns (HF's default
        ``sdpa`` attention returns an empty tuple there).  Both are fresh tensors outside autograd
        (``requires_grad=False``): ``loss.backward()`` gives the same gradients as without them, and no gradient flows
        through them.  Requesting either runs the top encoder layer on every token instead of the CLS rows alone.

        Gradients reach a floating-point ``pixel_values`` that requires grad, as in HF: ``x.grad`` is the gradient with
        respect to ``pixel_values`` as passed (for the collate_fn contract, the normalised image), in its dtype and on its
        device — saliency maps, SmoothGrad, Integrated Gradients.  With every parameter frozen
        (``model.requires_grad_(False)``) backward computes only that gradient: no weight gradients, no ``param.grad``,
        no data-parallel gradient sync.  uint8 input cannot require grad (torch forbids it).

        ``interpolate_pos_encoding=True`` (HF modeling_vit.py:60-99) accepts any H×W that is a multiple of 16 on both
        sides, for every input kind above, in train() and eval(), with labels, hidden states, attention maps and an input
        gradient.  The H/16 × W/16 patch grid gets position embeddings resized bicubically from the checkpoint's grid
        (``vitk_pos_interp``), and training sends their gradient back through the resize into ``position_embeddings``,
        which keeps its checkpoint shape.  As in HF, a square input of the config's size is not resized: it runs exactly
        the plain call.  Unlike HF, which floors H and W to whole patches, a size that is not a multiple of 16 is rejected.
        Each grid gets its own activation buffers and launch plans (built on the first call at that size); T = H·W/256 + 1
        above 4096 runs the top encoder layer on every token.  Hidden states are [B,T,D], attention maps [B,H,T,T] and
        ``x.grad`` has the input's shape.  The CUDA-graph wrappers of ``graph.py`` stay at the config size."""
        if pixel_values is None:
            raise ValueError("You have to specify pixel_values")                               # HF:440-441
        cfg = self.config
        want_attn = bool(cfg.output_attentions if output_attentions is None else output_attentions)
        want_hidden = bool(cfg.output_hidden_states if output_hidden_states is None else output_hidden_states)
        self._check_inputs(pixel_values, bool(interpolate_pos_encoding))
        if interpolate_pos_encoding and self._flat_params.device.type != "cuda":
            raise ValueError("interpolate_pos_encoding=True runs on the CUDA kernel path only: move the model with .cuda() "
                             "first — there is no CPU path")
        eng = self.engine()
        if labels is not None and cfg.problem_type is None:
            cfg.problem_type = "multi_label_classification"     # HF loss_utils.py:92-98 (float labels)
        need_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in self.param_list()) or
                                                 (pixel_values.is_floating_point() and pixel_values.requires_grad))
        extras = {"attentions": want_attn, "hidden_states": want_hidden}
        if need_grad:
            loss, logits = _VitFunction.apply(self, pixel_values, labels, extras, *self.param_list())
            hidden, attn = extras["out"]
        else:
            loss, logits, hidden, attn = eng.forward(pixel_values, labels, save=False, output_attentions=want_attn,
                                                     output_hidden_states=want_hidden)
        return ImageClassifierOutput(loss=loss if labels is not None else None, logits=logits, hidden_states=hidden,
                                     attentions=attn)


class _VitFunction(torch.autograd.Function):
    """One autograd node for the whole model.  Every parameter is an input of the node, so the usual autograd
    contract holds: backward RETURNS one gradient per parameter that requires grad and the engine's AccumulateGrad
    nodes populate ``param.grad`` — hooks, ``torch.autograd.grad``, frozen parameters and DistributedDataParallel's
    reducer all see what they expect.  The returned gradients are views of one flat fp32 buffer the kernels wrote:
    when ``param.grad`` is None autograd adopts the view without a copy, so the optimizer still finds all gradients
    contiguous; when ``param.grad`` is already populated (gradient accumulation) the kernels write a second buffer
    and autograd adds it in place.  ``pixel_values`` gets its gradient when it requires one (a fresh tensor: the
    engine's input-gradient GEMM allocates it).  Requested hidden states / attention maps leave through
    ``extras["out"]``, outside autograd."""

    @staticmethod
    def forward(ctx, model: ViTForImageClassification, pixel_values, labels, extras, *params):
        eng = model.engine()
        loss, logits, hidden, attn = eng.forward(pixel_values, labels, save=True, output_attentions=extras["attentions"],
                                                 output_hidden_states=extras["hidden_states"])
        extras["out"] = (hidden, attn)
        ctx.model = model
        ctx.ticket = eng.ticket
        ctx.has_labels = labels is not None
        ctx.x_dtype, ctx.x_device = pixel_values.dtype, pixel_values.device
        ctx.set_materialize_grads(False)
        if loss is None:
            loss = logits.new_zeros(())
        return loss, logits

    @staticmethod
    def backward(ctx, dloss, dlogits):
        model = ctx.model
        grads, dx = model.engine().backward(ctx.ticket, dloss if ctx.has_labels else None, dlogits, ctx.needs_input_grad[4:],
                                            input_grad=ctx.needs_input_grad[1])
        if dx is not None and (dx.dtype != ctx.x_dtype or dx.device != ctx.x_device):
            dx = dx.to(device=ctx.x_device, dtype=ctx.x_dtype)
        return (None, dx, None, None) + grads
