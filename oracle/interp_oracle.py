"""Oracle for ``interpolate_pos_encoding`` (inputs of another size than the checkpoint's).  TEST INFRASTRUCTURE ONLY.

Two parts:
  * the model with ``interpolate_pos_encoding`` in fp32, as HF computes it (``resize_pos`` uses ``F.interpolate`` exactly
    as HF:60-99 does; ``embeddings`` / ``forward`` / ``forward_backward`` are oracle/vit_oracle.py's with that table in
    place of the parameter, everything else reused from there);
  * an fp64 restatement of the resize as dense matrices, below.

HF (modeling_vit.py:60-99) resizes the s×s grid of position embeddings with ``F.interpolate(mode="bicubic",
align_corners=False)`` to the input's gh×gw patch grid.  That map is separable: per channel, out = Wy · X · Wxᵀ with
dense 1-D matrices Wy [gh, s] and Wx [gw, s].  Row o of a matrix holds torch's cubic-convolution weights (A = −0.75) of
output index o: source coordinate (o + 0.5)·n_in/n_out − 0.5 (not clamped), taps floor − 1 … floor + 2, each tap clamped
to [0, n_in − 1] with the weights of coinciding taps added (ATen UpSample.h: area_pixel_compute_source_index,
upsample_get_cubic_coefficients, upsample_get_value_bounded).  The adjoint is Wyᵀ · G · Wx.

tests/test_oracle_interp.py pins these matrices against F.interpolate in fp64; tests/test_gpu_interp.py checks
vitk_pos_interp / vitk_pos_interp_bwd against them.
"""
from __future__ import annotations

import math
from typing import Dict

import torch
import torch.nn.functional as F

from .vit_oracle import OracleConfig, bce_with_logits_mean, encoder_layer, im2col, layer_norm

A = -0.75


# --------------------------------------------------------------------------- the model with the flag (fp32, as HF)
def resize_pos(pos: torch.Tensor, height: int, width: int, patch: int) -> torch.Tensor:
    """ViTEmbeddings.interpolate_pos_encoding (HF:60-99): the [1, 1+s², D] table at the (height/p) × (width/p) grid —
    unchanged when that grid has the table's patch count and height == width, else row 0 kept and rows 1.. resized by
    F.interpolate(mode="bicubic", align_corners=False)."""
    num_positions = pos.shape[1] - 1
    gh, gw = height // patch, width // patch
    if gh * gw == num_positions and height == width:
        return pos
    s, dim = int(num_positions ** 0.5), pos.shape[-1]
    grid = pos[:, 1:].reshape(1, s, s, dim).permute(0, 3, 1, 2)
    grid = F.interpolate(grid, size=(gh, gw), mode="bicubic", align_corners=False)
    return torch.cat((pos[:, :1], grid.permute(0, 2, 3, 1).reshape(1, -1, dim)), dim=1)


def embeddings(p, cfg: OracleConfig, pixel_values: torch.Tensor, interpolate_pos_encoding: bool = False) -> torch.Tensor:
    """vit_oracle.embeddings (HF:100-128, :153-167) with the position table resized to the input's patch grid when
    ``interpolate_pos_encoding`` is set (HF:124-125)."""
    w = p["vit.embeddings.patch_embeddings.projection.weight"].reshape(cfg.hidden_size, -1)
    b = p["vit.embeddings.patch_embeddings.projection.bias"]
    e = im2col(pixel_values, cfg.patch_size) @ w.t() + b
    cls = p["vit.embeddings.cls_token"].expand(pixel_values.shape[0], -1, -1)
    pos = p["vit.embeddings.position_embeddings"]
    if interpolate_pos_encoding:
        pos = resize_pos(pos, pixel_values.shape[2], pixel_values.shape[3], cfg.patch_size)
    return torch.cat((cls, e), dim=1) + pos


def forward(p: Dict[str, torch.Tensor], cfg: OracleConfig, pixel_values: torch.Tensor, labels=None,
            interpolate_pos_encoding: bool = False):
    """ViTForImageClassification.forward (HF:620-653) with ``interpolate_pos_encoding`` → (loss | None, logits)."""
    h = embeddings(p, cfg, pixel_values, interpolate_pos_encoding)
    for i in range(cfg.num_hidden_layers):
        h = encoder_layer(p, cfg, i, h)
    z = layer_norm(h, p["vit.layernorm.weight"], p["vit.layernorm.bias"], cfg.layer_norm_eps)[:, 0, :]
    logits = z @ p["classifier.weight"].t() + p["classifier.bias"]
    loss = bce_with_logits_mean(logits, labels) if labels is not None else None
    return loss, logits


def forward_backward(p: Dict[str, torch.Tensor], cfg: OracleConfig, pixel_values, labels, interpolate_pos_encoding: bool = False):
    """One fwd+bwd in fp32; returns (loss, logits, {name: grad}); ``position_embeddings`` keeps its checkpoint shape."""
    leaves = {k: v.detach().clone().requires_grad_(True) for k, v in p.items()}
    loss, logits = forward(leaves, cfg, pixel_values, labels, interpolate_pos_encoding)
    loss.backward()
    return loss.detach(), logits.detach(), {k: v.grad for k, v in leaves.items()}


# --------------------------------------------------------------------------- fp64 matrices of the resize


def _cc1(x: float) -> float:       # |x| <= 1
    return ((A + 2) * x - (A + 3)) * x * x + 1


def _cc2(x: float) -> float:       # 1 < |x| < 2
    return ((A * x - 5 * A) * x + 8 * A) * x - 4 * A


def bicubic_matrix(n_in: int, n_out: int) -> torch.Tensor:
    """fp64 [n_out, n_in]: row o maps the n_in samples to output sample o."""
    W = torch.zeros(n_out, n_in, dtype=torch.float64)
    for o in range(n_out):
        src = (o + 0.5) * n_in / n_out - 0.5
        f = math.floor(src)
        t = src - f
        w = (_cc2(t + 1), _cc1(t), _cc1(1 - t), _cc2(2 - t))
        for k in range(4):
            W[o, min(max(f - 1 + k, 0), n_in - 1)] += w[k]
    return W


def pos_interp(pos: torch.Tensor, gh0: int, gw0: int, gh: int, gw: int) -> torch.Tensor:
    """[1 + gh0·gw0, D] → fp64 [1 + gh·gw, D]: row 0 copied, rows 1.. = Wy · grid · Wxᵀ per channel."""
    pos = pos.double()
    D = pos.shape[-1]
    grid = pos[1:].reshape(gh0, gw0, D)
    Wy, Wx = bicubic_matrix(gh0, gh), bicubic_matrix(gw0, gw)
    out = torch.einsum("yi,ijd,xj->yxd", Wy, grid, Wx).reshape(gh * gw, D)
    return torch.cat((pos[:1], out), dim=0)


def pos_interp_bwd(dout: torch.Tensor, gh: int, gw: int, gh0: int, gw0: int) -> torch.Tensor:
    """Adjoint of pos_interp: fp64 [1 + gh·gw, D] → [1 + gh0·gw0, D], row 0 passed through, rows 1.. = Wyᵀ · G · Wx."""
    dout = dout.double()
    D = dout.shape[-1]
    g = dout[1:].reshape(gh, gw, D)
    Wy, Wx = bicubic_matrix(gh0, gh), bicubic_matrix(gw0, gw)
    back = torch.einsum("yi,yxd,xj->ijd", Wy, g, Wx).reshape(gh0 * gw0, D)
    return torch.cat((dout[:1], back), dim=0)
