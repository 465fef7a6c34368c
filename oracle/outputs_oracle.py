"""CPU oracle of the forward's optional outputs (``output_hidden_states`` / ``output_attentions``).  TEST INFRASTRUCTURE
ONLY.  Built from the building blocks of ``vit_oracle`` and computing the same arithmetic as ``vit_oracle.forward``
(its logits are bit-identical), it also returns what HF 5.5.0's ``ViTForImageClassification`` returns under
``attn_implementation="eager"``; ``tests/test_oracle_outputs.py`` pins it against live HF."""
from __future__ import annotations

from typing import Dict

import torch

from .vit_oracle import OracleConfig, bce_with_logits_mean, embeddings, gelu_erf, layer_norm


def attention_probs(q, k, scale):
    """The attention weights eager_attention_forward returns (HF:185-190): softmax(QKᵀ·scale), no mask — the
    probabilities ``vit_oracle.attention`` multiplies V by."""
    s = (q @ k.transpose(-1, -2)) * scale
    return torch.softmax(s, dim=-1)


def forward_outputs(p: Dict[str, torch.Tensor], cfg: OracleConfig, pixel_values: torch.Tensor, labels=None):
    """ViTForImageClassification.forward with ``output_hidden_states=True, output_attentions=True`` under HF's eager
    attention → (loss | None, logits, hidden_states, attentions).
    hidden_states: L+1 tensors [B,T,D] — the embeddings output, then each encoder layer's output, the last one taken
    before the final LayerNorm (HF:426, capture_outputs(tie_last_hidden_states=False)); attentions: L tensors
    [B,H,T,T] of softmax probabilities (HF:185-190)."""
    H = cfg.num_attention_heads
    h = embeddings(p, cfg, pixel_values)
    hidden, attentions = [h], []
    for i in range(cfg.num_hidden_layers):                   # vit_oracle.encoder_layer (HF:328-346), keeping the weights
        pre = f"vit.encoder.layer.{i}."
        B, T, D = h.shape
        dh = D // H
        n1 = layer_norm(h, p[pre + "layernorm_before.weight"], p[pre + "layernorm_before.bias"], cfg.layer_norm_eps)

        def lin(x, name):
            return x @ p[pre + name + ".weight"].t() + p[pre + name + ".bias"]
        q = lin(n1, "attention.attention.query").view(B, T, H, dh).transpose(1, 2)
        k = lin(n1, "attention.attention.key").view(B, T, H, dh).transpose(1, 2)
        v = lin(n1, "attention.attention.value").view(B, T, H, dh).transpose(1, 2)
        pr = attention_probs(q, k, dh ** -0.5)
        attentions.append(pr)
        o = (pr @ v).transpose(1, 2).reshape(B, T, D)
        h1 = lin(o, "attention.output.dense") + h
        n2 = layer_norm(h1, p[pre + "layernorm_after.weight"], p[pre + "layernorm_after.bias"], cfg.layer_norm_eps)
        h = lin(gelu_erf(lin(n2, "intermediate.dense")), "output.dense") + h1
        hidden.append(h)
    z = layer_norm(h, p["vit.layernorm.weight"], p["vit.layernorm.bias"], cfg.layer_norm_eps)[:, 0, :]
    logits = z @ p["classifier.weight"].t() + p["classifier.bias"]
    loss = bce_with_logits_mean(logits, labels) if labels is not None else None
    return loss, logits, tuple(hidden), tuple(attentions)
