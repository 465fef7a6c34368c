"""CPU-only: the oracle's hidden states and attention maps against live HF eager attention, and the module's host logic
for ``output_attentions`` / ``output_hidden_states``."""
import pytest
import torch

import chest_x_ray_vit_b200 as pkg
from oracle import outputs_oracle as OO
from oracle import vit_oracle as O

TINY = dict(image_size=64, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256, num_labels=14)


def _inputs(cfg, batch=2, seed=5):
    g = torch.Generator().manual_seed(seed)
    x8, y = O.synth_inputs(cfg, batch, g)
    return O.normalize_gray(x8), y


def test_forward_outputs_matches_live_hf_eager():
    pytest.importorskip("transformers")
    from oracle.make_golden import hf_model
    cfg = O.TINY
    p = O.init_params(cfg, 3, 7)
    x, y = _inputs(cfg)
    m, _ = hf_model(cfg, p)
    m.set_attn_implementation("eager")
    with torch.no_grad():
        ref = m(pixel_values=x, labels=y, output_attentions=True, output_hidden_states=True)
        loss, logits, hs, attn = OO.forward_outputs(p, cfg, x, y)
    L, B, T, D, H = cfg.num_hidden_layers, 2, cfg.seq_len, cfg.hidden_size, cfg.num_attention_heads
    assert len(hs) == len(ref.hidden_states) == L + 1 and len(attn) == len(ref.attentions) == L
    for a, r in zip(hs, ref.hidden_states):
        assert a.shape == r.shape == (B, T, D) and a.dtype == torch.float32
        assert (a - r).abs().max() <= 1e-5 * max(1.0, r.abs().max().item())
    for a, r in zip(attn, ref.attentions):
        assert a.shape == r.shape == (B, H, T, T) and a.dtype == torch.float32
        assert (a - r).abs().max() <= 1e-6
    assert (logits - ref.logits).abs().max() <= 2e-5 and abs(loss.item() - ref.loss.item()) <= 1e-6
    # the last hidden state is the encoder output BEFORE the final LayerNorm
    normed = O.layer_norm(hs[-1], p["vit.layernorm.weight"], p["vit.layernorm.bias"], cfg.layer_norm_eps)
    assert (normed - ref.hidden_states[-1]).abs().max() > 1e-2


def test_forward_outputs_logits_equal_forward():
    cfg = O.TINY
    p = O.init_params(cfg, 0, 123)
    x, y = _inputs(cfg, 3, 1)
    with torch.no_grad():
        loss0, logits0 = O.forward(p, cfg, x, y)
        loss, logits, hs, attn = OO.forward_outputs(p, cfg, x, y)
    assert torch.equal(logits, logits0) and torch.equal(loss, loss0)
    for a in attn:                                     # rows are probability distributions
        assert torch.allclose(a.sum(-1), torch.ones(()), atol=1e-5)


def test_from_hf_copies_output_flags():
    tr = pytest.importorskip("transformers")
    hc = tr.ViTConfig(**TINY, output_attentions=True, output_hidden_states=True)
    c = pkg.ViTConfig.from_hf(hc)
    assert c.output_attentions is True and c.output_hidden_states is True
    c = pkg.ViTConfig.from_hf(tr.ViTConfig(**TINY))
    assert c.output_attentions is False and c.output_hidden_states is False
    assert pkg.ViTConfig().output_attentions is False and pkg.ViTConfig().output_hidden_states is False


def test_keyword_overrides_config_and_cpu_model_has_no_path(monkeypatch):
    m = pkg.ViTForImageClassification(pkg.ViTConfig(**TINY, output_attentions=True, output_hidden_states=True))
    seen = {}

    class FakeEngine:
        def forward(self, pixel_values, labels, save, output_attentions=False, output_hidden_states=False):
            seen.update(attentions=output_attentions, hidden_states=output_hidden_states, save=save)
            return None, torch.zeros(pixel_values.shape[0], 14), None, None

    monkeypatch.setattr(m, "engine", lambda: FakeEngine())
    x = torch.zeros(1, 3, 64, 64)
    with torch.no_grad():
        m(pixel_values=x)
        assert seen == dict(attentions=True, hidden_states=True, save=False)
        m(pixel_values=x, output_attentions=False, output_hidden_states=False)
        assert seen == dict(attentions=False, hidden_states=False, save=False)
        m(pixel_values=x, output_attentions=False)
        assert seen == dict(attentions=False, hidden_states=True, save=False)
    monkeypatch.undo()
    with pytest.raises(RuntimeError, match="no CPU path"):
        m(pixel_values=x, output_attentions=True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        pkg.ViTForImageClassification(pkg.ViTConfig(**TINY))(pixel_values=x, output_hidden_states=True)
