"""The oracle (oracle/vit_oracle.py) against the frozen HF golden vectors and, when
transformers is importable, against the live HF model.  CPU only."""
import os

import pytest
import torch

from oracle import vit_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _cfg(rec):
    return O.OracleConfig(**rec["cfg"])


def test_param_inventory_matches_survey():
    shapes = O.param_shapes(O.VIT_B16_384)
    assert len(shapes) == 200
    n = sum(torch.Size(s).numel() for s in shapes.values())
    assert n == 86_101_262
    assert sum(torch.Size(s).numel() for s in O.param_shapes(O.VIT_L16_384).values()) == 303_705_102
    assert sum(torch.Size(s).numel() for s in O.param_shapes(O.VIT_B16_224).values()) == 85_809_422


def test_tiny_full_gradients_match_hf_golden():
    rec = torch.load(os.path.join(GOLD, "tiny_b3.pt"), weights_only=False)
    cfg = _cfg(rec)
    p = O.init_params(cfg, 0, 123)
    x = O.normalize_gray(rec["x8"])
    loss, logits, grads = O.forward_backward(p, cfg, x, rec["y"])
    assert torch.allclose(logits, rec["logits"], atol=2e-5, rtol=0)
    assert abs(loss.item() - rec["loss"].item()) <= 1e-6 * abs(rec["loss"].item()) + 1e-7
    from oracle.make_golden import record_indices
    for k, g in rec["grad_sample"].items():
        if k.endswith("key.bias"):        # analytically zero (SURVEY App. C.6)
            assert grads[k].norm() < 1e-6
            continue
        nrm = rec["grad_norm"][k]
        assert abs(grads[k].norm().item() - nrm) <= 1e-3 * nrm + 2e-6, k
        assert torch.allclose(grads[k].flatten()[record_indices(rec, k, grads[k].numel())], g, atol=2e-6, rtol=1e-3), k
    st = {}
    O.adamw_step(p, grads, st)
    for k, v in rec["post_sample"].items():
        if k.endswith("key.bias"):
            continue   # Adam normalises rounding noise of a zero gradient
        assert torch.allclose(p[k].flatten()[record_indices(rec, k, p[k].numel())], v, atol=2e-5 * 1.01, rtol=0), k


def test_vitb16_384_matches_hf_golden():
    """BASELINE.json configs[0]: ViT-B/16@384, batch 2, one fwd+bwd on CPU fp32."""
    rec = torch.load(os.path.join(GOLD, "vitb16_384_b2.pt"), weights_only=False)
    cfg = _cfg(rec)
    p = O.init_params(cfg, 0, 123)
    x = O.normalize_gray(rec["x8"])
    loss, logits, grads = O.forward_backward(p, cfg, x, rec["y"])
    assert (logits - rec["logits"]).abs().max() < 1e-4
    assert abs(loss.item() - rec["loss"].item()) < 1e-5 * abs(rec["loss"].item())
    from oracle.make_golden import sample_indices
    for k, nrm in rec["grad_norm"].items():
        if k.endswith("key.bias"):
            assert grads[k].norm() < 1e-6
            continue
        assert abs(grads[k].norm().item() - nrm) <= 2e-3 * nrm + 1e-9, k
        s = grads[k].flatten()[sample_indices(k, grads[k].numel())]
        assert torch.allclose(s, rec["grad_sample"][k], atol=1e-3 * nrm / max(1.0, grads[k].numel() ** 0.5) + 1e-8, rtol=2e-2), k


def test_vitb16_224_logits_match_hf_golden():
    rec = torch.load(os.path.join(GOLD, "vitb16_224_b2.pt"), weights_only=False)
    cfg = _cfg(rec)
    p = O.init_params(cfg, 0, 123)
    with torch.no_grad():
        loss, logits = O.forward(p, cfg, O.normalize_gray(rec["x8"]), rec["y"])
    assert (logits - rec["logits"]).abs().max() < 1e-4
    assert abs(loss.item() - rec["loss"].item()) < 1e-5


def test_live_hf_agrees_on_tiny():
    tr = pytest.importorskip("transformers")
    from oracle.make_golden import hf_model
    cfg = O.TINY
    p = O.init_params(cfg, 3, 7)
    g = torch.Generator().manual_seed(5)
    x8, y = O.synth_inputs(cfg, 2, g)
    x = O.normalize_gray(x8)
    m, _ = hf_model(cfg, p)
    out = m(pixel_values=x, labels=y)
    loss, logits = O.forward(p, cfg, x, y)
    assert torch.allclose(out.logits, logits, atol=2e-5)
    assert abs(out.loss.item() - loss.item()) < 1e-6


def test_normalize_gray_is_totensor_normalize():
    x8 = torch.arange(0, 256, dtype=torch.uint8).view(1, 1, 16, 16)
    x = O.normalize_gray(x8, mean=(0.485, 0.456, 0.406), std=(0.229, 0.224, 0.225))
    assert x.shape == (1, 3, 16, 16)
    assert torch.allclose(x[0, 1, 0, 3], torch.tensor((3 / 255 - 0.456) / 0.224))


def test_im2col_matches_conv2d():
    torch.manual_seed(0)
    x = torch.randn(2, 3, 32, 32)
    w = torch.randn(8, 3, 16, 16)
    ref = torch.nn.functional.conv2d(x, w, stride=16).flatten(2).transpose(1, 2)
    got = O.im2col(x, 16) @ w.reshape(8, -1).t()
    assert torch.allclose(ref, got, atol=1e-3)
