"""Attention maps and hidden states (``output_attentions`` / ``output_hidden_states``): the vitk_attn_probs kernel against
fp32 softmax, the module against live HF eager attention and the oracle, and the behaviour around the default path."""
import os

import pytest
import torch

from oracle import outputs_oracle as OO
from oracle import vit_oracle as O

pytestmark = pytest.mark.gpu
dev = "cuda"
bf16 = torch.bfloat16
SCALE = 0.125
HS_TOL, HS_COS = 2e-2, 0.9999          # hidden states: max-abs ≤ HS_TOL·max|ref|, cosine per tensor
AT_TOL, AT_COS = 1e-2, 0.999           # attention maps: max-abs, cosine per tensor


@pytest.fixture(scope="module")
def ops():
    import chest_x_ray_vit_b200 as pkg
    pkg.ops.check_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    return pkg.ops


def _ref_probs(qkv, scale):
    x = qkv.float()
    q, k = x[:, :, 0].transpose(1, 2), x[:, :, 1].transpose(1, 2)       # [B,H,T,64]
    return torch.softmax((q @ k.transpose(-1, -2)) * scale, dim=-1)


def _probs_guarded(ops, qkv, lse, B, T, H, scale):
    """Runs the kernel into the front of a NaN-filled buffer and checks that the tail stays NaN."""
    n = B * H * T * T
    buf = torch.full((n + 8192,), float("nan"), device=dev)
    p = ops.attn_probs(qkv, lse, B, T, H, scale, out=buf[:n].view(B, H, T, T))
    torch.cuda.synchronize()
    assert torch.isnan(buf[n:]).all(), "attn_probs wrote past its [B, H, T, T] output"
    return p


def _check_rows(p):
    assert torch.isfinite(p).all() and p.min() >= 0 and p.max() <= 1
    assert (p.sum(-1) - 1).abs().max() <= 1e-3


# shapes like test_gpu_attention.py's: T from 17 to 1024, H up to 20, and the benchmarked B = 16 at T = 577
@pytest.mark.parametrize("B,T,H", [(1, 128, 1), (1, 64, 2), (2, 17, 2), (2, 129, 3), (2, 197, 12), (1, 256, 2), (2, 577, 12),
                                   (1, 300, 16), (1, 385, 2), (1, 640, 2), (1, 1024, 1), (16, 577, 12),
                                   (1, 130, 6), (1, 70, 20), (2, 129, 20)])
def test_attn_probs_matches_fp32_softmax(ops, B, T, H):
    g = torch.Generator().manual_seed(T * 10 + H)
    qkv = torch.randn(B, T, 3, H, 64, generator=g).to(dev).to(bf16)
    o, lse = ops.attn_fwd(qkv, B, T, H, SCALE)
    p = _probs_guarded(ops, qkv, lse, B, T, H, SCALE)
    ref = _ref_probs(qkv, SCALE)
    err = (p - ref).abs().max().item()
    assert err <= 2e-3, f"max-abs {err}"
    _check_rows(p)
    v = qkv[:, :, 2].float().transpose(1, 2)                              # [B,H,T,64]
    pv = (p @ v).transpose(1, 2).reshape(B, T, H * 64)
    of = o.view(B, T, H * 64).float()
    assert (pv - of).abs().max() <= 2e-2 * of.abs().max()


def test_attn_probs_large_logits(ops):
    B, T, H = 1, 577, 2
    g = torch.Generator().manual_seed(0)
    qkv = (torch.randn(B, T, 3, H, 64, generator=g) * 4).to(dev).to(bf16)
    _, lse = ops.attn_fwd(qkv, B, T, H, SCALE)
    _check_rows(_probs_guarded(ops, qkv, lse, B, T, H, SCALE))


def test_attn_probs_reference_maximum_jumps(ops):
    B, T, H = 1, 577, 1
    g = torch.Generator().manual_seed(4)
    qkv = torch.randn(B, T, 3, H, 64, generator=g)
    qkv[:, :, 0] *= 3.0
    qkv[:, 200:, 1] *= 6.0
    qkv[:, 400:, 1] *= 8.0
    qkv = qkv.to(dev).to(bf16)
    _, lse = ops.attn_fwd(qkv, B, T, H, SCALE)
    _check_rows(_probs_guarded(ops, qkv, lse, B, T, H, SCALE))


def test_attn_probs_rejects_bad_arguments(ops):
    import chest_x_ray_vit_b200 as pkg
    B, T, H = 1, 64, 2
    qkv = torch.randn(B, T, 3, H, 64, device=dev).to(bf16)
    _, lse = ops.attn_fwd(qkv, B, T, H, SCALE)
    out = torch.empty(B, H, T, T, device=dev)
    L = pkg._lib.lib()
    s = torch.cuda.current_stream().cuda_stream
    assert L.vitk_attn_probs(None, lse.data_ptr(), B, T, H, SCALE, out.data_ptr(), s) != 0
    assert L.vitk_attn_probs(qkv.data_ptr(), None, B, T, H, SCALE, out.data_ptr(), s) != 0
    assert L.vitk_attn_probs(qkv.data_ptr(), lse.data_ptr(), B, T, H, SCALE, None, s) != 0
    with pytest.raises(RuntimeError, match="NULL"):                        # an empty tensor has no storage
        ops.attn_probs(torch.empty(0, dtype=bf16, device=dev), torch.empty(0, device=dev), 0, T, H, SCALE,
                       out=torch.empty(0, device=dev))
    raw = torch.empty(qkv.numel() + 8, dtype=bf16, device=dev)
    mis = raw[1:1 + qkv.numel()]                                          # 2-byte offset
    mis.copy_(qkv.flatten())
    with pytest.raises(RuntimeError, match="aligned"):
        ops.attn_probs(mis, lse, B, T, H, SCALE, out=out)
    with pytest.raises(RuntimeError, match="scale"):
        ops.attn_probs(qkv, lse, B, T, H, -1.0, out=out)
    with pytest.raises(AssertionError):                                   # shape does not match the tensors
        ops.attn_probs(qkv, lse, B, T + 1, H, SCALE)
    assert L.vitk_attn_probs(qkv.data_ptr(), lse.data_ptr(), B, 0, H, SCALE, out.data_ptr(), s) != 0
    assert b"unsupported shape" in L.vitk_last_error()
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------- model
def _model(cfg: O.OracleConfig, params, train=False):
    from test_gpu_model import _model as make
    m = make(cfg, params)
    return m if train else m.eval()


def _compare(hidden, attn, ref_hidden, ref_attn, what):
    assert len(hidden) == len(ref_hidden) and len(attn) == len(ref_attn)
    worst = [1.0, 0.0, 1.0, 0.0]
    for a, r in zip(hidden, ref_hidden):
        a, r = a.float().cpu(), r.float()
        assert a.shape == r.shape and a.dtype == torch.float32
        err = (a - r).abs().max().item() / r.abs().max().item()
        cos = torch.nn.functional.cosine_similarity(a.flatten().double(), r.flatten().double(), dim=0).item()
        worst[0], worst[1] = min(worst[0], cos), max(worst[1], err)
        assert err <= HS_TOL and cos >= HS_COS, f"{what} hidden state: rel max-abs {err:.3e}, cosine {cos:.6f}"
    for a, r in zip(attn, ref_attn):
        a, r = a.float().cpu(), r.float()
        assert a.shape == r.shape and a.dtype == torch.float32
        err = (a - r).abs().max().item()
        cos = torch.nn.functional.cosine_similarity(a.flatten().double(), r.flatten().double(), dim=0).item()
        worst[2], worst[3] = min(worst[2], cos), max(worst[3], err)
        assert err <= AT_TOL and cos >= AT_COS, f"{what} attention: max-abs {err:.3e}, cosine {cos:.6f}"
    print(f"{what}: hidden states worst cosine {worst[0]:.7f}, rel max-abs {worst[1]:.3e}; "
          f"attentions worst cosine {worst[2]:.7f}, max-abs {worst[3]:.3e}")


@pytest.mark.parametrize("input_kind", ["u8", "f32"])
def test_tiny_matches_live_hf_eager(input_kind):
    pytest.importorskip("transformers")
    from oracle.make_golden import hf_model
    cfg = O.TINY
    params = O.init_params(cfg, 3, 7)
    g = torch.Generator().manual_seed(5)
    x8, y = O.synth_inputs(cfg, 3, g)
    hf, _ = hf_model(cfg, params)
    hf.set_attn_implementation("eager")
    with torch.no_grad():
        ref = hf(pixel_values=O.normalize_gray(x8), labels=y, output_attentions=True, output_hidden_states=True)
    m = _model(cfg, params)
    x = x8[:, 0].cuda() if input_kind == "u8" else O.normalize_gray(x8).cuda()
    with torch.no_grad():
        out = m(pixel_values=x, labels=y.cuda(), output_attentions=True, output_hidden_states=True)
    _compare(out.hidden_states, out.attentions, ref.hidden_states, ref.attentions, f"tiny {input_kind} vs HF eager")
    assert (out.logits.cpu() - ref.logits).abs().max() <= 2e-2


@pytest.mark.parametrize("train", [False, True])
def test_vitb16_384_matches_oracle(train):
    cfg = O.VIT_B16_384
    params = O.init_params(cfg, 0, 123)
    g = torch.Generator().manual_seed(1)
    x8, y = O.synth_inputs(cfg, 2, g)
    m = _model(cfg, params, train=train)
    out = m(pixel_values=x8[:, 0].cuda(), labels=y.cuda(), output_attentions=True, output_hidden_states=True)
    if train:
        assert out.loss.requires_grad
        out.loss.backward()
    torch.cuda.synchronize()
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        _, logits, hs, attn = OO.forward_outputs(params, cfg, O.normalize_gray(x8), y)
    _compare(out.hidden_states, out.attentions, hs, attn, f"ViT-B/16@384 b2 {'train' if train else 'eval'} vs oracle")
    assert (out.logits.detach().cpu() - logits).abs().max() <= 2e-2


# ---------------------------------------------------------------------------------------------------- behaviour
@pytest.mark.parametrize("train", [False, True])
def test_flagged_logits_equal_dense_top_mode(monkeypatch, train):
    """With either flag the top layer runs densely: the logits are those of VITK_CLS_ONLY_TOP=0, bit for bit."""
    cfg = O.VIT_B16_224
    params = O.init_params(cfg, 0, 123)
    g = torch.Generator().manual_seed(2)
    x8, y = O.synth_inputs(cfg, 4, g)
    x, y = x8[:, 0].cuda(), y.cuda()
    monkeypatch.delenv("VITK_CLS_ONLY_TOP", raising=False)
    m = _model(cfg, params, train)
    with torch.set_grad_enabled(train):
        plain = m(pixel_values=x, labels=y).logits.detach()
        flagged = m(pixel_values=x, labels=y, output_hidden_states=True).logits.detach()
        flagged_a = m(pixel_values=x, labels=y, output_attentions=True).logits.detach()
    monkeypatch.setenv("VITK_CLS_ONLY_TOP", "0")
    m_dense = _model(cfg, params, train)
    with torch.set_grad_enabled(train):
        dense = m_dense(pixel_values=x, labels=y).logits.detach()
    assert not m_dense.engine().cls_only_top and m.engine().cls_only_top
    assert torch.equal(flagged, dense) and torch.equal(flagged_a, dense)
    assert (flagged - plain).abs().max().item() <= 5e-3


def test_plain_forward_unchanged_after_flagged_call():
    import chest_x_ray_vit_b200 as pkg
    cfg = O.VIT_B16_224
    m = _model(cfg, O.init_params(cfg, 0, 123))
    g = torch.Generator().manual_seed(3)
    x = O.synth_inputs(cfg, 4, g)[0][:, 0].cuda()

    def plain():
        with torch.no_grad():
            n0 = pkg.ops.launch_count()
            logits = m(pixel_values=x).logits
            torch.cuda.synchronize()
            return pkg.ops.launch_count() - n0, logits
    plain()                      # first call launches kernel by kernel, the second captures: compare steady states
    plain()
    n_before, l_before = plain()
    with torch.no_grad():
        m(pixel_values=x, output_attentions=True, output_hidden_states=True)
    n_after, l_after = plain()
    assert n_after == n_before and torch.equal(l_after, l_before)


def test_train_gradients_unchanged_by_flags(monkeypatch):
    """The flags change the forward of the top layer only (dense instead of CLS rows alone); backward stays CLS-only.
    The gradients then move by as little as VITK_CLS_ONLY_TOP=0 moves them: both runs differ from the default in how the
    top layer's attention rounds (bf16 P in the dense kernel), which reaches every gradient through the CLS row.  On a
    B200 the worst per-tensor cosine against the plain step is 0.99995 with the flags and 0.99996 in the dense-top mode
    (the patch-embedding weight), while repeating either step gives cosine 1.0000000; hence 0.9999 and not 0.99999."""
    cfg = O.VIT_B16_224
    params = O.init_params(cfg, 0, 123)
    g = torch.Generator().manual_seed(4)
    x8, y = O.synth_inputs(cfg, 2, g)
    x, y = x8[:, 0].cuda(), y.cuda()
    monkeypatch.delenv("VITK_CLS_ONLY_TOP", raising=False)

    def grads(m, **kw):
        m.zero_grad(set_to_none=True)
        out = m(pixel_values=x, labels=y, **kw)
        out.loss.backward()
        return out, {k: p.grad.detach().double().clone() for k, p in m.named_parameters()}
    m = _model(cfg, params, train=True)
    _, ref = grads(m)
    out, got = grads(m, output_attentions=True, output_hidden_states=True)
    assert all(not t.requires_grad for t in out.hidden_states + out.attentions)
    monkeypatch.setenv("VITK_CLS_ONLY_TOP", "0")
    _, dense = grads(_model(cfg, params, train=True))
    assert len(ref) == 200

    def worst(a):
        w = (1.0, None)
        for k in ref:
            if k.endswith("key.bias"):          # analytically zero: the magnitude bound of test_gpu_model.py
                assert a[k].norm() <= 0.05 * ref[k.replace("key.bias", "query.bias")].norm() + 1e-7
                continue
            c = torch.nn.functional.cosine_similarity(a[k].flatten(), ref[k].flatten(), dim=0).item()
            w = min(w, (c, k))
        return w
    w_flags, w_dense = worst(got), worst(dense)
    print(f"gradients vs the plain step: worst cosine {w_flags[0]:.7f} ({w_flags[1]}) with the flags, "
          f"{w_dense[0]:.7f} ({w_dense[1]}) with VITK_CLS_ONLY_TOP=0")
    assert w_flags[0] >= 0.9999, w_flags
    assert 1 - w_flags[0] <= 2 * (1 - w_dense[0]) + 1e-6, (w_flags, w_dense)


@pytest.mark.parametrize("train", [False, True])
def test_outputs_are_fresh_tensors(train):
    cfg = O.TINY
    m = _model(cfg, O.init_params(cfg, 0, 123), train)
    g = torch.Generator().manual_seed(6)
    x1, y1 = O.synth_inputs(cfg, 2, g)
    x2, y2 = O.synth_inputs(cfg, 2, g)
    with torch.set_grad_enabled(train):
        a = m(pixel_values=x1[:, 0].cuda(), labels=y1.cuda(), output_attentions=True, output_hidden_states=True)
        keep = [t.clone() for t in a.hidden_states + a.attentions]
        b = m(pixel_values=x2[:, 0].cuda(), labels=y2.cuda(), output_attentions=True, output_hidden_states=True)
    torch.cuda.synchronize()
    for t, k in zip(a.hidden_states + a.attentions, keep):
        assert torch.equal(t, k)
    assert not torch.equal(a.hidden_states[1], b.hidden_states[1]) and not torch.equal(a.attentions[0], b.attentions[0])


@pytest.mark.parametrize("image_size,B", [(384, 16), (224, 64)])
def test_output_shapes(image_size, B):
    cfg = O.OracleConfig(image_size=image_size)
    m = _model(cfg, O.init_params(cfg, 0, 123))
    g = torch.Generator().manual_seed(7)
    x = O.synth_inputs(cfg, B, g)[0][:, 0].cuda()
    with torch.no_grad():
        out = m(pixel_values=x, output_attentions=True, output_hidden_states=True)
    L, T, D, H = cfg.num_hidden_layers, cfg.seq_len, cfg.hidden_size, cfg.num_attention_heads
    assert len(out.hidden_states) == L + 1 and all(t.shape == (B, T, D) for t in out.hidden_states)
    assert len(out.attentions) == L and all(t.shape == (B, H, T, T) for t in out.attentions)
    assert out.to_tuple()[1] is out.hidden_states and out.to_tuple()[2] is out.attentions
    last = out.attentions[-1]
    assert torch.isfinite(last).all() and (last.sum(-1) - 1).abs().max() <= 1e-3
