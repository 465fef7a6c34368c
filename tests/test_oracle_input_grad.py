"""CPU-only: the oracle's gradient with respect to ``pixel_values`` against live HF, and the module's host logic for an
input that requires grad (which autograd node runs, what reaches the engine, dtype and device of ``x.grad``)."""
import pytest
import torch

import chest_x_ray_vit_b200 as pkg
from oracle import vit_oracle as O

TINY = dict(image_size=64, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256, num_labels=14)


def _inputs(cfg, batch=3, seed=5):
    g = torch.Generator().manual_seed(seed)
    x8, y = O.synth_inputs(cfg, batch, g)
    return O.normalize_gray(x8), y


def _rel(a, r):
    return ((a - r).abs().max() / r.abs().max()).item()


@pytest.mark.parametrize("target", ["loss", "logit"])
def test_oracle_input_grad_matches_live_hf(target):
    pytest.importorskip("transformers")
    from oracle.make_golden import hf_model
    cfg = O.TINY
    p = O.init_params(cfg, 3, 7)
    x, y = _inputs(cfg)
    hf, _ = hf_model(cfg, p)
    hf.requires_grad_(False)
    xr = x.clone().requires_grad_()
    xo = x.clone().requires_grad_()
    if target == "loss":
        hf(pixel_values=xr, labels=y).loss.backward()
        O.forward(p, cfg, xo, y)[0].backward()
        ref, got = xr.grad, xo.grad
    else:
        (ref,) = torch.autograd.grad(hf(pixel_values=xr).logits[:, 3].sum(), xr)
        (got,) = torch.autograd.grad(O.forward(p, cfg, xo)[1][:, 3].sum(), xo)
    assert got.shape == ref.shape == x.shape and got.dtype == torch.float32
    assert ref.abs().max() > 0
    assert _rel(got, ref) <= 1e-5, _rel(got, ref)


class _FakeEngine:
    """Stands in for the CUDA engine: records what the module asks of it and returns a known input gradient."""

    def __init__(self):
        self.ticket = 0
        self.calls = []

    def forward(self, pixel_values, labels, save, output_attentions=False, output_hidden_states=False):
        self.calls.append(("forward", save))
        loss = torch.ones(()) if labels is not None else None
        return loss, torch.zeros(pixel_values.shape[0], 14), None, None

    def backward(self, ticket, dloss, dlogits, needs, input_grad=False):
        self.calls.append(("backward", any(needs), input_grad))
        B = dlogits.shape[0] if dlogits is not None else 2
        dx = torch.full((B, 3, 64, 64), 0.5) if input_grad else None
        return tuple(torch.zeros_like(p) if n else None for p, n in zip(self.params, needs)), dx


@pytest.fixture
def fake(monkeypatch):
    m = pkg.ViTForImageClassification(pkg.ViTConfig(**TINY))
    eng = _FakeEngine()
    eng.params = m.param_list()
    monkeypatch.setattr(m, "engine", lambda: eng)
    return m, eng


def test_frozen_model_with_input_requiring_grad_records_a_node(fake):
    m, eng = fake
    m.requires_grad_(False)
    x = torch.zeros(2, 3, 64, 64, requires_grad=True)
    out = m(pixel_values=x)
    assert out.logits.requires_grad and eng.calls == [("forward", True)]
    out.logits.sum().backward()
    assert eng.calls[-1] == ("backward", False, True)
    assert x.grad is not None and x.grad.dtype == torch.float32 and torch.all(x.grad == 0.5)
    assert all(p.grad is None for p in m.parameters())


def test_frozen_model_plain_input_stays_outside_autograd(fake):
    m, eng = fake
    m.requires_grad_(False)
    out = m(pixel_values=torch.zeros(2, 3, 64, 64))
    assert not out.logits.requires_grad and eng.calls == [("forward", False)]
    with torch.no_grad():
        m(pixel_values=torch.zeros(2, 3, 64, 64, requires_grad=True))
    assert eng.calls[-1] == ("forward", False)


def test_trainable_model_passes_both_requests(fake):
    m, eng = fake
    x = torch.zeros(2, 3, 64, 64, requires_grad=True)
    m(pixel_values=x, labels=torch.zeros(2, 14)).loss.backward()
    assert eng.calls[-1] == ("backward", True, True)
    assert x.grad is not None
    m(pixel_values=torch.zeros(2, 3, 64, 64), labels=torch.zeros(2, 14)).loss.backward()
    assert eng.calls[-1] == ("backward", True, False)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16, torch.float64])
def test_input_grad_takes_the_input_dtype(fake, dtype):
    m, _ = fake
    m.requires_grad_(False)
    x = torch.zeros(2, 3, 64, 64, dtype=dtype, requires_grad=True)
    (g,) = torch.autograd.grad(m(pixel_values=x).logits.sum(), x)
    assert g.dtype == dtype and g.device == x.device and g.shape == x.shape and torch.all(g == 0.5)


def test_uint8_input_cannot_require_grad():
    with pytest.raises(RuntimeError):
        torch.zeros(2, 64, 64, dtype=torch.uint8).requires_grad_()


def test_unpatch_argument_checks_need_no_device():
    """vitk_gemm_bf16 validates UNPATCH_F32's arguments on the host, before it touches a device or a pointer."""
    import ctypes as C
    ops, lib = pkg.ops, pkg._lib.lib()
    B, S, D = 2, 64, 128
    T = (S // 16) ** 2 + 1

    def rc(**over):
        kw = dict(M=B * T, N=768, K=D, ldd=S, rows_out=T, row_off=1, d=1 << 24, variant=2)
        kw.update(over)
        g = ops.GemmArgs()
        g.a, g.b, g.d = 1 << 20, 1 << 22, kw["d"]
        g.M, g.N, g.K = kw["M"], kw["N"], kw["K"]
        g.lda, g.ldb, g.ldd = D, 768, kw["ldd"]
        g.b_mn_major, g.epilogue, g.variant = 1, ops.EPI_UNPATCH_F32, kw["variant"]
        g.rows_out, g.row_off = kw["rows_out"], kw["row_off"]
        return lib.vitk_gemm_bf16(C.byref(g), None), lib.vitk_last_error().decode()

    assert ops.EPI_UNPATCH_F32 == 10
    for over, code, msg in [(dict(N=640), -1, "N = 768"), (dict(rows_out=T + 1, M=B * (T + 1)), -1, "square"),
                            (dict(rows_out=1, row_off=1, M=B), -1, "rows_out > row_off"), (dict(row_off=-1), -1, "row_off"),
                            (dict(ldd=S + 16), -1, "ldd"), (dict(M=B * T - 1), -1, "M % rows_out"),
                            (dict(d=(1 << 24) + 4), -2, "aligned"), (dict(), -1, "CTA-pair kernel does not support"),
                            (dict(variant=3), -1, "CTA-pair kernel does not support")]:
        r, err = rc(**over)
        assert r == code and msg in err, (over, r, err)
