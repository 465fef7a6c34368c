"""Gradients with respect to ``pixel_values``: the VITK_EPI_UNPATCH_F32 GEMM epilogue against torch, the module against
live HF and the oracle, the data-only backward of a frozen model, and the behaviour around the default path."""
import pytest
import torch
import torch.nn.functional as F

from oracle import vit_oracle as O

pytestmark = pytest.mark.gpu
dev = "cuda"
bf16 = torch.bfloat16
COS_MIN, NORM_TOL = 0.999, 0.03        # per image: cosine and norm ratio against an fp32 reference
REPEAT_COS = 0.99999                   # two runs of the same gradient through different plans


@pytest.fixture(scope="module")
def ops():
    import chest_x_ray_vit_b200 as pkg
    pkg.ops.check_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    return pkg.ops


# ---------------------------------------------------------------------------------------------------- kernel
def _fold(cols: torch.Tensor, B: int, S: int) -> torch.Tensor:
    """Adjoint of vit_oracle.im2col: [B, P, 768] → [B, 3, S, S] (a permutation, so exact)."""
    x = torch.zeros(B, 3, S, S, device=cols.device, dtype=cols.dtype, requires_grad=True)
    (g,) = torch.autograd.grad(O.im2col(x, 16), x, grad_outputs=cols)
    return g


def _operands(B, S, D, seed):
    T = (S // 16) ** 2 + 1
    g = torch.Generator().manual_seed(seed)
    dh = torch.randn(B * T, D, generator=g).to(dev).to(bf16)
    wp = (torch.randn(D, 768, generator=g) * 0.05).to(dev).to(bf16)
    return dh, wp, T


def _unpatch_guarded(ops, dh, wp, B, S, T, D, **kw):
    """Runs UNPATCH_F32 into the middle of a NaN-filled buffer; the guards on both sides must stay NaN."""
    n, pad = B * 3 * S * S, 4096
    buf = torch.full((n + 2 * pad,), float("nan"), device=dev)
    out = buf[pad:pad + n].view(B, 3, S, S)
    ops.gemm(dh, wp, B * T, 768, D, out, epilogue=ops.EPI_UNPATCH_F32, b_mn_major=True, ldd=S, rows_out=T, row_off=1, **kw)
    torch.cuda.synchronize()
    assert torch.isnan(buf[:pad]).all() and torch.isnan(buf[pad + n:]).all(), "UNPATCH_F32 wrote outside its image"
    assert torch.isfinite(out).all(), "UNPATCH_F32 left pixels unwritten"
    return out


@pytest.mark.parametrize("D", [128, 768, 1024])
@pytest.mark.parametrize("S,B", [(64, 3), (224, 2), (384, 1), (384, 16)])
def test_unpatch_matches_torch(ops, S, B, D):
    dh, wp, T = _operands(B, S, D, S + B + D)
    out = _unpatch_guarded(ops, dh, wp, B, S, T, D)
    ref = _fold((dh.float().view(B, T, D)[:, 1:] @ wp.float()), B, S)
    err = ((out - ref).abs().max() / ref.abs().max()).item()
    assert err <= 1e-5, f"relative max-abs {err:.3e}"


@pytest.mark.parametrize("tile_n", [128, 192, 256])
@pytest.mark.parametrize("S,B,D", [(384, 2, 768), (224, 3, 1024), (64, 5, 128)])
def test_unpatch_equals_folded_store_f32(ops, S, B, D, tile_n):
    """Same tiles, same K order: the scatter moves the bits of STORE_F32 on the compact patch rows, nothing else."""
    dh, wp, T = _operands(B, S, D, 7 * S + D)
    out = _unpatch_guarded(ops, dh, wp, B, S, T, D, variant=1, tile_n=tile_n)
    P = T - 1
    compact = dh.view(B, T, D)[:, 1:].reshape(B * P, D).contiguous()
    st = torch.empty(B * P, 768, device=dev)
    ops.gemm(compact, wp, B * P, 768, D, st, epilogue=ops.EPI_STORE_F32, b_mn_major=True, variant=1, tile_n=tile_n)
    assert torch.equal(out, _fold(st.view(B, P, 768), B, S))


def test_unpatch_rejects_bad_arguments(ops):
    B, S, D = 2, 64, 128
    dh, wp, T = _operands(B, S, D, 1)
    out = torch.empty(B, 3, S, S, device=dev)

    def run(**over):
        kw = dict(M=B * T, N=768, K=D, d=out, ldd=S, rows_out=T, row_off=1)
        kw.update(over)
        M, N, K, d = kw.pop("M"), kw.pop("N"), kw.pop("K"), kw.pop("d")
        ops.gemm(dh, wp, M, N, K, d, epilogue=ops.EPI_UNPATCH_F32, b_mn_major=True, **kw)

    with pytest.raises(RuntimeError, match=r"rc=-1\).*N = 768"):
        run(N=640)
    with pytest.raises(RuntimeError, match=r"rc=-1\).*square"):
        run(rows_out=T + 1, M=B * (T + 1))
    with pytest.raises(RuntimeError, match=r"rc=-1\).*rows_out > row_off"):
        run(rows_out=1, row_off=1, M=B)
    with pytest.raises(RuntimeError, match=r"rc=-1\).*ldd"):
        run(ldd=S + 16)
    with pytest.raises(RuntimeError, match=r"rc=-1\).*M % rows_out"):
        run(M=B * T - 1)
    raw = torch.empty(out.numel() + 4, device=dev)
    with pytest.raises(RuntimeError, match=r"rc=-2\).*aligned"):
        run(d=raw[1:1 + out.numel()])
    with pytest.raises(RuntimeError, match=r"rc=-1\).*CTA-pair kernel does not support"):
        run(variant=2)
    with pytest.raises(RuntimeError, match=r"rc=-1\).*CTA-pair kernel does not support"):
        run(variant=3)
    run()                                  # the same arguments, unaltered, are accepted
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------------------------------- model
def _model(cfg: O.OracleConfig, params):
    from test_gpu_model import _model as make
    return make(cfg, params)


def _inputs(cfg, B, seed):
    g = torch.Generator().manual_seed(seed)
    x8, y = O.synth_inputs(cfg, B, g)
    return O.normalize_gray(x8), y


def _oracle_grad(cfg, params, x, y=None, c=None):
    """fp32 reference gradient of the loss (c None) or of Σ logits[:, c] with respect to x, by autograd through the
    oracle — on the GPU, with TF32 off, so that ViT-B at batch 16 takes seconds."""
    torch.backends.cuda.matmul.allow_tf32 = False
    p = {k: v.to(dev) for k, v in params.items()}
    xr = x.detach().to(dev, torch.float32).clone().requires_grad_()
    loss, logits = O.forward(p, cfg, xr, y.to(dev) if y is not None else None)
    (g,) = torch.autograd.grad(loss if c is None else logits[:, c].sum(), xr)
    return g


def _per_image(got, ref, what, cos_min=COS_MIN, norm_tol=NORM_TOL):
    g, r = got.detach().double().cpu().flatten(1), ref.detach().double().cpu().flatten(1)
    cos = F.cosine_similarity(g, r, dim=1)
    ratio = g.norm(dim=1) / r.norm(dim=1)
    print(f"{what}: per-image cosine min {cos.min().item():.7f}, norm ratio {ratio.min().item():.5f} … {ratio.max().item():.5f}")
    assert cos.min().item() >= cos_min, (what, cos)
    assert (ratio - 1).abs().max().item() <= norm_tol, (what, ratio)


def _hf_grad(hf, x, y=None, c=None):
    xr = x.clone().requires_grad_()
    out = hf(pixel_values=xr, labels=y)
    (g,) = torch.autograd.grad(out.loss if c is None else out.logits[:, c].sum(), xr)
    return g


@pytest.mark.parametrize("frozen", [False, True])
def test_tiny_matches_live_hf_eager(frozen):
    pytest.importorskip("transformers")
    from oracle.make_golden import hf_model
    cfg = O.TINY
    params = O.init_params(cfg, 3, 7)
    x, y = _inputs(cfg, 3, 5)
    hf, _ = hf_model(cfg, params)
    hf.set_attn_implementation("eager")
    ref_loss, ref_logit = _hf_grad(hf, x, y), _hf_grad(hf, x, c=2)
    m = _model(cfg, params)
    if frozen:
        m.requires_grad_(False)
    xg = x.cuda().requires_grad_()
    m(pixel_values=xg, labels=y.cuda()).loss.backward()
    _per_image(xg.grad, ref_loss, f"tiny loss.backward() {'frozen' if frozen else 'trainable'} vs HF eager")
    xg2 = x.cuda().requires_grad_()
    (g,) = torch.autograd.grad(m(pixel_values=xg2).logits[:, 2].sum(), xg2)
    _per_image(g, ref_logit, f"tiny autograd.grad(logit) {'frozen' if frozen else 'trainable'} vs HF eager")
    assert xg2.grad is None


@pytest.mark.parametrize("cfg,B", [(O.VIT_B16_384, 2), (O.VIT_B16_384, 16), (O.VIT_B16_224, 2)],
                         ids=["vitb384_b2", "vitb384_b16", "vitb224_b2"])
def test_vitb_matches_oracle(cfg, B):
    params = O.init_params(cfg, 0, 123)
    x, y = _inputs(cfg, B, 11)
    m = _model(cfg, params)
    xg = x.cuda().requires_grad_()
    m(pixel_values=xg, labels=y.cuda()).loss.backward()
    _per_image(xg.grad, _oracle_grad(cfg, params, x, y), f"ViT-B/16@{cfg.image_size} b{B} loss vs oracle")
    m.requires_grad_(False)
    xg = x.cuda().requires_grad_()
    (g,) = torch.autograd.grad(m(pixel_values=xg).logits[:, 5].sum(), xg)
    _per_image(g, _oracle_grad(cfg, params, x, c=5), f"ViT-B/16@{cfg.image_size} b{B} frozen logit vs oracle")


# ---------------------------------------------------------------------------------------------------- frozen model
class _RecordingSync:
    """Stands in for a data-parallel gradient sync: records every call made to it."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        def f(*a, **k):
            self.calls.append(name)
            return set() if name == "bucket_end_layers" else None
        return f


def _plan_record(pl):
    return [n for _, _, n in pl.steps], [(g.a, g.b, g.M, g.N, g.K, g.epilogue, g.d) for g in pl._keep]


def test_frozen_model_runs_data_only_backward(ops):
    cfg = O.VIT_B16_224
    params = O.init_params(cfg, 0, 123)
    B = 4
    x, y = _inputs(cfg, B, 12)
    m = _model(cfg, params)
    xt = x.cuda().requires_grad_()
    m(pixel_values=xt, labels=y.cuda()).loss.backward()
    ref = xt.grad.clone()
    m.zero_grad(set_to_none=True)
    m.requires_grad_(False)
    eng = m.engine()
    flat = m.flat_grads()
    flat.view(torch.int32).fill_(0x7FA5A5A5)          # a NaN payload no kernel writes
    sentinel = flat.clone()
    sync = _RecordingSync()
    eng.grad_sync = sync
    try:
        for _ in range(3):                             # kernel by kernel, capture, replay
            xf = x.cuda().requires_grad_()
            m(pixel_values=xf, labels=y.cuda()).loss.backward()
            torch.cuda.synchronize()
            _per_image(xf.grad, ref, "frozen vs trainable x.grad", cos_min=REPEAT_COS, norm_tol=1e-4)
    finally:
        eng.grad_sync = None
    assert sync.calls == []
    assert all(p.grad is None for p in m.parameters())
    assert torch.equal(flat.view(torch.int32), sentinel.view(torch.int32))
    assert m._stage_grads is None
    ar = eng.arena(B, True)
    for from_loss in (True, False):
        names, gemms = _plan_record(ar.data_backward_plan(from_loss))
        full_names, full_gemms = _plan_record(ar.backward_plan(from_loss, False))
        assert not {"vitk_colsum_bf16", "vitk_embed_bwd", "fork", "join", "record", "python"} & set(names)
        assert all(e[5] != ops.EPI_ACCUM_F32 for e in gemms)
        assert gemms == [e for e in full_gemms if e[5] != ops.EPI_ACCUM_F32]     # the same data-gradient GEMMs
        pl = ar.data_backward_plan(from_loss)
        assert pl.side_stream is None and not pl.side_steps and not pl.sync_points
    sink = ar._sink["wc"]
    assert sink.numel() == cfg.num_labels * cfg.hidden_size


# ---------------------------------------------------------------------------------------------------- mixed and edges
def test_trainable_model_with_input_grad_keeps_parameter_gradients():
    cfg = O.VIT_B16_224
    params = O.init_params(cfg, 0, 123)
    x, y = _inputs(cfg, 2, 13)
    m = _model(cfg, params)

    def step(requires):
        m.zero_grad(set_to_none=True)
        xg = x.cuda().requires_grad_(requires)
        m(pixel_values=xg, labels=y.cuda()).loss.backward()
        return xg.grad, {k: p.grad.detach().double().clone() for k, p in m.named_parameters()}
    gx0, plain = step(False)
    gx, mixed = step(True)
    assert gx0 is None and gx is not None
    for k in plain:
        if k.endswith("key.bias"):                     # analytically zero
            continue
        c = F.cosine_similarity(mixed[k].flatten(), plain[k].flatten(), dim=0).item()
        assert c >= REPEAT_COS, (k, c)
    _per_image(gx, _oracle_grad(cfg, params, x, y), "trainable + x.requires_grad vs oracle")


def test_input_grad_accumulates_and_returns_fresh_tensors():
    cfg = O.TINY
    params = O.init_params(cfg, 0, 123)
    x, y = _inputs(cfg, 2, 14)
    m = _model(cfg, params)
    m.requires_grad_(False)
    xg = x.cuda().requires_grad_()
    m(pixel_values=xg, labels=y.cuda()).loss.backward()
    first = xg.grad.clone()
    m(pixel_values=xg, labels=y.cuda()).loss.backward()
    _per_image(xg.grad, 2 * first, "two backward calls vs 2× one", cos_min=REPEAT_COS, norm_tol=1e-4)
    (r1,) = torch.autograd.grad(m(pixel_values=xg).logits[:, 1].sum(), xg)
    keep = r1.clone()
    x2, _ = _inputs(cfg, 2, 15)
    x2g = x2.cuda().requires_grad_()
    torch.autograd.grad(m(pixel_values=x2g).logits[:, 1].sum(), x2g)
    torch.cuda.synchronize()
    assert torch.equal(r1, keep)


def test_input_dtype_and_device():
    cfg = O.TINY
    params = O.init_params(cfg, 0, 123)
    x, y = _inputs(cfg, 3, 16)
    m = _model(cfg, params)
    m.requires_grad_(False)
    ref = _oracle_grad(cfg, params, x, y)
    for xin in (x.cuda().half(), x.cuda().bfloat16(), x.clone(), x.clone().double()):
        xg = xin.requires_grad_()
        m(pixel_values=xg, labels=y.cuda()).loss.backward()
        assert xg.grad.dtype == xin.dtype and xg.grad.device == xin.device and xg.grad.shape == xin.shape
        _per_image(xg.grad.float(), ref, f"{xin.dtype} on {xin.device.type}", cos_min=0.99 if xin.dtype == bf16 else COS_MIN)


def test_output_attentions_with_input_grad():
    cfg = O.TINY
    params = O.init_params(cfg, 0, 123)
    x, y = _inputs(cfg, 2, 17)
    m = _model(cfg, params)
    m.requires_grad_(False)
    xg = x.cuda().requires_grad_()
    out = m(pixel_values=xg, labels=y.cuda(), output_attentions=True, output_hidden_states=True)
    assert len(out.attentions) == cfg.num_hidden_layers and not out.attentions[0].requires_grad
    out.loss.backward()
    _per_image(xg.grad, _oracle_grad(cfg, params, x, y), "output_attentions + x.requires_grad vs oracle")


def test_plain_step_unchanged_by_input_grad_calls():
    import chest_x_ray_vit_b200 as pkg
    cfg = O.VIT_B16_224
    params = O.init_params(cfg, 0, 123)
    x, y = _inputs(cfg, 2, 18)
    x, y = x.cuda(), y.cuda()
    m = _model(cfg, params)

    def plain(xp):
        m.zero_grad(set_to_none=True)
        n0 = pkg.ops.launch_count()
        m(pixel_values=xp, labels=y).loss.backward()
        torch.cuda.synchronize()
        assert xp.grad is None
        return pkg.ops.launch_count() - n0
    for _ in range(2):                                  # the first call launches kernel by kernel, the second captures
        plain(x)
    n_before = plain(x)
    ar = m.engine().arena(2, True)
    plans_before = [_plan_record(p) for p in (ar.fwd, ar.fwd_loss, ar.bwd_loss, ar.bwd_logits)]
    xg = x.clone().requires_grad_()
    m(pixel_values=xg, labels=y).loss.backward()        # full plan + input GEMM
    m.requires_grad_(False)
    xg = x.clone().requires_grad_()
    m(pixel_values=xg, labels=y).loss.backward()        # data-only plan + input GEMM
    m.requires_grad_(True)
    assert plain(x.clone()) == n_before
    assert [_plan_record(p) for p in (ar.fwd, ar.fwd_loss, ar.bwd_loss, ar.bwd_logits)] == plans_before
    assert m.engine().arena(2, True) is ar
