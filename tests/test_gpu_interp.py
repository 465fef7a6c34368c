"""Inputs of another size than the checkpoint's (``interpolate_pos_encoding``): the position-embedding resize and its
adjoint against fp64, the rectangular UNPATCH_F32 input-gradient epilogue, the module against live HF and the oracle at
other grids, the dense top layer above T = 4096, and arenas of several grids in one process."""
import pytest
import torch
import torch.nn.functional as F

from oracle import interp_oracle as I
from oracle import outputs_oracle as OO
from oracle import vit_oracle as O

pytestmark = pytest.mark.gpu
dev = "cuda"
bf16 = torch.bfloat16
LOGIT_TOL, LOSS_RTOL, COS_MIN = 2e-2, 1e-3, 0.999    # the project's model tolerances (test_gpu_model.py)
HS_TOL, HS_COS = 2e-2, 0.9999                        # hidden states (test_gpu_outputs.py)
AT_TOL, AT_COS = 1e-2, 0.999                         # attention maps (test_gpu_outputs.py)
REPEAT_COS = 0.99999                                 # the same input gradient through another run of the same plans
# the same parameter gradients from another run: split-K weight gradients add with fp32 atomics and the attention dQ
# of T > 128 is not bit-reproducible, so repeated gradients differ in the last bits; the patch-embedding weight, a sum
# over every token, shows it most (0.999989 measured on a B200 at 384 px, batch 2)
REPEAT_GRAD_COS = 0.9999


@pytest.fixture(scope="module")
def pkg():
    import chest_x_ray_vit_b200 as p
    p.ops.check_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    return p


def _guarded(n, pad=1024):
    buf = torch.full((n + 2 * pad,), float("nan"), device=dev)
    return buf, buf[pad:pad + n]


def _rel(a, r):
    return ((a.double() - r.double()).abs().max() / r.double().abs().max()).item()


# ---------------------------------------------------------------------------------------------------- resize kernels
GRIDS = [(3, 3), (28, 28), (32, 32), (40, 40), (24, 40), (64, 64), (1, 7), (1, 1), (5, 1)]


@pytest.mark.parametrize("D", [128, 768, 1024])
@pytest.mark.parametrize("s", [4, 14, 24])
@pytest.mark.parametrize("gh,gw", GRIDS, ids=lambda v: str(v))
def test_pos_interp_matches_fp64(pkg, s, gh, gw, D):
    g = torch.Generator().manual_seed(s * 7 + gh * 3 + gw + D)
    pos = torch.randn(1 + s * s, D, generator=g)
    n = (1 + gh * gw) * D
    buf, out = _guarded(n)
    n0 = pkg.ops.launch_count()
    pkg.ops.pos_interp(pos.to(dev), s, s, gh, gw, out=out.view(1 + gh * gw, D))
    torch.cuda.synchronize()
    assert pkg.ops.launch_count() - n0 == 1
    assert torch.isnan(buf[:1024]).all() and torch.isnan(buf[1024 + n:]).all(), "pos_interp wrote outside its output"
    got = out.view(1 + gh * gw, D).cpu()
    ref = I.pos_interp(pos, s, s, gh, gw)
    assert torch.equal(got[0], pos[0])
    err = _rel(got, ref)
    assert err <= 2e-6, f"relative max-abs {err:.3e}"


@pytest.mark.parametrize("D", [128, 768, 1024])
@pytest.mark.parametrize("s", [4, 14, 24])
@pytest.mark.parametrize("gh,gw", GRIDS, ids=lambda v: str(v))
def test_pos_interp_bwd_is_the_fp64_adjoint(pkg, s, gh, gw, D):
    g = torch.Generator().manual_seed(s * 11 + gh * 5 + gw + D)
    dout = torch.randn(1 + gh * gw, D, generator=g)
    init = torch.randn(1 + s * s, D, generator=g)              # dpos is accumulated onto
    n = (1 + s * s) * D
    buf, dpos = _guarded(n)
    dpos.copy_(init.flatten().to(dev))
    d_dev = dout.to(dev)
    pkg.ops.pos_interp_bwd(d_dev, gh, gw, s, s, dpos.view(1 + s * s, D))
    torch.cuda.synchronize()
    assert torch.isnan(buf[:1024]).all() and torch.isnan(buf[1024 + n:]).all(), "pos_interp_bwd wrote outside dpos"
    got = dpos.view(1 + s * s, D).cpu().double() - init.double()
    ref = I.pos_interp_bwd(dout, gh, gw, s, s)
    err = ((got - ref).abs().max() / ref.abs().max()).item()
    assert err <= 1e-5, f"relative max-abs {err:.3e}"
    # two runs from the same start give the same bits
    again = init.to(dev).contiguous()
    pkg.ops.pos_interp_bwd(d_dev, gh, gw, s, s, again)
    assert torch.equal(again, dpos.view(1 + s * s, D))
    # <R x, y> = <x, Rᵀ y>, both sides from the kernels, in fp64
    x = torch.randn(1 + s * s, D, generator=g)
    rx = pkg.ops.pos_interp(x.to(dev), s, s, gh, gw).cpu().double()
    rty = pkg.ops.pos_interp_bwd(d_dev, gh, gw, s, s, torch.zeros(1 + s * s, D, device=dev)).cpu().double()
    lhs, rhs = (rx * dout.double()).sum().item(), (x.double() * rty).sum().item()
    scale = (rx.abs() * dout.double().abs()).sum().item()
    assert abs(lhs - rhs) <= 1e-6 * scale, (lhs, rhs)


def test_pos_interp_rejects_bad_arguments(pkg):
    pos = torch.zeros(1 + 16, 128, device=dev)
    out = torch.zeros(1 + 64, 128, device=dev)
    lib = pkg._lib.lib()
    P, O_ = pos.data_ptr(), out.data_ptr()
    # (source, gh0, gw0, gh, gw, D, destination) of the forward; the backward gets the same grids the other way round
    for src, gh0, gw0, gh, gw, D, dst, msg in [(P, 4, 4, 0, 8, 128, O_, "grids"), (P, 4, 4, 8, 8, 126, O_, "multiple of 4"),
                                               (P, 4, 4, 8, 5000, 128, O_, "grids"), (P + 4, 4, 4, 8, 8, 128, O_, "aligned"),
                                               (None, 4, 4, 8, 8, 128, O_, "NULL")]:
        assert lib.vitk_pos_interp(src, gh0, gw0, gh, gw, D, dst, None) == (-2 if msg == "aligned" else -1)
        assert msg in lib.vitk_last_error().decode()
        assert lib.vitk_pos_interp_bwd(dst if src else None, gh, gw, gh0, gw0, D, src if src else P, None) < 0
        assert msg in lib.vitk_last_error().decode()
    torch.cuda.synchronize()
    assert not out.any() and not pos.any()


# ---------------------------------------------------------------------------------------------------- rectangular UNPATCH
def _fold(cols, B, Hi, Wi):
    x = torch.zeros(B, 3, Hi, Wi, device=cols.device, dtype=cols.dtype, requires_grad=True)
    (g,) = torch.autograd.grad(O.im2col(x, 16), x, grad_outputs=cols)
    return g


@pytest.mark.parametrize("tile_n", [128, 256])
@pytest.mark.parametrize("gh,gw", [(4, 6), (24, 32), (32, 24), (40, 40)], ids=lambda v: str(v))
def test_unpatch_rectangular(pkg, gh, gw, tile_n):
    ops = pkg.ops
    B, D = 2, 768
    P, T = gh * gw, gh * gw + 1
    g = torch.Generator().manual_seed(gh * 100 + gw)
    dh = torch.randn(B * T, D, generator=g).to(dev).to(bf16)
    wp = (torch.randn(D, 768, generator=g) * 0.05).to(dev).to(bf16)
    n = B * 3 * 16 * gh * 16 * gw
    buf, flat = _guarded(n, 4096)
    out = flat.view(B, 3, 16 * gh, 16 * gw)
    ops.gemm(dh, wp, B * T, 768, D, out, epilogue=ops.EPI_UNPATCH_F32, b_mn_major=True, ldd=16 * gw, rows_out=T, row_off=1,
             rows_in=gw, variant=1, tile_n=tile_n)
    torch.cuda.synchronize()
    assert torch.isnan(buf[:4096]).all() and torch.isnan(buf[4096 + n:]).all(), "UNPATCH_F32 wrote outside its image"
    assert torch.isfinite(out).all(), "UNPATCH_F32 left pixels unwritten"
    ref = _fold(dh.float().view(B, T, D)[:, 1:] @ wp.float(), B, 16 * gh, 16 * gw)
    assert _rel(out, ref) <= 1e-5
    compact = dh.view(B, T, D)[:, 1:].reshape(B * P, D).contiguous()
    st = torch.empty(B * P, 768, device=dev)
    ops.gemm(compact, wp, B * P, 768, D, st, epilogue=ops.EPI_STORE_F32, b_mn_major=True, variant=1, tile_n=tile_n)
    assert torch.equal(out, _fold(st.view(B, P, 768), B, 16 * gh, 16 * gw))
    with pytest.raises(RuntimeError, match=r"rc=-1\).*rows_in"):
        ops.gemm(dh, wp, B * T, 768, D, out, epilogue=ops.EPI_UNPATCH_F32, b_mn_major=True, ldd=16 * gw, rows_out=T,
                 row_off=1, rows_in=P + 1)
    with pytest.raises(RuntimeError, match=r"rc=-1\).*ldd"):
        ops.gemm(dh, wp, B * T, 768, D, out, epilogue=ops.EPI_UNPATCH_F32, b_mn_major=True, ldd=16 * gw + 16, rows_out=T,
                 row_off=1, rows_in=gw)


# ---------------------------------------------------------------------------------------------------- module
def _model(cfg, params):
    from test_gpu_model import _model as make
    return make(cfg, params)


def _images(B, Hi, Wi, seed, ncls=14):
    g = torch.Generator().manual_seed(seed)
    x8 = torch.randint(0, 256, (B, 1, Hi, Wi), dtype=torch.uint8, generator=g)
    y = (torch.rand(B, ncls, generator=g) < 0.2).float()
    return x8, y


def _check_grads(m, ref, what):
    worst = 1.0
    for k, p in m.named_parameters():
        gk, r = p.grad.detach().double().cpu(), ref[k].detach().double().cpu()
        assert gk.shape == r.shape, k
        if k.endswith("key.bias"):          # analytically zero
            qn = m.get_parameter(k.replace("key.bias", "query.bias")).grad.norm().item()
            assert gk.norm().item() <= 0.05 * qn + 1e-7, k
            continue
        c = F.cosine_similarity(gk.flatten(), r.flatten(), dim=0).item()
        worst = min(worst, c)
        assert c >= COS_MIN and abs(gk.norm().item() / r.norm().item() - 1) < 0.03, (k, c)
    pc = F.cosine_similarity(m.vit.embeddings.position_embeddings.grad.double().cpu().flatten(),
                             ref["vit.embeddings.position_embeddings"].double().cpu().flatten(), dim=0).item()
    print(f"{what}: worst gradient cosine {worst:.6f}, position_embeddings {pc:.6f}")


def _per_image(got, ref, what):
    g, r = got.detach().double().cpu().flatten(1), ref.detach().double().cpu().flatten(1)
    cos = F.cosine_similarity(g, r, dim=1)
    ratio = g.norm(dim=1) / r.norm(dim=1)
    print(f"{what}: input gradient per-image cosine min {cos.min().item():.7f}, norm ratio {ratio.min().item():.5f} … "
          f"{ratio.max().item():.5f}")
    assert cos.min().item() >= COS_MIN and (ratio - 1).abs().max().item() <= 0.03


def _check_outputs(hidden, attn, ref_hidden, ref_attn, what):
    worst_h, worst_a = 1.0, 1.0
    for a, r in zip(hidden, ref_hidden):
        a, r = a.double().cpu(), r.double().cpu()
        assert a.shape == r.shape
        assert (a - r).abs().max().item() <= HS_TOL * r.abs().max().item()
        worst_h = min(worst_h, F.cosine_similarity(a.flatten(), r.flatten(), dim=0).item())
    for a, r in zip(attn, ref_attn):
        a, r = a.double().cpu(), r.double().cpu()
        assert a.shape == r.shape
        assert (a - r).abs().max().item() <= AT_TOL
        worst_a = min(worst_a, F.cosine_similarity(a.flatten(), r.flatten(), dim=0).item())
    print(f"{what}: hidden-state cosine min {worst_h:.6f}, attention-map cosine min {worst_a:.6f}")
    assert worst_h >= HS_COS and worst_a >= AT_COS


def _oracle_outputs(p, cfg, x):
    """Hidden states and attention maps of the oracle with the flag (oracle/outputs_oracle.py, interpolated embeddings)."""
    h = I.embeddings(p, cfg, x, True)
    hs, maps = [h], []
    H, D = cfg.num_attention_heads, cfg.hidden_size
    for i in range(cfg.num_hidden_layers):
        pre = f"vit.encoder.layer.{i}."
        n1 = O.layer_norm(h, p[pre + "layernorm_before.weight"], p[pre + "layernorm_before.bias"], cfg.layer_norm_eps)
        B, T, _ = h.shape
        q = (n1 @ p[pre + "attention.attention.query.weight"].t() + p[pre + "attention.attention.query.bias"])
        k = (n1 @ p[pre + "attention.attention.key.weight"].t() + p[pre + "attention.attention.key.bias"])
        maps.append(OO.attention_probs(q.view(B, T, H, 64).transpose(1, 2), k.view(B, T, H, 64).transpose(1, 2), 64 ** -0.5))
        h = O.encoder_layer(p, cfg, i, h)
        hs.append(h)
    return hs, maps


@pytest.mark.parametrize("Hi,Wi", [(96, 96), (64, 112)], ids=lambda v: str(v))
@pytest.mark.parametrize("kind", ["f32", "u8"])
@pytest.mark.parametrize("mode", ["train", "eval"])
def test_tiny_matches_live_hf_eager(pkg, Hi, Wi, kind, mode):
    pytest.importorskip("transformers")
    from oracle.make_golden import hf_model
    cfg = O.TINY
    params = O.init_params(cfg, 3, 7)
    x8, y = _images(3, Hi, Wi, Hi + Wi)
    x = O.normalize_gray(x8)
    hf, _ = hf_model(cfg, params)
    hf.set_attn_implementation("eager")
    xr = x.clone().requires_grad_()
    ref = hf(pixel_values=xr, labels=y, interpolate_pos_encoding=True, output_attentions=True, output_hidden_states=True)
    ref.loss.backward()
    m = _model(cfg, params)
    xin = x8[:, 0].cuda() if kind == "u8" else x.cuda().requires_grad_()
    if mode == "eval":
        m.eval()
        with torch.no_grad():
            out = m(pixel_values=xin, labels=y.cuda(), interpolate_pos_encoding=True, output_attentions=True,
                    output_hidden_states=True)
    else:
        out = m(pixel_values=xin, labels=y.cuda(), interpolate_pos_encoding=True, output_attentions=True,
                output_hidden_states=True)
    T = (Hi // 16) * (Wi // 16) + 1
    assert out.logits.shape == (3, 14) and out.hidden_states[0].shape == (3, T, cfg.hidden_size)
    assert out.attentions[0].shape == (3, cfg.num_attention_heads, T, T)
    dl = (out.logits.detach().cpu() - ref.logits.detach()).abs().max().item()
    rl = abs(out.loss.item() - ref.loss.item()) / abs(ref.loss.item())
    print(f"tiny {Hi}x{Wi} {kind} {mode} vs HF eager: logits max-abs {dl:.2e}, loss rel {rl:.2e}")
    assert dl <= LOGIT_TOL and rl <= LOSS_RTOL
    _check_outputs(out.hidden_states, out.attentions, ref.hidden_states, ref.attentions, f"tiny {Hi}x{Wi} {kind} {mode}")
    if mode == "train":
        out.loss.backward()
        _check_grads(m, {k: p.grad for k, p in hf.named_parameters()}, f"tiny {Hi}x{Wi} {kind}")
        assert m.vit.embeddings.position_embeddings.shape == (1, cfg.seq_len, cfg.hidden_size)
        if kind == "f32":
            assert xin.grad.shape == x.shape
            _per_image(xin.grad, xr.grad, f"tiny {Hi}x{Wi}")


def _oracle_step(cfg, params, x, y):
    p = {k: v.to(dev) for k, v in params.items()}
    leaves = {k: v.detach().clone().requires_grad_() for k, v in p.items()}
    xr = x.to(dev).requires_grad_()
    loss, logits = I.forward(leaves, cfg, xr, y.to(dev), interpolate_pos_encoding=True)
    loss.backward()
    return loss.detach(), logits.detach(), {k: v.grad for k, v in leaves.items()}, xr.grad


@pytest.mark.parametrize("Hi,Wi,B,outputs", [(512, 512, 2, True), (384, 640, 2, True), (512, 512, 16, False)],
                         ids=["512x512_b2", "384x640_b2", "512x512_b16"])
def test_vitb_at_other_sizes_matches_oracle(pkg, Hi, Wi, B, outputs):
    cfg = O.VIT_B16_384
    params = O.init_params(cfg, 0, 123)
    x8, y = _images(B, Hi, Wi, Hi * 3 + Wi + B)
    x = O.normalize_gray(x8)
    m = _model(cfg, params)
    xg = x.cuda().requires_grad_()
    out = m(pixel_values=xg, labels=y.cuda(), interpolate_pos_encoding=True, output_attentions=outputs,
            output_hidden_states=outputs)
    out.loss.backward()
    loss, logits, grads, xgrad = _oracle_step(cfg, params, x, y)
    dl = (out.logits.detach() - logits).abs().max().item()
    rl = abs(out.loss.item() - loss.item()) / abs(loss.item())
    print(f"ViT-B/16@384 at {Hi}x{Wi} b{B}: logits max-abs {dl:.2e}, loss rel {rl:.2e}")
    assert dl <= LOGIT_TOL and rl <= LOSS_RTOL
    _check_grads(m, grads, f"ViT-B/16@384 at {Hi}x{Wi} b{B}")
    _per_image(xg.grad, xgrad, f"ViT-B/16@384 at {Hi}x{Wi} b{B}")
    if outputs:
        with torch.no_grad():
            hs, maps = _oracle_outputs({k: v.to(dev) for k, v in params.items()}, cfg, x.to(dev))
        _check_outputs(out.hidden_states, out.attentions, hs, maps, f"ViT-B/16@384 at {Hi}x{Wi} b{B}")


def test_dense_top_layer_above_4096_tokens(pkg):
    cfg = O.TINY
    params = O.init_params(cfg, 1, 5)
    x8, y = _images(2, 1040, 1040, 9)
    x = O.normalize_gray(x8)
    m = _model(cfg, params)
    xg = x.cuda().requires_grad_()
    out = m(pixel_values=xg, labels=y.cuda(), interpolate_pos_encoding=True)
    out.loss.backward()
    ar = m.engine().arena(2, True, 65, 65)
    assert ar.T == 4226 and not ar.cls_top
    names = [n for _, _, n in ar.fwd_loss.steps]
    assert "vitk_attn_cls_fwd" not in names and names[0] == "vitk_pos_interp"
    assert "vitk_attn_cls_bwd" not in [n for _, _, n in ar.bwd_loss.steps]
    loss, logits, grads, xgrad = _oracle_step(cfg, params, x, y)
    dl = (out.logits.detach() - logits).abs().max().item()
    rl = abs(out.loss.item() - loss.item()) / abs(loss.item())
    print(f"tiny at 1040x1040 (T = 4226): logits max-abs {dl:.2e}, loss rel {rl:.2e}")
    assert dl <= LOGIT_TOL and rl <= LOSS_RTOL
    _check_grads(m, grads, "tiny at 1040x1040")
    _per_image(xg.grad, xgrad, "tiny at 1040x1040")


def _step(m, x, y, **kw):
    m.zero_grad(set_to_none=True)
    out = m(pixel_values=x, labels=y, **kw)
    out.loss.backward()
    torch.cuda.synchronize()
    return out.logits.detach().clone(), {k: p.grad.detach().clone() for k, p in m.named_parameters()}


def _same_grads(a, b, what):
    worst = 1.0
    for k in a:
        if k.endswith("key.bias"):
            continue
        c = F.cosine_similarity(a[k].double().flatten(), b[k].double().flatten(), dim=0).item()
        worst = min(worst, c)
        assert c >= REPEAT_GRAD_COS, (k, c)
    print(f"{what}: worst gradient cosine {worst:.7f}")


def test_flag_at_the_config_size_is_the_plain_call(pkg):
    cfg = O.TINY
    params = O.init_params(cfg, 0, 123)
    x8, y = _images(3, 64, 64, 4)
    m = _model(cfg, params)
    x, y = O.normalize_gray(x8).cuda(), y.cuda()
    lp, gp = _step(m, x, y)
    keys = set(m.engine().arenas)
    for flag in (True, False, None):
        lf, gf = _step(m, x, y, interpolate_pos_encoding=flag)
        assert torch.equal(lf, lp)
        _same_grads(gf, gp, f"flag={flag} at the config size vs the plain call")
        with torch.no_grad():
            assert torch.equal(m(pixel_values=x, interpolate_pos_encoding=flag).logits, m(pixel_values=x).logits)
    assert set(m.engine().arenas) - keys <= {(3, False, 4, 4)} and all(k[2:] == (4, 4) for k in m.engine().arenas)


def test_mixed_sizes_in_one_process(pkg):
    cfg = O.VIT_B16_384
    params = O.init_params(cfg, 0, 123)
    a8, ya = _images(2, 384, 384, 21)
    b8, yb = _images(2, 512, 512, 22)
    xa, xb = O.normalize_gray(a8).cuda(), O.normalize_gray(b8).cuda()
    ya, yb = ya.cuda(), yb.cuda()
    m = _model(cfg, params)
    eng = m.engine()
    la, ga = _step(m, xa, ya, interpolate_pos_encoding=True)
    lb, gb = _step(m, xb, yb, interpolate_pos_encoding=True)
    arenas = dict(eng.arenas)
    assert set(arenas) == {(2, True, 24, 24), (2, True, 32, 32)}
    la2, ga2 = _step(m, xa, ya)
    assert torch.equal(la2, la) and dict(eng.arenas) == arenas and all(eng.arenas[k] is arenas[k] for k in arenas)
    _same_grads(ga2, ga, "384 px after 512 px vs the first 384 px step")
    # two forwards of different grids, then the backward of the first: each grid keeps its own activations
    m.zero_grad(set_to_none=True)
    ob = m(pixel_values=xb, labels=yb, interpolate_pos_encoding=True)
    oa = m(pixel_values=xa, labels=ya, interpolate_pos_encoding=True)
    ob.loss.backward()
    torch.cuda.synchronize()
    assert torch.equal(ob.logits.detach(), lb) and torch.equal(oa.logits.detach(), la)
    _same_grads({k: p.grad for k, p in m.named_parameters()}, gb, "512 backward after a 384 forward vs the 512 step")
    # a plain step afterwards matches a fresh model's
    lf, gf = _step(_model(cfg, params), xa, ya)
    lp, gp = _step(m, xa, ya)
    assert torch.equal(lp, lf)
    _same_grads(gp, gf, "plain 384 step after mixed sizes vs a fresh model")


def test_frozen_model_at_512_runs_the_data_only_plan(pkg):
    cfg = O.VIT_B16_384
    params = O.init_params(cfg, 0, 123)
    x8, y = _images(2, 512, 512, 31)
    x, y = O.normalize_gray(x8).cuda(), y.cuda()
    m = _model(cfg, params)
    xt = x.clone().requires_grad_()
    m(pixel_values=xt, labels=y, interpolate_pos_encoding=True).loss.backward()
    m.zero_grad(set_to_none=True)
    m.requires_grad_(False)
    # at T = 1025 the attention dQ's non-reproducible last bits reach x.grad more than at 577: the trainable model's
    # x.grad is matched to 0.99997 (B200), so the bound here is 0.9999, and both are checked against the oracle
    _, _, _, ref = _oracle_step(cfg, params, x.cpu(), y.cpu())
    _per_image(xt.grad, ref, "trainable ViT-B/16@384 at 512x512 vs the oracle")
    for _ in range(2):
        xf = x.clone().requires_grad_()
        m(pixel_values=xf, labels=y, interpolate_pos_encoding=True).loss.backward()
        torch.cuda.synchronize()
        g, r = xf.grad.double().flatten(1), xt.grad.double().flatten(1)
        cos = F.cosine_similarity(g, r, dim=1).min().item()
        print(f"frozen vs trainable x.grad at 512x512: per-image cosine min {cos:.7f}")
        assert cos >= REPEAT_GRAD_COS
        assert ((g.norm(dim=1) / r.norm(dim=1)) - 1).abs().max().item() <= 1e-3
        _per_image(xf.grad, ref, "frozen ViT-B/16@384 at 512x512 vs the oracle")
    assert all(p.grad is None for p in m.parameters())
    ar = m.engine().arena(2, True, 32, 32)
    names = [n for _, _, n in ar.data_backward_plan(True).steps]
    assert "vitk_pos_interp_bwd" not in names and "vitk_embed_bwd" not in names


def test_optimizer_step_after_a_512_backward(pkg):
    cfg = O.VIT_B16_384
    params = O.init_params(cfg, 0, 123)
    x8, y = _images(2, 512, 512, 41)
    m = _model(cfg, params)
    opt = pkg.VitkAdamW(m, lr=1e-3)
    pe = m.vit.embeddings.position_embeddings
    before = pe.detach().clone()
    m(pixel_values=O.normalize_gray(x8).cuda(), labels=y.cuda(), interpolate_pos_encoding=True).loss.backward()
    assert pe.grad.shape == (1, 577, 768) and pe.grad.abs().max() > 0
    opt.step()
    torch.cuda.synchronize()
    assert pe.shape == (1, 577, 768) and not torch.equal(pe.detach(), before)
    moved = (pe.detach() - before).abs().amax(-1)[0]
    assert (moved > 0).all()          # every position, CLS included, received gradient through the resize
