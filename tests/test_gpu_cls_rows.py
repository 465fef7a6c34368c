"""The top encoder layer on the B CLS rows (engine.py: the cls_only_top branch of Arena._build_forward and the top
layer of Arena._build_backward).  The classifier reads only the CLS row of the last layer, so the engine runs that
layer's out-projection, LayerNorm and MLP on strided [B, ·] views of [B·T, ·] buffers (row stride T·width): GEMMs
with M = B and strided A / D / d2 / aux, weight gradients with K = B, LayerNorm with row_stride = T and column sums
with ldx = T·N.

The rows outside those views are never to be read or written: in training the non-CLS rows of dh hold stale
gradients of the previous step, and dh1 / do are read densely by the next kernels.  Every [B·T, ·] buffer of a
strided run therefore starts filled with a NaN bit pattern, and only the CLS rows of the inputs are copied in.
Afterwards every other row must still hold that exact pattern (no stray write) and every CLS row must be finite
(no stray read: a NaN that gets into a dot product, even multiplied by zero, stays NaN)."""
import math
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import vit_oracle as O

pytestmark = pytest.mark.gpu
dev = "cuda"
bf16, f32 = torch.bfloat16, torch.float32
POISON = {f32: 0x7FBADBAD, bf16: 0x7FBB}          # NaN bit patterns no kernel produces by arithmetic
BITS = {f32: torch.int32, bf16: torch.int16}
EPS = 1e-12

# (B, T, D, F): the tiny golden config (LayerNorm with one float4 per lane, N = 128); ViT-B/16 at 384 and 224;
# the two ViT-L/16@384 batches of test_gpu_model.
SHAPES = [(3, 17, 128, 256), (1, 577, 768, 3072), (2, 197, 768, 3072), (16, 577, 768, 3072), (1, 577, 1024, 4096),
          (8, 577, 1024, 4096)]
SHAPE_IDS = ["B{}-T{}-D{}-F{}".format(*s) for s in SHAPES]
PINNED = [(1, 128), (2, 128)]       # (variant, tile_n): one fixed tiling per kernel, so strided and dense runs agree bit for bit


@pytest.fixture(scope="module")
def ops():
    import chest_x_ray_vit_b200 as pkg
    pkg.ops.check_device(0)
    return pkg.ops


def cls_rows(t: torch.Tensor, B: int, T: int) -> torch.Tensor:
    """The B CLS rows of a [B·T, width] buffer, in place (row stride T·width): the view the engine's top layer uses.
    A 1-D [B·T] buffer (LayerNorm statistics) is taken as width 1."""
    t = t.view(t.shape[0], -1)
    width = t.shape[1]
    return t.view(B, T * width)[:, :width]


def _poisoned(rows: int, width: int, dtype) -> torch.Tensor:
    t = torch.empty((rows, width) if width else (rows,), dtype=dtype, device=dev)
    t.view(BITS[dtype]).fill_(POISON[dtype])
    return t


def _check_rows(bufs: dict, B: int, T: int):
    """Rows other than b·T keep the poison bit for bit; rows b·T are finite."""
    for name, t in bufs.items():
        rows = t.view(B, T, -1)
        assert bool((rows[:, 1:].view(BITS[t.dtype]) == POISON[t.dtype]).all()), f"{name}: a row outside the view was written"
        assert bool(torch.isfinite(rows[:, 0].float()).all()), f"{name}: a row of the view is not finite"


def _same_bits(x: torch.Tensor, y: torch.Tensor) -> bool:
    return torch.equal(x.contiguous().view(BITS[x.dtype]), y.contiguous().view(BITS[y.dtype]))


def _tol(K, ref):
    """test_gpu_gemm._tol: fp32 accumulation of bf16 products, weights of scale 0.05."""
    return 3e-3 * ref.abs().max().item() + 1e-3 * math.sqrt(K) * 0.05


def _bf16_tol(K, ref):
    return _tol(K, ref) + 2 ** -8 * ref.abs().max().item()


def _gen(seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    return lambda *shape: torch.randn(*shape, generator=g, device=dev)


def _weights(D, Fi, seed):
    r = _gen(seed)
    return {"wo": (r(D, D) * 0.05).to(bf16), "bo": r(D) * 0.5, "g2": 1 + 0.05 * r(D), "b2": 0.02 * r(D),
            "w1": (r(Fi, D) * 0.05).to(bf16), "bf1": r(Fi) * 0.5, "w2": (r(D, Fi) * 0.05).to(bf16), "bf2": r(D) * 0.5}


# ---------------------------------------------------------------------------------------------------- forward
def _forward_buffers(B, T, D, Fi, train, o, hin, strided):
    """Activation buffers of one layer as the arena lays them out (eval: hin = h1 = hout, no gp).  Strided: all poison
    but the CLS rows of the inputs o / hin; dense: o / hin copied whole."""
    M = B * T
    if strided:
        X = {"o": _poisoned(M, D, bf16), "hin": _poisoned(M, D, f32)}
        cls_rows(X["o"], B, T).copy_(cls_rows(o, B, T))
        cls_rows(X["hin"], B, T).copy_(cls_rows(hin, B, T))
    else:
        X = {"o": o.clone(), "hin": hin.clone()}
    X["h1"] = _poisoned(M, D, f32) if train else X["hin"]
    X["hout"] = _poisoned(M, D, f32) if train else X["hin"]
    X["n2"] = _poisoned(M, D, bf16)
    X["mean"], X["rstd"] = _poisoned(M, 0, f32), _poisoned(M, 0, f32)
    X["a"] = _poisoned(M, Fi, bf16)
    if train:
        X["gp"] = _poisoned(M, Fi, bf16)
    return X


def _run_forward(ops, X, W, B, T, strided, train, variant, tile_n):
    """out-proj (+bias +residual, fp32) → LayerNorm → fc1 (+bias, GELU, GELU') → fc2 (+bias +residual), in engine order.
    Returns the CLS rows of each output right after the launch that wrote it (eval overwrites h1 in place)."""
    D, Fi = W["wo"].shape[0], W["w1"].shape[0]
    M, rs = (B, T) if strided else (B * T, 1)
    view = (lambda t: cls_rows(t, B, T)) if strided else (lambda t: t)
    pin = dict(variant=variant, tile_n=tile_n)
    out = {}
    h1 = view(X["h1"])
    ops.gemm(view(X["o"]), W["wo"], M, D, D, h1, epilogue=ops.EPI_BIAS_RESID_F32, bias=W["bo"], aux=view(X["hin"]), **pin)
    out["h1"] = cls_rows(X["h1"], B, T).clone()
    ops.layernorm_fwd(h1, W["g2"], W["b2"], EPS, X["n2"], X["mean"], X["rstd"], row_stride=rs)
    ops.gemm(view(X["n2"]), W["w1"], M, Fi, D, view(X["a"]), epilogue=ops.EPI_BIAS_GELUG_BF16,
             d2=view(X["gp"]) if train else None, bias=W["bf1"], **pin)
    ops.gemm(view(X["a"]), W["w2"], M, D, Fi, view(X["hout"]), epilogue=ops.EPI_BIAS_RESID_F32, bias=W["bf2"], aux=h1, **pin)
    for k in ("n2", "mean", "rstd", "a", "gp", "hout"):
        if k in X:
            out[k] = cls_rows(X[k], B, T).clone()
    return out


def _check_forward_fp64(out, o, hin, W, B, T):
    """Each stage against fp64 on the bf16 / fp32 CLS-row operands it actually read."""
    D, Fi = W["wo"].shape[0], W["w1"].shape[0]
    o_c, hin_c = cls_rows(o, B, T).double(), cls_rows(hin, B, T).double()
    ref = o_c @ W["wo"].double().t() + W["bo"].double() + hin_c
    assert (out["h1"].double() - ref).abs().max() <= _tol(D, ref), "out-proj"
    h1 = out["h1"].double()
    ref = F.layer_norm(h1, (D,), W["g2"].double(), W["b2"].double(), EPS)
    assert (out["n2"].double() - ref).abs().max() <= 2 ** -8 * ref.abs().max() + 1e-6, "layernorm y"
    assert torch.allclose(out["mean"][:, 0].double(), h1.mean(1), atol=1e-5), "layernorm mean"
    assert torch.allclose(out["rstd"][:, 0].double(), torch.rsqrt(h1.var(1, unbiased=False) + EPS), rtol=1e-4), "layernorm rstd"
    u = out["n2"].double() @ W["w1"].double().t() + W["bf1"].double()
    act = F.gelu(u)
    assert (out["a"].double() - act).abs().max() <= _tol(D, u) + 2 ** -8 * act.abs().max(), "fc1 gelu"
    if "gp" in out:
        dgelu = 0.5 * (1 + torch.erf(u / math.sqrt(2))) + u * torch.exp(-0.5 * u * u) / math.sqrt(2 * math.pi)
        assert (out["gp"].double() - dgelu).abs().max() <= _tol(D, u) + 2 ** -8 * 1.2, "fc1 gelu'"
    ref = out["a"].double() @ W["w2"].double().t() + W["bf2"].double() + h1
    assert (out["hout"].double() - ref).abs().max() <= _tol(Fi, ref), "fc2"


@pytest.mark.parametrize("train", [True, False], ids=["train", "eval"])
@pytest.mark.parametrize("B,T,D,Fi", SHAPES, ids=SHAPE_IDS)
def test_top_layer_forward_rows(ops, B, T, D, Fi, train):
    r = _gen(B * T + D)
    W = _weights(D, Fi, D + Fi)
    o, hin = r(B * T, D).to(bf16), r(B * T, D)
    for variant, tile_n in PINNED:
        X = _forward_buffers(B, T, D, Fi, train, o, hin, strided=True)
        got = _run_forward(ops, X, W, B, T, True, train, variant, tile_n)
        _check_rows(X, B, T)
        Xd = _forward_buffers(B, T, D, Fi, train, o, hin, strided=False)
        want = _run_forward(ops, Xd, W, B, T, False, train, variant, tile_n)
        for k in want:
            assert _same_bits(got[k], want[k]), f"variant {variant}: {k} of the CLS rows differs from the dense launch"
    # the engine's own launches: automatic kernel and tiling choice for M = B
    X = _forward_buffers(B, T, D, Fi, train, o, hin, strided=True)
    got = _run_forward(ops, X, W, B, T, True, train, 0, 0)
    _check_rows(X, B, T)
    _check_forward_fp64(got, o, hin, W, B, T)


# ---------------------------------------------------------------------------------------------------- backward
def _backward_inputs(B, T, D, Fi, seed):
    """CLS rows of what the top layer's backward reads: dh (from head_bwd), the saved activations a / gp / n2 / o,
    the residual h1 with its LayerNorm statistics."""
    r = _gen(seed)
    h1 = r(B, D) * 1.7 + 0.3
    return {"dh": r(B, D).to(bf16), "a": F.gelu(r(B, Fi)).to(bf16), "gp": (r(B, Fi) * 0.4 + 0.5).to(bf16),
            "n2": r(B, D).to(bf16), "o": r(B, D).to(bf16), "h1": h1, "mean": h1.mean(1, keepdim=True),
            "rstd": torch.rsqrt(h1.var(1, unbiased=False, keepdim=True) + EPS)}


def _backward_buffers(I, B, T, D, Fi, strided):
    """[B·T, ·] buffers with the CLS rows of I.  Strided: every other row is poison (inputs and outputs alike);
    dense: every other row of the inputs is zero."""
    M = B * T
    width = {"dh": D, "a": Fi, "gp": Fi, "n2": D, "o": D, "h1": D, "mean": 0, "rstd": 0}
    X = {}
    for k, w in width.items():
        X[k] = _poisoned(M, w, I[k].dtype) if strided else torch.zeros((M, w) if w else (M,), dtype=I[k].dtype, device=dev)
        cls_rows(X[k], B, T).copy_(I[k])
    for k, w in (("du", Fi), ("dn", D), ("dh1", D), ("do", D)):
        X[k] = _poisoned(M, w, bf16)
    return X


def _run_backward(ops, X, W, B, T, strided, variant, tile_n):
    """Top-layer launches of _build_backward from after head_bwd up to the attention backward.  Returns the fp32
    accumulators (all started at one, or zero for dgamma / dbeta)."""
    D, Fi = W["wo"].shape[0], W["w1"].shape[0]
    M, rs = (B, T) if strided else (B * T, 1)
    view = (lambda t: cls_rows(t, B, T)) if strided else (lambda t: t)
    pin = dict(variant=variant, tile_n=tile_n)
    G = {"w2": torch.ones(D, Fi, device=dev), "bf2": torch.ones(D, device=dev), "w1": torch.ones(Fi, D, device=dev),
         "bf1": torch.ones(Fi, device=dev), "g2": torch.zeros(D, device=dev), "b2": torch.zeros(D, device=dev),
         "bo": torch.ones(D, device=dev), "wo": torch.ones(D, D, device=dev)}
    dh, du, dn, dh1, do = (view(X[k]) for k in ("dh", "du", "dn", "dh1", "do"))
    ops.gemm(dh, view(X["a"]), D, Fi, M, G["w2"], epilogue=ops.EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True, **pin)
    ops.colsum(dh, G["bf2"])
    ops.gemm(dh, W["w2"], M, Fi, D, du, epilogue=ops.EPI_MUL_BF16, b_mn_major=True, aux=view(X["gp"]), **pin)
    ops.gemm(du, view(X["n2"]), Fi, D, M, G["w1"], epilogue=ops.EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True, **pin)
    ops.colsum(du, G["bf1"])
    ops.gemm(du, W["w1"], M, D, Fi, dn, epilogue=ops.EPI_STORE_BF16, b_mn_major=True, **pin)
    ops.layernorm_bwd(X["dn"], view(X["h1"]), X["mean"], X["rstd"], W["g2"], X["dh"], G["g2"], G["b2"], dx=X["dh1"],
                      dxsum=G["bo"], row_stride=rs)
    ops.gemm(dh1, view(X["o"]), D, D, M, G["wo"], epilogue=ops.EPI_ACCUM_F32, a_mn_major=True, b_mn_major=True, **pin)
    ops.gemm(dh1, W["wo"], M, D, D, do, epilogue=ops.EPI_STORE_BF16, b_mn_major=True, **pin)
    return G


def _check_backward_fp64(X, G, I, W, B, T, data_grads: bool):
    """Accumulators against fp64 on the operands each launch read; with ``data_grads`` also du / dn / dh1 / do."""
    D = W["wo"].shape[0]
    c = {k: cls_rows(X[k], B, T).double() for k in ("du", "dn", "dh1")}
    dh = I["dh"].double()
    for name, a, b in (("w2", dh, I["a"]), ("w1", c["du"], I["n2"]), ("wo", c["dh1"], I["o"])):
        ref = a.t() @ b.double()
        assert (G[name].double() - 1 - ref).abs().max() <= _tol(B, ref) * 4, f"weight gradient {name}"
    for name, x in (("bf2", dh), ("bf1", c["du"]), ("bo", c["dh1"])):    # bo: the LayerNorm's dxsum
        assert torch.allclose(G[name].double(), 1 + x.sum(0), rtol=1e-4, atol=1e-3 * max(1.0, B ** 0.5)), f"column sum {name}"
    xr = I["h1"].double().requires_grad_(True)
    gr = W["g2"].double().requires_grad_(True)
    br = torch.zeros(D, dtype=torch.float64, device=dev, requires_grad=True)
    F.layer_norm(xr, (D,), gr, br, EPS).backward(c["dn"])
    assert torch.allclose(G["g2"].double(), gr.grad, rtol=2e-4, atol=2e-4 * gr.grad.abs().max().item()), "dgamma"
    assert torch.allclose(G["b2"].double(), br.grad, rtol=2e-4, atol=2e-4 * br.grad.abs().max().item()), "dbeta"
    if data_grads:
        ref = (dh @ W["w2"].double()) * I["gp"].double()
        assert (c["du"] - ref).abs().max() <= _bf16_tol(D, ref), "du"
        ref = c["du"] @ W["w1"].double()
        assert (c["dn"] - ref).abs().max() <= _bf16_tol(W["w1"].shape[0], ref), "dn"
        ref = xr.grad + dh
        assert (c["dh1"] - ref).abs().max() <= 2 ** -7 * ref.abs().max() + 1e-5, "dh1"
        ref = c["dh1"] @ W["wo"].double()
        assert (cls_rows(X["do"], B, T).double() - ref).abs().max() <= _bf16_tol(D, ref), "do"


@pytest.mark.parametrize("B,T,D,Fi", SHAPES, ids=SHAPE_IDS)
def test_top_layer_backward_rows(ops, B, T, D, Fi):
    W = _weights(D, Fi, D + Fi + 1)
    I = _backward_inputs(B, T, D, Fi, B * T + D + 1)
    for variant, tile_n in PINNED + [(0, 0)]:
        X = _backward_buffers(I, B, T, D, Fi, strided=True)
        G = _run_backward(ops, X, W, B, T, True, variant, tile_n)
        _check_rows(X, B, T)
        _check_backward_fp64(X, G, I, W, B, T, data_grads=variant == 0)
        if variant == 0:
            continue
        Xd = _backward_buffers(I, B, T, D, Fi, strided=False)
        _run_backward(ops, Xd, W, B, T, False, variant, tile_n)
        for k in ("du", "dn", "dh1", "do"):
            assert _same_bits(cls_rows(X[k], B, T), cls_rows(Xd[k], B, T)), \
                f"variant {variant}: {k} of the CLS rows differs from the dense launch"


# ---------------------------------------------------------------------------------------------------- LayerNorm
@pytest.mark.parametrize("M,rs", [(m, s) for s in (17, 577) for m in (1, 2, 7, 16)] + [(2000, 3)])
@pytest.mark.parametrize("D", [128, 256, 512, 768, 1024])
def test_layernorm_rows(ops, D, M, rs):
    """vitk_layernorm_{fwd,bwd}_rows with row_stride > 1, every hidden size (one warp per row for D = 128, a warp pair
    otherwise).  M = 2000 walks the backward's grid-stride loop, next-row prefetch and parity-indexed row exchange."""
    r = _gen(M * rs + D)
    x = r(M, D) * 1.7 + 0.3
    gamma, beta = 1 + 0.05 * r(D), 0.02 * r(D)
    dy, dres = r(M, D).to(bf16), r(M, D).to(bf16)
    xr = x.double().requires_grad_(True)
    gr, br = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    yr = F.layer_norm(xr, (D,), gr, br, EPS)
    yr.backward(dy.double())

    def spread(t, dtype):            # the rows of t at physical rows r·rs of a poisoned buffer
        buf = _poisoned(M * rs, D, dtype)
        buf.view(M, rs, D)[:, 0] = t
        return buf

    xb = spread(x, f32)
    xv = xb.view(M, rs * D)[:, :D]                      # ldx = rs·D, as h1's CLS rows
    y, mean, rstd = _poisoned(M * rs, D, bf16), _poisoned(M * rs, 0, f32), _poisoned(M * rs, 0, f32)
    ops.layernorm_fwd(xv, gamma, beta, EPS, y, mean, rstd, row_stride=rs)
    y1, mean1, rstd1 = ops.layernorm_fwd(x, gamma, beta, EPS)
    _check_rows({"x": xb, "y": y, "mean": mean, "rstd": rstd}, M, rs)
    for name, got, want in (("y", y, y1), ("mean", mean, mean1), ("rstd", rstd, rstd1)):
        assert _same_bits(got.view(M, rs, -1)[:, 0], want.view(M, -1)), f"{name} differs from the row_stride = 1 launch"
    yg = y.view(M, rs, D)[:, 0].double()
    assert (yg - yr).abs().max() <= 2 ** -8 * yr.abs().max() + 1e-6
    assert torch.allclose(mean1.double(), xr.mean(1), atol=1e-5)
    assert torch.allclose(rstd1.double(), torch.rsqrt(xr.var(1, unbiased=False) + EPS), rtol=1e-4)

    for extras in (True, False):     # with dres and dxsum, and without
        dyb = spread(dy, bf16)
        dresb = spread(dres, bf16) if extras else None
        dx = _poisoned(M * rs, D, bf16)
        dg, db = torch.zeros(D, device=dev), torch.zeros(D, device=dev)
        dxsum = torch.ones(D, device=dev) if extras else None
        ops.layernorm_bwd(dyb, xv, mean, rstd, gamma, dresb, dg, db, dx=dx, dxsum=dxsum, row_stride=rs)
        dx1 = ops.layernorm_bwd(dy, x, mean1, rstd1, gamma, dres if extras else None, torch.zeros(D, device=dev),
                                torch.zeros(D, device=dev), dxsum=torch.ones(D, device=dev) if extras else None)
        bufs = {"dy": dyb, "dx": dx, "mean": mean, "rstd": rstd}
        if extras:
            bufs["dres"] = dresb
        _check_rows(bufs, M, rs)
        dxg = dx.view(M, rs, D)[:, 0]
        assert _same_bits(dxg, dx1), f"dx differs from the row_stride = 1 launch (dres / dxsum: {extras})"
        ref = xr.grad + (dres.double() if extras else 0)
        assert (dxg.double() - ref).abs().max() <= 2 ** -7 * ref.abs().max() + 1e-5
        assert torch.allclose(dg.double(), gr.grad, rtol=2e-4, atol=2e-4 * gr.grad.abs().max().item())
        assert torch.allclose(db.double(), br.grad, rtol=2e-4, atol=2e-4 * br.grad.abs().max().item())
        if extras:
            assert torch.allclose(dxsum.double(), 1 + dxg.double().sum(0), rtol=1e-4, atol=1e-3 * max(1.0, M ** 0.5))


# ---------------------------------------------------------------------------------------------------- dense-top mode
def test_dense_top_layer_mode_matches_golden(monkeypatch):
    """VITK_CLS_ONLY_TOP=0 runs the top layer densely (the A/B reference of the CLS-only top layer): it must pass the
    tiny golden record like the default mode, and give the default mode's logits up to a quarter of the tolerance."""
    from test_gpu_model import GOLD, LOGIT_TOL, LOSS_RTOL, _check_grads, _model
    rec = torch.load(os.path.join(GOLD, "tiny_b3.pt"), weights_only=False)
    cfg = O.OracleConfig(**rec["cfg"])
    x, y = rec["x8"][:, 0].cuda(), rec["y"].cuda()
    monkeypatch.delenv("VITK_CLS_ONLY_TOP", raising=False)
    m_cls = _model(cfg, O.init_params(cfg, 0, 123))
    logits_cls = m_cls(pixel_values=x, labels=y).logits.detach().cpu()
    assert m_cls.engine().cls_only_top
    monkeypatch.setenv("VITK_CLS_ONLY_TOP", "0")          # read when the engine is built, at the first forward
    m = _model(cfg, O.init_params(cfg, 0, 123))
    out = m(pixel_values=x, labels=y)
    assert not m.engine().cls_only_top
    assert (out.logits.detach().cpu() - rec["logits"]).abs().max() <= LOGIT_TOL
    assert abs(out.loss.item() - rec["loss"].item()) <= LOSS_RTOL * abs(rec["loss"].item())
    out.loss.backward()
    _check_grads(m, rec["grad_sample"], rec)
    g1 = m.classifier.weight.grad.clone()
    m(pixel_values=x, labels=y).loss.backward()
    assert torch.allclose(m.classifier.weight.grad, 2 * g1, rtol=1e-3, atol=1e-7)
    gap = (out.logits.detach().cpu() - logits_cls).abs().max().item()
    print(f"dense-top vs CLS-only top: logits max-abs difference {gap:.3e}")
    assert gap <= LOGIT_TOL / 4
