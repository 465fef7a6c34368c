"""Fused attention forward/backward (csrc/attention.cu) and the CLS-row kernels (csrc/attention_cls.cu) through the C ABI,
row by row against the fp64 oracle (oracle/attention_oracle.py): every (image, token, head) row of O / dQ / dK / dV
within the calibrated TAU, lse within its absolute bound.  Around that: outputs inside guarded NaN buffers, inputs left
bit-identical, poisoned / exactly-sized / reused workspaces, determinism, work-item counts around the SM count,
contended schedules, a PDL chain on a side stream, and argument errors."""
import math

import pytest
import torch

from oracle import attention_oracle as A

pytestmark = pytest.mark.gpu
dev = "cuda"
bf16, f32, u8 = torch.bfloat16, torch.float32, torch.uint8
GUARD = 4096


@pytest.fixture(scope="module")
def ops():
    import chest_x_ray_vit_b200 as pkg
    pkg.ops.check_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    return pkg.ops


class Guarded:
    """``n`` elements of ``dtype`` at byte ``offset`` past a 4 KB guard and followed by another, in a buffer whose every
    byte starts as 0xFF (a NaN in bf16 and fp32).  The allocator hands out 512-byte aligned blocks, so the data pointer
    sits ``offset`` bytes past a 256-byte boundary."""

    def __init__(self, n, dtype, offset=16, like=None):
        size = torch.empty((), dtype=dtype).element_size()
        self.lo, self.hi = GUARD + offset, GUARD + offset + n * size
        self.raw = torch.full((self.hi + GUARD,), 0xFF, dtype=u8, device=dev)
        self.t = self.raw[self.lo:self.hi].view(dtype)
        assert self.t.data_ptr() % 256 == offset
        if like is not None:
            self.t.copy_(like.reshape(-1))

    def intact(self):
        return bool((self.raw[:self.lo] == 0xFF).all()) and bool((self.raw[self.hi:] == 0xFF).all())

    def untouched(self):
        return bool((self.raw == 0xFF).all())


def _bits(t):
    return t.contiguous().reshape(-1).view(u8)


def _same_bits(a, b):
    return torch.equal(_bits(a), _bits(b))


def _inputs(B, T, H, scale, family):
    qkv, do = A.inputs(B, T, H, scale, family)
    return qkv.to(dev), do.to(dev)


def _grads(dqkv, B, T, H):
    d = dqkv.view(B, T, 3, H, A.DH)
    return {"dq": d[:, :, 0], "dk": d[:, :, 1], "dv": d[:, :, 2]}


def _check(got, ref, what, names=A.ROWS, tokens=slice(None)):
    """Worst row per tensor within TAU (tokens: the token range compared); prints the worst rows."""
    r = {n: ref[n][:, tokens] for n in names}
    r["terms"] = {n: ref["terms"][n][:, tokens] for n in names}
    e = A.row_errors({n: got[n].reshape(ref[n].shape)[:, tokens] for n in names}, r, names)
    print(f"{what}: " + "  ".join(f"{n} {e[n]['worst']:.4f}@{e[n]['row']} (τ {A.TAU[n]})" for n in names))
    for n in names:
        assert e[n]["worst"] <= A.TAU[n], f"{what}: {n} row {e[n]['row']} off by {e[n]['worst']:.4f} > τ {A.TAU[n]}"


def _check_lse(lse, ref, what, tokens=slice(None)):
    err = (lse.double() - ref["lse"])[..., tokens].abs()
    tol = ref["lse_tol"][..., tokens]
    worst = (err / tol).max().item()
    assert torch.isfinite(lse[..., tokens]).all() and worst <= 1.0, f"{what}: lse off by {worst:.2f}× its bound"


def _check_dq(dq, dq_first, ref, T, what):
    """dQ of a second call: the same bits when every element got one reduce-add (T ≤ 128), within TAU otherwise."""
    if T <= 128:
        assert _same_bits(dq, dq_first), f"{what}: dQ differs between calls"
    else:
        _check({"dq": dq}, ref, what, names=("dq",))


# ---------------------------------------------------------------------------------------------------- dense kernels
@pytest.mark.parametrize("B,T,H,scale,family", A.SWEEP, ids=[A.case_id(*c) for c in A.SWEEP])
def test_attention_fwd_bwd(ops, B, T, H, scale, family):
    """The sweep, twice: fresh buffers and a zeroed workspace; then every buffer at a 16-byte offset (lse: 4 bytes)
    inside 0xFF guards, outputs starting as NaN and the workspace exactly attn_bwd_workspace_bytes long, filled with
    0xFF.  The second run must write every output element, nothing outside, leave qkv / o / do / lse alone and repeat
    the first: o, lse, dK and dV bit for bit (one CTA per item, fixed accumulation order), dQ as _check_dq."""
    what = A.case_id(B, T, H, scale, family)
    qkv, do = _inputs(B, T, H, scale, family)
    ref = A.reference(qkv, do, scale)
    o, lse = ops.attn_fwd(qkv, B, T, H, scale)
    ws = torch.zeros(ops.attn_bwd_workspace_bytes(B, T, H), dtype=u8, device=dev)
    dqkv = ops.attn_bwd(qkv, o, do.view(B * T, -1), lse, B, T, H, scale, workspace=ws)
    torch.cuda.synchronize()
    _check({"o": o, **_grads(dqkv, B, T, H)}, ref, what)
    _check_lse(lse, ref, what)

    gq, gdo = Guarded(qkv.numel(), bf16, like=qkv), Guarded(do.numel(), bf16, like=do)
    go, gl, gd = Guarded(o.numel(), bf16), Guarded(lse.numel(), f32, offset=4), Guarded(dqkv.numel(), bf16)
    gw = Guarded(ws.numel(), u8)
    ops.attn_fwd(gq.t, B, T, H, scale, go.t, gl.t)
    o2, lse2 = go.t.clone(), gl.t.clone()
    ops.attn_bwd(gq.t, go.t, gdo.t, gl.t, B, T, H, scale, gd.t, gw.t)
    torch.cuda.synchronize()
    for name, g in (("qkv", gq), ("do", gdo), ("o", go), ("lse", gl), ("dqkv", gd), ("workspace", gw)):
        assert g.intact(), f"{what}: a byte around {name} was written"
    assert torch.isfinite(o2.float()).all() and torch.isfinite(gd.t.float()).all(), f"{what}: an output element left unwritten"
    assert _same_bits(gq.t, qkv) and _same_bits(gdo.t, do), f"{what}: qkv or do changed"
    assert _same_bits(go.t, o2) and _same_bits(gl.t, lse2), f"{what}: attn_bwd changed o or lse"
    assert _same_bits(o2, o) and _same_bits(lse2, lse), f"{what}: the forward differs between calls"
    d1, d2 = _grads(dqkv, B, T, H), _grads(gd.t, B, T, H)
    assert _same_bits(d2["dk"], d1["dk"]) and _same_bits(d2["dv"], d1["dv"]), \
        f"{what}: dK / dV differ from the first call (0xFF workspace, offset buffers)"
    _check_dq(d2["dq"], d1["dq"], ref, T, what + " (second call)")


def test_workspace_reused_across_shapes(ops):
    """One workspace, sized for the largest shape and starting as 0xFF, serves smaller shapes in turn (the engine
    keeps one attn_ws for every layer); each result repeats that shape's run on a fresh workspace."""
    shapes = [(16, 577, 12), (2, 577, 12), (2, 197, 12), (1, 129, 3), (2, 17, 2), (3, 1, 4)]
    ws = torch.full((max(ops.attn_bwd_workspace_bytes(*s) for s in shapes),), 0xFF, dtype=u8, device=dev)
    for B, T, H in shapes:
        what = f"reused workspace B{B}-T{T}-H{H}"
        qkv, do = _inputs(B, T, H, 0.125, "randn")
        o, lse = ops.attn_fwd(qkv, B, T, H, 0.125)
        fresh = _grads(ops.attn_bwd(qkv, o, do.view(B * T, -1), lse, B, T, H, 0.125), B, T, H)
        reused = _grads(ops.attn_bwd(qkv, o, do.view(B * T, -1), lse, B, T, H, 0.125, workspace=ws), B, T, H)
        torch.cuda.synchronize()
        assert _same_bits(reused["dk"], fresh["dk"]) and _same_bits(reused["dv"], fresh["dv"]), what
        _check_dq(reused["dq"], fresh["dq"], A.reference(qkv, do, 0.125), T, what)


def _items_shape(items, T):
    """(B, T, H) with ⌈T/128⌉·H·B = items work items of attn_bwd."""
    nq = -(-T // 128)
    assert items % nq == 0
    n = items // nq
    H = max(h for h in range(1, 33) if n % h == 0)
    return n // H, T, H


@pytest.mark.parametrize("which", ["1", "sms-1", "sms", "sms+1", "2sms+1", "many"])
def test_work_items_around_sm_count(ops, which):
    """The persistent backward's grid is min(items, SMs) CTAs drawing from a counter: one item, a grid one short of /
    exactly / one past the SM count, two rounds plus one (T = 300: a CTA walks items of three key blocks), and ≫ SMs."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    items = {"1": 1, "sms-1": sms - 1, "sms": sms, "sms+1": sms + 1, "2sms+1": 2 * sms + 1}.get(which)
    if items is None:
        B, T, H = 32, 577, 12
    else:
        B, T, H = _items_shape(items, 300 if which == "2sms+1" and items % 3 == 0 else 100)
    what = f"{which} (B{B}-T{T}-H{H}, {-(-T // 128) * H * B} items, {sms} SMs)"
    qkv, do = _inputs(B, T, H, 0.125, "randn")
    ref = A.reference(qkv, do, 0.125)
    o, lse = ops.attn_fwd(qkv, B, T, H, 0.125)
    dqkv = ops.attn_bwd(qkv, o, do.view(B * T, -1), lse, B, T, H, 0.125)
    torch.cuda.synchronize()
    _check({"o": o, **_grads(dqkv, B, T, H)}, ref, what)
    _check_lse(lse, ref, what)


def _prepared(ops, B, T, H, scale=0.125, family="randn"):
    """Inputs, forward, reference and an uncontended backward of one case, plus zeroed output / workspace buffers."""
    qkv, do = _inputs(B, T, H, scale, family)
    o, lse = ops.attn_fwd(qkv, B, T, H, scale)
    base = ops.attn_bwd(qkv, o, do.view(B * T, -1), lse, B, T, H, scale)
    c = dict(B=B, T=T, H=H, scale=scale, qkv=qkv, do=do.view(B * T, -1), o=o, lse=lse, base=base,
             ref=A.reference(qkv, do, scale), out=torch.zeros_like(base),
             ws=torch.zeros(ops.attn_bwd_workspace_bytes(B, T, H), dtype=u8, device=dev))
    torch.cuda.synchronize()
    return c


def _launch(ops, c):
    ops.attn_bwd(c["qkv"], c["o"], c["do"], c["lse"], c["B"], c["T"], c["H"], c["scale"], c["out"], c["ws"])


def _check_contended(c, what):
    got, base = _grads(c["out"], c["B"], c["T"], c["H"]), _grads(c["base"], c["B"], c["T"], c["H"])
    assert _same_bits(got["dk"], base["dk"]) and _same_bits(got["dv"], base["dv"]), f"{what}: dK / dV differ"
    _check({"dq": got["dq"]}, c["ref"], what, names=("dq",))


def test_bwd_on_two_streams_at_once(ops):
    """Two backward passes with their own workspaces, launched on two streams without waiting on each other: whichever
    way their CTAs share the SMs, each result is that of its uncontended run."""
    cases = [_prepared(ops, 16, 577, 12), _prepared(ops, 8, 197, 12, 0.3, "onehot")]
    streams = [torch.cuda.Stream() for _ in cases]
    for s, c in zip(streams, cases):
        with torch.cuda.stream(s):
            _launch(ops, c)
    torch.cuda.synchronize()
    for i, c in enumerate(cases):
        _check_contended(c, f"stream {i}")


def test_bwd_beside_persistent_gemm(ops):
    """The backward launched while a persistent GEMM capped below the SM count (several ms of work) holds SMs on a side
    stream: its CTAs start late or not at all on those SMs, and the work-item draw must still give the same result."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    c = _prepared(ops, 16, 577, 12)
    M, N, K = 16384, 16384, 8192
    g = torch.Generator(device=dev).manual_seed(7)
    a = torch.randn(M, K, generator=g, device=dev).to(bf16)
    b = torch.randn(N, K, generator=g, device=dev).to(bf16)
    d = torch.empty(M, N, dtype=bf16, device=dev)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        ops.gemm(a, b, M, N, K, d, epilogue=ops.EPI_STORE_BF16, max_ctas=sms // 2)
    _launch(ops, c)
    torch.cuda.synchronize()
    _check_contended(c, "beside a GEMM")


def test_pdl_chain_on_a_side_stream(ops):
    """QKV GEMM → attn_fwd → a torch op writing do → attn_bwd on one fresh stream with no synchronisation in between
    (programmatic dependent launches inside the library, an ordinary kernel between them) gives what the same chain
    gives with a device synchronise after every launch."""
    B, T, H, scale = 2, 197, 12, 0.125
    D = H * A.DH
    g = torch.Generator(device=dev).manual_seed(11)
    x = torch.randn(B * T, D, generator=g, device=dev).to(bf16)
    w = (torch.randn(3 * D, D, generator=g, device=dev) * 0.05).to(bf16)
    bias = torch.randn(3 * D, generator=g, device=dev) * 0.1
    gain = (torch.randn(B * T, D, generator=g, device=dev) * 0.1).to(bf16)

    def chain(sync):
        qkv = torch.empty(B * T, 3 * D, dtype=bf16, device=dev)
        o, do = torch.empty(B * T, D, dtype=bf16, device=dev), torch.empty(B * T, D, dtype=bf16, device=dev)
        lse = torch.empty(B, H, T, device=dev)
        dqkv = torch.empty(B * T, 3 * D, dtype=bf16, device=dev)
        ws = torch.zeros(ops.attn_bwd_workspace_bytes(B, T, H), dtype=u8, device=dev)
        steps = [lambda: ops.gemm(x, w, B * T, 3 * D, D, qkv, epilogue=ops.EPI_BIAS_BF16, bias=bias),
                 lambda: ops.attn_fwd(qkv, B, T, H, scale, o, lse),
                 lambda: torch.mul(o, gain, out=do),
                 lambda: ops.attn_bwd(qkv, o, do, lse, B, T, H, scale, dqkv, ws)]
        torch.cuda.synchronize()
        with torch.cuda.stream(torch.cuda.Stream()):
            for step in steps:
                step()
                if sync:
                    torch.cuda.synchronize()
        torch.cuda.synchronize()
        return {"qkv": qkv, "o": o, "lse": lse, "do": do, **_grads(dqkv, B, T, H)}

    want, got = chain(True), chain(False)
    for k in ("qkv", "o", "lse", "do", "dk", "dv"):
        assert _same_bits(got[k], want[k]), f"{k} differs from the synchronised chain"
    ref = A.reference(got["qkv"].view(B, T, 3, H, A.DH), got["do"], scale)
    _check_dq(got["dq"], want["dq"], ref, T, "PDL chain")
    _check(got, ref, "PDL chain")


def test_attention_rejects_bad_arguments(ops):
    """Each bad call raises with the library's message and writes nothing."""
    import chest_x_ray_vit_b200 as pkg
    B, T, H, s = 2, 65, 3, 0.125
    qkv, do = _inputs(B, T, H, s, "randn")
    do = do.view(B * T, -1)
    o, lse = ops.attn_fwd(qkv, B, T, H, s)
    nbytes = ops.attn_bwd_workspace_bytes(B, T, H)
    out = {"o": Guarded(o.numel(), bf16), "lse": Guarded(lse.numel(), f32, offset=4), "dqkv": Guarded(qkv.numel(), bf16),
           "ws": Guarded(nbytes, u8)}
    go, gl, gd, gw = (out[k].t for k in ("o", "lse", "dqkv", "ws"))
    calls = {
        "attn_fwd": lambda q=qkv, o_=go, b=B, t=T, h=H, sc=s: ops.attn_fwd(q, b, t, h, sc, o_, gl),
        "attn_bwd": lambda q=qkv, o_=o, d=do, dq=gd, w=gw, b=B, t=T, h=H, sc=s:
            ops.attn_bwd(q, o_, d, lse, b, t, h, sc, dq, w),
        "attn_cls_fwd": lambda q=qkv, o_=go, b=B, t=T, h=H, sc=s: ops.attn_cls_fwd(q, b, t, h, sc, o_, gl),
        "attn_cls_bwd": lambda q=qkv, o_=o, d=do, dq=gd, b=B, t=T, h=H, sc=s: ops.attn_cls_bwd(q, o_, d, lse, b, t, h, sc, dq),
    }
    for name, call in calls.items():
        for bad in (dict(b=0), dict(t=0), dict(h=0), dict(t=1 << 24)):
            with pytest.raises(RuntimeError, match="unsupported shape"):
                call(**bad)
        for sc in (0.0, -0.125, math.nan):
            with pytest.raises(RuntimeError, match="scale"):
                call(sc=sc)
    with pytest.raises(RuntimeError, match="unsupported shape"):
        calls["attn_cls_fwd"](t=4097)
    with pytest.raises(RuntimeError, match="unsupported shape"):
        calls["attn_cls_bwd"](t=4097)
    # one pointer at a time 8 bytes past a 16-byte boundary
    mis = {"q": Guarded(qkv.numel(), bf16, 8, qkv).t, "o_": Guarded(o.numel(), bf16, 8, o).t,
           "d": Guarded(do.numel(), bf16, 8, do).t, "dq": Guarded(qkv.numel(), bf16, 8).t, "w": Guarded(nbytes, u8, 8).t}
    for name, args in (("attn_fwd", ("q", "o_")), ("attn_bwd", ("q", "o_", "d", "dq", "w")), ("attn_cls_fwd", ("q", "o_")),
                       ("attn_cls_bwd", ("q", "o_", "d", "dq"))):
        for a in args:
            with pytest.raises(RuntimeError, match="aligned"):
                calls[name](**{a: mis[a]})
    L = pkg._lib.lib()
    rc = L.vitk_attn_bwd(qkv.data_ptr(), o.data_ptr(), do.data_ptr(), lse.data_ptr(), B, T, H, s, gd.data_ptr(), None,
                         torch.cuda.current_stream().cuda_stream)
    assert rc != 0 and b"NULL" in L.vitk_last_error()
    torch.cuda.synchronize()
    for k, g in out.items():
        assert g.untouched(), f"a rejected call wrote into {k}"


# ---------------------------------------------------------------------------------------------------- CLS-row kernels
CLS_CASES = [(2, 17, 2, 0.125, "randn"), (3, 197, 12, 0.125, "randn"), (2, 577, 12, 0.125, "randn"),
             (1, 1024, 3, 0.125, "randn"), (3, 1, 12, 0.3, "randn"), (2, 2, 1, 0.125, "onehot"), (2, 577, 16, 0.3, "x4"),
             (1, 577, 12, 0.125, "jumps"), (1, 4096, 12, 0.125, "onehot"), (2, 4096, 1, 0.3, "x4"),
             (1, 4096, 16, 0.3, "randn")]


@pytest.mark.parametrize("B,T,H,scale,family", CLS_CASES, ids=[A.case_id(*c) for c in CLS_CASES])
def test_cls_row_attention_matches_dense_and_fp32(ops, B, T, H, scale, family):
    """Top-layer kernels (one query per head) with a gradient on token 0 only: row 0 of o / lse, and dense dK / dV with
    dQ on token 0, against the oracle row by row; the dense kernels on the same input as well.  o / lse / dqkv live in
    guarded NaN buffers: o and lse get row 0 only, dqkv every element (dQ exactly zero off token 0), nothing outside."""
    what = "CLS " + A.case_id(B, T, H, scale, family)
    qkv, do_full = _inputs(B, T, H, scale, family)
    do = torch.zeros_like(do_full)
    do[:, 0] = do_full[:, 0]
    ref = A.reference(qkv, do, scale)
    go, gl = Guarded(B * T * H * A.DH, bf16), Guarded(B * H * T, f32, offset=4)
    ops.attn_cls_fwd(qkv, B, T, H, scale, go.t, gl.t)
    torch.cuda.synchronize()
    o, lse = go.t.view(B, T, H, A.DH), gl.t.view(B, H, T)
    assert go.intact() and gl.intact()
    assert torch.isnan(o[:, 1:].float()).all() and torch.isnan(lse[:, :, 1:]).all(), f"{what}: a row other than 0 written"
    _check({"o": o}, ref, what + " fwd", names=("o",), tokens=slice(0, 1))
    _check_lse(lse, ref, what, tokens=slice(0, 1))
    gd = Guarded(qkv.numel(), bf16)
    ops.attn_cls_bwd(qkv, go.t, do.view(B * T, -1), gl.t, B, T, H, scale, gd.t)
    torch.cuda.synchronize()
    assert gd.intact(), f"{what}: a byte around dqkv was written"
    assert torch.isfinite(gd.t.float()).all(), f"{what}: a dqkv element left unwritten"
    got = _grads(gd.t, B, T, H)
    assert (got["dq"][:, 1:] == 0).all(), f"{what}: dQ is not zero off the CLS row"
    _check(got, ref, what + " bwd", names=("dq", "dk", "dv"))

    o_d, lse_d = ops.attn_fwd(qkv, B, T, H, scale)
    dense = ops.attn_bwd(qkv, o_d, do.view(B * T, -1), lse_d, B, T, H, scale)
    torch.cuda.synchronize()
    _check({"o": o_d, **_grads(dense, B, T, H)}, ref, what + " dense kernels")
    _check_lse(lse_d, ref, what + " dense kernels")
