"""HBM-bound kernels through the C ABI vs fp32 PyTorch / the oracle.  Needs a B200."""
import pytest
import torch

from oracle import vit_oracle as O

pytestmark = pytest.mark.gpu
dev = "cuda"


@pytest.fixture(scope="module")
def ops():
    import chest_x_ray_vit_b200 as pkg
    pkg.ops.check_device(0)
    return pkg.ops


@pytest.mark.parametrize("B,S", [(1, 16), (2, 64), (3, 384)])
@pytest.mark.parametrize("norm", [((0.5, 0.5, 0.5), (0.5, 0.5, 0.5)), ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))])
def test_patchify_u8_bit_exact(ops, B, S, norm):
    g = torch.Generator().manual_seed(B * 1000 + S)
    x8 = torch.randint(0, 256, (B, S, S), dtype=torch.uint8, generator=g)
    ref = O.im2col(O.normalize_gray(x8, *norm), 16).reshape(-1, 768).to(torch.bfloat16)
    got = ops.patchify_u8(x8.to(dev), *norm)
    torch.cuda.synchronize()
    assert torch.equal(got.cpu().view(torch.int16), ref.view(torch.int16))


@pytest.mark.parametrize("B,S", [(1, 32), (2, 384)])
def test_patchify_f32_bit_exact(ops, B, S):
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, 3, S, S, generator=g)
    ref = O.im2col(x, 16).reshape(-1, 768).to(torch.bfloat16)
    got = ops.patchify_f32(x.to(dev))
    assert torch.equal(got.cpu().view(torch.int16), ref.view(torch.int16))


@pytest.mark.parametrize("M,D", [(1, 768), (13, 768), (1154, 768), (9232, 768), (65, 128), (300, 1024), (300, 256), (77, 512)])
def test_layernorm_fwd_bwd(ops, M, D):
    g = torch.Generator().manual_seed(M + D)
    x = (torch.randn(M, D, generator=g) * 1.7 + 0.3).to(dev)
    gamma = (1 + 0.05 * torch.randn(D, generator=g)).to(dev)
    beta = (0.02 * torch.randn(D, generator=g)).to(dev)
    dy = torch.randn(M, D, generator=g).to(dev).to(torch.bfloat16)
    dres = torch.randn(M, D, generator=g).to(dev).to(torch.bfloat16)
    eps = 1e-12
    xr = x.clone().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    yr = torch.nn.functional.layer_norm(xr, (D,), gr, br, eps)
    yr.backward(dy.float())
    y, mean, rstd = ops.layernorm_fwd(x, gamma, beta, eps)
    assert (y.float() - yr).abs().max() <= 2 ** -8 * yr.abs().max() + 1e-6     # one bf16 rounding
    assert torch.allclose(mean, x.mean(1), atol=1e-5)
    assert torch.allclose(rstd, torch.rsqrt(x.var(1, unbiased=False) + eps), rtol=1e-4)
    dgamma = torch.zeros(D, device=dev)
    dbeta = torch.zeros(D, device=dev)
    dxsum = torch.ones(D, device=dev)
    dx = ops.layernorm_bwd(dy, x, mean, rstd, gamma, dres, dgamma, dbeta, dxsum=dxsum)
    ref_dx = xr.grad + dres.float()
    assert torch.allclose(dxsum, 1 + dx.float().sum(0), rtol=1e-4, atol=1e-3 * max(1.0, M ** 0.5))
    assert (dx.float() - ref_dx).abs().max() <= 2 ** -7 * ref_dx.abs().max() + 1e-5
    assert torch.allclose(dgamma, gr.grad, rtol=2e-4, atol=2e-4 * gr.grad.abs().max().item())
    assert torch.allclose(dbeta, br.grad, rtol=2e-4, atol=2e-4 * br.grad.abs().max().item())
    # dres = NULL and accumulation into dgamma/dbeta
    dx2 = ops.layernorm_bwd(dy, x, mean, rstd, gamma, None, dgamma, dbeta)
    assert (dx2.float() - xr.grad).abs().max() <= 2 ** -7 * xr.grad.abs().max() + 1e-5
    assert torch.allclose(dgamma, 2 * gr.grad, rtol=2e-4, atol=4e-4 * gr.grad.abs().max().item())


def test_layernorm_strided_rows(ops):
    """Final LayerNorm reads only the CLS rows: ldx = T·D."""
    g = torch.Generator().manual_seed(3)
    h = torch.randn(4, 5, 768, generator=g).to(dev)
    gamma, beta = torch.ones(768, device=dev), torch.zeros(768, device=dev)
    y, _, _ = ops.layernorm_fwd(h.view(4, 5 * 768)[:, :768], gamma, beta, 1e-12)
    ref = torch.nn.functional.layer_norm(h[:, 0], (768,), gamma, beta, 1e-12)
    assert (y.float() - ref).abs().max() < 0.02


@pytest.mark.parametrize("M,N,row_stride", [pytest.param(M, N, 1, id=f"{M}-{N}") for M, N in
                                              [(1, 8), (577, 768), (9232, 2304), (1000, 3072), (50, 264)]] +
                         [(16, 768, 577), (3, 3072, 197), (1, 1024, 577)])
def test_colsum(ops, M, N, row_stride):
    """row_stride > 1: x is every row_stride-th row of a larger buffer whose other rows are NaN (the bias gradients
    of the top layer sum the B CLS rows of a [B·T, N] buffer, ldx = T·N)."""
    g = torch.Generator().manual_seed(M)
    x = torch.randn(M, N, generator=g).to(dev).to(torch.bfloat16)
    if row_stride > 1:
        buf = torch.full((M * row_stride, N), float("nan"), device=dev, dtype=torch.bfloat16)
        buf[::row_stride] = x
        x = buf.view(M, row_stride * N)[:, :N]
    out = torch.ones(N, device=dev)
    ops.colsum(x, out)
    ref = 1 + x.double().sum(0)
    assert torch.allclose(out.double(), ref, atol=1e-3 * max(1.0, M ** 0.5))


def test_embed_cls_and_bwd(ops):
    B, T, D = 3, 17, 768
    g = torch.Generator().manual_seed(0)
    cls, pos = torch.randn(D, generator=g).to(dev), torch.randn(T, D, generator=g).to(dev)
    h = torch.zeros(B, T, D, device=dev)
    ops.embed_cls(cls, pos, B, T, D, h)
    assert torch.equal(h[:, 0], (cls + pos[0]).expand(B, D))
    assert h[:, 1:].abs().max() == 0
    dh = torch.randn(B, T, D, generator=g).to(dev).to(torch.bfloat16)
    dpos, dcls, dbias = torch.zeros(T, D, device=dev), torch.zeros(D, device=dev), torch.zeros(D, device=dev)
    dpatch = torch.empty(B * (T - 1), D, dtype=torch.bfloat16, device=dev)
    ops.embed_bwd(dh, B, T, D, dpos, dcls, dbias, dpatch)
    f = dh.float()
    assert torch.allclose(dpos, f.sum(0), atol=1e-5)
    assert torch.allclose(dcls, f[:, 0].sum(0), atol=1e-5)
    assert torch.allclose(dbias, f[:, 1:].sum((0, 1)), atol=1e-4)
    assert torch.equal(dpatch.view(B, T - 1, D), dh[:, 1:])


def test_cast_and_adamw(ops):
    n = 4 * 1000 + 8
    g = torch.Generator().manual_seed(0)
    p = torch.randn(n, generator=g).to(dev)
    p16 = torch.empty(n, dtype=torch.bfloat16, device=dev)
    ops.cast_f32_bf16(p, p16)
    assert torch.equal(p16, p.to(torch.bfloat16))
    ref = p.clone().requires_grad_(True)
    opt = torch.optim.AdamW([ref], lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)
    m, v = torch.zeros(n, device=dev), torch.zeros(n, device=dev)
    for t in range(1, 4):
        grad = torch.randn(n, generator=g).to(dev)
        ref.grad = grad.clone()
        opt.step()
        gcopy = grad.clone()
        ops.adamw(p, gcopy, m, v, p16, n, 1e-3, 0.9, 0.999, 1e-8, 0.01, 1 - 0.9 ** t, 1 - 0.999 ** t, zero_grad=(t == 2))
        assert torch.equal(gcopy, torch.zeros_like(grad) if t == 2 else grad)
        assert torch.allclose(p, ref.detach(), atol=2e-6, rtol=1e-5)
        assert torch.equal(p16, p.to(torch.bfloat16))
    # global-norm clip scale
    ss, sc = torch.zeros(1, device=dev), torch.zeros(1, device=dev)
    ops.sumsq(grad, ss)
    assert torch.allclose(ss, (grad.double() ** 2).sum().float(), rtol=1e-5)
    ops.clip_scale(ss, 1.0, sc)
    assert torch.allclose(sc, 1.0 / (grad.norm() + 1e-6), rtol=1e-5)


def test_sumsq_is_bit_reproducible_and_accumulates(ops):
    """Fixed summation order: replicas with identical gradients must get identical clip coefficients."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(86_101_264 // 8 * 8, generator=g).to(dev)            # the size of ViT-B's flat gradient buffer
    outs = []
    for _ in range(6):
        ss = torch.zeros(1, device=dev)
        ops.sumsq(x, ss)
        outs.append(ss.item())
    assert len(set(outs)) == 1, outs
    assert abs(outs[0] / (x.double() ** 2).sum().item() - 1) < 1e-5
    ss = torch.zeros(1, device=dev)
    ops.sumsq(x[:1024], ss)
    ops.sumsq(x[1024:4096], ss)
    assert torch.allclose(ss, (x[:4096].double() ** 2).sum().float(), rtol=1e-5)


def test_adamw_tick_device_step_counter(ops):
    step = torch.zeros(1, dtype=torch.int64, device=dev)
    bc = torch.zeros(2, device=dev)
    for t in range(1, 4):
        ops.adamw_tick(step, True, 0.9, 0.999, bc)
        assert step.item() == t
        assert torch.allclose(bc.cpu(), torch.tensor([1 - 0.9 ** t, (1 - 0.999 ** t) ** -0.5]), rtol=1e-5)
    ops.adamw_tick(step, False, 0.9, 0.999, bc)
    assert step.item() == 3


@pytest.mark.parametrize("B,H,W", [(5, 384, 384), (3, 224, 224), (2, 48, 48), (4, 16, 16), (2, 32, 80)])
def test_hflip_u8_is_the_mirror(ops, B, H, W):
    """RandomHorizontalFlip on the device: masked images are mirrored along W (even and odd numbers of 16-byte chunks per
    row), the others untouched — bit for bit what torch.flip / PIL's FLIP_LEFT_RIGHT gives before ToTensor+Normalize."""
    g = torch.Generator().manual_seed(B * 100 + W)
    x8 = torch.randint(0, 256, (B, H, W), dtype=torch.uint8, generator=g)
    mask = (torch.arange(B) % 2 == 0).to(torch.uint8)
    ref = torch.where(mask.bool()[:, None, None], torch.flip(x8, dims=[-1]), x8)
    d = x8.to(dev)
    out = ops.hflip_u8(d, mask.to(dev))
    assert out.data_ptr() == d.data_ptr() and torch.equal(d.cpu(), ref)
    ops.hflip_u8(d, torch.ones(B, dtype=torch.bool, device=dev))          # all images, bool mask
    assert torch.equal(d.cpu(), torch.flip(ref, dims=[-1]))
    norm = ((0.5, 0.5, 0.5), (0.5, 0.5, 0.5))
    if H % 16 == 0:
        got = ops.patchify_u8(d, *norm)                                   # flip, then the usual transform = the reference's order
        want = O.im2col(O.normalize_gray(torch.flip(ref, dims=[-1]), *norm), 16).reshape(-1, 768).to(torch.bfloat16)
        assert torch.equal(got.cpu().view(torch.int16), want.view(torch.int16))


def test_device_feeder_random_hflip(ops):
    """DeviceFeeder(hflip_p=…): per-image masks from a seeded generator, applied on the copy stream; the fed batches are
    the host batches mirrored where the mask says so, labels untouched."""
    import chest_x_ray_vit_b200 as pkg
    g = torch.Generator().manual_seed(3)
    batches = [{"pixel_values": torch.randint(0, 256, (6, 64, 64), dtype=torch.uint8, generator=g),
                "labels": torch.rand(6, 14, generator=g)} for _ in range(5)]
    feeder = pkg.data.DeviceFeeder(batches, device=dev, hflip_p=0.5, generator=torch.Generator().manual_seed(11))
    ref_gen = torch.Generator().manual_seed(11)
    flipped = 0
    for host, fed in zip(batches, feeder):
        mask = torch.rand(6, generator=ref_gen) < 0.5
        want = torch.where(mask[:, None, None], torch.flip(host["pixel_values"], dims=[-1]), host["pixel_values"])
        torch.cuda.current_stream().synchronize()
        assert torch.equal(fed["pixel_values"].cpu(), want) and torch.equal(fed["labels"].cpu(), host["labels"])
        flipped += int(mask.sum())
    assert 0 < flipped < 30
    with pytest.raises(ValueError, match="uint8"):
        next(iter(pkg.data.DeviceFeeder([{"pixel_values": torch.zeros(2, 3, 32, 32)}], device=dev, hflip_p=0.5)))
