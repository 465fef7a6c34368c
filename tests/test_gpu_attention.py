"""Fused attention forward/backward through the C ABI vs fp32 softmax(QKᵀ·s)·V with autograd."""
import pytest
import torch

pytestmark = pytest.mark.gpu
dev = "cuda"
bf16 = torch.bfloat16


@pytest.fixture(scope="module")
def ops():
    import chest_x_ray_vit_b200 as pkg
    pkg.ops.check_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    return pkg.ops


def _ref(qkv, do, scale):
    B, T, _, H, dh = qkv.shape
    x = qkv.float().requires_grad_(True)
    q, k, v = (x[:, :, i].transpose(1, 2) for i in range(3))      # [B,H,T,dh]
    s = (q @ k.transpose(-1, -2)) * scale
    lse = torch.logsumexp(s, dim=-1)
    o = (torch.softmax(s, dim=-1) @ v).transpose(1, 2).reshape(B, T, H * dh)
    o.backward(do.float())
    return o.detach(), lse.detach(), x.grad


# T covers: one partial tile (17, 64), one full tile, pair + narrow last key block (129, 197), a pair exactly (256), two pairs
# (300 → 3 tiles = pair + single; 385 → 4 tiles), the model's 577 (2 pairs + single, 65-key tail), 5 full tiles (640) and
# 8 key blocks (1024: the 3-deep K/V ring is recycled)
@pytest.mark.parametrize("B,T,H", [(1, 128, 1), (1, 64, 2), (2, 17, 2), (2, 129, 3), (2, 197, 12), (1, 256, 2), (2, 577, 12),
                                   (1, 300, 16), (1, 385, 2), (1, 640, 2), (1, 1024, 1), (16, 577, 12),
                                   (1, 130, 6), (1, 70, 20),       # head counts of every attn_delta instantiation (≤4, ≤8, ≤12, ≤16, >16)
                                   (2, 129, 20)])                  # H > 16 (attn_delta_kernel) with two images and two key blocks
def test_attention_fwd_bwd(ops, B, T, H):
    g = torch.Generator().manual_seed(T * 10 + H)
    qkv = (torch.randn(B, T, 3, H, 64, generator=g)).to(dev).to(bf16)
    do = (torch.randn(B, T, H * 64, generator=g) * 0.1).to(dev).to(bf16)
    scale = 0.125
    o_ref, lse_ref, dqkv_ref = _ref(qkv, do, scale)
    o, lse = ops.attn_fwd(qkv, B, T, H, scale)
    torch.cuda.synchronize()
    assert (o.view(B, T, -1).float() - o_ref).abs().max() <= 2e-2 * o_ref.abs().max()
    assert torch.allclose(lse, lse_ref, atol=2e-3, rtol=1e-4)
    dqkv = ops.attn_bwd(qkv, o, do.view(B * T, -1), lse, B, T, H, scale)
    torch.cuda.synchronize()
    got = dqkv.view(B, T, 3, H, 64).float()
    for i, name in enumerate("qkv"):
        r = dqkv_ref[:, :, i]
        err = (got[:, :, i] - r).abs().max().item()
        cos = torch.nn.functional.cosine_similarity(got[:, :, i].flatten(), r.flatten(), dim=0).item()
        assert err <= 3e-2 * r.abs().max().item() and cos > 0.9995, f"d{name}: err {err} cos {cos}"


def test_attention_large_logits(ops):
    """Rows dominated by one key (large scores) must not overflow the online softmax."""
    B, T, H = 1, 577, 2
    g = torch.Generator().manual_seed(0)
    qkv = (torch.randn(B, T, 3, H, 64, generator=g) * 4).to(dev).to(bf16)
    do = torch.randn(B, T, H * 64, generator=g).to(dev).to(bf16)
    o_ref, lse_ref, _ = _ref(qkv, do, 0.125)
    o, lse = ops.attn_fwd(qkv, B, T, H, 0.125)
    assert torch.isfinite(o.float()).all()
    assert (o.view(B, T, -1).float() - o_ref).abs().max() <= 3e-2 * o_ref.abs().max()
    assert torch.allclose(lse, lse_ref, atol=2e-2, rtol=1e-3)


def test_attention_reference_maximum_jumps(ops):
    """Later key blocks whose scores exceed the first block's maximum by far more than the lazy
    threshold (2^16), including jumps past the fp32 exponent range, must rescale exactly."""
    B, T, H = 1, 577, 1
    g = torch.Generator().manual_seed(4)
    qkv = torch.randn(B, T, 3, H, 64, generator=g)
    qkv[:, :, 0] *= 3.0
    qkv[:, 200:, 1] *= 6.0           # keys of blocks 1..4 produce much larger scores
    qkv[:, 400:, 1] *= 8.0
    qkv = qkv.to(dev).to(bf16)
    do = torch.randn(B, T, H * 64, generator=g).to(dev).to(bf16)
    o_ref, lse_ref, _ = _ref(qkv, do, 0.125)
    o, lse = ops.attn_fwd(qkv, B, T, H, 0.125)
    assert torch.isfinite(o.float()).all() and torch.isfinite(lse).all()
    assert (o.view(B, T, -1).float() - o_ref).abs().max() <= 3e-2 * o_ref.abs().max()
    assert torch.allclose(lse, lse_ref, atol=5e-2, rtol=2e-3)


@pytest.mark.parametrize("B,T,H", [(2, 17, 2), (3, 197, 12), (2, 577, 12), (1, 1024, 3)])
def test_cls_row_attention_matches_dense_and_fp32(ops, B, T, H):
    """Top-layer kernels (one query per head): forward against the dense flash kernel's row 0 and the fp32 reference,
    backward against the dense backward fed a gradient that is zero except on the CLS rows."""
    g = torch.Generator().manual_seed(100 + T + H)
    qkv = torch.randn(B, T, 3, H, 64, generator=g).to(dev).to(bf16)
    scale = 0.125
    do = torch.zeros(B, T, H * 64)
    do[:, 0] = torch.randn(B, H * 64, generator=g) * 0.1
    do = do.to(dev).to(bf16)
    o_ref, lse_ref, dqkv_ref = _ref(qkv, do, scale)
    o_dense, lse_dense = ops.attn_fwd(qkv, B, T, H, scale)
    o = torch.full((B * T, H * 64), float("nan"), dtype=bf16, device=dev)        # rows other than CLS must not be needed
    lse = torch.full((B, H, T), float("nan"), device=dev)
    ops.attn_cls_fwd(qkv, B, T, H, scale, o, lse)
    torch.cuda.synchronize()
    oc = o.view(B, T, -1)[:, 0].float()
    assert (oc - o_ref[:, 0]).abs().max() <= 2e-2 * o_ref[:, 0].abs().max()
    assert (oc - o_dense.view(B, T, -1)[:, 0].float()).abs().max() <= 2e-2 * o_ref[:, 0].abs().max()
    assert torch.allclose(lse[:, :, 0], lse_ref[:, :, 0], atol=2e-3, rtol=1e-4)
    assert torch.isnan(o.view(B, T, -1)[:, 1:].float()).all() and torch.isnan(lse[:, :, 1:]).all()      # nothing else written
    dqkv = ops.attn_cls_bwd(qkv, o, do.view(B * T, -1), lse, B, T, H, scale)
    dense = ops.attn_bwd(qkv, o_dense, do.view(B * T, -1), lse_dense, B, T, H, scale).view(B, T, 3, H, 64).float()
    torch.cuda.synchronize()
    got = dqkv.view(B, T, 3, H, 64).float()
    assert got[:, 1:, 0].abs().max() == 0                                       # dQ is zero off the CLS row
    for i, name in enumerate("qkv"):
        r = dqkv_ref[:, :, i]
        err = (got[:, :, i] - r).abs().max().item()
        cos = torch.nn.functional.cosine_similarity(got[:, :, i].flatten(), r.flatten(), dim=0).item()
        assert err <= 3e-2 * r.abs().max().item() and cos > 0.9995, f"d{name} vs fp32: err {err} cos {cos}"
        cosd = torch.nn.functional.cosine_similarity(got[:, :, i].flatten(), dense[:, :, i].flatten(), dim=0).item()
        assert cosd > 0.9995, f"d{name} vs dense kernel: cos {cosd}"
