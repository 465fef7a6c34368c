"""Fused final-LN + classifier + BCEWithLogits (+ gradients) vs fp32 PyTorch autograd."""
import pytest
import torch

pytestmark = pytest.mark.gpu
dev = "cuda"


@pytest.fixture(scope="module")
def ops():
    import chest_x_ray_vit_b200 as pkg
    return pkg.ops


@pytest.mark.parametrize("B,T,D,C", [(2, 5, 768, 14), (16, 577, 768, 14), (3, 2, 1024, 15), (1, 1, 128, 1),
                                     (2, 3, 8192, 64)])     # the largest D and C the kernels accept
def test_head_fwd_bwd(ops, B, T, D, C):
    g = torch.Generator().manual_seed(B + C)
    h = torch.randn(B, T, D, generator=g).to(dev)
    gamma = (1 + 0.05 * torch.randn(D, generator=g)).to(dev)
    beta = (0.02 * torch.randn(D, generator=g)).to(dev)
    Wc = (0.02 * torch.randn(C, D, generator=g)).to(dev)
    bc = (0.02 * torch.randn(C, generator=g)).to(dev)
    y = (torch.rand(B, C, generator=g) < 0.3).float().to(dev)
    hr, gr, br, wr, cr = (t.clone().requires_grad_(True) for t in (h, gamma, beta, Wc, bc))
    z = torch.nn.functional.layer_norm(hr, (D,), gr, br, 1e-12)[:, 0]
    lr = z @ wr.t() + cr
    loss_r = torch.nn.functional.binary_cross_entropy_with_logits(lr, y)
    (loss_r * 0.5).backward()

    logits = torch.empty(B, C, device=dev)
    loss = torch.empty(1, device=dev)
    dlog = torch.empty(B, C, device=dev)
    mean, rstd = torch.empty(B, device=dev), torch.empty(B, device=dev)
    ops.head_fwd(h, B, T, D, C, gamma, beta, 1e-12, Wc, bc, y, logits, loss, dlog, mean, rstd)
    assert torch.allclose(logits, lr, atol=1e-5)
    assert torch.allclose(loss[0], loss_r, rtol=1e-5)
    dh = torch.zeros(B, T, D, device=dev, dtype=torch.bfloat16)
    dW, db, dg, dbt = (torch.zeros_like(t) for t in (Wc, bc, gamma, beta))
    dloss = torch.full((1,), 0.5, device=dev)
    ops.head_bwd(h, mean, rstd, gamma, beta, Wc, B, T, D, C, dlog, dloss, dh, dW, db, dg, dbt)
    assert torch.allclose(dW, wr.grad, atol=1e-6, rtol=1e-4)
    assert torch.allclose(db, cr.grad, atol=1e-7, rtol=1e-4)
    assert torch.allclose(dg, gr.grad, atol=1e-6, rtol=1e-3)
    assert torch.allclose(dbt, br.grad, atol=1e-6, rtol=1e-3)
    assert (dh[:, 0].float() - hr.grad[:, 0]).abs().max() <= 2 ** -7 * hr.grad[:, 0].abs().max()
    assert dh[:, 1:].abs().max() == 0 if T > 1 else True
    # inference: no labels
    logits2 = torch.empty(B, C, device=dev)
    ops.head_fwd(h, B, T, D, C, gamma, beta, 1e-12, Wc, bc, None, logits2, None, None, None, None)
    assert torch.equal(logits2, logits)
