"""CPU-only: the oracle's ``interpolate_pos_encoding`` against live HF, the fp64 resize matrices against F.interpolate, and
the module's host-side checks of the flag."""
import pytest
import torch
import torch.nn.functional as F

import chest_x_ray_vit_b200 as pkg
from oracle import interp_oracle as I
from oracle import vit_oracle as O

TINY = dict(image_size=64, hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=256, num_labels=14)


def _rel(a, r):
    return ((a - r).abs().max() / r.abs().max()).item()


@pytest.mark.parametrize("H,W", [(48, 48), (96, 96), (64, 112), (112, 64)])
def test_oracle_with_flag_matches_live_hf(H, W):
    pytest.importorskip("transformers")
    from oracle.make_golden import hf_model
    cfg = O.TINY
    p = O.init_params(cfg, 3, 7)
    g = torch.Generator().manual_seed(H * 1000 + W)
    x = O.normalize_gray(torch.randint(0, 256, (3, 1, H, W), dtype=torch.uint8, generator=g))
    y = (torch.rand(3, cfg.num_labels, generator=g) < 0.3).float()
    hf, _ = hf_model(cfg, p)
    xr = x.clone().requires_grad_()
    out = hf(pixel_values=xr, labels=y, interpolate_pos_encoding=True)
    out.loss.backward()
    leaves = {k: v.detach().clone().requires_grad_() for k, v in p.items()}
    xo = x.clone().requires_grad_()
    loss, logits = I.forward(leaves, cfg, xo, y, interpolate_pos_encoding=True)
    loss.backward()
    assert (logits - out.logits).abs().max().item() <= 1e-5
    assert abs(loss.item() - out.loss.item()) <= 1e-6 * abs(out.loss.item())
    ref_grads = dict(hf.named_parameters())
    for k, v in leaves.items():
        r = ref_grads[k].grad
        assert v.grad.shape == r.shape, k
        if k.endswith("key.bias"):          # analytically zero: both are rounding noise
            assert v.grad.abs().max() <= 1e-6 and r.abs().max() <= 1e-6
            continue
        assert _rel(v.grad, r) <= 1e-4, (k, _rel(v.grad, r))
    pos_g = leaves["vit.embeddings.position_embeddings"].grad
    assert pos_g.shape == (1, cfg.seq_len, cfg.hidden_size) and pos_g.abs().max() > 0
    assert _rel(xo.grad, xr.grad) <= 1e-5
    # forward_backward takes the flag too, and without it stays the plain path
    l2, lg2, g2 = I.forward_backward(p, cfg, x, y, interpolate_pos_encoding=True)
    assert torch.equal(lg2, logits.detach()) and torch.equal(g2["vit.embeddings.position_embeddings"], pos_g)


def test_flag_at_the_config_size_is_the_plain_path():
    cfg = O.TINY
    p = O.init_params(cfg, 0, 123)
    x, y = O.synth_inputs(cfg, 2, torch.Generator().manual_seed(1))
    x = O.normalize_gray(x)
    assert torch.equal(I.forward(p, cfg, x, y, True)[1], O.forward(p, cfg, x, y)[1])
    assert torch.equal(I.forward(p, cfg, x, y)[1], O.forward(p, cfg, x, y)[1])
    pos = p["vit.embeddings.position_embeddings"]
    assert I.resize_pos(pos, 64, 64, 16) is pos
    # a grid with the same number of patches but another shape is resized, as in HF
    assert I.resize_pos(pos, 32, 128, 16).shape == pos.shape and not torch.equal(I.resize_pos(pos, 32, 128, 16), pos)


@pytest.mark.parametrize("n_in,n_out", [(24, 32), (24, 40), (24, 64), (14, 28), (4, 9), (24, 3), (24, 16), (14, 1), (24, 1),
                                        (4, 1), (1, 5), (24, 24), (4, 4)],
                         ids=lambda v: str(v))
def test_bicubic_matrix_matches_f_interpolate(n_in, n_out):
    g = torch.Generator().manual_seed(n_in * 100 + n_out)
    x = torch.randn(1, 3, n_in, n_in, dtype=torch.float64, generator=g)
    W = I.bicubic_matrix(n_in, n_out)
    assert W.shape == (n_out, n_in)
    ref = F.interpolate(x, size=(n_out, n_out), mode="bicubic", align_corners=False)
    got = torch.einsum("yi,ncij,xj->ncyx", W, x, W)
    assert (got - ref).abs().max().item() <= 1e-12
    if n_in == n_out:
        assert torch.equal(W, torch.eye(n_in, dtype=torch.float64))


@pytest.mark.parametrize("s,gh,gw", [(24, 32, 32), (24, 24, 40), (24, 40, 24), (14, 1, 9), (4, 3, 1), (24, 24, 24)])
def test_pos_interp_reference_matches_hf_resize_and_its_adjoint(s, gh, gw):
    D = 16
    g = torch.Generator().manual_seed(s + gh + gw)
    pos = torch.randn(1, 1 + s * s, D, dtype=torch.float64, generator=g)
    grid = pos[:, 1:].reshape(1, s, s, D).permute(0, 3, 1, 2)
    hf = F.interpolate(grid, size=(gh, gw), mode="bicubic", align_corners=False).permute(0, 2, 3, 1).reshape(-1, D)
    got = I.pos_interp(pos[0], s, s, gh, gw)
    assert torch.equal(got[0], pos[0, 0]) and (got[1:] - hf).abs().max().item() <= 1e-12
    # the adjoint against autograd of F.interpolate, and <R x, y> = <x, Rᵀ y>
    dout = torch.randn(1 + gh * gw, D, dtype=torch.float64, generator=g)
    leaf = pos.clone().requires_grad_()
    lg = leaf[:, 1:].reshape(1, s, s, D).permute(0, 3, 1, 2)
    r = torch.cat((leaf[0, :1], F.interpolate(lg, size=(gh, gw), mode="bicubic", align_corners=False)
                   .permute(0, 2, 3, 1).reshape(-1, D)))
    (ag,) = torch.autograd.grad(r, leaf, grad_outputs=dout)
    back = I.pos_interp_bwd(dout, gh, gw, s, s)
    assert (back - ag[0]).abs().max().item() <= 1e-12
    assert abs((got * dout).sum().item() - (pos[0] * back).sum().item()) <= 1e-9


def test_host_validation_of_the_flag():
    m = pkg.ViTForImageClassification(pkg.ViTConfig(**TINY))
    for x in (torch.zeros(1, 3, 72, 64), torch.zeros(1, 3, 64, 50), torch.zeros(1, 3, 0, 64), torch.zeros(1, 3, 64, 0),
              torch.zeros(1, 72, 64, dtype=torch.uint8), torch.zeros(1, 1, 64, 8, dtype=torch.uint8)):
        with pytest.raises(ValueError, match=r"interpolate_pos_encoding=True needs a height and width that are positive "
                                             r"multiples of 16"):
            m(pixel_values=x, interpolate_pos_encoding=True)
    # a valid size on a CPU-resident model names the flag, before the generic "no CPU path" error
    for x in (torch.zeros(1, 3, 96, 128), torch.zeros(1, 3, 64, 64), torch.zeros(2, 96, 96, dtype=torch.uint8)):
        with pytest.raises(ValueError, match=r"interpolate_pos_encoding=True runs on the CUDA kernel path only"):
            m(pixel_values=x, interpolate_pos_encoding=True)
    # without the flag (False or None) another size keeps HF's error
    for flag in (False, None):
        with pytest.raises(ValueError, match="doesn't match model"):
            m(pixel_values=torch.zeros(1, 3, 96, 96), interpolate_pos_encoding=flag)
    with pytest.raises(ValueError, match="channel dimension"):
        m(pixel_values=torch.zeros(1, 1, 96, 96), interpolate_pos_encoding=True)
