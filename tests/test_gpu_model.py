"""End-to-end parity of the drop-in module on a B200 against (a) the golden vectors frozen from
HF transformers 5.5.0 fp32 CPU and (b) the CPU oracle on the same seeded inputs.
Tolerances are BASELINE.json's north_star: logits max-abs <= 2e-2, loss rel <= 1e-3,
per-parameter gradient cosine >= 0.999 (key.bias gradients are analytically zero: magnitude
bound instead, SURVEY App. C.6)."""
import os

import pytest
import torch

from oracle import vit_oracle as O

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
LOGIT_TOL, LOSS_RTOL, COS_MIN = 2e-2, 1e-3, 0.999


def _model(cfg: O.OracleConfig, params):
    import chest_x_ray_vit_b200 as pkg
    c = pkg.ViTConfig(image_size=cfg.image_size, hidden_size=cfg.hidden_size, num_hidden_layers=cfg.num_hidden_layers,
                      num_attention_heads=cfg.num_attention_heads, intermediate_size=cfg.intermediate_size,
                      num_labels=cfg.num_labels)
    m = pkg.ViTForImageClassification(c)
    m.load_state_dict(params, strict=True)
    return m.cuda().train()


def _check_grads(m, ref_grads, rec=None):
    """``ref_grads``: whole reference gradients, or with ``rec`` (a golden record) its sampled ``grad_sample`` entries,
    whose cosine is taken over the kept elements and whose norms are the record's whole-tensor ``grad_norm``."""
    from oracle.make_golden import record_indices
    worst = (1.0, None)
    got = {k: p.grad.detach().float().cpu() for k, p in m.named_parameters()}
    for k, r in ref_grads.items():
        g = got[k]
        if k.endswith("key.bias"):
            qn = got[k.replace("key.bias", "query.bias")].norm()
            assert g.norm() <= 0.05 * qn + 1e-7, (k, g.norm().item(), qn.item())
            continue
        gs = g.flatten() if rec is None else g.flatten()[record_indices(rec, k, g.numel())]
        rn = r.norm().item() if rec is None else rec["grad_norm"][k]
        cos = torch.nn.functional.cosine_similarity(gs.double(), r.flatten().double(), dim=0).item()
        if cos < worst[0]:
            worst = (cos, k)
        assert cos >= COS_MIN, f"{k}: cosine {cos}"
        assert abs(g.norm().item() / rn - 1) < 0.03, f"{k}: norm ratio {g.norm().item() / rn}"
    return worst


@pytest.mark.parametrize("input_kind", ["u8", "f32"])
def test_tiny_matches_hf_golden(input_kind):
    rec = torch.load(os.path.join(GOLD, "tiny_b3.pt"), weights_only=False)
    cfg = O.OracleConfig(**rec["cfg"])
    m = _model(cfg, O.init_params(cfg, 0, 123))
    x = rec["x8"][:, 0].cuda() if input_kind == "u8" else O.normalize_gray(rec["x8"]).cuda()
    out = m(pixel_values=x, labels=rec["y"].cuda())
    assert (out.logits.cpu() - rec["logits"]).abs().max() <= LOGIT_TOL
    assert abs(out.loss.item() - rec["loss"].item()) <= LOSS_RTOL * abs(rec["loss"].item())
    out.loss.backward()
    _check_grads(m, rec["grad_sample"], rec)
    # second backward pass accumulates (PyTorch semantics): grads double
    g1 = m.classifier.weight.grad.clone()
    m(pixel_values=x, labels=rec["y"].cuda()).loss.backward()
    assert torch.allclose(m.classifier.weight.grad, 2 * g1, rtol=1e-3, atol=1e-7)


def test_vitb16_384_b2_matches_hf_golden_and_oracle():
    """BASELINE.json configs[0] on the GPU: logits/loss vs the HF golden, all 200 gradients vs the
    CPU oracle (itself pinned to the same golden in tests/test_oracle.py)."""
    rec = torch.load(os.path.join(GOLD, "vitb16_384_b2.pt"), weights_only=False)
    cfg = O.OracleConfig(**rec["cfg"])
    params = O.init_params(cfg, 0, 123)
    m = _model(cfg, params)
    out = m(pixel_values=rec["x8"][:, 0].cuda(), labels=rec["y"].cuda())
    dl = (out.logits.cpu() - rec["logits"]).abs().max().item()
    rl = abs(out.loss.item() - rec["loss"].item()) / abs(rec["loss"].item())
    out.loss.backward()
    torch.cuda.synchronize()
    torch.set_num_threads(os.cpu_count() or 1)
    _, _, ref = O.forward_backward(params, cfg, O.normalize_gray(rec["x8"]), rec["y"])
    worst = _check_grads(m, ref)
    print(f"vitb16_384 b2: logits max-abs {dl:.3e}, loss rel {rl:.3e}, worst grad cosine {worst[0]:.6f} ({worst[1]})")
    assert dl <= LOGIT_TOL and rl <= LOSS_RTOL
    for k, nrm in rec["grad_norm"].items():          # and the HF-frozen gradient norms
        if not k.endswith("key.bias"):
            assert abs(m.get_parameter(k).grad.norm().item() / nrm - 1) < 0.03, k


def test_vitb16_224_inference_matches_hf_golden():
    rec = torch.load(os.path.join(GOLD, "vitb16_224_b2.pt"), weights_only=False)
    cfg = O.OracleConfig(**rec["cfg"])
    m = _model(cfg, O.init_params(cfg, 0, 123)).eval()
    with torch.no_grad():
        out = m(pixel_values=O.normalize_gray(rec["x8"]).cuda())
        assert out.loss is None
        assert (out.logits.cpu() - rec["logits"]).abs().max() <= LOGIT_TOL
        out = m(pixel_values=rec["x8"][:, 0].cuda(), labels=rec["y"].cuda())
        assert abs(out.loss.item() - rec["loss"].item()) <= LOSS_RTOL * abs(rec["loss"].item())


def test_vitb16_384_b16_matches_oracle():
    """BASELINE.json configs[1] — the configuration bench.py times (ViT-B/16@384, batch 16): logits, loss and all
    200 gradients against the fp32 CPU oracle on the same seeded inputs (a few seconds of host time)."""
    cfg = O.VIT_B16_384
    params = O.init_params(cfg, 0, 123)
    m = _model(cfg, params)
    g = torch.Generator().manual_seed(1)
    x8, y = O.synth_inputs(cfg, 16, g)
    out = m(pixel_values=x8[:, 0].cuda(), labels=y.cuda())
    out.loss.backward()
    torch.cuda.synchronize()
    torch.set_num_threads(os.cpu_count() or 1)
    loss_ref, logits_ref, ref = O.forward_backward(params, cfg, O.normalize_gray(x8), y)
    dl = (out.logits.cpu() - logits_ref).abs().max().item()
    rl = abs(out.loss.item() - loss_ref.item()) / abs(loss_ref.item())
    worst = _check_grads(m, ref)
    print(f"vitb16_384 b16: logits max-abs {dl:.3e}, loss rel {rl:.3e}, worst grad cosine {worst[0]:.6f} ({worst[1]})")
    assert dl <= LOGIT_TOL and rl <= LOSS_RTOL


def test_batch16_shard_linearity_and_determinism():
    """Size-independent properties at the benchmarked batch: batch-shard linearity of the mean-loss gradient
    (the DP identity of SURVEY §4, through the gradient-accumulation path) and determinism of the forward."""
    cfg = O.VIT_B16_384
    params = O.init_params(cfg, 0, 123)
    m = _model(cfg, params)
    g = torch.Generator().manual_seed(1)
    x8, y = O.synth_inputs(cfg, 16, g)
    x8, y = x8[:, 0].cuda(), y.cuda()
    out = m(pixel_values=x8, labels=y)
    out.loss.backward()
    full = m.flat_grads().clone()
    logits_full = out.logits.clone()
    m.zero_grad(set_to_none=True)
    for s in range(2):                      # two shards of 8, accumulated, each scaled by 1/2
        o = m(pixel_values=x8[8 * s:8 * s + 8], labels=y[8 * s:8 * s + 8])
        assert torch.allclose(o.logits, logits_full[8 * s:8 * s + 8], atol=2e-3)
        (o.loss * 0.5).backward()
    acc = torch.cat([p.grad.flatten() for p in m.parameters()])
    ref = torch.cat([m.layout.view(full, n).flatten() for n in m.layout.names])
    cos = torch.nn.functional.cosine_similarity(acc.double(), ref.double(), dim=0).item()
    assert cos > 0.9999, cos
    out2 = m(pixel_values=x8, labels=y)
    assert torch.equal(out2.logits, logits_full)


def _train_steps(m, opt, x, y, n, clip=None, loss_scale=1.0):
    losses = []
    for _ in range(n):
        out = m(pixel_values=x, labels=y)
        (out.loss * loss_scale).backward()
        if clip is not None:
            torch.nn.utils.clip_grad_norm_(m.parameters(), clip)
        opt.step()
        opt.zero_grad(set_to_none=True)
        losses.append(out.loss.item())
    return losses


@pytest.mark.parametrize("clip,loss_scale", [(None, 1.0), (1.0, 1.0), (1.0, 1e-3)])
def test_vitk_adamw_matches_torch_adamw_with_clip(clip, loss_scale):
    """VitkAdamW(max_grad_norm) — the optimizer bench.py times — against clip_grad_norm_ + torch.optim.AdamW
    (HF trainer.py:1755-1760) on IDENTICAL gradients, three steps: replica A computes the gradients, replica B receives
    copies of them as ordinary ``param.grad`` tensors (which also exercises the fold of foreign gradients into the flat
    buffer).  Same gradients in, so the post-step parameters must agree to fp32 rounding.  With loss_scale 1 the global
    gradient norm is 2.24 (> 1: the clip is active); with 1e-3 it is inactive and eps matters."""
    rec = torch.load(os.path.join(GOLD, "tiny_b3.pt"), weights_only=False)
    cfg = O.OracleConfig(**rec["cfg"])
    import chest_x_ray_vit_b200 as pkg
    x, y = rec["x8"][:, 0].cuda(), rec["y"].cuda()
    lr = 1e-3
    ma, mb = _model(cfg, O.init_params(cfg, 0, 123)), _model(cfg, O.init_params(cfg, 0, 123))
    ob = pkg.VitkAdamW(mb, lr=lr, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01, max_grad_norm=clip)
    # torch's AdamW decays every parameter it is given; HF (trainer.py:1280-1290) and VitkAdamW exclude biases / LayerNorm
    nd = [p for n, p in ma.named_parameters() if ma.layout.kinds[n] == "nodecay"]
    dc = [p for n, p in ma.named_parameters() if ma.layout.kinds[n] != "nodecay"]
    oa = torch.optim.AdamW([{"params": dc, "weight_decay": 0.01}, {"params": nd, "weight_decay": 0.0}], lr=lr,
                           betas=(0.9, 0.999), eps=1e-8)
    worst, losses = 0.0, []
    for it in range(3):
        out = ma(pixel_values=x, labels=y)
        (out.loss * loss_scale).backward()
        losses.append(out.loss.item())
        for pa, pb in zip(ma.parameters(), mb.parameters()):
            pb.grad = pa.grad.detach().clone()
        if clip is not None:
            total = torch.nn.utils.clip_grad_norm_(ma.parameters(), clip).item()
        oa.step()
        ob.step()
        if clip is not None:
            gn = ob.grad_norm().item()
            assert abs(gn / total - 1) < 1e-4, (gn, total)
            if it == 0:
                assert (gn > 1.0) == (loss_scale == 1.0), gn          # the case really exercises clip on / clip off
        oa.zero_grad(set_to_none=True)
        ob.zero_grad(set_to_none=True)
        for (k, pa), (_, pb) in zip(ma.named_parameters(), mb.named_parameters()):
            d = (pa.detach() - pb.detach()).abs().max().item()
            worst = max(worst, d)
            assert d <= 2e-3 * lr, (it, k, d)           # a step moves a parameter by up to lr; 0.2 % of that
    assert losses[2] < losses[0]
    print(f"VitkAdamW vs torch AdamW (clip={clip}, loss_scale={loss_scale}): max |Δparam| over 3 steps {worst:.3e}")


def test_vitk_adamw_trajectory_tracks_torch_adamw():
    """Two independently trained replicas (eager torch AdamW + clip_grad_norm_ vs VitkAdamW(max_grad_norm=1)), three
    steps each on their OWN gradients.  Gradients are reproducible only up to the order of fp32 atomics (bf16
    roundings downstream flip), and Adam turns a sign-uncertain gradient element into a ±lr difference, so the
    comparison is statistical: losses agree, and all but a small fraction of elements agree to a tenth of a step."""
    rec = torch.load(os.path.join(GOLD, "tiny_b3.pt"), weights_only=False)
    cfg = O.OracleConfig(**rec["cfg"])
    import chest_x_ray_vit_b200 as pkg
    x, y = rec["x8"][:, 0].cuda(), rec["y"].cuda()
    lr = 1e-3
    ma, mb = _model(cfg, O.init_params(cfg, 0, 123)), _model(cfg, O.init_params(cfg, 0, 123))
    oa = torch.optim.AdamW(ma.parameters(), lr=lr, weight_decay=0.0)
    ob = pkg.VitkAdamW(mb, lr=lr, weight_decay=0.0, max_grad_norm=1.0)
    la = _train_steps(ma, oa, x, y, 3, clip=1.0)
    lb = _train_steps(mb, ob, x, y, 3)
    assert abs(la[0] - lb[0]) < 1e-6 and la[2] < la[0] and abs(la[2] - lb[2]) < 1e-4, (la, lb)   # (the loss mean is a 3-way fp32 atomic sum)
    da = torch.cat([(pa.detach() - pb.detach()).abs().flatten() for pa, pb in zip(ma.parameters(), mb.parameters())])
    frac = (da > 0.1 * lr).float().mean().item()
    print(f"trajectories after 3 steps: {100 * frac:.3f}% of elements differ by more than lr/10, mean |Δ| {da.mean().item():.2e}")
    assert frac < 0.02 and da.mean().item() < 0.02 * lr and da.max().item() <= 6.5 * lr


def test_vitk_adamw_clip_post_step_matches_hf_goldens():
    """One VitkAdamW(max_grad_norm=1.0) step against the post-step parameters frozen from HF + torch.optim.AdamW on the
    CPU: the tiny config (every element of tensors up to 2048 elements, 2048 sampled ones of larger tensors) and
    ViT-B/16@384 batch 2 (64 sampled elements per parameter).  The goldens were
    stepped without clipping; a first AdamW step moves every element by lr·g/(|g|+eps), which a positive rescale of g
    leaves unchanged except where |g| ~ eps, hence the same tolerance with the clip active (global norms 2.24 and 11.4).
    An element is "off" when it differs by more than half a step, i.e. its gradient had the other sign than HF's fp32
    one (bf16 noise on a near-zero gradient): at most 2 % of all elements, 10 % of any one parameter."""
    import chest_x_ray_vit_b200 as pkg
    from oracle.make_golden import record_indices
    for fname in ("tiny_b3.pt", "vitb16_384_b2.pt"):
        rec = torch.load(os.path.join(GOLD, fname), weights_only=False)
        cfg = O.OracleConfig(**rec["cfg"])
        m = _model(cfg, O.init_params(cfg, 0, 123))
        opt = pkg.VitkAdamW(m, lr=2e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, max_grad_norm=1.0)
        m(pixel_values=rec["x8"][:, 0].cuda(), labels=rec["y"].cuda()).loss.backward()
        opt.step()
        assert opt.grad_norm().item() > 1.0
        bad = tot = 0
        for k, p in m.named_parameters():
            if k.endswith("key.bias"):
                continue                                 # analytically zero gradient: the update direction is rounding noise
            p = p.detach().cpu()
            v = rec["post_sample"][k]
            p = p.flatten()[record_indices(rec, k, p.numel())]
            nb = ((p - v).abs() > 1.0e-5).sum().item()
            assert nb <= 0.10 * v.numel() + 1, (fname, k, nb, v.numel())
            bad, tot = bad + nb, tot + v.numel()
        print(f"{fname}: {bad}/{tot} post-step elements off by more than lr/2")
        assert bad <= 0.02 * tot, (fname, bad, tot)


def test_vitk_adamw_state_dict_round_trip():
    """save -> load -> step gives the same parameters as stepping on (Trainer's save_strategy='epoch' writes optimizer.pt)."""
    import chest_x_ray_vit_b200 as pkg
    cfg = O.TINY
    g = torch.Generator().manual_seed(3)
    x8, y = O.synth_inputs(cfg, 2, g)
    x, y = x8[:, 0].cuda(), y.cuda()
    ma = _model(cfg, O.init_params(cfg, 0, 123))
    oa = pkg.VitkAdamW(ma, lr=1e-3, max_grad_norm=1.0)
    _train_steps(ma, oa, x, y, 2)
    sd_m = {k: v.clone() for k, v in ma.state_dict().items()}
    sd_o = oa.state_dict()
    assert sd_o["vitk"]["step"] == 2 and sd_o["vitk"]["exp_avg"].abs().sum().item() > 0
    import io
    buf = io.BytesIO()
    torch.save(sd_o, buf)                           # what Trainer does with optimizer.state_dict()
    buf.seek(0)
    sd_o = torch.load(buf, weights_only=False)
    mb = _model(cfg, sd_m)
    ob = pkg.VitkAdamW(mb, lr=1e-3, max_grad_norm=1.0)
    ob.load_state_dict(sd_o)
    _train_steps(ma, oa, x, y, 1)
    _train_steps(mb, ob, x, y, 1)
    def mean_diff(a, b):
        return torch.cat([(pa.detach() - pb.detach()).abs().flatten() for pa, pb in zip(a.parameters(), b.parameters())]).mean().item()
    # the two replicas recompute their own (atomics-order-dependent) gradients, so compare on average, not element by element
    assert mean_diff(ma, mb) < 2e-5, mean_diff(ma, mb)
    mc = _model(cfg, sd_m)                          # without the state the trajectories differ (guards against a vacuous pass)
    oc = pkg.VitkAdamW(mc, lr=1e-3, max_grad_norm=1.0)
    _train_steps(mc, oc, x, y, 1)
    assert mean_diff(ma, mc) > 1e-4, mean_diff(ma, mc)


def test_autograd_contract_hooks_frozen_params_and_autograd_grad():
    """Every parameter is an input of the autograd node: gradients are RETURNED to autograd (adopted without a copy
    when param.grad is None), so hooks fire, torch.autograd.grad works, and frozen parameters get no gradient and
    are not touched by either optimizer."""
    import chest_x_ray_vit_b200 as pkg
    cfg = O.TINY
    g = torch.Generator().manual_seed(4)
    x8, y = O.synth_inputs(cfg, 2, g)
    x, y = x8[:, 0].cuda(), y.cuda()
    m = _model(cfg, O.init_params(cfg, 0, 123))
    fired = []
    m.classifier.weight.register_hook(lambda gr: fired.append(gr.shape))
    m.classifier.bias.register_post_accumulate_grad_hook(lambda p: fired.append("post"))
    m(pixel_values=x, labels=y).loss.backward()
    assert len(fired) == 2
    flat = m.flat_grads()
    for n, p in m.named_parameters():               # adopted, not copied: param.grad aliases the flat buffer
        assert p.grad.data_ptr() == flat.data_ptr() + 4 * m.layout.offset[n], n
    ref = {n: p.grad.clone() for n, p in m.named_parameters()}
    m.zero_grad(set_to_none=True)
    # torch.autograd.grad
    wq = m.vit.encoder.layer[0].attention.attention.query.weight
    (gq,) = torch.autograd.grad(m(pixel_values=x, labels=y).loss, [wq])
    assert torch.allclose(gq, ref["vit.encoder.layer.0.attention.attention.query.weight"], rtol=1e-3, atol=1e-7)
    assert all(p.grad is None for p in m.parameters())
    # classifier-only fine-tuning
    for n, p in m.named_parameters():
        p.requires_grad_(n.startswith("classifier"))
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    opt = pkg.VitkAdamW(m, lr=1e-2, weight_decay=0.1, max_grad_norm=1.0)
    m(pixel_values=x, labels=y).loss.backward()
    assert all((p.grad is not None) == n.startswith("classifier") for n, p in m.named_parameters())
    gn_ref = torch.sqrt(sum(ref[n].double().pow(2).sum() for n in ref if n.startswith("classifier"))).item()
    opt.step()
    assert abs(opt.grad_norm().item() / gn_ref - 1) < 1e-3           # the clip norm counts trainable gradients only
    opt.zero_grad()
    for n, p in m.named_parameters():
        moved = (p.detach() - before[n]).abs().max().item()
        assert (moved > 0) == n.startswith("classifier"), (n, moved)
    out = m(pixel_values=x, labels=y)                # the bf16 shadow of frozen GEMM weights is still intact
    assert torch.isfinite(out.loss)


def test_ddp_wrapped_module_reduces_and_steps():
    """HF Trainer under torchrun wraps the model in DistributedDataParallel (the reference's 8-replica path): the
    reducer must see every gradient become ready, twice in a row.  World size 1 (NCCL on this GPU) exercises the
    reducer's bookkeeping — the failure mode is 'Expected to have finished reduction in the prior iteration'."""
    import socket
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP
    if dist.is_initialized():
        pytest.skip("a process group already exists in this process")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1,
                            device_id=torch.device("cuda", 0))
    try:
        cfg = O.TINY
        g = torch.Generator().manual_seed(4)
        x8, y = O.synth_inputs(cfg, 2, g)
        x, y = x8[:, 0].cuda(), y.cuda()
        m = _model(cfg, O.init_params(cfg, 0, 123))
        ref = _model(cfg, O.init_params(cfg, 0, 123))
        ddp = DDP(m, device_ids=[0])
        oa = torch.optim.AdamW(ddp.parameters(), lr=1e-3, weight_decay=0.0)
        ob = torch.optim.AdamW(ref.parameters(), lr=1e-3, weight_decay=0.0)
        for _ in range(2):
            ddp(pixel_values=x, labels=y).loss.backward()
            ref(pixel_values=x, labels=y).loss.backward()
            for (k, pa), (_, pb) in zip(m.named_parameters(), ref.named_parameters()):
                assert torch.allclose(pa.grad, pb.grad, rtol=1e-3, atol=1e-6), k
            oa.step(); ob.step()
            oa.zero_grad(set_to_none=True); ob.zero_grad(set_to_none=True)
        for pa, pb in zip(m.parameters(), ref.parameters()):
            assert (pa - pb).abs().max().item() < 1e-5
    finally:
        dist.destroy_process_group()


def test_no_grad_and_custom_loss_on_logits():
    cfg = O.TINY
    m = _model(cfg, O.init_params(cfg, 0, 123))
    g = torch.Generator().manual_seed(2)
    x8, y = O.synth_inputs(cfg, 2, g)
    x8, y = x8[:, 0].cuda(), y.cuda()
    out = m(pixel_values=x8)                    # no labels: logits only, user-side loss
    loss = torch.nn.functional.binary_cross_entropy_with_logits(out.logits, y)
    loss.backward()
    ga = m.flat_grads().clone()
    m.zero_grad(set_to_none=True)
    m(pixel_values=x8, labels=y).loss.backward()
    assert torch.allclose(ga, m.flat_grads(), rtol=1e-4, atol=1e-7)
    with pytest.raises(RuntimeError, match="overwritten"):
        o1 = m(pixel_values=x8, labels=y)
        m(pixel_values=x8, labels=y)
        o1.loss.backward()


@pytest.mark.parametrize("batch", [1, 8])
def test_vit_large_16_384_matches_oracle(batch):
    """BASELINE.json configs[4] (ViT-L/16@384: D=1024, H=16, F=4096, L=24) at its per-GPU batch of 8 (and batch 1):
    logits / loss and every gradient against the fp32 CPU oracle."""
    cfg = O.VIT_L16_384
    params = O.init_params(cfg, 0, 123)
    g = torch.Generator().manual_seed(11)
    x8, y = O.synth_inputs(cfg, batch, g)
    m = _model(cfg, params)
    out = m(pixel_values=x8[:, 0].cuda(), labels=y.cuda())
    out.loss.backward()
    torch.cuda.synchronize()
    torch.set_num_threads(os.cpu_count() or 1)
    loss_ref, logits_ref, ref = O.forward_backward(params, cfg, O.normalize_gray(x8), y)
    dl = (out.logits.cpu() - logits_ref).abs().max().item()
    rl = abs(out.loss.item() - loss_ref.item()) / abs(loss_ref.item())
    worst = _check_grads(m, ref)
    print(f"vit-L b{batch}: logits max-abs {dl:.3e}, loss rel {rl:.3e}, worst grad cosine {worst[0]:.6f} ({worst[1]})")
    assert dl <= LOGIT_TOL and rl <= LOSS_RTOL


def test_vitb16_224_batch_sweep_is_batch_invariant():
    """BASELINE.json configs[3]: inference at 224 px; logits of an image must not depend on the batch it is in."""
    cfg = O.VIT_B16_224
    m = _model(cfg, O.init_params(cfg, 0, 123)).eval()
    g = torch.Generator().manual_seed(5)
    x8 = torch.randint(0, 256, (64, 224, 224), dtype=torch.uint8, generator=g).cuda()
    with torch.no_grad():
        big = m(pixel_values=x8).logits
        for bs in (1, 2, 7, 32):
            part = m(pixel_values=x8[:bs]).logits
            assert (part - big[:bs]).abs().max() < 5e-3, bs
    assert torch.isfinite(big).all()
