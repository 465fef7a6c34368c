"""Freeze golden vectors from the real third-party implementation the reference calls.

Runs ``transformers.ViTForImageClassification`` (what /root/reference/ViT-Training.py:83-90
constructs) in fp32 on the CPU, on weights produced by ``oracle.vit_oracle.init_params``
(deterministic CPU generator, so the weights themselves need not be committed), and
writes small fixtures under tests/golden/:

  tiny_b3.pt .......... TINY config, batch 3: inputs, logits, loss, per-parameter gradient
                        norms, and every element (tensors of at most TINY_SAMPLE elements) or
                        TINY_SAMPLE distinct sampled elements of each gradient and of each
                        post-AdamW-step parameter
  vitb16_384_b2.pt .... BASELINE.json configs[0] (ViT-B/16@384, batch 2): inputs,
                        logits, loss, per-parameter gradient norms and 64 sampled
                        gradient entries per parameter, same for post-step params
  vitb16_224_b2.pt .... the 197-token variant (configs[3]) logits only

Run here (needs transformers; not needed on the GPU box):
    python oracle/make_golden.py
Versions are recorded inside each file.
"""
from __future__ import annotations

import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import vit_oracle as O  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def hf_model(cfg: O.OracleConfig, params):
    import transformers
    from transformers import ViTConfig, ViTForImageClassification
    hc = ViTConfig(image_size=cfg.image_size, patch_size=cfg.patch_size, hidden_size=cfg.hidden_size,
                   num_hidden_layers=cfg.num_hidden_layers, num_attention_heads=cfg.num_attention_heads,
                   intermediate_size=cfg.intermediate_size, num_labels=cfg.num_labels,
                   problem_type="multi_label_classification")
    m = ViTForImageClassification(hc).train()
    missing = m.load_state_dict(params, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return m, transformers.__version__


TINY_SAMPLE = 2048       # keeps tiny_b3.pt far below 1 MB (all gradients and post-step parameters would be 2.9 MB)


def sample_indices(name: str, numel: int, n: int = 64) -> torch.Tensor:
    g = torch.Generator().manual_seed(abs(hash_name(name)) % (2 ** 31))
    return torch.randint(0, numel, (min(n, numel),), generator=g)


def kept_indices(name: str, numel: int, n: int) -> torch.Tensor:
    """All elements of a tensor of at most ``n``, else ``n`` distinct ones drawn with a per-name seed (sorted)."""
    if numel <= n:
        return torch.arange(numel)
    g = torch.Generator().manual_seed(abs(hash_name(name)) % (2 ** 31))
    return torch.randperm(numel, generator=g)[:n].sort().values


def record_indices(rec: dict, name: str, numel: int) -> torch.Tensor:
    """Flat indices of parameter ``name`` that the ``grad_sample`` / ``post_sample`` entries of ``rec`` hold."""
    n = rec.get("n_sample")
    return sample_indices(name, numel) if n is None else kept_indices(name, numel, n)


def hash_name(name: str) -> int:
    h = 2166136261
    for ch in name.encode():
        h = ((h ^ ch) * 16777619) & 0xFFFFFFFF
    return h


def run(cfg: O.OracleConfig, batch: int, n_sample=None, step: bool = True):
    """``n_sample`` None: 64 elements per tensor drawn with replacement (sample_indices); else kept_indices(n_sample)."""
    torch.manual_seed(0)
    params = O.init_params(cfg, seed=0, perturb_seed=123)
    g = torch.Generator().manual_seed(1)
    x8, y = O.synth_inputs(cfg, batch, g)
    x = O.normalize_gray(x8)
    m, ver = hf_model(cfg, params)
    out = m(pixel_values=x, labels=y)
    out.loss.backward()
    grads = {k: v.grad.detach().clone() for k, v in m.named_parameters()}
    rec = {"hf_version": ver, "torch_version": torch.__version__, "batch": batch,
           "cfg": cfg.__dict__, "x8": x8, "y": y,
           "logits": out.logits.detach().clone(), "loss": out.loss.detach().clone()}
    if step:
        opt = torch.optim.AdamW(m.parameters(), lr=2e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)
        opt.step()
        post = {k: v.detach().clone() for k, v in m.named_parameters()}
    if n_sample is not None:
        rec["n_sample"] = n_sample
    rec["grad_norm"] = {k: v.norm().item() for k, v in grads.items()}
    rec["grad_sample"] = {k: v.flatten()[record_indices(rec, k, v.numel())].clone() for k, v in grads.items()}
    if step:
        rec["post_sample"] = {k: v.flatten()[record_indices(rec, k, v.numel())].clone() for k, v in post.items()}
    return rec


def main():
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(os.cpu_count() or 1)
    torch.save(run(O.TINY, 3, n_sample=TINY_SAMPLE), os.path.join(OUT, "tiny_b3.pt"))
    torch.save(run(O.VIT_B16_384, 2), os.path.join(OUT, "vitb16_384_b2.pt"))
    r = run(O.VIT_B16_224, 2, step=False)
    r = {k: r[k] for k in ("hf_version", "torch_version", "batch", "cfg", "x8", "y", "logits", "loss")}
    torch.save(r, os.path.join(OUT, "vitb16_224_b2.pt"))
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
