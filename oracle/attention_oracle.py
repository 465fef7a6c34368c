"""fp64 oracle of the fused attention kernels (csrc/attention.cu, csrc/attention_cls.cu) and the per-row error metric
their tests assert.  TEST INFRASTRUCTURE ONLY.

* ``reference(qkv, do, scale)``: O, lse and dQ / dK / dV of softmax(Q·Kᵀ·scale)·V in float64 from the bf16 inputs,
  on whichever device the inputs live.
* ``emulate_kernel(qkv, do, scale)``: the same with the kernels' roundings (attention.cu, the comment above
  attn_bwd_kernel): fp32 scores and exponentials, P rounded to bf16 before P·V and Pᵀ·dO, dS = P∘(dP − Δ) rounded to
  bf16 before dSᵀ·Q and dS·K, Δ from the bf16 O and dO, bf16 outputs.  It calibrates ``TAU`` without a GPU
  (tests/test_oracle_attention.py).
* ``row_errors(got, ref)``: every (image, token, head) 64-vector of O / dQ / dK / dV is a row; a row's error is
  ‖got − ref‖₂ / max(‖ref‖₂, median row norm of that tensor, ‖terms‖ / 16, 10⁻⁶ · the tensor's largest ‖terms‖),
  where ‖terms‖ is the root-sum-square of the norms of the terms the row sums (``reference``'s "terms").  A global
  cosine or max-abs bound lets one wrong row in 577 through; this metric does not.  The two floors only matter for rows far smaller
  than what they are summed from: a peaked softmax row makes dS = P∘(dP − Δ) a difference of nearly equal terms (and
  at T = 1 dQ = dK = 0 exactly), which bf16 operands can only resolve to a fraction of the terms; and a row of
  vanishing probabilities (family "jumps") underflows fp32.

``SWEEP`` lists the (B, T, H, scale, family) cases the GPU tests run and the CPU calibration covers, ``inputs`` builds
each case's qkv / do from a CPU generator, so both see the same bits.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch

DH = 64
ROWS = ("o", "dq", "dk", "dv")

# Per-row bound of each tensor.  Calibrated on the CPU (tests/test_oracle_attention.py): over every SWEEP case the
# emulated kernel's worst row error is at most TAU/2 (EMULATED_WORST), and each mutant of the reference that changes a
# case (a dropped key, keys truncated to a multiple of 16, the last query left out of dK/dV, K of two heads swapped,
# 0.125 in place of the scale) exceeds TAU by at least MUTANT_MARGIN there.
TAU = {"o": 0.01, "dq": 0.03, "dk": 0.03, "dv": 0.012}
MUTANT_MARGIN = 4.0
# What that calibration measured (the CPU test keeps these honest): the emulation's worst row over the sweep, and the
# smallest (worst row error / TAU, worst tensor) each mutant reaches over the cases it changes.
EMULATED_WORST = {"o": 0.0035, "dq": 0.0136, "dk": 0.0126, "dv": 0.0047}
MUTANT_MIN_MARGIN = {"last key dropped": 13.7, "keys truncated to 16k": 83.2, "last query left out of dK/dV": 13.4,
                     "K of two heads swapped": 79.1, "scale 0.125": 32.3}
# lse against fp64, per query: |Δlse| ≤ LSE_ATOL + LSE_REL · max_j |S_ij| (fp32 scores of 64 bf16 products, ex2/lg2).
LSE_ATOL, LSE_REL = 1e-4, 2e-5
TERMS_FLOOR, TINY_FLOOR = 1 / 16, 1e-6

FAMILIES = ("randn", "x4", "jumps", "onehot")

# T crosses the 16-column rounding (15/16/17), the 64-query sub-block (63/64/65), the 128-key tile (127/128/129), odd
# sub-block counts (191/193), ring recycling (1025, 2048); H covers every Δ-kernel instantiation (≤4, ≤8, ≤12, ≤16 and
# the generic loop for H > 16, several times for 32).  The first seventeen are the cases the suite had before.
SWEEP = [
    (1, 128, 1, 0.125, "randn"), (1, 64, 2, 0.125, "randn"), (2, 17, 2, 0.125, "randn"), (2, 129, 3, 0.125, "randn"),
    (2, 197, 12, 0.125, "randn"), (1, 256, 2, 0.125, "randn"), (2, 577, 12, 0.125, "randn"),
    (1, 300, 16, 0.125, "randn"), (1, 385, 2, 0.125, "randn"), (1, 640, 2, 0.125, "randn"),
    (1, 1024, 1, 0.125, "randn"), (16, 577, 12, 0.125, "randn"), (1, 130, 6, 0.125, "randn"),
    (1, 70, 20, 0.125, "randn"), (2, 129, 20, 0.125, "randn"),
    (1, 577, 2, 0.125, "x4"), (1, 577, 1, 0.125, "jumps"),
    (3, 1, 4, 0.3, "randn"), (2, 2, 5, 0.05, "onehot"), (2, 15, 8, 0.3, "randn"), (1, 16, 9, 0.05, "x4"),
    (4, 63, 13, 0.125, "onehot"), (2, 65, 17, 0.3, "randn"), (1, 127, 32, 0.05, "randn"),
    (2, 191, 5, 0.3, "onehot"), (1, 193, 4, 0.05, "jumps"), (1, 255, 13, 0.125, "x4"), (1, 257, 9, 0.3, "onehot"),
    (2, 513, 3, 0.05, "randn"), (1, 1025, 2, 0.3, "onehot"), (1, 2048, 3, 0.3, "x4"), (1, 2048, 1, 0.05, "onehot"),
    (64, 197, 12, 0.125, "randn"),            # ViT-B/16 at 224 px
    (16, 577, 16, 0.125, "onehot"),           # ViT-L/16 at 384 px
]


def case_id(B: int, T: int, H: int, scale: float, family: str) -> str:
    return f"B{B}-T{T}-H{H}-s{scale}-{family}"


def inputs(B: int, T: int, H: int, scale: float, family: str, seed: Optional[int] = None):
    """qkv bf16 [B,T,3,H,64] and do bf16 [B,T,H·64] on the CPU.
    randn: unit normal, do ×0.1.  x4: qkv ×4 (scores of std ≈ 16, rows dominated by one key).  jumps: Q ×3, keys
    200.. ×6 and 400.. ×48, so later key blocks exceed the first block's maximum by far more than the forward's lazy
    rescale threshold.  onehot: each query is a multiple of one random key, scaled so that the key's score is
    ln(9T) and its probability ≈ 0.85 – 0.9."""
    g = torch.Generator().manual_seed(T * 10 + H + 1000 * FAMILIES.index(family) if seed is None else seed)
    qkv = torch.randn(B, T, 3, H, DH, generator=g)
    if family == "x4":
        qkv *= 4
    elif family == "jumps":
        qkv[:, :, 0] *= 3.0
        qkv[:, 200:, 1] *= 6.0
        qkv[:, 400:, 1] *= 8.0
    elif family == "onehot":
        k = qkv[:, :, 1]                                                   # [B,T,H,64]
        pick = torch.randint(0, T, (B, T, H), generator=g)
        kp = torch.gather(k, 1, pick[..., None].expand(B, T, H, DH))
        qkv[:, :, 0] = kp * (math.log(9 * T) / (scale * (kp * kp).sum(-1, keepdim=True)))
    do = torch.randn(B, T, H * DH, generator=g) * (0.1 if family == "randn" else 1.0)
    return qkv.to(torch.bfloat16), do.to(torch.bfloat16)


def _heads(qkv, do, dtype):
    """q, k, v, dO as [B,H,T,64] of ``dtype``."""
    B, T, _, H, dh = qkv.shape
    q, k, v = (qkv[:, :, i].transpose(1, 2).to(dtype) for i in range(3))
    return q, k, v, do.reshape(B, T, H, dh).transpose(1, 2).to(dtype)


def _tokens(x):
    """[B,H,T,64] → [B,T,H,64]."""
    return x.transpose(1, 2).contiguous()


def reference(qkv: torch.Tensor, do: torch.Tensor, scale: float, *, keys: Optional[int] = None,
              dkv_queries: Optional[int] = None) -> Dict[str, torch.Tensor]:
    """float64 O / dQ / dK / dV [B,T,H,64] and lse [B,H,T] of softmax(Q·Kᵀ·scale)·V from bf16 qkv [B,T,3,H,64] and dO
    [B,T,H·64] (or [B·T, H·64]); also the lse bound "lse_tol" [B,H,T] and each row's "terms" [B,T,H] (row_errors).
    ``keys`` (attend to the first ``keys`` keys only) and ``dkv_queries`` (only the first ``dkv_queries`` queries
    contribute to dK / dV) exist for the mutants of the sensitivity test."""
    q, k, v, g = _heads(qkv, do, torch.float64)
    T = q.shape[2]
    s = (q @ k.transpose(-1, -2)) * scale
    lse_tol = LSE_ATOL + LSE_REL * s.abs().amax(-1)
    if keys is not None and keys < T:
        s[..., keys:] = -math.inf
    lse = torch.logsumexp(s, -1)
    p = torch.nan_to_num(torch.exp(s - lse[..., None]), nan=0.0)           # no key left: P = 0
    o = p @ v
    dp = g @ v.transpose(-1, -2)
    ds = p * (dp - (g * o).sum(-1, keepdim=True))
    dq = scale * (ds @ k)
    if dkv_queries is not None and dkv_queries < T:
        p, ds = p.clone(), ds.clone()
        p[..., dkv_queries:, :] = 0
        ds[..., dkv_queries:, :] = 0
    dk = scale * (ds.transpose(-1, -2) @ q)
    dv = p.transpose(-1, -2) @ g
    # Root-sum-square of the terms of each row's sum, the scale of its rounding error: O_i = Σ_j P_ij V_j,
    # dV_j = Σ_i P_ij dO_i, dQ_i = s Σ_j dS_ij K_j, dK_j = s Σ_i dS_ij Q_i, with |dS_ij| counted as P_ij (|dP_ij| +
    # ‖O_i‖‖dO_i‖): the second part bounds |Δ_i| and the error of a Δ taken from a rounded O
    w = (p * (dp.abs() + (o.norm(dim=-1) * g.norm(dim=-1))[..., None])) ** 2
    rss = lambda m, x: (m @ (x * x).sum(-1, keepdim=True)).sqrt().squeeze(-1).transpose(1, 2).contiguous()   # [B,T,H]
    terms = {"o": rss(p * p, v), "dv": rss((p * p).transpose(-1, -2), g), "dq": scale * rss(w, k),
             "dk": scale * rss(w.transpose(-1, -2), q)}
    return {"o": _tokens(o), "dq": _tokens(dq), "dk": _tokens(dk), "dv": _tokens(dv), "lse": lse, "lse_tol": lse_tol,
            "terms": terms}


def emulate_kernel(qkv: torch.Tensor, do: torch.Tensor, scale: float) -> Dict[str, torch.Tensor]:
    """The kernels' arithmetic in fp32 with their bf16 roundings (outputs as float32 holding bf16 values, lse fp32)."""
    bf = torch.bfloat16
    q, k, v, g = _heads(qkv, do, torch.float32)
    s = (q @ k.transpose(-1, -2)) * scale
    m = s.amax(-1, keepdim=True)
    pt = torch.exp(s - m)                                  # forward: P̃ against the row maximum, bf16 into P̃·V
    l = pt.sum(-1, keepdim=True)                           # the row sum in fp32 (before the rounding)
    o = ((pt.to(bf).float() @ v) / l).to(bf).float()
    lse = (m + torch.log(l)).squeeze(-1)
    p = torch.exp(s - lse[..., None])                      # backward: P from the stored lse
    delta = (o * g).sum(-1, keepdim=True)                  # Δ from the bf16 O and dO
    ds = p * (g @ v.transpose(-1, -2) - delta)
    p16, ds16 = p.to(bf).float(), ds.to(bf).float()
    dv = (p16.transpose(-1, -2) @ g).to(bf).float()
    dk = (scale * (ds16.transpose(-1, -2) @ q)).to(bf).float()
    dq = (scale * (ds16 @ k)).to(bf).float()
    return {"o": _tokens(o), "dq": _tokens(dq), "dk": _tokens(dk), "dv": _tokens(dv), "lse": lse}


def row_errors(got: Dict[str, torch.Tensor], ref: Dict[str, torch.Tensor], names=ROWS) -> Dict[str, dict]:
    """Per tensor: ``worst`` row error, the ``row`` (image, token, head) where it occurs, and the global relative L2
    ``rel_l2``.  ``got`` may be in any float type and any shape with the same element order as ``ref`` [B,T,H,64]; a
    non-finite row counts as an infinite error."""
    out = {}
    for name in names:
        r = ref[name].double()
        x = got[name].reshape(r.shape).double()
        rn = r.reshape(-1, DH).norm(dim=1)
        en = (x - r).reshape(-1, DH).norm(dim=1)
        en = torch.where(torch.isfinite(en), en, torch.full_like(en, math.inf))
        tn = ref["terms"][name].reshape(-1).double()
        den = torch.maximum(rn, TERMS_FLOOR * tn).clamp(min=max(rn.median().item(), TINY_FLOOR * tn.max().item(), 1e-300))
        err = en / den
        i = int(err.argmax())
        out[name] = {"worst": err[i].item(), "row": tuple(int(c) for c in torch.unravel_index(torch.tensor(i), r.shape[:-1])),
                     "rel_l2": ((x - r).norm() / r.norm().clamp(min=1e-300)).item()}
    return out

