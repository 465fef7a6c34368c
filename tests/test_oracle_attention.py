"""CPU-only: the fp64 attention oracle (oracle/attention_oracle.py) against autograd, the calibration of the per-row
bounds TAU against an emulation of the kernels' roundings, and the metric's sensitivity to plausible kernel bugs."""
import functools

import pytest
import torch

from oracle import attention_oracle as A


def cpu_shape(B, T, H, budget=1 << 23):
    """The sweep case at the same T with B, then H, halved until B·H·T² score elements fit ``budget``."""
    while B > 1 and B * H * T * T > budget:
        B = (B + 1) // 2
    while H > 1 and B * H * T * T > budget:
        H = (H + 1) // 2
    return B, T, H


@functools.lru_cache(maxsize=4)
def _case(B, T, H, scale, family):
    b, t, h = cpu_shape(B, T, H)
    qkv, do = A.inputs(B, T, H, scale, family)
    qkv = qkv[:b, :, :, :h].contiguous()
    do = do.view(B, T, H, A.DH)[:b, :, :h].reshape(b, T, h * A.DH).contiguous()
    return qkv, do, A.reference(qkv, do, scale)


def _swap_heads(qkv):
    """K of the first and last head exchanged in the last image."""
    x = qkv.clone()
    x[-1, :, 1, 0], x[-1, :, 1, -1] = qkv[-1, :, 1, -1], qkv[-1, :, 1, 0]
    return x


MUTANTS = {
    "last key dropped": lambda qkv, do, s: A.reference(qkv, do, s, keys=qkv.shape[1] - 1),
    "keys truncated to 16k": lambda qkv, do, s: A.reference(qkv, do, s, keys=qkv.shape[1] // 16 * 16),
    "last query left out of dK/dV": lambda qkv, do, s: A.reference(qkv, do, s, dkv_queries=qkv.shape[1] - 1),
    "K of two heads swapped": lambda qkv, do, s: A.reference(_swap_heads(qkv), do, s),
    "scale 0.125": lambda qkv, do, s: A.reference(qkv, do, 0.125),
}
IDS = [A.case_id(*c) for c in A.SWEEP]


@pytest.mark.parametrize("B,T,H", [(2, 17, 3), (1, 129, 2), (3, 1, 2), (1, 2, 1)])
@pytest.mark.parametrize("scale", [0.125, 0.3])
def test_reference_matches_autograd(B, T, H, scale):
    qkv, do = A.inputs(B, T, H, scale, "randn")
    ref = A.reference(qkv, do, scale)
    x = qkv.double().requires_grad_(True)
    q, k, v = (x[:, :, i].transpose(1, 2) for i in range(3))
    s = (q @ k.transpose(-1, -2)) * scale
    o = torch.softmax(s, dim=-1) @ v
    o.transpose(1, 2).reshape(B, T, -1).backward(do.double())
    want = {"o": o.transpose(1, 2), "lse": torch.logsumexp(s, -1), "dq": x.grad[:, :, 0], "dk": x.grad[:, :, 1],
            "dv": x.grad[:, :, 2]}
    for name, w in want.items():
        err = (ref[name] - w.detach()).abs().max().item()
        assert err <= 1e-12 * max(1.0, w.abs().max().item()), f"{name}: {err}"


def test_row_errors_sees_one_row():
    qkv, do, ref = _case(2, 577, 3, 0.125, "randn")
    got = {n: ref[n].clone() for n in A.ROWS}
    got["dk"][1, 576, 2] = 0                               # the last key of the last (head, image) tail block
    got["dv"][0, 5, 1, 7] = float("nan")
    e = A.row_errors(got, ref)
    assert e["o"]["worst"] == 0 and e["dq"]["worst"] == 0
    assert e["dk"]["row"] == (1, 576, 2) and e["dk"]["worst"] >= min(1.0, ref["dk"][1, 576, 2].norm().item() /
                                                                       ref["dk"].norm(dim=-1).median().item())
    assert e["dk"]["rel_l2"] < 0.1                         # what a global measure makes of it
    assert e["dv"]["row"] == (0, 5, 1) and e["dv"]["worst"] == float("inf")


@pytest.mark.parametrize("B,T,H,scale,family", A.SWEEP, ids=IDS)
def test_emulated_kernel_within_half_tau(B, T, H, scale, family):
    """The kernels' roundings, emulated, stay within TAU/2 on every row; lse within half its bound."""
    qkv, do, ref = _case(B, T, H, scale, family)
    em = A.emulate_kernel(qkv, do, scale)
    e = A.row_errors(em, ref)
    lse = ((em["lse"].double() - ref["lse"]).abs() / ref["lse_tol"]).max().item()
    print(f"{A.case_id(B, T, H, scale, family)} at {cpu_shape(B, T, H)}: "
          + "  ".join(f"{n} {e[n]['worst']:.4f} (τ {A.TAU[n]})" for n in A.ROWS) + f"  lse/bound {lse:.3f}")
    for n in A.ROWS:
        assert e[n]["worst"] <= A.TAU[n] / 2, f"{n}: emulated worst row {e[n]['worst']:.4f} at {e[n]['row']}"
        assert e[n]["worst"] <= A.EMULATED_WORST[n], f"{n}: the recorded EMULATED_WORST is out of date"
    assert lse <= 0.5


@pytest.mark.parametrize("B,T,H,scale,family", A.SWEEP, ids=IDS)
def test_mutants_exceed_tau(B, T, H, scale, family):
    """Every mutant that changes the case's result moves some row of some tensor by ≥ MUTANT_MARGIN·TAU."""
    qkv, do, ref = _case(B, T, H, scale, family)
    line = []
    for name, mutant in MUTANTS.items():
        got = mutant(qkv, do, scale)
        e = A.row_errors(got, ref)
        if max(e[n]["rel_l2"] for n in A.ROWS) < 1e-9:      # this mutant changes nothing here (e.g. T % 16 == 0)
            continue
        margin = max(e[n]["worst"] / A.TAU[n] for n in A.ROWS)
        line.append(f"{name}: {margin:.1f}")
        assert margin >= A.MUTANT_MARGIN, f"{name}: worst row only {margin:.2f} τ"
        assert margin >= A.MUTANT_MIN_MARGIN[name], f"{name}: the recorded MUTANT_MIN_MARGIN is out of date"
    print(f"{A.case_id(B, T, H, scale, family)} margins (× τ): " + ", ".join(line))
