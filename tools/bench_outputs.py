"""Cost of the forward's optional outputs (output_attentions / output_hidden_states) on one GPU.

1. vitk_attn_probs alone at (B, T, H) = (16, 577, 12) and (64, 197, 12): CUDA events around 200 back-to-back launches
   into one output.  The output (256 MB and 119 MB) is written, never read, so the kernel is held against HBM write
   bandwidth: the measured peak of MEASURED_PEAKS.json when present, and a write-only fill of 1 GB timed in the same run.
2. Eval forwards of ViT-B/16 at 384 px, batch 16: plain, hidden states only, attentions only, both — ms per forward,
   including the returned tensors (the host waits for each forward to finish).

Usage: python tools/bench_outputs.py [--out FILE]   (the text printed is also written to FILE)
"""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import chest_x_ray_vit_b200 as pkg  # noqa: E402

ops = pkg.ops
dev = "cuda"
lines = []


def say(s=""):
    print(s, flush=True)
    lines.append(s)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # the card name still identifies the number
        q = f"power limit unavailable ({e})"
    return f"{name}; power limit, max SM clock: {q}"


def events_ms(fn, n):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    ops.check_device(0)
    say(f"card: {card()}")
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm_meas = json.load(open(pk))["hbm_gbs"] if os.path.exists(pk) else None
    fill = torch.empty(1 << 28, dtype=torch.float32, device=dev)            # 1 GB
    fill.fill_(0.0)
    t_fill = events_ms(lambda: fill.fill_(1.0), 50)
    fill_gbs = fill.numel() * 4 / t_fill / 1e6
    del fill
    say(f"HBM write reference: MEASURED_PEAKS.json hbm_gbs = {hbm_meas if hbm_meas else 'not present'}; "
        f"torch fill_ of 1 GB in this run: {fill_gbs:.0f} GB/s")
    say()
    say("vitk_attn_probs alone (200 launches between one event pair; output > the 126 MB L2, written once per launch)")
    for B, T, H in ((16, 577, 12), (64, 197, 12)):
        g = torch.Generator().manual_seed(0)
        qkv = torch.randn(B, T, 3, H, 64, generator=g).to(dev).to(torch.bfloat16)
        _, lse = ops.attn_fwd(qkv, B, T, H, 0.125)
        probs = torch.empty(B, H, T, T, device=dev)
        for _ in range(5):
            ops.attn_probs(qkv, lse, B, T, H, 0.125, out=probs)
        ms = events_ms(lambda: ops.attn_probs(qkv, lse, B, T, H, 0.125, out=probs), 200)
        nbytes = B * H * T * T * 4
        gbs = nbytes / ms / 1e6
        vs = f"{gbs / hbm_meas:.2f} of measured peak, " if hbm_meas else ""
        say(f"  B={B:3d} T={T} H={H}: output {nbytes / 2**20:6.1f} MiB  {ms * 1e3:7.1f} us  {gbs:6.0f} GB/s  "
            f"({vs}{gbs / fill_gbs:.2f} of the fill)")
        del qkv, lse, probs
    say()
    say("ViT-B/16 @ 384 px, batch 16, eval forward (no_grad), ms per forward incl. the returned tensors")
    m = pkg.ViTForImageClassification(pkg.ViTConfig()).cuda().eval()
    g = torch.Generator().manual_seed(1)
    x = torch.randint(0, 256, (16, 384, 384), dtype=torch.uint8, generator=g).to(dev)
    modes = (("plain", {}), ("hidden states", {"output_hidden_states": True}), ("attentions", {"output_attentions": True}),
             ("both", {"output_attentions": True, "output_hidden_states": True}))
    res = {k: [] for k, _ in modes}
    with torch.no_grad():
        for _, kw in modes:                 # build and capture every plan first
            for _ in range(3):
                m(pixel_values=x, **kw)
        torch.cuda.synchronize()
        for _ in range(5):                  # alternate the modes: a drift of the clock hits all four alike
            for name, kw in modes:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(4):
                    out = m(pixel_values=x, **kw)
                    del out
                e1.record()
                torch.cuda.synchronize()
                res[name].append(e0.elapsed_time(e1) / 4)
    base = sorted(res["plain"])[2]
    for name, _ in modes:
        t = sorted(res[name])[2]
        say(f"  {name:14s} {t:7.2f} ms  (+{t - base:6.2f} ms)   runs: " + " ".join(f"{v:.2f}" for v in res[name]))
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
