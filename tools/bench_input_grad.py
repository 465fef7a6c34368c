"""Cost of the gradient with respect to pixel_values on one GPU.

1. The VITK_EPI_UNPATCH_F32 GEMM alone at B·T = 9232 (batch 16, 384 px), N = K = 768, against a STORE_F32 GEMM of the
   same shape into a row-major [9232, 768] fp32 output (single-CTA kernel, as UNPATCH uses, and the library's own
   choice).  CUDA events around 200 back-to-back launches; both outputs (28 MB) are written, never read.  The
   difference is the cost of the NCHW scatter.
2. A saliency call — forward + backward to x, Σ logits[:, c] as the target — of ViT-B/16 at batch 16 / 384 px and
   batch 64 / 224 px: frozen model (data-only backward plan + the input GEMM) against trainable model (full backward
   plan + the input GEMM), with a trainable step without input gradient and a no-grad forward for reference; ms per
   call, modes alternated, the host waiting for each call.

Usage: python tools/bench_input_grad.py [--out FILE]   (the text printed is also written to FILE)
"""
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


def gemm_leg():
    B, S, D = 16, 384, 768
    T = (S // 16) ** 2 + 1
    M = B * T
    g = torch.Generator().manual_seed(0)
    dh = torch.randn(M, D, generator=g).to(dev).to(torch.bfloat16)
    wp = (torch.randn(D, 768, generator=g) * 0.05).to(dev).to(torch.bfloat16)
    img = torch.empty(B, 3, S, S, device=dev)
    rows = torch.empty(M, 768, device=dev)
    flops = 2.0 * M * 768 * D
    cases = (("UNPATCH_F32 (single-CTA)", lambda: ops.gemm(dh, wp, M, 768, D, img, epilogue=ops.EPI_UNPATCH_F32,
                                                             b_mn_major=True, ldd=S, rows_out=T, row_off=1), img.numel() * 4),
             ("STORE_F32 single-CTA", lambda: ops.gemm(dh, wp, M, 768, D, rows, epilogue=ops.EPI_STORE_F32, b_mn_major=True,
                                                       variant=1), rows.numel() * 4),
             ("STORE_F32 library choice", lambda: ops.gemm(dh, wp, M, 768, D, rows, epilogue=ops.EPI_STORE_F32,
                                                           b_mn_major=True), rows.numel() * 4))
    say(f"GEMM alone: M = B·T = {M} (batch {B}, {S} px), N = K = 768, {flops / 1e9:.1f} GFLOP; "
        "200 launches between one event pair, 5 repeats alternated")
    res = {name: [] for name, _, _ in cases}
    for _, fn, _ in cases:
        for _ in range(10):
            fn()
    torch.cuda.synchronize()
    for _ in range(5):
        for name, fn, _ in cases:
            res[name].append(events_ms(fn, 200))
    for name, _, nbytes in cases:
        t = sorted(res[name])[2]
        say(f"  {name:26s} {t * 1e3:7.2f} us  {flops / t / 1e9:6.0f} TFLOP/s  writes {nbytes / 1e6:5.1f} MB "
            f"({nbytes / t / 1e6:5.0f} GB/s)   runs: " + " ".join(f"{v * 1e3:.2f}" for v in res[name]))
    say()


def saliency_leg(S, B, reps=5, calls=4):
    torch.manual_seed(1)
    m = pkg.ViTForImageClassification(pkg.ViTConfig(image_size=S)).cuda().train()
    x = (torch.rand(B, 3, S, S, device=dev) * 2 - 1)

    def frozen():
        xg = x.detach().requires_grad_()
        m(pixel_values=xg).logits[:, 3].sum().backward()

    def trainable_input():
        m.zero_grad(set_to_none=True)
        xg = x.detach().requires_grad_()
        m(pixel_values=xg).logits[:, 3].sum().backward()

    def trainable_plain():
        m.zero_grad(set_to_none=True)
        m(pixel_values=x).logits[:, 3].sum().backward()

    def forward_only():
        with torch.no_grad():
            m(pixel_values=x)
    modes = (("frozen: data-only + input GEMM", False, frozen), ("trainable: full + input GEMM", True, trainable_input),
             ("trainable, no input grad", True, trainable_plain), ("forward only (no_grad)", False, forward_only))
    for _, trainable, fn in modes:          # build and capture every plan first
        m.requires_grad_(trainable)
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    res = {name: [] for name, _, _ in modes}
    for _ in range(reps):                   # alternate the modes: a drift of the clock hits all of them alike
        for name, trainable, fn in modes:
            m.requires_grad_(trainable)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(calls):
                fn()
            e1.record()
            torch.cuda.synchronize()
            res[name].append(e0.elapsed_time(e1) / calls)
    say(f"ViT-B/16 @ {S} px, batch {B}: saliency call (forward + backward to x), ms per call")
    t = {name: sorted(v)[len(v) // 2] for name, v in res.items()}
    fwd = t["forward only (no_grad)"]
    for name, _, _ in modes:
        extra = f"  backward {t[name] - fwd:6.2f} ms" if name != "forward only (no_grad)" else ""
        say(f"  {name:32s} {t[name]:7.2f} ms{extra}   runs: " + " ".join(f"{v:.2f}" for v in res[name]))
    f, tr = t["frozen: data-only + input GEMM"], t["trainable: full + input GEMM"]
    say(f"  frozen / trainable call: {f / tr:.3f};  backward: {(f - fwd) / (tr - fwd):.3f}")
    say()
    del m


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    ops.check_device(0)
    torch.backends.cuda.matmul.allow_tf32 = False
    say(f"card: {card()}")
    say()
    gemm_leg()
    saliency_leg(384, 16)
    saliency_leg(224, 64)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
