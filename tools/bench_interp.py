"""Cost of running the 384-px ViT-B/16 at other resolutions (``interpolate_pos_encoding=True``) on one GPU.

1. ms per training step (forward + backward + VitkAdamW) at batch 16 for 384 px (the plain call), 448, 512 and 640 px,
   each with its algorithmic GFLOP per image on the dense convention of bench.py (every token through every layer, the
   CLS-only top layer counted dense; backward = 2 × forward).  Sizes alternated, 5 repeats of 5 steps, median reported.
2. ms per eval forward (torch.no_grad) at 512 px, batch 16 and 64.
3. vitk_pos_interp and vitk_pos_interp_bwd alone (D = 768, 24×24 → 32×32 and → 40×40): CUDA events around 200
   back-to-back launches; the share of the HBM bound counts the bytes each kernel must move once (table read once,
   output written once; the adjoint reads dout and reads + writes dpos) at the data sheet's 7.7 TB/s.  The tables fit in
   L2, so after the first launch the reads come from there: the share can exceed what HBM alone would allow.

Usage: python tools/bench_interp.py [--out FILE]   (the text printed is also written to FILE)
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
HBM_BPS = 7.7e12
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


def gf_per_image(S, D=768, L=12, Fi=3072, C=14, train=True):
    """Algorithmic GFLOP per image at S×S px, dense convention (bench.py): 2·M·N·K of every GEMM, QKᵀ and PV."""
    P = (S // 16) ** 2
    T = P + 1
    fwd = 2 * P * 768 * D + L * (2 * T * D * 3 * D + 2 * 2 * T * T * D + 2 * T * D * D + 2 * 2 * T * D * Fi) + 2 * D * C
    return fwd * (3 if train else 1) / 1e9


def step_leg(sizes=(384, 448, 512, 640), B=16, reps=5, steps=5):
    torch.manual_seed(0)
    m = pkg.ViTForImageClassification(pkg.ViTConfig(image_size=384)).cuda().train()
    opt = pkg.VitkAdamW(m, lr=1e-5)
    data = {S: (torch.rand(B, 3, S, S, device=dev) * 2 - 1, (torch.rand(B, 14, device=dev) < 0.1).float()) for S in sizes}

    def step(S):
        x, y = data[S]
        kw = {} if S == 384 else {"interpolate_pos_encoding": True}
        m(pixel_values=x, labels=y, **kw).loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
    for S in sizes:                      # build and capture every plan first
        for _ in range(3):
            step(S)
    torch.cuda.synchronize()
    res = {S: [] for S in sizes}
    for _ in range(reps):
        for S in sizes:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                step(S)
            e1.record()
            torch.cuda.synchronize()
            res[S].append(e0.elapsed_time(e1) / steps)
    say(f"ViT-B/16 (384-px checkpoint), batch {B}: training step (forward + backward + VitkAdamW), ms per step")
    base = None
    for S in sizes:
        t = sorted(res[S])[len(res[S]) // 2]
        gf = gf_per_image(S)
        base = base or t
        tag = "plain call" if S == 384 else "interpolate_pos_encoding=True"
        say(f"  {S:4d} px  T = {(S // 16) ** 2 + 1:5d}  {t:8.2f} ms  {B * 1e3 / t:7.1f} img/s  {gf:6.1f} GF/image  "
            f"{B * gf / t:7.1f} TFLOP/s algorithmic  ({tag}; {t / base:.2f}× 384 px)   runs: "
            + " ".join(f"{v:.2f}" for v in res[S]))
    say()
    return m


def eval_leg(m, S=512, batches=(16, 64), reps=5, calls=5):
    m.eval()
    say(f"ViT-B/16 (384-px checkpoint) at {S} px: eval forward (torch.no_grad), ms per call")
    for B in batches:
        x = torch.rand(B, 3, S, S, device=dev) * 2 - 1
        with torch.no_grad():
            for _ in range(3):
                m(pixel_values=x, interpolate_pos_encoding=True)
            torch.cuda.synchronize()
            runs = []
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(calls):
                    m(pixel_values=x, interpolate_pos_encoding=True)
                e1.record()
                torch.cuda.synchronize()
                runs.append(e0.elapsed_time(e1) / calls)
        t = sorted(runs)[len(runs) // 2]
        gf = gf_per_image(S, train=False)
        say(f"  batch {B:3d}  {t:8.2f} ms  {B * 1e3 / t:7.1f} img/s  {gf:6.1f} GF/image  {B * gf / t:7.1f} TFLOP/s algorithmic"
            f"   runs: " + " ".join(f"{v:.2f}" for v in runs))
        del x
    say()
    m.train()


def events_us(fn, n=200):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n * 1e3


def kernel_leg(s=24, D=768, grids=((32, 32), (40, 40))):
    say(f"vitk_pos_interp / vitk_pos_interp_bwd alone, D = {D}, {s}×{s} table; 200 launches between one event pair, "
        "5 repeats, median")
    pos = torch.randn(1 + s * s, D, device=dev)
    dpos = torch.zeros(1 + s * s, D, device=dev)
    for gh, gw in grids:
        out = torch.empty(1 + gh * gw, D, device=dev)
        fwd_bytes = (pos.numel() + out.numel()) * 4
        bwd_bytes = (out.numel() + 2 * dpos.numel()) * 4
        cases = (("pos_interp", lambda: ops.pos_interp(pos, s, s, gh, gw, out=out), fwd_bytes),
                 ("pos_interp_bwd", lambda: ops.pos_interp_bwd(out, gh, gw, s, s, dpos), bwd_bytes))
        for name, fn, nbytes in cases:
            for _ in range(10):
                fn()
            torch.cuda.synchronize()
            t = sorted(events_us(fn) for _ in range(5))[2]
            bound = nbytes / HBM_BPS * 1e6
            say(f"  {name:15s} {s}×{s} → {gh}×{gw}  {t:7.2f} us  moves {nbytes / 1e6:5.2f} MB  HBM bound {bound:5.2f} us  "
                f"({bound / t * 100:5.1f} % of it)")
    say()


def main():
    out_path = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    ops.check_device(0)
    say(f"card: {card()}")
    say()
    kernel_leg()
    m = step_leg()
    eval_leg(m)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
