#!/usr/bin/env python
"""Headline benchmark: ViT-B/16@384 training images/sec (BASELINE.json) on N B200s of one node.

  python bench.py --gpus 1 --steps 20 --warmup 5
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference --steps 5 --warmup 2      # HF fp32 CPU step on the host cores
  python bench.py --steps 20 --warmup 5 --dump-outputs DIR   # + the last timed step's outputs as DIR/*.npy

A step = forward + backward + AdamW (global-norm clip 1.0, as HF Trainer runs it) on a per-GPU
batch of 16 synthetic 384×384 images.  `value` is timed with CUDA events with the inputs already
in HBM; `e2e` goes through the public nn.Module call with the reference's collate contract
(fp32 [B,3,384,384] + fp32 labels) coming from pinned host memory every step and the loss read
back to the host.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ViT-B/16@384 train images/sec"
UNIT = "images/s"
TRAIN_GF_PER_IMG = 332.222          # SURVEY §8(d): algorithmic fwd+bwd GFLOP per image, ViT-B/16@384
PER_GPU_BATCH = 16
# BASELINE.json configs (SURVEY §8(d) algorithmic GFLOP per image: forward, forward+backward)
CONFIGS = {
    "vitb384": {"metric": METRIC, "name": "ViT-B/16@384", "batch": 16, "fwd_gf": 110.967, "train_gf": 332.222,
                "model": {}},                                                                    # configs[1] / configs[2]
    "vitl384": {"metric": "ViT-L/16@384 train images/sec", "name": "ViT-L/16@384", "batch": 8, "fwd_gf": 382.131,
                "train_gf": 1145.486,                                                            # configs[4]
                "model": {"hidden_size": 1024, "num_hidden_layers": 24, "num_attention_heads": 16, "intermediate_size": 4096}},
    "vitb224-infer": {"metric": "ViT-B/16@224 inference images/sec", "name": "ViT-B/16@224", "batch": 64, "fwd_gf": 35.126,
                      "train_gf": 105.147, "model": {"image_size": 224}},                        # configs[3]
}


def measured_traffic():
    """dram bytes per launch of the dominant kernel from the latest committed ncu --set full summary."""
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_roofline_traffic.json")))
    if not files:
        return None
    try:
        return float(json.load(open(files[-1]))["dram_bytes_per_launch"])
    except Exception:
        return None


def measured_traffic_detail():
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "*_roofline_traffic.json")))
    if not files:
        return None
    try:
        d = json.load(open(files[-1]))
        return {"file": os.path.relpath(files[-1], ROOT), "per_shape": d.get("per_shape"), "launches_profiled": d.get("launches_profiled")}
    except Exception:
        return None


def pick_peak(pk, clocks):
    """Which measured bf16 peak a number is held against: the burst figure (cuBLAS timed alone at boost clocks) unless
    the clock record of the SAME window shows the part power-capped or well below its maximum SM clock — the state
    MEASURED_PEAKS' sustained figure was taken in (1327 MHz at 993 W)."""
    if clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz"):
        capped = "sw_power_cap" in (clocks.get("reasons") or []) or clocks["sm_mhz"] < 0.85 * clocks["sm_max_mhz"]
        if capped:
            return "sustained", pk["tflops_sustained"]
    return "burst", pk["tflops_burst"]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_sustained": d["bf16_tflops_sustained"], "tflops_burst": d["bf16_tflops"], "hbm_gbs": d["hbm_gbs"],
                "src": "measured"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "src": "fallback"}


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock, power and clock-event (throttle) reasons of one GPU every ~10 ms from a background
    thread through NVML (what `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` reads) while the
    timed region runs; falls back to an nvidia-smi subprocess when pynvml is unavailable."""
    REASONS = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4,
               "hw_power_brake_slowdown": 0x80}

    def __init__(self, gpu_index: int):
        import threading
        self.samples = []
        self.stop_flag = False
        self.mode = None
        self.proc = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[gpu_index]) if vis and vis.split(",")[gpu_index].strip().isdigit() else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.mode = "nvml"
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception:
            q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
            self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
            try:
                self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                              "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
                self.mode = "smi"
            except OSError:
                pass

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.samples.append((sm, pw, rs))
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        if self.mode == "nvml":
            self.stop_flag = True
            self.t.join(timeout=2)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": ["no samples"]}
            reasons = sorted(n for n, bit in self.REASONS.items() if any(r & bit for _, _, r in self.samples))
            return {"sm_mhz": statistics.median(s for s, _, _ in self.samples), "sm_max_mhz": self.max_sm,
                    "power_w_max": max(p for _, p, _ in self.samples), "samples": len(self.samples), "reasons": reasons,
                    "source": "NVML, 10 ms period, during the timed region"}
        if self.mode != "smi":
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        reasons = set()
        for r in rows:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if r[col].strip().lower() == "active":
                    reasons.add(name)
        return {"sm_mhz": statistics.median(float(r[1]) for r in rows), "sm_max_mhz": float(rows[0][2]),
                "power_w_max": max(float(r[3]) for r in rows), "samples": len(rows), "reasons": sorted(reasons),
                "source": "nvidia-smi -lms 20 during the timed region"}


# ----------------------------------------------------------------------------- reference arm (CPU)
def hf_cpu_step_fn(batch: int):
    """The reference's own implementation of the path: HF ViTForImageClassification fp32 on the
    host cores (ViT-Training.py:83-90 + Trainer's fwd/bwd/AdamW).  Falls back to the oracle port
    when transformers is not importable.  Returns (step_fn, kind)."""
    import torch
    from oracle import vit_oracle as O
    cfg = O.VIT_B16_384
    torch.manual_seed(0)
    params = O.init_params(cfg, 0, 123)
    g = torch.Generator().manual_seed(1)
    x8, y = O.synth_inputs(cfg, batch, g)
    x = O.normalize_gray(x8)
    try:
        from oracle.make_golden import hf_model
        m, _ = hf_model(cfg, params)
        opt = torch.optim.AdamW(m.parameters(), lr=2e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0)

        def step():
            out = m(pixel_values=x, labels=y)
            out.loss.backward()
            torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
            opt.step()
            opt.zero_grad(set_to_none=True)
            return float(out.loss)
        return step, "reference"
    except Exception:                                   # transformers missing on this box
        state = {}

        def step():
            loss, _, grads = O.forward_backward(params, cfg, x, y)
            O.adamw_step(params, grads, state)
            return float(loss)
        return step, "port"


def time_cpu(batch: int, steps: int, warmup: int):
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, kind = hf_cpu_step_fn(batch)
    for _ in range(warmup):
        step()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        ts.append(time.perf_counter() - t0)
    total = sum(ts)
    return {"value": batch * steps / total, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind,
            "sample": f"{steps} fwd+bwd+AdamW steps of batch {batch} (ViT-B/16@384 fp32, HF transformers on CPU), "
                      f"{warmup} warm-up; median {statistics.median(ts):.3f} s/step"}, total / steps


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = 2
    cb, s_per_step = time_cpu(batch, args.steps, args.warmup)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "ViT-B/16@384 fwd+bwd+AdamW(clip 1.0), 14-label BCEWithLogits; CPU sample batch 2 per step",
                       "per_gpu_batch": PER_GPU_BATCH, "sample_batch": batch},
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def gemm_flops_of_plan(plan):
    return [plan.gemm_flops.get(i) for i in range(len(plan.steps))]


def instrumented_gemm_time(ar, plans, stream):
    """Run the plans once with a CUDA-event pair around every GEMM launch (same stream the kernels
    run on); returns (Σ algorithmic FLOPs, Σ ms, launches) over all GEMM launches."""
    import torch
    tot_f, evs, n = 0.0, [], 0
    torch.cuda.synchronize()
    torch.cuda._sleep(4_000_000)   # ≈2 ms head start: the host enqueues ahead of the GPU, so each event pair brackets
                                   # device time only (an idle GPU would add the host's launch latency to every interval)
    for plan in plans:
        fl = gemm_flops_of_plan(plan)
        for (fn, a, name), f in zip(plan.steps, fl):
            if fn is None:
                if name == "python":
                    a[0]()
                continue           # fork / join markers: this replay is single-stream
            if f is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                rc = fn(*a, stream)
                e1.record()
                evs.append((e0, e1))
                tot_f += f
                n += 1
            else:
                rc = fn(*a, stream)
            assert rc == 0, name
    torch.cuda.synchronize()
    return tot_f, sum(a.elapsed_time(b) for a, b in evs), n


def gemm_chain_time(plans, stream, reps=3):
    """All GEMM launches of the plans back to back on the launch stream (programmatic-dependent-launch chain intact, as
    in the step) inside ONE CUDA-event pair; returns (Σ algorithmic FLOPs, best ms, launches).  The buffers hold a real
    step's data, so shapes, epilogues and memory footprints are the step's own."""
    import torch
    calls, tot_f = [], 0.0
    for plan in plans:
        for (fn, a, name), f in zip(plan.steps, gemm_flops_of_plan(plan)):
            if fn is not None and f is not None:
                calls.append((fn, a))
                tot_f += f
    best = float("inf")
    for _ in range(reps):
        torch.cuda.synchronize()
        torch.cuda._sleep(4_000_000)      # head start: the host enqueues ahead of the GPU
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for fn, a in calls:
            rc = fn(*a, stream)
            assert rc == 0
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    return tot_f, best, len(calls)


DUMP_PARAM_SAMPLE = 1 << 22         # fp32 parameters kept by --dump-outputs: 16 MB of ViT-B's 344 MB (ViT-L: 1.2 GB)


def last_step_outputs(model, B, loss):
    """On-device copies of what the last timed training step computed, taken before any later leg overwrites it: the
    loss, the logits (the arena buffer the module's output is cloned from; the backward and the optimizer leave it
    alone) and a fixed seeded sample of the updated fp32 master parameters."""
    import torch
    flat = model.flat_parameters()
    g = torch.Generator().manual_seed(0)
    idx = torch.randint(0, flat.numel(), (min(DUMP_PARAM_SAMPLE, flat.numel()),), generator=g).to(flat.device)
    return {"loss": torch.tensor([loss], dtype=torch.float32), "logits": model.engine().arena(B, True).logits.clone(),
            "params_sample": flat[idx]}


def write_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def build_model(conf, dev):
    import torch
    import chest_x_ray_vit_b200 as pkg
    from oracle import vit_oracle as O      # only for the seeded synthetic-parameter / input recipe (outside timed regions)
    cfg = pkg.ViTConfig(**conf["model"])
    ocfg = O.OracleConfig(image_size=cfg.image_size, hidden_size=cfg.hidden_size, num_hidden_layers=cfg.num_hidden_layers,
                          num_attention_heads=cfg.num_attention_heads, intermediate_size=cfg.intermediate_size)
    torch.manual_seed(0)
    model = pkg.ViTForImageClassification(cfg)
    model.load_state_dict(O.init_params(ocfg, 0, 123))
    return model.to(dev), cfg


def run_ours(args):
    import torch
    import torch.distributed as dist
    import chest_x_ray_vit_b200 as pkg
    from chest_x_ray_vit_b200.data import DeviceFeeder
    from chest_x_ray_vit_b200.parallel import GradSync, PeerGradSync, broadcast_parameters
    from oracle import vit_oracle as O      # only for the seeded synthetic-input recipe and the cpu_baseline leg

    conf = CONFIGS[args.config]
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    pkg.ops.check_device(local)

    B, K, W = (args.batch or conf["batch"]), args.steps, args.warmup
    model, cfg = build_model(conf, dev)
    model.train()
    S = cfg.image_size
    train_gf = conf["train_gf"]
    if world > 1:
        broadcast_parameters(model)
        sync = args.sync if args.sync != "auto" else ("peer" if world <= 4 else "nccl")
        if sync == "peer":
            # symmetric memory needs P2P mappings between all GPUs of the job: if any rank cannot set it up, every rank
            # falls back to the NCCL sync together (the choice is agreed with a MIN all-reduce)
            ok = 1
            try:
                PeerGradSync.attach(model, layers_per_bucket=args.layers_per_bucket)
            except Exception as e:                          # noqa: BLE001
                sys.stderr.write(f"[rank {rank}] PeerGradSync unavailable ({type(e).__name__}: {e}); using NCCL\n")
                ok = 0
            flag = torch.tensor([ok], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if flag.item() == 0:
                sync = "nccl"
                model._engine = None
        if sync == "nccl":
            GradSync.attach(model, layers_per_bucket=args.layers_per_bucket)
    elif os.environ.get("VITK_BENCH_SEGMENTED") == "1":
        # diagnostic: one GPU running the N>1 launch plan (backward cut into graph segments at the bucket boundaries, host
        # callbacks in between) with nothing to communicate — isolates what the segmentation itself costs
        GradSync.attach(model, layers_per_bucket=args.layers_per_bucket)
    opt = pkg.VitkAdamW(model, lr=2e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, max_grad_norm=1.0)

    g = torch.Generator().manual_seed(1 + rank)
    nbuf = 4                                               # rotating distinct synthetic batches
    x8 = torch.randint(0, 256, (nbuf, B, S, S), dtype=torch.uint8, generator=g)
    yh = (torch.rand(nbuf, B, cfg.num_labels, generator=g) < 0.1).float()
    x_dev = [O.normalize_gray(x8[i].unsqueeze(1)).cuda() for i in range(nbuf)]      # fp32 [B,3,S,S] resident in HBM
    y_dev = [yh[i].cuda() for i in range(nbuf)]

    if args.graph:
        stepper = pkg.graph.GraphedTrainStep(model, opt)
        step = stepper
    else:
        def step(x, y):
            out = model(pixel_values=x, labels=y)
            out.loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            return out.loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(n, sample_clocks):
        """n steps on device-resident inputs inside one CUDA-event pair; returns (ms max over ranks, launches, clocks, loss)."""
        sampler = ClockSampler(local) if (sample_clocks and (rank == 0 or world > 1)) else None
        n0 = pkg.ops.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(n):
            loss = step(x_dev[i % nbuf], y_dev[i % nbuf])
        e1.record()
        barrier()
        own_ms = e0.elapsed_time(e1)
        t = torch.tensor([own_ms], device=dev)
        launches = pkg.ops.launch_count() - n0
        clocks = sampler.stop() if sampler else None
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            if clocks is not None:
                # every rank's own device time and SM clock / power: the step is as fast as the slowest GPU of the box
                mine = {"rank": rank, "ms_per_step": own_ms / n, "sm_mhz": clocks.get("sm_mhz"), "power_w_max": clocks.get("power_w_max"),
                        "reasons": clocks.get("reasons")}
                allr = [None] * world
                dist.all_gather_object(allr, mine)
                if rank == 0:
                    clocks["per_rank"] = allr
        return t.item(), launches, clocks, float(loss.detach())

    # ---------------- device-resident timing (`value`)
    for i in range(W):
        step(x_dev[i % nbuf], y_dev[i % nbuf])
    barrier()
    ms_max, launches, clocks, last_loss = timed(K, True)
    value = world * B * K / (ms_max / 1e3)
    dump = last_step_outputs(model, B, last_loss) if (args.dump_outputs and rank == 0) else None

    # ---------------- end-to-end through the public API with host buffers (`e2e`)
    # the reference's collate contract (fp32 [B,3,S,S] + fp32 labels, ViT-Training.py:77-80) in pinned host memory, fed by
    # the package's DeviceFeeder (pinned → copy stream → double-buffered device slots); loss read back every step
    xh = [O.normalize_gray(x8[i].unsqueeze(1)).pin_memory() for i in range(nbuf)]
    yp = [yh[i].pin_memory() for i in range(nbuf)]
    loss_host = torch.zeros(K, dtype=torch.float32).pin_memory()

    def host_batches(n):
        for i in range(n):
            yield {"pixel_values": xh[i % nbuf], "labels": yp[i % nbuf]}

    def e2e_loop(n, record_loss):
        feeder = DeviceFeeder(host_batches(n), device=dev)
        for i, batch in enumerate(feeder):
            l = step(batch["pixel_values"], batch["labels"])
            if record_loss:
                loss_host[i].copy_(l.detach(), non_blocking=True)
        return feeder

    e2e_loop(max(2, W // 2), False)
    barrier()
    e2e_sampler = ClockSampler(local) if rank == 0 else None
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    feeder = e2e_loop(K, True)
    f1.record()
    barrier()
    e2e_clocks = e2e_sampler.stop() if e2e_sampler else None
    t2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / (t2.item() / 1e3)
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": feeder.h2d_bytes // K * world, "d2h_bytes_per_step": 4 * world,
           "input": f"fp32 [B,3,{S},{S}] + fp32 labels [B,14] from pinned host memory through chest_x_ray_vit_b200.data.DeviceFeeder "
                    "(copy stream, double-buffered device slots), loss read back every step",
           "ms_per_step": t2.item() / K, "last_loss": float(loss_host[K - 1]), "clocks": e2e_clocks,
           "order": "timed right after `value` (same power state), before the `sustained` loop"}

    # ---------------- the same loop for >= 3 s: what the step does once the part has had time to reach its power state
    sustained = None
    if args.sustained_seconds > 0:
        n_sus = max(K, int(args.sustained_seconds * 1e3 / (ms_max / K)) + 1)
        s_ms, _, s_clocks, _ = timed(n_sus, True)
        sustained = {"value": world * B * n_sus / (s_ms / 1e3), "unit": UNIT, "steps": n_sus, "seconds": s_ms / 1e3,
                     "ms_per_step": s_ms / n_sus, "clocks": s_clocks}

    # ---------------- roofline of the dominant kernel (all tcgen05 GEMM launches of a step)
    roof = None
    if rank == 0:
        pk = peaks()
        eng = model.engine()
        ar = eng.arena(B, True)
        eng.grad_sync = None                                # single-rank measurement: no collectives here
        stream = torch.cuda.current_stream().cuda_stream
        ar.labels.copy_(y_dev[0])
        pkg.ops.patchify_f32(x_dev[0], out=ar.apatch)
        for _ in range(2):
            flops, gms, n = instrumented_gemm_time(ar, [ar.fwd_loss, ar.bwd_loss], stream)
        per_launch = flops / (gms / 1e3) / 1e12
        cflops, cms, cn = gemm_chain_time([ar.fwd_loss, ar.bwd_loss], stream)
        achieved = cflops / (cms / 1e3) / 1e12
        model._grads_clean = False                          # the replayed backward plans wrote into the gradient buffer
        step_tf = value / world * train_gf / 1e3
        step_kind, step_peak = pick_peak(pk, clocks)
        roof = {"bound": "tensor", "kernel": "gemm2_bf16_kernel / gemm_bf16_kernel (all forward/dgrad/wgrad launches of one step)",
                "achieved": achieved, "peak": pk["tflops_burst"], "unit": "TFLOP/s", "frac": achieved / pk["tflops_burst"],
                "frac_burst": achieved / pk["tflops_burst"], "frac_sustained": achieved / pk["tflops_sustained"],
                "peak_burst": pk["tflops_burst"], "peak_sustained": pk["tflops_sustained"],
                "peak_choice": f"burst: the GEMM chain is timed as an isolated {cms:.1f} ms burst after an idle gap (boost clocks), "
                               "the state MEASURED_PEAKS' burst figure was taken in",
                "traffic": measured_traffic(), "traffic_detail": measured_traffic_detail(),
                "launches_per_step": cn, "gemm_ms_per_step": cms,
                "how": "one CUDA-event pair around the step's GEMM launches issued back to back on the launch stream "
                       "(average launch duration = that time / launches)",
                "achieved_event_pair_per_launch": per_launch, "gemm_ms_per_step_event_pair_per_launch": gms,
                "peak_source": pk["src"],
                "step_tflops": step_tf, "step_tensor_frac": step_tf / step_peak, "step_tensor_frac_peak": step_kind,
                "step_tensor_frac_burst": step_tf / pk["tflops_burst"], "step_tensor_frac_sustained": step_tf / pk["tflops_sustained"]}
        if sustained is not None:
            kind, peak = pick_peak(pk, sustained["clocks"])
            stf = sustained["value"] / world * train_gf / 1e3
            sustained.update({"step_tflops": stf, "step_tensor_frac": stf / peak, "step_tensor_frac_peak": kind})
    if world > 1:
        dist.barrier()

    if rank == 0:
        cb = None
        if world == 1 and not args.no_cpu_baseline and args.config == "vitb384":
            cb, _ = time_cpu(2, 5, 2)
        line = {"metric": conf["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic",
                "config": {"workload": f"{conf['name']} fwd+bwd+AdamW(clip 1.0), 14-label BCEWithLogits, batch {B}/GPU "
                                       f"(global {B * world}), bf16 compute / fp32 master+grads",
                           "per_gpu_batch": B, "global_batch": B * world, "tokens": cfg.seq_len, "parallelism": f"dp{world}",
                           "l2": "per-step working set (GBs of saved activations + params/grads/moments) exceeds the 126 MB L2; "
                                 "4 rotating input batches", "train_gflop_per_image": train_gf,
                           "cuda_graph": bool(args.graph),
                           "grad_sync": (None if world == 1 else ("PeerGradSync: symmetric memory + copy engines over NVLink"
                                                                  if sync == "peer" else "GradSync: bucketed NCCL all-reduce"))},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "loss": last_loss}
        if sustained is not None:
            line["sustained"] = sustained
        if cb is not None:
            line["cpu_baseline"] = cb
        if dump is not None:
            write_outputs(args.dump_outputs, dump)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_infer_sweep(args):
    """BASELINE.json configs[3]: ViT-B/16@224 (197 tokens) inference-only throughput, batch 1 … 512, one B200.
    eval() + no_grad forward through the public module call on device-resident fp32 [B,3,224,224] inputs; per batch
    size: images/s (CUDA events over `steps` forwards after `warmup`), fraction of the measured bf16 burst peak against
    SURVEY App. B.1's 35.126 GF/image."""
    import torch
    import chest_x_ray_vit_b200 as pkg
    from oracle import vit_oracle as O
    conf = CONFIGS["vitb224-infer"]
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    pkg.ops.check_device(0)
    model, cfg = build_model(conf, dev)
    model.eval()
    pk = peaks()
    g = torch.Generator().manual_seed(1)
    sweep = []
    batches = args.batch_sweep
    nbuf = 4
    total_launches = 0
    sampler = ClockSampler(0)
    with torch.no_grad():
        for B in batches:
            x8 = torch.randint(0, 256, (nbuf, B, 224, 224), dtype=torch.uint8, generator=g)
            xs = [O.normalize_gray(x8[i].unsqueeze(1)).cuda() for i in range(nbuf)]
            fwd = pkg.graph.GraphedForward(model, xs[0]) if args.graph else (lambda x: model(pixel_values=x).logits)
            for i in range(max(args.warmup, 3)):
                fwd(xs[i % nbuf])
            n = args.steps if B >= 32 else args.steps * 4
            torch.cuda.synchronize()
            n0 = pkg.ops.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                out = fwd(xs[i % nbuf])
            e1.record()
            torch.cuda.synchronize()
            total_launches += pkg.ops.launch_count() - n0
            ms = e0.elapsed_time(e1) / n
            ips = B / (ms / 1e3)
            sweep.append({"batch": B, "images_per_s": ips, "ms_per_forward": ms,
                          "tensor_frac_burst": ips * conf["fwd_gf"] / 1e3 / pk["tflops_burst"], "finite": bool(torch.isfinite(out).all())})
            del xs
    clocks = sampler.stop()
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"logits": out})      # the last timed forward, at the last batch size
    best = max(sweep, key=lambda r: r["images_per_s"])
    line = {"metric": conf["metric"], "value": best["images_per_s"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": best["ms_per_forward"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic",
            "config": {"workload": f"ViT-B/16@224 eval()+no_grad forward, batch sweep {batches}; value = best batch ({best['batch']})",
                       "tokens": cfg.seq_len, "fwd_gflop_per_image": conf["fwd_gf"], "cuda_graph": bool(args.graph),
                       "l2": "4 rotating input batches; weights (172 MB bf16) exceed L2"},
            "sweep": sweep, "clocks": clocks, "gpu_launches": int(total_launches)}
    print(json.dumps(line), flush=True)


def main():
    # libraries (NCCL's version banner, …) write to fd 1: route everything to stderr and keep the real stdout for
    # the single JSON line
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="vitb384", choices=sorted(CONFIGS),
                    help="vitb384 = BASELINE configs[1]/[2] (the headline, default); vitl384 = configs[4]; vitb224-infer = configs[3]")
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the config's — 16 for ViT-B, 8 for ViT-L)")
    ap.add_argument("--batch-sweep", type=lambda v: [int(x) for x in v.split(",")], default=[1, 2, 4, 8, 16, 32, 64, 128, 256, 512],
                    help="vitb224-infer: batch sizes")
    ap.add_argument("--sustained-seconds", type=float, default=0.0,
                    help="after the K timed steps, keep stepping for this long and report it as `sustained` (default 0: skip, "
                         "so that --steps is the number of timed training steps)")
    ap.add_argument("--graph", action="store_true", help="replay the step from a captured CUDA graph (chest_x_ray_vit_b200.graph)")
    ap.add_argument("--layers-per-bucket", type=lambda v: [int(x) for x in v.split(",")], default=[3, 3, 3, 2, 1], help="encoder layers per all-reduce bucket, in the order layers finish backward; last entry repeats (3 layers = 85 MB; tapered so the all-reduce left after backward is short)")
    ap.add_argument("--sync", default="auto", choices=["auto", "peer", "nccl"],
                    help="gradient all-reduce at N>1: copy engines over NVLink peer memory (PeerGradSync) or NCCL (GradSync); auto = "
                         "peer up to 4 GPUs (measured 0.973 vs 0.953 at N=2), NCCL at 8 (0.912 vs 0.905)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32): loss, logits and a fixed "
                         "seeded sample of the updated parameters (training), logits (vitb224-infer); inputs are seeded, "
                         "so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs records the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        if args.warmup < 3:
            args.warmup = 3
        if args.config == "vitb224-infer":
            run_infer_sweep(args)
        else:
            run_ours(args)


if __name__ == "__main__":
    main()
