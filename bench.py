#!/usr/bin/env python
"""Benchmark of the CtrLoRA denoising hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

Workload (BASELINE.json configs[1]): SD1.5 UNet + ControlNet (LoRA rank 128), 512x512 (latent 4x64x64), batch 4,
DDIM with classifier-free guidance 7.5.  One "step" = one DDIM step = eps for the conditional and unconditional
branches (one batch-8 pass of ControlNet + UNet) + the fused DDIM update.  Weights are random (no checkpoints
offline), inputs synthetic.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference ...                           # the reference's algorithm on the host CPU (oracle port)
    python bench.py ... --dump-outputs DIR                         # also write the last timed step's outputs as DIR/*.npy

N > 1 (torchrun): sampling does not exchange anything between images, so ranks are independent replicas
("replicas only", DESIGN.md §Multi-GPU); value = N * K steps / max-over-ranks time.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH, LATENT, CTX_TOKENS, CTX_DIM, CFG_SCALE = 4, 64, 77, 768, 7.5
CONFIG = os.path.join(ROOT, "configs", "ctrlora_finetune_sd15_rank128.yaml")
GF_PER_IMAGE_PASS = 1103.4  # algorithmic forward GFLOP of ControlNet(r=128) + UNet per image (BASELINE.md §2)


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def random_weights_(model, seed):
    """Variance-preserving random weights written straight on the GPU (same scale rules as oracle/synth.py)."""
    gen = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            g = torch.randn(p.shape, device=p.device, generator=gen)
            if "lora_layer.down" in name:
                g *= 1.0 / p.shape[0]
            elif "lora_layer.up" in name:
                g *= 0.05
            elif p.dim() >= 2:
                g *= (p[0].numel()) ** -0.5
            elif name.endswith(".weight"):
                g = 1.0 + 0.1 * g
            else:
                g *= 0.1
            p.copy_(g)


def build_model(device, seed=0, config=None):
    from ctrlora_b200 import dropin
    dropin.activate()
    from cldm.model import create_model
    model = create_model(config or CONFIG, init_weights=False)
    model = model.to(device).eval()
    random_weights_(model, seed)
    return model


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()

    def run(self):
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop_evt.wait(0.2)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=5)
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None,
                "sm_max_mhz": float(self.rows[0][1]) if self.rows and self.rows[0][1].replace(".", "").isdigit() else None,
                "samples": len(self.rows), "reasons": sorted(reasons)}


def ncu_gemm_traffic():
    """DRAM bytes of the GEMM family per DDIM step from the committed ncu launch list of this same workload
    (profiles/r2_shares_ddim_step.json, written by tools/launch_shares.py from `ncu --metrics ...dram__bytes...` over
    tools/profile_step.py); None when the capture is absent."""
    path = os.path.join(ROOT, "profiles", "r2_shares_ddim_step.json")
    try:
        fam = json.load(open(path))["families"]["gemm_tcgen05"]
        return fam["dram_bytes"] if fam["dram_bytes"] > 0 else None, os.path.relpath(path, ROOT)
    except Exception:
        return None, None


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("bf16_tflops_sustained", 1412.1), d.get("hbm_gbs", 6569.6), "measured (MEASURED_PEAKS.json)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


DUMP_MAX_ELEMENTS = 1 << 20  # a larger output is dumped as a sample of this many elements
DUMP_MAX_BYTES = 64 << 20


def host_copy(t):
    """fp32 host copy of an output for --dump-outputs: the whole tensor, or the same seeded sample of its elements in
    every run when it is larger than DUMP_MAX_ELEMENTS."""
    t = t.detach()
    if t.numel() > DUMP_MAX_ELEMENTS:
        idx = torch.randint(t.numel(), (DUMP_MAX_ELEMENTS,), generator=torch.Generator().manual_seed(0))
        t = t.reshape(-1)[idx.to(t.device)]
    return t.float().cpu()


def write_outputs(path, outputs):
    """outputs {name: host tensor} -> path/<name>.npy (float32), so that two builds can be compared output for output"""
    import numpy as np
    arrays = {name: t.numpy().astype(np.float32) for name, t in outputs.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, f"outputs to dump take {total} bytes, more than {DUMP_MAX_BYTES}"
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


def cpu_reference_pass(model_state, threads, n_images=1, seed=1):
    """One apply_model of the reference's algorithm (oracle port) on the host cores; returns seconds."""
    from oracle import ctrlora_oracle as O
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n_images, 4, LATENT, LATENT, generator=g)
    hint = torch.randn(n_images, 4, LATENT, LATENT, generator=g)
    ctx = torch.randn(n_images, CTX_TOKENS, CTX_DIM, generator=g)
    t = torch.full((n_images,), 501, dtype=torch.long)
    t0 = time.perf_counter()
    with torch.no_grad():
        O.apply_model(model_state, x, t, ctx, hint, 8, 320)
    return time.perf_counter() - t0


def cpu_state_dict(seed=0):
    """fp32 weights for the CPU oracle (same architecture, random values; generated on the host)."""
    from ctrlora_b200 import dropin
    dropin.activate()
    from cldm.model import create_model
    model = create_model(CONFIG, init_weights=False)
    g = torch.Generator().manual_seed(seed)
    sd = {}
    with torch.no_grad():
        for name, p in model.state_dict().items():
            if not name.startswith(("control_model.", "model.diffusion_model.")):
                continue
            v = torch.randn(p.shape, generator=g)
            if "lora_layer.down" in name:
                v *= 1.0 / p.shape[0]
            elif "lora_layer.up" in name:
                v *= 0.05
            elif p.dim() >= 2:
                v *= (p[0].numel()) ** -0.5
            elif name.endswith(".weight"):
                v = 1.0 + 0.1 * v
            else:
                v *= 0.1
            sd[name] = v
    return sd


def pick_cpu_threads(model_state=None):
    """Thread count for the CPU arm, measured on this box.  A micro-probe (conv + GEMM of the path's shapes) at 16 / 32 / 64 /
    all cores shortlists the two fastest counts; when the model is available one batch-1 apply_model at each of them decides
    (torch's intra-op scaling on this model is far from linear and differs between box classes: the round-1 runs of this arm
    spread 3.5x).  Returns (threads, host cores, {threads: probe ms})."""
    import torch.nn.functional as F
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (16, 32, 64, cores) if c <= cores} or {cores})
    x = torch.randn(1, 320, 64, 64)
    w = torch.randn(320, 320, 3, 3)
    a, b = torch.randn(4096, 320), torch.randn(320, 1280)
    probe = {}
    for c in cands:
        torch.set_num_threads(c)
        for _ in range(2):
            F.conv2d(x, w, padding=1); a @ b
        t0 = time.perf_counter()
        for _ in range(6):
            F.conv2d(x, w, padding=1); a @ b
        probe[c] = round((time.perf_counter() - t0) / 6 * 1e3, 3)
    short = sorted(cands, key=lambda c: probe[c])[:2]
    best = short[0]
    if model_state is not None and len(short) > 1:
        model_ms = {}
        for c in short:
            cpu_reference_pass(model_state, c)          # warm-up at this thread count
            model_ms[c] = cpu_reference_pass(model_state, c)
        best = min(model_ms, key=model_ms.get)
        probe.update({f"apply_model@{c}": round(v, 3) for c, v in model_ms.items()})
    torch.set_num_threads(best)
    return best, cores, probe


def cpu_reference_step(model_state, seed=1):
    """One DDIM step of the workload on the host: the reference's two apply_model calls (cond, uncond: cldm/ddim_hacked.py:188-192)
    over the batch of 4 -- executed image by image (8 batch-1 passes: every image's work is done, nothing is extrapolated;
    at batch 4 the reference's materialised [4, 8, 4096, 4096] fp32 attention matrices thrash the host caches and one step takes
    160 s on the 128-core box instead of ~25 s) -- then the CFG combine and the DDIM update."""
    from oracle import ctrlora_oracle as O
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(BATCH, 4, LATENT, LATENT, generator=g)
    hint = torch.randn(BATCH, 4, LATENT, LATENT, generator=g)
    ctx = torch.randn(BATCH, CTX_TOKENS, CTX_DIM, generator=g)
    uc = torch.randn(BATCH, CTX_TOKENS, CTX_DIM, generator=g)
    t = torch.full((1,), 501, dtype=torch.long)
    t0 = time.perf_counter()
    with torch.no_grad():
        e_c = torch.cat([O.apply_model(model_state, x[i:i + 1], t, ctx[i:i + 1], hint[i:i + 1], 8, 320) for i in range(BATCH)])
        e_u = torch.cat([O.apply_model(model_state, x[i:i + 1], t, uc[i:i + 1], hint[i:i + 1], 8, 320) for i in range(BATCH)])
        tab = O.ddim_tables(O.register_schedule(), 50, 0.0)
        O.ddim_update(x, O.cfg_combine(e_c, e_u, CFG_SCALE), tab, 25)
    return time.perf_counter() - t0


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (oracle port; /root/reference is a Python tree that
    cannot travel to the GPU box), same config / metric / unit.  One 'step' = one full DDIM step of the workload (two
    batch-4 apply_model passes + the update), not an extrapolated sample; the step count is cut to fit a few minutes."""
    if rank != 0:
        return
    sd = cpu_state_dict()
    threads, cores, probe = pick_cpu_threads(sd)
    budget_s = 240.0
    t_first = cpu_reference_step(sd)  # warm-up (also sizes the run)
    steps = max(3, min(args.steps, int(budget_s / t_first) - 1))
    times = sorted(cpu_reference_step(sd) for _ in range(steps))
    t_step = times[len(times) // 2]  # median: the arm has to be reproducible, a single stalled step must not move it
    value = 1.0 / t_step
    line = {"impl": "reference", "metric": "ddim_steps_per_sec", "value": value, "unit": "steps/s (batch 4, CFG)",
            "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": t_step * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.gpus),
            "cpu_baseline": {"value": value, "unit": "steps/s (batch 4, CFG)", "cores": threads, "host_cores": cores,
                             "kind": "port", "thread_probe_ms": probe,
                             "sample": f"{steps} full DDIM steps (8 image passes + CFG + update each), median {t_step:.2f} s, "
                                       f"min {times[0]:.2f} s, max {times[-1]:.2f} s"},
            "e2e": {"value": value, "unit": "steps/s (batch 4, CFG)", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_reference_gpu(args, rank, world):
    """--impl reference-gpu: the library comparator SURVEY.md §8(d) asks for -- the reference's algorithm (oracle port: plain
    torch ops = cuDNN / cuBLAS / ATen eager, N x N attention matrix materialised like the reference) on the SAME B200, in
    fp32 and under bf16 autocast.  Two sequential batch-4 passes per step like the reference's sampler.  Not a product path."""
    if rank != 0:
        return
    from oracle import ctrlora_oracle as O
    dev = torch.device("cuda", 0)
    sd = {k: v.to(dev) for k, v in cpu_state_dict().items()}
    g = torch.Generator().manual_seed(1)
    x = torch.randn(BATCH, 4, LATENT, LATENT, generator=g).to(dev)
    hint = torch.randn(BATCH, 4, LATENT, LATENT, generator=g).to(dev)
    ctx = torch.randn(BATCH, CTX_TOKENS, CTX_DIM, generator=g).to(dev)
    uc = torch.randn(BATCH, CTX_TOKENS, CTX_DIM, generator=g).to(dev)
    t = torch.full((BATCH,), 501, dtype=torch.long, device=dev)
    tab = O.ddim_tables(O.register_schedule(), 50, 0.0)

    def step():
        e_c = O.apply_model(sd, x, t, ctx, hint, 8, 320)
        e_u = O.apply_model(sd, x, t, uc, hint, 8, 320)
        return O.ddim_update(x, O.cfg_combine(e_c.float(), e_u.float(), CFG_SCALE), tab, 25)

    res = {}
    for name, ctxmgr in (("fp32", torch.autocast("cuda", enabled=False)), ("bf16_autocast", torch.autocast("cuda", dtype=torch.bfloat16))):
        with torch.no_grad(), ctxmgr:
            for _ in range(max(3, args.warmup)):
                step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step()
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        res[name] = {"ms_per_step": ms, "steps_per_sec": 1e3 / ms}
    line = {"impl": "reference-gpu", "metric": "ddim_steps_per_sec", "value": res["fp32"]["steps_per_sec"],
            "unit": "steps/s (batch 4, CFG)", "n_gpus": 1, "steps": args.steps, "warmup": max(3, args.warmup),
            "ms_per_step": res["fp32"]["ms_per_step"], "higher_is_better": True, "dtype": "f32 (torch eager, TF32 off)",
            "data": "synthetic", "config": workload_config(1), "variants": res,
            "note": "oracle port on cuda:0 = the reference's op sequence through cuDNN/cuBLAS/ATen; comparator only"}
    print(json.dumps(line))


def workload_config(n):
    return {"workload": "configs[1]: SD1.5 UNet + ControlNet LoRA rank-128, DDIM step with CFG 7.5, batch 4, 512x512 "
                        "(latent 4x64x64), 77x768 context; cond+uncond batched as one batch-8 pass",
            "batch_per_gpu": BATCH, "cfg_scale": CFG_SCALE, "ddim_steps_schedule": 50,
            "parallelism": f"replicas x{n}" if n > 1 else "single GPU",
            "l2": "no flush needed: 2.7 GB of fp16 weights stream through the 126 MB L2 every step"}


TRAIN_BATCH = 16
TF_PER_IMAGE_TRAIN = 2.11  # algorithmically necessary TFLOP per image of one finetune step at rank 128 (BASELINE.md §2)


def run_train(args, rank, local_rank, world, device, outputs=None):
    """BASELINE.json configs[2]: ctrlora_finetune_sd15_rank128 training step, synthetic pairs, batch 16 per GPU,
    data-parallel with ONE NCCL all-reduce of the flat trainable-gradient buffer per step.  Returns a dict; the last timed
    step's loss and the trained parameters go to `outputs` when it is given."""
    import torch.distributed as dist
    from ctrlora_b200 import dropin
    dropin.activate()
    from ctrlora_b200.train import FinetuneTrainer
    lora_rank = getattr(args, "lora_rank", 128)
    cfg = os.path.join(ROOT, "configs", f"ctrlora_finetune_sd15_rank{lora_rank}.yaml")
    model = build_model(device, seed=0, config=cfg)  # identical replicas
    trainer = FinetuneTrainer(model, lr=1e-5)
    B = getattr(args, "train_batch", TRAIN_BATCH)
    gen = torch.Generator().manual_seed(200 + rank)
    host = {"x0": torch.randn(B, 4, LATENT, LATENT, generator=gen).pin_memory(),
            "hint": torch.randn(B, 4, LATENT, LATENT, generator=gen).pin_memory(),
            "ctx": torch.randn(B, CTX_TOKENS, CTX_DIM, generator=gen).pin_memory(),
            "t": torch.randint(0, 1000, (B,), generator=gen).pin_memory(),
            "noise": torch.randn(B, 4, LATENT, LATENT, generator=gen).pin_memory()}
    order = ("x0", "hint", "ctx", "t", "noise")
    dev = [host[k].to(device) for k in order]
    trainer.capture(*dev)
    import gc
    gc.collect()
    gc.freeze()  # static module tree: keep generation-2 collections out of the timed loops

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        trainer.step(*dev)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = trainer.step(*dev)
    e1.record()
    barrier()
    if outputs is not None:  # before the next step overwrites the graph's loss buffer and the parameters
        outputs.update(train_loss=host_copy(loss), train_params=host_copy(trainer.G.flat_p))
    ms_dev = e0.elapsed_time(e1)
    loss_host = torch.empty(1).pin_memory()
    h2d = sum(host[k].numel() * host[k].element_size() for k in order)
    for _ in range(2):
        trainer.step(*[host[k].to(device, non_blocking=True) for k in order])
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        loss = trainer.step(*[host[k].to(device, non_blocking=True) for k in order])
        loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    t = torch.tensor([ms_dev, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = t.tolist()
    peak_tf, _, peak_src = measured_peaks()
    ips = world * B * args.steps / (ms_dev / 1e3)
    spread = replica_spread(trainer, world)
    return {"metric": "train_images_per_sec", "value": ips, "unit": f"images/s (512x512, rank {lora_rank})", "batch_per_gpu": B,
            "lora_rank": lora_rank,
            "ms_per_step": ms_dev / args.steps, "loss": float(loss_host.item()),
            "e2e": {"value": world * B * args.steps / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4},
            "allreduce_bytes_per_step": trainer.G.numel * 4 if world > 1 else 0, "trainable_params": trainer.G.numel,
            "replica_param_spread": spread,
            "roofline": {"bound": "tensor", "achieved": ips / world * TF_PER_IMAGE_TRAIN, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": ips / world * TF_PER_IMAGE_TRAIN / peak_tf, "peak_source": peak_src,
                         "note": "algorithmically necessary 2.11 TFLOP/image (no recompute, no frozen weight grads)"}}


PRETRAIN_BATCH = 8
TF_PER_IMAGE_PRETRAIN = 2.33  # the finetune step's 2.11 TF + dense weight gradients of every ControlNet conv / linear
# (= their forward cost: conv 122.4 + Linear 95.8 GF, SURVEY.md §8d) -- algorithmically necessary work per image


def run_pretrain(args, rank, local_rank, world, device, outputs=None):
    """BASELINE.json configs[3]: ctrlora_pretrain_sd15_9tasks_rank128, one task per mini-batch from the multi-task
    schedule (per-rank un-seeded permutations in the reference -> ranks generally train different tasks in a step), batch 8
    per GPU (global 64 on 8 GPUs).  All ControlNet parameters + the task's LoRA set are trained.  The last timed step's
    loss and the trained parameters go to `outputs` when it is given."""
    import numpy as np
    import torch.distributed as dist
    from ctrlora_b200 import dropin
    dropin.activate()
    from ctrlora_b200.scheduler import TaskSchedule
    from ctrlora_b200.train import PretrainTrainer
    cfg = os.path.join(ROOT, "configs", "ctrlora_pretrain_sd15_9tasks_rank128.yaml")
    model = build_model(device, seed=0, config=cfg)
    trainer = PretrainTrainer(model, lr=1e-5)
    B = PRETRAIN_BATCH
    gen = torch.Generator().manual_seed(300 + rank)
    host = {"x0": torch.randn(B, 4, LATENT, LATENT, generator=gen).pin_memory(),
            "hint": torch.randn(B, 4, LATENT, LATENT, generator=gen).pin_memory(),
            "ctx": torch.randn(B, CTX_TOKENS, CTX_DIM, generator=gen).pin_memory(),
            "t": torch.randint(0, 1000, (B,), generator=gen).pin_memory(),
            "noise": torch.randn(B, 4, LATENT, LATENT, generator=gen).pin_memory()}
    order = ("x0", "hint", "ctx", "t", "noise")
    dev = [host[k].to(device) for k in order]
    trainer.capture(*dev)  # one graph per task, shared memory pool
    np.random.seed(1000 + rank)  # a different permutation stream per rank, like the reference's un-seeded ranks
    sched = TaskSchedule(trainer.tasks, largest_dataset_size=B * 64, batch_size=B)
    tasks = []
    while len(tasks) < args.warmup + 2 * args.steps + 4:
        tasks += list(sched)
    it = iter(tasks)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        trainer.step(*dev, task=next(it))
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = trainer.step(*dev, task=next(it))
    e1.record()
    barrier()
    if outputs is not None:
        outputs.update(pretrain_loss=host_copy(loss), pretrain_params=host_copy(trainer.G.flat_p))
    ms_dev = e0.elapsed_time(e1)
    loss_host = torch.empty(1).pin_memory()
    h2d = sum(host[k].numel() * host[k].element_size() for k in order)
    for _ in range(2):
        trainer.step(*[host[k].to(device, non_blocking=True) for k in order], task=next(it))
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        loss = trainer.step(*[host[k].to(device, non_blocking=True) for k in order], task=next(it))
        loss_host.copy_(loss, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    t = torch.tensor([ms_dev, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = t.tolist()
    peak_tf, _, peak_src = measured_peaks()
    ips = world * B * args.steps / (ms_dev / 1e3)
    lay = trainer.layout
    spread = replica_spread(trainer, world)
    return {"metric": "pretrain_images_per_sec", "value": ips, "unit": "images/s (512x512, 9 tasks, rank 128)",
            "batch_per_gpu": B, "global_batch": B * world, "ms_per_step": ms_dev / args.steps, "loss": float(loss_host.item()),
            "tasks": len(trainer.tasks), "skipped_steps": trainer.skipped_steps,
            "e2e": {"value": world * B * args.steps / (ms_e2e / 1e3), "unit": "images/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": 4},
            "trainable_params": trainer.G.numel, "controlnet_params": lay["base"][1], "replica_param_spread": spread,
            "allreduce_cuts": trainer._overlap_cuts() if world > 1 else [],
            "allreduce_bytes_per_step": (4 * (lay["base"][1] + min(world, len(trainer.tasks)) * lay["lora"][trainer.tasks[0]][1])
                                         if world > 1 else 0),
            "roofline": {"bound": "tensor", "achieved": ips / world * TF_PER_IMAGE_PRETRAIN, "peak": peak_tf, "unit": "TFLOP/s",
                         "frac": ips / world * TF_PER_IMAGE_PRETRAIN / peak_tf, "peak_source": peak_src,
                         "note": "algorithmically necessary 2.33 TFLOP/image (finetune step + dense ControlNet weight gradients)"}}


def replica_spread(trainer, world):
    """max over the flat parameter buffer of |p_rank - p_rank0|: data-parallel replicas must stay bit-identical (every
    gradient element reduced exactly once before AdamW); 0.0 expected, None on one GPU"""
    if world <= 1:
        return None
    import torch.distributed as dist
    ref = trainer.G.flat_p.clone()
    dist.broadcast(ref, src=0)
    d = (trainer.G.flat_p - ref).abs().max()
    dist.all_reduce(d, op=dist.ReduceOp.MAX)
    return float(d.item())


def attention_roofline(device, batch=2 * BATCH, heads=8, n=LATENT * LATENT, d=40, reps=20):
    """CUDA-event time of the step's dominant attention launch (64x64 self-attention of a CFG batch) on its own."""
    from ctrlora_b200 import ops
    g = torch.Generator(device=device).manual_seed(7)
    mk = lambda *s: (torch.randn(*s, device=device, generator=g) * 0.5).half()
    q, k, v = mk(batch * n, heads * d), mk(batch * n, heads * d), mk(batch * n, heads * d)
    vt = v.view(batch, n, heads, d).permute(0, 2, 3, 1).contiguous()
    out = torch.empty_like(q)
    for _ in range(3):
        ops.attention(q, k, vt, batch, heads, n, n, d, out=out)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        ops.attention(q, k, vt, batch, heads, n, n, d, out=out)
    e1.record()
    torch.cuda.synchronize()
    exps = float(batch) * heads * n * n
    return {"us": e0.elapsed_time(e1) * 1e3 / reps, "exps": exps, "flops": 4.0 * exps * d}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--lora-rank", type=int, default=128, choices=[32, 64, 128, 256, 512],
                    help="training workload only: BASELINE.json configs[4] rank sweep (default: the rank-128 headline)")
    ap.add_argument("--train-batch", type=int, default=TRAIN_BATCH, help="training workload: images per GPU per step")
    ap.add_argument("--workload", default="sample+train", choices=["sample", "train", "sample+train", "pretrain"],
                    help="sample: configs[1] DDIM step (the headline line); train: configs[2] finetune step; default: both, "
                         "the training result rides in the line's 'train' key")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (DDIM x_prev / pred_x0; training loss and a fixed sample "
                         "of the trained parameters) to DIR/<name>.npy; the inputs are seeded, so two builds can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank, local_rank, world = dist_env()
    outputs = {} if args.dump_outputs and rank == 0 else None
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.impl == "reference-gpu":
        run_reference_gpu(args, rank, world)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    from ctrlora_b200 import dropin, ops
    dropin.activate()
    if args.workload == "pretrain":
        res = run_pretrain(args, rank, local_rank, world, device, outputs)
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        if rank == 0:
            line = {"metric": res["metric"], "value": res["value"], "unit": res["unit"], "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "fp16 (fp32 accumulate, fp32 master weights)", "data": "synthetic",
                    "config": {"workload": "configs[3]: ctrlora_pretrain_sd15_9tasks_rank128, multi-task schedule, batch 8 per "
                                           "GPU (global 64 on 8 GPUs), 512x512 (latent 4x64x64)",
                               "batch_per_gpu": PRETRAIN_BATCH, "parallelism": f"dp{world}"},
                    "e2e": res["e2e"], "roofline": res["roofline"], "pretrain": res}
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return
    if args.workload == "train":
        res = run_train(args, rank, local_rank, world, device, outputs)
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        if rank == 0:
            line = {"metric": res["metric"], "value": res["value"], "unit": res["unit"], "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                    "vs_baseline": None, "dtype": "fp16 (fp32 accumulate, fp32 master weights)", "data": "synthetic",
                    "config": {"workload": "configs[2]: ctrlora_finetune_sd15_rank128 training step, synthetic pairs, batch 16 "
                                           "per GPU, 512x512 (latent 4x64x64)", "batch_per_gpu": TRAIN_BATCH,
                               "parallelism": f"dp{world}"},
                    "e2e": res["e2e"], "roofline": res["roofline"], "train": res}
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return
    from cldm.ddim_hacked import DDIMSampler
    model = build_model(device, seed=rank)
    sampler = DDIMSampler(model, batched_cfg=True, use_cuda_graph=True)
    sampler.make_schedule(50, ddim_eta=0.0, verbose=False)
    S = len(sampler.ddim_timesteps)

    gen = torch.Generator().manual_seed(100 + rank)
    host = {"x": torch.randn(BATCH, 4, LATENT, LATENT, generator=gen).pin_memory(),
            "hint": torch.randn(BATCH, 4, LATENT, LATENT, generator=gen).pin_memory(),
            "ctx": torch.randn(BATCH, CTX_TOKENS, CTX_DIM, generator=gen).pin_memory(),
            "uc": torch.randn(BATCH, CTX_TOKENS, CTX_DIM, generator=gen).pin_memory()}
    dev = {k: v.to(device) for k, v in host.items()}
    cond = {"c_crossattn": [dev["ctx"]], "c_concat": [dev["hint"]]}
    ucond = {"c_crossattn": [dev["uc"]], "c_concat": [dev["hint"]]}

    def step(i, x, c=cond, u=ucond):
        index = S - 1 - (i % S)
        ts = torch.full((BATCH,), int(sampler.ddim_timesteps[index]), device=device, dtype=torch.long)
        return sampler.p_sample_ddim(x, c, ts, index=index, unconditional_guidance_scale=CFG_SCALE,
                                     unconditional_conditioning=u)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- launches per step (counted on an un-graphed pass through the C ABI)
    ops.LAUNCHES = 0
    x = dev["x"]
    with sampler.run_mode():
        for i in range(args.warmup):  # includes weight preparation, LoRA folding and the graph capture
            x, _ = step(i, x)
    torch.cuda.synchronize()
    def one_step_in_run():
        with sampler.run_mode():
            step(0, dev["x"])

    launches_per_step = ops.count_launches(one_step_in_run, sampler)

    # The module tree (3 000 modules, ~10^6 Python objects) is static from here on: move it out of the cyclic collector's
    # reach, as a serving process would -- a generation-2 pass over it costs ~100 ms and, landing inside the 20-step
    # end-to-end loop, moved that figure between 49 and 64 steps/s from run to run (tools/debug_e2e.py: 15.54 ms/step steady).
    import gc
    gc.collect()
    gc.freeze()

    # ---- (1) device-resident throughput
    clocks = ClockSampler(local_rank)
    clocks.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    x = dev["x"]
    with sampler.run_mode():  # the K steps of a sampling run share their conditioning (as in DDIMSampler.sample)
        for i in range(args.steps):
            x, pred_x0 = step(i, x)
    e1.record()
    barrier()
    ms_dev = e0.elapsed_time(e1)
    clk = clocks.stop()
    if outputs is not None:
        outputs.update(x_prev=host_copy(x), pred_x0=host_copy(pred_x0))

    # ---- (2) end to end through the public API with host buffers: H2D of the step's inputs, D2H of its result
    out_host = torch.empty(BATCH, 4, LATENT, LATENT).pin_memory()
    stats_host = torch.empty(BATCH).pin_memory()
    h2d = sum(host[k].numel() * 4 for k in ("x", "hint", "ctx", "uc")) + BATCH * 8
    d2h = out_host.numel() * 4 + stats_host.numel() * 4

    def e2e_step(i):
        d = {k: host[k].to(device, non_blocking=True) for k in ("x", "hint", "ctx", "uc")}
        c = {"c_crossattn": [d["ctx"]], "c_concat": [d["hint"]]}
        u = {"c_crossattn": [d["uc"]], "c_concat": [d["hint"]]}
        xp, _ = step(i, d["x"], c, u)
        out_host.copy_(xp, non_blocking=True)
        stats_host.copy_(sampler.last_stats, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the caller reads the result before issuing the next step
        host["x"].copy_(out_host)

    for i in range(3):
        e2e_step(i)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(args.steps):
        e2e_step(i)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)

    # ---- roofline of the dominant kernel (tcgen05 implicit GEMM): the step's GEMM launches are recorded on an
    # un-graphed step, then replayed back to back from one CUDA graph between two CUDA events (ops.replay_gemms)
    gemm_stats = ops.replay_gemms(one_step_in_run, sampler)
    attn_stats = attention_roofline(device)

    t = torch.tensor([ms_dev, ms_e2e], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = t.tolist()
    train_result = None
    if "train" in args.workload:
        del sampler, model
        torch.cuda.empty_cache()
        train_result = run_train(args, rank, local_rank, world, device, outputs)
    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)
    if rank == 0:
        peak_tf, peak_hbm, peak_src = measured_peaks()
        value = world * args.steps / (ms_dev / 1e3)
        e2e_value = world * args.steps / (ms_e2e / 1e3)
        ach = gemm_stats["flops"] / (gemm_stats["ms"] * 1e-3) / 1e12 if gemm_stats["ms"] > 0 else 0.0
        line = {"metric": "ddim_steps_per_sec", "value": value, "unit": "steps/s (batch 4, CFG)", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_dev / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16 (fp32 accumulate)",
                "data": "synthetic", "config": workload_config(world), "clocks": clk,
                "e2e": {"value": e2e_value, "unit": "steps/s (batch 4, CFG)", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / args.steps},
                "gpu_launches": launches_per_step * args.steps,
                "images_per_sec": value * BATCH,
                "model_tflops": value / world * 2 * BATCH * GF_PER_IMAGE_PASS / 1e3,
                "roofline": {"kernel": "gemm_tcgen05_kernel (all convs + linears of one step, replayed back to back from a CUDA graph)",
                             "bound": "tensor",
                             "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                             "peak_source": peak_src + ", sustained bf16/fp16 dense", "traffic": ncu_gemm_traffic()[0],
                             "traffic_unit": "DRAM bytes per step, all GEMM launches (ncu dram__bytes_read+write)",
                             "traffic_source": ncu_gemm_traffic()[1],
                             "launches": gemm_stats["launches"], "gflop_per_step": gemm_stats["flops"] / 1e9,
                             "share_of_step": gemm_stats["ms"] / (ms_dev / args.steps)}}
        # second kernel of the step (19 % of it): the d_head-40 self-attention of the 64x64 level, bound by exp2 throughput
        sm_mhz = (clk or {}).get("sm_mhz") or 1900.0
        peak_exp = 16.0 * torch.cuda.get_device_properties(device).multi_processor_count * sm_mhz * 1e6 / 1e12
        a_ach = attn_stats["exps"] / (attn_stats["us"] * 1e-6) / 1e12
        line["roofline_attention"] = {
            "kernel": "attention_stream64s_kernel (7 launches per step: 8 img x 8 heads x 4096 x 4096, d = 40)",
            "bound": "mufu (16 ex2 per clock per SM at the sampled SM clock)", "achieved": a_ach, "peak": peak_exp,
            "unit": "Texp/s", "frac": a_ach / peak_exp, "us_per_launch": attn_stats["us"],
            "tensor_tflops": attn_stats["flops"] / (attn_stats["us"] * 1e-6) / 1e12,
            "share_of_step": 7 * attn_stats["us"] * 1e-3 / (ms_dev / args.steps)}
        if train_result is not None:
            line["train"] = train_result
            # BASELINE.json's second headline metric, lifted to the top level so that the scaling record keeps it
            line["train_images_per_sec"] = train_result["value"]
            line["train_ms_per_step"] = train_result["ms_per_step"]
            line["train_e2e_images_per_sec"] = train_result["e2e"]["value"]
        if not args.no_cpu_baseline:
            sd = cpu_state_dict()
            threads, cores, probe = pick_cpu_threads(sd)  # includes warm-up passes at the chosen thread count
            tp = cpu_reference_step(sd)
            line["cpu_baseline"] = {"value": 1.0 / tp, "unit": "steps/s (batch 4, CFG)", "cores": threads, "host_cores": cores,
                                    "kind": "port", "thread_probe_ms": probe,
                                    "sample": f"ONE full DDIM step (8 image passes + CFG + update) after warm-up passes, {tp:.2f} s"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
