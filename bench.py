#!/usr/bin/env python
"""bench.py — rays/s (training) and fps (inference) of the Instant-NGP hot path on B200 (driver contract: task statement).

    python bench.py --gpus N --steps K --warmup W [--config NAME]     # this repository (CUDA, sm_100a)
    python bench.py --impl reference --gpus N --steps K ... [--config NAME]   # reference restatement on host cores

A training "step" = one pass of the hot path over one batch of synthetic rays:
get_rays -> ray/AABB -> occupancy march -> hash encode -> MLP(+SH) -> composite -> MSE -> backward ->
[grad all-reduce] -> fused Adam, plus update_density_grid every 16th step exactly like the reference's loop
(train.py:168-201).  An inference "step" = one 800x800 frame of gui.py:115-145 (get_rays + render(test_time=True)).

--config selects one of BASELINE.json's five configurations (default = configs[1], the one the metric is quoted on):
  lego_fp32_1024  configs[0]  Lego shape, batch 1024, fp32 hash encoder (the reference's CPU-runnable case)
  lego_half       configs[1]  Lego shape, batch 8192, fp16 hash encoder
  garden16        configs[2]  360_v2-garden shape: scale 16 (6 cascades), max_res 4096, exp_step_factor 1/256, batch 8192
  lego_8x         configs[3]  = lego_half per GPU, meant for --gpus 8 (global batch 65536, one NCCL all-reduce per step)
  frame800        configs[4]  800x800 test-time frame, fps
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 23
BATCH = 8192                  # rays per GPU of the default configuration (scripts/ use it)
UPDATE_INTERVAL = 16          # train.py:57-58
PREWARM = 20                  # extra untimed steps before the W warm-up steps
DENSITY_THRESHOLD = 0.01 * 1024 / 3 ** 0.5  # train.py:180
DUMP_SAMPLE = 1 << 20         # --dump-outputs: hash-table entries written (the full table can exceed 64 MB)

CONFIGS = {
    "lego_fp32_1024": dict(index=0, kind="train", n_rays=1024, half=False, scale=0.5, max_res=1024, esf=0.0,
                           img_wh=(800, 800), focal=1111.111, radius=1.4, cap=384,
                           workload="BASELINE configs[0]: Synthetic-NeRF Lego shape, batch 1024 rays/GPU, fp32 hash "
                                    "encoder L=16 T=2^19 F=2"),
    "lego_half": dict(index=1, kind="train", n_rays=8192, half=True, scale=0.5, max_res=1024, esf=0.0,
                      img_wh=(800, 800), focal=1111.111, radius=1.4, cap=384,
                      workload="BASELINE configs[1]: Synthetic-NeRF Lego shape, batch 8192 rays/GPU, fp16 hash encoder "
                               "L=16 T=2^19 F=2"),
    "garden16": dict(index=2, kind="train", n_rays=8192, half=True, scale=16.0, max_res=4096, esf=1.0 / 256,
                     img_wh=(1297, 840), focal=960.0, radius=1.3, cap=1024,
                     workload="BASELINE configs[2]: 360_v2 garden shape, scale 16 (6 occupancy cascades, multi-cascade "
                              "grids play the role of scene contraction), max_res 4096, exp_step_factor 1/256, "
                              "background 0, batch 8192 rays/GPU, fp16 hash encoder"),
    "lego_8x": dict(index=3, kind="train", n_rays=8192, half=True, scale=0.5, max_res=1024, esf=0.0,
                    img_wh=(800, 800), focal=1111.111, radius=1.4, cap=384,
                    workload="BASELINE configs[3]: Lego shape, 8192 rays per GPU sharded over the ranks (65536 at "
                             "--gpus 8) + one NCCL gradient all-reduce per step, fp16 hash encoder"),
    "frame800": dict(index=4, kind="frame", half=True, scale=0.5, max_res=1024, esf=0.0, img_wh=(800, 800),
                     focal=1111.111, radius=1.396,
                     workload="BASELINE configs[4]: 800x800 full-frame test-time ray march (gui.py path), occupancy "
                              "grid loaded, fps"),
}

# algorithmic bytes / flops per sample (SURVEY.md §8d): [fp16 encoder, fp32 encoder]
BYTES_PER_SAMPLE = {"hash_fwd": (588, 1164), "hash_bwd": (1100, 1164), "mlp_fwd": (86, 156), "mlp_bwd": (150, 284),
                    "ray_head": (22 + 32, 28 + 44), "march": (32, 32), "composite_fwd": (22, 28)}
FLOP_PER_SAMPLE = {"mlp_fwd": 18816, "mlp_bwd": 37632}
ADAM_BYTES_PER_PARAM = 34     # p, g, m, v read; p, m, v written; fp16 shadow written; grad zeroed (DESIGN.md §4)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return (float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1418.0))),
                "measured (MEASURED_PEAKS.json: HBM copy GB/s, sustained dense bf16 TFLOP/s)")
    return 6650.0, 1418.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(config, kernel, samples):
    """DRAM bytes per launch of `kernel` from the committed `ncu --set full` capture of this very command
    (profiles/r2_traffic.json, written by scripts/ncu_traffic.py).  None when no capture of this workload exists or
    the kernel was not captured; scaled by the sample ratio when the live sample count differs by more than 5 %."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f).get(config)
    if not d or kernel not in d.get("kernels", {}):
        return None, None
    src = d.get("source") or "profiles/r2_traffic.json (ncu --set full, one graph step, dram__bytes_read.sum + dram__bytes_write.sum)"
    if samples and abs(d["samples"] - samples) > 0.05 * samples:
        # the capture ran with another sample count (the count depends on how far the model has trained): per-sample
        # streams dominate these kernels' DRAM traffic, so the captured bytes are scaled by the ratio of the counts
        k = samples / d["samples"]
        return d["kernels"][kernel]["dram_bytes"] * k, src + f"; captured at {int(d['samples'])} samples, scaled x{k:.3f} to the live count"
    return d["kernels"][kernel]["dram_bytes"], src


# --------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def n_samples(self):
        return len(self.lines)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write what the timed path computed in its last step as <out_dir>/<name>.npy (float32, or
    float64 where the value is float64), so that two builds can be compared output for output on identical inputs.
    The hash-table gradient is accumulated with atomics, so two runs agree to float-reordering tolerance, not bitwise."""
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        total += a.nbytes
        np.save(os.path.join(out_dir, name + ".npy"), a)
    assert total <= 64 << 20, total


# --------------------------------------------------------------------------------------------------
def init_weights_numpy(seed, max_res=1024, half=True):
    """Random-init parameters shared by both arms: table U(-1e-4,1e-4) in half mode (hash_encoder_half.py:299),
    U(0,1) in fp32 mode (hash_encoder.py:227, torch.nn.init.uniform_); xavier-uniform MLP (networks.py:306-312)."""
    from taichi_nerfs_b200.layout import make_hash_layout
    rng = np.random.default_rng(seed)
    lay = make_hash_layout(2 ** 19, 16, 16, max_res, 2)
    u = rng.random((lay.total_entries, 2), dtype=np.float32)
    table = ((u * 2 - 1) * 1e-4).astype(np.float32) if half else u
    shapes = [(64, 32), (16, 64), (64, 32), (64, 64), (3, 64)]
    ws = [(rng.uniform(-1, 1, s) * math.sqrt(6.0 / (s[0] + s[1]))).astype(np.float32) for s in shapes]
    return lay, table, ws


def dist_setup(n_gpus):
    import torch
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    elif n_gpus > 1:
        raise SystemExit("--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    return world, rank, local


def mlp_params(model):
    return [model.xyz_encoder.hidden_layers[0].weight, model.xyz_encoder.output_layer.weight,
            model.rgb_net.hidden_layers[0].weight, model.rgb_net.hidden_layers[1].weight,
            model.rgb_net.output_layer.weight]


def make_timed(torch, world, dev):
    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return float(ms)
    return timed


# --------------------------------------------------------------------------------------------------
def run_train(args, cfg_name, cfg):
    import torch
    world, rank, local = dist_setup(args.gpus)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)

    from datasets.ray_utils import get_rays
    from datasets.synthetic import SyntheticLego
    from modules.networks import NGP
    from taichi_nerfs_b200 import _lib
    from taichi_nerfs_b200.fast_step import StaticTrainStep
    from taichi_nerfs_b200.trainer import NGPTrainer

    BATCH, half, esf = cfg["n_rays"], cfg["half"], cfg["esf"]
    torch.manual_seed(SEED + rank)
    lay, table, ws = init_weights_numpy(SEED, cfg["max_res"], half)
    model = NGP(scale=cfg["scale"], max_res=cfg["max_res"], half_opt=half).to(dev)
    with torch.no_grad():
        model.pos_encoder.hash_table.copy_(torch.from_numpy(table).view_as(model.pos_encoder.hash_table))
        for p, w in zip(mlp_params(model), ws):
            p.copy_(torch.from_numpy(w))
    ds = SyntheticLego(batch_size=BATCH, seed=SEED + rank, img_wh=cfg["img_wh"], focal=cfg["focal"],
                       radius=cfg["radius"]).to(dev)
    model.mark_invisible_cells(ds.K, ds.poses, ds.img_wh)
    with torch.autocast("cuda", dtype=torch.float16):
        model.update_density_grid(DENSITY_THRESHOLD, warmup=True)
    occupied = float(np.unpackbits(model.density_bitfield.cpu().numpy()).mean())
    trainer = NGPTrainer(model, lr=1e-2, max_steps=20000)

    n_total = args.steps + args.warmup
    batches = [ds[0] for _ in range(n_total)]                      # device-resident inputs
    host_batches = [{k: v.cpu().pin_memory() for k, v in b.items() if k in ("direction", "pose", "rgb")}
                    for b in batches]

    sample_counts = []
    fast = StaticTrainStep(trainer, BATCH, samples_per_ray_capacity=cfg["cap"], exp_step_factor=esf,
                           overlap_optimizer=not args.no_overlap)
    # the training set stays resident in HBM (train.py: `train_dataset.to(device)`), and the step draws its own
    # batch on the device (datasets/base.py:34-61 + get_rays as the first node of the graph)
    ds.build_image_bank()
    fast.attach_ray_source(ds.rays, ds.poses, ds.directions, seed=SEED + rank)

    def grid_update(step_idx):
        with torch.autocast("cuda", dtype=torch.float16):
            if step_idx % UPDATE_INTERVAL == 0:
                fast.flush()   # overlap mode: the grid update must see the parameters of the last step
                model.update_density_grid(DENSITY_THRESHOLD, warmup=step_idx < 256)

    def graph_step(step_idx, b):
        """StaticTrainStep: b None -> batch drawn on the device inside the graph; else caller-provided batch."""
        grid_update(step_idx)
        if b is None:
            loss = fast.step_sampled()
        else:
            rays_o, rays_d = get_rays(b["direction"], b["pose"])
            loss = fast.step(rays_o, rays_d, b["rgb"])
        sample_counts.append(fast.counter[0].clone())
        return loss

    def module_step(step_idx, b):
        """reference-shaped plugin API: render() (autograd Functions) + MSE + backward + NGPTrainer.optimizer_step"""
        grid_update(step_idx)
        rays_o, rays_d = get_rays(b["direction"], b["pose"])
        loss, results = trainer.step(rays_o, rays_d, b["rgb"], exp_step_factor=esf)
        sample_counts.append(results["rm_samples"])
        return loss

    use_graph = args.path == "graph"
    timed = make_timed(torch, world, dev)

    if args.ncu_window > 0:
        # the same steps the timed region starts with (state after the pre-warm = the initial state)
        keep = [t.clone() for t in (trainer.flat_param, trainer.exp_avg, trainer.exp_avg_sq, trainer.step_dev,
                                     trainer.hyper, trainer.scale_state, fast.sample_step)]
        for s in range(PREWARM):
            graph_step(1 + s % 8, None)
        fast.flush()
        for t, k in zip((trainer.flat_param, trainer.exp_avg, trainer.exp_avg_sq, trainer.step_dev, trainer.hyper,
                         trainer.scale_state, fast.sample_step), keep):
            t.copy_(k)
        if trainer._shadow_full is not None:
            trainer._shadow_full.copy_(trainer.flat_param)
        trainer.flat_grad.zero_()
        for s in range(args.warmup):
            graph_step(1 + s, None)
        fast.flush()
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for s in range(args.ncu_window):
            graph_step(args.warmup + 1 + s, None)
        fast.flush()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        if rank == 0:
            print(json.dumps({"ncu_window_steps": args.ncu_window, "config": cfg_name,
                              "samples_per_step": [int(c) for c in sample_counts[-args.ncu_window:]]}))
        return

    # ---- device-resident arm ("value") -------------------------------------------------------------
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    # The pre-warm below runs a clock-dependent number of steps.  The timed workload must not depend on it (every
    # step trains the model, which changes the next occupancy grid and with it the samples per ray), so the complete
    # training state is put back afterwards: the timed region always starts from "random init + one grid update".
    snap = {"param": trainer.flat_param.clone(), "m": trainer.exp_avg.clone(), "v": trainer.exp_avg_sq.clone(),
            "step_dev": trainer.step_dev.clone(), "hyper": trainer.hyper.clone(), "scale": trainer.scale_state.clone(),
            "shadow": None if trainer._shadow_full is None else trainer._shadow_full.clone(),
            "grid": model.density_grid.clone(), "bits": model.density_bitfield.clone(),
            "grid_step": model.__dict__.get("_grid_step", 0), "sample_step": fast.sample_step.clone(),
            "step_count": trainer.step_count, "rng": torch.cuda.get_rng_state(dev)}

    def restore_state():
        fast.flush()
        trainer.flat_param.copy_(snap["param"])
        trainer.exp_avg.copy_(snap["m"])
        trainer.exp_avg_sq.copy_(snap["v"])
        trainer.step_dev.copy_(snap["step_dev"])
        trainer.hyper.copy_(snap["hyper"])
        trainer.scale_state.copy_(snap["scale"])
        if snap["shadow"] is not None:
            trainer._shadow_full.copy_(snap["shadow"])
        trainer.flat_grad.zero_()
        model.density_grid.copy_(snap["grid"])
        model.density_bitfield.copy_(snap["bits"])
        model.__dict__["_grid_step"] = snap["grid_step"]
        fast.sample_step.copy_(snap["sample_step"])
        trainer.step_count = snap["step_count"]
        torch.cuda.set_rng_state(snap["rng"], dev)   # --path modules: the marching noise comes from torch's RNG
    # untimed pre-warm beyond --warmup: the caching allocator must have seen the range of per-step
    # sample counts (every new size is a cudaMalloc) and the clocks must have ramped up
    step_fn = (lambda i, k: graph_step(i, None)) if use_graph else (lambda i, k: module_step(i, batches[k]))
    # ... and nvidia-smi (100 ms period, slow to start on a fresh box) must have sampled the clocks UNDER THIS LOAD:
    # keep stepping in blocks of 16 until rank 0's sampler has delivered a few samples (bounded at 4 s; the decision is
    # shared by all ranks so that every rank runs the same number of collective steps)
    t_pre, s = time.perf_counter(), 0
    while True:
        for _ in range(16):
            step_fn(1 + s % 8, s % n_total)
            s += 1
        torch.cuda.synchronize()
        more = torch.tensor([1.0 if (rank == 0 and clocks.proc is not None and clocks.n_samples() < 5
                                     and time.perf_counter() - t_pre < 4.0) else 0.0], device=dev)
        if world > 1:
            torch.distributed.all_reduce(more, op=torch.distributed.ReduceOp.MAX)
        if s >= PREWARM and float(more) == 0.0:
            break
    restore_state()
    for s in range(args.warmup):
        step_fn(s, s)
    launches0 = _lib.launch_count()
    graph0 = fast.graph_kernel_launches

    last_loss = []

    def timed_steps():
        for k in range(args.steps):
            last_loss[:] = [step_fn(args.warmup + k, args.warmup + k)]
        fast.flush()   # every one of the K updates is applied inside the timed region
    ms_total = timed(timed_steps)
    if args.dump_outputs and rank == 0:
        # the step's loss and the parameters it leaves (a fixed, seeded sample of the hash table, all MLP weights)
        P = model.pos_encoder.total_param_size
        pick = np.sort(np.random.default_rng(SEED).choice(P, min(P, DUMP_SAMPLE), replace=False))
        dump_outputs(args.dump_outputs, {
            "loss": last_loss[0].detach().float().reshape(1).cpu().numpy(),
            "samples": sample_counts[-1].reshape(1).cpu().numpy().astype(np.float64),
            "hash_table_sample": trainer.flat_param[torch.from_numpy(pick).to(dev)].cpu().numpy(),
            "mlp_params": trainer.flat_param[P:].cpu().numpy()})
    trainer.p2p_check()   # (several ranks) no peer barrier gave up waiting
    clock_info = clocks.stop() if rank == 0 else None
    launches = _lib.launch_count() - launches0            # eager launches of libngp_b200 kernels
    launches += fast.graph_kernel_launches - graph0       # + kernel nodes executed by CUDA-graph replays
    ms_step = ms_total / args.steps
    value = world * BATCH / (ms_step * 1e-3)
    spr = float(torch.stack([c.float() for c in sample_counts[-args.steps:]]).mean()) / BATCH

    # ---- end-to-end arms: host buffers, H2D inputs + D2H loss every step ----------------------------------
    def e2e_arm(step):
        def e2e_step(step_idx, hb):
            b = {k: v.to(dev, non_blocking=True) for k, v in hb.items()}
            loss = step(step_idx, b)
            return float(loss.detach().float().cpu())   # device->host read of the step's result
        base = args.warmup + args.steps
        for s in range(min(3, args.warmup)):
            e2e_step(base + s, host_batches[s])

        def run():
            for k in range(args.steps):
                e2e_step(base + 3 + k, host_batches[args.warmup + k])
            fast.flush()
        ms = timed(run)
        return world * BATCH / (ms / args.steps * 1e-3), ms / args.steps
    e2e_graph, ms_e2e_graph = e2e_arm(graph_step)        # public API: StaticTrainStep.step (train.py --graph_step)
    fast.flush()
    e2e_mod, ms_e2e_mod = e2e_arm(module_step)           # public API: render() + NGPTrainer.step (train.py default)
    h2d = sum(v.numel() * v.element_size() for v in host_batches[0].values())

    # ---- per-kernel rooflines, timed live with CUDA events on the buffers of a real step -----------------------
    roof = kernel_roofline(torch, cfg_name, cfg, fast, trainer, dev, ms_step)

    # ---- amortised density-grid update --------------------------------------------------------------------
    def upd():
        with torch.autocast("cuda", dtype=torch.float16):
            model.update_density_grid(DENSITY_THRESHOLD, warmup=True)
    upd()
    upd_ms = timed(upd)

    psnr = None
    if world == 1 and args.psnr_steps > 0:
        from taichi_nerfs_b200.psnr import train_vs_teacher
        del fast
        torch.cuda.empty_cache()
        r = train_vs_teacher(dev, steps=args.psnr_steps)
        if r is None:
            psnr = {"unavailable": "teacher fixture (oracle/_ref/lego_deployment) not staged"}
        else:
            psnr = {k: r[k] for k in ("psnr", "psnr_views", "steps", "batch", "train_views", "test_views", "image_wh",
                                      "steps_per_s", "rays_per_s", "path")}
            psnr["vs"] = ("teacher = the reference's shipped trained Lego deployment model rendered by this CUDA path; "
                          "PSNR on held-out teacher views (protocol of train.py:237-304); the reference's published "
                          "35.0 dB is on the real Lego test set, not available offline")

    if rank != 0:
        return
    overlap_txt = ("" if args.no_overlap else "; optimizer of step k runs on a parallel graph branch beside ray_aabb + "
                   "marching of step k+1 (flushed before every grid update and at the end of the timed region)")
    line = {
        "metric": "rays/sec (8192-ray batch, Lego shape)" if cfg_name in ("lego_half", "lego_8x")
                  else f"rays/sec ({BATCH}-ray batch, {cfg_name})",
        "value": value, "unit": "rays/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f16" if half else "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"] + "; random-init table+MLP, occupancy B (one warm-up grid update)",
                   "name": cfg_name, "rays_per_gpu": BATCH, "global_batch": world * BATCH, "samples_per_ray": spr,
                   "occupied_fraction": occupied, "parallelism": f"ray-sharded dp{world}, " + (
                       "no collective" if world == 1 else
                       "peer-memory optimizer step: NVLink P2P reduce-scatter + Adam on the owned 1/N + fp16 all-gather "
                       "in ONE kernel per rank (csrc/p2p.cu), no NCCL in the step" if trainer.p2p is not None else
                       "1 NCCL all-reduce/step"),
                   "l2": "no flush: per-step working set (~%d MB of per-sample tensors) exceeds the 126 MB L2; "
                         "new rays every step" % int(spr * BATCH * (2010 if half else 2872) / 1e6),
                   "density_grid_update": f"inside timed loop every {UPDATE_INTERVAL} steps (warm-up mode); "
                                          f"{upd_ms:.3f} ms each",
                   "step_path": ("StaticTrainStep: batch sampling (resident training set) + whole step = one CUDA-graph "
                                 "replay, sample count stays on the device" + overlap_txt) if use_graph else
                                "modules API: render() + torch.autograd + fused Adam"},
        "e2e": {"value": e2e_graph, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e_graph,
                "api": "StaticTrainStep.step(rays_o, rays_d, rgb) — train.py --graph_step; pinned host batch -> H2D -> "
                       "get_rays -> one graph replay -> loss D2H"},
        "e2e_modules": {"value": e2e_mod, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                        "ms_per_step": ms_e2e_mod,
                        "api": "reference-shaped plugin API: render(model, rays_o, rays_d) (HashEncoder / VolumeRenderer "
                               "autograd Functions, raymarching_train) + F.mse_loss + backward + NGPTrainer.optimizer_step "
                               "— train.py default path"},
        "gpu_launches": int(launches),
        "clocks": clock_info,
        "roofline": roof,
    }
    if psnr is not None:
        line["psnr"] = psnr
    if world == 1:
        line["cpu_baseline"] = cpu_baseline(cfg_name, cfg, budget_s=args.cpu_budget)
    print(json.dumps(line))


def kernel_roofline(torch, cfg_name, cfg, fast, trainer, dev, ms_step):
    """Times each kernel of the graph step alone (CUDA events on the launching stream, L2 flushed between repeats)
    on the buffers of one real step (same sample count S, same rays) and reports every kernel against the roofline
    that bounds it; top-level fields describe the dominant (slowest) kernel."""
    from taichi_nerfs_b200 import ops
    hbm_peak, tf_peak, peak_src = measured_peaks()
    col = 0 if cfg["half"] else 1
    fast.flush()
    fast.step_sampled()          # leave the buffers of a complete step behind
    fast.flush()
    torch.cuda.synchronize()
    S = int(fast.counter[0])
    flush = torch.empty(256 * 1024 * 1024, device=dev, dtype=torch.uint8)

    def t(fn, reps=5):
        out = []
        for _ in range(reps):
            flush.fill_(1)                      # evict L2 (126 MB) between repeats
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return statistics.median(out)

    def march():
        fast.counter.zero_()
        fast._enqueue_march()
    n_param = trainer.flat_param.numel()
    sp, sg, sm, sv = (trainer.flat_param.clone(), torch.randn_like(trainer.flat_grad) * 1e-3,
                      trainer.exp_avg.clone(), trainer.exp_avg_sq.clone())
    ssh = None if trainer._shadow_full is None else trainer._shadow_full.clone()
    times = {
        "hash_fwd": t(fast._k_hash_fwd),
        "mlp_fwd": t(fast._k_mlp_fwd),
        "ray_head": t(fast._k_head),
        "mlp_bwd": t(fast._k_mlp_bwd),
        "hash_bwd": t(fast._k_hash_bwd),
        "adam": t(lambda: ops.adam_step(sp, sg, sm, sv, 1e-3, 5, param_f16=ssh, zero_grad=True)),
    }
    t_cnt = t(lambda: fast.counter.zero_())
    times["march"] = max(t(march) - t_cnt, 1e-4)
    fast.counter[0] = S
    trainer.flat_grad.zero_()    # the timed backward kernels accumulated into it
    trainer.found_inf.zero_()
    del sp, sg, sm, sv, ssh, flush

    kernels = {}
    for k, ms in times.items():
        if k == "adam":
            b = ADAM_BYTES_PER_PARAM * n_param
        else:
            b = BYTES_PER_SAMPLE[k][col] * S
        e = {"ms": ms, "bound": "hbm", "achieved": b / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
             "step_share": ms / ms_step}
        e["frac"] = e["achieved"] / hbm_peak
        if k in FLOP_PER_SAMPLE:   # the one place a dense contraction exists: also against the tensor pipe
            tf = FLOP_PER_SAMPLE[k] * S / (ms * 1e-3) / 1e12
            e.update({"tensor_achieved": tf, "tensor_peak": tf_peak, "tensor_unit": "TFLOP/s", "tensor_frac": tf / tf_peak})
        kernels[k] = e
    top = max(times, key=times.get)
    traffic, traffic_src = ncu_traffic(cfg_name, top, S)
    out = {"kernel": top, "bound": "hbm", "achieved": kernels[top]["achieved"], "peak": hbm_peak, "unit": "GB/s",
           "frac": kernels[top]["frac"], "traffic": traffic, "traffic_unit": "bytes/launch",
           "traffic_source": traffic_src, "peak_source": peak_src, "samples": S,
           "algorithmic_bytes_per_sample": BYTES_PER_SAMPLE.get(top, (None, None))[col],
           "kernel_ms": times, "kernels": kernels,
           "sum_kernel_ms": sum(times.values()), "ms_per_step": ms_step,
           "note": "fp16 table (21.8 MiB) + fp32 grad (43.6 MiB) fit the 126 MB L2: the hash gathers / atomics never "
                   "reach HBM, their limiter is the SM's L1TEX/LSU wavefront rate (one 128-B line per cycle per SM for "
                   "divergent loads, ~1.3 cycles per lane for scattered RED) — DESIGN.md §4; algorithmic GB/s over the "
                   "HBM peak is what the contract asks for and can exceed the DRAM traffic by 10x"}
    return out


# --------------------------------------------------------------------------------------------------
def run_frame(args, cfg_name, cfg):
    """configs[4]: fps of one 800x800 test-time frame through the gui.py path (get_rays + render(test_time=True))."""
    import torch
    world, rank, local = dist_setup(args.gpus)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1 and rank != 0:      # single-GPU configuration: replicas would only repeat the same frame
        torch.distributed.barrier()
        return
    from datasets.ray_utils import get_ray_directions, get_rays
    from datasets.teacher import load_teacher, render_views
    from modules.networks import NGP
    from modules.rendering import render
    from taichi_nerfs_b200 import _lib, ops

    w, h = cfg["img_wh"]
    K = torch.tensor([[cfg["focal"], 0, w / 2], [0, cfg["focal"], h / 2], [0, 0, 1]], dtype=torch.float32)
    directions = get_ray_directions(h, w, K).to(dev)
    teacher = load_teacher(dev)
    info = {}
    if teacher is not None and args.frame_train_steps > 0:
        # trained weights + trained occupancy grid: the stock L=16 fp16 model fitted to the reference's shipped Lego model
        from taichi_nerfs_b200.psnr import train_vs_teacher
        r = train_vs_teacher(dev, steps=args.frame_train_steps, teacher=teacher)
        model = r["model"]
        info["weights"] = (f"stock L=16 T=2^19 F=2 fp16 model trained {r['steps']} steps on {r['train_views']} views of the "
                           f"reference's shipped Lego model ({r['psnr']:.2f} dB on held-out teacher views), occupancy grid "
                           "as trained")
        info["train_psnr"] = r["psnr"]
        from modules.utils import read_aot_array
        from datasets.teacher import teacher_dir
        pose = torch.from_numpy(read_aot_array(os.path.join(teacher_dir(), "pose.bin")).reshape(3, 4).copy()).to(dev)
        info["pose"] = "the reference demo's pose.bin"
    else:
        from datasets.synthetic import hemisphere_poses
        lay, table, ws = init_weights_numpy(SEED, cfg["max_res"], True)
        model = NGP(scale=cfg["scale"], max_res=cfg["max_res"], half_opt=True).to(dev)
        bits = np.load(os.path.join(ROOT, "tests", "golden", "lego_bitfield.npz"))["bitfield"]
        with torch.no_grad():
            model.pos_encoder.hash_table.copy_(torch.from_numpy(table))
            for p, wt in zip(mlp_params(model), ws):
                p.copy_(torch.from_numpy(wt))
            model.density_bitfield.copy_(torch.from_numpy(bits))
        pose = hemisphere_poses(1, cfg["radius"], SEED)[0].to(dev)
        info["weights"] = "random-init stock model, occupancy A = the reference's trained Lego bitfield (teacher not staged)"
    model.eval()
    pose_host = pose.cpu().pin_memory()

    def frame(p):
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            rays_o, rays_d = get_rays(directions, p)                       # gui.py:118-127
            return render(model, rays_o, rays_d, test_time=True, exp_step_factor=cfg["esf"])   # gui.py:129-137

    timed = make_timed(torch, 1, dev)
    if args.ncu_window > 0:
        for _ in range(5):
            frame(pose)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        for _ in range(args.ncu_window):
            res = frame(pose)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"ncu_window_steps": args.ncu_window, "config": cfg_name,
                          "samples_per_step": int(res["total_samples"])}))
        return
    clocks = ClockSampler(local)
    clocks.start()
    t_pre, k = time.perf_counter(), 0
    while k < max(args.warmup, 3) + 5 or (clocks.proc is not None and clocks.n_samples() < 5
                                          and time.perf_counter() - t_pre < 4.0):
        res = frame(pose)
        k += 1
    launches0 = _lib.launch_count()
    timed_frames = []
    ms = timed(lambda: timed_frames.extend(frame(pose) for _ in range(args.steps))) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: timed_frames[-1][k].float().cpu().numpy() for k in ("rgb", "depth", "opacity")})
    del timed_frames
    launches = _lib.launch_count() - launches0
    clock_info = clocks.stop()
    total_samples = int(res["total_samples"])
    fr = next(iter(model.__dict__.get("_frame_renderers", {}).values()), None)
    if fr is not None and fr.coarse is not None:   # how much of the box the empty-space leap has to respect
        words = fr.coarse.cpu().numpy().view(np.uint32)
        info["coarse_supercells_occupied"] = float(sum(bin(int(x)).count("1") for x in words)) / (32 * len(words))

    def e2e_frame():
        p = pose_host.to(dev, non_blocking=True)
        out = frame(p)
        return out["rgb"].float().cpu()          # the image goes back to the host (the GUI blits it)
    for _ in range(3):
        img = e2e_frame()
    ms_e2e = timed(lambda: [e2e_frame() for _ in range(args.steps)]) / args.steps

    psnr_teacher = None
    if teacher is not None:
        gold = render_views(teacher, directions, pose[None])[0]
        mse = float(((img.to(dev).clamp(0, 1) - gold) ** 2).mean())
        psnr_teacher = -10 * math.log10(max(mse, 1e-12))

    # per-kernel roofline of the frame path on the frame's own samples
    hbm_peak, tf_peak, peak_src = measured_peaks()
    roof = frame_roofline(torch, ops, model, directions, pose, cfg, dev, hbm_peak, tf_peak, peak_src, ms)
    line = {
        "metric": "fps (800x800 full-frame test-time ray march)", "value": 1e3 / ms, "unit": "frames/s", "n_gpus": 1,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": cfg["workload"], "name": cfg_name, "rays": w * h, "samples_evaluated": total_samples,
                   "samples_per_ray": total_samples / (w * h), "psnr_vs_teacher_frame": psnr_teacher,
                   "l2": "no flush: one frame touches ~%d MB of per-sample tensors (> 126 MB L2)"
                         % int(total_samples * 692 / 1e6), **info},
        "e2e": {"value": 1e3 / ms_e2e, "unit": "frames/s", "h2d_bytes_per_step": 48, "d2h_bytes_per_step": w * h * 12,
                "ms_per_step": ms_e2e,
                "api": "gui.py path: pose (host) -> get_rays -> render(model, rays_o, rays_d, test_time=True) -> "
                       "rgb image copied to the host"},
        "gpu_launches": int(launches), "clocks": clock_info, "roofline": roof,
        "cpu_baseline": cpu_baseline(cfg_name, cfg, budget_s=args.cpu_budget),
    }
    print(json.dumps(line))
    if world > 1:
        torch.distributed.barrier()


def frame_roofline(torch, ops, model, directions, pose, cfg, dev, hbm_peak, tf_peak, peak_src, ms_frame):
    from datasets.ray_utils import get_rays
    from taichi_nerfs_b200.fused_mlp import mlp_weights
    rays_o, rays_d = get_rays(directions, pose)
    rays_o, rays_d = rays_o.float().contiguous(), rays_d.float().contiguous()
    n = rays_o.shape[0]
    hits = ops.ray_aabb_intersect(rays_o, rays_d, model.scale)
    zeros = torch.zeros(n, device=dev)
    counter, rays_a = ops.raymarching_train_count(rays_o, rays_d, hits, model.density_bitfield, zeros, model.cascades,
                                                  model.scale, cfg["esf"], model.grid_size, 1024)
    S = int(counter[0])
    f32 = dict(device=dev, dtype=torch.float32)
    xyzs, dirs, deltas, ts = (torch.empty(S, 3, **f32), torch.empty(S, 3, **f32), torch.empty(S, **f32),
                              torch.empty(S, **f32))
    ops.raymarching_train_write(rays_o, rays_d, hits, model.density_bitfield, zeros, model.cascades, model.scale,
                                cfg["esf"], model.grid_size, counter, rays_a, xyzs, dirs, deltas, ts)
    enc = model.pos_encoder
    table = enc.table_f16()
    W = [w.detach() for w in mlp_weights(model)]
    aabb = model.xyz_min.flatten().tolist() + (model.xyz_max - model.xyz_min).flatten().tolist()
    emb = ops.hash_encode_fwd(xyzs, table, enc._clayout, enc.out_dim, aabb=aabb)
    sig, rgbs = ops.mlp_fwd(emb, dirs, W)
    cap = S + 4096
    cnt2 = torch.zeros(2, device=dev, dtype=torch.int32)
    ra2 = torch.empty(n, 3, device=dev, dtype=torch.int32)
    bx, bd, bdl, bts = (torch.empty(cap, 3, **f32), torch.empty(cap, 3, **f32), torch.empty(cap, **f32),
                        torch.empty(cap, **f32))
    flush = torch.empty(256 * 1024 * 1024, device=dev, dtype=torch.uint8)

    def t(fn, reps=5):
        out = []
        for _ in range(reps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            out.append(e0.elapsed_time(e1))
        return statistics.median(out)

    def march():
        cnt2.zero_()
        ops.raymarching_frame(rays_o, rays_d, hits, model.density_bitfield, model.cascades, model.scale, cfg["esf"],
                              model.grid_size, 1024, cnt2, ra2, bx, bd, bdl, bts)
    times = {
        "march": max(t(march) - t(lambda: cnt2.zero_()), 1e-4),
        "hash_fwd": t(lambda: ops.hash_encode_fwd(xyzs, table, enc._clayout, enc.out_dim, aabb=aabb)),
        "mlp_fwd": t(lambda: ops.mlp_fwd(emb, dirs, W)),
        "composite_fwd": t(lambda: ops.composite_train_fwd(sig, rgbs, deltas, ts, rays_a, 1e-4)),
    }
    kernels = {}
    for k, ms in times.items():
        b = BYTES_PER_SAMPLE[k][0] * S + (44 * n if k == "march" else 0)
        e = {"ms": ms, "bound": "hbm", "achieved": b / (ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
             "step_share": ms / ms_frame}
        e["frac"] = e["achieved"] / hbm_peak
        if k in FLOP_PER_SAMPLE:
            tf = FLOP_PER_SAMPLE[k] * S / (ms * 1e-3) / 1e12
            e.update({"tensor_achieved": tf, "tensor_peak": tf_peak, "tensor_unit": "TFLOP/s", "tensor_frac": tf / tf_peak})
        kernels[k] = e
    top = max(times, key=times.get)
    whole = (692 * S + 44 * n) / (ms_frame * 1e-3) / 1e9
    return {"kernel": top, "bound": "hbm", "achieved": kernels[top]["achieved"], "peak": hbm_peak, "unit": "GB/s",
            "frac": kernels[top]["frac"], "traffic": None, "peak_source": peak_src, "samples": S, "rays": n,
            "kernel_ms": times, "kernels": kernels,
            "whole_frame": {"algorithmic_bytes": 692 * S + 44 * n, "achieved": whole, "frac": whole / hbm_peak,
                            "note": "692 B/sample + 44 B/ray (SURVEY.md §8d, unfused boundaries) over the frame time"}}


# --------------------------------------------------------------------------------------------------
def oracle_workload(cfg, n_rays, seed):
    """Builds the CPU-arm model (same random init, occupancy B computed by the oracle) and ray batches."""
    from oracle import oracle as O
    from oracle import train_step as TS
    O.build()
    half, scale = cfg["half"], cfg["scale"]
    lay, table, ws = init_weights_numpy(SEED, cfg["max_res"], half)
    rng = np.random.default_rng(seed)
    cascades = max(1 + int(math.ceil(math.log2(2 * scale))), 1)
    g = 128
    if cfg["kind"] == "frame":   # occupancy A: the reference's trained Lego bitfield
        bitfield = np.load(os.path.join(ROOT, "tests", "golden", "lego_bitfield.npz"))["bitfield"]
    else:
        # occupancy B: density at a jittered point of every cell, threshold = min(mean, 5.91) (networks.py:255-290)
        coords = np.stack(np.meshgrid(np.arange(g), np.arange(g), np.arange(g), indexing="ij"), -1).reshape(-1, 3).astype(np.int32)
        mort = O.morton3d(coords).astype(np.int64)
        grid = np.zeros((cascades, g ** 3), np.float32)
        tab = table.astype(np.float16).reshape(-1) if half else table.reshape(-1)
        for c in range(cascades):
            s = min(2.0 ** (c - 1), scale)
            hg = s / g
            xyz = (coords / (g - 1) * 2 - 1) * (s - hg) + (rng.random((g ** 3, 3)) * 2 - 1) * hg
            xn = ((xyz + scale) / (2 * scale)).astype(np.float32)
            emb = O.hash_encode_fwd(xn, tab, lay)
            dens, _ = O.mlp_fwd(emb, np.tile(np.array([[0, 0, 1]], np.float32), (g ** 3, 1)), ws)
            grid[c, mort] = dens
        thr = min(float(grid[grid > 0].mean()), DENSITY_THRESHOLD)
        bitfield = O.packbits(grid.reshape(-1), thr)
    model = TS.OracleModel(lay, table, ws, bitfield, scale=scale, cascades=cascades, half=half)
    w, h = cfg["img_wh"]

    def batch(i):
        o, d = TS.make_rays(n_rays, seed=seed * 1000 + i, radius=cfg["radius"], img=w, focal=cfg["focal"], img_h=h)
        r = np.random.default_rng(seed * 1000 + i)
        return o, d, r.random((n_rays, 3), dtype=np.float32), r.random(n_rays, dtype=np.float32)
    return TS, model, batch


def host_threads():
    """Force the OpenMP team to every core this process may run on (torchrun exports OMP_NUM_THREADS=1) and return
    (cores available, threads a parallel region really used)."""
    from oracle import oracle as O
    cores = len(os.sched_getaffinity(0))
    os.environ["OMP_NUM_THREADS"] = str(cores)
    O.build()
    return cores, O.set_threads(cores)


def oracle_frame(cfg, stride):
    """CPU arm of frame800: forward render (AABB -> march -> encode -> MLP -> composite) of every `stride`-th pixel in
    both directions of one 800x800 frame; returns (seconds, rays, samples)."""
    TS, model, _ = oracle_workload(cfg, 0, SEED)
    w, h = cfg["img_wh"]
    c = np.array([0.70147288, -1.0291882, 0.63064414])           # the reference demo's camera position (pose.bin)
    fwd = -c / np.linalg.norm(c)
    right = np.cross(fwd, [0, 0, 1.0])
    right /= np.linalg.norm(right)
    down = np.cross(fwd, right)
    u, v = np.meshgrid(np.arange(0, w, stride), np.arange(0, h, stride))
    dc = np.stack([(u.ravel() - w / 2 + .5) / cfg["focal"], (v.ravel() - h / 2 + .5) / cfg["focal"],
                   np.ones(u.size)], -1)
    d = (dc[:, 0:1] * right + dc[:, 1:2] * down + dc[:, 2:3] * fwd).astype(np.float32)
    o = np.tile(c.astype(np.float32), (d.shape[0], 1))
    noise = np.zeros(d.shape[0], np.float32)
    TS.forward(model, o[:1024], d[:1024], noise[:1024])          # warm-up
    t0 = time.perf_counter()
    _, cache = TS.forward(model, o, d, noise)
    return time.perf_counter() - t0, d.shape[0], cache["S"]


def cpu_baseline(cfg_name, cfg, budget_s=20.0):
    cores, used = host_threads()
    if cfg["kind"] == "frame":
        stride = 4
        dt, rays, S = oracle_frame(cfg, stride)
        w, h = cfg["img_wh"]
        return {"value": 1.0 / (dt * (w * h) / rays), "unit": "frames/s", "cores": used, "cores_available": cores,
                "kind": "port",
                "sample": f"every {stride}th pixel in x and y of one 800x800 frame ({rays} rays, {S} samples, {dt:.2f} s) "
                          f"through oracle/ngp_oracle.c forward (OpenMP, {used} threads), random-init stock model, the "
                          "reference's trained Lego occupancy; fps scaled by the ray count"}
    n_rays = cfg["n_rays"]
    TS, model, batch = oracle_workload(cfg, n_rays, SEED)
    o, d, gt, nz = batch(0)
    TS.train_step(model, o, d, gt, nz, exp_step_factor=cfg["esf"])      # warm-up
    t0, steps, samples = time.perf_counter(), 0, 0
    while steps < 1 or (time.perf_counter() - t0 < budget_s and steps < 64):
        o, d, gt, nz = batch(steps + 1)
        _, cache = TS.train_step(model, o, d, gt, nz, exp_step_factor=cfg["esf"])
        samples += cache["S"]
        steps += 1
    dt = time.perf_counter() - t0
    return {"value": steps * n_rays / dt, "unit": "rays/s", "cores": used, "cores_available": cores, "kind": "port",
            "sample": f"{steps} full train steps of {n_rays} rays (the same {cfg_name} workload, occupancy B, "
                      f"{samples / max(steps * n_rays, 1):.0f} samples/ray) through oracle/ngp_oracle.c "
                      f"(OpenMP, {used} threads)"}


def run_reference(args, cfg_name, cfg):
    """Reference arm: the reference's algorithm on the host cores (the Taichi reference itself cannot be installed
    offline — see DESIGN.md — so this is the strict-fp32 C/OpenMP restatement, kind=port).  SAME configuration as the
    CUDA arm: same rays per step, same model, same occupancy; only the number of timed steps is capped so the run
    ends within a few minutes (a 8192-ray CPU step takes seconds)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores, used = host_threads()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if cfg["kind"] == "frame":
        stride = 4
        dts = []
        for _ in range(max(1, min(args.steps, 3))):
            dt, rays, S = oracle_frame(cfg, stride)
            dts.append(dt)
        w, h = cfg["img_wh"]
        value = 1.0 / (statistics.median(dts) * (w * h) / rays)
        sample = (f"{len(dts)} renders of every {stride}th pixel in x and y of the 800x800 frame ({rays} rays, {S} samples "
                  f"each), fps scaled by the ray count; {used} OpenMP threads of {cores} cores")
        unit, metric, ms = "frames/s", "fps (800x800 full-frame test-time ray march)", 1e3 / value
        steps_done = len(dts)
    else:
        n_rays = cfg["n_rays"]
        TS, model, batch = oracle_workload(cfg, n_rays, SEED)
        t0 = time.perf_counter()
        TS.train_step(model, *batch(0), exp_step_factor=cfg["esf"])     # warm-up step (also the time probe)
        probe = time.perf_counter() - t0
        budget = args.ref_budget
        warm = max(0, min(args.warmup - 1, int(0.25 * budget / max(probe, 1e-3))))
        steps_done = max(1, min(args.steps, int(0.75 * budget / max(probe, 1e-3))))
        for s in range(warm):
            TS.train_step(model, *batch(1 + s), exp_step_factor=cfg["esf"])
        t0 = time.perf_counter()
        samples = 0
        for k in range(steps_done):
            _, cache = TS.train_step(model, *batch(100 + k), exp_step_factor=cfg["esf"])
            samples += cache["S"]
        dt = time.perf_counter() - t0
        value = steps_done * n_rays / dt
        sample = (f"{steps_done} timed steps (of the {args.steps} requested: a CPU step takes {dt / steps_done:.1f} s) x "
                  f"{n_rays} rays per step = the full batch of this configuration, "
                  f"{samples / (steps_done * n_rays):.0f} samples/ray; {used} OpenMP threads of {cores} cores")
        unit, ms = "rays/s", dt / steps_done * 1e3
        metric = ("rays/sec (8192-ray batch, Lego shape)" if cfg_name in ("lego_half", "lego_8x")
                  else f"rays/sec ({n_rays}-ray batch, {cfg_name})")
    print(json.dumps({
        "impl": "reference", "metric": metric, "value": value, "unit": unit,
        "n_gpus": world, "steps": steps_done, "steps_requested": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16" if cfg["half"] else "f32", "data": "synthetic",
        "config": {"workload": cfg["workload"] + " — restated on the CPU (oracle/ngp_oracle.c, kind=port): same "
                               "model, same occupancy recipe, same rays per step; rank 0 only", "name": cfg_name,
                   "rays_per_gpu": cfg.get("n_rays"), "sample": sample},
        "cpu_baseline": {"value": value, "unit": unit, "cores": used, "cores_available": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="lego_half", choices=sorted(CONFIGS),
                    help="which BASELINE.json configuration to run (default: configs[1], the one the metric is quoted on)")
    ap.add_argument("--cpu-budget", type=float, default=12.0, help="seconds of CPU work for cpu_baseline")
    ap.add_argument("--ref-budget", type=float, default=150.0,
                    help="reference arm: wall-clock budget (s) for warm-up + timed steps at the FULL batch size")
    ap.add_argument("--path", default="graph", choices=["graph", "modules"],
                    help="value arm — graph: StaticTrainStep (one CUDA graph per step, sync-free); "
                         "modules: render()+autograd through the reference-shaped module API")
    ap.add_argument("--no-overlap", action="store_true",
                    help="graph path: run the optimizer at the end of its own step instead of next to the next "
                         "step's marching")
    ap.add_argument("--psnr-steps", type=int, default=2000,
                    help="train configs, 1 GPU: also train the stock model this many steps on views of the reference's "
                         "shipped Lego model and report PSNR on held-out views (0 = skip)")
    ap.add_argument("--frame-train-steps", type=int, default=2000,
                    help="frame800: steps of teacher training that produce the rendered model (0 = random weights)")
    ap.add_argument("--ncu-window", type=int, default=0,
                    help="profiling aid: wrap this many extra steps in cudaProfilerStart/Stop "
                         "(use with `ncu --profile-from-start off`); numbers printed under ncu are not bench values")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed to DIR/<name>.npy "
                         "(train: loss, sample count, a seeded sample of the hash table, MLP weights; frame: rgb, "
                         "depth, opacity), at most 64 MB")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.ncu_window > 0):
        ap.error("--dump-outputs applies to the timed CUDA path only")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    cfg = CONFIGS[args.config]
    if args.impl == "reference":
        run_reference(args, args.config, cfg)
    elif cfg["kind"] == "frame":
        run_frame(args, args.config, cfg)
    else:
        run_train(args, args.config, cfg)


if __name__ == "__main__":
    main()
