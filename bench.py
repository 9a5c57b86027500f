#!/usr/bin/env python
"""Benchmark of the DeepBedMap ESRGAN hot path on B200 (contract: see DESIGN.md "Measurement").

Two metrics (BASELINE.json names both), selected with --metric:

  --metric inference (default)  BASELINE configs[2]: whole-Antarctic tiled inference on a synthetic continent-sized
      grid (X 1x1x4502x5502, W1 1x1x45020x55020, W2 1x2x9004x11004, W3 1x1x4502x5502 -> 18000 x 22000 px at 250 m =
      396 Mpx), reference tile geometry, 12-RRDB generator, random-init weights. One step = one whole-continent pass;
      N GPUs split the 396 tiles into N contiguous runs (strong scaling).
        value    Mpx/s with the grids resident in HBM, predictions left on the device
        e2e      Mpx/s through predict_continent() with pinned HOST grids in and a HOST DEM out
        roofline dominant kernel (umma_trunk_kernel): algorithmic FLOPs / CUDA-event time vs measured bf16 peak
        parity   one full-size interior tile of this very continent: bf16 path vs the fp32 CPU oracle run for the
                 cpu_baseline leg (relative L2, max-abs in output units and in metres) and vs the fp32 CUDA path
        train    the second metric as a sub-object (same fields as --metric train)
        configs  BASELINE configs[0] (batch-1 latency) and configs[1] (batch-128 forward), each with its CPU leg
  --metric train  BASELINE configs[3]: ESRGAN train steps/s, D-step + G-step on a batch of 128 per GPU
      (srgan_train.py:1286-1308), data parallel (weak scaling), with roofline / e2e (host minibatch in, metrics out)
      / cpu_baseline (3 oracle steps at batch 128).

  --impl reference  the reference arm: the reference graph restated on the CPU (oracle/, torch fp32, all host
      cores; Chainer 7 is not installable in this image -- probed at run time, kind "port") on a bounded sample per
      step, same metric / config as the B200 arm.

  --dump-outputs DIR  after the timed steps, what the last one computed, as DIR/<name>.npy: inference writes
      continent_sample (2^23 seeded pixels of the 18000 x 22000 DEM inside its NaN frame); train writes train_metrics
      (d_loss, d_accuracy, g_loss, g_psnr, g_ssim) and 2^22 seeded parameters of each model after that step. The inputs
      are seeded, so two builds run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

MPX = 396.0  # 18000 x 22000 output pixels
FULL = dict(final_shape=(18000, 22000), ary_shape=(1000, 1000), grid=(4502, 5502))
BED_STD_M = 800.0           # spread of the synthetic BEDMAP2-like input; calibrates output units to metres
GFLOP_PER_SAMPLE_STEP = 6.4995   # SURVEY 8d: algorithmic work of a train step per sample, G forward counted once
TRUNK_MAC_PER_PX = 9 * 128 * 64 + 36 * 239616 + 9 * 64 * 64   # pre-res + 36 RDB + post-res (SURVEY App. A)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1383.0), d.get("hbm_gbs", 6547.2), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def infer_config(args, world):
    return {"workload": "configs[2] whole-Antarctic tiled inference, 396 tiles -> 18000x22000 px @250 m"
            if args.scale == 1.0 else f"DEBUG scaled continent x{args.scale}",
            "num_residual_blocks": 12, "batch_tiles": args.batch_tiles, "tile_split": f"contiguous/{world}",
            "l2": "inputs (10.9 GB) and per-layer activations exceed the 126 MB L2; no flush needed"}


def train_config(world, batch=128):
    return {"workload": "configs[3] ESRGAN training step: D-step + G-step (srgan_train.py:1286-1308), batch 128 per GPU, "
                        "11x11 / 110x110 / 22x22 / 11x11 tiles -> 36x36",
            "num_residual_blocks": 12, "batch_per_gpu": batch, "global_batch": batch * world,
            "parallelism": f"dp{world}",
            "l2": "a step streams 77 MB of fp32 gradients + 154 MB of Adam state and ~1 GB of saved activations: "
                  "larger than the 126 MB L2, no flush needed"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.rows = []
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [s.strip() for s in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]),
                "power_w_max": max(float(r[2]) for r in self.rows), "samples": len(self.rows), "reasons": reasons}


def synth_grids_device(grid, seed=42):
    """Synthetic continent in the physical regime of SURVEY 8(d) config 3; identical on every rank."""
    H, W = grid
    g = torch.Generator(device="cuda").manual_seed(seed)
    X = (torch.randn(1, 1, H, W, generator=g, device="cuda") * 800.0 - 500.0).clamp_(-5000.0, 4500.0)
    W1 = torch.rand(1, 1, 10 * H, 10 * W, generator=g, device="cuda") * 4000.0
    W2 = torch.randn(1, 2, 2 * H, 2 * W, generator=g, device="cuda") * 200.0
    W3 = torch.rand(1, 1, H, W, generator=g, device="cuda") * 1000.0
    return X, W1, W2, W3


def dist_setup():
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import datetime
        import torch.distributed as dist
        torch.cuda.set_device(local)
        # short watchdog: a mismatched collective must fail in minutes, not burn the GPU box for ten
        dist.init_process_group("nccl", device_id=torch.device("cuda", local), timeout=datetime.timedelta(seconds=180))
    else:
        torch.cuda.set_device(0)
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(ms, world):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])
    return ms


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / (np.linalg.norm(b) + 1e-300))


DUMP_LIMIT_BYTES = 64 << 20


def seeded_sample(t, n, seed=0):
    """``t`` flattened to the host if it has at most ``n`` elements, else ``n`` of its elements at fixed, seeded
    positions in ascending order: the same positions on every run, so two builds compare element for element."""
    flat = t.reshape(-1)
    if flat.numel() <= n:
        return flat.cpu().numpy()
    idx = np.sort(np.random.RandomState(seed).randint(0, flat.numel(), size=n))
    return flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()


def dump_outputs(out_dir, arrays):
    """--dump-outputs: writes each array as <out_dir>/<name>.npy."""
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT_BYTES
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------------------
# CPU legs: the oracle port timed on this box's host cores. bench.py's cpu_baseline / --impl reference legs are the
# only place outside tests/ and smoke() where oracle/ is executed -- as the baseline, never as the product.
# ------------------------------------------------------------------------------------------------------------
def reference_kind():
    """Chainer 7 (the reference's engine) is not installable in this image; probe anyway so that a box that has it
    (site-packages or baseline/_ref) is reported. The timed code is the oracle port either way."""
    sys.path.insert(0, os.path.join(ROOT, "baseline", "_ref"))
    try:
        import chainer  # noqa: F401
        found = f"chainer {chainer.__version__} importable (not wired: the notebooks' other imports are absent)"
    except Exception as ex:
        found = f"chainer not importable ({type(ex).__name__})"
    finally:
        sys.path.pop(0)
    return "port", found


def cpu_threads():
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    return cores


def continent_flop_weight():
    """Computed output pixels (incl. halos) of the 396-tile plan: the FLOP-weighted tile mix."""
    from oracle import deepbedmap_oracle as O
    return sum(16 * (y1 - y0 - 2) * (x1 - x0 - 2) for (y0, y1, x0, x1, _, _) in O.tile_plan())


def cpu_tile_forward(ins, nb=12, reps=1, warm=0):
    """fp32 oracle forward of one lowres crop (batch 1) on all host cores -> (seconds per forward, output)."""
    from oracle import deepbedmap_oracle as O
    params = O.to_torch(O.init_generator_params(nb, seed=0), torch.float32)
    tin = [torch.as_tensor(np.asarray(a, np.float32)) for a in ins]
    y = None
    with torch.no_grad():
        for _ in range(warm):
            O.generator_forward(params, *tin, num_residual_blocks=nb, fast_deform=True)
        t0 = time.perf_counter()
        for _ in range(reps):
            y = O.generator_forward(params, *tin, num_residual_blocks=nb, fast_deform=True)
        dt = (time.perf_counter() - t0) / reps
    return dt, y.numpy()


def cpu_inference_rate(crop, reps=1, warm=0):
    """Times the oracle on one crop x crop lowres window of physical-regime input and extrapolates to the continent
    by computed-pixel count. -> (Mpx/s, seconds per forward, sample text)."""
    from oracle import deepbedmap_oracle as O
    ins = O.synthetic_inputs(1, crop, crop, regime="physical")
    ins = (ins[0],) + tuple(np.clip(a, 0, None) for a in ins[1:])
    dt, _ = cpu_tile_forward(ins, reps=reps, warm=warm)
    px = (4 * (crop - 2)) ** 2
    total = continent_flop_weight()
    sample = (f"{reps} fp32 forward(s) of one {crop}x{crop} lowres crop (-> {4 * (crop - 2)}^2 px), {dt:.2f} s each, "
              f"extrapolated x{total / px:.0f} by computed-pixel count to the 396-tile continent")
    return MPX / (dt * total / px), dt, sample


def cpu_train_step_time(batch=128, steps=3, warm=0, nb=12):
    """Oracle D-step + G-step (reference-literal dataflow: two generator forwards, autograd backward, Chainer Adam)
    in fp32 on all host cores -> seconds per step."""
    from oracle import deepbedmap_oracle as O
    rng = np.random.RandomState(42)
    arrays = {"X": rng.rand(batch, 1, 11, 11), "W1": rng.rand(batch, 1, 110, 110), "W2": rng.rand(batch, 2, 22, 22),
              "W3": rng.rand(batch, 1, 11, 11), "Y": rng.rand(batch, 1, 36, 36)}
    ta = {k: torch.as_tensor(v, dtype=torch.float32) for k, v in arrays.items()}
    gp = O.to_torch(O.init_generator_params(nb, seed=0), torch.float32)
    dp = O.to_torch(O.init_discriminator_params(seed=1), torch.float32)
    g_opt, d_opt = O.ChainerAdam(1.6e-4), O.ChainerAdam(1.6e-4)
    ts = []
    for i in range(warm + steps):
        t0 = time.perf_counter()
        O.train_eval_discriminator(ta, gp, dp, d_opt, num_residual_blocks=nb)
        O.train_eval_generator(ta, gp, dp, g_opt, num_residual_blocks=nb)
        if i >= warm:
            ts.append(time.perf_counter() - t0)
    return float(np.mean(ts))


def cpu_forward_time(batch, reps, warm=1, nb=12):
    """fp32 oracle forward of ``batch`` 11x11 tiles (configs[0] / configs[1]) -> median seconds."""
    from oracle import deepbedmap_oracle as O
    params = O.to_torch(O.init_generator_params(nb, seed=0), torch.float32)
    tin = [torch.as_tensor(a) for a in O.synthetic_inputs(batch)]
    ts = []
    with torch.no_grad():
        for i in range(warm + reps):
            t0 = time.perf_counter()
            O.generator_forward(params, *tin, num_residual_blocks=nb, fast_deform=True)
            if i >= warm:
                ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def run_reference(args):
    """--impl reference: rank 0 alone, CPU only, same metric / unit / config as the B200 arm. Each step is a bounded
    sample sized so that the driver's --steps 20 --warmup 5 ends within a few minutes; ms_per_step is the measured
    time of that sample, ``value`` its extrapolation to the whole workload (stated in cpu_baseline.sample)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    cores = cpu_threads()
    kind, probe = reference_kind()
    vals, secs, sample = [], [], ""
    if args.metric == "train":
        b = args.cpu_train_batch
        for i in range(args.warmup + args.steps):
            dt = cpu_train_step_time(batch=b, steps=1)
            if i >= args.warmup:
                secs.append(dt)
                vals.append(1.0 / (dt * 128.0 / b) * world)
        v = float(np.mean(vals))
        sample = (f"per step: one D-step + G-step of the fp32 oracle at batch {b} ({np.mean(secs):.2f} s), scaled x{128 // b} "
                  f"to the batch of 128; one CPU host stands for every rank (x{world})")
        metric, unit, scaling, cfg = "train steps/s (D-step + G-step, batch 128 per GPU)", "steps/s", "weak", train_config(world)
    else:
        for i in range(args.warmup + args.steps):
            v, dt, sample = cpu_inference_rate(args.cpu_crop)
            if i >= args.warmup:
                vals.append(v)
                secs.append(dt)
        v = float(np.mean(vals))
        metric, unit, scaling, cfg = "continent inference output Mpx/s", "Mpx/s", "strong", infer_config(args, world)
    line = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": v, "unit": unit, "cores": cores, "kind": kind, "sample": sample,
                             "reference_engine_probe": probe},
            "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# inference legs
# ------------------------------------------------------------------------------------------------------------
def instrumented_roofline(model, grids, kw, peak_tf):
    """Re-runs a strip of tiles with CUDA events (on the launching stream) around every tcgen05 conv launch: the
    persistent trunk kernel (dominant) and the per-layer conv kernel."""
    from deepbedmap_b200 import ops, tiler
    recs = {"umma_trunk_kernel": [], "umma_conv3x3_kernel": []}
    orig = ops.call

    def wrapped(name, *a):
        if name not in ("dbm_trunk_umma", "dbm_conv3x3_umma"):
            return orig(name, *a)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig(name, *a)
        e1.record()
        if name == "dbm_trunk_umma":
            n, h, w = a[2], a[3], a[4]
            recs["umma_trunk_kernel"].append((e0, e1, model._ws[(n, h, w)]["flops"]))
        else:
            cin, coutp, n, h, w = a[2], a[5], a[6], a[7], a[8]
            cout = 18 if (coutp == 32 and a[12] is None) else coutp   # offset convs: 18 real channels
            recs["umma_conv3x3_kernel"].append((e0, e1, 2.0 * 9 * cin * cout * n * h * w))

    ops.call = wrapped
    c_api = model.c_model_api
    model.c_model_api = False   # the strip needs the per-kernel calls: same kernels and tables, composed from Python
    try:
        sub = dict(kw)
        sub["final_shape"] = (min(kw["final_shape"][0], 3000), min(kw["final_shape"][1], 6000))
        tiler.predict_continent(model, None, None, None, None, grids=grids, to_host=False, **sub)
        torch.cuda.synchronize()
    finally:
        ops.call = orig
        model.c_model_api = c_api
    out = {}
    for k, v in recs.items():
        if not v:
            continue
        ms = sum(a.elapsed_time(b) for a, b, _ in v)
        fl = sum(f for _, _, f in v)
        out[k] = {"tflops": fl / (ms * 1e-3) / 1e12, "launches_timed": len(v), "avg_launch_us": ms * 1e3 / len(v),
                  "flops_per_launch_avg": fl / len(v), "ms_total": ms}
    dom = max(out, key=lambda k: out[k]["ms_total"])
    ach = out[dom]["tflops"]
    traffic, traffic_src = trunk_traffic(out[dom]["flops_per_launch_avg"]) if dom == "umma_trunk_kernel" else (None, None)
    return {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
            "traffic": traffic, "traffic_source": traffic_src,
            "kernel": dom, "launches_timed": out[dom]["launches_timed"],
            "avg_launch_us": out[dom]["avg_launch_us"], "flops_per_launch_avg": out[dom]["flops_per_launch_avg"],
            "algorithmic": "2*9*Cin*Cout FLOP per pixel per pass summed over the pass table (DESIGN.md 4)",
            "all_tcgen05_conv_kernels": {k: {kk: vv for kk, vv in v.items() if kk != "ms_total"} | {
                "frac": v["tflops"] / peak_tf} for k, v in out.items()}}


def trunk_traffic(flops_per_launch):
    """DRAM bytes of the trunk kernel per launch: dram__bytes_read.sum + dram__bytes_write.sum of the round's
    `ncu --set full` capture (profiles/trunk_traffic.json: bytes and FLOPs of the captured launch), scaled to this
    run's average launch by its algorithmic FLOPs. ncu counters cannot be read inside an unprofiled run."""
    p = os.path.join(ROOT, "profiles", "trunk_traffic.json")
    if not os.path.exists(p):
        return None, "no capture on record"
    d = json.load(open(p))
    return d["dram_bytes"] / d["flops"] * flops_per_launch, d["source"]


def tile_parity(model, grids, cpu: bool):
    """One full-size interior tile of the benchmark continent (tile row 9, column 11 of the 18 x 22 plan): the bf16
    path against the fp32 CUDA path and -- when the CPU leg runs -- against the fp32 CPU oracle of the same crop.
    Also returns the CPU seconds of that forward (the cpu_baseline sample)."""
    from deepbedmap_b200 import GeneratorModel, tiler
    plan = tiler.tile_plan(FULL["final_shape"])
    y0, y1, x0, x1 = plan[9 * 22 + 11][:4]
    r0 = grids.row0
    crop = (grids.X[:, :, y0 - r0:y1 - r0, x0:x1],
            grids.W1[:, :, 10 * (y0 - r0):10 * (y1 - r0), 10 * x0:10 * x1].clamp(min=0),
            grids.W2[:, :, 2 * (y0 - r0):2 * (y1 - r0), 2 * x0:2 * x1].clamp(min=0),
            grids.W3[:, :, y0 - r0:y1 - r0, x0:x1].clamp(min=0))
    crop = tuple(c.contiguous() for c in crop)
    y16 = model.forward(*crop).array[0, 0].cpu().numpy()
    m32 = GeneratorModel(num_residual_blocks=12, residual_scaling=0.1, precision="fp32", seed=0)
    y32 = m32.forward(*crop).array[0, 0].cpu().numpy()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    m32.forward(*crop)
    e1.record()
    torch.cuda.synchronize()
    ms32 = e0.elapsed_time(e1)
    e0.record()
    model.forward(*crop)
    e1.record()
    torch.cuda.synchronize()
    ms16 = e0.elapsed_time(e1)
    del m32
    torch.cuda.empty_cache()
    # split-bf16 tensor-core path (precision="bf16x3"): the fp32-grade option at tensor-core speed
    m3 = GeneratorModel(num_residual_blocks=12, residual_scaling=0.1, precision="bf16x3", seed=0)
    y3 = m3.forward(*crop).array[0, 0].cpu().numpy()
    e0.record()
    m3.forward(*crop)
    e1.record()
    torch.cuda.synchronize()
    ms3 = e0.elapsed_time(e1)
    del m3
    torch.cuda.empty_cache()
    std = float(y32.std())
    to_m = BED_STD_M / std
    out = {"tile": f"interior tile (row 9, col 11): lowres crop [{y0}:{y1}, {x0}:{x1}] -> {y16.shape[0]}x{y16.shape[1]} px, "
                   "12 RRDB, bench weights",
           "metres": f"output units x ({BED_STD_M:.0f} m / std(output)): the random-init network's output unit is arbitrary, "
                     "so errors are quoted for an output calibrated to the spread of the bed-elevation input",
           "output_std": std,
           "precision_modes": {"bf16": {"ms_per_tile": ms16, "what": "tensor-core path (the benchmarked one)"},
                               "bf16x3": {"ms_per_tile": ms3, "what": "split-bf16 tensor-core path, precision='bf16x3': hi + lo "
                                          "bf16 terms, three MMAs per K chunk in the trunk and the upsample convs, stem and "
                                          "deformable layers fp32; error below as bf16x3_vs_fp32_cpu_oracle"},
                               "fp32": {"ms_per_tile": ms32, "what": "exact CUDA-core path, precision='fp32', error below "
                                        "as fp32_cuda_vs_fp32_cpu_oracle"}},
           "bf16x3_vs_fp32_cuda": {"rel_l2": rel_l2(y3, y32), "max_abs": float(np.abs(y3 - y32).max()),
                                   "max_abs_m": float(np.abs(y3 - y32).max()) * to_m},
           "bf16_vs_fp32_cuda": {"rel_l2": rel_l2(y16, y32), "max_abs": float(np.abs(y16 - y32).max()),
                                 "max_abs_m": float(np.abs(y16 - y32).max()) * to_m}}
    secs = None
    if cpu:
        secs, yc = cpu_tile_forward([c.cpu().numpy() for c in crop])
        yc = yc[0, 0]
        for name, y in (("bf16_vs_fp32_cpu_oracle", y16), ("bf16x3_vs_fp32_cpu_oracle", y3),
                        ("fp32_cuda_vs_fp32_cpu_oracle", y32)):
            out[name] = {"rel_l2": rel_l2(y, yc), "max_abs": float(np.abs(y - yc).max()),
                         "max_abs_m": float(np.abs(y - yc).max()) * to_m}
        out["rel_l2"] = out["bf16_vs_fp32_cpu_oracle"]["rel_l2"]
        out["max_abs_m"] = out["bf16_vs_fp32_cpu_oracle"]["max_abs_m"]
    else:
        out["rel_l2"] = out["bf16_vs_fp32_cuda"]["rel_l2"]
        out["max_abs_m"] = out["bf16_vs_fp32_cuda"]["max_abs_m"]
    return out, secs, (y1 - y0, x1 - x0)


def small_tile_configs(peak_tf, cpu: bool):
    """BASELINE configs[0] (batch 1, one 11x11 tile: latency) and configs[1] (batch 128 forward) with their CPU legs
    (SURVEY 8d: median of 20 / 3 forwards)."""
    from deepbedmap_b200 import GeneratorModel
    from oracle import deepbedmap_oracle as O   # input generator only (host side)
    m = GeneratorModel(num_residual_blocks=12, residual_scaling=0.1, precision="bf16", seed=0)
    out = {}
    for key, batch, reps in (("configs[0] batch 1 latency", 1, 20), ("configs[1] batch 128 forward", 128, 20)):
        host = [torch.from_numpy(a).pin_memory() for a in O.synthetic_inputs(batch)]
        dev = [t.cuda() for t in host]
        for _ in range(5):
            m.forward(*dev)
        torch.cuda.synchronize()
        dts = []
        for _ in range(reps):   # device-resident inputs, CUDA events
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            m.forward(*dev)
            e1.record()
            torch.cuda.synchronize()
            dts.append(e0.elapsed_time(e1))
        e2e = []
        for _ in range(reps):   # host arrays in, host prediction out (wall clock)
            t0 = time.perf_counter()
            m.forward(*host).array.cpu()
            e2e.append((time.perf_counter() - t0) * 1e3)
        ms, ms_e2e = float(np.median(dts)), float(np.median(e2e))
        gflop = 1.690720 * batch
        rec = {"batch": batch, "ms": ms, "ms_e2e_host_in_host_out": ms_e2e, "tiles_per_s": batch / ms * 1e3,
               "gflop_forward": gflop, "tflops": gflop / ms, "frac_of_bf16_peak": gflop / ms / peak_tf,
               "timing": f"median of {reps}"}
        if cpu:
            cs = cpu_forward_time(batch, reps=20 if batch == 1 else 3)
            rec["cpu_baseline"] = {"ms": cs * 1e3, "cores": os.cpu_count(), "kind": "port",
                                   "sample": f"median of {20 if batch == 1 else 3} fp32 oracle forwards at batch {batch}"}
            rec["speedup_vs_cpu_e2e"] = cs * 1e3 / ms_e2e
        out[key] = rec
    out["configs[4] depth / width sweep"] = config5_sweep(peak_tf)
    return out


def config5_sweep(peak_tf):
    """BASELINE configs[4]: forward of deeper / wider generators (the reference's Optuna search space:
    num_residual_blocks 8-14 and ESRGAN's 23, srgan_train.py:454; inter_channels 32 / 64, :283-284) at large batch
    (1024 training tiles) and on one full continent tile; whole-forward TFLOP/s and fraction of the measured bf16 peak."""
    from deepbedmap_b200 import GeneratorModel

    def macs_per_trunk_px(nb, g):
        stem = 32 * (9 + 900 + 72 + 9)
        rdb = 9 * (64 * g + (64 + g) * g + (64 + 2 * g) * g + (64 + 3 * g) * g + (64 + 4 * g) * 64)
        head = 4 * 9 * 64 * 64 + 16 * 9 * 64 * 64 + 16 * 9 * 64 * (18 + 64) + 16 * 9 * 64 * (18 + 1)
        return stem + 9 * 128 * 64 + 3 * nb * rdb + 9 * 64 * 64 + head

    rows = []
    for label, n, h in (("1024 tiles 11x11", 1024, 11), ("1 tile 288x288", 1, 288)):
        gen = torch.Generator(device="cuda").manual_seed(42)
        ins = (torch.rand(n, 1, h, h, generator=gen, device="cuda"), torch.rand(n, 1, 10 * h, 10 * h, generator=gen, device="cuda"),
               torch.rand(n, 2, 2 * h, 2 * h, generator=gen, device="cuda"), torch.rand(n, 1, h, h, generator=gen, device="cuda"))
        for inter in (32, 64):
            for nb in (8, 12, 23):
                m = GeneratorModel(num_residual_blocks=nb, inter_channels=inter, precision="bf16")
                for _ in range(2):
                    m.forward(*ins)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(3):
                    m.forward(*ins)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / 3
                gflop = 2.0 * macs_per_trunk_px(nb, inter) * n * (h - 2) ** 2 / 1e9
                rows.append({"workload": label, "num_residual_blocks": nb, "inter_channels": inter, "gflop_forward": gflop,
                             "ms": ms, "tflops": gflop / ms, "frac_of_bf16_peak": gflop / ms / peak_tf})
                del m
                torch.cuda.empty_cache()
    return rows


def run_inference(args, rank, world, local):
    from deepbedmap_b200 import GeneratorModel, _lib, tiler
    peak_tf, peak_hbm, peak_src = measured_peaks()
    if args.scale != 1.0:
        fy = max(1000, int(FULL["final_shape"][0] * args.scale) // 1000 * 1000)
        fx = max(1000, int(FULL["final_shape"][1] * args.scale) // 1000 * 1000)
        final_shape, grid = (fy, fx), (fy // 4 + 2, fx // 4 + 2)
    else:
        final_shape, grid = FULL["final_shape"], FULL["grid"]
    mpx = final_shape[0] * final_shape[1] / 1e6
    kw = dict(final_shape=final_shape, ary_shape=(1000, 1000), stride=(1000, 1000), xtrapad=(18, 18),
              batch_tiles=args.batch_tiles)

    model = GeneratorModel(num_residual_blocks=12, residual_scaling=0.1, precision="bf16", seed=0)
    X, W1, W2, W3 = synth_grids_device(grid)
    grids = tiler.ContinentGrids(X, W1, W2, W3)

    def step():
        return tiler.predict_continent(model, None, None, None, None, grids=grids, to_host=False, **kw)

    for _ in range(args.warmup):
        step()
    barrier(world)
    l0 = _lib.kernel_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        e0.record()
        for _ in range(args.steps):
            y_hat = step()
        e1.record()
        barrier(world)
    launches = _lib.kernel_launches() - l0   # counted inside the library, one per kernel launch
    ms = max_over_ranks(e0.elapsed_time(e1), world)
    value = mpx * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        # the DEM is 1.58 GB: 2^23 seeded pixels of the part the tiles write (their abutting windows), not of the
        # frame the reference leaves NaN, which nothing computes
        plan = tiler.tile_plan(final_shape, kw["ary_shape"], kw["stride"], kw["xtrapad"])
        ys, ye = min(t[4] for t in plan), max(t[5] for t in plan)
        xs, xe = min(t[6] for t in plan), max(t[7] for t in plan)
        dump_outputs(args.dump_outputs, {"continent_sample": seeded_sample(y_hat[0, ys:ye, xs:xe], 1 << 23)})
    del y_hat

    # every rank runs the instrumented strip (predict_continent ends in a collective); rank 0's CUDA-event timings
    # are the ones reported
    roof = instrumented_roofline(model, grids, kw, peak_tf)
    barrier(world)

    # ---- parity of one benchmark tile (+ the CPU baseline sample: the same forward on the host cores) ----
    parity = cpu = None
    do_cpu = (not args.no_cpu) and world == 1 and rank == 0
    if rank == 0 and args.scale == 1.0:
        cores = cpu_threads()
        parity, secs, (th, tw) = tile_parity(model, grids, do_cpu)
        if do_cpu:
            total = continent_flop_weight()
            px = 16 * (th - 2) * (tw - 2)
            kind, probe = reference_kind()
            cpu = {"value": MPX / (secs * total / px), "unit": "Mpx/s", "cores": cores, "kind": kind,
                   "sample": f"1 fp32 oracle forward of one full {th}x{tw} interior tile of this continent ({secs:.1f} s), "
                             f"extrapolated x{total / px:.0f} by computed-pixel count to the 396-tile mix",
                   "reference_engine_probe": probe}
    barrier(world)

    # ---- end to end: pinned host grids -> host DEM ----
    e2e = None
    if not args.no_e2e:
        # each rank keeps only the band of grid rows under its own tiles on the host (what it uploads)
        plan = tiler.tile_plan(final_shape)
        band = tiler.rank_row_band(plan, rank, world) if world > 1 else (0, grid[0])
        host = tiler.HostBand(*[torch.empty(t[:, :, s * band[0]:s * band[1]].shape, dtype=torch.float32,
                                            pin_memory=True).copy_(t[:, :, s * band[0]:s * band[1]])
                                for t, s in ((X, 1), (W1, 10), (W2, 2), (W3, 1))], row0=band[0], full_rows=grid[0])
        torch.cuda.synchronize()
        del grids, X, W1, W2, W3
        torch.cuda.empty_cache()
        h2d = 4 * (grid[0] * grid[1] * (1 + 100 + 8 + 1))
        sink = tiler.HostDEM(final_shape)   # rank 0 owns it; other ranks map the same pinned shared memory
        tiler.predict_continent(model, host, out=sink, **kw)  # warm-up
        barrier(world)
        t0 = time.perf_counter()
        n_e2e = max(1, min(args.steps, 2))
        for _ in range(n_e2e):
            out = tiler.predict_continent(model, host, out=sink, **kw)
        barrier(world)
        dt = max_over_ranks((time.perf_counter() - t0) * 1e3, world)
        e2e = {"value": mpx * n_e2e / (dt * 1e-3), "unit": "Mpx/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": int(final_shape[0] * final_shape[1] * 4), "steps": n_e2e,
               "api": "deepbedmap_b200.predict_continent(model, host grids, out=HostDEM): band-wise H2D of each rank's "
                      "rows overlapped with compute; every rank streams its finished tile rows into the pinned host DEM"}
        if rank == 0:
            assert out is not None and out.shape == (1, final_shape[0], final_shape[1])
            assert np.isfinite(out[0, 76:-76:97, 76:-76:89]).all()
        del host, out
        sink.close()

    train = configs = None
    if not args.no_train:
        try:
            train = train_bench(rank, world, local, steps=args.train_steps, warmup=5, cpu=do_cpu, peak_tf=peak_tf)
        except Exception as ex:  # reported, never hidden
            train = {"error": repr(ex)[:300]}
    if not args.no_configs and rank == 0:
        try:
            configs = small_tile_configs(peak_tf, do_cpu)
        except Exception as ex:
            configs = {"error": repr(ex)[:300]}
    barrier(world)

    if rank == 0:
        line = {"metric": "continent inference output Mpx/s", "value": value, "unit": "Mpx/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "bf16 (fp32 accumulate, fp32 residual stream)",
                "data": "synthetic", "config": infer_config(args, world),
                "clocks": clocks.summary(), "e2e": e2e, "gpu_launches": launches, "roofline": roof,
                "roofline_peak_source": peak_src, "cpu_baseline": cpu, "parity": parity, "train": train,
                "configs": configs}
        print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
# training legs
# ------------------------------------------------------------------------------------------------------------
def train_kernel_strip(step_fn, n_steps=2):
    """CUDA events (each on the stream the call is launched on) around every C-ABI call of ``n_steps`` EAGER steps:
    per entry point total time and launches; the three trunk kernels also get their algorithmic TFLOP/s."""
    from deepbedmap_b200 import ops
    recs = []
    orig = ops.call

    def wrapped(name, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig(name, *a)
        e1.record()
        recs.append((name, a[1] if name == "dbm_flat_wgrad" else 0, e0, e1))

    ops.call = wrapped
    try:
        for _ in range(n_steps):
            step_fn()
        torch.cuda.synchronize()
    finally:
        ops.call = orig
    agg = {}
    for name, units, e0, e1 in recs:
        d = agg.setdefault(name, {"ms": 0.0, "launches": 0, "max_units": 0, "by_units": {}})
        t = e0.elapsed_time(e1)
        d["ms"] += t
        d["launches"] += 1
        if name == "dbm_flat_wgrad":
            d["by_units"].setdefault(units, []).append(t)
            d["max_units"] = max(d["max_units"], units)
    return agg, n_steps


def train_bench(rank, world, local, steps=50, warmup=5, batch=128, cpu=False, peak_tf=None, dump_dir=None):
    from deepbedmap_b200 import _lib
    from deepbedmap_b200 import train as T
    if peak_tf is None:
        peak_tf = measured_peaks()[0]
    g, g_opt, d, d_opt = T.compile_srgan_model()
    gen = torch.Generator(device="cuda").manual_seed(42 + rank)
    r = lambda *s: torch.rand(*s, generator=gen, device="cuda")
    shapes = {"X": (batch, 1, 11, 11), "W1": (batch, 1, 110, 110), "W2": (batch, 2, 22, 22), "W3": (batch, 1, 11, 11),
              "Y": (batch, 1, 36, 36)}
    arrays = {k: r(*s) for k, s in shapes.items()}

    # the per-minibatch body of trainer() (srgan_train.py:1286-1308): both steps on the same device batch,
    # the generator step reusing the graph-keeping forward the discriminator step ran (weights unchanged between)
    def eager_step():   # returns the five metrics as GraphedTrainStep.step does
        return (T.train_eval_discriminator(arrays, g, d, d_opt, share_generator_forward=True),
                T.train_eval_generator(arrays, g, d, g_opt))

    launch = "CUDA graph replay (deepbedmap_b200.train.GraphedTrainStep)"
    graphed = None
    try:
        # the step (and, data parallel, its bucketed NCCL all-reduces) is captured once as a CUDA graph and replayed
        graphed = T.GraphedTrainStep(arrays, g, g_opt, d, d_opt)
        step = lambda a=arrays: graphed.step(a)
    except Exception as ex:   # reported in the line, never hidden
        launch = f"eager (graph capture failed: {repr(ex)[:120]})"
        step = lambda a=arrays: eager_step()
    for _ in range(warmup):
        step()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        e0.record()
        for _ in range(steps):
            metrics = step()
        e1.record()
        barrier(world)
    ms = max_over_ranks(e0.elapsed_time(e1), world) / steps
    eager_launches = None
    if dump_dir and rank == 0:   # before the end-to-end steps below train the models further
        dump_outputs(dump_dir, {"train_metrics": np.array([*metrics[0], *metrics[1]], np.float64),
                                "generator_params_sample": seeded_sample(g.flat, 1 << 22),
                                "discriminator_params_sample": seeded_sample(d.flat, 1 << 22)})

    # ---- end to end: a fresh pinned HOST minibatch per step -> H2D -> step -> five metrics back on the host ----
    host_batches = [{k: torch.rand(*s).pin_memory() for k, s in shapes.items()} for _ in range(4)]
    for i in range(3):
        step(host_batches[i % 4])
    barrier(world)
    t0 = time.perf_counter()
    for i in range(steps):
        metrics = step(host_batches[i % 4])
    barrier(world)
    ms_e2e = max_over_ranks((time.perf_counter() - t0) * 1e3, world) / steps
    h2d = sum(int(np.prod(s)) * 4 for s in shapes.values())

    # ---- kernel strip (eager launches, events per call) ----
    if graphed is not None:
        graphed.refresh()
    l1 = _lib.kernel_launches()
    agg, ns = train_kernel_strip(eager_step)
    eager_launches = (_lib.kernel_launches() - l1) // ns
    if graphed is not None:
        graphed.refresh()
    trunk_gflop = 2.0 * TRUNK_MAC_PER_PX * 81 * batch / 1e9
    kernels = {}
    for name, dd in sorted(agg.items(), key=lambda kv: -kv[1]["ms"])[:12]:
        kernels[name] = {"ms_per_step": dd["ms"] / ns, "launches_per_step": dd["launches"] // ns}
    for name in ("dbm_trunk_local_fwd", "dbm_trunk_local_bwd"):
        if name in agg:
            t = agg[name]["ms"] / agg[name]["launches"]
            kernels[name].update(gflop=trunk_gflop, tflops=trunk_gflop / t, frac=trunk_gflop / t / peak_tf)
    if "dbm_flat_wgrad" in agg:
        ts = agg["dbm_flat_wgrad"]["by_units"][agg["dbm_flat_wgrad"]["max_units"]]
        t = float(np.mean(ts))
        kernels["dbm_flat_wgrad"].update(trunk_launch_ms=t, gflop=trunk_gflop, tflops=trunk_gflop / t,
                                         frac=trunk_gflop / t / peak_tf)
    sum_ms = sum(dd["ms"] for dd in agg.values()) / ns
    dom = max(("dbm_trunk_local_fwd", "dbm_trunk_local_bwd", "dbm_flat_wgrad"),
              key=lambda k: kernels.get(k, {}).get("trunk_launch_ms", kernels.get(k, {}).get("ms_per_step", 0.0)))
    gflop_step = GFLOP_PER_SAMPLE_STEP * batch
    ach = gflop_step / ms   # per GPU: GFLOP / ms = TFLOP/s
    roof = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
            "traffic": None, "scope": "whole step per GPU: 6.4995 GFLOP/sample x 128 (SURVEY 8d, generator forward "
                                      "counted once) / graph-replayed step time",
            "kernel": {"dbm_flat_wgrad": "flat_wgrad_kernel (trunk weight gradient)",
                       "dbm_trunk_local_fwd": "local_trunk_kernel<fwd>", "dbm_trunk_local_bwd": "local_trunk_kernel<bwd>"}[dom],
            "dominant_kernel": {k: v for k, v in kernels[dom].items()},
            "strip": {"what": f"CUDA events around every C-ABI call of {ns} eager steps (launch gaps included, streams "
                              "overlap: shares, not a sum)", "sum_ms_per_step": sum_ms, "entry_points": kernels}}
    out = {"metric": "train steps/s (D-step + G-step, batch 128 per GPU)", "value": 1e3 / ms, "unit": "steps/s",
           "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": ms, "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16 tensor-core operands / fp32 accumulation for every 3x3 conv of G and D (fwd, dgrad, wgrad); fp32 "
                    "stem, bilinear sampling, BN, losses, Adam",
           "data": "synthetic", "config": train_config(world, batch), "clocks": clocks.summary(),
           "samples_per_s": batch * world * 1e3 / ms, "algorithmic_tflops": gflop_step * world / ms,
           "e2e": {"value": 1e3 / ms_e2e, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 28,
                   "api": "GraphedTrainStep.step(host minibatch): pinned host arrays -> device, graph replay, the step's "
                          "five metrics read back", "last_metrics": [list(map(float, metrics[0])), list(map(float, metrics[1]))]},
           "gpu_launches": (eager_launches or 0) * steps,
           "gpu_launches_note": (f"{eager_launches} kernels of this library per step (counted inside the library on eager "
                                 "steps)" + (", replayed from one CUDA graph launch per step" if graphed is not None else "")),
           "roofline": roof,
           "generator_forward": "one per step, shared by the D-step and the G-step (the reference runs it twice with "
                                "unchanged weights; SURVEY 8d counts it once)",
           "launch": launch,
           "allreduce": "bucketed, launched from inside backward (NCCL, overlapped)" if world > 1 else "none (1 GPU)"}
    if cpu and rank == 0:
        cores = cpu_threads()
        kind, probe = reference_kind()
        cs = cpu_train_step_time(batch=batch, steps=3)
        out["cpu_baseline"] = {"value": 1.0 / cs, "unit": "steps/s", "cores": cores, "kind": kind,
                               "sample": f"3 D-step + G-step of the fp32 oracle at batch {batch} (reference-literal dataflow: "
                                         f"two generator forwards), {cs:.1f} s each", "reference_engine_probe": probe}
    else:
        out["cpu_baseline"] = None
    del graphed
    return out


def run_train(args, rank, world, local):
    peak_tf, _, peak_src = measured_peaks()
    do_cpu = (not args.no_cpu) and world == 1
    line = train_bench(rank, world, local, steps=args.steps, warmup=max(args.warmup, 3), cpu=do_cpu, peak_tf=peak_tf,
                       dump_dir=args.dump_outputs)
    line["roofline_peak_source"] = peak_src
    if rank == 0:
        print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--metric", default="inference", choices=["inference", "train"])
    ap.add_argument("--batch-tiles", type=int, default=4)
    ap.add_argument("--cpu-crop", type=int, default=144,
                    help="--impl reference: lowres crop edge of the per-step CPU sample (a full tile is 288)")
    ap.add_argument("--cpu-train-batch", type=int, default=32,
                    help="--impl reference --metric train: batch of the per-step CPU sample (scaled to 128)")
    ap.add_argument("--train-steps", type=int, default=50)
    ap.add_argument("--scale", type=float, default=1.0, help="debug only: shrink the continent (invalid as a result)")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (float32 / float64, "
                         "a fixed seeded sample of outputs too large to keep whole, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 2 if args.metric == "inference" else 50
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3
    rank, world, local = dist_setup()
    if args.metric == "train":
        run_train(args, rank, world, local)
    else:
        run_inference(args, rank, world, local)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
