#!/usr/bin/env python
"""Benchmark of the HyperReel per-ray rendering hot path on B200 (contract: see the task prompt / DESIGN.md section 5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one pass of the hot path (sample net -> intersect -> VM gather -> decode -> composite) over one
synthetic batch of 65 536 rays x 32 samples per GPU, Technicolor-shape model (technicolor_z_plane: C_in=8,
K=12 keyframes of 50 frames, comps [8,0,0], SH-27, final-size 1007x1007x503 grid, 62 MiB of tables),
seeded random-init sample net, "trained-like" density tables.  The model is built through the registry path with its
defaults (tensor-core sample net).  Weak scaling: every rank renders its own 65 536-ray shard and its finished tile lands
in every rank's gather buffer (ray_shard.render_sharded: peer-memory epilogue, else one NCCL all_gather), inside the timed
region.  Rank 0 prints ONE JSON line; extra keys carry the other BASELINE configurations (DoNeRF shape S=16, Neural-3D
shape S=64), strong-scaling points and the stated baselines (reference's op sequence on the host CPUs and, eagerly, on
the same B200).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

RAYS_PER_GPU = 65536
WORKLOAD = "technicolor_z_plane"
N_VOXELS = 512000000  # final grid 1007x1007x503 (utils/tensorf_utils.py:65-68)
DENSITY_GAIN = 30.0
PARAM_SEED = 11
CPU_SAMPLE_RAYS = int(os.environ.get("HR_BENCH_CPU_RAYS", "8192"))  # bounded CPU sample (the env override is for the CPU test)
L2_FLUSH_BYTES = 512 << 20
METRIC = "Mrays/s at 65k-ray x 32-sample batch"

# the other single-GPU BASELINE configurations, reported as extra keys (rays per GPU: one 800x800 DoNeRF frame; one eighth
# of a 2704x2028 Neural-3D frame = the per-GPU share of BASELINE config 4)
EXTRA_WORKLOADS = {
    "donerf_sphere_s16": dict(builtin="donerf_sphere", over=dict(n_voxels=216000000, z_channels=16), rays=640000,
                              what="DoNeRF shape (BASELINE config 2): 800x800 frame, 16 samples/ray, sphere primitives, grid 600^3, comps [8,4,4], RGB"),
    "neural3d_s64": dict(builtin="neural_3d_z_plane", over=dict(n_voxels=262144000), rays=685464,
                         what="Neural-3D shape (BASELINE config 4): 1/8 of a 2704x2028 frame, 64 samples/ray, grid 823x617x514, K=12, comps [8,4,4], SH-27"),
}


def algorithmic_bytes_per_ray(sig) -> int:
    """SURVEY.md section 8(d): 4*C_in + 12 + S * sum_fields sum_planes 4*C*(4 + T), T = 4 dynamic / 2 static."""
    c = sig.cfg
    T = 4 if c.dynamic else 2
    per_sample = 0
    for comps in (c.n_sigma, c.n_app):
        for i in range(3):
            per_sample += 4 * int(comps[i]) * (4 + T)
    return 4 * c.c_in + 12 + c.n_samples * per_sample


def executed_bytes_per_ray(sig) -> int:
    """What the render kernel actually fetches: the dynamic second factor is pre-blended per keyframe at upload
    (hr_api.cu:pack_time_lines), so it costs 2 taps like a static line; plus the ray and the heads row."""
    c = sig.cfg
    per_sample = 0
    for comps in (c.n_sigma, c.n_app):
        for i in range(3):
            per_sample += 4 * int(comps[i]) * (4 + 2)
    return 4 * c.c_in + 12 + 4 * c.mlp_out + c.n_samples * per_sample


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def measured_tensor_peak():
    """Dense bf16 TFLOP/s: burst figure of MEASURED_PEAKS.json (cuBLAS 8192^3), else the profiling recipe's fallback."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        if "bf16_tflops" in d:
            return float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", 0.0)), "measured (MEASURED_PEAKS.json bf16_tflops, cuBLAS burst)"
    return 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


def usable_cpus() -> int:
    """Host threads this process may really use: the affinity mask, cut by a cgroup CPU quota when there is one
    (os.cpu_count() ignores both; round 1 asked a 128-thread pool from a box that granted far fewer)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, math.ceil(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, math.ceil(q / per)))
            break
        except Exception:
            continue
    return max(1, n)


def cpu_model() -> str:
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = max((int(r[1]) for r in self.rows if r[1].isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.rows)}


def build_workload(builtin=WORKLOAD, over=None, gain=DENSITY_GAIN, app_gain=1.0):
    import hyperreel_b200 as hb
    from hyperreel_b200.state import seeded_state_dict

    cfg, ds = hb.configs.get(builtin, **(over or dict(n_voxels=N_VOXELS)))
    sig = hb.lower(cfg, ds)
    sd = seeded_state_dict(sig, seed=PARAM_SEED, density_gain=gain, app_gain=app_gain)
    return hb, cfg, ds, sig, sd


def workload_config(sig, n: int, world: int) -> dict:
    """The `config` object, identical in both arms (the reference arm times a bounded sample of this workload and says so
    in its cpu_baseline.sample)."""
    return {"workload": f"{WORKLOAD}: {n} rays x {sig.n_samples} samples per GPU, grid 1007x1007x503, K=12, comps [8,0,0], SH-27",
            "rays_per_gpu": n, "samples_per_ray": sig.n_samples,
            "parallelism": f"ray-shard x{world}, finished rgb tiles gathered on every rank",
            "l2": f"flushed between timed iterations ({L2_FLUSH_BYTES >> 20} MiB memset)",
            "params": f"seed {PARAM_SEED}, density gain {DENSITY_GAIN} (trained-like)"}


def time_oracle(cfg, ds, sd, sig, hb, steps: int, warmup: int, rays_n: int, device: str = "cpu"):
    """The reference's op sequence restated (oracle port, same torch ops as the reference: F.grid_sample gathers, boolean-
    mask compaction, cumprod), eager PyTorch.  device='cpu': all usable host threads.  device='cuda': the same eager ops on
    the B200 -- the "beat eager PyTorch on the same GPU" baseline of SURVEY.md 2.3.  Returns (Mrays/s from the median step,
    median ms, threads, rgb of the last step)."""
    import torch
    from oracle.hyperreel_oracle import HyperReelOracle

    threads = usable_cpus()
    torch.set_num_threads(threads)
    dev = torch.device(device)
    rays = hb.rays.for_signature(sig, rays_n, seed=5).to(dev)
    with torch.device(dev):
        orc = HyperReelOracle(hb.config.to_plain(cfg), ds, {k: v.to(dev) for k, v in sd.items()}, gather="grid_sample")
        ts = []
        for i in range(warmup + steps):
            if dev.type == "cuda":
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            rgb = orc.render(rays.clone())
            if dev.type == "cuda":
                torch.cuda.synchronize()
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return rays_n / med / 1e6, med * 1e3, threads, rgb


def cpu_baseline_object(mrays, cores, sig, extra=""):
    return {"value": mrays, "unit": "Mrays/s", "cores": cores, "kind": "port", "cpu": cpu_model(),
            "sample": f"{CPU_SAMPLE_RAYS} rays x {sig.n_samples} samples per step (bounded sample of the 65536-ray batch), oracle port = the "
                      f"reference's torch ops (grid_sample gathers) on {cores} host threads, median step{extra}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    hb, cfg, ds, sig, sd = build_workload()
    steps, warm = max(args.steps, 1), max(min(args.warmup, 2), 1)
    mrays, ms, cores, rgb = time_oracle(cfg, ds, sd, sig, hb, steps, warm, CPU_SAMPLE_RAYS)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"rgb": rgb})
    line = {
        "impl": "reference", "metric": METRIC, "value": mrays, "unit": "Mrays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(sig, args.rays, max(args.gpus, 1)),
        "cpu_baseline": cpu_baseline_object(mrays, cores, sig),
        "e2e": {"value": mrays, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def ncu_summary():
    """Numbers of the committed ncu --set full capture of the render kernel (profiles/render_kernel_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "render_kernel_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f)
    return {}


def make_render(hb, cfg, ds, sd, mlp=None):
    kw = {} if mlp is None else {"mlp_mode": mlp}
    model = hb.LightfieldModel(cfg, dataset=ds, **kw)  # registry defaults: the tensor-core sample net
    render = hb.RenderLightfield(model, None, cfg.render, net_chunk=1 << 22)
    render.load_state_dict(sd, strict=False)
    render.eval()
    return model, render


def timed_steps(torch, step, steps, flush):
    """Total ms of `steps` timed calls of `step`, and what the last call returned."""
    evs = []
    out = None
    for _ in range(steps):
        flush.zero_()  # evict L2 between timed iterations
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = step()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs), out


def dump_outputs(out_dir, arrays):
    """Write each output array as `<out_dir>/<name>.npy` (float32), so that two builds can be compared output for output."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def kernel_times(torch, model, step, steps, flush):
    model.timing(True)
    for _ in range(steps):
        flush.zero_()
        step()
    torch.cuda.synchronize()
    tm = model.timing_read()
    model.timing(False)
    return tm


def roofline_object(sig, n, tm, peak, peak_src, ncu=None, kernel="render_kernel (fused intersect+gather+decode+composite)"):
    bpr = algorithmic_bytes_per_ray(sig)
    achieved = (bpr * n / (tm["render_ms"] * 1e-3) / 1e9) if tm["render_ms"] > 0 else 0.0
    obj = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
           "traffic": None, "kernel": kernel, "algorithmic_bytes_per_ray": bpr, "executed_bytes_per_ray": executed_bytes_per_ray(sig),
           "kernel_ms": tm["render_ms"], "peak_source": peak_src, "sample_net_kernel_ms": tm["mlp_ms"]}
    if ncu:
        obj["traffic"] = ncu.get("dram_bytes_per_launch")
        if ncu.get("dram_bytes_per_launch") and tm["render_ms"] > 0:
            obj["dram_frac"] = ncu["dram_bytes_per_launch"] / (tm["render_ms"] * 1e-3) / 1e9 / peak
        for k in ("l1_wavefront_pct", "warps_active_pct", "ncu_source"):
            if k in ncu:
                obj[k] = ncu[k]
    return obj


def run_extra_workloads(torch, hb, dev, flush, steps, peak, peak_src):
    out = {}
    for key, spec in EXTRA_WORKLOADS.items():
        hb_, cfg, ds, sig, sd = build_workload(spec["builtin"], spec["over"], gain=100.0, app_gain=6.0)
        model, render = make_render(hb, cfg, ds, sd)
        n = spec["rays"]
        rays = hb.rays.for_signature(sig, n, seed=5).to(dev)

        def step():
            return render(rays)["rgb"]

        for _ in range(3):
            step()
        torch.cuda.synchronize()
        ms = timed_steps(torch, step, steps, flush)[0] / steps
        tm = kernel_times(torch, model, step, steps, flush)
        out[key] = {"workload": spec["what"], "rays": n, "samples_per_ray": sig.n_samples, "value": n / (ms * 1e-3) / 1e6,
                    "unit": "Mrays/s", "ms_per_step": ms, "steps": steps,
                    "roofline": roofline_object(sig, n, tm, peak, peak_src)}
        del model, render, rays
        torch.cuda.empty_cache()
    return out


def run_train_step(torch, hb, dev, steps):
    """BASELINE config 3 ("train+render"): INRSystem.training_step (forward in training mode, MSE, backward through the
    render-backward kernel and the sample net, one Adam per optimiser group, re-pack of the updated parameters) on the
    Technicolor shape at the final grid.  Reported per batch size: whole-step ms and the render-backward kernel alone with the
    bytes it reduces into the gradient tables (24*C bytes per sample, field and VM group: 4 plane taps + 2 line taps)."""
    hb_, cfg, ds, sig, sd = build_workload(gain=600.0, app_gain=6.0)
    system = hb.INRSystem(hb.to_cfg({"model": cfg, "training": {"ray_chunk": 1 << 20, "iters_per_epoch": 4000}, "dataset": ds}))
    system.load_state_dict(sd)
    system.to(dev)
    system.configure_optimizers()
    model = system.render_fn.model
    c = sig.cfg
    red_bytes_per_ray = c.n_samples * sum(24 * int(x) for comps in (c.n_sigma, c.n_app) for x in comps)
    peak, peak_src = measured_peaks()
    out = {"what": "technicolor_z_plane, grid 1007x1007x503, K=12: INRSystem.training_step (image loss only), fp32; sample-net "
                   "Linear layers forward/backward as torch (cuBLAS SGEMM) ops, everything else hand-written kernels",
           "batches": []}
    for n in (16384, 65536):
        g = torch.Generator().manual_seed(3)
        batch = {"coords": hb.rays.for_signature(sig, n, seed=9).to(dev), "rgb": torch.rand(n, 3, generator=g).to(dev)}
        for _ in range(3):
            system.training_step(batch)
        torch.cuda.synchronize()
        evs = []
        for _ in range(steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            system.training_step(batch)
            b.record()
            evs.append((a, b))
        torch.cuda.synchronize()
        ms = sum(a.elapsed_time(b) for a, b in evs) / steps
        model.timing(True)
        for _ in range(steps):
            system.training_step(batch)
        torch.cuda.synchronize()
        tm = model.timing_read()
        model.timing(False)
        bw = tm["backward_ms"]
        out["batches"].append({"rays": n, "train_step_ms": ms, "Mrays_per_s": n / (ms * 1e-3) / 1e6,
                               "render_backward_kernel_ms": bw,
                               "roofline": {"bound": "l2 atomics (reported against the HBM copy peak)", "unit": "GB/s",
                                            "reduction_bytes_per_ray": red_bytes_per_ray,
                                            "achieved": (red_bytes_per_ray * n / (bw * 1e-3) / 1e9) if bw > 0 else None,
                                            "peak": peak, "frac": (red_bytes_per_ray * n / (bw * 1e-3) / 1e9 / peak) if bw > 0 else None,
                                            "peak_source": peak_src}})
    del system
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (hyperreel_b200 has no CPU path); use --impl reference for the CPU baseline")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from hyperreel_b200.ray_shard import render_sharded

    hb, cfg, ds, sig, sd = build_workload()
    model, render = make_render(hb, cfg, ds, sd, args.mlp)
    n = args.rays
    N = world * n
    # the global batch: rank r owns rows [r*n, (r+1)*n) (contiguous ranges, SURVEY.md 8e); every rank holds all rays, as a
    # frame renderer would (rays come from the camera, hr_generate_rays)
    rays_all = torch.cat([hb.rays.for_signature(sig, n, seed=5 + r) for r in range(world)], 0)
    rays_host = rays_all[rank * n:(rank + 1) * n].clone().pin_memory()
    rays_all = rays_all.to(dev)
    rays = rays_all[rank * n:(rank + 1) * n]
    flush = torch.empty(L2_FLUSH_BYTES // 4, dtype=torch.float32, device=dev)
    gather_mode = "single GPU"

    def step():
        if world > 1:
            return render_sharded(rays_all, render)  # the product path: each rank renders its shard, tiles land everywhere
        return render(rays)["rgb"]

    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        out = step()
    torch.cuda.synchronize()
    if world > 1:
        from hyperreel_b200 import ray_shard
        gather_mode = "nccl all_gather" if ray_shard._p2p_broken else "peer-memory epilogue (hr_render_scatter) + signal barrier"
        # the gathered frame must be what one GPU renders alone
        local_full = torch.cat([render(rays_all[r * n:(r + 1) * n])["rgb"] for r in range(world)], 0)
        assert torch.equal(out, local_full), "gathered tiles differ from a local re-render"
        del local_full
    BAD = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown")
    remeasured = False
    while True:
        launches0 = model.launch_count()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        total_ms, last_out = timed_steps(torch, step, args.steps, flush)
        if world > 1:
            dist.barrier()
        launches = model.launch_count() - launches0
        # a timed region that saw a hardware / thermal slowdown is measured again, once (sw_power_cap is kept and reported)
        bad = torch.tensor([1 if (not remeasured and any(r in BAD for r in sampler.summary()["reasons"])) else 0], device=dev)
        if world > 1:
            dist.all_reduce(bad, op=dist.ReduceOp.MAX)
        if int(bad.item()) == 0:
            break
        remeasured = True
        time.sleep(2.0)
    if args.dump_outputs and rank == 0:  # copied now: later passes reuse the model's buffers
        dump_outputs(args.dump_outputs, {"rgb": last_out})
    del last_out
    # per-kernel durations for the roofline: a second pass with the library's CUDA events around each kernel (kept out of
    # the headline loop so the event records do not sit between the two kernels of a step)
    tm = kernel_times(torch, model, step, args.steps, flush)
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = N / (ms_per_step * 1e-3) / 1e6

    # ---- end to end through the host-buffer API: pinned rays in, rgb out, copies inside the timed region ----
    rgb_host = torch.empty((n, 3), dtype=torch.float32).pin_memory()
    for _ in range(3):
        model.render_host(rays_host, rgb_host)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e2e_t = []
    for _ in range(args.steps):
        flush.zero_()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.render_host(rays_host, rgb_host)
        e2e_t.append(time.perf_counter() - t0)
    e2e_ms = sum(e2e_t) / len(e2e_t) * 1e3
    t2 = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t2, op=dist.ReduceOp.MAX)
    e2e_val = N / (float(t2.item()) * 1e-3) / 1e6

    # ---- strong scaling (multi-GPU): a fixed total batch split over the ranks, through render_sharded ----
    strong = None
    if world > 1:
        strong = []
        for total in (65536, 262144, 1048576, 4194304):  # BASELINE config 5: the 65k - 4M sweep
            rs = torch.cat([hb.rays.for_signature(sig, min(total, 1 << 20), seed=77)] * max(1, total >> 20), 0)[:total].to(dev)

            def sstep():
                return render_sharded(rs, render)

            for _ in range(3):
                got = sstep()
            torch.cuda.synchronize()
            lo = (rank * 7919) % max(total - 4096, 1)
            assert torch.equal(got[lo:lo + 4096], render(rs[lo:lo + 4096])["rgb"]), "strong-scaling tiles differ from a local re-render"
            dist.barrier()
            k = max(3, args.steps // 4)
            ms = torch.tensor([timed_steps(torch, sstep, k, flush)[0] / k], device=dev, dtype=torch.float64)
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            strong.append({"rays_total": total, "rays_per_gpu": total // world, "ms_per_step": float(ms.item()),
                           "value": total / (float(ms.item()) * 1e-3) / 1e6, "unit": "Mrays/s", "steps": k})
            del rs
    # ---- BASELINE config 4: one full Neural-3D frame (2704 x 2028 rays, 64 samples) ray-sharded over the ranks ----
    frame = None
    if world > 1 and not args.no_extras:
        spec = EXTRA_WORKLOADS["neural3d_s64"]
        _, fcfg, fds, fsig, fsd = build_workload(spec["builtin"], spec["over"], gain=100.0, app_gain=6.0)
        fmodel, frender = make_render(hb, fcfg, fds, fsd)
        total = 2704 * 2028
        fr = torch.cat([hb.rays.for_signature(fsig, 1 << 20, seed=91)] * 6, 0)[:total].to(dev)

        def fstep():
            return render_sharded(fr, frender)

        for _ in range(2):
            got = fstep()
        torch.cuda.synchronize()
        lo = (rank * 104729) % (total - 4096)
        assert torch.equal(got[lo:lo + 4096], frender(fr[lo:lo + 4096])["rgb"]), "frame tiles differ from a local re-render"
        dist.barrier()
        k = 3
        ms = torch.tensor([timed_steps(torch, fstep, k, flush)[0] / k], device=dev, dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        frame = {"workload": "Neural-3D shape (BASELINE config 4): full 2704x2028 frame, 64 samples/ray, grid 823x617x514, K=12, comps [8,4,4], "
                             "SH-27, ray-sharded over the ranks through render_sharded", "rays_total": total,
                 "rays_per_gpu": total // world, "ms_per_frame": float(ms.item()), "frames_per_s": 1e3 / float(ms.item()),
                 "value": total / (float(ms.item()) * 1e-3) / 1e6, "unit": "Mrays/s", "steps": k}
        del fr, fmodel, frender
        torch.cuda.empty_cache()
    # the timed regions last a few milliseconds, far less than one nvidia-smi poll: keep the same step running for about
    # 1.5 s more (a fixed count, so that every rank issues the same number of barriers) so that the clock /
    # throttle-reason samples are taken under this load
    for _ in range(5000):
        step()
    torch.cuda.synchronize()
    sampler.stop_flag.set()
    sampler.join(timeout=2)

    extras = None
    baselines = {}
    if rank == 0 and world == 1 and not args.no_extras:
        peak, peak_src = measured_peaks()
        extras = run_extra_workloads(torch, hb, dev, flush, max(3, args.steps // 4), peak, peak_src)
        try:
            extras["train_step"] = run_train_step(torch, hb, dev, max(3, args.steps // 4))
        except Exception as e:  # the render line must survive a failure of the next-tier row
            extras["train_step"] = {"unavailable": repr(e)[:300]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:  # the reference's op sequence, eager PyTorch, on this same B200 (full 65 536-ray batch)
            mr, ms, _, _ = time_oracle(cfg, ds, sd, sig, hb, 5, 2, n, device=f"cuda:{local}")
            baselines["torch_eager_b200"] = {"value": mr, "unit": "Mrays/s", "ms_per_step": ms, "rays": n,
                                             "what": "oracle port (the reference's torch op sequence: grid_sample gathers, mask compaction, cumprod) "
                                                     "run eagerly on cuda:0, fp32, median of 5 after 2 warm-ups; a stated baseline"}
        except Exception as e:  # never let a baseline break the bench line
            baselines["torch_eager_b200"] = {"unavailable": repr(e)[:200]}
        torch.cuda.empty_cache()

    if rank == 0:
        peak, peak_src = measured_peaks()
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            mr, _, cores, _ = time_oracle(cfg, ds, sd, sig, hb, 5, 1, CPU_SAMPLE_RAYS)
            cpu = cpu_baseline_object(mr, cores, sig, extra=" of 5 after 1 warm-up")
        # sample net (tensor-core bound): algorithmic MACs of the six Linear layers x 3 split products x 2 flop
        macs = sum(o * i for o, i in sig.mlp_layer_shapes)
        tpeak, tsust, tsrc = measured_tensor_peak()
        tc = model.sig.cfg.mlp_mode == 1
        products = 3 if tc else 1
        tach = (2.0 * products * macs * n / (tm["mlp_ms"] * 1e-3) / 1e12) if tm["mlp_ms"] > 0 else 0.0
        cfg_obj = workload_config(sig, n, world)
        cfg_obj["gather"] = gather_mode
        cfg_obj["sample_net"] = "bf16x3 on tcgen05 (registry default)" if tc else "fp32 CUDA cores"
        line = {
            "metric": METRIC, "value": value, "unit": "Mrays/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 (sample net bf16x3 split on tcgen05, fp32 accumulate)" if tc else "f32",
            "data": "synthetic", "config": cfg_obj,
            "e2e": {"value": e2e_val, "unit": "Mrays/s", "h2d_bytes_per_step": n * sig.c_in * 4, "d2h_bytes_per_step": n * 12,
                    "ms_per_step": float(t2.item()),
                    "path": "hr_render_host per rank: pinned rays read zero-copy over PCIe by the sample net's encoder warps (the H2D "
                            "transfer, inside the timed region), rgb stored by the render kernel's epilogue straight into the pinned "
                            "host buffer (the D2H transfer, posted writes over PCIe); wall clock per call incl. the final sync"},
            "gpu_launches": int(launches),
            "clocks": dict(sampler.summary(), remeasured=remeasured),
            "roofline": roofline_object(sig, n, tm, peak, peak_src, ncu_summary()),
            "roofline_sample_net": {"bound": "tensor" if tc else "fp32 simt", "achieved": tach, "peak": tpeak,
                                    "unit": "TFLOP/s", "frac": tach / tpeak if tpeak else None, "peak_sustained": tsust,
                                    "useful_frac": (tach / products) / tpeak if tpeak else None,
                                    "kernel": "mlp_tc2_kernel (bf16 hi/lo split, 3 tcgen05.mma per k-step)" if tc else "mlp_simt_kernel",
                                    "algorithmic_macs_per_ray": macs, "executed_flop_per_ray": 2 * products * macs,
                                    "kernel_ms": tm["mlp_ms"], "peak_source": tsrc},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if baselines:
            line["baselines"] = baselines
        if extras is not None:
            line["extra_workloads"] = extras
        if strong is not None:
            line["strong"] = strong
        if frame is not None:
            line["frame_neural3d"] = frame
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--mlp", default=os.environ.get("HR_BENCH_MLP"), choices=[None, "auto", "fp32", "bf16x3"],
                    help="A/B only: the default (None) is whatever the registry path picks")
    ap.add_argument("--rays", type=int, default=RAYS_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the rgb the timed path returned in its last timed step as DIR/rgb.npy (float32)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
