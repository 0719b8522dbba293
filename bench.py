#!/usr/bin/env python
"""Benchmark of the 3DHumanGAN generator hot path on B200 (and its CPU reference arm).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload C2|C2native|C5|tiny] [--dump-outputs DIR]

One "step" = one `Map3DGenerator.forward` over one batch of synthetic latents + random SMPL-like poses
(train-mode BatchNorm, as the reference's trainer runs the generator) at BASELINE.json configs[1]:
batch 8 per GPU, 512x512, render 96x96, 32 samples per ray.  Prints ONE JSON line (rank 0):

  value        images/s, whole job, inputs already resident in HBM, CUDA-event timed, max over ranks
  e2e          images/s through the public module API with pinned HOST inputs (latents + pose conditions
               copied H2D every step) and the generated images read back D2H every step
  roofline     dominant kernel: algorithmic bytes (or FLOPs) per launch / mean CUDA-event duration vs the
               measured peak in MEASURED_PEAKS.json
  cpu_baseline the CPU oracle (port of the reference's PyTorch path) on the host cores, bounded sample
  --impl reference   times that CPU arm on its own (rank 0 only)
  --dump-outputs DIR after the timed steps, rank 0 writes what the timed path returned in its last step as DIR/<name>.npy

Multi-GPU (`torchrun ... bench.py --gpus N`): weak scaling, 8 images per rank, SyncBatchNorm statistics
all-reduced over NCCL inside the forward (18 small all-reduces), no other data-path collective.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "images_per_sec_G_fwd_512x512"
UNIT = "images/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DUMP_BYTES = 60 * 2 ** 20          # --dump-outputs writes at most this much data (headroom under 64 MB for the .npy headers)


_REAL_STDOUT = None


def claim_stdout():
    """Keep stdout to the ONE JSON line: libraries write banners to file descriptor 1 (NCCL prints its version there at
    NCCL_DEBUG=WARN/VERSION), so fd 1 is pointed at stderr for the rest of the process and the JSON line goes to a private
    duplicate of the original stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        d["_source"] = "measured"
        return d
    return dict(FALLBACK_PEAKS, _source="fallback")


def ncu_traffic(entry, workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the newest committed `ncu --set full`
    capture of this workload (profiles/r2_ncu_traffic.json, written from tools/profile_r2.sh's export: the mean over the 18
    half-block launches of one forward, all variants); null for workloads / kernels that were not captured.  (A profiler cannot
    run inside the timed process; the capture is refreshed whenever the kernel changes.)"""
    p = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    if not os.path.exists(p):
        return None
    d = json.load(open(p)).get(entry, {}).get(workload)
    return None if d is None else d["dram_bytes_per_launch_mean_of_18"]


def dump_outputs(path, outputs):
    """Write every output as <path>/<name>.npy, float64 as float64 and anything else as float32.  When together they exceed
    DUMP_BYTES, each array is replaced by the same fraction of its elements (flattened) at positions drawn from a fixed seed,
    so that runs with the same arguments, on any build, write files that compare element for element."""
    import numpy as np
    arrays = {}
    for name, v in outputs.items():
        t = v.detach().cpu() if torch.is_tensor(v) else torch.as_tensor(v)
        arrays[name] = (t.double() if t.dtype == torch.float64 else t.float()).numpy()
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_BYTES:
            flat = a.reshape(-1)
            keep = int(flat.size * DUMP_BYTES / total)
            a = flat[np.sort(np.random.default_rng(0).choice(flat.size, keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def workload_cfg(pkg, name):
    cfg = pkg.configs.baseline_config(name)
    cfg["nerf_noise"] = 0.0
    return cfg


# --------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores (bounded sample)
# --------------------------------------------------------------------------------------------------
def cpu_sample(pkg, name, steps, warmup, sample_div=4):
    """Times `oracle.port.generator_forward` for ONE image on a 1/sample_div^2 sub-grid of the workload
    (gen and render resolutions divided by sample_div, same 32 samples per ray, same dims) and scales
    by the pixel ratio.  Returns (images_per_sec, cores, description, median seconds per pass, outputs of the last pass)."""
    from oracle import port
    cores = host_cores()
    torch.set_num_threads(cores)
    cfg = workload_cfg(pkg, name)
    full_px = cfg["gen_height"] * cfg["gen_width"]
    cfg.update(gen_height=cfg["gen_height"] // sample_div, gen_width=cfg["gen_width"] // sample_div,
               render_height=cfg["render_height"] // sample_div, render_width=cfg["render_width"] // sample_div)
    frac = cfg["gen_height"] * cfg["gen_width"] / full_px
    params = port.init_generator_params(cfg, seed=0)
    cond = pkg.synthetic.make_conditions(1, seed=1)
    z = torch.randn(1, cfg["latent_dim"], generator=torch.Generator().manual_seed(2))
    R, S = cfg["render_height"] * cfg["render_width"], cfg["num_steps"]
    torch.manual_seed(3)
    u, noise = pkg.rng.draw_render_noise(1, R, S, "cpu", cfg["sample_dist"])
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            out = port.generator_forward(params, z, cond, cfg, u, noise, training=True)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    times.sort()
    t = times[len(times) // 2]                       # median pass
    desc = (f"oracle.port.generator_forward, 1 image on a {cfg['gen_height']}x{cfg['gen_width']} / render "
            f"{cfg['render_height']}x{cfg['render_width']}x{S} sub-grid ({frac:.4f} of the workload's pixels), "
            f"median of {len(times)} passes {t:.2f} s (min {times[0]:.2f}, max {times[-1]:.2f}), scaled by pixel count; fp32, "
            f"torch {torch.__version__}, {cores} threads = len(os.sched_getaffinity(0)) (os.cpu_count() = {os.cpu_count()})")
    return frac / t, cores, desc, t, out


def host_cores():
    """Cores this process may actually run on (cgroup / affinity aware): `os.cpu_count()` reports the machine's 128 even when
    the container is given a fraction of them, and 128 torch threads on fewer cores made the round-1 CPU arm swing 19x."""
    try:
        n = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):      # cgroup v2 / v1 CPU quota
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                quota, period = txt[0], float(txt[1])
            else:
                quota, period = txt[0], float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota not in ("max", "-1"):
                n = max(1, min(n, int(float(quota) / period + 0.999)))
            break
        except (OSError, ValueError, IndexError):
            continue
    return n


def run_reference(args, pkg):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    warm = 1
    ips, cores, desc, t, out = cpu_sample(pkg, args.workload, steps, warm)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    cfg = workload_cfg(pkg, args.workload)
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": t * 1000.0, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": describe(cfg, args.workload, 8), "timing": "host wall clock, bounded sample"},
        "cpu_baseline": {"value": ips, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": ips, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def describe(cfg, name, batch):
    return (f"{name}: Map3DGenerator.forward, batch {batch}/GPU, gen {cfg['gen_height']}x{cfg['gen_width']}, render "
            f"{cfg['render_height']}x{cfg['render_width']}, {cfg['num_steps']} samples/ray, hidden {cfg['hidden_dim']}, "
            f"train-mode BatchNorm, random init, synthetic SMPL-like poses")


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index):
        self.path = tempfile.mktemp(suffix=".csv")
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        rows = [r.split(", ") for r in open(self.path).read().strip().splitlines() if r.count(",") >= 6]
        os.unlink(self.path)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].strip().lower() == "active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}


def kernel_costs(cfg, B):
    """Algorithmic work per launch of each kernel (DESIGN.md 'Kernels'): FLOPs of the fp32-equivalent
    contraction and compulsory HBM bytes."""
    HW = cfg["gen_height"] * cfg["gen_width"]
    R, S = cfg["render_height"] * cfg["render_width"], cfg["num_steps"]
    C = 256
    act = B * HW * C * 4
    return {
        # mean over the 18 half-block launches of a forward: read x + write out, + the residual input of the second half of blocks
        # 4..8 (5 launches), + the 3-channel ToRGB accumulator of 6 launches (read + write)
        "hg_spade_conv": {"flops": 2.0 * B * HW * C * C, "bytes": 2.0 * act + (5.0 / 18.0) * act + (6.0 / 18.0) * 2.0 * B * HW * 3 * 4},
        "hg_render_mlp": {"flops": 938496.0 * B * R * S, "bytes": B * R * S * (36 + 1) * 4.0 + B * R * 260 * 4.0},
        "hg_geo_features": {"flops": 8.0 * B * R * S * 6890, "bytes": B * R * S * (36 + 1 + 1) * 4.0},
    }


def parity_gate(pkg, G, cfg, z, cond, kw, dev, tol=1e-3):
    """One forward of the benchmarked batch through the module, compared with `oracle.port.generator_forward` run on the
    same device in fp32 (TF32 off) on the same parameters, latents, poses and random draws.  Raises if the images differ by
    more than `tol` (relative L2) or are not finite: a fast kernel with different results is not a result."""
    from oracle import port                              # checker only (never on the timed path)
    rng = importlib.import_module("3dhumangan_b200.rng")
    B = z.shape[0]
    R, S = cfg["render_height"] * cfg["render_width"], cfg["num_steps"]
    g = torch.Generator(device=dev).manual_seed(1234)
    u = torch.rand(B, R, S, 1, device=dev, generator=g)
    noise = torch.randn(B, R, S, 1, device=dev, generator=g)
    state = {k: v.detach().clone() for k, v in G.state_dict().items()}       # the forward advances buffers (BN, spectral u/v)
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False
    orig = rng.draw_render_noise
    rng.draw_render_noise = lambda *a, **k: (u, noise)
    try:
        with torch.no_grad():
            out = G(z, cond, **kw)
            ref = port.generator_forward(state, z, cond, cfg, u, noise, training=True)
    finally:
        rng.draw_render_noise = orig
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    # The reference's own compositing makes alpha of the LAST sample a step function of sign(sigma_last) (delta = 1e10,
    # volume_rendering.py:20-21,33): a ray whose last density is within rounding of zero is background in one fp32
    # evaluation and opaque in another (CPU vs GPU torch disagree on the same rays).  With 73 728 rays per batch a few
    # such rays are expected, each an O(1) difference on ~100 pixels.  The gate therefore trims the 0.1 % worst elements
    # (reported) and requires the relative L2 of the remaining 99.9 % below `tol`.
    res, plain, outliers = {}, {}, {}
    for key in ("rgbs", "rgbs_render"):
        a, b = out[key].double(), ref[key].double()
        if not bool(torch.isfinite(a).all()):
            raise SystemExit(f"bench parity gate: {key} is not finite")
        e2 = (a - b).square().reshape(-1)
        plain[key] = float(e2.sum().sqrt() / b.norm())
        k = max(1, int(e2.numel() * 1e-3))
        kept = e2.sum() - torch.topk(e2, k).values.sum()
        res[key] = float(kept.clamp_min(0).sqrt() / b.norm())
        outliers[key] = int((e2.sqrt() > 1e-2 * b.abs().max()).sum())
    del ref, state
    torch.cuda.empty_cache()
    if max(res.values()) > tol:
        raise SystemExit(f"bench parity gate FAILED: relative L2 vs oracle {res} (untrimmed {plain}) > {tol}")
    return {"checker": "oracle.port.generator_forward on the same device, fp32, TF32 off", "batch": B, "tol": tol,
            "rel_l2_trimmed_99.9pct": res, "rel_l2_all": plain, "elements_off_by_more_than_1pct_of_max": outliers}


def run_gpu(args, pkg):
    import torch.distributed as dist
    abi = importlib.import_module("3dhumangan_b200.abi")
    gen = importlib.import_module("3dhumangan_b200.modules.generator")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("bench.py --gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    abi.require_device()

    cfg = workload_cfg(pkg, args.workload)
    B = args.batch
    torch.manual_seed(0)
    G = gen.Map3DGenerator(**cfg).to(dev)
    G.set_device(dev)
    G.train()
    passes_mode = args.precision
    kw = dict(cfg, hg_precision=passes_mode, hg_cuda_graph=not args.no_graph, hg_cuda_graph_nccl=not args.no_graph)

    # host (pinned) inputs: per-rank latents and poses
    cond_h = {k: v.pin_memory() for k, v in pkg.synthetic.make_conditions(B, seed=1 + rank).items()}
    z_h = torch.randn(B, cfg["latent_dim"], generator=torch.Generator().manual_seed(2 + rank)).pin_memory()
    out_h = torch.empty(B, 3, cfg["gen_height"], cfg["gen_width"]).pin_memory()
    h2d = z_h.numel() * 4 + sum(v.numel() * v.element_size() for v in cond_h.values())
    d2h = out_h.numel() * 4
    cond_d = {k: v.to(dev) for k, v in cond_h.items()}
    z_d = z_h.to(dev)

    # Parity gate BEFORE anything is timed: this rank's batch, at the benchmarked size, through the same module call,
    # against the oracle executed on the device in true fp32 (before the process group exists: single-GPU BatchNorm
    # statistics on both sides; the cross-rank statistics are covered by tests/test_gpu_multi.py).
    parity = None if args.no_parity else parity_gate(pkg, G, cfg, z_d, cond_d, dict(kw, hg_cuda_graph=False), dev)

    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")      # keep stdout to the one JSON line
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")   # the watchdog must not query events of a capturing stream
        dist.init_process_group("nccl", device_id=dev)

    last = {}                         # what the module returned in the latest resident step (--dump-outputs)

    def step_resident():
        with torch.no_grad():
            last.update(G(z_d, cond_d, **kw))
        return last["rgbs"]

    def step_e2e():
        with torch.no_grad():
            c = {k: v.to(dev, non_blocking=True) for k, v in cond_h.items()}
            z = z_h.to(dev, non_blocking=True)
            out_h.copy_(G(z, c, **kw)["rgbs"], non_blocking=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    for _ in range(max(args.warmup, 3)):
        step_resident()
    torch.cuda.synchronize()

    sampler = ClockSampler(local) if rank == 0 else None
    ms_total = timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)

    # Per-kernel device time: the same step launched eagerly with a CUDA-event pair around every launch of the
    # C ABI (a captured graph cannot carry timing events).  Also counts this library's launches per step.
    kw_eager = dict(kw, hg_cuda_graph=False)

    def step_eager():
        with torch.no_grad():
            return G(z_d, cond_d, **kw_eager)["rgbs"]

    step_eager()
    torch.cuda.synchronize()
    abi.TIMING = []
    launches0 = abi.LAUNCHES
    ms_eager = timed(step_eager, args.steps)
    launches = abi.LAUNCHES - launches0
    timing, abi.TIMING = abi.TIMING, None

    for _ in range(2):
        step_e2e()
    ms_e2e = timed(step_e2e, args.steps)

    # the TIMED path is the graph replay: same seed + same buffers => its pixels must equal the eager launch sequence that
    # the parity gate compared with the oracle
    graph_vs_eager = None
    if not args.no_parity:
        bufs = {k: v.detach().clone() for k, v in G.named_buffers()}
        torch.cuda.manual_seed(4321)
        a = step_resident().double().clone()
        for k, v in G.named_buffers():
            v.copy_(bufs[k])
        torch.cuda.manual_seed(4321)
        b = step_eager().double()
        graph_vs_eager = float((a - b).norm() / b.norm())
        del a, b, bufs
    if os.environ.get("HG3D_BENCH_DEBUG") and rank == 0:
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        t0 = time.perf_counter()
        with torch.no_grad():
            ev[0].record()
            c = {k: v.to(dev, non_blocking=True) for k, v in cond_h.items()}
            z = z_h.to(dev, non_blocking=True)
            ev[1].record()
            t1 = time.perf_counter()
            r = G(z, c, **kw)["rgbs"]
            ev[2].record()
            t2 = time.perf_counter()
            out_h.copy_(r, non_blocking=True)
            ev[3].record()
        t3 = time.perf_counter()
        torch.cuda.synchronize()
        t4 = time.perf_counter()
        sys.stderr.write("e2e breakdown (device ms): h2d %.2f forward %.2f d2h %.2f | host ms: h2d-issue %.2f forward-issue %.2f "
                         "d2h-issue %.2f drain %.2f\n" % (ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]),
                                                        (t1 - t0) * 1e3, (t2 - t1) * 1e3, (t3 - t2) * 1e3, (t4 - t3) * 1e3))

    imgs = B * world * args.steps
    value = imgs / (ms_total / 1000.0)
    e2e = imgs / (ms_e2e / 1000.0)

    run_leg = args.workload == "C2" and not args.no_train
    if rank != 0:
        if run_leg:
            getattr(G, "_graphs", {}).clear()
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            try:
                train_leg(args, pkg, dev, rank, world, args.train_batch, args.train_steps, 3, args.precision, args.train_split)
            except Exception:
                import traceback
                traceback.print_exc()
        _leave(world, G)
        return

    # per-kernel device time from the events recorded inside the timed region
    per = {}
    for name, s, e in timing:
        d = per.setdefault(name, [0.0, 0])
        d[0] += s.elapsed_time(e)
        d[1] += 1
    breakdown = {k: {"ms_per_step": v[0] / args.steps, "launches_per_step": v[1] / args.steps, "ms_per_launch": v[0] / v[1]}
                 for k, v in sorted(per.items(), key=lambda kv: -kv[1][0])}
    pk = peaks()
    costs = kernel_costs(cfg, B)
    dom = next(iter(breakdown))
    roof = None
    if dom in costs:
        sec = breakdown[dom]["ms_per_launch"] / 1000.0
        fl, by = costs[dom]["flops"], costs[dom]["bytes"]
        mult = 3.0 if passes_mode == "fp32x3" else 1.0
        t_tensor = fl * mult / (pk["bf16_tflops"] * 1e12)
        t_hbm = by / (pk["hbm_gbs"] * 1e9)
        if t_hbm >= t_tensor:
            roof = {"bound": "hbm", "achieved": by / sec / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s"}
        else:
            roof = {"bound": "tensor", "achieved": fl / sec / 1e12, "peak": pk["bf16_tflops"], "unit": "TFLOP/s"}
        roof["frac"] = roof["achieved"] / roof["peak"]
        roof.update(kernel=dom, traffic=ncu_traffic(dom, args.workload), peak_source=pk["_source"], algorithmic_flops_per_launch=fl,
                    algorithmic_bytes_per_launch=by, mma_passes=int(mult),
                    tensor_frac_issued=fl * mult / sec / (pk["bf16_tflops"] * 1e12),
                    hbm_frac=by / sec / (pk["hbm_gbs"] * 1e9))

    cpu = None
    if world == 1 and not args.no_cpu:
        ips, cores, desc, _, _ = cpu_sample(pkg, args.workload, 3, 1)
        cpu = {"value": ips, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (bf16x3 split on tcgen05, fp32 accumulate)" if passes_mode == "fp32x3" else "bf16",
        "data": "synthetic",
        "config": {"workload": describe(cfg, args.workload, B), "global_batch": B * world,
                   "parallelism": f"dp{world} (SyncBatchNorm statistics all-reduced over NCCL)" if world > 1 else "single GPU",
                   "l2": "every synthesis activation is %.2f GB (>> 126 MB L2): inputs larger than L2, no flush needed"
                         % (B * 256 * cfg["gen_height"] * cfg["gen_width"] * 4 / 1e9),
                   "precision": passes_mode,
                   "launch": "eager" if (args.no_graph or getattr(G, "_graph_broken", False)) else
                   "whole forward replayed as one CUDA graph" + (" (NCCL all-reduces captured)" if world > 1 else "")},
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "parity_checked": parity is not None and graph_vs_eager is not None and graph_vs_eager < 1e-3,
        "parity": None if parity is None else dict(parity, graph_replay_vs_eager_rel_l2=graph_vs_eager),
        "eager_ms_per_step": ms_eager / args.steps,
        "clocks": clocks,
        "roofline": roof,
        "cpu_baseline": cpu,
        "kernels": breakdown,
        "train_step": None,
    }
    # Second metric of BASELINE.json (G+D training iteration) in the same run, on every rank, so that the driver's
    # N = 1, 2, 4, 8 scaling runs carry both curves.  The forward line must survive a failure or a hang of this leg:
    # a watchdog on rank 0 prints the line without it after 15 minutes.
    if run_leg:
        import threading

        def give_up():
            line["train_step"] = {"error": "training leg did not finish within 900 s"}
            emit(line)
            os._exit(0)

        dog = threading.Timer(900.0, give_up)
        dog.daemon = True
        dog.start()
        getattr(G, "_graphs", {}).clear()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        try:
            line["train_step"] = train_leg(args, pkg, dev, rank, world, args.train_batch, args.train_steps, 3, args.precision,
                                           args.train_split)
        except Exception as err:
            import traceback
            traceback.print_exc()
            line["train_step"] = {"error": f"{type(err).__name__}: {str(err)[:300]}"}
        # BASELINE.json pins the training configuration at bf16: the same iteration with single-pass bf16 products (fp32
        # storage and accumulation; the analogue of the reference's autocast mode), next to the fp32x3 headline
        # Single-GPU runs only: the decision to enter a leg must be identical on every rank (it builds DDP wrappers, i.e.
        # collectives), and only rank 0 holds the first leg's result.
        if world == 1 and args.precision == "fp32x3" and not args.no_train_bf16 and isinstance(line["train_step"], dict) \
                and "error" not in line["train_step"]:
            try:
                leg = train_leg(args, pkg, dev, rank, world, args.train_batch, args.train_steps, 2, "bf16", args.train_split)
                if leg is not None:
                    leg.pop("kernels", None)
                line["train_step_bf16"] = leg
            except Exception as err:
                import traceback
                traceback.print_exc()
                line["train_step_bf16"] = {"error": f"{type(err).__name__}: {str(err)[:300]}"}
        dog.cancel()
    emit(line)
    _leave(world, G)


def train_leg(args, pkg, dev, rank, world, B, steps, warm, precision, split, dump=None):
    """BASELINE.json's second metric: one G+D training iteration (discriminator step, then generator step) per step through
    `train_step.Trainer` -- the mirror of the reference's PhaseTrainer (DDP wrappers with their gradient all-reduce over
    NCCL when world > 1, SyncBatchNorm statistics all-reduced inside the generator, five Adam groups, clip, EMA, R1 on its
    2-of-8 phase schedule).  B images per GPU per iteration, in `split` micro-batches (the reference's `batch_split`).
    Returns the sub-object that goes into the JSON line (rank 0) or None.  With `dump`, the two losses of the last timed
    iteration are written there (dump_outputs)."""
    import torch.distributed as dist
    abi = importlib.import_module("3dhumangan_b200.abi")
    gen = importlib.import_module("3dhumangan_b200.modules.generator")
    disc = importlib.import_module("3dhumangan_b200.modules.discriminator")
    ts = importlib.import_module("3dhumangan_b200.train_step")
    cfg = workload_cfg(pkg, "C2")
    cfg["nerf_noise"] = 0.5                      # SURVEY.md §8d: C3 trains with sigma noise
    cfg["batch_split"] = split
    cfg["hg_precision"] = precision
    torch.manual_seed(0)
    G = gen.Map3DGenerator(**cfg).to(dev).train()
    G.set_device(dev)
    D = disc.UNetDiscriminator(**cfg).to(dev).train()
    trainer = ts.Trainer(G, D, cfg, amp=False)
    Hg, Wg = cfg["gen_height"], cfg["gen_width"]
    gcpu = torch.Generator().manual_seed(5 + rank)
    host = dict(z_d=torch.randn(B, cfg["latent_dim"], generator=gcpu), z_g=torch.randn(B, cfg["latent_dim"], generator=gcpu),
                images=torch.randn(B, 3, Hg, Wg, generator=gcpu).clamp_(-1, 1),
                labels=torch.randint(1, cfg["label_dim"], (B, Hg, Wg), generator=gcpu))
    host = {k: v.pin_memory() for k, v in host.items()}
    cond_h = {k: v.pin_memory() for k, v in pkg.synthetic.make_conditions(B, seed=1 + rank).items()}
    h2d = sum(v.numel() * v.element_size() for v in list(host.values()) + list(cond_h.values()))
    resident = {k: v.to(dev) for k, v in host.items()}
    resident["cond"] = {k: v.to(dev) for k, v in cond_h.items()}
    loss_h = torch.empty(2).pin_memory()

    last = []

    def step_resident():
        last[:] = trainer.iteration(resident)

    def step_e2e():
        batch = {k: v.to(dev, non_blocking=True) for k, v in host.items()}
        batch["cond"] = {k: v.to(dev, non_blocking=True) for k, v in cond_h.items()}
        d, g = trainer.iteration(batch)
        loss_h.copy_(torch.stack([d.float(), torch.as_tensor(g, device=dev).float()]), non_blocking=True)

    per_iter = []
    host_ms = []          # host time spent enqueueing an iteration (no synchronisation inside): ~ the GPU time => launch bound

    def timed(fn, n, record=False):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        ev[0].record()
        for i in range(n):
            r1 = bool(cfg["phases"][D.step % len(cfg["phases"])]["do_r1"])
            t0 = time.perf_counter()
            fn()
            ev[i + 1].record()
            if record:
                host_ms.append((time.perf_counter() - t0) * 1e3)
                per_iter.append([r1, ev[i], ev[i + 1]])
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([ev[0].elapsed_time(ev[n])], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    torch.cuda.reset_peak_memory_stats()
    for _ in range(warm):
        step_resident()
    sampler = ClockSampler(dev.index) if rank == 0 else None
    abi.LAUNCHES = 0
    ms_total = timed(step_resident, steps, record=True)
    launches = abi.LAUNCHES
    clocks = sampler.stop() if sampler else None
    if dump:
        dump_outputs(dump, {"d_loss": last[0], "g_loss": last[1]})
    ms_e2e = timed(step_e2e, steps)
    finite = bool(torch.isfinite(loss_h).all())
    it_ms = [(r1, a.elapsed_time(b)) for r1, a, b in per_iter]
    ms_r1 = [m for r1, m in it_ms if r1]
    ms_plain = [m for r1, m in it_ms if not r1]
    abi.TIMING = []
    torch.cuda.synchronize()
    step_resident()
    torch.cuda.synchronize()
    per = {}
    for name, s_, e_ in abi.TIMING:
        d = per.setdefault(name, [0.0, 0])
        d[0] += s_.elapsed_time(e_)
        d[1] += 1
    abi.TIMING = None
    peak_mem = torch.cuda.max_memory_allocated() / 1e9
    del trainer, G, D, resident
    torch.cuda.empty_cache()
    if rank != 0:
        return None
    imgs = B * world * steps
    # reference-equivalent work of an iteration (SURVEY.md §8d table): 10.8 TFLOP per image as the reference executes it
    eq_tflops = 10.8 * imgs / (ms_total / 1e3)
    pk = peaks()
    return {
        "metric": "images_per_sec_GD_train_step_512x512", "value": imgs / (ms_total / 1e3), "unit": UNIT, "n_gpus": world,
        "steps": steps, "warmup": warm, "ms_per_step": ms_total / steps, "scaling": "weak",
        "dtype": "f32 (bf16x3 split on tcgen05, fp32 accumulate)" if precision == "fp32x3" else "bf16 products, fp32 storage",
        "config": {"workload": f"C3: one discriminator step + one generator step per iteration (train_step.Trainer = PhaseTrainer's "
                               f"steps: segmentation loss, R1 on its 2-of-8 phase schedule with r1_lambda = {cfg['r1_lambda']} as in "
                               f"configs/map3d.py:98-191, five Adam groups, grad clip 1, EMA), {B} images/GPU/iteration in {split} "
                               f"micro-batch(es) of {B // split} (the reference's batch_split), 512x512, render 96x96, 32 samples/ray, "
                               f"hidden 256, random init, synthetic images / labels / poses; no path-length regulariser exists in the reference",
                   "global_batch": B * world,
                   "parallelism": (f"dp{world}: DistributedDataParallel(find_unused_parameters=True) gradient all-reduce over NCCL for G and D "
                                   f"+ SyncBatchNorm statistics") if world > 1 else "single GPU",
                   "precision": precision, "launch": "eager"},
        "e2e": {"value": imgs / (ms_e2e / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                "ms_per_step": ms_e2e / steps},
        "gpu_launches": launches, "losses_finite": finite, "clocks": clocks, "peak_mem_gb": peak_mem,
        "iteration_ms": {"do_r1": (sum(ms_r1) / len(ms_r1)) if ms_r1 else None,
                         "plain": (sum(ms_plain) / len(ms_plain)) if ms_plain else None,
                         "r1_iterations_timed": len(ms_r1), "plain_iterations_timed": len(ms_plain),
                         "schedule": "do_r1 on 2 of 8 phases (configs/map3d.py:104-113)",
                         "host_enqueue_ms": sum(host_ms) / max(1, len(host_ms))},
        "roofline": {"bound": "tensor", "achieved": eq_tflops / world, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                     "frac": eq_tflops / world / pk["bf16_tflops_sustained"], "traffic": None,
                     "note": "reference-equivalent FLOPs of the whole iteration (10.8 TFLOP/image, SURVEY.md 8d) per GPU vs the "
                             "sustained bf16 tensor peak; fp32x3 issues 3 MMA passes per product"},
        "kernels": {k: {"ms_per_step": v[0], "launches_per_step": v[1]} for k, v in sorted(per.items(), key=lambda kv: -kv[1][0])},
    }


def run_train(args, pkg):
    """--workload C3: only the G+D training-iteration metric, as its own JSON line."""
    import torch.distributed as dist
    abi = importlib.import_module("3dhumangan_b200.abi")
    rank, world, local = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("WORLD_SIZE", "1"), ("LOCAL_RANK", "0")))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=dev)
    abi.require_device()
    leg = train_leg(args, pkg, dev, rank, world, args.train_batch, args.steps, max(args.warmup, 3), args.precision, args.train_split,
                    dump=args.dump_outputs if rank == 0 else None)
    if rank == 0:
        leg.update(higher_is_better=True, vs_baseline=None, data="synthetic", cpu_baseline=None)
        emit(leg)
    _leave(world, None)


def _leave(world, G):
    """End a multi-rank run without tearing NCCL down: destroying a communicator whose kernels are still referenced
    by live CUDA graphs blocks, so drop the graphs, drain the device and leave the process directly."""
    if world <= 1:
        return
    if G is not None:
        getattr(G, "_graphs", {}).clear()
    torch.cuda.synchronize()
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C2", choices=["C2", "C2native", "C5", "tiny", "C3"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--precision", default=os.environ.get("HG3D_PRECISION", "fp32x3"), choices=["fp32x3", "bf16"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying a CUDA graph")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity gate (profiling runs)")
    ap.add_argument("--no-train", action="store_true", help="skip the G+D training-iteration leg of the default run")
    ap.add_argument("--no-train-bf16", action="store_true", help="skip the additional bf16 training-iteration leg")
    ap.add_argument("--train-batch", type=int, default=16, help="images per GPU per training iteration (config C3: 16)")
    ap.add_argument("--train-split", type=int, default=2, help="micro-batches per iteration (the reference's batch_split)")
    ap.add_argument("--train-steps", type=int, default=4, help="timed training iterations in the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    claim_stdout()
    pkg = importlib.import_module("3dhumangan_b200")
    if args.impl == "reference":
        if args.workload == "C3":
            emit({"impl": "reference", "unavailable": "the CPU arm times the generator forward (C2); a CPU training "
                                                       "iteration at 512x512 does not fit a bounded sample"})
            return
        run_reference(args, pkg)
    elif args.workload == "C3":
        run_train(args, pkg)
    else:
        run_gpu(args, pkg)


if __name__ == "__main__":
    main()
