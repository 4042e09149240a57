#!/usr/bin/env python
"""Benchmark of the TriNeRFLet reconstruction hot path on B200 (contract: see the task statement / DESIGN.md section 5).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config small|base_light|large] [--scaling weak|strong]
    python bench.py ... --dump-outputs DIR                              also write the last timed step's results as .npy
    python bench.py --mode render [--max-steps 4096]                    full-frame 800x800 inference, ray-tile sharded
    python bench.py --impl reference ...                                the reference's CPU path on the host cores
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Metric (BASELINE.json): rays/s per training step (fwd+bwd): one step = encoder.get_planes() (multilevel IDWT,
outside autocast) + render of N rays (near/far, march, tri-plane sampling, sigma/color MLP, composite) + MSE +
wavelet L1 regulariser + backward down to the coefficient / MLP gradients (+ NCCL gradient exchange at N > 1),
in the order of reconstruction/nerf/utils.py:1138-1166.  The optimizer step and the density-grid refresh are
outside the metric (SURVEY.md 8d) and reported separately under "extras" (incl. the amortised cost of the
every-16th dense step + update_extra_state).

`--impl reference` times the reference's CPU implementation of the same path (the oracle port: pytorch_wavelets and
the CUDA-only extensions cannot run on a CPU here) on the host cores, on a bounded sample of the same workload.
"""
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

METRIC = "rays/sec per training step (fwd+bwd)"
METRIC_RENDER = "rays/sec full-frame render (800x800, inference)"
UNIT = "rays/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--config", default="base_light", help="small | base_light | large (BASELINE.json configs[1..3]); tiny / cpu for tests")
    ap.add_argument("--mode", default="train", choices=["train", "render"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: the config's rays PER GPU; strong: the config's rays in total, sharded over the GPUs")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rays", type=int, default=0, help="rays per step (default: the config's)")
    ap.add_argument("--max-steps", type=int, default=4096, help="render mode: max_steps of the marcher (BASELINE configs[4]: 4096)")
    ap.add_argument("--infer-chunk", type=int, default=8, help="render mode: iterations per read of the device-driven loop state (0 = host loop)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the measurements outside the contract line (optimizer, grid refresh, GPU reference, next rows)")
    ap.add_argument("--no-next-rows", action="store_true", help="skip the extras.next_rows measurements (feeder, render loops)")
    ap.add_argument("--occupancy-radius", type=float, default=0.75,
                    help="radius of the occupied ball (SURVEY.md 8d: 0.75 = the metric's scene, 0.4 = the sparse preset that exposes the plane-bound regime)")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="N > 1: gradient exchange by this package's peer-memory kernels (multimem / P2P) or by NCCL (bf16 dirty tiles)")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from Python instead of replaying the captured CUDA graph")
    ap.add_argument("--cpu-budget", type=float, default=25.0, help="seconds of CPU work for the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (train: the loss and "
                         "every parameter gradient; render: image, depth, weights_sum), float32; a gradient larger than its share "
                         "of 64 MB is written as a sample at fixed seeded positions")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """arrays: name -> tensor.  Writes float32 <name>.npy files, at most DUMP_BYTES in all: a tensor with more elements than
    its share is flattened and sampled at sorted positions drawn from a generator seeded by its size, so that two runs (or two
    builds) with the same arguments write the same positions."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // 4 // max(len(arrays), 1)
    for name, t in arrays.items():
        a = t.detach().float()
        if a.numel() > cap:
            idx = np.unique(np.random.default_rng(a.numel()).integers(0, a.numel(), size=cap))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


# ---------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed regions (NVML, every 2 ms in a thread; a timed region of a few
    steps is shorter than nvidia-smi's start-up time, so the CLI loop of the profiling recipe is only the fallback)."""
    REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu, self.sm, self.mask, self.max_mhz = gpu_index, [], 0, None
        self.h = self.nv = self.proc = None
        self.active = False
        self.stop_flag = False
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[gpu_index]) if vis and all(t.strip().isdigit() for t in vis.split(",")) else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            if self.active:
                try:
                    self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                    self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                except Exception:
                    pass
            time.sleep(0.002)

    def start(self):
        if self.nv is not None:
            self.active = True
            return
        try:
            self.rows = []
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.rows.append([c.strip() for c in ln.split(",")]) for ln in self.proc.stdout],
                             daemon=True).start()
        except Exception:
            self.proc = None

    def pause(self):
        self.active = False

    def stop(self):
        self.active = False
        self.stop_flag = True
        if self.nv is not None:
            sm = sorted(self.sm)
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(n for b, n in self.REASONS if self.mask & b), "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def load_peaks():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(peaks["hbm_gbs"]), float(peaks.get("bf16_tflops", 1671.7)), "measured (MEASURED_PEAKS.json: hbm_gbs, bf16_tflops burst)"
    except Exception:
        return 6650.0, 1670.0, "fallback 6650 GB/s / 1670 TFLOP/s (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------------
# algorithmic bytes / flops (SURVEY.md 8d) per kernel, from the scalar arguments the profiler hook records
# ---------------------------------------------------------------------------------------------------------
_SPARSE = ("tnl_idwt_level_forward_sparse", "tnl_idwt_level_backward_sparse")
_PARTS_POS = {"tnl_idwt_level_forward_sparse": -1, "tnl_idwt_level_backward_sparse": -1}


def kernel_key(name, meta):
    """One entry per KERNEL: the work-list IDWT entry points launch one kernel per bit of `parts` (bit 0: the active blocks =
    the real (adjoint) transform, bit 1: the clean blocks = a streaming |yh| / lambda*sign pass); the training step issues them
    as separate calls, so the recorded `parts` argument splits them."""
    if name in _SPARSE:
        parts = int(meta[_PARTS_POS[name]]) & 3
        return f"{name}[{ {1: 'active', 2: 'clean', 3: 'active+clean'}.get(parts, parts) }]"
    return name


def algorithmic_bytes(name, meta, C, m_valid, plan=None):
    g = 12 * C * 4
    if name in ("tnl_idwt_level_forward", "tnl_idwt_level_backward"):
        n, c = meta[0], meta[1]
        return 2 * (3 * c * (2 * n) ** 2 * 4)            # read all coefficients of the level + write its planes (= 2 P_level)
    if name in _SPARSE and plan is not None:
        # work-list mode: px = one (plane, channel) layer of n x n coefficients.  Forward reads x + 3 bands on the active
        # blocks, the 3 bands only (|yh| sum) on the clean ones, writes 4 px of planes per active coefficient position;
        # backward reads the 4 px of incoming gradient on the active blocks + the 3 bands everywhere (regulariser sign),
        # writes all 4 gradient layers.
        n, c = meta[0], meta[1]
        lvl = int(round(math.log2(n / plan.n0)))
        px = 3 * c * n * n * 4
        a = plan.stats["active_fraction_forward"][lvl]
        b = plan.stats["active_fraction_backward"][lvl]
        parts = int(meta[-1])
        if name.endswith("forward_sparse"):
            clean = (b - a) if plan.defer_clean_abs else (1 - a)
            return px * (((parts & 1) and a * (4 + 4)) + ((parts & 2) and clean * 3))
        return px * (((parts & 1) and b * (4 + 3 + 4)) + ((parts & 2) and (1 - b) * (3 + 4)))
    if name == "tnl_sample_planes_forward":
        return m_valid * (12 + g)
    if name == "tnl_sample_planes_backward":
        return m_valid * 2 * g
    if name == "tnl_mlp_forward":
        return m_valid * (2 * 3 * C + 28)            # fp16 feature row + dirs in, sigma + rgb out
    if name == "tnl_mlp_backward":
        return m_valid * (2 * 2 * 3 * C + 28)        # feature row in, feature-gradient row out (fp16), dirs, g_sigma, g_rgb
    if name == "tnl_composite_rays_train_forward":
        return m_valid * 24 + meta[1] * 32
    if name == "tnl_composite_rays_train_backward":
        return m_valid * 40 + meta[1] * 32
    if name == "tnl_march_rays_train":
        return meta[3] * 36 + m_valid * 32
    return None


def mlp_params(C, hidden):
    return 3 * C * hidden + hidden * 16 + 31 * hidden + hidden * hidden + 3 * hidden


def algorithmic_flops(name, C, hidden, m_valid):
    """SURVEY.md 8d: 2 * params per point forward, 6 * params per point forward + backward (recompute counted once: the
    algorithm's flops, not the kernel's)."""
    if name == "tnl_mlp_forward":
        return 2.0 * mlp_params(C, hidden) * m_valid
    if name == "tnl_mlp_backward":
        return 4.0 * mlp_params(C, hidden) * m_valid
    return None


def step_bytes(P, C, M, N):
    return 5 * P + M * (3 * 12 * C * 4 + 152) + N * 120


# ---------------------------------------------------------------------------------------------------------
# CPU reference arm (oracle port), BASELINE.md section 4
# ---------------------------------------------------------------------------------------------------------
def cpu_step_sample(cfg, n_rays, budget_s, seed=0):
    """One DIRECTLY timed reference step on the host cores with a bounded number of rays: the IDWT forward + backward run in
    full, the ray part on n_sample rays; scaled to the metric's unit by scaling the (per-ray independent) ray part linearly
    to n_rays.  Nothing else is modelled or fitted."""
    import torch
    from oracle import pipeline
    from trinerflet_b200 import scene
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sc = scene.make_scene()
    bits = scene.packbits_cpu(scene.ball_density_grid(1.5, 0.75), 0.5).numpy()
    P_GB = 3 * cfg["C"] * cfg["R"] ** 2 * 4 / 1e9
    est_idwt = 2.4 * P_GB * (16.0 / cores)                 # ~3.5 s for base-light on 16 cores (measured, round 1)
    planes_sub = 3 if est_idwt < 0.6 * budget_s else 1
    n_sample = int(max(256, min(n_rays, 4096, (budget_s - est_idwt * planes_sub / 3) / 1.5e-4 / max(16.0 / cores, 1.0))))
    batch = scene.sample_batch(sc, n_sample, torch.Generator().manual_seed(seed))
    r = pipeline.timed_step_sample(cfg["C"], cfg["R"], cfg["S"], cfg["hidden"], batch, bits, n_sample, seed, planes_sub)
    idwt = (r["idwt_fwd_s"] + r["idwt_bwd_s"]) * 3.0 / planes_sub
    r.update(cores=cores, n_sample=n_sample, planes_sub=planes_sub, idwt_seconds=idwt,
             scaled_step_seconds=idwt + r["rays_s"] * n_rays / n_sample)
    r["value"] = n_rays / r["scaled_step_seconds"]
    r["sample"] = (f"one step timed directly: multilevel IDWT fwd+bwd in full ({planes_sub}/3 planes at R={cfg['R']}"
                   f"{', x3: the planes are independent batch entries' if planes_sub < 3 else ''}) = {idwt:.2f} s, + march/sample/MLP/composite "
                   f"fwd+bwd on {n_sample} of the {n_rays} rays = {r['rays_s']:.2f} s, the ray part scaled x{n_rays / n_sample:.1f} (rays are independent)")
    return r


def run_reference(args, cfg, n_rays):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    per_step_budget = max(3.0, min(12.0, 150.0 / max(1, args.steps + args.warmup)))
    vals = []
    t_wall = time.perf_counter()
    for i in range(args.warmup + args.steps):
        r = cpu_step_sample(cfg, n_rays, per_step_budget, seed=i)
        if i >= args.warmup:
            vals.append(r)
    t_wall = time.perf_counter() - t_wall
    step_s = sum(v["scaled_step_seconds"] for v in vals) / len(vals)
    value = n_rays / step_s
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.config}: C={cfg['C']} R={cfg['R']} levels={cfg['S']} rays={n_rays} (CPU oracle port; bounded sample per step, see cpu_baseline.sample)"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": vals[-1]["cores"], "kind": "port", "sample": vals[-1]["sample"],
                         "measured_seconds_per_sampled_step": round(sum(v["step_s"] for v in vals) / len(vals), 3),
                         "ms_per_step_note": "ms_per_step = the sampled step scaled to the full ray count (value = rays / ms_per_step); the run's wall time is steps x measured_seconds_per_sampled_step",
                         "wall_seconds": round(t_wall, 1)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_leg(args, cfg, n_rays):
    """cpu_baseline of our line: (a) BASELINE.md section 4 measured directly (CPU config, 65 536 points, fwd+bwd, median of 5);
    (b) the metric's own workload on a bounded sample (cpu_step_sample)."""
    import torch
    from oracle import pipeline
    torch.set_num_threads(os.cpu_count() or 1)
    a = pipeline.cpu_config_benchmark(iters=5, warmup=2)
    r = cpu_step_sample(cfg, n_rays, args.cpu_budget)
    return {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": r["sample"],
            "measured_seconds_sampled_step": round(r["step_s"], 3), "idwt_seconds": round(r["idwt_seconds"], 3),
            "rays_seconds_on_sample": round(r["rays_s"], 3), "n_sample_rays": r["n_sample"],
            "cpu_config": {k: (round(v, 5) if isinstance(v, float) else v) for k, v in a.items()},
            "cpu_config_note": "BASELINE.md section 4: reference torch path (TriPlaneVolume C=16 R=512 S=8 + sigma/color MLP, fp32) fwd+bwd on 65536 random points, measured directly, median"}


# ---------------------------------------------------------------------------------------------------------
# GPU reference baseline (BASELINE.md section 4, last bullet): the reference's own CUDA kernels (oracle/_ref, compiled
# unmodified) + the torch library ops its Python calls (conv_transpose2d IDWT, grid_sample, autocast nn.Linear) on this GPU
# ---------------------------------------------------------------------------------------------------------
def reference_gpu_step(cfg, n_rays, batches, mean_count, radius, steps=3):
    import torch
    from oracle import gpu_reference
    return gpu_reference.timed_training_steps(cfg["C"], cfg["R"], cfg["S"], cfg["hidden"], batches, mean_count, radius, steps)


# ---------------------------------------------------------------------------------------------------------
# extras.next_rows: step feeder + inference loops (SURVEY.md 8f-2 / 8f-3)
# ---------------------------------------------------------------------------------------------------------
def next_rows(args, net, ts, sc, n_rays, dev, use_graph):
    import torch
    from trinerflet_b200 import rays, scene
    out = {}
    try:
        if use_graph:
            H, W = scene.H_IMG, scene.W_IMG
            images = torch.rand(sc.poses.shape[0], H * W, 3, device=dev)          # resident targets (768 MB fp32)
            feeder = rays.RayFeeder(sc.poses.to(dev), sc.intrinsics, H, W, images, seed=0).shuffle()
            for b in range(3):
                ts.replay_from_feeder(feeder, b, n_rays).item()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for b in range(args.steps):
                ts.replay_from_feeder(feeder, 3 + b, n_rays).item()
            e1.record()
            torch.cuda.synchronize()
            out["e2e_device_feeder_rays_per_s"] = n_rays / (e0.elapsed_time(e1) / args.steps * 1e-3)
            out["e2e_device_feeder_note"] = "rays_o / rays_d / targets generated by tnl_rays_from_ids into the graph's static inputs, loss read back every step; 0 H2D bytes per step"
            del feeder, images
    except Exception as ex:  # pragma: no cover
        out["e2e_device_feeder_rays_per_s"] = f"failed: {ex}"
    return out


def _make_net(cfg, dev, radius):
    from trinerflet_b200 import scene
    from trinerflet_b200.network import NeRFNetwork
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=cfg["C"], triplane_resolution=cfg["R"],
                      triplane_wavelet_levels=cfg["S"], hidden_dim=cfg["hidden"], hidden_dim_color=cfg["hidden"]).to(dev)
    scene.init_model_(net, seed=0)                      # identical replicas on every rank
    scene.install_ball_occupancy(net, radius)
    return net


def _dist_setup():
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    return world, rank, local_rank, dev


# ---------------------------------------------------------------------------------------------------------
# full-frame render (BASELINE.json configs[4]): 800x800, max_steps 4096, ray tiles sharded over the GPUs, final gather
# ---------------------------------------------------------------------------------------------------------
def run_render(args, cfg):
    import torch
    import torch.distributed as dist
    from trinerflet_b200 import _lib, parallel, scene
    world, rank, local_rank, dev = _dist_setup()
    _lib.load()
    net = _make_net(cfg, dev, args.occupancy_radius)
    net.eval()
    net.infer_chunk = args.infer_chunk
    sc = scene.make_scene()
    frames = [scene.full_frame(sc, i % sc.poses.shape[0]) for i in range(args.warmup + args.steps)]
    N = frames[0][0].shape[0]
    n_local = int(parallel.tile_shard_indices(N, rank, world).numel()) if world > 1 else N
    host = [tuple(t.contiguous().pin_memory() for t in f) for f in frames]      # the frame's rays (every rank takes its tiles of them)
    devf = [tuple(t.to(dev) for t in f) for f in host]
    kw = dict(bg_color=1, max_steps=args.max_steps, dt_gamma=0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def render_frame(ro, rd):
        """this rank's round-robin ray tiles through the marching loop + the final gather (the only collective)"""
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            return parallel.render_frame_sharded(net, ro, rd, rank, world, **kw)

    # planes: reconstructed once and cached for the whole run, as in the reference's eval (SURVEY.md 3.3)
    with torch.no_grad():
        net.encoder.get_planes()
        net.encoder.reset_cahce()
    torch.cuda.synchronize()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    with torch.no_grad():
        net.encoder.get_planes()
    p1.record()
    torch.cuda.synchronize()
    planes_ms = p0.elapsed_time(p1)
    c0 = _lib.launch_count
    for i in range(args.warmup):
        render_frame(*devf[i])
    launches_per_frame = (_lib.launch_count - c0) / max(args.warmup, 1)
    clocks = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        o = render_frame(*devf[args.warmup + i])
    e1.record()
    barrier()
    if rank == 0:
        clocks.pause()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {k: o[k] for k in ("image", "depth", "weights_sum")})
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_frame = float(ms) / args.steps
    # ---- e2e: host rays in, sharded render + gather, frame out on rank 0, every frame ----
    barrier()
    if rank == 0:
        clocks.start()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(args.steps):
        ro, rd = (t.to(dev, non_blocking=True) for t in host[args.warmup + i])
        o = render_frame(ro, rd)
        if rank == 0:
            img_host, d_host, w_host = o['image'].cpu(), o['depth'].cpu(), o['weights_sum'].cpu()
        else:
            torch.cuda.synchronize()
    f1.record()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    ms2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms2) / args.steps
    samples = None
    loop = getattr(net, "last_infer_loop", None)
    if rank == 0:
        peak, tpeak, peak_src = load_peaks()
        C, R = cfg["C"], cfg["R"]
        P = 3 * C * R * R * 4
        line = {
            "metric": METRIC_RENDER, "value": N / (ms_frame * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_frame, "frames_per_s": 1e3 / ms_frame, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": {"workload": f"full-frame render: {args.config} C={C} R={R}, 800x800 = {N} rays, max_steps={args.max_steps}, perturb=False, ball occupancy r={args.occupancy_radius:g}, random-init",
                       "parallelism": f"round-robin tiles of 256 rays over {world} GPU(s) ({n_local} rays on rank 0), replicated planes (built once, cached), no collective until the final gather (inside the timed region)",
                       "loop": (f"device-driven inference loop, {args.infer_chunk} iterations per state read" if args.infer_chunk else "host-driven loop (one 4-byte read per iteration)"),
                       "l2": "a different camera every frame; planes (1.6 GB) exceed the 126 MB L2"},
            "clocks": clk,
            "e2e": {"value": N / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": N * 24 * world, "d2h_bytes_per_step": N * 20,
                    "frames_per_s": 1e3 / ms_e2e},
            "gpu_launches": int(launches_per_frame * args.steps),
            "extras": {"planes_build_ms_once": round(planes_ms, 3), "planes_GBps": round(2 * P / 1e9 / (planes_ms * 1e-3), 1),
                       "iterations": (loop.iterations_done if loop else None), "state_reads": (loop.reads if loop else None)},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------
# training step
# ---------------------------------------------------------------------------------------------------------
def main():
    args = parse()
    import torch
    from trinerflet_b200 import scene
    cfg = scene.CONFIGS[args.config]
    if args.mode == "render":
        if args.impl == "reference":
            print(json.dumps({"impl": "reference", "unavailable": "the reference's full-frame render needs its CUDA extensions; no CPU path exists for --cuda_ray inference"}))
            return
        run_render(args, cfg)
        return
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    total_rays = args.rays or cfg["rays"]
    n_rays = total_rays if args.scaling == "weak" else -(-total_rays // world_env)      # rays per GPU per step
    if args.impl == "reference":
        run_reference(args, cfg, total_rays)
        return

    import torch.distributed as dist
    from trinerflet_b200 import _lib, trainer

    world, rank, local_rank, dev = _dist_setup()
    _lib.load()

    C, R, S, hidden = cfg["C"], cfg["R"], cfg["S"], cfg["hidden"]
    net = _make_net(cfg, dev, args.occupancy_radius)
    opt = trainer.default_opt()
    ts = trainer.TrainStep(net, opt, optimizer=None, world_size=world, exchange=args.exchange)
    sc = scene.make_scene()
    gen = torch.Generator().manual_seed(1234 + rank)     # each rank draws its own shard of the global batch
    total = args.warmup + args.steps
    host = [tuple(t.pin_memory() for t in scene.sample_batch(sc, n_rays, gen)) for _ in range(total + 3)]
    devb = [tuple(t.to(dev) for t in b) for b in host]
    torch.manual_seed(100 + rank)

    # establish the steady state: mean_count > 0 (no D2H sync in march_rays_train), M rounded up to 128
    net.train()
    ts.forward_backward(*devb[-1], update_grid=False)
    net.mean_count = int(net.step_counter[0, 0].item())
    net.local_step = 0
    m_valid = net.mean_count
    P = 3 * C * R * R * 4

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def eager_step(b):
        net.zero_grad(set_to_none=True)
        return ts.forward_backward(*b, update_grid=False)

    use_graph = not args.no_graph
    if use_graph:
        c0 = _lib.launch_count
        ts.capture(*devb[-2], warmup=0)
        ts._graph_kernel_count = _lib.launch_count - c0

    def one_step(b):
        return ts.replay(*b) if use_graph else eager_step(b)

    for i in range(args.warmup):
        one_step(devb[i])
    # ---- timed region: device-resident inputs ----
    clocks = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    if rank == 0:
        clocks.start()
    launches0 = _lib.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        loss = one_step(devb[args.warmup + i])
    e1.record()
    barrier()
    launches = _lib.launch_count - launches0
    if use_graph:   # replays do not pass through the Python launch counter: kernels per captured step x steps (+ the exchange's)
        launches = ts._graph_kernel_count * args.steps + launches
    if rank == 0:
        clocks.pause()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": loss, **{"grad." + n: p.grad for n, p in net.named_parameters() if p.grad is not None}})
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    counts = net.step_counter[:, 0].float().max().reshape(1)     # samples of the (graph-captured) step slot
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(counts, op=dist.ReduceOp.SUM)
        counts /= world
    ms_per_step = float(ms) / args.steps
    m_valid = float(counts)
    value = n_rays * world / (ms_per_step * 1e-3)

    # ---- e2e: host (pinned) buffers in, loss out, every step ----
    barrier()
    if rank == 0:
        clocks.start()       # the end-to-end region is a timed region under load too
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    h2d = d2h = 0
    for i in range(args.steps):
        hb = host[args.warmup + i]
        b = hb if use_graph else tuple(t.to(dev, non_blocking=True) for t in hb)   # graph mode: H2D into the static buffers
        h2d = sum(t.numel() * t.element_size() for t in hb)
        loss = one_step(b)
        _ = loss.item()
        d2h = 4
    f1.record()
    barrier()
    clk = clocks.stop() if rank == 0 else None
    ms2 = torch.tensor([f0.elapsed_time(f1)], device=dev)
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_value = n_rays * world / (float(ms2) / args.steps * 1e-3)

    if world > 1:              # everything below is rank 0's own work: release the other ranks first
        dist.barrier()
    if rank == 0:
        # ---- per-kernel times (CUDA events around every ABI call on the launching stream) ----
        ts.world_size = 1          # rank-0-only section: no collectives from here on
        if ts.reducer is not None:
            ts.reducer.world_size = 1
        exchange_note = ts.exchange_note
        ts.exch = None             # (the peer exchange's cross-rank barriers would wait for ranks that are done)
        net.encoder.external_grad_buffer = None
        ts.prefetch_planes = False   # per-kernel events must not overlap kernels of two streams
        _lib.profile_start()
        nprof = min(args.steps, 5)
        for i in range(nprof):
            eager_step(devb[args.warmup + i])
        prof = _lib.profile_stop()
        ts.prefetch_planes = True
        peak, tpeak, peak_src = load_peaks()
        kernels = {}
        for name, recs in prof.items():
            groups = {}
            for r in recs:
                groups.setdefault(kernel_key(name, r[1]), []).append(r)
            for key, rs in groups.items():
                t = sum(r[0] for r in rs) / nprof
                by = sum((algorithmic_bytes(name, r[1], C, m_valid, ts._plan) or 0) for r in rs) / nprof
                fl = algorithmic_flops(name, C, hidden, m_valid)
                kernels[key] = {"ms_per_step": round(t, 4), "launches_per_step": len(rs) / nprof,
                                "algorithmic_GB_per_step": round(by / 1e9, 4),
                                "achieved_GBps": round(by / 1e9 / (t * 1e-3), 1) if t > 0 and by else None,
                                "hbm_frac": round(by / 1e9 / (t * 1e-3) / peak, 4) if t > 0 and by else None}
                if fl:
                    kernels[key]["algorithmic_TFLOP_per_step"] = round(fl / 1e12, 4)
                    kernels[key]["achieved_TFLOPps"] = round(fl / 1e12 / (t * 1e-3), 1)
                    kernels[key]["tensor_frac"] = round(fl / 1e12 / (t * 1e-3) / tpeak, 4)
        # DRAM bytes per kernel measured by ncu (dram__bytes_read.sum + dram__bytes_write.sum, one --set full capture of a
        # step of this config, summarised under profiles/), per step
        traffic_tab = {}
        try:
            traffic_tab = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        except Exception:
            pass
        dom = max((k for k in kernels if kernels[k]["achieved_GBps"]), key=lambda k: kernels[k]["ms_per_step"])
        kd = kernels[dom]
        tr = traffic_tab.get(dom) or traffic_tab.get(dom.split("[")[0])
        traffic = None
        if tr and args.config == tr.get("config"):
            traffic = round(tr["dram_bytes_per_step"] / kd["launches_per_step"] / 1e9, 4)
        tensor_bound = dom in ("tnl_mlp_forward", "tnl_mlp_backward")
        if tensor_bound:
            # the MLP heads: the tensor pipe (fed from shared memory), not HBM, is what the kernel is designed against
            roofline = {"bound": "tensor", "kernel": dom, "achieved": kd["achieved_TFLOPps"], "peak": tpeak, "unit": "TFLOP/s",
                        "frac": kd["tensor_frac"], "traffic": traffic, "traffic_unit": "GB/launch",
                        "algorithmic_TFLOP_per_launch": round(kd["algorithmic_TFLOP_per_step"] / kd["launches_per_step"], 5),
                        "hbm_frac_of_same_kernel": kd["hbm_frac"]}
        else:
            roofline = {"bound": "hbm", "kernel": dom, "achieved": kd["achieved_GBps"], "peak": peak, "unit": "GB/s",
                        "frac": kd["hbm_frac"], "traffic": traffic, "traffic_unit": "GB/launch",
                        "algorithmic_GB_per_launch": round(kd["algorithmic_GB_per_step"] / kd["launches_per_step"], 4)}
        roofline.update(peak_source=peak_src, launch_ms=round(kd["ms_per_step"] / kd["launches_per_step"], 4),
                        attribution="per kernel (CUDA events around each launch; the work-list IDWT calls are split by their `parts` argument)")
        # B_step: what the reference's (dense) data flow has to move per step (SURVEY.md 8d).  The work-list IDWT and the
        # cell-sorted gather move far less than that through DRAM, so step_frac_of_hbm_roofline is DENSE-EQUIVALENT throughput;
        # the DRAM utilisation proper is actual_dram_GB_per_step / time (ncu dram bytes of every kernel of one step).
        Bstep = step_bytes(P, C, m_valid, n_rays)
        extras = {"sparse_allreduce_tile_fraction": (round(ts.reducer.fraction, 4) if ts.reducer is not None else None),
                  "idwt_worklist": (ts._plan.stats if ts._plan is not None else None),
                  "M_samples_per_step": m_valid, "B_step_GB": round(Bstep / 1e9, 3),
                  "step_achieved_GBps": round(Bstep / 1e9 / (ms_per_step * 1e-3), 1),
                  "step_frac_of_hbm_roofline": round(Bstep / 1e9 / (ms_per_step * 1e-3) / peak, 4),
                  "step_frac_note": "dense-equivalent: B_step (SURVEY.md 8d, the reference's data flow) / time / peak; see dram_frac for the DRAM utilisation proper",
                  "kernels": kernels}
        step_tr = traffic_tab.get("_step")
        if step_tr and args.config == step_tr.get("config"):
            extras["actual_dram_GB_per_step"] = round(step_tr["dram_bytes_per_step"] / 1e9, 3)
            extras["dram_frac"] = round(step_tr["dram_bytes_per_step"] / 1e9 / (ms_per_step * 1e-3) / peak, 4)
            extras["dram_note"] = f"sum of ncu dram__bytes_read+write over the kernels of one step ({step_tr.get('source', 'profiles/')}) / this run's step time / peak"
        if not args.no_extras:
            measure_extras(args, cfg, net, ts, opt, devb, dev, extras, ms_per_step, m_valid, peak, use_graph, sc, n_rays, world)
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_leg(args, cfg, total_rays)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": {"workload": f"{args.config}: C={C} R={R} wavelet_levels={S} ({int(round(math.log2(S)))} IDWT levels), hidden={hidden}, "
                                   f"{n_rays} rays/GPU/step, synthetic 800x800 Blender-shaped scene, ball occupancy r={args.occupancy_radius:g}, random-init",
                       "rays_per_gpu": n_rays, "global_rays": n_rays * world,
                       "parallelism": (f"ray-sharded dp{world} ({args.scaling} scaling), replicated coefficients; dirty tiles of the plane gradient + MLP gradients "
                                       f"all-reduced between the render backward and the IDWT backward: {exchange_note}" if world > 1 else "single GPU"),
                       "timed_region": "get_planes (work-list IDWT over the occupied tiles) + render + loss + backward (+ gradient exchange); optimizer and density-grid refresh excluded (metric definition), see extras",
                       "launch": ("one CUDA-graph replay per step" if (world == 1 or "peer memory" in (exchange_note or "")) else "two CUDA-graph replays per step around the NCCL exchange") if use_graph else "eager Python launches",
                       "l2": f"inputs ({P / 1e9:.2f} GB of coefficients/planes per pass) exceed the 126 MB L2; a different ray batch every step"},
            "clocks": clk, "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu, "extras": extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_extras(args, cfg, net, ts, opt, devb, dev, extras, ms_per_step, m_valid, peak, use_graph, sc, n_rays, world):
    """Everything outside the contract line (rank 0, no collectives): encoder metric, optimizer, amortised grid refresh, the
    GPU reference baseline, the next rows.  A failure turns into a "failed: ..." string."""
    import torch
    from trinerflet_b200 import trainer
    C, R = cfg["C"], cfg["R"]
    P = 3 * C * R * R * 4

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    # ---- SURVEY.md 8d encoder metric: DENSE multilevel IDWT forward / backward, 2P / t ----
    try:
        enc = net.encoder

        def dense_fwd():
            enc.reset_cahce()
            with torch.no_grad():
                enc.get_planes()

        t_f = timed(dense_fwd)
        enc.reset_cahce()
        planes = enc.get_planes()
        gy = torch.randn_like(planes)

        def dense_bwd():
            net.zero_grad(set_to_none=True)
            torch.autograd.backward([planes], [gy], retain_graph=True)

        t_b = timed(dense_bwd)
        del planes, gy
        enc.reset_cahce()
        net.zero_grad(set_to_none=True)
        extras["encoder_dense_idwt"] = {"fwd_ms": round(t_f, 4), "fwd_GBps": round(2 * P / 1e9 / (t_f * 1e-3), 1), "fwd_hbm_frac": round(2 * P / 1e9 / (t_f * 1e-3) / peak, 4),
                                        "bwd_ms": round(t_b, 4), "bwd_GBps": round(2 * P / 1e9 / (t_b * 1e-3), 1), "bwd_hbm_frac": round(2 * P / 1e9 / (t_b * 1e-3) / peak, 4),
                                        "note": "all levels, all blocks (the path of grid-refresh steps and of inference); algorithmic bytes 2P per direction"}
    except Exception as ex:  # pragma: no cover
        extras["encoder_dense_idwt"] = f"failed: {ex}"
    # ---- optimizer (outside the metric) ----
    try:
        for fused, key in ((False, "ms_per_step_with_optimizer"), (True, "ms_per_step_with_fused_optimizer")):
            optim = trainer.make_optimizer(net, 1e-2, fused=fused)
            ts2 = trainer.TrainStep(net, opt, optimizer=optim, world_size=1)
            ts2.step(*devb[0], update_grid=False)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(3):
                ts2.step(*devb[i], update_grid=False)
            torch.cuda.synchronize()
            extras[key] = round((time.perf_counter() - t0) / 3 * 1e3, 3)
            del optim, ts2
            torch.cuda.empty_cache()
    except Exception as ex:  # pragma: no cover
        extras["ms_per_step_with_optimizer"] = f"failed: {ex}"
    # ---- every 16th step: dense planes + update_extra_state; amortised over the 16-step cycle ----
    try:
        saved = (net.density_grid.clone(), net.density_bitfield.clone(), net.mean_density, net.iter_density, net.mean_count, net.local_step)
        ts3 = trainer.TrainStep(net, opt, optimizer=None, world_size=1)
        res = {}
        for label, it in (("partial_sweep", 16), ("full_sweep", 0)):
            for rep in range(2):          # the first pass of each kind pays one-time allocations (1.6 GB dense planes + gradients): time the second
                net.density_grid.copy_(saved[0]); net.density_bitfield.copy_(saved[1])
                net.mean_density, net.iter_density = saved[2], it
                net.mark_bitfield_changed()
                net.zero_grad(set_to_none=True)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                ts3.forward_backward(*devb[0], update_grid=True)
                torch.cuda.synchronize()
                res[label] = (time.perf_counter() - t0) * 1e3
        net.density_grid.copy_(saved[0]); net.density_bitfield.copy_(saved[1])
        net.mean_density, net.iter_density, net.mean_count, net.local_step = saved[2], saved[3], saved[4], saved[5]
        net.mark_bitfield_changed()
        extras["grid_refresh_step_ms"] = {k: round(v, 3) for k, v in res.items()}
        extras["amortised_ms_per_step_incl_grid_refresh"] = round((res["partial_sweep"] + 15 * ms_per_step) / 16, 4)
        extras["amortised_note"] = ("(one dense-IDWT step with update_extra_state [2 x 128^3/2 cells, steady state] + 15 steady-state steps) / 16; the first 16 "
                                    "refreshes of a stage sweep all 2 x 128^3 cells (full_sweep)")
        del ts3
        net.zero_grad(set_to_none=True)
        torch.cuda.empty_cache()
    except Exception as ex:  # pragma: no cover
        extras["grid_refresh_step_ms"] = f"failed: {ex}"
    # ---- GPU reference baseline: reference CUDA kernels + torch library ops on this GPU ----
    if world == 1:
        try:
            r = reference_gpu_step(cfg, n_rays, devb[:4], int(m_valid), args.occupancy_radius)
            extras["reference_gpu_ms_per_step"] = round(r["ms_per_step"], 3)
            extras["reference_gpu"] = r
            torch.cuda.empty_cache()
        except Exception as ex:  # pragma: no cover
            extras["reference_gpu_ms_per_step"] = f"failed: {type(ex).__name__}: {ex}"
    if world == 1 and not args.no_next_rows:
        extras["next_rows"] = next_rows(args, net, ts, sc, n_rays, dev, use_graph)


if __name__ == "__main__":
    main()
