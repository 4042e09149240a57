"""Cost of camera pose refinement on one GPU, base_light: ms per eager training step (RayFeeder.select_batch + TrainStep.step with
FusedAdam) without and with pose refinement (rays drawn from CameraPoses() so that they require grad), the two alternated round
by round, CUDA events around `--steps` steady-state steps, medians over `--rounds`.  Then the two new backward kernels at the
step's own sizes (CUDA events around each ABI call of a profiled refinement step), and tnl_rays_from_ids_backward for B = 100
and B = 1000 images.  tnl_rays_backward reads ts + g_xyz + g_dirs = 28 B per sample (plus 24 B per ray and the ray table); the
rate below is those bytes over its time.

The card's name, power limit and max SM clock are read in the same run and written next to the numbers.
    python profiles/bench_pose_refine.py [--out profiles/r07_bench_pose_refine.json] [--steps 10] [--rounds 3]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q)


def setup(cfg):
    from trinerflet_b200 import rays, scene, trainer
    from trinerflet_b200.network import NeRFNetwork
    from trinerflet_b200.optim import FusedAdam
    from trinerflet_b200.poses import CameraPoses
    c = scene.CONFIGS[cfg]
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=c["C"],
                      triplane_resolution=c["R"], triplane_wavelet_levels=c["S"], hidden_dim=c["hidden"],
                      hidden_dim_color=c["hidden"]).cuda()
    scene.init_model_(net, seed=0)
    scene.install_ball_occupancy(net, 0.75)
    sc = scene.make_scene()
    poses = sc.poses.cuda()
    images = torch.rand(poses.shape[0], scene.H_IMG, scene.W_IMG, 3, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    feeder = rays.RayFeeder(poses, sc.intrinsics, scene.H_IMG, scene.W_IMG, images, seed=0)
    cams = CameraPoses(poses)
    opt = FusedAdam(net.get_params(1e-2) + cams.get_params(1e-4), betas=(0.9, 0.99), eps=1e-15)
    ts = trainer.TrainStep(net, trainer.default_opt(), opt, world_size=1)
    return ts, feeder, cams, c["rays"]


def one_step(ts, feeder, cams, bs, b, refine):
    data = feeder.select_batch(b % feeder.steps_per_epoch(bs), bs, poses=cams() if refine else None)
    ts.step(data['rays_o'][0], data['rays_d'][0], data['images'][0], update_grid=False)


def timed(ts, feeder, cams, bs, steps, refine):
    for b in range(2):
        one_step(ts, feeder, cams, bs, b, refine)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for b in range(steps):
        one_step(ts, feeder, cams, bs, b, refine)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def kernel_times(ts, feeder, cams, bs, reps=5):
    from trinerflet_b200 import _lib
    rec = {}
    for b in range(reps):
        _lib.profile_start()
        one_step(ts, feeder, cams, bs, b, True)
        for name, v in _lib.profile_stop().items():
            rec.setdefault(name, []).extend(v)
    med = lambda xs: sorted(xs)[len(xs) // 2]   # noqa: E731
    rb = rec["tnl_rays_backward"]
    N, M = rb[0][1][1], rb[0][1][2]
    t_rb = med([ms for ms, _ in rb])
    byt = 28 * M + (24 + 24 + 12) * N
    out = dict(N=N, M=M, tnl_rays_backward_ms=t_rb, tnl_rays_backward_bytes=byt, tnl_rays_backward_GBps=byt / t_rb / 1e6,
               tnl_rays_from_ids_backward_ms_B100=med([ms for ms, _ in rec["tnl_rays_from_ids_backward"]]),
               march_train_ts_ms=med([ms for ms, _ in rec["tnl_march_rays_train_ts"]]))
    return out


def pose_bwd_B(B, n, reps=50):
    from trinerflet_b200 import _lib
    g = torch.Generator(device="cuda").manual_seed(B)
    ids = torch.randint(0, B * 800 * 800, (n,), device="cuda", generator=g)
    go, gd = torch.randn(n, 3, device="cuda", generator=g), torch.randn(n, 3, device="cuda", generator=g)
    gP = torch.empty(B, 4, 4, device="cuda")

    def run():
        _lib.call("tnl_rays_from_ids_backward", _lib.ptr(go), _lib.ptr(gd), B, 1111.0, 1111.0, 400.0, 400.0, 800, 800, _lib.ptr(ids),
                  0, n, _lib.ptr(gP), _lib.stream())
    for _ in range(3):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--config", default="base_light")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    res = dict(card=card(), config=a.config, steps=a.steps, rounds=a.rounds)
    ts, feeder, cams, bs = setup(a.config)
    off, on = [], []
    for _ in range(a.rounds):
        off.append(timed(ts, feeder, cams, bs, a.steps, False))
        on.append(timed(ts, feeder, cams, bs, a.steps, True))
    med = lambda xs: sorted(xs)[len(xs) // 2]   # noqa: E731
    res.update(rays_per_step=bs, ms_per_step_default=off, ms_per_step_pose_refine=on, median_default=med(off),
               median_pose_refine=med(on), ratio_of_medians=med(on) / med(off))
    res["kernels"] = kernel_times(ts, feeder, cams, bs)
    res["kernels"]["tnl_rays_from_ids_backward_ms_synthetic"] = {f"B={B}": pose_bwd_B(B, bs) for B in (100, 1000)}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
