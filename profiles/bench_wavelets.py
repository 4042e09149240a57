"""Per-wavelet cost of the tri-plane reconstruction at the base-light geometry (C = 32, 64^2 -> 2048^2, 5 levels), for every
wavelet of the reference's pad table (bior6.8, haar, bior2.2, bior2.6, bior4.4).  One run on one GPU, CUDA events:

  * dense IDWT level kernels: forward and backward (with the fused regulariser gradient, as the training step issues it) per
    level and in total; algorithmic bytes 2P per level (P = 3*C*(2n)^2*4, read the level's coefficients + write its planes,
    bench.py's count) over kernel time, against the HBM3e data-sheet rate of the B200 (7.7 TB/s).  The levels up to 512^2
    fit in the 126 MB L2 after the first pass; the two top levels (1.6 GB / 400 MB of output) do not;
  * the base-light training step (60 000 rays, ball occupancy of radius 0.75, fp16 autocast, work-list IDWT) through
    TrainStep graph replay, the wavelets alternated round by round so that drift of the shared machine spreads over all.

The card's name, power limit and max SM clock are read in the same run and written next to the numbers.
    python profiles/bench_wavelets.py [--out profiles/r03_bench_wavelets.json] [--steps 20] [--rounds 3]"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

WAVES = ["bior6.8", "haar", "bior2.2", "bior2.6", "bior4.4"]
HBM_PEAK_GBS = 7700.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q)


def events_ms(fn, reps, warm=3):
    for _ in range(warm):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def level_times(wave, C=32, n0=64, levels=5, reps=20):
    from trinerflet_b200._lib import ptr, stream
    from trinerflet_b200.idwt_plan import idwt_call
    from trinerflet_b200.triplane_encoder import cl_empty_coefs, cl_empty_planes
    g1 = torch.ones(1, device="cuda")
    rows = []
    for l in range(levels):
        n = n0 * 2 ** l
        x = cl_empty_planes(C, n, device="cuda").normal_()
        yh = cl_empty_coefs(C, n, device="cuda").normal_()
        out = cl_empty_planes(C, 2 * n, device="cuda")
        asum = torch.zeros(1, device="cuda")
        gx, gyh = cl_empty_planes(C, n, device="cuda"), cl_empty_coefs(C, n, device="cuda")
        fwd = events_ms(lambda: idwt_call("tnl_idwt_level_forward", wave, ptr(x), ptr(yh), ptr(out), n, C, ptr(asum), stream()), reps)
        bwd = events_ms(lambda: idwt_call("tnl_idwt_level_backward", wave, ptr(out), ptr(gx), ptr(gyh), n, C, ptr(yh), ptr(g1), 1.0, 0, 3,
                                          stream()), reps)
        two_p = 2 * 3 * C * (2 * n) ** 2 * 4
        rows.append(dict(n=n, out=2 * n, fwd_ms=fwd, bwd_ms=bwd, fwd_GBps=two_p / fwd / 1e6, bwd_GBps=two_p / bwd / 1e6,
                         fwd_frac_hbm_peak=two_p / fwd / 1e6 / HBM_PEAK_GBS, bwd_frac_hbm_peak=two_p / bwd / 1e6 / HBM_PEAK_GBS))
        del x, yh, out, gx, gyh
    two_p_all = sum(2 * 3 * C * (2 * r["n"]) ** 2 * 4 for r in rows)
    fwd_t, bwd_t = sum(r["fwd_ms"] for r in rows), sum(r["bwd_ms"] for r in rows)
    return dict(levels=rows, fwd_total_ms=fwd_t, bwd_total_ms=bwd_t, fwd_total_GBps=two_p_all / fwd_t / 1e6,
                bwd_total_GBps=two_p_all / bwd_t / 1e6, fwd_total_frac_hbm_peak=two_p_all / fwd_t / 1e6 / HBM_PEAK_GBS,
                bwd_total_frac_hbm_peak=two_p_all / bwd_t / 1e6 / HBM_PEAK_GBS)


def make_step(wave, cfg, n_rays, batches):
    from trinerflet_b200 import scene, trainer
    from trinerflet_b200.network import NeRFNetwork
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=cfg["C"], triplane_resolution=cfg["R"],
                      triplane_wavelet_levels=cfg["S"], hidden_dim=cfg["hidden"], hidden_dim_color=cfg["hidden"],
                      wavelet_type=wave).cuda()
    scene.init_model_(net, seed=0)
    scene.install_ball_occupancy(net, 0.75)
    ts = trainer.TrainStep(net, trainer.default_opt(), optimizer=None, world_size=1)
    net.train()
    torch.manual_seed(100)
    ts.forward_backward(*batches[-1], update_grid=False)
    net.mean_count = int(net.step_counter[0, 0].item())     # steady state, as bench.py establishes it
    net.local_step = 0
    ts.capture(*batches[-2], warmup=0)
    return net, ts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "r03_bench_wavelets.json"))
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_wavelets: needs a CUDA device (no CPU measurement)")
    from trinerflet_b200 import _lib, scene
    _lib.load()
    res = dict(card=card(), geometry="base_light: C=32, 64^2 -> 2048^2 (5 levels), 60000 rays, ball occupancy r=0.75",
               hbm_peak_GBps_datasheet=HBM_PEAK_GBS, idwt_dense={}, train_step={})
    for wave in WAVES:
        res["idwt_dense"][wave] = level_times(wave, reps=args.reps)
        print(wave, "idwt fwd %.3f ms bwd %.3f ms" % (res["idwt_dense"][wave]["fwd_total_ms"], res["idwt_dense"][wave]["bwd_total_ms"]),
              flush=True)
    cfg = scene.CONFIGS["base_light"]
    n_rays = cfg["rays"]
    sc = scene.make_scene()
    gen = torch.Generator().manual_seed(1234)
    batches = [tuple(t.cuda() for t in scene.sample_batch(sc, n_rays, gen)) for _ in range(args.warmup + args.steps + 2)]
    steps = {w: make_step(w, cfg, n_rays, batches) for w in WAVES}
    times = {w: [] for w in WAVES}
    for r in range(args.rounds):
        for wave in (WAVES if r % 2 == 0 else WAVES[::-1]):
            net, ts = steps[wave]
            for i in range(args.warmup):
                ts.replay(*batches[i])
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                loss = ts.replay(*batches[args.warmup + i])
            e1.record()
            torch.cuda.synchronize()
            times[wave].append(e0.elapsed_time(e1) / args.steps)
            assert torch.isfinite(torch.as_tensor(float(loss)))
    for wave in WAVES:
        t = sorted(times[wave])
        res["train_step"][wave] = dict(ms_per_step_rounds=times[wave], ms_per_step_median=t[len(t) // 2],
                                       rays_per_s_median=n_rays / (t[len(t) // 2] * 1e-3), samples_per_step=int(steps[wave][0].mean_count))
        print(wave, "train step %.3f ms (rounds %s)" % (t[len(t) // 2], ", ".join("%.3f" % v for v in times[wave])), flush=True)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(card=res["card"], out=args.out)))


if __name__ == "__main__":
    main()
