"""Cost of torch.use_deterministic_algorithms(True) on one GPU: ms per training step (TrainStep.step: forward, backward,
FusedAdam) with the flag off and on, at the small, base_light and large configs, the two modes alternated round by round
(three rounds of each by default), CUDA events around `--steps` steady-state steps of the same batch size.

What the mode costs is all in these numbers: the fixed-point scatter (four 64-bit REDs per corner instead of one vector RED,
plus its scale, zero and convert passes), the unfused _SamplePlanes + _FieldMLP path (no scatter inside the MLP backward), the
slot reduction of the weight gradients, torch's deterministic reductions, and torch's NaN fill of fresh allocations.

The card's name, power limit and max SM clock are read in the same run and written next to the numbers.
    python profiles/bench_deterministic.py [--out profiles/r05_bench_deterministic.json] [--steps 10] [--rounds 3]"""
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


def make_step(cfg):
    from trinerflet_b200 import scene, trainer
    from trinerflet_b200.network import NeRFNetwork
    c = scene.CONFIGS[cfg]
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=c["C"],
                      triplane_resolution=c["R"], triplane_wavelet_levels=c["S"], hidden_dim=c["hidden"],
                      hidden_dim_color=c["hidden"]).cuda()
    scene.init_model_(net, seed=0)
    scene.install_ball_occupancy(net, 0.75)
    ts = trainer.TrainStep(net, trainer.default_opt(), trainer.make_optimizer(net, 1e-2, fused=True), world_size=1)
    sc = scene.make_scene()
    batch = tuple(t.cuda() for t in scene.sample_batch(sc, c["rays"], torch.Generator().manual_seed(1)))
    return ts, batch


def timed(ts, batch, steps, det):
    torch.use_deterministic_algorithms(det)
    for _ in range(2):                      # warm-up of this mode's kernels and allocations
        ts.step(*batch, update_grid=False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        ts.step(*batch, update_grid=False)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--configs", default="small,base_light,large")
    a = ap.parse_args()
    from trinerflet_b200 import _lib
    prev = torch.are_deterministic_algorithms_enabled()
    res = dict(card=card(), steps=a.steps, rounds=a.rounds, configs={})
    try:
        for cfg in a.configs.split(","):
            ts, batch = make_step(cfg)
            off, on = [], []
            for _ in range(a.rounds):
                off.append(timed(ts, batch, a.steps, False))
                on.append(timed(ts, batch, a.steps, True))
            res["configs"][cfg] = dict(ms_per_step_off=off, ms_per_step_on=on,
                                       ratio_of_medians=sorted(on)[len(on) // 2] / sorted(off)[len(off) // 2])
            print(cfg, json.dumps(res["configs"][cfg]), flush=True)
            del ts, batch
            _lib._workspaces.clear()
            torch.cuda.empty_cache()
    finally:
        torch.use_deterministic_algorithms(prev)
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
