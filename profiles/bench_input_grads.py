"""Cost of the input-gradient paths on one GPU, CUDA events, the variants alternated round by round:

  * the fused MLP backward with and without the direction gradient (tnl_mlp_backward_dirs vs tnl_mlp_backward), 64-wide heads
    (C = 32) and 128-wide heads (C = 48), M = 3.8 M samples, fp16 feature stream;
  * the position gradient of the plane gather at the base-light geometry (C = 32, R = 2048, 3.8 M samples in a ball of radius
    0.75 * bound, visited in cell order, fp16 feature gradient, fp16 coordinates): the plane scatter alone
    (tnl_sample_planes_backward), the position gradient alone (tnl_sample_planes_backward_xyz), and the two launched back to back
    as _SamplePlanes.backward issues them when both gradients are needed.

The card's name, power limit and max SM clock are read in the same run and written next to the numbers.
    python profiles/bench_input_grads.py [--out profiles/r04_bench_input_grads.json] [--reps 20] [--rounds 3]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

M = 3_800_000
BOUND = 1.5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q)


def events_ms(fn, reps):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def points(g):
    x = torch.randn(M, 3, generator=g)
    x = x / x.norm(dim=-1, keepdim=True) * torch.rand(M, 1, generator=g) ** (1 / 3) * 0.75 * BOUND
    d = torch.randn(M, 3, generator=g)
    return x.cuda(), (d / d.norm(dim=-1, keepdim=True)).cuda()


def mlp_cases(g, x, d):
    from oracle import field as of
    from trinerflet_b200._lib import MlpDims, call, ptr, stream
    from trinerflet_b200.network import pack_mlp_weights
    cases = {}
    for C, H in ((32, 64), (48, 128)):
        W = [w.cuda() for w in of.init_mlp_weights(C, H, H, gen=g)]
        dims = MlpDims(3 * C, H, H)
        packed = pack_mlp_weights(dims, W)
        feat = (0.5 * torch.randn(M, 3 * C, generator=g)).half().cuda()
        gs, grgb = torch.randn(M, device="cuda"), torch.randn(M, 3, device="cuda")
        g_feat = torch.empty_like(feat)
        gW = [torch.zeros_like(w) for w in W]
        g_dirs = torch.empty(M, 3, device="cuda")
        args = (ctypes.byref(dims), ptr(packed), ptr(feat), 1, ptr(d), M, None, ptr(gs), ptr(grgb), ptr(g_feat), *[ptr(w) for w in gW])
        cases[f"mlp_backward_H{H}_C{C}"] = lambda a=args: call("tnl_mlp_backward", *a, stream())
        cases[f"mlp_backward_dirs_H{H}_C{C}"] = lambda a=args, gd=g_dirs: call("tnl_mlp_backward_dirs", *a, ptr(gd), stream())
    return cases


def sample_cases(g, x):
    from trinerflet_b200._lib import call, ptr, stream
    from trinerflet_b200.triplane_encoder import _inv_bound, cell_sort, cl_empty_planes
    C, R = 32, 2048
    planes = cl_empty_planes(C, R, device="cuda").normal_()
    g_planes = cl_empty_planes(C, R, device="cuda", zero=True)
    perm = cell_sort(x, BOUND)
    g_feat = torch.randn(M, 3 * C, generator=g).half().cuda()
    g_xyz = torch.empty(M, 3, device="cuda")
    inv = _inv_bound(BOUND)
    scatter = lambda: call("tnl_sample_planes_backward", ptr(g_feat), 1, ptr(x), M, R, C, inv, 1, None, ptr(perm), ptr(g_planes), stream())   # noqa: E731
    xyz = lambda: call("tnl_sample_planes_backward_xyz", ptr(g_feat), 1, ptr(planes), ptr(x), M, R, C, inv, 1, None, ptr(perm), ptr(g_xyz),  # noqa: E731
                       stream())
    return {"sample_scatter": scatter, "sample_xyz": xyz, "sample_scatter_then_xyz": lambda: (scatter(), xyz())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r04_bench_input_grads.json")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    g = torch.Generator().manual_seed(0)
    x, d = points(g)
    cases = {**mlp_cases(g, x, d), **sample_cases(g, x)}
    res = {k: [] for k in cases}
    for _ in range(a.rounds):
        for k, fn in cases.items():
            res[k].append(round(events_ms(fn, a.reps), 4))
    out = dict(card=card(), M=M, reps=a.reps, rounds=a.rounds, ms=res, ms_min={k: min(v) for k, v in res.items()})
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
