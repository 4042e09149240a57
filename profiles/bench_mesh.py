"""Times mesh extraction (trinerflet_b200.mesh) for the base-light model at 256^3 and 512^3, and the marching cubes alone at
1024^3; prints and writes one JSON document.

  sweep_ms          extract_fields: density() under fp16 autocast over the lattice in 128^3 chunks into a device volume
  mc_ms             marching_cubes on that volume, outputs copied to the host as numpy arrays (what a caller receives);
                    mc_count_ms / mc_emit_ms are the two ABI calls alone (CUDA events)
  extract_geometry_ms  the whole extract_geometry call
  reference_shaped_ms  the reference's path restated here: the chunked sweep with a .cpu() per chunk, then the numpy
                    marching cubes of oracle/mesh.py on the CPU (our restatement, not mcubes, which is not available)

Timings are medians over --reps runs after one warm-up run; every timed region ends in a device synchronisation.  The
threshold is the median of the 256^3 volume (the random-init field has no natural level), the same at every resolution.

    python profiles/bench_mesh.py [--reps 5] [--out r06_bench_mesh.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def _gpu():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = (s.strip() for s in out.split(","))
    except Exception as ex:  # pragma: no cover
        name, power = torch.cuda.get_device_name(0), f"unknown ({ex})"
    return {"gpu": name, "power_limit": power}


def _timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), out


def _abi_ms(u, thr):
    from trinerflet_b200 import _lib, mesh
    _lib.profile_start()
    mesh.marching_cubes(u, thr)
    rec = _lib.profile_stop()
    return rec["tnl_mc_count"][0][0], rec["tnl_mc_emit"][0][0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--config", default="base_light")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_mesh.py times the GPU path: it needs a CUDA device"
    from oracle import mesh as om
    from trinerflet_b200 import mesh, scene
    from trinerflet_b200.network import NeRFNetwork
    c = scene.CONFIGS[args.config]
    net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=c["C"], triplane_resolution=c["R"],
                      triplane_wavelet_levels=c["S"], hidden_dim=c["hidden"], hidden_dim_color=c["hidden"]).cuda()
    scene.init_model_(net, seed=0)
    net.eval()
    bmin, bmax = net.aabb_infer[:3], net.aabb_infer[3:]

    def query(pts):
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            return net.density(pts.to("cuda"))["sigma"]

    res = {"config": args.config, **_gpu(), "reps": args.reps, "rows": []}
    thr = None
    for n in (256, 512):
        sweep_ms, u = _timed(lambda: mesh.extract_fields(bmin, bmax, n, query), args.reps)
        if thr is None:
            thr = float(u.float().median())
            res["threshold"] = thr
        mc_ms, (v, t) = _timed(lambda: mesh.marching_cubes(u, thr), args.reps)
        count_ms, emit_ms = _abi_ms(u, thr)
        e2e_ms, _ = _timed(lambda: mesh.extract_geometry(bmin, bmax, n, thr, query), args.reps)
        row = {"resolution": n, "vertices": int(v.shape[0]), "triangles": int(t.shape[0]), "sweep_ms": sweep_ms, "mc_ms": mc_ms,
               "mc_count_ms": count_ms, "mc_emit_ms": emit_ms, "extract_geometry_ms": e2e_ms}
        if n == 256:
            t0 = time.perf_counter()
            u_host = om.extract_fields(bmin, bmax, n, query)
            t1 = time.perf_counter()
            om.marching_cubes(u_host, thr)
            t2 = time.perf_counter()
            row.update(reference_shaped_sweep_ms=(t1 - t0) * 1e3, reference_shaped_numpy_mc_ms=(t2 - t1) * 1e3,
                       reference_shaped_ms=(t2 - t0) * 1e3, reference_shaped_runs=1)
        else:
            row.update(reference_shaped_ms="not measured")
        del u
        res["rows"].append(row)
        print(json.dumps(row), flush=True)
    # marching cubes alone at 1024^3 on an analytic ball generated on the device (a base-light sweep at 1024^3 is not timed)
    n, r = 1024, 400.0
    a = torch.arange(n, device="cuda", dtype=torch.float32) - (n - 1) / 2 - 0.137
    u = r - torch.sqrt(a[:, None, None] ** 2 + a[None, :, None] ** 2 + a[None, None, :] ** 2)
    mc_ms, (v, t) = _timed(lambda: mesh.marching_cubes(u, 0.0), args.reps)
    count_ms, emit_ms = _abi_ms(u, 0.0)
    row = {"resolution": 1024, "volume": "analytic ball r=400", "vertices": int(v.shape[0]), "triangles": int(t.shape[0]),
           "sweep_ms": "not measured", "mc_ms": mc_ms, "mc_count_ms": count_ms, "mc_emit_ms": emit_ms,
           "extract_geometry_ms": "not measured", "reference_shaped_ms": "not measured"}
    res["rows"].append(row)
    print(json.dumps(row), flush=True)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
