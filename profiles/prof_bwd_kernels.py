"""Device time per steady-state training step of the kernels of the render backward's critical path, from torch.profiler
(CUDA activities) over TNL_STEPS eager steps: the tcgen05 MLP backward (k_mlp_tc_bwd, fused with the plane scatter or not)
and the separate plane-gradient scatter (k_sample_bwd4) where the step still launches it.  Runs on any revision of the
package, so two builds can be compared kernel by kernel.  TNL_CONFIG selects the workload (default base_light).
Prints one JSON line: {kernel name: ms per step} plus the card's name."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from torch.profiler import ProfilerActivity, profile

from trinerflet_b200 import scene, trainer
from trinerflet_b200.network import NeRFNetwork

name = os.environ.get("TNL_CONFIG", "base_light")
cfg = scene.CONFIGS[name]
steps = int(os.environ.get("TNL_STEPS", "10"))
net = NeRFNetwork(bound=1.5, cuda_ray=True, density_thresh=10, min_near=0.2, triplane_channels=cfg["C"],
                  triplane_resolution=cfg["R"], triplane_wavelet_levels=cfg["S"], hidden_dim=cfg["hidden"],
                  hidden_dim_color=cfg["hidden"]).cuda()
scene.init_model_(net, 0)
scene.install_ball_occupancy(net, 0.75)
ts = trainer.TrainStep(net, trainer.default_opt(), None)
sc = scene.make_scene()
g = torch.Generator().manual_seed(0)
batches = [tuple(t.cuda() for t in scene.sample_batch(sc, cfg["rays"], g)) for _ in range(steps + 3)]
ts.forward_backward(*batches[0], update_grid=False)
net.mean_count = int(net.step_counter[0, 0].item())
net.local_step = 0
for b in batches[1:3]:      # warm-up
    net.zero_grad(set_to_none=True)
    ts.forward_backward(*b, update_grid=False)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for b in batches[3:]:
        net.zero_grad(set_to_none=True)
        ts.forward_backward(*b, update_grid=False)
    torch.cuda.synchronize()
per = {}
for ev in prof.key_averages():
    if "k_mlp_tc_bwd" in ev.key or "k_sample_bwd4" in ev.key:
        per[ev.key] = round(ev.device_time_total / 1e3 / steps, 4)
print(json.dumps({"config": name, "samples": net.mean_count, "steps": steps, "device": torch.cuda.get_device_name(0),
                  "ms_per_step": per, "sum_ms_per_step": round(sum(per.values()), 4)}))
