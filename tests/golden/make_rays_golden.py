"""Generates tests/golden/rays_ref.npz by importing the REFERENCE's own get_rays / shuffle_data / select_batch from
/root/reference/reconstruction/nerf/utils.py (read-only) and running them on the CPU in fp32.  Build container only.

    python tests/golden/make_rays_golden.py

UI / IO imports of nerf/utils.py (cv2, trimesh, lpips, ...) are replaced by inert stubs exactly as in make_golden.py;
the three functions under test are the reference's real code.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import make_golden  # noqa: E402
from trinerflet_b200 import scene  # noqa: E402


def main():
    make_golden._install_stubs()
    sys.path.insert(0, make_golden.require_reference(make_golden.REF))
    from nerf.utils import get_rays, shuffle_data, select_batch

    out = {}
    # ---- case A: Blender-shaped intrinsics (800x800), 5 poses, explicit random pixel subset + corner pixels --------------
    sc = scene.make_scene(seed=0)
    poses = sc.poses[:5].contiguous()
    intr = np.array(sc.intrinsics, np.float64)             # provider.py:681 keeps a float64 numpy array
    H = W = 800
    torch.manual_seed(7)
    full = get_rays(poses, intr, H, W, -1)                 # all pixels
    g = torch.Generator().manual_seed(7)
    pick = torch.cat([torch.tensor([0, W - 1, (H - 1) * W, H * W - 1, 400 * W + 400]),
                      torch.randint(0, H * W, (2043,), generator=g)])
    out.update(A_poses=poses.numpy(), A_intr=intr, A_H=H, A_W=W, A_inds=pick.numpy(),
               A_rays_o=full['rays_o'][:, pick].numpy(), A_rays_d=full['rays_d'][:, pick].numpy())
    assert torch.equal(full['inds'][0], torch.arange(H * W))

    # ---- case B: non-square small images (H=37, W=53), fx != fy, off-centre principal point, B=4, N random (utils.py:118)
    H, W = 37, 53
    intr_b = np.array([61.25, 58.5, 25.75, 19.125], np.float64)
    poses_b = scene.make_poses(4, seed=3)
    torch.manual_seed(11)
    sub = get_rays(poses_b, intr_b, H, W, 257)             # torch.randint indices, shared by the B poses
    full_b = get_rays(poses_b, intr_b, H, W, -1)
    out.update(B_poses=poses_b.numpy(), B_intr=intr_b, B_H=H, B_W=W, B_inds=sub['inds'].numpy(),
               B_rays_o=sub['rays_o'].numpy(), B_rays_d=sub['rays_d'].numpy(),
               B_full_o=full_b['rays_o'].numpy(), B_full_d=full_b['rays_d'].numpy())

    # ---- case C: the step feeder: all rays + images -> shuffle_data -> select_batch (first, middle and ragged last batch)
    images = torch.rand(4, H * W, 4, generator=g)
    all_data = dict(rays_o=full_b['rays_o'].clone(), rays_d=full_b['rays_d'].clone(), images=images.clone())
    torch.manual_seed(13)
    shuffled = shuffle_data(all_data)
    torch.manual_seed(13)
    perm = torch.randperm(4 * H * W)                       # the permutation shuffle_data drew (utils.py:230)
    assert torch.equal(shuffled['images'], images.view(-1, 4)[perm])
    bs = 1000
    out.update(C_images=images.numpy(), C_perm=perm.numpy(), C_bs=bs)
    for b in (0, 3, (4 * H * W) // bs):
        sel = select_batch(shuffled, b, bs, 'cpu')
        out[f"C_b{b}_rays_o"] = sel['rays_o'][0].numpy()
        out[f"C_b{b}_rays_d"] = sel['rays_d'][0].numpy()
        out[f"C_b{b}_images"] = sel['images'][0].numpy()
    np.savez_compressed(os.path.join(HERE, "rays_ref.npz"), **out)
    print("rays_ref.npz:", {k: v.shape for k, v in out.items() if hasattr(v, 'shape') and v.ndim})


if __name__ == "__main__":
    main()
