"""NeRFRenderer -- the `--cuda_ray` renderer of reconstruction/nerf/renderer.py (run_cuda :257-381,
update_extra_state :448-542, mark_untrained_grid :383-446, render :545-577) on the trinerflet_b200 kernels.

Same constructor arguments, buffers (`aabb_train`, `aabb_infer`, `density_grid`, `density_bitfield`,
`step_counter`) and host-visible state (`mean_density`, `iter_density`, `mean_count`, `local_step`), same RNG
call sequence (torch.rand / torch.randint, so a seeded run consumes the generator exactly like the reference).
The pure-PyTorch sampler `run` (:126-254) is not used with --cuda_ray and is out of scope.
"""
import math

import numpy as np
import torch
import torch.nn as nn

from . import _lib, raymarching
from ._lib import call, ptr, stream


class NeRFRenderer(nn.Module):
    def __init__(self, bound=1, cuda_ray=False, density_scale=1, min_near=0.2, density_thresh=0.01, bg_radius=-1,
                 **kwargs):
        super().__init__()
        self.bound = bound
        self.cascade = 1 + math.ceil(math.log2(bound))
        self.grid_size = 128
        self.density_scale = density_scale
        self.min_near = min_near
        self.density_thresh = density_thresh
        self.bg_radius = bg_radius
        if bg_radius > 0:
            raise NotImplementedError("background model (bg_radius > 0) is outside the hot path: every reference config "
                                      "uses bg_radius = -1 (SURVEY.md 2.1 #3)")
        box = torch.FloatTensor([-bound, -bound, -bound, bound, bound, bound])
        self.register_buffer('aabb_train', box)
        self.register_buffer('aabb_infer', box.clone())
        self.cuda_ray = cuda_ray
        if cuda_ray:
            H3 = self.grid_size ** 3
            self.register_buffer('density_grid', torch.zeros([self.cascade, H3]))
            self.register_buffer('density_bitfield', torch.zeros(self.cascade * H3 // 8, dtype=torch.uint8))
            self.mean_density = 0
            self.iter_density = 0
            self.register_buffer('step_counter', torch.zeros(16, 2, dtype=torch.int32))
            self.mean_count = 0
            self.local_step = 0
        # bumped whenever density_bitfield changes (update_extra_state, reset_extra_state, load_state_dict, or a caller that
        # writes the buffer itself and calls mark_bitfield_changed()): everything derived from the bitfield -- the IDWT work
        # lists and the dirty-tile list of the multi-GPU exchange (trainer.TrainStep) -- is rebuilt when it lags behind
        self.bitfield_generation = 0

    def mark_bitfield_changed(self):
        self.bitfield_generation += 1

    def _load_from_state_dict(self, state_dict, prefix, *args, **kwargs):
        super()._load_from_state_dict(state_dict, prefix, *args, **kwargs)
        if prefix + "density_bitfield" in state_dict:
            self.mark_bitfield_changed()

    # subclasses provide the field --------------------------------------------------------------
    def forward(self, x, d, n_valid=None):
        raise NotImplementedError()

    def density(self, x):
        raise NotImplementedError()

    def reset_extra_state(self):
        if not self.cuda_ray:
            return
        self.density_grid.zero_()
        self.mean_density = 0
        self.iter_density = 0
        self.step_counter.zero_()
        self.mean_count = 0
        self.local_step = 0

    def run(self, *args, **kwargs):
        raise NotImplementedError("trinerflet_b200 implements the --cuda_ray path only (renderer.py:257-381)")

    # ------------------------------------------------------------------------------------------
    def _finish(self, image, depth, weights_sum, nears, fars, bg_color, prefix):
        # renderer.py:317-320 / 370-374 (depth of rays that miss the box is 0/0 = NaN there too)
        image = image + (1 - weights_sum).unsqueeze(-1) * bg_color
        depth = torch.clamp(depth - nears, min=0) / (fars - nears)
        return image.view(*prefix, 3), depth.view(*prefix)

    def run_cuda(self, rays_o, rays_d, dt_gamma=0, bg_color=None, perturb=False, force_all_rays=False, max_steps=1024,
                 T_thresh=1e-4, **kwargs):
        prefix = rays_o.shape[:-1]
        rays_o = rays_o.contiguous().view(-1, 3)
        rays_d = rays_d.contiguous().view(-1, 3)
        N = rays_o.shape[0]
        device = rays_o.device
        aabb = self.aabb_train if self.training else self.aabb_infer
        nears, fars = raymarching.near_far_from_aabb(rays_o, rays_d, aabb, self.min_near)
        if bg_color is None:
            bg_color = 1
        out = {}
        if self.training:
            counter = self.step_counter[self.local_step % 16]
            counter.zero_()
            self.local_step += 1
            xyzs, dirs, deltas, rays = raymarching.march_rays_train(
                rays_o, rays_d, self.bound, self.density_bitfield, self.cascade, self.grid_size, nears, fars, counter,
                self.mean_count, perturb, 128, force_all_rays, dt_gamma, max_steps)
            # rows >= counter[0] are zero padding no ray refers to (SURVEY.md App. A-13): the field kernels skip them
            sigmas, rgbs = self(xyzs, dirs, n_valid=counter[0:1])
            sigmas = self.density_scale * sigmas
            weights_sum, depth, image = raymarching.composite_rays_train(sigmas, rgbs, deltas, rays, T_thresh)
            image, depth = self._finish(image, depth, weights_sum, nears, fars, bg_color, prefix)
            out['weights_sum'] = weights_sum
        else:
            weights_sum = torch.zeros(N, dtype=torch.float32, device=device)
            depth = torch.zeros(N, dtype=torch.float32, device=device)
            image = torch.zeros(N, 3, dtype=torch.float32, device=device)
            chunk = int(getattr(self, "infer_chunk", 0))
            budget = max(N, int(getattr(self, "infer_row_budget", 0)))   # rows per iteration (reference: N; see DeviceRayLoop)
            if chunk > 0 and N > 0:
                # device-driven loop (SURVEY.md 8f-3): `chunk` iterations are issued per read of the loop state; sample
                # buffers live for the whole frame; identical per-ray results (opt-in: model.infer_chunk = 8)
                loop = raymarching.DeviceRayLoop(rays_o, rays_d, nears, fars, self.bound, self.density_bitfield, self.cascade,
                                                 self.grid_size, dt_gamma, max_steps, perturb, row_budget=budget)
                # every live iteration marches >= 1 sample per ray, so the loop needs at most max_steps iterations
                for _ in range(-(-int(max_steps) // chunk) + 1):
                    for _ in range(chunk):
                        xyzs, dirs = loop.begin_iteration()
                        sigmas, rgbs = self(xyzs, dirs, n_valid=loop.n_valid)
                        sigmas = self.density_scale * sigmas
                        loop.end_iteration(sigmas, rgbs, weights_sum, depth, image, T_thresh)
                    if loop.poll():
                        break
                else:
                    raise RuntimeError("device-driven inference loop did not terminate")
                self.last_infer_loop = loop
                n_alive = 0
            else:
                n_alive = N
            rays_alive = torch.arange(n_alive, dtype=torch.int32, device=device)
            rays_t = nears.clone()
            step = 0
            while step < max_steps and n_alive > 0:
                n_step = max(min(budget // n_alive, 8), 1)
                xyzs, dirs, deltas = raymarching.march_rays(
                    n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, self.bound, self.density_bitfield, self.cascade,
                    self.grid_size, nears, fars, 128, perturb if step == 0 else False, dt_gamma, max_steps)
                sigmas, rgbs = self(xyzs, dirs)
                sigmas = self.density_scale * sigmas
                raymarching.composite_rays(n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth,
                                           image, T_thresh)
                # device-side compaction; only the 4-byte count crosses to the host (the reference's boolean
                # indexing at renderer.py:364 synchronises as well and moves no less)
                rays_alive, cnt = raymarching.compact_rays_alive(rays_alive, n_alive)
                n_alive = int(cnt.item())
                rays_alive = rays_alive[:n_alive]
                step += n_step
            image, depth = self._finish(image, depth, weights_sum, nears, fars, bg_color, prefix)
            weights_sum = weights_sum.view(*prefix)
        out['depth'] = depth
        out['image'] = image
        out['weights_sum'] = weights_sum
        return out

    # ------------------------------------------------------------------------------------------
    def _all_cells(self):
        """[H^3, 3] int32 cell coordinates in the reference's meshgrid('ij') order and their Morton codes."""
        H = self.grid_size
        dev = self.density_bitfield.device
        a = torch.arange(H, dtype=torch.int32, device=dev)
        xx, yy, zz = torch.meshgrid(a, a, a, indexing='ij')
        coords = torch.stack([xx.reshape(-1), yy.reshape(-1), zz.reshape(-1)], dim=-1)
        return coords, raymarching.morton3D(coords)

    @torch.no_grad()
    def mark_untrained_grid(self, poses, intrinsic, S=64):
        """renderer.py:383-446: density_grid = -1 for cells no training camera sees."""
        if not self.cuda_ray:
            return
        if isinstance(poses, np.ndarray):
            poses = torch.from_numpy(poses)
        fx, fy, cx, cy = intrinsic
        H = self.grid_size
        count = torch.zeros_like(self.density_grid)
        poses = poses.to(count.device)
        B = poses.shape[0]
        ax = torch.arange(H, dtype=torch.int32, device=count.device).split(S)
        for xs in ax:
            for ys in ax:
                for zs in ax:
                    xx, yy, zz = torch.meshgrid(xs, ys, zs, indexing='ij')
                    coords = torch.stack([xx.reshape(-1), yy.reshape(-1), zz.reshape(-1)], dim=-1)
                    indices = raymarching.morton3D(coords).long()
                    world = (2 * coords.float() / (H - 1) - 1).unsqueeze(0)
                    for cas in range(self.cascade):
                        bound = min(2 ** cas, self.bound)
                        hgs = bound / H
                        cas_world = world * (bound - hgs)
                        for head in range(0, B, S):
                            R = poses[head:head + S, :3, :3]
                            cam = (cas_world - poses[head:head + S, :3, 3].unsqueeze(1)) @ R
                            seen = (cam[:, :, 2] > 0) \
                                & (torch.abs(cam[:, :, 0]) < cx / fx * cam[:, :, 2] + hgs * 2) \
                                & (torch.abs(cam[:, :, 1]) < cy / fy * cam[:, :, 2] + hgs * 2)
                            count[cas, indices] += seen.sum(0).reshape(-1)
        self.density_grid[count == 0] = -1
        print(f'[mark untrained grid] {(count == 0).sum()} from {H ** 3 * self.cascade}')

    def _sweep_cells(self, cas, idx32, tmp_grid):
        """Jittered cell-centre density of the Morton cells `idx32` of cascade `cas`, written to tmp_grid[cas, idx]
        (renderer.py:477-488, 507-518): positions, field query and the scatter are three launches, nothing returns to the host."""
        H = self.grid_size
        bound_c = min(2 ** cas, self.bound)
        n = idx32.shape[0]
        noise = torch.rand(n, 3, device=idx32.device, dtype=torch.float32)  # == torch.rand_like(cas_xyzs)
        xyz = torch.empty(n, 3, device=idx32.device, dtype=torch.float32)
        call("tnl_grid_cell_positions", ptr(idx32), n, H, float(bound_c), ptr(noise), ptr(xyz), stream())
        sigmas = self.density(xyz)['sigma'].reshape(-1).detach().float().contiguous()
        if _lib.deterministic():
            # duplicate cells of the partial sweep: torch's deterministic index_put_, the reference's own statement
            # (tmp_grid[cas, indices] = sigmas), instead of the kernel where one of the writers wins
            tmp_grid[cas].index_put_((idx32.long(),), sigmas * float(self.density_scale))
        else:
            call("tnl_grid_scatter", ptr(idx32), ptr(sigmas), n, float(self.density_scale), ptr(tmp_grid[cas]), stream())

    @property
    def mean_density(self):
        """renderer.py:528.  Kept on the device by update_extra_state; the float is fetched (one 4-byte read) only when somebody
        looks at it -- the reference reads it back inside every update."""
        t = self.__dict__.get("_mean_density_t")
        if t is not None:
            self.__dict__["_mean_density"] = float(t.item())
            self.__dict__["_mean_density_t"] = None
        return self.__dict__.get("_mean_density", 0)

    @mean_density.setter
    def mean_density(self, v):
        self.__dict__["_mean_density"] = v
        self.__dict__["_mean_density_t"] = None

    @torch.no_grad()
    def update_extra_state(self, decay=0.95, S=128):
        """renderer.py:448-542 with the same RNG call sequence (torch.rand / torch.randint draws, in the reference's order, so a
        seeded run consumes the generator identically) and ONE host synchronisation: the two data-dependent integers the
        reference's own control flow needs on the host -- the occupied-cell counts that bound `torch.randint` in the partial
        sweep (:500-501) and the sample-count average `mean_count` (:538-539) -- are fetched together up front.  The threshold
        (mean density) stays on the device: EMA-max + mean + packbits are two kernels (tnl_grid_ema_update_sum,
        tnl_packbits_mean)."""
        if not self.cuda_ray:
            return
        H = self.grid_size
        dev = self.density_bitfield.device
        total_step = min(16, self.local_step)
        partial = self.iter_density >= 16
        # ---- the one read-back: [occupied cells per cascade (partial sweep only), sum of the step counters] ----
        head = []
        if partial:
            occ_mask = self.density_grid > 0
            head.append(occ_mask.sum(dim=1).to(torch.int64))
        if total_step > 0:
            head.append(self.step_counter[:total_step, 0].sum().to(torch.int64).reshape(1))
        host = torch.cat(head).tolist() if head else []
        n_occ = host[:self.cascade] if partial else None
        tmp_grid = torch.full_like(self.density_grid, -1.0)
        if not partial:  # full sweep: every cell of every cascade, in the reference's meshgrid('ij') order
            cells = self.__dict__.get("_cells_cache")
            if cells is None or cells.device != dev:
                cells = self._all_cells()[1].int().contiguous()
                self.__dict__["_cells_cache"] = cells
            for cas in range(self.cascade):
                self._sweep_cells(cas, cells, tmp_grid)
        else:  # H^3/4 uniform cells + H^3/4 cells drawn from the occupied set, per cascade
            N = H ** 3 // 4
            for cas in range(self.cascade):
                coords = torch.randint(0, H, (N, 3), device=dev)
                indices = raymarching.morton3D(coords)
                if n_occ[cas] > 0:
                    occ = torch.nonzero_static(occ_mask[cas], size=int(n_occ[cas])).squeeze(-1)
                    pick = torch.randint(0, int(n_occ[cas]), [N], dtype=torch.long, device=dev)
                    indices = torch.cat([indices.long(), occ[pick]], dim=0)
                self._sweep_cells(cas, indices.int().contiguous(), tmp_grid)
        flat = self.density_grid.view(-1)
        acc = torch.empty(1, dtype=torch.float64, device=dev)
        mean_t = torch.empty(1, dtype=torch.float32, device=dev)
        call("tnl_grid_ema_update_sum", ptr(flat), ptr(tmp_grid.view(-1)), flat.numel(), float(decay), ptr(acc), stream())
        if _lib.deterministic():   # the kernel's sum adds one double atomic per block: torch's deterministic reduction instead
            acc.copy_(torch.clamp(flat, min=0).sum(dtype=torch.float64).reshape(1))
        self.iter_density += 1
        call("tnl_packbits_mean", ptr(flat), flat.numel(), ptr(acc), float(self.density_thresh), ptr(mean_t), ptr(self.density_bitfield),
             stream())
        self.__dict__["_mean_density_t"] = mean_t
        self.mark_bitfield_changed()
        if total_step > 0:
            self.mean_count = int(host[-1] / total_step)
        self.local_step = 0

    def render(self, rays_o, rays_d, staged=False, max_ray_batch=4096, **kwargs):
        if not self.cuda_ray:
            raise NotImplementedError("trinerflet_b200 implements the --cuda_ray path only")
        return self.run_cuda(rays_o, rays_d, **kwargs)  # never staged with cuda_ray (renderer.py:557-576)
