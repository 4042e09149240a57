"""On-device step feeder (SURVEY.md 8f-2): the reference's ray generation and batch selection, call-compatible.

  get_rays(poses, intrinsics, H, W, N=-1, error_map=None, patch_size=1)
        same signature, index selection and result dict as reconstruction/nerf/utils.py:64-149; the index draws are the
        reference's own torch calls (randint / multinomial, on the poses' device), the per-ray arithmetic is
        `tnl_rays_from_ids` (csrc/rays.cu).
  RayFeeder
        shuffle_data + select_batch (utils.py:228-243) over the ray tables of NeRFDataset_all (nerf/provider.py:683-711)
        WITHOUT the tables: poses and images stay resident in HBM, an epoch is one device permutation of ray ids, a batch
        is one kernel launch that generates rays_o / rays_d and gathers the targets for a slice of it.  No host work, no
        H2D copy and no D2H read per step (the reference: CPU randperm over 64 M rays per epoch, pageable copy per step).

No CPU path: tensors must be CUDA tensors (trinerflet_b200._lib raises otherwise).
"""
import math

import torch

from . import _lib
from .parallel import shard_range


def _intr(intrinsics):
    fx, fy, cx, cy = (float(v) for v in intrinsics)
    return fx, fy, cx, cy


def rays_from_ids(poses, intrinsics, H, W, ray_ids=None, first_id=0, n=None, images=None, out=None):
    """poses [B,4,4] fp32 CUDA; ray_ids int64 [n] flat ids into the [B*H*W] table (or None: first_id .. first_id+n-1);
    images [B,H*W,C] / [B,H,W,C] fp32 (optional) -> rays_o [n,3], rays_d [n,3] (, targets [n,C]).
    out = (rays_o, rays_d[, targets]): write into these contiguous fp32 buffers (e.g. the static inputs of a captured
    CUDA graph) instead of allocating.
    When the poses require grad (and grad mode is on), rays_o / rays_d are differentiable in them
    (tnl_rays_from_ids_backward); the targets never are."""
    poses = poses.contiguous().float()
    B = poses.shape[0]
    fx, fy, cx, cy = _intr(intrinsics)
    if ray_ids is not None:
        ray_ids = ray_ids.contiguous()
        if ray_ids.dtype != torch.int64:
            ray_ids = ray_ids.long()
        n = ray_ids.numel()
    pose_grad = poses.requires_grad and torch.is_grad_enabled()
    if out is not None:
        if pose_grad:
            raise RuntimeError("rays_from_ids: `out` buffers cannot carry a pose gradient (the poses require grad)")
        for t, width in zip(out, (3, 3, images.shape[-1] if images is not None else 0)):
            if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n * width:
                raise RuntimeError("rays_from_ids: `out` buffers must be contiguous fp32 with n rows")
    if images is not None:
        if images.dtype != torch.float32 or not images.is_contiguous():
            raise RuntimeError("rays_from_ids: images must be a contiguous fp32 tensor [B,H*W,C] or [B,H,W,C]")
        if images.numel() != B * H * W * images.shape[-1]:
            raise RuntimeError("rays_from_ids: images do not match B*H*W")
    geom = (B, fx, fy, cx, cy, int(H), int(W), int(first_id), int(n))
    if pose_grad:
        return _PoseRays.apply(poses, ray_ids, images, geom)
    return _rays_from_ids(poses.detach(), ray_ids, images, geom, out)


def _rays_from_ids(poses, ray_ids, images, geom, out=None):
    B, fx, fy, cx, cy, H, W, first_id, n = geom
    if out is not None:
        rays_o, rays_d = out[0], out[1]
    else:
        rays_o = torch.empty(n, 3, device=poses.device, dtype=torch.float32)
        rays_d = torch.empty(n, 3, device=poses.device, dtype=torch.float32)
    targets, ci = None, 0
    if images is not None:
        ci = images.shape[-1]
        targets = out[2] if out is not None else torch.empty(n, ci, device=poses.device, dtype=torch.float32)
    _lib.call("tnl_rays_from_ids", _lib.ptr(poses), B, fx, fy, cx, cy, H, W, _lib.ptr(ray_ids), first_id, n,
              _lib.ptr(images), ci, _lib.ptr(rays_o), _lib.ptr(rays_d), _lib.ptr(targets), _lib.stream())
    return (rays_o, rays_d) if images is None else (rays_o, rays_d, targets)


class _PoseRays(torch.autograd.Function):
    """rays_from_ids as a function of the poses: rays_d = R dir(pix), rays_o = pose[:3,3], so
    g_pose[b][r][c] = sum over the rays of image b of g_d[r] dir[c] (c < 3), g_pose[b][r][3] = sum g_o[r], bottom row 0."""

    @staticmethod
    def forward(ctx, poses, ray_ids, images, geom):
        res = _rays_from_ids(poses, ray_ids, images, geom)
        if images is not None:
            ctx.mark_non_differentiable(res[2])
        ctx.save_for_backward(ray_ids)
        ctx.geom = geom
        return res

    @staticmethod
    def backward(ctx, g_o, *rest):
        g_d = rest[0]
        (ray_ids,) = ctx.saved_tensors
        B, fx, fy, cx, cy, H, W, first_id, n = ctx.geom
        g_o = g_o.contiguous().float() if g_o is not None else None
        g_d = g_d.contiguous().float() if g_d is not None else None
        dev = (g_o if g_o is not None else g_d).device
        g_poses = torch.empty(B, 4, 4, device=dev, dtype=torch.float32)
        _lib.call("tnl_rays_from_ids_backward", _lib.ptr(g_o), _lib.ptr(g_d), B, fx, fy, cx, cy, H, W, _lib.ptr(ray_ids),
                  first_id, n, _lib.ptr(g_poses), _lib.stream())
        return g_poses, None, None, None


@torch.amp.autocast("cuda", enabled=False)
def get_rays(poses, intrinsics, H, W, N=-1, error_map=None, patch_size=1):
    """Drop-in for reconstruction/nerf/utils.py:64-149.  Returns {'rays_o','rays_d' [B,N,3], 'inds' [B,N]
    (, 'inds_coarse')} with the reference's index selection: N<=0 all pixels; patch_size>1 random patches (:94-112);
    error_map None -> torch.randint shared by the B poses (:114-116); else multinomial on the 128x128 error map (:117-131)."""
    device = poses.device
    B = poses.shape[0]
    results = {}
    if N > 0:
        N = min(N, H * W)
        if patch_size > 1:
            num_patch = N // (patch_size ** 2)
            inds_x = torch.randint(0, H - patch_size, size=[num_patch], device=device)
            inds_y = torch.randint(0, W - patch_size, size=[num_patch], device=device)
            inds = torch.stack([inds_x, inds_y], dim=-1)
            pi, pj = torch.meshgrid(torch.arange(patch_size, device=device), torch.arange(patch_size, device=device), indexing='ij')
            offsets = torch.stack([pi.reshape(-1), pj.reshape(-1)], dim=-1)
            inds = (inds.unsqueeze(1) + offsets.unsqueeze(0)).view(-1, 2)
            inds = inds[:, 0] * W + inds[:, 1]
            inds = inds.expand([B, inds.shape[0]])
        elif error_map is None:
            inds = torch.randint(0, H * W, size=[N], device=device).expand([B, N])
        else:
            inds_coarse = torch.multinomial(error_map.to(device), N, replacement=False)
            inds_x, inds_y = inds_coarse // 128, inds_coarse % 128
            sx, sy = H / 128, W / 128
            inds_x = (inds_x * sx + torch.rand(B, N, device=device) * sx).long().clamp(max=H - 1)
            inds_y = (inds_y * sy + torch.rand(B, N, device=device) * sy).long().clamp(max=W - 1)
            inds = inds_x * W + inds_y
            results['inds_coarse'] = inds_coarse
        results['inds'] = inds
        n = inds.shape[1]
        ids = (inds + (torch.arange(B, device=device) * (H * W)).unsqueeze(1)).reshape(-1)
        rays_o, rays_d = rays_from_ids(poses, intrinsics, H, W, ray_ids=ids)
    else:
        n = H * W
        results['inds'] = torch.arange(H * W, device=device).expand([B, H * W])
        rays_o, rays_d = rays_from_ids(poses, intrinsics, H, W, first_id=0, n=B * H * W)
    results['rays_o'] = rays_o.view(B, n, 3)
    results['rays_d'] = rays_d.view(B, n, 3)
    return results


class RayFeeder:
    """Device-resident replacement of `all_data` + shuffle_data + select_batch (nerf/utils.py:228-243, :1126-1135).

        feeder = RayFeeder(poses, intrinsics, H, W, images)       # images [B,H,W,C] fp32 in HBM (or None)
        feeder.shuffle()                                          # once per epoch (reference: shuffle_data)
        for b in range(feeder.steps_per_epoch(num_rays)):
            data = feeder.select_batch(b, num_rays)               # {'rays_o','rays_d','images'} each [1,n,.]

    `select_batch` returns the rows perm[b*bs:(b+1)*bs] of the flattened ray tables, exactly what the reference's
    shuffle_data/select_batch pair yields for the same permutation (last batch ragged).  world_size/rank shard a batch
    into contiguous slices for the ray-sharded multi-GPU step (every rank draws the same permutation from `seed`)."""

    def __init__(self, poses, intrinsics, H, W, images=None, seed=None, rank=0, world_size=1):
        self.poses = poses.contiguous().float()
        _lib.ptr(self.poses)                               # raises unless the poses live on a CUDA device: there is no CPU path
        self.intrinsics = _intr(intrinsics)
        self.H, self.W = int(H), int(W)
        self.B = self.poses.shape[0]
        self.images = None
        if images is not None:
            self.images = images.to(self.poses.device, torch.float32).reshape(self.B, self.H * self.W, -1).contiguous()
        self.rank, self.world_size = rank, world_size
        self.gen = torch.Generator(device=self.poses.device)
        if seed is not None:
            self.gen.manual_seed(seed)
        self.perm = None

    @property
    def n_rays(self):
        return self.B * self.H * self.W

    def steps_per_epoch(self, batch_size):
        return math.ceil(self.n_rays / batch_size)

    def shuffle(self, perm=None):
        """draw the epoch's permutation on the device (or install a given one, e.g. the reference's, for parity tests)"""
        if perm is None:
            perm = torch.randperm(self.n_rays, device=self.poses.device, generator=self.gen)
        self.perm = perm.to(self.poses.device, torch.int64).contiguous()
        return self

    def batch_ids(self, batch_idx, batch_size):
        if self.perm is None:
            self.shuffle()
        ids = self.perm[batch_idx * batch_size:(batch_idx + 1) * batch_size]
        if self.world_size > 1:
            lo, hi = shard_range(ids.numel(), self.rank, self.world_size)
            ids = ids[lo:hi]
        return ids

    def select_batch(self, batch_idx, batch_size, out=None, poses=None):
        """poses: [B,4,4] to draw the rays from instead of the feeder's own (e.g. poses.CameraPoses()(): refined poses that
        require grad, so the batch's rays carry the pose gradient; the targets do not)"""
        ids = self.batch_ids(batch_idx, batch_size)
        if poses is not None and tuple(poses.shape) != (self.B, 4, 4):
            raise RuntimeError(f"select_batch: poses must be [{self.B},4,4], got {list(poses.shape)}")
        out = rays_from_ids(self.poses if poses is None else poses, self.intrinsics, self.H, self.W, ray_ids=ids,
                            images=self.images, out=out)
        res = {'rays_o': out[0].unsqueeze(0), 'rays_d': out[1].unsqueeze(0)}
        if self.images is not None:
            res['images'] = out[2].unsqueeze(0)
        return res

