"""Drop-in for the reference's `raymarching` module (aux_libs/raymarching/raymarching.py:19-372):
same function names, positional signatures, defaults, dtypes and in-place semantics, implemented on the
sm_100a kernels of libtrinerflet_b200.so through the C ABI.  `renderer.py` call sites
(reconstruction/nerf/renderer.py:142,235,269,274,287,305,316,354,362,414,473,497,502,534) run unchanged.

Differences by design (DESIGN.md):
  * march_rays_train allocates sample slots with a deterministic scan in ray order, so `rays[i] = (i, off, cnt)`
    (the reference's order is an atomicAdd race, raymarching.cu:405-406);
  * kernels run on the current torch stream (the reference uses the legacy default stream);
  * extra helper `compact_rays_alive` keeps the inference loop on the device.
"""
import torch
from torch.autograd import Function
from torch.amp import custom_bwd, custom_fwd

from . import _lib
from ._lib import call, ptr, stream

_fwd32 = custom_fwd(device_type="cuda", cast_inputs=torch.float32)
_bwd = custom_bwd(device_type="cuda")


def _cuda_f32(t):
    if not t.is_cuda:
        t = t.cuda()
    return t.contiguous().float()


class _near_far_from_aabb(Function):
    @staticmethod
    @_fwd32
    def forward(ctx, rays_o, rays_d, aabb, min_near=0.2):
        """raymarching.py:22-47. rays_o/d [N,3], aabb [6] -> nears [N], fars [N]."""
        rays_o = _cuda_f32(rays_o).view(-1, 3)
        rays_d = _cuda_f32(rays_d).view(-1, 3)
        aabb = _cuda_f32(aabb)
        N = rays_o.shape[0]
        nears = torch.empty(N, dtype=rays_o.dtype, device=rays_o.device)
        fars = torch.empty(N, dtype=rays_o.dtype, device=rays_o.device)
        call("tnl_near_far_from_aabb", ptr(rays_o), ptr(rays_d), ptr(aabb), N, float(min_near), ptr(nears), ptr(fars),
             stream())
        # piecewise-constant in the rays through the box faces' min / max: no ray gradient flows through nears / fars
        ctx.mark_non_differentiable(nears, fars)
        return nears, fars


near_far_from_aabb = _near_far_from_aabb.apply


class _sph_from_ray(Function):
    @staticmethod
    @_fwd32
    def forward(ctx, rays_o, rays_d, radius):
        """raymarching.py:55-78."""
        rays_o = _cuda_f32(rays_o).view(-1, 3)
        rays_d = _cuda_f32(rays_d).view(-1, 3)
        N = rays_o.shape[0]
        coords = torch.empty(N, 2, dtype=rays_o.dtype, device=rays_o.device)
        call("tnl_sph_from_ray", ptr(rays_o), ptr(rays_d), float(radius), N, ptr(coords), stream())
        return coords


sph_from_ray = _sph_from_ray.apply


class _morton3D(Function):
    @staticmethod
    def forward(ctx, coords):
        """raymarching.py:85-102. coords [N,3] int -> indices [N] int32."""
        if not coords.is_cuda:
            coords = coords.cuda()
        coords = coords.int().contiguous()
        N = coords.shape[0]
        indices = torch.empty(N, dtype=torch.int32, device=coords.device)
        call("tnl_morton3d", ptr(coords), N, ptr(indices), stream())
        return indices


morton3D = _morton3D.apply


class _morton3D_invert(Function):
    @staticmethod
    def forward(ctx, indices):
        """raymarching.py:108-124. indices [N] int -> coords [N,3] int32."""
        if not indices.is_cuda:
            indices = indices.cuda()
        indices = indices.int().contiguous()
        N = indices.shape[0]
        coords = torch.empty(N, 3, dtype=torch.int32, device=indices.device)
        call("tnl_morton3d_invert", ptr(indices), N, ptr(coords), stream())
        return coords


morton3D_invert = _morton3D_invert.apply


class _packbits(Function):
    @staticmethod
    @_fwd32
    def forward(ctx, grid, thresh, bitfield=None):
        """raymarching.py:132-153. grid [C, H^3] fp32 -> bitfield [C*H^3/8] uint8 (bit i of byte n = grid[8n+i] > thresh)."""
        grid = _cuda_f32(grid)
        C, H3 = grid.shape[0], grid.shape[1]
        N = C * H3 // 8
        if bitfield is None:
            bitfield = torch.empty(N, dtype=torch.uint8, device=grid.device)
        call("tnl_packbits", ptr(grid), N, float(thresh), ptr(bitfield), stream())
        return bitfield


packbits = _packbits.apply


def _workspace(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


class _march_rays_train(Function):
    @staticmethod
    @_fwd32
    def forward(ctx, rays_o, rays_d, bound, density_bitfield, C, H, nears, fars, step_counter=None, mean_count=-1,
                perturb=False, align=-1, force_all_rays=False, dt_gamma=0, max_steps=1024, ray_grad=False):
        """raymarching.py:164-233. Returns xyzs [M,3], dirs [M,3], deltas [M,2], rays [N,3].
        ray_grad (set by march_rays_train): record each row's t for the ray backward."""
        shapes = (rays_o.shape, rays_d.shape)
        rays_o = _cuda_f32(rays_o).view(-1, 3)
        rays_d = _cuda_f32(rays_d).view(-1, 3)
        if not density_bitfield.is_cuda:
            density_bitfield = density_bitfield.cuda()
        density_bitfield = density_bitfield.contiguous()
        nears, fars = _cuda_f32(nears), _cuda_f32(fars)
        dev = rays_o.device
        N = rays_o.shape[0]
        M = N * max_steps
        if not force_all_rays and mean_count > 0:
            if align > 0:
                mean_count += align - mean_count % align
            M = mean_count
        if step_counter is None:
            step_counter = torch.zeros(2, dtype=torch.int32, device=dev)
        if perturb:
            noises = torch.rand(N, dtype=rays_o.dtype, device=dev)
        else:
            noises = torch.zeros(N, dtype=rays_o.dtype, device=dev)
        rays = torch.empty(N, 3, dtype=torch.int32, device=dev)
        lib = _lib.load()
        # (one float per ray and step of scratch lets the call skip the second traversal; beyond 1 GiB the plain two-pass march)
        need = lib.tnl_march_rays_train_workspace_fast(N, int(max_steps))
        ws = _workspace(need if need <= (1 << 30) else lib.tnl_march_rays_train_workspace(N), dev)

        ts = None

        def run(M_, xyzs, dirs, deltas):
            nonlocal ts
            if ray_grad:    # the same march, plus the ray parameter of every row for the backward
                ts = torch.empty(M_, dtype=torch.float32, device=dev) if M_ > 0 else None
                call("tnl_march_rays_train_ts", ptr(rays_o), ptr(rays_d), ptr(density_bitfield), float(bound), float(dt_gamma),
                     int(max_steps), N, int(C), int(H), int(M_), ptr(nears), ptr(fars), ptr(xyzs), ptr(dirs), ptr(deltas),
                     ptr(ts), ptr(rays), ptr(step_counter), ptr(noises), ptr(ws), ws.numel(), stream())
                return
            call("tnl_march_rays_train", ptr(rays_o), ptr(rays_d), ptr(density_bitfield), float(bound), float(dt_gamma),
                 int(max_steps), N, int(C), int(H), int(M_), ptr(nears), ptr(fars), ptr(xyzs), ptr(dirs), ptr(deltas),
                 ptr(rays), ptr(step_counter), ptr(noises), ptr(ws), ws.numel(), stream())

        if force_all_rays or mean_count <= 0:
            # The reference allocates N*max_steps rows (about 2 GB at N = 60k), marches, reads the count back and
            # slices (raymarching.py:205-231).  Same result without the giant buffer: count first (M = 0 writes no
            # samples), read the count (the reference syncs here too), then march into an exactly sized buffer.
            saved = step_counter.clone()
            run(0, None, None, None)
            m = int(step_counter[0].item()) - int(saved[0].item())
            step_counter.copy_(saved)
            if align > 0:
                m += align - m % align
            m = min(m, M)
            # (torch.empty: the call itself zero-fills the rows no ray owns -- same contents as the reference's zero-initialised
            #  buffers, raymarching.py:205-207, without 120 MB of memset per step)
            xyzs = torch.empty(m, 3, dtype=rays_o.dtype, device=dev)
            dirs = torch.empty(m, 3, dtype=rays_o.dtype, device=dev)
            deltas = torch.empty(m, 2, dtype=rays_o.dtype, device=dev)
            run(m, xyzs, dirs, deltas)
        else:
            xyzs = torch.empty(M, 3, dtype=rays_o.dtype, device=dev)
            dirs = torch.empty(M, 3, dtype=rays_o.dtype, device=dev)
            deltas = torch.empty(M, 2, dtype=rays_o.dtype, device=dev)
            run(M, xyzs, dirs, deltas)
        if ray_grad:
            ctx.mark_non_differentiable(deltas, rays)
            ctx.save_for_backward(rays, ts, rays_o, rays_d)
            ctx.meta = (float(bound), shapes)
        return xyzs, dirs, deltas, rays

    @staticmethod
    @_bwd
    def backward(ctx, grad_xyzs, grad_dirs, grad_deltas, grad_rays):
        rays, ts, rays_o, rays_d = ctx.saved_tensors
        bound, (shape_o, shape_d) = ctx.meta
        N, M = rays.shape[0], (ts.shape[0] if ts is not None else 0)
        g_xyz = grad_xyzs.contiguous().float() if grad_xyzs is not None else None
        g_dirs = grad_dirs.contiguous().float() if grad_dirs is not None else None
        g_o = torch.empty_like(rays_o)
        g_d = torch.empty_like(rays_d)
        # (rows no ray owns are never read, so the rows past the sample count need no n_valid here)
        call("tnl_rays_backward", ptr(rays), ptr(ts), ptr(rays_o), ptr(rays_d), bound, ptr(g_xyz), ptr(g_dirs), None, N, M,
             ptr(g_o), ptr(g_d), stream())
        return (g_o.view(shape_o) if ctx.needs_input_grad[0] else None, g_d.view(shape_d) if ctx.needs_input_grad[1] else None,
                *([None] * 14))


def march_rays_train(rays_o, rays_d, bound, density_bitfield, C, H, nears, fars, step_counter=None, mean_count=-1,
                     perturb=False, align=-1, force_all_rays=False, dt_gamma=0, max_steps=1024):
    """raymarching.py:164-233 (same positional signature).  When rays_o or rays_d requires grad and grad mode is on, xyzs and
    dirs are differentiable in the rays with every sample's ray parameter t held fixed: xyz = clamp(o + t d, -bound, bound),
    dirs = d (tnl_rays_backward); deltas and rays are not.  Otherwise the call and its outputs are exactly those of the plain
    march.  (Grad mode is read here: inside Function.forward it is always off.)"""
    ray_grad = torch.is_grad_enabled() and (rays_o.requires_grad or rays_d.requires_grad)
    return _march_rays_train.apply(rays_o, rays_d, bound, density_bitfield, C, H, nears, fars, step_counter, mean_count, perturb,
                                   align, force_all_rays, dt_gamma, max_steps, ray_grad)


class _composite_rays_train(Function):
    @staticmethod
    @_fwd32
    def forward(ctx, sigmas, rgbs, deltas, rays, T_thresh=1e-4):
        """raymarching.py:241-269. -> weights_sum [N], depth [N], image [N,3] (indexed by ray id)."""
        sigmas = sigmas.contiguous()
        rgbs = rgbs.contiguous()
        deltas = deltas.contiguous()
        rays = rays.contiguous()
        M, N = sigmas.shape[0], rays.shape[0]
        weights_sum = torch.empty(N, dtype=sigmas.dtype, device=sigmas.device)
        depth = torch.empty(N, dtype=sigmas.dtype, device=sigmas.device)
        image = torch.empty(N, 3, dtype=sigmas.dtype, device=sigmas.device)
        call("tnl_composite_rays_train_forward", ptr(sigmas), ptr(rgbs), ptr(deltas), ptr(rays), M, N, float(T_thresh),
             ptr(weights_sum), ptr(depth), ptr(image), stream())
        ctx.save_for_backward(sigmas, rgbs, deltas, rays, weights_sum, depth, image)
        ctx.dims = [M, N, T_thresh]
        return weights_sum, depth, image

    @staticmethod
    @_bwd
    def backward(ctx, grad_weights_sum, grad_depth, grad_image):
        """raymarching.py:273-288 (grad_depth is ignored, as in the reference)."""
        grad_weights_sum = grad_weights_sum.contiguous()
        grad_image = grad_image.contiguous()
        sigmas, rgbs, deltas, rays, weights_sum, depth, image = ctx.saved_tensors
        M, N, T_thresh = ctx.dims
        grad_sigmas = torch.empty_like(sigmas)      # every row is written by the call (zeros where the reference leaves its
        grad_rgbs = torch.empty_like(rgbs)          # zero-initialised buffers untouched, raymarching.py:283-284)
        call("tnl_composite_rays_train_backward", ptr(grad_weights_sum), ptr(grad_image), ptr(sigmas), ptr(rgbs),
             ptr(deltas), ptr(rays), ptr(weights_sum), ptr(image), M, N, float(T_thresh), ptr(grad_sigmas),
             ptr(grad_rgbs), stream())
        return grad_sigmas, grad_rgbs, None, None, None


composite_rays_train = _composite_rays_train.apply


class _march_rays(Function):
    @staticmethod
    @_fwd32
    def forward(ctx, n_alive, n_step, rays_alive, rays_t, rays_o, rays_d, bound, density_bitfield, C, H, near, far,
                align=-1, perturb=False, dt_gamma=0, max_steps=1024):
        """raymarching.py:300-346. -> xyzs, dirs, deltas of n_alive*n_step rows (padded up to `align`)."""
        rays_o = _cuda_f32(rays_o).view(-1, 3)
        rays_d = _cuda_f32(rays_d).view(-1, 3)
        dev = rays_o.device
        M = n_alive * n_step
        if align > 0:
            M += align - (M % align)
        xyzs = torch.zeros(M, 3, dtype=rays_o.dtype, device=dev)
        dirs = torch.zeros(M, 3, dtype=rays_o.dtype, device=dev)
        deltas = torch.zeros(M, 2, dtype=rays_o.dtype, device=dev)
        if perturb:
            noises = torch.rand(n_alive, dtype=rays_o.dtype, device=dev)
        else:
            noises = torch.zeros(n_alive, dtype=rays_o.dtype, device=dev)
        call("tnl_march_rays", int(n_alive), int(n_step), ptr(rays_alive), ptr(rays_t), ptr(rays_o), ptr(rays_d),
             float(bound), float(dt_gamma), int(max_steps), int(C), int(H), ptr(density_bitfield.contiguous()), ptr(near),
             ptr(far), ptr(xyzs), ptr(dirs), ptr(deltas), ptr(noises), stream())
        return xyzs, dirs, deltas


march_rays = _march_rays.apply


class _composite_rays(Function):
    @staticmethod
    @_fwd32
    def forward(ctx, n_alive, n_step, rays_alive, rays_t, sigmas, rgbs, deltas, weights_sum, depth, image, T_thresh=1e-2):
        """raymarching.py:354-370. In place on rays_alive, rays_t, weights_sum, depth, image."""
        call("tnl_composite_rays", int(n_alive), int(n_step), float(T_thresh), ptr(rays_alive), ptr(rays_t),
             ptr(sigmas.contiguous()), ptr(rgbs.contiguous()), ptr(deltas.contiguous()), ptr(weights_sum), ptr(depth),
             ptr(image), stream())
        return tuple()


composite_rays = _composite_rays.apply


def compact_rays_alive(rays_alive, n_alive=None):
    """Device-side equivalent of `rays_alive = rays_alive[rays_alive >= 0]` (renderer.py:364).
    Returns (compacted int32 tensor of the same capacity, count as a 1-element device tensor)."""
    n = rays_alive.shape[0] if n_alive is None else int(n_alive)
    out = torch.empty_like(rays_alive)
    cnt = torch.zeros(1, dtype=torch.int32, device=rays_alive.device)
    lib = _lib.load()
    ws = _workspace(lib.tnl_compact_alive_workspace(n), rays_alive.device)
    call("tnl_compact_alive", ptr(rays_alive), n, ptr(out), ptr(cnt), ptr(ws), ws.numel(), stream())
    return out, cnt


class DeviceRayLoop:
    """Device-driven form of the inference loop of NeRFRenderer.run_cuda (reconstruction/nerf/renderer.py:342-368; SURVEY.md
    8f-3).  n_alive, n_step = max(min(N // n_alive, 8), 1), the step budget and the alive-list compaction live in `ctrl` on
    the device (tnl_infer_plan / tnl_march_rays_dev / tnl_composite_rays_dev / tnl_compact_alive_dev), the sample buffers are
    allocated once per frame, and the host reads the state back only when `poll()` is called -- the reference (and the
    host-driven calls above) synchronise once per iteration.  Per-ray results are identical to the host-driven loop.

        loop = DeviceRayLoop(rays_o, rays_d, nears, fars, bound, bitfield, cascade, H, dt_gamma, max_steps, perturb)
        while True:
            for _ in range(chunk):
                xyzs, dirs = loop.begin_iteration()
                sigmas, rgbs = field(xyzs, dirs, n_valid=loop.n_valid)
                loop.end_iteration(sigmas, rgbs, weights_sum, depth, image, T_thresh)
            if loop.poll():
                break
    """

    def __init__(self, rays_o, rays_d, nears, fars, bound, density_bitfield, C, H, dt_gamma=0, max_steps=1024, perturb=False,
                 row_budget=0):
        self.rays_o = _cuda_f32(rays_o).view(-1, 3)
        self.rays_d = _cuda_f32(rays_d).view(-1, 3)
        dev = self.rays_o.device
        self.N = N = self.rays_o.shape[0]
        self.nears, self.fars = _cuda_f32(nears), _cuda_f32(fars)
        self.bound, self.C, self.H = float(bound), int(C), int(H)
        self.dt_gamma, self.max_steps = float(dt_gamma), int(max_steps)
        self.bitfield = density_bitfield.contiguous()
        self.ctrl = torch.tensor([0, 0, 0, 0, 0, 0, N, 0], dtype=torch.int32, device=dev)
        self.n_valid = self.ctrl[3:4]                      # n_alive * n_step of the running iteration, on the device
        self.lists = [torch.arange(N, dtype=torch.int32, device=dev), torch.empty(N, dtype=torch.int32, device=dev)]
        self.rays_t = self.nears.clone()
        # rows marched per iteration: n_alive * n_step <= budget.  The reference's budget is the N of the call (renderer.py:352:
        # n_step = max(min(N // n_alive, 8), 1)); a ray-tile shard of a frame passes the frame's ray count instead, so that it
        # marches as many samples per ray and iteration as the unsharded frame would (per-ray results do not depend on n_step)
        self.budget = B = max(N, int(row_budget))
        rows = B + 128 - B % 128                           # n_alive * n_step <= budget always; same padding rule as march_rays
        self.xyzs = torch.zeros(rows, 3, dtype=torch.float32, device=dev)
        self.dirs = torch.zeros(rows, 3, dtype=torch.float32, device=dev)
        self.deltas = torch.zeros(rows, 2, dtype=torch.float32, device=dev)
        self.noises = torch.rand(N, dtype=torch.float32, device=dev) if perturb else None   # first iteration only (renderer.py:354)
        self.ws = _workspace(_lib.load().tnl_compact_alive_workspace(N), dev)
        self.cap = N                                       # the host's upper bound of n_alive (sizes the grids)
        self.iterations_issued = 0
        self.reads = 0

    def _rows_cap(self):
        m = min(self.budget, 8 * self.cap)
        return min(m + 128 - m % 128, self.xyzs.shape[0])

    def begin_iteration(self):
        """plan + march -> views of the sample buffers the field has to evaluate (rows >= *n_valid are stale: skip them)"""
        if self.cap <= 0:
            raise RuntimeError("DeviceRayLoop: the loop has finished")
        call("tnl_infer_plan", ptr(self.ctrl), self.budget, self.max_steps, stream())
        noises = self.noises if self.iterations_issued == 0 else None
        call("tnl_march_rays_dev", ptr(self.ctrl), self.cap, ptr(self.lists[0]), ptr(self.rays_t), ptr(self.rays_o), ptr(self.rays_d),
             self.bound, self.dt_gamma, self.max_steps, self.C, self.H, ptr(self.bitfield), ptr(self.fars), ptr(self.xyzs),
             ptr(self.dirs), ptr(self.deltas), ptr(noises), stream())
        r = self._rows_cap()
        return self.xyzs[:r], self.dirs[:r]

    def end_iteration(self, sigmas, rgbs, weights_sum, depth, image, T_thresh=1e-2):
        """composite into weights_sum / depth / image (in place) and compact the alive list"""
        sigmas = sigmas.detach().float().contiguous()
        rgbs = rgbs.detach().float().contiguous()
        r = self._rows_cap()
        if sigmas.shape[0] < r or rgbs.shape[0] < r:
            raise RuntimeError("DeviceRayLoop: sigmas / rgbs must cover the rows returned by begin_iteration()")
        call("tnl_composite_rays_dev", ptr(self.ctrl), self.cap, float(T_thresh), ptr(self.lists[0]), ptr(self.rays_t), ptr(sigmas),
             ptr(rgbs), ptr(self.deltas), ptr(weights_sum), ptr(depth), ptr(image), stream())
        call("tnl_compact_alive_dev", ptr(self.ctrl), self.cap, ptr(self.lists[0]), ptr(self.lists[1]), ptr(self.ws), self.ws.numel(),
             stream())
        self.lists.reverse()
        self.iterations_issued += 1

    def poll(self):
        """read the loop state (one D2H copy + sync); tightens the grid bound; True when the loop has finished"""
        c = self.ctrl.cpu()
        self.reads += 1
        self.cap = int(c[6])
        self.iterations_done = int(c[4])
        return self.cap <= 0 or int(c[2]) >= self.max_steps
