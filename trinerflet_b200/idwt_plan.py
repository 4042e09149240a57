"""Work lists for the plane reconstruction on the training hot path.

During training the feature planes are only sampled -- and only receive gradient -- inside the texel tiles that the
occupancy grid marks (`tnl_mark_dirty_tiles`, the same tile set the multi-GPU gradient exchange uses).  The reference
reconstructs and differentiates the full planes every step (pytorch_wavelets is dense); here the multilevel IDWT and its
adjoint run over per-level lists of blocks instead (tnl_idwt_level_forward_sparse / _backward_sparse):

  forward   level l reconstructs a block iff its output is read later: at the top level the dirty tiles themselves,
            below it every block whose output lies in the (4-pixel) input halo of an active block one level up;
  backward  level l processes a block iff the incoming gradient can be non-zero on its (8-pixel) input halo; all other
            blocks get g_x = 0 and g_yh = (regulariser gradient only) from a streaming pass.

The parts of the returned planes that belong to inactive blocks are NOT written; this is only valid for consumers that
stay inside the marked tiles (the ray-marched sampler of a training step).  Anything that reads the planes elsewhere
(density-grid refresh, inference outside the grid, export) must use the dense path (plan = None).

A block is 16 x 16 coefficients of its level (32 x 32 output pixels); the lists hold vertical runs of blocks,
{plane, first column, first row, last row + 1} in coefficient units.
"""
import numpy as np
import torch
import torch.nn.functional as F

from ._lib import call, ptr, stream

TILE = 32          # top-level tile edge in plane texels == one block of the top level
# wavelet name -> TNL_WAVELET_* id (include/trinerflet_b200.h)
WAVELET_IDS = {'bior6.8': 0, 'haar': 1, 'bior2.2': 2, 'bior2.6': 3, 'bior4.4': 4}
MAX_ACTIVE_RUN = 6  # blocks per active item (96 rows: halo overhead 8/96)
MAX_CLEAN_RUN = 8


def _runs(mask, max_len):
    """mask [K, nb] bool -> (k, start, end) arrays of the maximal runs of True along axis 1, split to <= max_len."""
    K, nb = mask.shape
    pad = np.zeros((K, 1), dtype=np.int8)
    d = np.diff(np.concatenate([pad, mask.astype(np.int8), pad], axis=1), axis=1)
    ks, starts = np.nonzero(d == 1)
    _, ends = np.nonzero(d == -1)
    if ks.size == 0:
        return ks, starts, ends
    pieces = (ends - starts + max_len - 1) // max_len
    idx = np.repeat(np.arange(ks.size), pieces)
    first = np.cumsum(pieces) - pieces
    j = np.arange(idx.size) - first[idx]
    s = starts[idx] + j * max_len
    e = np.minimum(s + max_len, ends[idx])
    return ks[idx], s, e


def _items(block_map, active, max_len):
    """block_map [3, nb(rows), nb(cols)] bool -> int32 [n, 4] items {plane, m0, row_lo, row_hi} over runs of `active`."""
    nb = block_map.shape[1]
    cols = np.ascontiguousarray(np.transpose(block_map, (0, 2, 1))).reshape(3 * nb, nb)   # [(plane, bx), by]
    k, s, e = _runs(cols if active else ~cols, max_len)
    out = np.empty((k.size, 4), dtype=np.int32)
    out[:, 0] = k // nb
    out[:, 1] = (k % nb) * 16
    out[:, 2] = s * 16
    out[:, 3] = e * 16
    return out


def level_maps(flags, levels):
    """flags [3, T, T] bool (top-level dirty tiles) -> (fwd_maps, bwd_maps), lists over levels 0 .. L-1 of bool block maps."""
    f = flags[None].float()                 # [1, 3, T, T]: planes as channels
    fwd = [None] * levels
    a = f
    for l in reversed(range(levels)):
        fwd[l] = a
        if l > 0:   # output tile k of level l-1 (32 px) is read by blocks 2k-1 .. 2k+2 of level l (16 px each, 4 px halo)
            a = F.max_pool2d(a, kernel_size=4, stride=2, padding=1)
    bwd = [None] * levels
    g = f
    for l in reversed(range(levels)):
        b = F.max_pool2d(g, kernel_size=3, stride=1, padding=1)   # block k reads fine tiles k-1 .. k+1 (8 px halo)
        bwd[l] = b
        if l > 0:
            g = F.max_pool2d(b, kernel_size=2, stride=2)           # its g_x lands in tile k // 2 of the level below
    return [m[0] > 0 for m in fwd], [m[0] > 0 for m in bwd]


def idwt_call(name, wave, *args):
    """Issue the IDWT entry point `name` (tnl_idwt_level_*, arguments ending with the stream) for wavelet `wave`.  bior6.8
    goes through the entry points without suffix, whose names and argument positions the benchmark's per-kernel
    attribution reads; the other wavelets through `name`_wavelet, with the wavelet id before the stream."""
    if wave == 'bior6.8':
        call(name, *args)
    else:
        call(name + "_wavelet", *args[:-1], WAVELET_IDS[wave], args[-1])


class IdwtPlan:
    def __init__(self, R, n0, levels, C, device):
        if levels < 1 or n0 % 16 != 0 or R != n0 * 2 ** levels or R % TILE != 0:
            raise ValueError("work-list IDWT needs base resolution % 16 == 0 and at least one wavelet level")
        self.R, self.n0, self.levels, self.C, self.device = R, n0, levels, C, device
        self.version = 0          # bumped whenever a list buffer is reallocated (captured CUDA graphs must be rebuilt)
        self.fwd = [None] * levels   # per level: dict(active, clean, counts, cap_active, cap_clean)
        self.bwd = [None] * levels
        self.gap = [None] * levels
        self.stats = {}
        # set by the training step when it drives the backward itself (SplitIdwtBackward): the forward then skips the
        # |yh| pass over the clean blocks and the backward's clean part, which reads those coefficients anyway, adds it
        self.defer_clean_abs = False
        self.on_planes_ready = None   # called once, right after the last active forward level has been issued
        self.zero = None              # tiles of the plane-gradient buffer the backward reads: dict(ids, count, cap)

    def _store(self, slot_list, l, active, clean):
        slot = slot_list[l]
        if slot is None or active.shape[0] > slot["cap_active"] or clean.shape[0] > slot["cap_clean"]:
            cap_a = max(64, 2 * active.shape[0])
            cap_c = max(64, 2 * clean.shape[0])
            slot = dict(active=torch.zeros(cap_a, 4, dtype=torch.int32, device=self.device),
                        clean=torch.zeros(cap_c, 4, dtype=torch.int32, device=self.device),
                        counts=torch.zeros(2, dtype=torch.int32, device=self.device), cap_active=cap_a, cap_clean=cap_c)
            slot_list[l] = slot
            self.version += 1
        if active.shape[0]:
            slot["active"][:active.shape[0]].copy_(torch.from_numpy(active), non_blocking=False)
        if clean.shape[0]:
            slot["clean"][:clean.shape[0]].copy_(torch.from_numpy(clean), non_blocking=False)
        slot["counts"].copy_(torch.tensor([active.shape[0], clean.shape[0]], dtype=torch.int32))
        slot["n_active"], slot["n_clean"] = int(active.shape[0]), int(clean.shape[0])

    def _active_items(self, block_map, target_ctas=4 * 148):
        """Runs of active blocks, as long as possible (halo overhead 8 rows per item) but short enough that the coarse
        levels, which have few blocks, still spread over the machine (a CTA streams its rows sequentially)."""
        chunks = max(1, self.C // 16)
        run = MAX_ACTIVE_RUN
        items = _items(block_map, True, run)
        while run > 1 and items.shape[0] * chunks < target_ctas:
            run -= 1
            items = _items(block_map, True, run)
        return items

    def update(self, flags):
        """flags: uint8/bool [3 * T * T] or [3, T, T] device tensor from tnl_mark_dirty_tiles (T = R / 32)."""
        T = self.R // TILE
        f = flags.reshape(3, T, T) > 0
        fwd_maps, bwd_maps = level_maps(f, self.levels)
        frac_f, frac_b = [], []
        for l in range(self.levels):
            mf, mb = fwd_maps[l].cpu().numpy(), bwd_maps[l].cpu().numpy()
            self._store(self.fwd, l, self._active_items(mf), _items(mf, False, MAX_CLEAN_RUN))
            self._store(self.bwd, l, self._active_items(mb), _items(mb, False, MAX_CLEAN_RUN))
            # blocks the backward treats as active but the forward does not reconstruct: with defer_clean_abs their |yh| is
            # counted neither by the forward's active blocks nor by the backward's clean part -> a (small) list of their own
            self._store(self.gap, l, np.zeros((0, 4), dtype=np.int32), _items(mb & ~mf, True, MAX_CLEAN_RUN))
            frac_f.append(float(mf.mean()))
            frac_b.append(float(mb.mean()))
        # the backward's active top-level blocks read the incoming gradient on their 8-pixel halo: tiles k-1 .. k+1
        z = F.max_pool2d(bwd_maps[-1][None].float(), kernel_size=3, stride=1, padding=1)[0] > 0
        ids = torch.nonzero(z.reshape(-1)).squeeze(-1).int()
        if self.zero is None or ids.numel() > self.zero["cap"]:
            cap = max(64, 2 * ids.numel())
            self.zero = dict(ids=torch.zeros(cap, dtype=torch.int32, device=self.device),
                             count=torch.zeros(1, dtype=torch.int32, device=self.device), cap=cap)
            self.version += 1
        self.zero["ids"][:ids.numel()].copy_(ids)
        self.zero["count"].fill_(int(ids.numel()))
        self.stats = dict(active_fraction_forward=frac_f, active_fraction_backward=frac_b, tile_fraction=float(f.float().mean()),
                          zero_fill_fraction=float(z.float().mean()))
        return self

    def zero_gradient_tiles(self, g_planes_dense):
        """Zero the tiles of a (channels-last, dense-storage) plane-gradient buffer that the work-list backward reads."""
        call("tnl_tiles_zero", ptr(g_planes_dense), ptr(self.zero["ids"]), ptr(self.zero["count"]), self.zero["cap"], self.R, self.C,
             TILE, stream())

    @staticmethod
    def from_model(model, margin=2, plan=None):
        """Build / refresh the plan from the model's density bitfield (call after every update_extra_state)."""
        enc = model.encoder
        R, C = enc.plane_resolution, enc.number_of_features
        levels = len(enc.planes_features_wavelet_coefs)
        n0 = enc.planes_features.shape[2]
        if plan is None:
            plan = IdwtPlan(R, n0, levels, C, model.density_bitfield.device)
        T = R // TILE
        flags = torch.empty(3 * T * T, dtype=torch.uint8, device=model.density_bitfield.device)
        call("tnl_mark_dirty_tiles", ptr(model.density_bitfield), model.cascade, model.grid_size, float(model.bound), R, TILE, margin,
             ptr(flags), stream())
        return plan.update(flags)

    # ---- per-level launches ------------------------------------------------------------------------------------------
    def forward_level(self, l, x, yh, out, n, abs_sum, parts=3, wave='bior6.8'):
        """parts: 1 = reconstruct the active blocks, 2 = |yh| sum of the clean blocks, 3 = both."""
        s = self.fwd[l]
        idwt_call("tnl_idwt_level_forward_sparse", wave, ptr(x), ptr(yh), ptr(out), n, self.C, ptr(abs_sum), ptr(s["active"]),
                  ptr(s["clean"]), ptr(s["counts"]), s["cap_active"], s["cap_clean"], int(parts), stream())

    def forward_gap_abs(self, l, yh, n, abs_sum):
        """abs_sum += sum |yh| over the blocks that are active in the backward but not reconstructed by the forward."""
        s = self.gap[l]
        call("tnl_idwt_level_forward_sparse", ptr(yh), ptr(yh), ptr(yh), n, self.C, ptr(abs_sum), ptr(s["active"]), ptr(s["clean"]),
             ptr(s["counts"]), 0, s["cap_clean"], 2, stream())

    def backward_level(self, l, g, g_x, g_yh, n, yh, reg_grad, reg_coef, parts=3, abs_sum=None, wave='bior6.8'):
        """parts: 1 = active blocks only, 2 = clean blocks only (independent of g), 3 = both.
        abs_sum: the clean part adds sum |yh| of its blocks (see defer_clean_abs)."""
        s = self.bwd[l]
        idwt_call("tnl_idwt_level_backward_sparse", wave, ptr(g) if g is not None else None, ptr(g_x), ptr(g_yh), n, self.C,
                  ptr(yh) if yh is not None else None, ptr(reg_grad) if reg_grad is not None else None, float(reg_coef),
                  ptr(s["active"]), ptr(s["clean"]), ptr(s["counts"]), s["cap_active"], s["cap_clean"], int(parts),
                  ptr(abs_sum) if abs_sum is not None else None, stream())
