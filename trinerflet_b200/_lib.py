"""ctypes binding of libtrinerflet_b200.so (the C ABI of include/trinerflet_b200.h).

There is deliberately no fallback: if the shared library is missing or a call fails, the caller gets a
RuntimeError.  torch is used only for device memory and the current CUDA stream.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libtrinerflet_b200.so")

_c = ctypes
_vp, _u32, _f32, _int, _sz = _c.c_void_p, _c.c_uint32, _c.c_float, _c.c_int, _c.c_size_t


class MlpDims(ctypes.Structure):
    _fields_ = [("in_dim", _u32), ("hidden", _u32), ("hidden_c", _u32)]


_DP = ctypes.POINTER(MlpDims)

# name -> (restype, argtypes); must list every symbol of include/trinerflet_b200.h (tests/test_abi.py checks)
SIGNATURES = {
    "tnl_abi_version": (_int, []),
    "tnl_last_error": (_c.c_char_p, []),
    "tnl_near_far_from_aabb": (_int, [_vp, _vp, _vp, _u32, _f32, _vp, _vp, _vp]),
    "tnl_sph_from_ray": (_int, [_vp, _vp, _f32, _u32, _vp, _vp]),
    "tnl_morton3d": (_int, [_vp, _u32, _vp, _vp]),
    "tnl_morton3d_invert": (_int, [_vp, _u32, _vp, _vp]),
    "tnl_packbits": (_int, [_vp, _u32, _f32, _vp, _vp]),
    "tnl_march_rays_train_workspace": (_sz, [_u32]),
    "tnl_march_rays_train_workspace_fast": (_sz, [_u32, _u32]),
    "tnl_march_rays_train": (_int, [_vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp,
                                    _vp, _vp, _vp, _vp, _sz, _vp]),
    "tnl_march_rays_train_ts": (_int, [_vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp,
                                       _vp, _vp, _vp, _vp, _sz, _vp]),
    "tnl_rays_backward": (_int, [_vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp]),
    "tnl_composite_rays_train_forward": (_int, [_vp, _vp, _vp, _vp, _u32, _u32, _f32, _vp, _vp, _vp, _vp]),
    "tnl_composite_rays_train_backward": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _u32, _f32, _vp, _vp, _vp]),
    "tnl_march_rays": (_int, [_u32, _u32, _vp, _vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp,
                              _vp, _vp]),
    "tnl_composite_rays": (_int, [_u32, _u32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tnl_compact_alive_workspace": (_sz, [_u32]),
    "tnl_compact_alive": (_int, [_vp, _u32, _vp, _vp, _vp, _sz, _vp]),
    "tnl_infer_plan": (_int, [_vp, _u32, _u32, _vp]),
    "tnl_march_rays_dev": (_int, [_vp, _u32, _vp, _vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tnl_composite_rays_dev": (_int, [_vp, _u32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tnl_compact_alive_dev": (_int, [_vp, _u32, _vp, _vp, _vp, _sz, _vp]),
    "tnl_sh_encode_forward": (_int, [_vp, _vp, _u32, _u32, _vp]),
    "tnl_sh_encode_backward": (_int, [_vp, _vp, _u32, _u32, _vp, _vp]),
    "tnl_idwt_level_forward": (_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp]),
    "tnl_idwt_level_backward": (_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp, _f32, _u32, _u32, _vp]),
    "tnl_sample_planes_forward": (_int, [_vp, _vp, _u32, _u32, _u32, _f32, _int, _vp, _vp, _vp, _int, _vp]),
    "tnl_sample_planes_backward": (_int, [_vp, _int, _vp, _u32, _u32, _u32, _f32, _int, _vp, _vp, _vp, _vp]),
    "tnl_sample_planes_backward_plane": (_int, [_vp, _int, _vp, _u32, _u32, _u32, _f32, _int, _vp, _vp, _vp, _u32, _vp]),
    "tnl_sample_planes_backward_det_workspace": (_sz, [_u32, _u32]),
    "tnl_sample_planes_backward_det": (_int, [_vp, _int, _vp, _u32, _u32, _u32, _f32, _int, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp,
                                              _sz, _vp]),
    "tnl_sample_planes_backward_coords": (_int, [_vp, _vp, _vp, _u32, _u32, _u32, _f32, _int, _vp, _vp]),
    "tnl_sample_planes_backward_xyz": (_int, [_vp, _int, _vp, _vp, _u32, _u32, _u32, _f32, _int, _vp, _vp, _vp, _vp]),
    "tnl_cell_sort_workspace": (_sz, [_u32, _u32]),
    "tnl_cell_sort": (_int, [_vp, _u32, _vp, _f32, _u32, _vp, _vp, _sz, _vp]),
    "tnl_mlp_packed_bytes": (_sz, [_DP]),
    "tnl_mlp_pack_weights": (_int, [_DP, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tnl_mlp_forward": (_int, [_DP, _vp, _vp, _int, _vp, _u32, _vp, _vp, _vp, _vp, _vp]),
    "tnl_mlp_backward": (_int, [_DP, _vp, _vp, _int, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tnl_mlp_backward_dirs": (_int, [_DP, _vp, _vp, _int, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "tnl_mlp_backward_det_workspace": (_sz, [_DP, _int, _u32]),
    "tnl_mlp_backward_det": (_int, [_DP, _vp, _vp, _int, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "tnl_mlp_backward_scatter": (_int, [_DP, _vp, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _u32, _u32, _f32, _int, _vp, _vp, _vp,
                                        _vp, _vp, _vp, _vp]),
    "tnl_idwt_level_forward_sparse": (_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp, _u32, _u32, _u32, _vp]),
    "tnl_idwt_level_backward_sparse": (_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp, _f32, _vp, _vp, _vp, _u32, _u32, _u32, _vp, _vp]),
    "tnl_idwt_level_forward_wavelet": (_int, [_vp, _vp, _vp, _u32, _u32, _vp, _u32, _vp]),
    "tnl_idwt_level_backward_wavelet": (_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp, _f32, _u32, _u32, _u32, _vp]),
    "tnl_idwt_level_forward_sparse_wavelet": (_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp, _u32, _u32, _u32, _u32, _vp]),
    "tnl_idwt_level_backward_sparse_wavelet": (_int, [_vp, _vp, _vp, _u32, _u32, _vp, _vp, _f32, _vp, _vp, _vp, _u32, _u32, _u32, _vp,
                                                      _u32, _vp]),
    "tnl_tiles_zero": (_int, [_vp, _vp, _vp, _u32, _u32, _u32, _u32, _vp]),
    "tnl_mlp_tc_profile": (_int, [_vp]),
    "tnl_umma_bench": (_int, [_int] * 8 + [_vp, _vp]),
    "tnl_umma_bench2": (_int, [_u32] * 8 + [_int] * 6 + [_vp, _vp]),
    "tnl_umma_probe": (_int, [_vp, _int, _int, _vp, _int, _int, _int, _int, _int, _int, _int, _vp, _int, _vp]),
    "tnl_mark_dirty_tiles": (_int, [_vp, _u32, _u32, _f32, _u32, _u32, _u32, _vp, _vp]),
    "tnl_tiles_pack": (_int, [_vp, _vp, _u32, _u32, _u32, _u32, _vp, _int, _vp]),
    "tnl_tiles_unpack": (_int, [_vp, _vp, _u32, _u32, _u32, _u32, _f32, _int, _vp, _vp]),
    "tnl_tiles_allreduce": (_int, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _u32, _u32, _u32, _f32, _vp]),
    "tnl_flat_allreduce": (_int, [_vp, _vp, _u32, _u32, _u32, _f32, _vp]),
    "tnl_grad_nonfinite": (_int, [_vp, ctypes.c_uint64, _vp, _vp]),
    "tnl_adam_prepare": (_int, [_vp, _vp, _f32, _f32, _vp]),
    "tnl_adam_step": (_int, [_vp, _vp, _vp, _vp, ctypes.c_uint64, _vp, _vp, _vp, _f32, _f32, _f32, _f32, _f32, _vp]),
    "tnl_grid_cell_positions": (_int, [_vp, _u32, _u32, _f32, _vp, _vp, _vp]),
    "tnl_grid_ema_update_sum": (_int, [_vp, _vp, _u32, _f32, _vp, _vp]),
    "tnl_packbits_mean": (_int, [_vp, _u32, _vp, _f32, _vp, _vp, _vp]),
    "tnl_grid_scatter": (_int, [_vp, _vp, _u32, _f32, _vp, _vp]),
    "tnl_rays_from_ids": (_int, [_vp, _u32, _f32, _f32, _f32, _f32, _u32, _u32, _vp, ctypes.c_int64, _u32, _vp, _u32, _vp, _vp,
                                 _vp, _vp]),
    "tnl_rays_from_ids_backward": (_int, [_vp, _vp, _u32, _f32, _f32, _f32, _f32, _u32, _u32, _vp, ctypes.c_int64, _u32, _vp, _vp]),
    "tnl_mc_workspace": (_sz, [_u32, _u32, _u32]),
    "tnl_mc_count": (_int, [_vp, _u32, _u32, _u32, _c.c_double, _vp, _sz, _vp, _vp]),
    "tnl_mc_emit": (_int, [_vp, _u32, _u32, _u32, _c.c_double, _vp, _sz, _c.c_int64, _c.c_int64, _vp, _vp, _vp]),
}

_lib = None


def load():
    """Load the shared library (once). Raises if it has not been built: there is no CPU path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"trinerflet_b200: {LIB_PATH} not found. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C trinerflet_b200/csrc`. There is no CPU / PyTorch fallback for this path.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the ABI and this table ever diverge
        fn.restype = res
        fn.argtypes = args
    if lib.tnl_abi_version() != 1:
        raise RuntimeError("trinerflet_b200: ABI version mismatch")
    _lib = lib
    return lib


def stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def deterministic():
    """True under torch.use_deterministic_algorithms(True): the package then launches its order-independent kernels (the
    fixed-point plane-gradient scatter, the slot-ordered MLP weight-gradient reduction) and torch's deterministic reductions
    instead of fp32 / fp64 atomics, so a single-GPU training step gives the same bits for the same inputs."""
    return torch.are_deterministic_algorithms_enabled()


def alert_nondeterministic(what):
    """torch's rule for an operation without a deterministic implementation: in deterministic mode raise, or warn under
    warn_only=True."""
    if not deterministic():
        return
    msg = f"trinerflet_b200: {what} has no deterministic implementation (torch.use_deterministic_algorithms is on)"
    if torch.is_deterministic_algorithms_warn_only_enabled():
        import warnings
        warnings.warn(msg)
    else:
        raise RuntimeError(msg)


_workspaces = {}


def workspace(key, nbytes, device):
    """A persistent device scratch buffer of at least nbytes (one per key and device), reused by every call: the
    deterministic kernels need gigabytes at the larger configs, and torch fills fresh allocations in deterministic mode."""
    k = (key, str(device))
    buf = _workspaces.get(k)
    if buf is None or buf.numel() < nbytes:
        _workspaces[k] = None
        buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
        _workspaces[k] = buf
    return buf


def ptr(t):
    """Device pointer of a CUDA tensor (None -> NULL). The tensor must be contiguous in the layout the ABI expects."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("trinerflet_b200: tensor must live on a CUDA device (no CPU path)")
    return ctypes.c_void_p(t.data_ptr())


def check(rc, what):
    if rc != 0:
        msg = load().tnl_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"trinerflet_b200.{what} failed (rc={rc}): {msg}")


# number of kernels each ABI call launches (for the launch counter the benchmark reports)
KERNELS_PER_CALL = {"tnl_march_rays_train": 6, "tnl_march_rays_train_ts": 7, "tnl_sample_planes_backward_det": 4, "tnl_mlp_backward_det": 2, "tnl_composite_rays_train_backward": 2, "tnl_compact_alive": 3, "tnl_compact_alive_dev": 3, "tnl_cell_sort": 5,
                    "tnl_mlp_pack_weights": 2, "tnl_mc_count": 2}
# work-list IDWT calls launch one kernel per requested part (position of the `parts` argument from the end)
_PARTS_ARG = {"tnl_idwt_level_forward_sparse": -2, "tnl_idwt_level_backward_sparse": -3,
              "tnl_idwt_level_forward_sparse_wavelet": -3, "tnl_idwt_level_backward_sparse_wavelet": -4}
launch_count = 0
_profile = None  # when enabled: name -> list of (start_event, end_event, scalar_args)


def profile_start():
    """Record a CUDA-event pair around every ABI call on the current stream (bench.py roofline measurement)."""
    global _profile
    _profile = {}


def profile_stop():
    """-> {name: [(milliseconds, scalar_args), ...]}; synchronises the device."""
    global _profile
    rec, _profile = _profile, None
    torch.cuda.synchronize()
    out = {}
    for name, evs in (rec or {}).items():
        out[name] = [(e0.elapsed_time(e1), meta) for e0, e1, meta in evs]
    return out


def call(name, *args):
    global launch_count
    fn = getattr(load(), name)
    if name in _PARTS_ARG:
        launch_count += bin(int(args[_PARTS_ARG[name]]) & 3).count("1")
    else:
        launch_count += KERNELS_PER_CALL.get(name, 1)
    if _profile is None:
        check(fn(*args), name)
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    rc = fn(*args)
    e1.record()
    _profile.setdefault(name, []).append((e0, e1, tuple(a for a in args if isinstance(a, (int, float)))))
    check(rc, name)
