"""Camera pose refinement: a per-image se(3) correction of the training poses, optimised with the field.

    cams = CameraPoses(train_poses)                       # [B,4,4] cam2world, e.g. from COLMAP / LLFF
    optimizer = Adam(model.get_params(lr) + cams.get_params(1e-3), betas=(0.9, 0.99), eps=1e-15)
    data = feeder.select_batch(b, bs, poses=cams())      # rays carry the pose gradient
    step.forward_backward(data['rays_o'][0], data['rays_d'][0], data['images'][0]); step.optimizer_step()

The correction is applied in the camera frame, pose_b @ exp(xi_b), xi_b = delta[b] = (omega, v): omega a rotation vector
(radians), v a translation in scene units, both in the camera's own axes.  The gradient reaches delta through the ray feeder
(tnl_rays_from_ids_backward) and the training march (tnl_rays_backward).
"""
import torch
import torch.nn as nn

# |omega|^2 below which the exp map's coefficients come from their Taylor series (truncation < 1e-13 relative there)
_SERIES_THETA2 = 1e-2


def _hat(w):
    """[..., 3] -> [..., 3, 3] cross-product matrix"""
    z = torch.zeros_like(w[..., 0])
    x, y, c = w[..., 0], w[..., 1], w[..., 2]
    return torch.stack([torch.stack([z, -c, y], -1), torch.stack([c, z, -x], -1), torch.stack([-y, x, z], -1)], -2)


def se3_exp(xi):
    """[..., 6] (omega, v) -> [..., 4, 4] rigid transform [[R, V v], [0, 1]] with R = I + A W + B W^2, V = I + B W + C W^2,
    W = hat(omega), A = sin t / t, B = (1 - cos t) / t^2, C = (t - sin t) / t^3.  Near t = 0 the coefficients are their series in
    t^2 = |omega|^2, so the value and the gradient at xi = 0 are exact (exp(0) = I)."""
    w, v = xi[..., :3], xi[..., 3:]
    th2 = (w * w).sum(-1)
    small = th2 < _SERIES_THETA2
    # closed form on a safe argument (the branch not taken must not produce NaN gradients)
    t2 = torch.where(small, torch.ones_like(th2), th2)
    t = torch.sqrt(t2)
    s, h = torch.sin(t), torch.sin(0.5 * t)
    A_c = s / t
    B_c = 2 * h * h / t2                  # (1 - cos t) / t^2 without the cancellation of 1 - cos t
    C_c = (t - s) / (t2 * t)
    A_s = 1 - th2 / 6 * (1 - th2 / 20 * (1 - th2 / 42))
    B_s = 0.5 - th2 / 24 * (1 - th2 / 30 * (1 - th2 / 56))
    C_s = 1 / 6 - th2 / 120 * (1 - th2 / 42 * (1 - th2 / 72))
    A = torch.where(small, A_s, A_c)[..., None, None]
    B = torch.where(small, B_s, B_c)[..., None, None]
    C = torch.where(small, C_s, C_c)[..., None, None]
    W = _hat(w)
    W2 = W @ W
    eye = torch.eye(3, dtype=xi.dtype, device=xi.device).expand(W.shape)
    R = eye + A * W + B * W2
    V = eye + B * W + C * W2
    tr = (V @ v.unsqueeze(-1))
    top = torch.cat([R, tr], -1)
    bottom = torch.zeros_like(top[..., :1, :])
    bottom[..., 0, 3] = 1
    return torch.cat([top, bottom], -2)


class CameraPoses(nn.Module):
    """poses [B,4,4] cam2world (tensor or array; kept as a buffer in its dtype and device) -> forward() = pose_b @ exp(xi_b),
    [B,4,4], with a zero-initialised learnable delta [B,6] (omega, v) in the camera frame.  fixed: image indices whose pose
    is not refined (their delta gets exactly zero gradient and stays 0 under Adam).  At delta = 0, forward() returns the
    poses bit for bit (the composition is an elementwise product and sum, never a TF32 matmul)."""

    def __init__(self, poses, fixed=None):
        super().__init__()
        poses = torch.as_tensor(poses).detach().clone()
        if poses.dim() != 3 or tuple(poses.shape[1:]) != (4, 4):
            raise ValueError(f"CameraPoses: poses must be [B,4,4], got {list(poses.shape)}")
        B = poses.shape[0]
        self.register_buffer("poses", poses)
        self.delta = nn.Parameter(torch.zeros(B, 6, dtype=poses.dtype, device=poses.device))
        free = torch.ones(B, dtype=torch.bool)
        if fixed is not None:
            free[torch.as_tensor(fixed, dtype=torch.long).reshape(-1)] = False
        self.register_buffer("free", free.to(poses.device))

    def forward(self):
        xi = torch.where(self.free.unsqueeze(-1), self.delta, torch.zeros_like(self.delta))
        E = se3_exp(xi)
        return (self.poses.unsqueeze(-1) * E.unsqueeze(-3)).sum(-2)

    def get_params(self, lr):
        """optimizer parameter groups, as NeRFNetwork.get_params: Adam(model.get_params(lr) + cams.get_params(lr_pose))"""
        return [{'params': [self.delta], 'lr': lr}]
