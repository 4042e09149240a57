"""TEST INFRASTRUCTURE ONLY: the reference's field as its literal torch op sequence, for input gradients.

Unlike oracle/field.py, which emulates the fp16-autocast rounding points explicitly, this builds the graph the reference
runs (reconstruction/triplaneencoder/triplane_encoder.py:293-332, reconstruction/nerf/network.py:118-166) and leaves the
precision to the ambient state: under torch.autocast('cuda', torch.float16) autocast itself inserts the casts, in fp32 or
fp64 nothing is rounded.  torch.autograd.grad of its outputs is the arbiter of the position and direction gradients.
"""
import torch
import torch.nn.functional as F

from oracle.field import plane_axes_tensor, sh16, trunc_exp


def inv_bound(bound, dtype):
    """CUDA evaluates `tensor / python_scalar` as tensor * (1/scalar) in the tensor's precision"""
    return torch.tensor(1.0, dtype=dtype) / torch.tensor(bound, dtype=dtype)


def sample(planes, x, bound):
    """planes logical [3,C,R,R], x [M,3] -> features [M, 3C]: coords * 1/bound, the projection matmul with the plane axes,
    grid_sample (bilinear, border, align_corners=True), permute / view"""
    axes = plane_axes_tensor(x.dtype).to(x.device)
    u = x * inv_bound(bound, x.dtype).to(x.device)
    proj = torch.matmul(u.unsqueeze(0), axes)                                   # [3, M, 2]
    s = F.grid_sample(planes.to(x.dtype) if x.dtype == torch.float64 else planes, proj.unsqueeze(2), mode="bilinear",
                      padding_mode="border", align_corners=True)                 # [3, C, M, 1]
    M = x.shape[0]
    return s.permute(2, 0, 1, 3).reshape(M, -1)


def density(planes, x, W, bound):
    W1, W2 = W[0], W[1]
    h = F.relu(F.linear(sample(planes, x, bound), W1))
    h = F.linear(h, W2)
    return trunc_exp(h[..., 0].float() if h.dtype == torch.float16 else h[..., 0]), h[..., 1:]


def field(planes, x, d, W, bound):
    """-> sigma [M], rgb [M,3] of the reference's NeRFNetwork.forward"""
    sigma, geo = density(planes, x, W, bound)
    sh = sh16(d.float() if d.dtype == torch.float16 else d)
    h = torch.cat([sh, geo], dim=-1)
    h = F.relu(F.linear(h, W[2]))
    h = F.relu(F.linear(h, W[3]))
    return sigma, torch.sigmoid(F.linear(h, W[4]))


def input_grads(planes, x, d, W, bound, g_sigma, g_rgb):
    """torch.autograd.grad((sigma, rgb), (x, d), (g_sigma, g_rgb)) of the literal graph, under the ambient autocast state"""
    x = x.detach().clone().requires_grad_(True)
    d = d.detach().clone().requires_grad_(True)
    sigma, rgb = field(planes, x, d, W, bound)
    return torch.autograd.grad((sigma, rgb), (x, d), (g_sigma.to(sigma.dtype), g_rgb.to(rgb.dtype)))
