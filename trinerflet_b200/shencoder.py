"""Drop-in for the reference's `shencoder` package (aux_libs/shencoder/sphere_harmonics.py:14-87), degree <= 4.
As in the reference, the input gradient is computed when the inputs require grad (sphere_harmonics.py:84); it is
once-differentiable.  Inside NeRFNetwork the SH evaluation is fused into the MLP kernels; this module serves stand-alone
callers and the fp32 library path of the heads."""
import torch
import torch.nn as nn
from torch.autograd import Function
from torch.autograd.function import once_differentiable
from torch.amp import custom_bwd, custom_fwd

from ._lib import call, ptr, stream


class _sh_encoder(Function):
    @staticmethod
    @custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, inputs, degree, calc_grad_inputs=False):
        inputs = inputs.contiguous()
        B = inputs.shape[0]
        outputs = torch.empty(B, degree ** 2, dtype=inputs.dtype, device=inputs.device)
        call("tnl_sh_encode_forward", ptr(inputs), ptr(outputs), B, int(degree), stream())
        ctx.save_for_backward(inputs if calc_grad_inputs else None)
        ctx.degree = int(degree)
        return outputs

    @staticmethod
    @once_differentiable
    @custom_bwd(device_type="cuda")
    def backward(ctx, grad):
        (inputs,) = ctx.saved_tensors
        if inputs is None:
            return None, None, None
        grad = grad.contiguous().float()
        grad_inputs = torch.empty_like(inputs)
        call("tnl_sh_encode_backward", ptr(grad), ptr(inputs), inputs.shape[0], ctx.degree, ptr(grad_inputs), stream())
        return grad_inputs, None, None


sh_encode = _sh_encoder.apply


class SHEncoder(nn.Module):
    def __init__(self, input_dim=3, degree=4):
        super().__init__()
        self.input_dim = input_dim
        self.degree = degree
        self.output_dim = degree ** 2
        assert self.input_dim == 3, "SH encoder only support input dim == 3"
        assert 0 < self.degree <= 4, "trinerflet_b200 SH encoder supports degree in [1, 4] (reference hot path uses 4)"

    def __repr__(self):
        return f"SHEncoder: input_dim={self.input_dim} degree={self.degree}"

    def forward(self, inputs, size=1):
        inputs = inputs / size
        prefix_shape = list(inputs.shape[:-1])
        inputs = inputs.reshape(-1, self.input_dim)
        outputs = sh_encode(inputs, self.degree, inputs.requires_grad)
        return outputs.reshape(prefix_shape + [self.output_dim])
