"""Linear rational spline transformer of Dolatabadi et al. 2020 (API of
torchflows/.../transformers/spline/linear_rational.py:9-182).

Per element 4K parameters: u_x = h[:K] (width logits), u_y = h[K:2K] (heights are parameterised as u_x + u_y/100),
u_lambda = h[2K:3K] (position of the intermediate knot inside each bin, through a sigmoid), u_d = h[3K:4K-1] (interior
derivative logits, /100, edges fixed at 1), u_w0 = h[4K-1] (weight of the first knot).  Forward, inverse and backward are one
kernel launch each (csrc/b2f_transformer.cu, math in csrc/b2f_lrs.cuh) instead of ~90 ATen launches and a boolean-mask copy of
h.  With the default n_bins = 8 (32 parameters per element), coupling and MADE layers built on it are ops of fused flow programs:
the same device math runs inside the whole-flow kernels, one launch per direction, the sequential MADE direction included, and
one fused backward.  Other bin counts run as a composite (conditioner GEMMs + the stand-alone kernel)."""
import math
from typing import Tuple, Union

import torch

from torchflows_b200 import _native as N
from torchflows_b200.bijections.finite.autoregressive.transformers.spline.base import MonotonicSpline


class LinearRational(MonotonicSpline):
    _tkind_forward = N.T_LRS_FWD
    _tkind_inverse = N.T_LRS_INV

    def __init__(self, event_shape: Union[torch.Size, Tuple[int, ...]], boundary: float = 50.0, **kwargs):
        super().__init__(event_shape, min_input=-boundary, max_input=boundary, min_output=-boundary,
                         max_output=boundary, **kwargs)
        if not 1 <= self.n_bins <= 64:
            raise NotImplementedError('LinearRational kernels support 1 <= n_bins <= 64')
        self.boundary = float(boundary)
        self.min_bin_width = 1e-2
        self.min_bin_height = 1e-2
        self.min_d = 1e-5
        self.const = math.log(math.exp(1 - self.min_d) - 1)
        self.eps = 5e-10

    @property
    def parameter_shape_per_element(self) -> torch.Size:
        return torch.Size((4 * self.n_bins,))

    @property
    def default_parameters(self) -> torch.Tensor:
        return torch.zeros(self.parameter_shape)

    def _kernel_args(self):
        return self.n_bins, self.boundary
