"""Architecture presets (API of torchflows/.../autoregressive/architectures.py:31-223).

Every preset is ``ElementwiseAffine -> [ReversePermutation -> <base> -> ActNorm] x n_layers -> ElementwiseAffine ->
ActNorm``.  With the default arguments the whole stack lowers to one libb2f flow program, i.e. ``log_prob`` and
``sample`` are one kernel launch each."""
from typing import Optional, Tuple, Type, Union

import torch

from torchflows_b200.bijections.base import BijectiveComposition
from torchflows_b200.bijections.finite.autoregressive.layers import (ActNorm, AffineCoupling,
                                                                    AffineForwardMaskedAutoregressive,
                                                                    AffineInverseMaskedAutoregressive,
                                                                    ElementwiseAffine, InverseAffineCoupling,
                                                                    LRSCoupling, LRSForwardMaskedAutoregressive,
                                                                    LRSInverseMaskedAutoregressive,
                                                                    RQSCoupling, RQSForwardMaskedAutoregressive,
                                                                    RQSInverseMaskedAutoregressive, ShiftCoupling)
from torchflows_b200.bijections.finite.autoregressive.layers_base import (CouplingBijection,
                                                                         InverseMaskedAutoregressiveBijection,
                                                                         MaskedAutoregressiveBijection)
from torchflows_b200.bijections.finite.matrix.permutation import ReversePermutationMatrix
from torchflows_b200.utils import event_size


class AutoregressiveArchitecture(BijectiveComposition):
    def __init__(self, event_shape: Union[Tuple[int, ...], torch.Size, int],
                 base_bijection: Type[Union[CouplingBijection, MaskedAutoregressiveBijection,
                                            InverseMaskedAutoregressiveBijection]],
                 context_shape: Optional[Union[Tuple[int, ...], torch.Size, int]] = None, n_layers: int = 2, **kwargs):
        if isinstance(event_shape, int):
            event_shape = (event_shape,)
        event_shape = tuple(event_shape)
        graphical = kwargs.get('edge_list') is not None
        stack = [ElementwiseAffine(event_shape=event_shape, context_shape=context_shape)]
        for _ in range(n_layers):
            if not graphical:
                stack.append(ReversePermutationMatrix(event_shape=event_shape, context_shape=context_shape))
            stack.append(base_bijection(event_shape=event_shape, context_shape=context_shape, **kwargs))
            stack.append(ActNorm(event_shape=event_shape))
        stack.append(ElementwiseAffine(event_shape=event_shape, context_shape=context_shape))
        stack.append(ActNorm(event_shape=event_shape, context_shape=context_shape))
        super().__init__(stack)


class NICE(AutoregressiveArchitecture):
    """Dinh et al. 2015: additive coupling."""

    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=ShiftCoupling, **kwargs)


class RealNVP(AutoregressiveArchitecture):
    """Dinh et al. 2017: affine coupling (an elementwise affine map for 1-D events)."""

    def __init__(self, event_shape, **kwargs):
        shape = (event_shape,) if isinstance(event_shape, int) else tuple(event_shape)
        base = ElementwiseAffine if event_size(shape) == 1 else AffineCoupling
        super().__init__(event_shape, base_bijection=base, **kwargs)


class InverseRealNVP(AutoregressiveArchitecture):
    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=InverseAffineCoupling, **kwargs)


class MAF(AutoregressiveArchitecture):
    """Papamakarios et al. 2018: one-pass density, sequential sampling."""

    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=AffineForwardMaskedAutoregressive, **kwargs)


class IAF(AutoregressiveArchitecture):
    """Kingma et al. 2017: one-pass sampling, sequential density."""

    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=AffineInverseMaskedAutoregressive, **kwargs)


class CouplingRQNSF(AutoregressiveArchitecture):
    """Durkan et al. 2019: rational-quadratic spline coupling."""

    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=RQSCoupling, **kwargs)


class MaskedAutoregressiveRQNSF(AutoregressiveArchitecture):
    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=RQSForwardMaskedAutoregressive, **kwargs)


class InverseAutoregressiveRQNSF(AutoregressiveArchitecture):
    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=RQSInverseMaskedAutoregressive, **kwargs)


class CouplingLRS(AutoregressiveArchitecture):
    """Dolatabadi et al. 2020: linear rational spline coupling (architectures.py:166-178).  With the default n_bins = 8 the
    whole preset is one fused flow program on the generic FP32 kernel (csrc/b2f_flow.cu): conditioners, spline
    (csrc/b2f_lrs.cuh), permutations and ActNorm in one launch per direction, and one fused backward."""

    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=LRSCoupling, **kwargs)


class MaskedAutoregressiveLRS(AutoregressiveArchitecture):
    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=LRSForwardMaskedAutoregressive, **kwargs)


class InverseAutoregressiveLRS(AutoregressiveArchitecture):
    def __init__(self, event_shape, **kwargs):
        super().__init__(event_shape, base_bijection=LRSInverseMaskedAutoregressive, **kwargs)
