"""Autoregressive layer bases (API of torchflows/.../autoregressive/layers_base.py:14-318).

Each class pairs a conditioner with a transformer like the reference, and adds ``lower(direction)``: the
description of the layer as one op of a fused libb2f flow program (conditioner GEMMs + transformer + log-det
in one kernel, ``h`` never written to HBM).  Rational-quadratic and linear rational splines with n_bins = 8 are fused
like the affine transformers.  Configurations outside the fused path (non-default conditioner depth / nonlinearity,
globally learned parameter subsets, n_bins != 8) are detected at construction time and run as a *composite*:
conditioner as library GEMMs, transformer as the stand-alone transformer kernel."""
import os
from typing import Any, List, Optional, Tuple, Type, Union

import torch
import torch.nn as nn

from torchflows_b200 import _native as N
from torchflows_b200 import _program as prog
from torchflows_b200.bijections.base import Bijection
from torchflows_b200.bijections.finite.autoregressive.conditioning.context import Concatenation
from torchflows_b200.bijections.finite.autoregressive.conditioning.coupling_masks import (HalfSplit, PartialCoupling,
                                                                                           make_coupling)
from torchflows_b200.bijections.finite.autoregressive.conditioning.transforms import (MADE, ConditionerTransform,
                                                                                       FeedForward, Linear)
from torchflows_b200.bijections.finite.autoregressive.transformers.base import ScalarTransformer, TensorTransformer
from torchflows_b200.bijections.finite.autoregressive.transformers.spline.linear_rational import LinearRational
from torchflows_b200.bijections.finite.autoregressive.transformers.spline.rational_quadratic import RationalQuadratic
from torchflows_b200.utils import flatten_event, get_batch_shape, unflatten_event


class _TF32Linear(torch.autograd.Function):
    """y = x @ W^T + b as library GEMMs on the tensor cores (TF32) in BOTH directions.  torch's global
    ``allow_tf32`` switch is read when a GEMM executes, so a plain ``F.linear`` under a scoped switch would run its
    backward GEMMs in fp32 SIMT; this Function scopes the switch around its own forward and backward."""

    @staticmethod
    def _scoped(fn):
        previous = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        try:
            return fn()
        finally:
            torch.backends.cuda.matmul.allow_tf32 = previous

    @staticmethod
    def forward(ctx, x, weight, bias):
        ctx.save_for_backward(x, weight)
        return _TF32Linear._scoped(lambda: torch.addmm(bias, x, weight.t()))

    @staticmethod
    def backward(ctx, g):
        x, weight = ctx.saved_tensors
        g = g.contiguous()
        gx = _TF32Linear._scoped(lambda: g @ weight) if ctx.needs_input_grad[0] else None
        gw = _TF32Linear._scoped(lambda: g.t() @ x) if ctx.needs_input_grad[1] else None
        gb = g.sum(dim=0) if ctx.needs_input_grad[2] else None
        return gx, gw, gb


class _WideCoupling(torch.autograd.Function):
    """One wide-conditioner spline coupling layer on libb2f's tcgen05 GEMM pipeline (csrc/b2f_wide.cu): conditioner GEMMs,
    spline and log-det in the forward; recompute, spline backward, dgrad and wgrad GEMMs in the backward.  Only the layer
    input is kept for the backward."""

    @staticmethod
    def forward(ctx, x2, W1, b1, W2, b2, tkind, n_bins, boundary):
        training = any(ctx.needs_input_grad[:5])
        y, ld, keep = N.wide_coupling_forward(tkind, x2, W1, b1, W2, b2, n_bins, boundary, for_backward=training)
        ctx.save_for_backward(x2, W1, b1, W2, b2)
        ctx.cfg = (tkind, n_bins, boundary)
        # packed operands + hidden activations of this call, reusable by the backward while the parameters are unchanged
        ctx.keep = keep
        ctx.versions = tuple(t._version for t in (W1, b1, W2, b2))
        return y, ld

    @staticmethod
    def backward(ctx, gy, gld):
        x2, W1, b1, W2, b2 = ctx.saved_tensors
        tkind, n_bins, boundary = ctx.cfg
        keep = ctx.keep if ctx.versions == tuple(t._version for t in (W1, b1, W2, b2)) else None
        gx, gW1, gb1, gW2, gb2 = N.wide_coupling_backward(tkind, x2, gy, gld, W1, b1, W2, b2, n_bins, boundary, keep=keep)
        ctx.keep = None
        return gx, gW1, gb1, gW2, gb2, None, None, None


def _fits_fused_kernel(n_dim: int, n_hidden: int, kind: int = N.OP_ELEMENTWISE, tkind: int = N.T_AFFINE_FWD,
                       n_bins: int = 0) -> bool:
    """Can a layer of this shape run -- and TRAIN -- inside the fused flow kernels?  Forward: mirror of the shared-memory
    budget of csrc/b2f_flow.cu at its smallest tile (32 samples): the sample tile [32][D|1] plus the hidden activations
    [32][H|1].  Backward: the library is asked (b2f_flow_backward_fits: the backward kernel keeps a gradient tile next to
    the sample tile and stages spline weights per warp, so it runs out of shared memory first -- at D = 768 for MADE
    layers).  Layers that do not fit (e.g. D=1024 with n_hidden=1024) run as a composite: library GEMMs for the
    conditioner and the stand-alone transformer kernel."""
    forward = 4 * (2 * 32 * (n_dim | 1) + 2 * 32 * (n_hidden | 1) + 3 * n_dim + 32 * 24 * 8 + 1024) <= 200 * 1024
    return forward and N.flow_backward_fits(kind, tkind, max(n_hidden, 1), n_bins, n_dim)


def _transformer_fusable(tr) -> bool:
    if isinstance(tr, (RationalQuadratic, LinearRational)):
        return tr.n_bins == 8
    # Affine / InverseAffine / Shift; Scale has stand-alone kernels only
    return isinstance(tr, ScalarTransformer) and 0 <= tr._tkind_forward <= N.T_RQ_INV


class AutoregressiveBijection(Bijection):
    def __init__(self, event_shape, transformer: Union[TensorTransformer, ScalarTransformer],
                 conditioner_transform: Optional[ConditionerTransform], l2_regularization: bool = False,
                 l2_coef: float = 0.01, **kwargs):
        super().__init__(event_shape=event_shape, **kwargs)
        self.conditioner_transform = conditioner_transform
        self.transformer = transformer
        self.l2_regularization = l2_regularization
        self.l2_coef = l2_coef

    def regularization(self, *aux: Tuple[Any, ...]):
        """l2_coef * sum of squared trainable parameters (layers_base.py:38-48)."""
        if self.l2_regularization and self.l2_coef > 0:
            return self.sq_norm_param() * self.l2_coef
        return torch.tensor(0.0)

    def _tkind(self, direction: str) -> int:
        return self.transformer._tkind_forward if direction == 'forward' else self.transformer._tkind_inverse

    def _spline_args(self):
        tr = self.transformer
        return (tr.n_bins, tr.boundary) if isinstance(tr, (RationalQuadratic, LinearRational)) else (0, 0.0)


class CouplingBijection(AutoregressiveBijection):
    """x = (x_A, x_B): x_A passes through and parameterises the transformer applied to x_B."""

    def __init__(self, event_shape, transformer_class: Type[TensorTransformer], context_shape=None,
                 coupling: PartialCoupling = None, conditioner_transform_class: Type[ConditionerTransform] = FeedForward,
                 coupling_kwargs: dict = None, conditioner_kwargs: dict = None, transformer_kwargs: dict = None,
                 l2_regularization: bool = True, **kwargs):
        coupling_kwargs, conditioner_kwargs = coupling_kwargs or {}, conditioner_kwargs or {}
        transformer_kwargs = transformer_kwargs or {}
        if coupling is None:
            coupling = make_coupling(event_shape, **coupling_kwargs)
        transformer = transformer_class(event_shape=coupling.target_shape, **transformer_kwargs)
        conditioner_transform = conditioner_transform_class(
            input_event_shape=coupling.constant_shape, context_shape=context_shape,
            parameter_shape=transformer.parameter_shape, **conditioner_kwargs)
        super().__init__(event_shape=event_shape, transformer=transformer, conditioner_transform=conditioner_transform,
                         context_shape=context_shape, l2_regularization=l2_regularization, **kwargs)
        self.coupling = coupling
        ct = conditioner_transform
        # a context tensor is concatenated to the conditioner input (conditioning/context.py:46-60): such layers run
        # as a composite (conditioner = library GEMMs on [x_A, context], transformer = stand-alone kernel)
        self._fusable = (context_shape is None and isinstance(coupling, HalfSplit) and type(ct) is FeedForward
                         and ct.n_layers == 2 and ct.nonlinearity is nn.Tanh and ct.is_plain
                         and _transformer_fusable(transformer)
                         and _fits_fused_kernel(self.n_dim, ct.n_hidden, N.OP_COUPLING, transformer._tkind_forward,
                                                self._spline_args()[0]))
        # Context-conditioned (conditioning/context.py:46-60: the hidden layer sees [x_A, context]): W1 [x_A, c]^T + b1 =
        # W1[:, :n_A] x_A + (b1 + W1[:, n_A:] c), i.e. the same coupling op with a PER-ROW hidden bias (B2F_FLAG_ROW_BIAS);
        # the bias (B, H) is one small product per call, h = conditioner output still never exists in memory.
        self._fusable_ctx = (context_shape is not None and isinstance(coupling, HalfSplit) and type(ct) is FeedForward
                             and ct.n_layers == 2 and ct.nonlinearity is nn.Tanh and ct.is_plain
                             and type(ct.context_combiner) is Concatenation and _transformer_fusable(transformer)
                             and _fits_fused_kernel(self.n_dim, ct.n_hidden, N.OP_COUPLING, transformer._tkind_forward,
                                                    self._spline_args()[0]))
        # too wide for the whole-flow kernels (e.g. n_dim = 1024, n_hidden = 1024): the layer runs on the tcgen05 GEMM
        # pipeline of csrc/b2f_wide.cu (spline as the output-layer GEMM's epilogue, h never in memory)
        wide_ok = (context_shape is None and isinstance(coupling, HalfSplit)
                   and type(ct) is FeedForward and ct.n_layers == 2 and ct.nonlinearity is nn.Tanh and ct.is_plain
                   and isinstance(transformer, RationalQuadratic)
                   and N.wide_eligible(self.n_dim, ct.n_hidden, transformer.n_bins))
        self._wide = not self._fusable and wide_ok
        # Spline couplings that DO fit the whole-flow kernels can also train through the per-layer GEMM pipeline
        # (B2F_WIDE_TRAINING=1): measured on CouplingRQNSF(256), 131072 rows, it is a tie with the whole-flow backward kernel
        # (7.56 vs 7.50 ms per step: both are bound by the latency of the spline backward arithmetic), so it is off by
        # default and the fp32-faithful recompute of the whole-flow kernel keeps the gradients of the default widths.
        self._wide_training = False
        self._wide_ok = wide_ok

    def _trains_wide(self) -> bool:
        if os.environ.get('B2F_WIDE_TRAINING') != '1' or not (self._fusable and self._wide_ok):
            return False
        return torch.is_grad_enabled() and any(p.requires_grad and p.is_cuda for p in self.conditioner_transform.parameters())

    # -- reference API ---------------------------------------------------------------------------------------
    def get_constant_part(self, x: torch.Tensor) -> torch.Tensor:
        batch_shape = get_batch_shape(x, self.event_shape)
        return flatten_event(x, self.event_shape)[..., self.coupling.source_mask.view(-1)].view(
            *batch_shape, *self.coupling.constant_shape)

    def get_transformed_part(self, x: torch.Tensor) -> torch.Tensor:
        batch_shape = get_batch_shape(x, self.event_shape)
        return flatten_event(x, self.event_shape)[..., self.coupling.target_mask.view(-1)].view(
            *batch_shape, *self.coupling.target_shape)

    def set_transformed_part(self, x: torch.Tensor, x_transformed: torch.Tensor):
        batch_shape = get_batch_shape(x, self.event_shape)
        x[..., self.coupling.target_mask] = x_transformed.reshape(*batch_shape, -1)

    def partition_and_predict_parameters(self, x: torch.Tensor, context: torch.Tensor):
        batch_shape = get_batch_shape(x, self.event_shape)
        h = self.conditioner_transform(self.get_constant_part(x), context=context)
        return h.view(*batch_shape, *self.transformer.parameter_shape)

    # -- fused path ------------------------------------------------------------------------------------------
    #: BijectiveComposition hands the context to lower() (see _segments)
    lowers_with_context: bool = True

    def lower(self, direction: str, context: torch.Tensor = None) -> Optional[List[prog.LoweredOp]]:
        if context is not None:
            return self._lower_with_context(direction, context)
        if not self._fusable or self._trains_wide():
            return None
        seq = self.conditioner_transform.sequential
        n_bins, boundary = self._spline_args()
        return [prog.LoweredOp(kind=N.OP_COUPLING, tkind=self._tkind(direction),
                               leafs=[seq[0].weight, seq[0].bias, seq[2].weight, seq[2].bias],
                               n_hidden=seq[0].out_features, n_bins=n_bins, boundary=boundary, owner=self)]

    def _lower_with_context(self, direction: str, context: torch.Tensor) -> Optional[List[prog.LoweredOp]]:
        ct = self.conditioner_transform
        if not self._fusable_ctx or not context.is_cuda or context.dtype != torch.float32:
            return None
        seq = ct.sequential
        n_a = ct.context_combiner.n_input_dims
        c2 = flatten_event(context, ct.context_shape).reshape(-1, ct.context_combiner.n_context_dims)
        w1 = seq[0].weight
        row_bias = torch.addmm(seq[0].bias, c2, w1[:, n_a:].t())          # (B, H): b1 + W1[:, n_A:] c
        n_bins, boundary = self._spline_args()
        return [prog.LoweredOp(kind=N.OP_COUPLING, tkind=self._tkind(direction),
                               leafs=[w1[:, :n_a], row_bias, seq[2].weight, seq[2].bias],
                               n_hidden=seq[0].out_features, n_bins=n_bins, boundary=boundary, flags=N.FLAG_ROW_BIAS,
                               owner=self)]

    #: composite path only: run the conditioner's library GEMMs on the tensor cores in TF32 for spline layers (the same
    #: precision the fused tcgen05 kernel uses; affine / shift layers always stay in fp32, SURVEY Appendix C)
    composite_tf32: bool = True

    def _conditioner_gemms(self, xa, context):
        ct = self.conditioner_transform
        use_tf32 = (self.composite_tf32 and isinstance(self.transformer, RationalQuadratic) and xa.is_cuda
                    and context is None and type(ct) is FeedForward and ct.is_plain)
        if not use_tf32:
            return ct(xa, context=context)
        a = xa.reshape(-1, xa.shape[-1])
        for module in ct.sequential:
            if isinstance(module, nn.Linear):
                a = _TF32Linear.apply(a, module.weight, module.bias)
            elif isinstance(module, nn.Unflatten):
                continue
            else:
                a = module(a)
        return a.reshape(*xa.shape[:-1], -1)

    def _run_wide(self, x: torch.Tensor, direction: str):
        batch_shape = get_batch_shape(x, self.event_shape)
        xf = flatten_event(x, self.event_shape).reshape(-1, self.n_dim)
        seq = self.conditioner_transform.sequential
        n_bins, boundary = self._spline_args()
        y, log_det = _WideCoupling.apply(xf, seq[0].weight, seq[0].bias, seq[2].weight, seq[2].bias,
                                         self._tkind(direction), n_bins, boundary)
        return unflatten_event(y.reshape(*batch_shape, self.n_dim), self.event_shape), log_det.reshape(batch_shape)

    def _composite(self, x: torch.Tensor, context, direction: str):
        """Conditioner as library GEMMs, transformer as the stand-alone kernel (non-default configurations)."""
        if (self._wide or self._trains_wide()) and context is None and x.is_cuda and x.dtype == torch.float32:
            return self._run_wide(x, direction)
        batch_shape = get_batch_shape(x, self.event_shape)
        xf = flatten_event(x, self.event_shape)
        fn = self.transformer.forward if direction == 'forward' else self.transformer.inverse
        if isinstance(self.coupling, HalfSplit):
            ds = self.n_dim // 2
            xa, xb = xf[..., :ds], xf[..., ds:]
            h = self._conditioner_gemms(xa, context).view(*batch_shape, *self.transformer.parameter_shape)
            yb, log_det = fn(xb.contiguous(), h)
            out = torch.cat([xa, yb.reshape(*batch_shape, -1)], dim=-1)
        else:
            src = self.coupling.source_mask.view(-1).to(x.device)
            tgt = self.coupling.target_mask.view(-1).to(x.device)
            h = self.conditioner_transform(xf[..., src], context=context).view(*batch_shape,
                                                                               *self.transformer.parameter_shape)
            yb, log_det = fn(xf[..., tgt].contiguous(), h)
            out = xf.clone()
            out[..., tgt] = yb
        return unflatten_event(out, self.event_shape), log_det

    def _run_direction(self, x: torch.Tensor, context, direction: str):
        if context is not None:
            ops = self._lower_with_context(direction, context) if x.is_cuda else None
            if ops is None:
                return self._composite(x, context, direction)
            batch_shape = get_batch_shape(x, self.event_shape)
            y2, ld, _ = prog.run_program(ops, x.reshape(-1, self.n_dim))
            return y2.reshape(x.shape), ld.reshape(batch_shape)
        fused = self._fusable and not self._trains_wide()
        return self._run_fused(x, direction) if fused else self._composite(x, context, direction)

    def forward(self, x: torch.Tensor, context: torch.Tensor = None) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run_direction(x, context, 'forward')

    def inverse(self, z: torch.Tensor, context: torch.Tensor = None) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run_direction(z, context, 'inverse')


class MaskedAutoregressiveBijection(AutoregressiveBijection):
    """MADE conditioner + scalar transformer.  ``forward`` is one pass; ``inverse`` is sequential over the
    event dimensions -- the reference re-runs the full network D times (layers_base.py:213-223); here it is one
    persistent kernel with incrementally updated hidden pre-activations (cost of one pass)."""

    #: reproduce the reference's last-iteration log-det in the sequential direction (SURVEY Appendix B.3)
    sequential_log_det_reference_quirk: bool = True

    def __init__(self, event_shape, transformer_class: Type[ScalarTransformer], context_shape=None,
                 transformer_kwargs: dict = None, conditioner_kwargs: dict = None, l2_regularization: bool = True,
                 **kwargs):
        conditioner_kwargs, transformer_kwargs = conditioner_kwargs or {}, transformer_kwargs or {}
        transformer = transformer_class(event_shape=event_shape, **transformer_kwargs)
        conditioner_transform = MADE(input_event_shape=event_shape, transformed_event_shape=event_shape,
                                     parameter_shape_per_element=transformer.parameter_shape_per_element,
                                     context_shape=context_shape, **conditioner_kwargs)
        super().__init__(transformer.event_shape, transformer, conditioner_transform,
                         l2_regularization=l2_regularization, **kwargs)
        ct = conditioner_transform
        if not (ct.n_layers == 2 and ct.is_plain and isinstance(transformer, ScalarTransformer)):
            raise NotImplementedError('masked autoregressive layers are implemented for the default MADE depth '
                                      '(n_layers=2) and predicted parameters only')
        # transformers without a whole-flow kernel (splines with n_bins != 8) run as a composite: masked conditioner
        # GEMMs + the stand-alone transformer kernel, the sequential direction as the reference's D-step loop
        # With a context, MADE concatenates it to x and gives the context columns degrees n_dim+1.. (transforms.py:
        # 222-226).  Hidden units that see a context column therefore have a degree > n_dim, and the strict output mask
        # (transforms.py:254) cuts every such unit off from every output: the context provably never reaches h.  The
        # fused kernels therefore use the first n_dim input columns only; the check below guards the argument.
        self._n_context_cols = ct.n_input_event_dims - self.n_dim
        if self._n_context_cols > 0:
            m1, m2 = ct.sequential[0].mask, ct.sequential[2].mask
            sees_context = (m1[:, self.n_dim:] != 0).any(dim=1).float()
            if float((m2 @ sees_context).abs().sum()) != 0.0:
                raise NotImplementedError('MADE masks let the context reach the outputs; this configuration is not fused')
        fin = ct.sequential[0].mask[:, :self.n_dim].sum(dim=1).to(torch.int32)
        self.register_buffer('_fin_steps', fin, persistent=False)
        # event sizes whose backward tile no longer fits shared memory (D >= 768) run as a composite, see _composite_*
        # (linear rational spline layers with a context stay composite)
        self._fusable = (_transformer_fusable(transformer)
                         and not (isinstance(transformer, LinearRational) and self._n_context_cols > 0)
                         and _fits_fused_kernel(self.n_dim, ct.n_hidden, N.OP_MADE, transformer._tkind_forward,
                                                self._spline_args()[0]))

    def _lower(self, one_pass: bool, transformer_direction: str):
        seq = self.conditioner_transform.sequential
        n_bins, boundary = self._spline_args()
        flags = 0 if self.sequential_log_det_reference_quirk else N.FLAG_SEQ_LOGDET_EXACT
        w1, m1 = seq[0].weight, seq[0].mask
        if self._n_context_cols > 0:
            w1, m1 = w1[:, :self.n_dim], m1[:, :self.n_dim]
        consts = [m1, seq[2].mask] + ([] if one_pass else [self._fin_steps])
        return [prog.LoweredOp(kind=N.OP_MADE if one_pass else N.OP_MADE_SEQ, tkind=self._tkind(transformer_direction),
                               leafs=[w1, seq[0].bias, seq[2].weight, seq[2].bias], consts=consts,
                               n_hidden=seq[0].out_features, n_bins=n_bins, boundary=boundary, flags=flags, owner=self)]

    def lower(self, direction: str):
        if not self._fusable:
            return None
        return self._lower(True, 'forward') if direction == 'forward' else self._lower(False, 'inverse')

    def apply_conditioner_transformer(self, inputs, context, forward: bool = True):
        h = self.conditioner_transform(inputs, context)
        return self.transformer.forward(inputs, h) if forward else self.transformer.inverse(inputs, h)

    # -- composite path (layers too large for the fused kernels) ------------------------------------------------------
    def _composite_one_pass(self, x: torch.Tensor, context, transformer_forward: bool):
        """Masked conditioner as library GEMMs, transformer as the stand-alone kernel (layers_base.py:202-211)."""
        return self.apply_conditioner_transformer(x, context, forward=transformer_forward)

    def _composite_sequential(self, z: torch.Tensor, context, transformer_forward: bool):
        """The reference's D-step loop (layers_base.py:213-223), one dimension fixed per iteration.  With the default
        ``sequential_log_det_reference_quirk`` the log-det is the last iteration's, as in the reference; otherwise it is
        the exact one, evaluated by one extra pass in the opposite direction at the result."""
        batch_shape = get_batch_shape(z, self.event_shape)
        x = flatten_event(z, self.event_shape)
        log_det = None
        for i in range(self.n_dim):
            tmp, log_det = self.apply_conditioner_transformer(unflatten_event(x, self.event_shape), context,
                                                              forward=transformer_forward)
            tmp = flatten_event(tmp, self.event_shape)
            x = torch.cat([x[..., :i], tmp[..., i:i + 1], x[..., i + 1:]], dim=-1)
        out = unflatten_event(x, self.event_shape)
        if not self.sequential_log_det_reference_quirk:
            log_det = -self.apply_conditioner_transformer(out, context, forward=not transformer_forward)[1]
        return out, log_det.reshape(batch_shape)

    def forward(self, x: torch.Tensor, context: torch.Tensor = None) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run_fused(x, 'forward') if self._fusable else self._composite_one_pass(x, context, True)

    def inverse(self, z: torch.Tensor, context: torch.Tensor = None) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run_fused(z, 'inverse') if self._fusable else self._composite_sequential(z, context, False)


class InverseMaskedAutoregressiveBijection(MaskedAutoregressiveBijection):
    """forward = sequential direction (with transformer.inverse), inverse = one pass (layers_base.py:226-234)."""

    def lower(self, direction: str):
        if not self._fusable:
            return None
        return self._lower(False, 'inverse') if direction == 'forward' else self._lower(True, 'forward')

    def forward(self, x: torch.Tensor, context: torch.Tensor = None) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run_fused(x, 'forward') if self._fusable else self._composite_sequential(x, context, False)

    def inverse(self, z: torch.Tensor, context: torch.Tensor = None) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run_fused(z, 'inverse') if self._fusable else self._composite_one_pass(z, context, True)


class ElementwiseBijection(AutoregressiveBijection):
    """Per-element transformer with globally learned parameters ``value`` (layers_base.py:237-318).  The
    reference materialises ``value`` repeated over the batch (:300-303); the kernels broadcast it."""

    def __init__(self, event_shape, transformer_class: Type[ScalarTransformer], context_shape=None,
                 transformer_kwargs: dict = None, fill_value: Union[float, torch.Tensor] = None,
                 conditioner_transform_class: Type[ConditionerTransform] = Linear, conditioner_kwargs: dict = None,
                 **kwargs):
        transformer = transformer_class(event_shape=event_shape, **(transformer_kwargs or {}))
        if context_shape is None:
            if fill_value is None:
                value = torch.randn(*transformer.parameter_shape)
            elif isinstance(fill_value, torch.Tensor):
                if fill_value.shape != transformer.parameter_shape:
                    raise ValueError('Shape of fill_value must match the transformer parameter shape')
                value = fill_value
            else:
                value = torch.full(size=tuple(transformer.parameter_shape), fill_value=float(fill_value))
            super().__init__(event_shape=event_shape, context_shape=None, transformer=transformer,
                             conditioner_transform=None, **kwargs)
            self.register_parameter('value', nn.Parameter(value))
            self.use_global_parameters = True
        else:
            # parameters predicted from the context by a conditioner (default: one Linear layer), layers_base.py:281-296
            conditioner_transform = conditioner_transform_class(
                input_event_shape=None, context_shape=context_shape, parameter_shape=transformer.parameter_shape,
                **(conditioner_kwargs or {}))
            super().__init__(event_shape=event_shape, context_shape=context_shape, transformer=transformer,
                             conditioner_transform=conditioner_transform, **kwargs)
            self.register_buffer('value', torch.empty(size=()))
            self.use_global_parameters = False

    def prepare_h(self, context: torch.Tensor, batch_shape):
        """Global parameters: broadcast over the batch as a stride-0 view (no copy).  Context-conditioned: predicted."""
        if self.use_global_parameters:
            return self.value.expand(*batch_shape, *self.value.shape)
        if context is None:
            raise RuntimeError('Context must be provided')
        return self.conditioner_transform(x=None, context=context)

    #: BijectiveComposition hands the context to lower() (see _segments)
    lowers_with_context: bool = True
    #: context-conditioned layers join the flow program with per-row parameters (False: stand-alone transformer kernel)
    fuse_context: bool = True

    def lower(self, direction: str, context: torch.Tensor = None):
        tk = self._tkind(direction)
        if tk not in (N.T_AFFINE_FWD, N.T_AFFINE_INV) or not _fits_fused_kernel(self.n_dim, 1):
            return None
        if self.use_global_parameters:
            return [prog.LoweredOp(kind=N.OP_ELEMENTWISE, tkind=tk, leafs=[self.value], owner=self)]
        if context is None or not self.fuse_context or not context.is_cuda or context.dtype != torch.float32:
            return None
        # context-conditioned (layers_base.py:281-296): the layer's own conditioner predicts (B, D, 2) parameters from the
        # context; the op carries them per row (B2F_FLAG_ROW_BIAS on an elementwise op) and the layer stays inside the program
        h = self.conditioner_transform(x=None, context=context).reshape(-1, self.n_dim, 2)
        return [prog.LoweredOp(kind=N.OP_ELEMENTWISE, tkind=tk, leafs=[h], flags=N.FLAG_ROW_BIAS, owner=self)]

    def column_op(self, direction: str):
        """(kind, value) of this layer as one op of a per-column run (csrc/b2f_colrun.cu), for event sizes the whole-flow
        kernels do not take; None if the layer is not a global-parameter affine map."""
        tk = self._tkind(direction)
        if self.use_global_parameters and tk in (N.T_AFFINE_FWD, N.T_AFFINE_INV) and self.n_dim % 4 == 0 \
                and self.value.is_cuda and self.value.dtype == torch.float32:
            return (N.COL_AFFINE_FWD if tk == N.T_AFFINE_FWD else N.COL_AFFINE_INV, self.value)
        return None

    def _run_direction(self, x, direction, context=None):
        if self.lower(direction) is not None:
            return self._run_fused(x, direction)
        batch_shape = get_batch_shape(x, self.event_shape)
        h = self.prepare_h(context, batch_shape)       # stride-0 view (global) or per-sample parameters (context)
        fn = self.transformer.forward if direction == 'forward' else self.transformer.inverse
        return fn(x, h)

    def forward(self, x: torch.Tensor, context: torch.Tensor = None) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run_direction(x, "forward", context)

    def inverse(self, z: torch.Tensor, context: torch.Tensor = None) -> Tuple[torch.Tensor, torch.Tensor]:
        return self._run_direction(z, "inverse", context)
