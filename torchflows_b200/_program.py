"""Lowering of bijection layers to libb2f flow programs and the autograd bridge.

A *lowered op* describes one layer applied in one direction:

    LoweredOp(kind, tkind, leafs=[module parameters], consts=[buffers], n_hidden, n_bins, boundary, flags, owner)

``leafs`` are the reference-layout parameters (what ``state_dict`` holds); the kernels want the last
Linear weight in *tile layout* ([element][hidden][param], see include/b2f.h) and MADE weights pre-multiplied
by their masks, so ``kernel_params`` derives those once per parameter version and caches them on the layer.
``FlowFunction`` is the single ``torch.autograd.Function`` through which every fused call goes.
"""
import dataclasses
import os
import warnings
from dataclasses import dataclass, field
from typing import List, Optional, Sequence

import torch

from . import _native as N
from . import _tca, _tcm, _tcq


@dataclass
class LoweredOp:
    kind: int
    tkind: int = 0
    leafs: List[torch.Tensor] = field(default_factory=list)    # differentiable inputs (reference layout)
    consts: List[torch.Tensor] = field(default_factory=list)   # masks, finalisation steps
    n_hidden: int = 0
    n_bins: int = 0
    boundary: float = 0.0
    flags: int = 0
    owner: Optional[torch.nn.Module] = None                    # cache holder


def params_per_element(tkind: int, n_bins: int) -> int:
    if tkind in (N.T_LRS_FWD, N.T_LRS_INV):
        return 4 * n_bins
    return {N.T_SHIFT_ADD: 1, N.T_SHIFT_SUB: 1, N.T_AFFINE_FWD: 2, N.T_AFFINE_INV: 2}.get(tkind, 3 * n_bins - 1)


#: spline transformer kinds: their sequential MADE direction reports the reference's last-iteration log-det by default
SPLINE_TKINDS = (N.T_RQ_FWD, N.T_RQ_INV, N.T_LRS_FWD, N.T_LRS_INV)


def padded(P: int) -> int:
    return P if P <= 2 else (P + 3) // 4 * 4


def to_tile_layout(W2: torch.Tensor, n_elem: int, P: int) -> torch.Tensor:
    """(n_elem*P, H) with row index e*P+p  ->  (n_elem, H, PP) zero padded, contiguous."""
    H = W2.shape[1]
    t = W2.reshape(n_elem, P, H).transpose(1, 2)
    PP = padded(P)
    if PP != P:
        t = torch.nn.functional.pad(t, (0, PP - P))
    return t.contiguous()


def from_tile_layout(G: torch.Tensor, n_elem: int, P: int) -> torch.Tensor:
    """Inverse of to_tile_layout for gradients: (n_elem, H, PP) -> (n_elem*P, H)."""
    return G[..., :P].transpose(1, 2).reshape(n_elem * P, G.shape[1])


def kernel_params(op: LoweredOp) -> List[Optional[torch.Tensor]]:
    """Tensors in the layout b2f_op.p[] expects (cached per parameter version on op.owner)."""
    if op.kind == N.OP_FLIP:
        return []
    if op.kind == N.OP_ELEMENTWISE:
        return [op.leafs[0].detach().reshape(-1, 2).contiguous()]
    W1, b1, W2, b2 = op.leafs
    if op.flags & N.FLAG_ROW_BIAS:
        # context-conditioned coupling: W1 is the x_A block of the first layer and b1 the per-row hidden bias, both made for
        # this call (never cached: a recycled allocation would alias a stale entry); only the output layer's layout is cached
        P = params_per_element(op.tkind, op.n_bins)
        n_elem = W2.shape[0] // P
        cache = getattr(op.owner, '_b2f_cache', None)
        if cache is None:
            cache = {}
            if op.owner is not None:
                object.__setattr__(op.owner, '_b2f_cache', cache)
        key, ver = ('rowbias', op.kind, op.tkind), ((W2.data_ptr(), W2._version), (b2.data_ptr(), b2._version))
        hit = cache.get(key)
        if hit is None or hit[0] != ver:
            with torch.no_grad():
                hit = (ver, [to_tile_layout(W2.detach(), n_elem, P), b2.detach().contiguous()])
            cache[key] = hit
        return [W1.detach().contiguous(), b1.detach().contiguous(), hit[1][0], hit[1][1]]
    key = (op.kind, op.tkind)
    ver = tuple((t.data_ptr(), t._version) for t in op.leafs)
    cache = getattr(op.owner, '_b2f_cache', None)
    if cache is None:
        cache = {}
        if op.owner is not None:
            object.__setattr__(op.owner, '_b2f_cache', cache)
    hit = cache.get(key)
    if hit is not None and hit[0] == ver:
        return hit[1]
    P = params_per_element(op.tkind, op.n_bins)
    n_elem = W2.shape[0] // P
    with torch.no_grad():
        if op.kind == N.OP_COUPLING:
            out = [W1.detach().contiguous(), b1.detach().contiguous(), to_tile_layout(W2.detach(), n_elem, P),
                   b2.detach().contiguous()]
        else:
            m1, m2 = op.consts[0], op.consts[1]
            out = [(W1.detach() * m1).contiguous(), b1.detach().contiguous(),
                   to_tile_layout(W2.detach() * m2, n_elem, P), b2.detach().contiguous()]
            if op.kind == N.OP_MADE_SEQ:
                out.append(op.consts[2])
    cache[key] = (ver, out)
    return out


def round_tf32(t: torch.Tensor) -> torch.Tensor:
    """Round fp32 to the nearest tf32 value (10 explicit mantissa bits), kept in fp32 storage."""
    return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def umma_canonical(mat: torch.Tensor) -> torch.Tensor:
    """[rows, K] -> flat tensor in the K-major no-swizzle UMMA operand order of csrc/b2f_umma.cuh:
    float offset(row, k) = (row//8)*K*8 + (k//4)*32 + (row%8)*4 + k%4."""
    rows, K = mat.shape
    return mat.reshape(rows // 8, 8, K // 4, 4).permute(0, 2, 1, 3).contiguous().reshape(-1)


_TC_GEOM = {  # transformer kind -> (parameter columns per element CPE, elements per GEMM2 chunk EPC, 3xTF32 split)
    N.T_RQ_FWD: (24, 8, False), N.T_RQ_INV: (24, 8, False),
    N.T_AFFINE_FWD: (2, 64, True), N.T_AFFINE_INV: (2, 64, True),
    N.T_SHIFT_ADD: (1, 128, True), N.T_SHIFT_SUB: (1, 128, True),
}


def tc_eligible(op: LoweredOp, D: int) -> bool:
    """Mirror of try_launch_flow_tc's per-op conditions (csrc/b2f_flow_tc.cu)."""
    if op.kind not in (N.OP_COUPLING, N.OP_MADE) or op.tkind not in _TC_GEOM or D % 16 != 0 or D < 32:
        return False
    if op.flags & N.FLAG_ROW_BIAS:           # context-conditioned layer (per-row hidden bias): generic kernel
        return False
    x3 = _TC_GEOM[op.tkind][2]
    if x3:
        return D <= 128 and 1 <= op.n_hidden <= 20
    return op.n_bins == 8 and D <= 256 and 1 <= op.n_hidden <= 30


def tc_operands(op: LoweredOp, flipped: bool, D: int):
    """Tensor-core operand layouts of a coupling layer (include/b2f.h, B2F_FLAG_TC_OPERANDS), cached per parameter
    version: W1c [32 x K1] and W2c [chunks][N2 x K2] with the bias folded in as two K columns.  Affine / shift layers
    use the 3xTF32 split along K: [w_hi | w_lo | w_hi]."""
    W1, b1, W2, b2 = op.leafs
    key = ('tc', bool(flipped))
    ver = tuple((t.data_ptr(), t._version) for t in op.leafs)
    cache = getattr(op.owner, '_b2f_cache', None)
    if cache is None:
        cache = {}
        object.__setattr__(op.owner, '_b2f_cache', cache)
    hit = cache.get(key)
    if hit is not None and hit[0] == ver:
        return hit[1]
    cpe, epc, x3 = _TC_GEOM[op.tkind]
    made = op.kind == N.OP_MADE
    with torch.no_grad():
        if made:       # masks folded into the weight tiles
            W1, W2 = W1.detach() * op.consts[0], W2.detach() * op.consts[1]
        H = W1.shape[0]
        Ks = D if made else D // 2           # source columns (K of GEMM1), in PHYSICAL order
        Dh = D if made else D // 2           # target elements
        P = params_per_element(op.tkind, op.n_bins)
        w1 = W1.detach().flip(1) if flipped else W1.detach()
        w1_hi = round_tf32(w1)
        W1p = W1.new_zeros(32, (3 if x3 else 1) * Ks)
        W1p[:H, :Ks] = w1_hi
        if x3:
            W1p[:H, Ks:2 * Ks] = round_tf32(w1 - w1_hi)
            W1p[:H, 2 * Ks:] = w1_hi
        w1c = umma_canonical(W1p)
        K2 = ((3 if x3 else 1) * H + 2 + 7) // 8 * 8
        n_chunks = (Dh + epc - 1) // epc
        M = W2.new_zeros(n_chunks * epc, cpe, K2)
        w2 = W2.detach().reshape(Dh, P, H)
        w2_hi = round_tf32(w2)
        M[:Dh, :P, :H] = w2_hi
        kb = H
        if x3:
            M[:Dh, :P, H:2 * H] = round_tf32(w2 - w2_hi)
            M[:Dh, :P, 2 * H:3 * H] = w2_hi
            kb = 3 * H
        bias = b2.detach().reshape(Dh, P)
        b_hi = round_tf32(bias)
        M[:Dh, :P, kb] = b_hi
        M[:Dh, :P, kb + 1] = round_tf32(bias - b_hi)
        # every chunk [N2 x K2] into canonical order in one go: (chunk, row/8, k/4, row%8, k%4)
        w2c = M.reshape(n_chunks, (epc * cpe) // 8, 8, K2 // 4, 4).permute(0, 1, 3, 2, 4).contiguous().reshape(-1)
    out = (w1c, w2c)
    cache[key] = (ver, out)
    return out


def seq_fold_eligible(ops: Sequence[LoweredOp], D: int, flags: int) -> bool:
    """Can the sequential spline layers of this program run in the folded formulation (rows kernel, B2F_FLAG_SEQ_FOLDED)?
    Cheap mirror of the rows kernel's main conditions; the library rejects the rest and the caller retries unfolded."""
    if (flags & N.FLOW_MODE_PRECISE) or os.environ.get('B2F_DISABLE_ROWS') or os.environ.get('B2F_NO_SEQ_FOLD') \
            or D % 8 != 0 or D > 1024:
        return False
    seq = [op for op in ops if op.kind == N.OP_MADE_SEQ and op.tkind in (N.T_RQ_FWD, N.T_RQ_INV)]
    return bool(seq) and all(op.n_bins == 8 and op.n_hidden <= 15 and not getattr(op.owner, '_b2f_no_seq_fold', False)
                             for op in seq)


def seq_folded_operands(op: LoweredOp):
    """[element][hidden][24] folded output layer and [element][24] folded bias of a sequential spline MADE layer (include/b2f.h,
    B2F_FLAG_SEQ_FOLDED; columns of csrc/b2f_rqfast.cuh), masks multiplied in, cached per parameter version."""
    W1, b1, W2, b2 = op.leafs
    ver = tuple((t.data_ptr(), t._version) for t in (W2, b2))
    cache = getattr(op.owner, '_b2f_cache', None)
    if cache is None:
        cache = {}
        if op.owner is not None:
            object.__setattr__(op.owner, '_b2f_cache', cache)
    key = ('seqfold', op.kind, op.tkind)
    hit = cache.get(key)
    if hit is not None and hit[0] == ver:
        return hit[1]
    with torch.no_grad():
        n_elem = W2.shape[0] // 23
        Wf, bf = _tcq.fold_output_layer(W2.detach().float() * op.consts[1].to(W2.device), b2.detach().float(), n_elem)
        out = (Wf.permute(0, 2, 1).contiguous(), bf.contiguous())
    cache[key] = (ver, out)
    return out


def op_dicts(ops: Sequence[LoweredOp], grads: Optional[List[List[Optional[torch.Tensor]]]] = None,
             D: Optional[int] = None, tcq_plan: Optional['_tcq.Plan'] = None, tca_plan=None, tcm_plan=None,
             fold_seq: bool = False):
    """b2f_op descriptors of a program.  ``tcq_plan``: the program is laid out for the second-generation spline kernel
    (csrc/b2f_flow_tcq.cu): every coupling op carries its blob in p[4], the first one the program blob in p[5]."""
    out = []
    flipped = False
    n_coupling = 0
    for i, op in enumerate(ops):
        p, flags = list(kernel_params(op)), op.flags
        if op.kind == N.OP_FLIP:
            flipped = not flipped
        elif tcm_plan is not None and op.kind == N.OP_MADE:           # one-pass MADE spline kernel (csrc/b2f_flow_tcm.cu)
            p = p[:4] + [tcm_plan.layer_blobs[n_coupling], tcm_plan.program_blob if n_coupling == 0 else None]
            flags |= N.FLAG_TCM_OPERANDS
            n_coupling += 1
        elif tcq_plan is not None and op.kind == N.OP_COUPLING:
            p = p[:4] + [tcq_plan.layer_blobs[n_coupling], tcq_plan.program_blob if n_coupling == 0 else None]
            flags |= N.FLAG_TCQ_OPERANDS
            n_coupling += 1
        elif tca_plan is not None and op.kind == N.OP_COUPLING:       # multi-tile affine kernel (csrc/b2f_flow_tca.cu)
            p = p[:4] + [tca_plan.layer_blobs[n_coupling], tca_plan.program_blob if n_coupling == 0 else None]
            flags |= N.FLAG_TCA_OPERANDS
            n_coupling += 1
        elif fold_seq and grads is None and op.kind == N.OP_MADE_SEQ and op.tkind in (N.T_RQ_FWD, N.T_RQ_INV):
            wf, bf = seq_folded_operands(op)
            p = p[:2] + [wf, bf] + p[4:]
            flags |= N.FLAG_SEQ_FOLDED
        elif D is not None and grads is None and tc_eligible(op, D):
            w1c, w2c = tc_operands(op, flipped, D)
            p = p[:4] + [w1c, w2c]
            flags |= N.FLAG_TC_OPERANDS | (N.FLAG_TC_FLIPPED if flipped else 0)
        out.append(dict(kind=op.kind, tkind=op.tkind, n_hidden=op.n_hidden, n_bins=op.n_bins, boundary=op.boundary,
                        flags=flags, p=p, g=(grads[i] if grads is not None else [])))
    return out


class _Cfg:
    """Non-tensor arguments of FlowFunction."""

    def __init__(self, ops, want_log_prob, base_loc, base_log_scale, flags):
        self.ops, self.want_log_prob = list(ops), want_log_prob
        self.base_loc, self.base_log_scale, self.flags = base_loc, base_log_scale, flags


class FlowFunction(torch.autograd.Function):
    """y, log_det, log_prob = program(x).  Forward: one b2f_flow_apply launch.  Backward: one
    b2f_flow_backward launch that recomputes the conditioner outputs per tile (h is never materialised)."""

    @staticmethod
    def forward(ctx, x2, cfg: _Cfg, *leafs):
        # the forward kernel keeps every conditioner layer's input for the backward kernel when it can (tensor-core
        # kernel): the backward pass then starts from the output y and skips its own forward recompute
        y, ld, lp, ws = N.flow_apply(op_dicts(cfg.ops, D=x2.shape[1]), x2, True, True, cfg.want_log_prob, cfg.base_loc,
                                     cfg.base_log_scale, cfg.flags, save_layer_inputs=not (cfg.flags & N.FLOW_LOGP_OF_INPUT))
        ctx.cfg = cfg
        ctx.ws = ws
        ctx.save_for_backward(x2 if ws is None else y, *leafs)
        if lp is None:
            lp = x2.new_empty(0)
            ctx.mark_non_differentiable(lp)
        return y, ld, lp

    @staticmethod
    def backward(ctx, gy, gld, glp):
        cfg = ctx.cfg
        x2 = ctx.saved_tensors[0]
        ops = cfg.ops
        for op in ops:
            if op.kind == N.OP_MADE_SEQ and op.tkind in SPLINE_TKINDS and not (op.flags & N.FLAG_SEQ_LOGDET_EXACT):
                raise NotImplementedError(
                    'gradients through the sequential direction of a spline MADE layer are implemented for the exact '
                    'log-determinant only: set layer.sequential_log_det_reference_quirk = False (the reference returns '
                    'the log-det of its last iteration, SURVEY Appendix B.3)')
        if cfg.flags & N.FLOW_LOGP_OF_INPUT:
            raise NotImplementedError('the fused LOGP_OF_INPUT variant is inference-only; with gradients Flow.sample '
                                      'evaluates the base density separately')
        dev = x2.device
        grads, leaf_grads = [], []
        for op in ops:
            kp = kernel_params(op)
            g = [None] * len(kp)
            if op.kind == N.OP_ELEMENTWISE:
                if op.leafs[0].requires_grad:
                    g[0] = torch.zeros_like(kp[0])
            elif op.kind in (N.OP_COUPLING, N.OP_MADE, N.OP_MADE_SEQ):
                if any(t.requires_grad for t in op.leafs):
                    g = [torch.zeros_like(t) for t in kp[:4]] + [None] * (len(kp) - 4)
            grads.append(g)
        B, D = x2.shape
        od = op_dicts(ops, grads)          # holds the per-call operand tensors (row-bias ops) alive until the launch below
        arr = N.make_ops(od)
        flags = cfg.flags
        if ctx.ws is not None:
            ws, flags = ctx.ws, flags | N.FLOW_WS_FILLED       # x2 is the forward output here
        else:
            ws_bytes = N.lib().b2f_flow_backward_workspace(arr, len(ops), B, D)
            ws = torch.empty(max(int(ws_bytes), 4) // 4, device=dev, dtype=torch.float32)
        need_gx = ctx.needs_input_grad[0]
        gx = torch.empty_like(x2)

        def c(t):
            return None if t is None else t.contiguous()
        glp_ = c(glp) if (cfg.want_log_prob and glp is not None) else None
        with torch.cuda.device(dev):
            N.check(N.lib().b2f_flow_backward(arr, len(ops), N.ptr(x2), N.ptr(c(gy)), N.ptr(c(gld)), N.ptr(glp_),
                                              N.ptr(cfg.base_loc), N.ptr(cfg.base_log_scale), N.ptr(gx), N.ptr(ws),
                                              B, D, flags, N.stream_ptr(dev)))
        for op, g in zip(ops, grads):
            if op.kind == N.OP_ELEMENTWISE:
                leaf_grads.append(None if g[0] is None else g[0].reshape(op.leafs[0].shape))
            elif op.kind in (N.OP_COUPLING, N.OP_MADE, N.OP_MADE_SEQ):
                if g[0] is None:
                    leaf_grads.extend([None] * 4)
                    continue
                P = params_per_element(op.tkind, op.n_bins)
                n_elem = op.leafs[2].shape[0] // P
                gW1, gb1, gW2, gb2 = g[0], g[1], from_tile_layout(g[2], n_elem, P), g[3]
                if op.kind in (N.OP_MADE, N.OP_MADE_SEQ):
                    gW1, gW2 = gW1 * op.consts[0], gW2 * op.consts[1]
                leaf_grads.extend([gW1, gb1, gW2, gb2])
        del od
        return (gx if need_gx else None, None, *leaf_grads)


_warned_seq_exact = False
_MODE_FLAGS = {'default': 0, 'precise': N.FLOW_MODE_PRECISE, 'fast': N.FLOW_MODE_FAST_KNOTS}
_mode = 'default'


def set_math_mode(mode: str) -> str:
    """Arithmetic mode of the fused flow kernels (process-wide); returns the previous mode.
    'default': deterministic spline knots (bin indices bit-reproducible against the CPU oracle), SFU approximations
               only after the bin search.
    'precise': libm-grade exp / log / division everywhere.
    'fast'   : additionally takes the softmax exponentials of the knots from the SFU: fewest instructions, same value
               tolerances, bin indices may differ from the oracle at exact ties."""
    global _mode
    if mode not in _MODE_FLAGS:
        raise ValueError(f'mode must be one of {sorted(_MODE_FLAGS)}')
    previous, _mode = _mode, mode
    return previous


def run_program(ops: Sequence[LoweredOp], x2: torch.Tensor, want_log_prob=False, base_loc=None, base_log_scale=None,
                flags=0, want_y=True):
    """x2: (B, D).  Returns y, log_det, log_prob (None unless requested).  Programs longer than B2F_MAX_OPS are
    chained (log-dets add, the base density is evaluated by the last launch)."""
    x2 = N.require_cuda_f32(x2, 'input')
    ops = list(ops)
    flags |= _MODE_FLAGS[_mode]
    if len(ops) > N.MAX_OPS:
        if flags & N.FLOW_LOGP_OF_INPUT:
            raise N.B2FError('program too long for LOGP_OF_INPUT')
        y, ld_total = x2, None
        chunks = [ops[i:i + N.MAX_OPS] for i in range(0, len(ops), N.MAX_OPS)]
        for ci, chunk in enumerate(chunks):
            last = ci == len(chunks) - 1
            y, ld, lp = run_program(chunk, y, want_log_prob and last, base_loc, base_log_scale, flags)
            ld_total = ld if ld_total is None else ld_total + ld
        if want_log_prob:
            lp = lp - ld + ld_total
        return y, ld_total, (lp if want_log_prob else None)
    leafs = [t for op in ops for t in op.leafs]
    needs_grad = torch.is_grad_enabled() and (x2.requires_grad or any(t.requires_grad for t in leafs))
    if needs_grad:
        # The reference's last-iteration log-det of a sequential spline layer (SURVEY Appendix B.3) has no fused gradient:
        # when gradients are needed the layer is lowered with the exact log-determinant instead (same value to ~1e-5 at
        # initialisation, a well-defined objective afterwards), so that fit() / variational_fit() work out of the box.
        quirky = [i for i, op in enumerate(ops) if op.kind == N.OP_MADE_SEQ and op.tkind in SPLINE_TKINDS
                  and not (op.flags & N.FLAG_SEQ_LOGDET_EXACT)]
        if quirky:
            global _warned_seq_exact
            if not _warned_seq_exact:
                _warned_seq_exact = True
                warnings.warn('gradients through the sequential direction of a spline masked-autoregressive layer use the '
                              'exact log-determinant (the reference reports the log-det of its last iteration, which has '
                              'no fused gradient); set layer.sequential_log_det_reference_quirk = False to use the exact '
                              'value for inference as well')
            for i in quirky:
                ops[i] = dataclasses.replace(ops[i], flags=ops[i].flags | N.FLAG_SEQ_LOGDET_EXACT)
        y, ld, lp = FlowFunction.apply(x2, _Cfg(ops, want_log_prob, base_loc, base_log_scale, flags), *leafs)
        return y, ld, (lp if want_log_prob else None)
    D = x2.shape[1]
    plan = None
    if (not (flags & N.FLOW_MODE_PRECISE) and not os.environ.get('B2F_DISABLE_TCQ') and not os.environ.get('B2F_DISABLE_TC')
            and _tcq.eligible(ops, D)):
        plan = _tcq.cached_plan(ops, D, base_loc, base_log_scale)
    fold = seq_fold_eligible(ops, D, flags)
    try:
        y, ld, lp = N.flow_apply(op_dicts(ops, D=D, tcq_plan=plan, tca_plan=_tca_plan(ops, D, base_loc, base_log_scale, flags),
                                          tcm_plan=_tcm_plan(ops, D, base_loc, base_log_scale, flags), fold_seq=fold),
                                 x2.detach(), want_y, True, want_log_prob, base_loc, base_log_scale, flags)
    except N.B2FError as e:
        if not fold or 'B2F_FLAG_SEQ_FOLDED' not in str(e):
            raise
        _no_seq_fold(ops)              # the rows kernel does not take this program: plain operands from now on
        y, ld, lp = N.flow_apply(op_dicts(ops, D=D), x2.detach(), want_y, True, want_log_prob, base_loc, base_log_scale, flags)
    return y, ld, lp


def _no_seq_fold(ops):
    for op in ops:
        if op.kind == N.OP_MADE_SEQ and op.owner is not None:
            object.__setattr__(op.owner, '_b2f_no_seq_fold', True)


def _tcm_plan(ops, D, base_loc, base_log_scale, flags):
    """Operand plan of the one-pass MADE spline kernel if the program is one it takes, else None."""
    if (flags & N.FLOW_MODE_PRECISE) or os.environ.get('B2F_DISABLE_TCM') or os.environ.get('B2F_DISABLE_TC') \
            or not _tcm.eligible(ops, D):
        return None
    return _tcm.cached_plan(ops, D, base_loc, base_log_scale)


def _tca_plan(ops, D, base_loc, base_log_scale, flags):
    """Operand plan of the multi-tile affine kernel if the program is one it takes, else None."""
    if (flags & N.FLOW_MODE_PRECISE) or os.environ.get('B2F_DISABLE_TCA') or os.environ.get('B2F_DISABLE_TC') \
            or not _tca.eligible(ops, D):
        return None
    return _tca.cached_plan(ops, D, base_loc, base_log_scale)


# ---- Flow.sample with the library's own base draws (b2f_flow_sample, csrc/b2f_philox.cuh) -----------------------------------
def next_noise_stream(device=None, n_elements: int = 0):
    """(seed, offset) of the next base draws: a fresh 62-bit Philox key from torch's CPU generator per call -- the stream the
    reference itself consumes (gaussian.py:42 draws torch.randn on the CPU) -- so torch.manual_seed makes sampling
    reproducible and re-seeding restarts it; no device synchronisation."""
    return int(torch.randint(0, 2 ** 62, (1,), dtype=torch.int64).item()), 0


def run_sample_program(ops: Sequence[LoweredOp], B: int, D: int, device, want_log_prob=False, base_loc=None,
                       base_log_scale=None, seed=None, offset=0):
    """Inverse-direction program applied to base draws made by the library: returns (x:(B, D), log_prob or None) where
    log_prob = base density of the draw + log_det (Flow.sample(return_log_prob=True), flows.py:710-712).  Inference only."""
    ops = list(ops)
    flags = _MODE_FLAGS[_mode] | N.FLOW_LOGP_OF_INPUT
    if seed is None:
        seed, offset = next_noise_stream(device, B * D)
    plan = None
    if (not (flags & N.FLOW_MODE_PRECISE) and not os.environ.get('B2F_DISABLE_TCQ') and not os.environ.get('B2F_DISABLE_TC')
            and _tcq.eligible(ops, D)):
        plan = _tcq.cached_plan(ops, D, base_loc, base_log_scale)
    tca = _tca_plan(ops, D, base_loc, base_log_scale, flags) if plan is None else None
    tcm = _tcm_plan(ops, D, base_loc, base_log_scale, flags) if plan is None and tca is None else None
    fold = seq_fold_eligible(ops, D, flags)
    try:
        return N.flow_sample(op_dicts(ops, D=D, tcq_plan=plan, tca_plan=tca, tcm_plan=tcm, fold_seq=fold), B, D, device,
                             want_log_prob, base_loc, base_log_scale, flags, seed, offset,
                             in_kernel=plan is not None or tca is not None or tcm is not None)
    except N.B2FError as e:
        if not fold or 'B2F_FLAG_SEQ_FOLDED' not in str(e):
            raise
        _no_seq_fold(ops)
        return N.flow_sample(op_dicts(ops, D=D), B, D, device, want_log_prob, base_loc, base_log_scale, flags, seed, offset)


# ---- runs of per-column layers outside whole-flow programs (csrc/b2f_colrun.cu) ---------------------------------------------
class ColumnRunFunction(torch.autograd.Function):
    """y = run(x), log_det_sum (one float, the same log-determinant for every row) of a run of ElementwiseAffine / ActNorm /
    ReversePermutation layers at an event size the whole-flow kernels do not take; one pass over the batch each way."""

    @staticmethod
    def forward(ctx, x2, kinds, *values):
        y, lds = N.column_run_apply(kinds, values, x2)
        ctx.kinds = kinds
        ctx.n_values = len(values)
        ctx.save_for_backward(x2, *[v for v in values if v is not None])
        ctx.present = [v is not None for v in values]
        return y, lds

    @staticmethod
    def backward(ctx, gy, g_lds):
        saved = ctx.saved_tensors
        x2, it = saved[0], iter(saved[1:])
        values = [next(it) if p else None for p in ctx.present]
        need = [ctx.needs_input_grad[2 + i] for i in range(ctx.n_values)]
        if gy is None:
            gy = torch.zeros_like(x2)
        gx, gvalues = N.column_run_backward(ctx.kinds, values, need, x2, gy.contiguous(), g_lds)
        return (gx, None) + tuple(gvalues)


def run_column_ops(col_ops, x2: torch.Tensor):
    """col_ops: [(N.COL_* kind, value tensor or None)] in application order.  Returns (y, log_det:(B,))."""
    x2 = N.require_cuda_f32(x2, 'input')
    log_det = None
    for i in range(0, len(col_ops), N.COL_MAX_OPS):
        chunk = col_ops[i:i + N.COL_MAX_OPS]
        kinds = tuple(k for k, _ in chunk)
        values = [v for _, v in chunk]
        x2, lds = ColumnRunFunction.apply(x2, kinds, *values)
        log_det = lds if log_det is None else log_det + lds
    return x2, log_det.expand(x2.shape[0])
