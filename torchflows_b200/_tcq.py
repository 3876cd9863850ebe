"""Operand layout of the spline-coupling tensor-core kernel (csrc/b2f_flow_tcq.cu, include/b2f.h B2F_FLAG_TCQ_OPERANDS).

The kernel runs a whole CouplingRQNSF-style program (ElementwiseAffine / ActNorm, ReversePermutation, RQS coupling layers:
architectures.py:44-54 of the reference) and wants everything that does not depend on the batch precomputed:

* every run of elementwise layers is an affine map per column; it is never executed as a pass of its own.  It is
  applied where the column is touched anyway: when a coupling layer reads its target element (``pre``), when it writes
  it back (``post`` = the run that follows the layer), when the base density is accumulated (``fin``), or -- for the
  half that feeds the conditioner -- in one materialisation pass over that half (``src``);
* the ReversePermutation only decides which *physical* half is the source: weights are permuted instead of data;
* the last Linear of the conditioner is folded into the 24 columns per element the spline epilogue consumes
  (csrc/b2f_rqfast.cuh): log2(e) * u_x, log2(e)/1000 * u_y, differences of the padded derivative logits.

All of it is computed with torch ops on the device (no host synchronisation) and cached per parameter version.
"""
import math
from typing import List, Optional, Sequence

import torch

from . import _native as N

LOG2E = 1.4426950408889634
RQ_EDGE_U = math.log(math.expm1(1 - 1e-5))      # rational_quadratic.py:38
AFFINE_C0 = math.log(1 - 1e-10)                 # affine.py:22
AFFINE_M = 1e-10
MAGIC = 0x51435442                              # 'BTCQ'
HDR = 8                                         # header floats (int32 bit patterns) in front of every layer blob
CPE = 24                                        # GEMM2 columns per element
EPC = 2                                         # elements per GEMM2 chunk (one chunk = one epilogue group's work unit)


def round_tf32(t: torch.Tensor) -> torch.Tensor:
    return ((t.contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


def canonical(mat: torch.Tensor) -> torch.Tensor:
    """[rows, K] -> K-major no-swizzle UMMA operand order (csrc/b2f_umma.cuh)."""
    rows, K = mat.shape
    return mat.reshape(rows // 8, 8, K // 4, 4).permute(0, 2, 1, 3).contiguous().reshape(-1)


def eligible(ops: Sequence, D: int) -> bool:
    """Mirror of try_launch_flow_tcq's conditions: spline coupling programs, D a multiple of 32 in [32, 256], both
    halves transformed by some layer, even number of flips."""
    if D % 32 != 0 or D < 32 or D > 256 or len(ops) > N.MAX_OPS:
        return False
    flip, written, n_c = False, set(), 0
    for op in ops:
        if op.kind == N.OP_FLIP:
            flip = not flip
        elif op.kind == N.OP_ELEMENTWISE:
            if op.tkind not in (N.T_AFFINE_FWD, N.T_AFFINE_INV) or (op.flags & N.FLAG_ROW_BIAS):
                return False
        elif op.kind == N.OP_COUPLING:
            if op.flags & N.FLAG_ROW_BIAS:              # context-conditioned layer: generic kernel
                return False
            if op.tkind not in (N.T_RQ_FWD, N.T_RQ_INV) or op.n_bins != 8 or not (1 <= op.n_hidden <= 30):
                return False
            written.add(0 if flip else 1)
            n_c += 1
        else:
            return False
    return (not flip) and n_c >= 1 and written == {0, 1}


def layer_blob_floats(D: int, H: int) -> int:
    Dh, K2 = D // 2, (H + 2 + 7) // 8 * 8
    return HDR + 32 * Dh + 32 + (Dh // EPC) * (EPC * CPE) * K2 + Dh * 8 + Dh * 2 + 4


def fold_output_layer(W2: torch.Tensor, b2: torch.Tensor, Dh: int):
    """(Dh*23, H), (Dh*23) in the reference layout (row = e*23 + p, rational_quadratic.py:125-127) ->
    Wf (Dh, 24, H), bf (Dh, 24): the folded columns of csrc/b2f_rqfast.cuh."""
    H = W2.shape[1]
    w = W2.reshape(Dh, 23, H).double()
    b = b2.reshape(Dh, 23).double()
    Wf = w.new_zeros(Dh, 24, H)
    bf = b.new_zeros(Dh, 24)
    Wf[:, 0:8] = LOG2E * w[:, 0:8]
    bf[:, 0:8] = LOG2E * b[:, 0:8]
    Wf[:, 8:16] = (LOG2E / 1000.0) * w[:, 8:16]
    bf[:, 8:16] = (LOG2E / 1000.0) * b[:, 8:16]
    # padded derivative logits relative to c: a = [c, u_d, c] / 1000   (the pad value is divided by 1000 as well)
    aw = w.new_zeros(Dh, 9, H)
    ab = b.new_zeros(Dh, 9)
    aw[:, 1:8] = w[:, 16:23] / 1000.0
    ab[:, 1:8] = b[:, 16:23] / 1000.0
    ab[:, 0] = RQ_EDGE_U / 1000.0
    ab[:, 8] = RQ_EDGE_U / 1000.0
    Wf[:, 16:24] = aw[:, 1:9] - aw[:, 0:8]
    bf[:, 16:24] = ab[:, 1:9] - ab[:, 0:8]
    return Wf.float(), bf.float()


def derivative_logit_bound(W2: torch.Tensor, b2: torch.Tensor, Dh: int) -> torch.Tensor:
    """sup |a - c| over all inputs and knots of the padded derivative logits a = c + [c, u_d, c]/1000 (|tanh| <= 1, so
    |u_d| <= sum_h |w| + |b| on the unfolded derivative rows): admits csrc/b2f_rqfast.cuh delta_poly when below
    kDeltaPolyBound.  Never 0 (the edge logits contribute c/1000), which the kernel reads as "no bound"."""
    H = W2.shape[1]
    w = W2.reshape(Dh, 23, H)[:, 16:23].double()
    b = b2.reshape(Dh, 23)[:, 16:23].double()
    interior = (w.abs().sum(dim=2) + b.abs()).max() / 1000.0
    return torch.clamp(interior, min=abs(RQ_EDGE_U) / 1000.0).float()


def _elementwise_affine(op, flip: bool):
    """(a, b, sum log|a|) of one ElementwiseAffine / ActNorm op as z = a*x + b per PHYSICAL column
    (affine.py:33-59; layers_base.py:300-318)."""
    value = op.leafs[0].detach().reshape(-1, 2).float()
    alpha = torch.exp(AFFINE_C0 + value[:, 0] / 2) + AFFINE_M
    la = torch.log(alpha)
    if op.tkind == N.T_AFFINE_FWD:
        a, b, ld = alpha, value[:, 1], la.sum()
    else:
        a, b, ld = 1.0 / alpha, -value[:, 1] / alpha, -la.sum()
    if flip:
        a, b = a.flip(0), b.flip(0)
    return a, b, ld


class Plan:
    """Blobs of one program: ``layer_blobs[i]`` for the i-th coupling op, ``program_blob`` for the program."""

    def __init__(self):
        self.layer_blobs: List[torch.Tensor] = []
        self.program_blob: Optional[torch.Tensor] = None
        self.layers: List[dict] = []           # decoded pieces, kept for the CPU emulator in tests/
        self.fin_a = self.fin_b = self.in_a = self.in_b = None
        self.const_ld = self.const_lp = None
        self.final_pass = [False, False]


def build_plan(ops: Sequence, D: int, base_loc: Optional[torch.Tensor], base_log_scale: Optional[torch.Tensor]) -> Plan:
    dev = ops[0].leafs[0].device if ops[0].leafs else None
    for op in ops:
        if op.leafs:
            dev = op.leafs[0].device
            break
    Dh = D // 2
    f32 = dict(device=dev, dtype=torch.float32)
    A, B = torch.ones(D, **f32), torch.zeros(D, **f32)
    pending = [False, False]
    const_ld = torch.zeros((), **f32)
    flip, last = False, None
    plan = Plan()
    half = (slice(0, Dh), slice(Dh, D))
    with torch.no_grad():
        for op in ops:
            if op.kind == N.OP_FLIP:
                flip = not flip
            elif op.kind == N.OP_ELEMENTWISE:
                a, b, ld = _elementwise_affine(op, flip)
                const_ld = const_ld + ld
                for h in (0, 1):
                    c = half[h]
                    if last is not None and last['tgt_half'] == h:      # rides on the write-back of the layer before
                        last['post_b'] = a[c] * last['post_b'] + b[c]
                        last['post_a'] = a[c] * last['post_a']
                    else:
                        B[c] = a[c] * B[c] + b[c]
                        A[c] = a[c] * A[c]
                        pending[h] = True
            else:
                s = 1 if flip else 0
                t = 1 - s
                W1, b1, W2, b2 = (x.detach().float() for x in op.leafs)
                H = W1.shape[0]
                bound_d = derivative_logit_bound(W2, b2, Dh)
                layer = dict(src_half=s, tgt_half=t, src_pass=pending[s], H=H, K2=(H + 2 + 7) // 8 * 8,
                             boundary=float(op.boundary), inverse=op.tkind == N.T_RQ_INV,
                             src_a=A[half[s]].clone(), src_b=B[half[s]].clone(),
                             pre_a=A[half[t]].clone(), pre_b=B[half[t]].clone(),
                             post_a=torch.ones(Dh, **f32), post_b=torch.zeros(Dh, **f32),
                             W1=(W1.flip(1) if flip else W1), b1=b1, bound_d=bound_d)
                Wf, bf = fold_output_layer(W2, b2, Dh)
                if flip:                      # physical order of the target columns is the reverse of the logical one
                    Wf, bf = Wf.flip(0), bf.flip(0)
                layer['Wf'], layer['bf'] = Wf, bf
                A[:] = 1.0
                B[:] = 0.0
                pending = [False, False]
                last = layer
                plan.layers.append(layer)
        # end of program: what is still pending is applied by the final pass (y) and by the base density (fin)
        ls = base_log_scale.detach().float() if base_log_scale is not None else torch.zeros(D, **f32)
        loc = base_loc.detach().float() if base_loc is not None else torch.zeros(D, **f32)
        inv_s = torch.exp(-ls)
        plan.fin_a, plan.fin_b = A.clone(), B.clone()
        plan.final_pass = list(pending)
        plan.in_a, plan.in_b = inv_s, -loc * inv_s
        plan.const_ld = const_ld
        plan.const_lp = -(0.5 * math.log(2 * math.pi) * D + ls.sum())
        last_writer = {}
        for i, layer in enumerate(plan.layers):
            last_writer[layer['tgt_half']] = i
        for i, layer in enumerate(plan.layers):
            c = half[layer['tgt_half']]
            if last_writer[layer['tgt_half']] == i:
                layer['fin_a'] = A[c] * inv_s[c]
                layer['fin_b'] = (B[c] - loc[c]) * inv_s[c]
            else:
                layer['fin_a'] = torch.zeros(Dh, **f32)
                layer['fin_b'] = torch.zeros(Dh, **f32)
        # ---- serialise -------------------------------------------------------------------------------------------------
        for layer in plan.layers:
            H, K2 = layer['H'], layer['K2']
            n_chunks = Dh // EPC
            hdr = torch.tensor([MAGIC, layer['src_half'], int(layer['src_pass']), H, K2, n_chunks, Dh, 0],
                               dtype=torch.int32, device=dev).view(torch.float32)
            W1p = torch.zeros(32, Dh, **f32)
            W1p[:H] = round_tf32(layer['W1'])
            b1p = torch.zeros(32, **f32)
            b1p[:H] = layer['b1']
            M = torch.zeros(Dh, CPE, K2, **f32)
            M[:, :, :H] = round_tf32(layer['Wf'])
            b_hi = round_tf32(layer['bf'])
            M[:, :, H] = b_hi
            M[:, :, H + 1] = round_tf32(layer['bf'] - b_hi)
            w2c = M.reshape(n_chunks, (EPC * CPE) // 8, 8, K2 // 4, 4).permute(0, 1, 3, 2, 4).contiguous().reshape(-1)
            tp = torch.stack([layer['pre_a'], layer['pre_b'], layer['post_a'], layer['post_b'], layer['fin_a'],
                              layer['fin_b'], torch.zeros(Dh, **f32), torch.zeros(Dh, **f32)], dim=1).reshape(-1)
            sp = torch.stack([layer['src_a'], layer['src_b']], dim=1).reshape(-1)
            # |tanh| <= 1, so |column| <= sum_h |w| + |b|: proves the ranges the fast spline variant relies on
            absum = layer['Wf'].abs().sum(dim=2) + layer['bf'].abs()
            misc = torch.stack([absum[:, 0:8].max(), absum[:, 8:16].max(), layer['bound_d'], torch.zeros((), **f32)])
            layer['bound_L'], layer['bound_Dl'] = misc[0], misc[1]
            layer['M'] = M
            blob = torch.cat([hdr, canonical(W1p), b1p, w2c, tp, sp, misc]).contiguous()
            assert blob.numel() == layer_blob_floats(D, H)
            plan.layer_blobs.append(blob)
        flags = torch.tensor([MAGIC, int(plan.final_pass[0]), int(plan.final_pass[1]), len(plan.layers)],
                             dtype=torch.int32, device=dev).view(torch.float32)
        consts = torch.stack([plan.const_ld.reshape(()), plan.const_lp.reshape(()).float(), torch.zeros((), **f32),
                              torch.zeros((), **f32)])
        plan.program_blob = torch.cat([flags, consts, torch.stack([plan.fin_a, plan.fin_b], dim=1).reshape(-1),
                                       torch.stack([plan.in_a, plan.in_b], dim=1).reshape(-1)]).contiguous()
    return plan


def program_blob_floats(D: int) -> int:
    return 8 + 4 * D


def cached_plan(ops: Sequence, D: int, base_loc, base_log_scale) -> Plan:
    """Plan of a program, rebuilt when any parameter (or the base distribution) changed."""
    tensors = [t for op in ops for t in op.leafs] + [t for t in (base_loc, base_log_scale) if t is not None]
    ver = tuple((t.data_ptr(), t._version) for t in tensors) + tuple((op.kind, op.tkind) for op in ops)
    owner = next((op.owner for op in ops if op.kind == N.OP_COUPLING and op.owner is not None), None)
    cache = getattr(owner, '_b2f_cache', None) if owner is not None else None
    if cache is None:
        cache = {}
        if owner is not None:
            object.__setattr__(owner, '_b2f_cache', cache)
    key = ('tcq', base_loc is None, base_log_scale is None) + tuple(op.tkind for op in ops)
    hit = cache.get(key)
    if hit is not None and hit[0] == ver:
        return hit[1]
    plan = build_plan(ops, D, base_loc, base_log_scale)
    cache[key] = (ver, plan)
    return plan
