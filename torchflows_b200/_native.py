"""ctypes binding of libb2f.so (include/b2f.h).  There is no fallback: if the library is missing or the
tensors are not CUDA fp32 the call fails loudly."""
import ctypes
import os
from typing import Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('B2F_LIB') or os.path.join(_HERE, 'lib', 'libb2f.so')      # B2F_LIB: A/B builds of the library

# enum b2f_transformer
T_SHIFT_ADD, T_SHIFT_SUB, T_AFFINE_FWD, T_AFFINE_INV, T_RQ_FWD, T_RQ_INV = range(6)
# stand-alone transformer kernels only (b2f_transformer_apply / _backward), never part of a flow program
T_LRS_FWD, T_LRS_INV, T_SCALE_FWD, T_SCALE_INV = range(6, 10)
# enum b2f_op_kind
OP_ELEMENTWISE, OP_FLIP, OP_COUPLING, OP_MADE, OP_MADE_SEQ = range(5)
MAX_OPS = 40
FLAG_SEQ_LOGDET_EXACT = 1
FLAG_TC_OPERANDS = 2
FLAG_TC_FLIPPED = 4
FLAG_TCQ_OPERANDS = 8
FLAG_TCA_OPERANDS = 16
FLAG_TCM_OPERANDS = 32
FLAG_ROW_BIAS = 64
FLAG_SEQ_FOLDED = 128
FLOW_LOGP_OF_INPUT = 1
FLOW_MODE_PRECISE = 2
FLOW_MODE_FAST_KNOTS = 4
FLOW_WS_FILLED = 8
KERNEL_NONE, KERNEL_GENERIC, KERNEL_TC, KERNEL_ROWS, KERNEL_TCQ, KERNEL_TCA, KERNEL_TCM = range(7)

INVERSE_KIND = {T_SHIFT_ADD: T_SHIFT_SUB, T_SHIFT_SUB: T_SHIFT_ADD, T_AFFINE_FWD: T_AFFINE_INV,
                T_AFFINE_INV: T_AFFINE_FWD, T_RQ_FWD: T_RQ_INV, T_RQ_INV: T_RQ_FWD, T_LRS_FWD: T_LRS_INV,
                T_LRS_INV: T_LRS_FWD, T_SCALE_FWD: T_SCALE_INV, T_SCALE_INV: T_SCALE_FWD}


class B2FError(RuntimeError):
    pass


class Op(ctypes.Structure):
    """struct b2f_op (include/b2f.h)."""
    _fields_ = [('kind', ctypes.c_int32), ('tkind', ctypes.c_int32), ('n_hidden', ctypes.c_int32),
                ('n_bins', ctypes.c_int32), ('boundary', ctypes.c_float), ('flags', ctypes.c_int32),
                ('p', ctypes.c_void_p * 6), ('g', ctypes.c_void_p * 6)]


class WideLayer(ctypes.Structure):
    """struct b2f_wide_layer (include/b2f.h)."""
    _fields_ = [('D', ctypes.c_int32), ('H', ctypes.c_int32), ('tkind', ctypes.c_int32), ('n_bins', ctypes.c_int32),
                ('boundary', ctypes.c_float), ('reserved', ctypes.c_int32), ('W1', ctypes.c_void_p), ('b1', ctypes.c_void_p),
                ('W2', ctypes.c_void_p), ('b2', ctypes.c_void_p)]


class ColOp(ctypes.Structure):
    """struct b2f_colop (include/b2f.h)."""
    _fields_ = [('kind', ctypes.c_int32), ('reserved', ctypes.c_int32), ('value', ctypes.c_void_p), ('gvalue', ctypes.c_void_p)]


COL_AFFINE_FWD, COL_AFFINE_INV, COL_FLIP, COL_MAX_OPS = 0, 1, 2, 8
_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B2FError(f'{LIB_PATH} is missing: build it with `python build_native.py product` '
                           '(torchflows_b200 has no CPU or PyTorch fallback for its kernels)')
        L = ctypes.CDLL(LIB_PATH)
        vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_float
        L.b2f_last_error.restype = ctypes.c_char_p
        L.b2f_abi_version.restype = i32
        L.b2f_last_flow_kernel.restype = i32
        L.b2f_params_per_element.argtypes = [i32, i32]
        L.b2f_padded_params.argtypes = [i32]
        L.b2f_flow_apply.argtypes = [ctypes.POINTER(Op), i32, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp]
        L.b2f_flow_apply_saving.argtypes = [ctypes.POINTER(Op), i32, vp, vp, vp, vp, vp, vp, vp, ctypes.POINTER(i32), i64,
                                            i32, i32, vp]
        L.b2f_flow_backward.argtypes = [ctypes.POINTER(Op), i32, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i32, vp]
        L.b2f_flow_backward_workspace.argtypes = [ctypes.POINTER(Op), i32, i64, i32]
        L.b2f_flow_backward_workspace.restype = i64
        L.b2f_flow_backward_fits.argtypes = [ctypes.POINTER(Op), i32, i32]
        L.b2f_flow_backward_fits.restype = i32
        L.b2f_flow_backward_shape.argtypes = [ctypes.POINTER(Op), i32, i32, i32, ctypes.POINTER(i32 * 3)]
        L.b2f_flow_backward_shape.restype = i32
        L.b2f_transformer_apply.argtypes = [i32, vp, vp, vp, vp, vp, i64, i32, i64, i32, f32, i32, vp]
        L.b2f_transformer_backward.argtypes = [i32, vp, vp, vp, vp, vp, vp, i64, i32, i64, i32, f32, i32, vp]
        L.b2f_column_stats.argtypes = [vp, vp, vp, i64, i32, vp]
        L.b2f_debug_umma_gemm.argtypes = [vp, vp, vp, i32, i32, vp]
        u64 = ctypes.c_uint64
        L.b2f_flow_sample.argtypes = [ctypes.POINTER(Op), i32, vp, vp, vp, vp, vp, vp, i64, i32, i32, u64, u64, vp]
        L.b2f_philox_normal.argtypes = [vp, i64, i32, vp, vp, u64, u64, vp]
        L.b2f_gauss_log_prob.argtypes = [vp, vp, vp, vp, i64, i32, vp]
        L.b2f_gauss_log_prob_backward.argtypes = [vp, vp, vp, vp, vp, i64, i32, vp]
        L.b2f_column_run_apply.argtypes = [ctypes.POINTER(ColOp), i32, vp, vp, vp, i64, i32, vp]
        L.b2f_column_run_backward.argtypes = [ctypes.POINTER(ColOp), i32, vp, vp, vp, vp, vp, i64, i32, vp]
        L.b2f_wide_coupling_workspace.argtypes = [i64, i32, i32, i32]
        L.b2f_wide_coupling_workspace.restype = i64
        L.b2f_wide_coupling_forward.argtypes = [ctypes.POINTER(WideLayer), vp, vp, vp, i64, vp, i64, vp, i64, i32, vp]
        L.b2f_wide_coupling_backward.argtypes = [ctypes.POINTER(WideLayer), vp, vp, vp, vp, vp, vp, vp, vp, i64, vp, i64, vp, i64,
                                                 i32, vp]
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise B2FError(f'libb2f error {rc}: {lib().b2f_last_error().decode()}')


def require_cuda_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda:
        raise B2FError(f'{name} must be a CUDA tensor: torchflows_b200 runs this path only as sm_100a kernels '
                       f'(no CPU fallback); got device {t.device}')
    if t.dtype != torch.float32:
        raise B2FError(f'{name} must be float32, got {t.dtype}')
    return t.contiguous()


def ptr(t: Optional[torch.Tensor]):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def stream_ptr(device) -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def make_ops(ops: Sequence[dict]):
    """ops: dicts with kind, tkind, n_hidden, n_bins, boundary, flags, p (list of tensors), g (list of tensors)."""
    if len(ops) > MAX_OPS:
        raise B2FError(f'flow program of {len(ops)} ops exceeds B2F_MAX_OPS={MAX_OPS}')
    arr = (Op * max(len(ops), 1))()
    for i, o in enumerate(ops):
        a = arr[i]
        a.kind, a.tkind = o['kind'], o.get('tkind', 0)
        a.n_hidden, a.n_bins = o.get('n_hidden', 0), o.get('n_bins', 0)
        a.boundary, a.flags = o.get('boundary', 0.0), o.get('flags', 0)
        for j, t in enumerate(o.get('p', [])):
            a.p[j] = None if t is None else t.data_ptr()
        for j, t in enumerate(o.get('g', [])):
            a.g[j] = None if t is None else t.data_ptr()
    return arr


def flow_apply(ops: Sequence[dict], x: torch.Tensor, want_y=True, want_log_det=True, want_log_prob=False,
               base_loc=None, base_log_scale=None, flags=0, save_layer_inputs=False):
    """x: (B, D) CUDA fp32 contiguous.  Returns (y | None, log_det | None, log_prob | None); with save_layer_inputs a fourth
    item: the workspace holding every conditioner layer's input for flow_backward (None if the kernel that ran cannot
    save them -- b2f_flow_apply_saving)."""
    x = require_cuda_f32(x, 'flow input')
    B, D = x.shape
    # all-sequential programs (IAF / IA-RQNSF densities) run in place in their output buffer (csrc/b2f_flow_rows.cu): give
    # them one even when the caller only wants the log-density
    kinds = [o['kind'] for o in ops]
    scratch_y = (not want_y) and OP_MADE_SEQ in kinds and all(k in (OP_ELEMENTWISE, OP_FLIP, OP_MADE_SEQ) for k in kinds)
    y = torch.empty_like(x) if (want_y or scratch_y) else None
    ld = torch.empty(B, device=x.device, dtype=torch.float32) if want_log_det else None
    lp = torch.empty(B, device=x.device, dtype=torch.float32) if want_log_prob else None
    arr = make_ops(ops)
    with torch.cuda.device(x.device):
        if not save_layer_inputs:
            check(lib().b2f_flow_apply(arr, len(ops), ptr(x), ptr(y), ptr(ld), ptr(lp), ptr(base_loc),
                                       ptr(base_log_scale), B, D, flags, stream_ptr(x.device)))
            return (y if want_y else None), ld, lp
        ws_bytes = int(lib().b2f_flow_backward_workspace(arr, len(ops), B, D))
        ws = torch.empty(max(ws_bytes, 4) // 4, device=x.device, dtype=torch.float32)
        saved = ctypes.c_int32(0)
        check(lib().b2f_flow_apply_saving(arr, len(ops), ptr(x), ptr(y), ptr(ld), ptr(lp), ptr(base_loc),
                                          ptr(base_log_scale), ptr(ws), ctypes.byref(saved), B, D, flags,
                                          stream_ptr(x.device)))
    return (y if want_y else None), ld, lp, (ws if saved.value else None)


def transformer_apply(tkind, x2: torch.Tensor, h: torch.Tensor, h_row_stride: int, n_bins=8, boundary=50.0,
                      want_bins=False, flags=0):
    """x2: (n_rows, E).  h: any CUDA fp32 tensor whose rows are h_row_stride floats apart."""
    x2 = require_cuda_f32(x2, 'transformer input')
    h = require_cuda_f32(h, 'transformer parameters')
    n_rows, E = x2.shape
    out = torch.empty_like(x2)
    ld = torch.empty(n_rows, device=x2.device, dtype=torch.float32)
    k = torch.empty((n_rows, E), device=x2.device, dtype=torch.int32) if want_bins else None
    with torch.cuda.device(x2.device):
        check(lib().b2f_transformer_apply(tkind, ptr(x2), ptr(h), ptr(out), ptr(ld), ptr(k), n_rows, E, h_row_stride,
                                          n_bins, boundary, flags, stream_ptr(x2.device)))
    return out, ld, k


def transformer_backward(tkind, x2, h, h_row_stride, gout, gld, n_bins=8, boundary=50.0, flags=0):
    n_rows, E = x2.shape
    P = lib().b2f_params_per_element(tkind, n_bins)
    gx = torch.empty_like(x2)
    gh = torch.empty((n_rows, E, P), device=x2.device, dtype=torch.float32)
    with torch.cuda.device(x2.device):
        check(lib().b2f_transformer_backward(tkind, ptr(x2), ptr(h), ptr(gout), ptr(gld), ptr(gx), ptr(gh), n_rows, E,
                                             h_row_stride, n_bins, boundary, flags, stream_ptr(x2.device)))
    return gx, gh


def flow_backward_fits(kind: int, tkind: int, n_hidden: int, n_bins: int, D: int) -> bool:
    """Can b2f_flow_backward take a program with a layer of this shape at event size D (shared-memory footprint of the
    backward kernel, csrc/b2f_flow_bwd.cu)?  Host-only query: no device, no parameters needed."""
    arr = (Op * 1)()
    arr[0].kind, arr[0].tkind, arr[0].n_hidden, arr[0].n_bins = kind, tkind, n_hidden, n_bins
    return bool(lib().b2f_flow_backward_fits(arr, 1, D))


def flow_backward_shape(ops: Sequence[dict], D: int, flags=0):
    """(TM, NT, wst_stride) that flow_backward would launch for this program, or None if the backward kernel cannot take
    it.  wst_stride > 0: spline layers take the tensor-core GEMM path.  Host-only; honours the B2F_BWD_TM / B2F_BWD_NT /
    B2F_BWD_NO_MMA overrides and FLOW_MODE_PRECISE in `flags` as the launch does."""
    arr = make_ops(ops)
    out = (ctypes.c_int32 * 3)()
    if not lib().b2f_flow_backward_shape(arr, len(ops), D, flags, ctypes.byref(out)):
        return None
    return tuple(out)


def last_flow_kernel() -> int:
    """Which kernel this thread's last flow_apply launched (KERNEL_GENERIC / KERNEL_TC / KERNEL_ROWS / KERNEL_TCQ)."""
    return int(lib().b2f_last_flow_kernel())


def column_stats(x2: torch.Tensor):
    """Per-column sum and sum of squares of x2:(B, D) in fp64 (ActNorm initialisation)."""
    B, D = x2.shape
    s = torch.zeros(D, device=x2.device, dtype=torch.float64)
    q = torch.zeros(D, device=x2.device, dtype=torch.float64)
    with torch.cuda.device(x2.device):
        check(lib().b2f_column_stats(ptr(x2), ptr(s), ptr(q), B, D, stream_ptr(x2.device)))
    return s, q


def debug_umma_gemm(A: torch.Tensor, B: torch.Tensor) -> torch.Tensor:
    """C[128,N] = A[128,K] @ B[N,K]^T on the tensor cores (tf32), diagnostic entry point."""
    A, B = require_cuda_f32(A, 'A'), require_cuda_f32(B, 'B')
    assert A.shape[0] == 128 and A.shape[1] == B.shape[1]
    C = torch.empty(128, B.shape[0], device=A.device, dtype=torch.float32)
    with torch.cuda.device(A.device):
        check(lib().b2f_debug_umma_gemm(ptr(A), ptr(B), ptr(C), B.shape[0], A.shape[1], stream_ptr(A.device)))
    return C


# ---- wide-conditioner spline coupling layer (csrc/b2f_wide.cu) -------------------------------------------------------------
def wide_eligible(D: int, H: int, n_bins: int) -> bool:
    """Mirror of check_layer in csrc/b2f_wide.cu."""
    return D >= 64 and D % 64 == 0 and H >= 1 and n_bins == 8


WIDE_FOR_BACKWARD, WIDE_KEPT = 1, 2
_wide_ws = {}


def _wide_buffer(device, role: str, need: int) -> torch.Tensor:
    """Shared buffers of the wide layer kernels, one per (device, role) that only grows: the layers of a flow run one
    after the other on one stream and nothing in them outlives a call (what must survive until the backward is allocated
    per call instead, see wide_coupling_forward).  Callers that drive wide layers from SEVERAL streams or threads at once
    must give each its own buffers (the C ABI takes them as arguments; this cache is a convenience of the Python side)."""
    key = (device.type, device.index, role)
    buf = _wide_ws.get(key)
    if buf is None or buf.numel() * 4 < need:
        _wide_ws[key] = buf = torch.empty((need + 3) // 4, device=device, dtype=torch.float32)
    return buf


def _wide_layer(D, H, tkind, n_bins, boundary, W1, b1, W2, b2) -> WideLayer:
    L = WideLayer()
    L.D, L.H, L.tkind, L.n_bins, L.boundary, L.reserved = D, H, tkind, n_bins, float(boundary), 0
    L.W1, L.b1, L.W2, L.b2 = W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr()
    return L


def wide_coupling_forward(tkind, x2, W1, b1, W2, b2, n_bins=8, boundary=50.0, for_backward=False):
    """x2: (B, D).  Returns (y, log_det, keep): with for_backward, `keep` holds the packed operands and hidden activations
    of this call for wide_coupling_backward (None otherwise)."""
    x2 = require_cuda_f32(x2, 'coupling input')
    W1, b1, W2, b2 = (require_cuda_f32(t, 'conditioner parameter') for t in (W1, b1, W2, b2))
    B, D = x2.shape
    H = W1.shape[0]
    y = torch.empty_like(x2)
    ld = torch.empty(B, device=x2.device, dtype=torch.float32)
    with torch.cuda.device(x2.device):
        L = lib()
        if for_backward:
            keep = torch.empty((int(L.b2f_wide_coupling_workspace(B, D, H, 1)) + 3) // 4, device=x2.device, dtype=torch.float32)
        else:
            keep = _wide_buffer(x2.device, 'keep', int(L.b2f_wide_coupling_workspace(B, D, H, 0)))
        scratch = _wide_buffer(x2.device, 'scratch', int(L.b2f_wide_coupling_workspace(B, D, H, 2)))
        layer = _wide_layer(D, H, tkind, n_bins, boundary, W1, b1, W2, b2)
        check(L.b2f_wide_coupling_forward(ctypes.byref(layer), ptr(x2), ptr(y), ptr(ld), B, ptr(keep), keep.numel() * 4,
                                          ptr(scratch), scratch.numel() * 4, WIDE_FOR_BACKWARD if for_backward else 0,
                                          stream_ptr(x2.device)))
    return y, ld, (keep if for_backward else None)


def wide_coupling_backward(tkind, x2, gy, gld, W1, b1, W2, b2, n_bins=8, boundary=50.0, keep=None):
    """Returns (gx, gW1, gb1, gW2, gb2) given the layer input x2 and upstream gradients (either may be None).  `keep`: what
    wide_coupling_forward(..., for_backward=True) returned for the same x2 and (unchanged) parameters."""
    x2 = require_cuda_f32(x2, 'coupling input')
    W1, b1, W2, b2 = (require_cuda_f32(t, 'conditioner parameter') for t in (W1, b1, W2, b2))
    gy = None if gy is None else require_cuda_f32(gy, 'upstream gradient')
    gld = None if gld is None else require_cuda_f32(gld, 'upstream gradient')
    B, D = x2.shape
    H = W1.shape[0]
    gx = torch.empty_like(x2)
    gW1, gb1, gW2, gb2 = (torch.empty_like(t) for t in (W1, b1, W2, b2))
    with torch.cuda.device(x2.device):
        L = lib()
        flags = WIDE_KEPT if keep is not None else 0
        if keep is None:
            keep = _wide_buffer(x2.device, 'keep', int(L.b2f_wide_coupling_workspace(B, D, H, 1)))
        scratch = _wide_buffer(x2.device, 'scratch', int(L.b2f_wide_coupling_workspace(B, D, H, 3)))
        layer = _wide_layer(D, H, tkind, n_bins, boundary, W1, b1, W2, b2)
        check(L.b2f_wide_coupling_backward(ctypes.byref(layer), ptr(x2), ptr(gy), ptr(gld), ptr(gx), ptr(gW1), ptr(gb1),
                                           ptr(gW2), ptr(gb2), B, ptr(keep), keep.numel() * 4, ptr(scratch),
                                           scratch.numel() * 4, flags, stream_ptr(x2.device)))
    return gx, gW1, gb1, gW2, gb2


# ---- runs of per-column layers (csrc/b2f_colrun.cu) --------------------------------------------------------------------------
def _col_ops(kinds, values, gvalues=None):
    arr = (ColOp * len(kinds))()
    for i, (k, v) in enumerate(zip(kinds, values)):
        arr[i].kind = k
        arr[i].value = None if v is None else v.data_ptr()
        g = None if gvalues is None else gvalues[i]
        arr[i].gvalue = None if g is None else g.data_ptr()
    return arr


def column_run_apply(kinds, values, x2: torch.Tensor):
    """kinds: COL_* per op; values: the (D, 2) parameter tensor per op (None for flips).  Returns (y, log_det_sum[1])."""
    x2 = require_cuda_f32(x2, 'column run input')
    B, D = x2.shape
    y = torch.empty_like(x2)
    lds = torch.empty(1, device=x2.device, dtype=torch.float32)
    with torch.cuda.device(x2.device):
        check(lib().b2f_column_run_apply(_col_ops(kinds, values), len(kinds), ptr(x2), ptr(y), ptr(lds), B, D, stream_ptr(x2.device)))
    return y, lds


def column_run_backward(kinds, values, need_grad, x2, gy, g_lds):
    """Returns (gx, [gvalue or None per op])."""
    x2, gy = require_cuda_f32(x2, 'column run input'), require_cuda_f32(gy, 'upstream gradient')
    B, D = x2.shape
    gx = torch.empty_like(x2)
    gvalues = [torch.empty_like(v) if (v is not None and ng) else None for v, ng in zip(values, need_grad)]
    scratch = torch.empty(2 * D, device=x2.device, dtype=torch.float32)
    with torch.cuda.device(x2.device):
        check(lib().b2f_column_run_backward(_col_ops(kinds, values, gvalues), len(kinds), ptr(x2), ptr(gy), ptr(g_lds), ptr(gx),
                                            ptr(scratch), B, D, stream_ptr(x2.device)))
    return gx, gvalues


# ---- base draws made by the library (csrc/b2f_philox.cuh) -------------------------------------------------------------------
def philox_normal(n_rows: int, D: int, device, seed: int, offset: int, loc=None, log_scale=None) -> torch.Tensor:
    """(n_rows, D) draws loc + exp(log_scale) * n from the counter-based stream (seed, offset)."""
    out = torch.empty((n_rows, D), device=device, dtype=torch.float32)
    with torch.cuda.device(device):
        check(lib().b2f_philox_normal(ptr(out), n_rows, D, ptr(loc), ptr(log_scale), seed, offset, stream_ptr(device)))
    return out


def flow_sample(ops: Sequence[dict], B: int, D: int, device, want_log_prob=False, base_loc=None, base_log_scale=None, flags=0,
                seed=0, offset=0, in_kernel=False):
    """b2f_flow_sample: (x:(B, D), log_prob | None).  in_kernel: the program is laid out for the spline tensor-core kernel,
    which draws its tiles in registers; every other program gets a (B, D) scratch for the materialised stream."""
    if not torch.device(device).type == 'cuda':
        raise B2FError(f'sampling runs only as sm_100a kernels (no CPU fallback); got device {device}')
    y = torch.empty((B, D), device=device, dtype=torch.float32)
    lp = torch.empty(B, device=device, dtype=torch.float32) if want_log_prob else None
    arr = make_ops(ops)
    with torch.cuda.device(device):
        scratch = None if in_kernel else torch.empty((B, D), device=device, dtype=torch.float32)
        rc = lib().b2f_flow_sample(arr, len(ops), ptr(y), None, ptr(lp), ptr(base_loc), ptr(base_log_scale), ptr(scratch), B, D,
                                   flags, seed, offset, stream_ptr(device))
        if rc == -2 and scratch is None:        # B2F_ERR_UNSUPPORTED: the kernel declined the program after all
            scratch = torch.empty((B, D), device=device, dtype=torch.float32)
            rc = lib().b2f_flow_sample(arr, len(ops), ptr(y), None, ptr(lp), ptr(base_loc), ptr(base_log_scale), ptr(scratch), B,
                                       D, flags, seed, offset, stream_ptr(device))
        check(rc)
    return y, lp


# ---- base density over rows (csrc/b2f_colrun.cu) ------------------------------------------------------------------------------
def gauss_log_prob(z2: torch.Tensor, loc, log_scale) -> torch.Tensor:
    z2 = require_cuda_f32(z2, 'base density input')
    B, D = z2.shape
    lp = torch.empty(B, device=z2.device, dtype=torch.float32)
    with torch.cuda.device(z2.device):
        check(lib().b2f_gauss_log_prob(ptr(z2), ptr(loc), ptr(log_scale), ptr(lp), B, D, stream_ptr(z2.device)))
    return lp


def gauss_log_prob_backward(z2: torch.Tensor, loc, log_scale, g: torch.Tensor) -> torch.Tensor:
    g = require_cuda_f32(g, 'upstream gradient')
    B, D = z2.shape
    gz = torch.empty_like(z2)
    with torch.cuda.device(z2.device):
        check(lib().b2f_gauss_log_prob_backward(ptr(z2), ptr(loc), ptr(log_scale), ptr(g), ptr(gz), B, D, stream_ptr(z2.device)))
    return gz
