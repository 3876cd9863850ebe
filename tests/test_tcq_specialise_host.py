"""CPU checks of the spline tensor-core kernel's specialisations (csrc/b2f_rqfast.cuh, torchflows_b200/_tcq.py): the
polynomial knot derivative against fp64, the output-only inverse map against the full one, and the host-proven bound on
the derivative logits that admits the polynomial."""
import ctypes
import itertools
import math
import os
import subprocess
import types

import numpy as np
import pytest
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope='module')
def lib(tmp_path_factory):
    so = str(tmp_path_factory.mktemp('tcq_specialise') / 'libtcq_specialise.so')
    subprocess.run(['g++', '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared', '-x', 'c++',
                    os.path.join(_HERE, 'tcq_specialise_host.cpp'), '-o', so], check=True)
    h = ctypes.CDLL(so)
    h.ts_edge_u.restype = ctypes.c_float
    h.ts_delta_poly_bound.restype = ctypes.c_float
    return h


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def delta_poly(lib, u):
    u = np.ascontiguousarray(u, dtype=np.float32)
    out = np.empty_like(u)
    lib.ts_delta_poly(_p(u), _p(out), ctypes.c_int64(u.size))
    return out


def test_delta_poly_within_one_ulp(lib):
    """1e-5 + softplus(c + u) for |u| <= kDeltaPolyBound, against fp64 at the same fp32 logit: <= 1 ulp of fp32."""
    bound = float(lib.ts_delta_poly_bound())
    assert bound == 1.0 / 32.0
    c = float(lib.ts_edge_u())
    u = np.concatenate([np.linspace(-bound, bound, 1 << 20, dtype=np.float64),
                        [0.0, c / 1000.0, -c / 1000.0, bound, -bound]]).astype(np.float32)
    d = delta_poly(lib, u).astype(np.float64)
    ref = np.log1p(np.exp(c + u.astype(np.float64))) + 1e-5
    ulp = np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64)
    err = np.abs(d - ref) / ulp
    assert err.max() <= 1.0, (err.max(), u[err.argmax()])


def folded(n, gen, scale_d=3.0):
    """24 folded columns per element from raw parameters (the fold of _tcq.fold_output_layer): widths / heights logits
    within the fast variant's bounds, derivative logits u_d of size scale_d."""
    u = torch.randn(n, 23, generator=gen, dtype=torch.float64)
    u[:, 16:] *= scale_d
    g = torch.empty(n, 24, dtype=torch.float64)
    g[:, 0:8] = u[:, 0:8] * (1 / math.log(2))
    g[:, 8:16] = u[:, 8:16] * (1 / math.log(2)) / 1000.0
    c = math.log(math.expm1(1 - 1e-5))
    a = torch.cat([torch.full((n, 1), c, dtype=torch.float64), u[:, 16:23], torch.full((n, 1), c, dtype=torch.float64)], 1)
    a = a / 1000.0
    g[:, 16:24] = a[:, 1:9] - a[:, 0:8]
    return g.float().numpy()


def inverse(lib, x, g, b, dpoly, ld):
    x = np.ascontiguousarray(x, dtype=np.float32)
    g = np.ascontiguousarray(g, dtype=np.float32)
    out, ld2 = np.empty_like(x), np.empty_like(x)
    lib.ts_inverse(_p(x), _p(g), _p(out), _p(ld2), ctypes.c_int64(x.size), ctypes.c_float(b), ctypes.c_int(int(dpoly)),
                   ctypes.c_int(int(ld)))
    return out, ld2


@pytest.mark.parametrize('dpoly', [False, True])
def test_output_only_inverse_is_bit_identical(lib, dpoly):
    """LD = false computes the same transformed values bit for bit and leaves the log-det alone."""
    gen = torch.Generator().manual_seed(7)
    n, b = 200000, 5.0
    g = folded(n, gen)
    x = (torch.rand(n, generator=gen) * 2.2 - 1.1).numpy() * b      # includes the identity tails beyond +-b
    out_ld, ld2 = inverse(lib, x, g, b, dpoly, True)
    out, ld2_none = inverse(lib, x, g, b, dpoly, False)
    assert np.array_equal(out.view(np.int32), out_ld.view(np.int32))
    assert np.isfinite(ld2).all() and np.isnan(ld2_none).all()


def test_delta_poly_inverse_matches_sfu_softplus(lib):
    gen = torch.Generator().manual_seed(8)
    n, b = 200000, 5.0
    g = folded(n, gen, scale_d=10.0)
    x = (torch.rand(n, generator=gen) * 2 - 1).numpy() * b
    o1, l1 = inverse(lib, x, g, b, True, True)
    o0, l0 = inverse(lib, x, g, b, False, True)
    assert (np.abs(o1 - o0) <= 1e-6 * (1 + np.abs(o0))).all()
    # ld2 is the difference of two lg2 results of order 16 (den^2 and the forward derivative's numerator), where one
    # ulp is already 1.9e-6
    assert (np.abs(l1 - l0) <= 4e-6).all()


def brute_force_bound(W2, b2, Dh):
    """max over knots, elements and every corner of [-1, 1]^H (where a linear map of tanh outputs peaks) of
    |u_d| / 1000, and the padded edge logit c / 1000."""
    H = W2.shape[1]
    corners = torch.tensor(list(itertools.product((-1.0, 1.0), repeat=H)), dtype=torch.float64)      # (2^H, H)
    w = W2.double().reshape(Dh, 23, H)[:, 16:23]
    b = b2.double().reshape(Dh, 23)[:, 16:23]
    vals = torch.einsum('ekh,ch->ekc', w, corners) + b[..., None]
    return max(vals.abs().max().item() / 1000.0, abs(math.log(math.expm1(1 - 1e-5))) / 1000.0)


@pytest.mark.parametrize('H,scale', [(10, 1.0), (7, 40.0), (3, 1e-4)])
def test_derivative_logit_bound_in_plan(H, scale):
    """misc[2] of a layer blob is the brute-force bound on |a - c| (the last case: the edge logit dominates)."""
    from torchflows_b200 import _native as N
    from torchflows_b200 import _tcq
    D = 32
    Dh = D // 2
    gen = torch.Generator().manual_seed(H)
    W1 = torch.randn(H, Dh, generator=gen)
    b1 = torch.randn(H, generator=gen)
    W2 = torch.randn(Dh * 23, H, generator=gen) * scale
    b2 = torch.randn(Dh * 23, generator=gen) * scale
    op = types.SimpleNamespace(kind=N.OP_COUPLING, tkind=N.T_RQ_INV, leafs=(W1, b1, W2, b2), boundary=50.0)
    plan = _tcq.build_plan([op], D, None, None)
    misc2 = plan.layer_blobs[0][-2].item()
    ref = brute_force_bound(W2, b2, Dh)
    assert misc2 == pytest.approx(ref, rel=1e-6)
    assert misc2 == pytest.approx(_tcq.derivative_logit_bound(W2, b2, Dh).item(), rel=0)
