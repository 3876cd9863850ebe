"""Specialisations of the spline tensor-core kernel (csrc/b2f_flow_tcq.cu): the output-only launch that Flow.sample uses
when nobody reads a log-det (bit-identical samples), and the polynomial knot derivative admitted by a host-proven bound on
the derivative logits (log_prob within 1e-6 of the SFU softplus, within the 1e-4 oracle tolerance; a layer above the
bound keeps the SFU path).  B2F_TCQ_ALWAYS_LD / B2F_TCQ_NO_DPOLY select the general variants per launch."""
import contextlib
import os

import pytest
import torch

from oracle.flow_oracle import OracleFlow

pytestmark = pytest.mark.gpu
LP_TOL = 1e-4
DPOLY_BOUND = 1.0 / 32.0        # rqf::kDeltaPolyBound


@contextlib.contextmanager
def env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    try:
        for k, v in kv.items():
            os.environ[k] = v
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def close(a, b, what, atol, rtol):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert torch.isfinite(a).all(), what
    err = (a - b).abs() - (atol + rtol * b.abs())
    assert (err <= 0).all(), f'{what}: max abs diff {(a - b).abs().max().item():.3e}, worst excess {err.max().item():.3e}'


def derivative_rows(flow, D):
    """(weight, bias) of every coupling conditioner's output layer (rows e * 23 + p, p >= 16: derivative logits)."""
    P = D // 2 * 23
    ws = [p for p in flow.parameters() if p.dim() == 2 and p.shape[0] == P]
    bs = [p for p in flow.parameters() if p.dim() == 1 and p.shape[0] == P]
    assert len(ws) == len(bs) > 0
    return list(zip(ws, bs))


def make(D, dev, state='T', scale_d=1.0):
    from torchflows_b200 import Flow
    import torchflows_b200.architectures as arch
    torch.manual_seed(200 + D)
    flow = Flow(arch.CouplingRQNSF(D)).to(dev)
    with torch.no_grad():
        for w, b in derivative_rows(flow, D):
            w.view(D // 2, 23, -1)[:, 16:] *= scale_d
            b.view(D // 2, 23)[:, 16:] *= scale_d
    if state == 'T':                    # ActNorm data-initialised by one training-mode pass
        g = torch.Generator().manual_seed(5)
        flow.train()
        with torch.no_grad():
            flow.log_prob((torch.randn(4096, D, generator=g) * 1.3 + 0.2).to(dev))
    flow.eval()
    sd = {k: v.detach().cpu() for k, v in flow.state_dict().items()}
    return flow, OracleFlow('CouplingRQNSF', (D,), sd)


def max_bound(flow, D):
    from torchflows_b200 import _tcq
    return max(_tcq.derivative_logit_bound(w.detach(), b.detach(), D // 2).item() for w, b in derivative_rows(flow, D))


def oracle_chunked(fn, x, chunk=8192):
    return torch.cat([fn(x[i:i + chunk]) for i in range(0, x.shape[0], chunk)])


@pytest.mark.parametrize('D,B', [(256, (1 << 20) + 77), (64, 1000), (32, 5)])
def test_sample_without_log_prob_is_bit_identical(D, B):
    """Flow.sample(n) runs the output-only kernel; under the same seed it equals the samples of the log-det kernel, both
    from sample(n, return_log_prob=True) and forced by B2F_TCQ_ALWAYS_LD (full tiles through TMA, the ragged last tile
    through the epilogue warps)."""
    from torchflows_b200 import _native as N
    dev = torch.device('cuda:0')
    flow, _ = make(D, dev)
    with torch.no_grad():
        torch.manual_seed(9)
        xs = flow.sample(B, no_grad=True)
        assert N.last_flow_kernel() == N.KERNEL_TCQ
        torch.manual_seed(9)
        xs_lp, lp = flow.sample(B, no_grad=True, return_log_prob=True)
        with env(B2F_TCQ_ALWAYS_LD='1'):
            torch.manual_seed(9)
            xs_ld = flow.sample(B, no_grad=True)
        torch.cuda.synchronize()
    assert torch.isfinite(xs).all() and torch.isfinite(lp).all()
    assert torch.equal(xs, xs_lp)
    assert torch.equal(xs, xs_ld)
    del xs, xs_lp, xs_ld


@pytest.mark.parametrize('scale_d', [1.0, 5.0])
def test_dpoly_matches_sfu_softplus_and_oracle(scale_d):
    """Benchmark shape (CouplingRQNSF(256), state T), derivative rows as initialised and scaled by 5: the bound admits
    the polynomial; log_prob agrees with the SFU softplus to 1e-6, both variants with the oracle to 1e-4."""
    dev = torch.device('cuda:0')
    D = 256
    flow, oracle = make(D, dev, scale_d=scale_d)
    assert max_bound(flow, D) < DPOLY_BOUND
    B = 32768 + 77
    g = torch.Generator().manual_seed(12)
    x = torch.randn(B, D, generator=g) * 1.5
    z = torch.randn(B, D, generator=g)
    res = {}
    for name, kv in (('poly', {}), ('sfu', {'B2F_TCQ_NO_DPOLY': '1'})):
        with env(**kv), torch.no_grad():
            lp = flow.log_prob(x.to(dev))
            xs = flow._sample_from_base(z.to(dev), no_grad=True)
            torch.manual_seed(4)
            xn = flow.sample(B, no_grad=True)
            res[name] = (lp, xs, xn)
    (lp1, xs1, xn1), (lp0, xs0, xn0) = res['poly'], res['sfu']
    assert not torch.equal(lp1, lp0)               # the two variants really ran different code
    close(lp1, lp0, 'log_prob poly vs sfu', 1e-6, 1e-6)
    # Samples are not held to 1e-6: the inverse map amplifies an ulp of the knot derivative where the spline is flat, and
    # a later layer's conditioner reads the result through a TF32 rounding that a 1-ulp difference can flip (2^-11
    # relative).  Any two fp32-faithful evaluations differ by up to ~1e-4 there, the parent commit and this one included.
    for what, a, b in (('sample', xs1, xs0), ('Flow.sample', xn1, xn0)):
        close(a, b, f'{what} poly vs sfu', 2e-4, 2e-4)
    lp_ref = oracle_chunked(oracle.log_prob, x)
    xs_ref = oracle_chunked(oracle.sample_from_noise, z)
    for name, (lp, xs, _) in res.items():
        close(lp, lp_ref, f'log_prob ({name})', LP_TOL, LP_TOL)
        close(xs, xs_ref, f'sample ({name})', 2e-3, 1e-4)


def test_layer_above_bound_takes_sfu_path():
    """Derivative rows scaled by 20 put the bound above 1/32: the kernel keeps the SFU softplus (bit-identical with and
    without B2F_TCQ_NO_DPOLY) and still matches the oracle."""
    dev = torch.device('cuda:0')
    D = 128
    flow, oracle = make(D, dev, scale_d=20.0)
    assert max_bound(flow, D) > DPOLY_BOUND
    B = 128 * 40 + 9
    g = torch.Generator().manual_seed(13)
    x = torch.randn(B, D, generator=g) * 1.5
    z = torch.randn(B, D, generator=g)
    res = {}
    for name, kv in (('default', {}), ('sfu', {'B2F_TCQ_NO_DPOLY': '1'})):
        with env(**kv), torch.no_grad():
            res[name] = (flow.log_prob(x.to(dev)), flow._sample_from_base(z.to(dev), no_grad=True))
    assert torch.equal(res['default'][0], res['sfu'][0])
    assert torch.equal(res['default'][1], res['sfu'][1])
    close(res['default'][0], oracle.log_prob(x), 'log_prob', LP_TOL, LP_TOL)
    close(res['default'][1], oracle.sample_from_noise(z), 'sample', 2e-3, 1e-4)
