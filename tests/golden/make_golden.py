"""Generate the golden input/output vectors under tests/golden/ by running the REAL reference.

Run in the build container only (the reference lives at /root/reference and does not travel to
the GPU box):

    python tests/golden/make_golden.py

It imports ``torchflows`` from /root/reference (torchflows v1.2.0, unmodified), builds transformers
and presets under fixed seeds, evaluates them on CPU in fp32, and stores inputs, weights
(``state_dict``) and outputs.  The fixtures pin ``oracle/`` (tests/test_oracle_golden.py) and are the
reference-produced half of the GPU parity tests (tests/test_gpu_*.py).
"""
import io
import os
import sys
import warnings

import torch

REF = os.environ.get('TORCHFLOWS_REF', '/root/reference')
sys.path.insert(0, REF)
warnings.filterwarnings('ignore')

from torchflows.flows import Flow  # noqa: E402
from torchflows.bijections.finite.autoregressive import architectures as ref_arch  # noqa: E402
from torchflows.bijections.finite.autoregressive.transformers.linear.affine import (  # noqa: E402
    Affine, InverseAffine, Shift)
from torchflows.bijections.finite.autoregressive.transformers.spline.rational_quadratic import (  # noqa: E402
    RationalQuadratic)

OUT = os.path.dirname(os.path.abspath(__file__))
PART_BYTES = 900_000        # no file of the repository is larger than 1 MB


def _nbytes(obj):
    buf = io.BytesIO()
    torch.save(obj, buf)
    return buf.tell()


def save(obj, name):
    """torch.save(obj) as tests/golden/<name>; a list of cases (or a dict of such lists) larger than PART_BYTES goes to
    numbered parts <stem>/00.pt, 01.pt, ... of whole cases instead, which tests/conftest.py (golden) joins back."""
    path = os.path.join(OUT, name)
    if _nbytes(obj) <= PART_BYTES:
        torch.save(obj, path)
        print(name, os.path.getsize(path) // 1024, 'KiB')
        return
    keys = list(obj) if isinstance(obj, dict) else [None]
    items = [(k, c) for k in keys for c in (obj if k is None else obj[k])]
    parts, size = [[]], 0
    for k, c in items:
        n = _nbytes(c)
        if parts[-1] and size + n > PART_BYTES:
            parts.append([])
            size = 0
        parts[-1].append((k, c))
        size += n
    stem = os.path.splitext(path)[0]
    os.makedirs(stem, exist_ok=True)
    for i, part in enumerate(parts):
        out = [c for _, c in part] if keys == [None] else {k: [c for kk, c in part if kk == k] for k in keys}
        torch.save(out, os.path.join(stem, f'{i:02d}.pt'))
        print(f'{name} part {i:02d}', os.path.getsize(os.path.join(stem, f'{i:02d}.pt')) // 1024, 'KiB')


def rq_bin_index(tr: RationalQuadratic, v, h, direction):
    """Bin index the reference uses (rational_quadratic.py:75-76,82 / :147), -1 outside the bounds."""
    k_out = torch.full(v.shape, -1, dtype=torch.int64)
    mask = (v > tr.min_input) & (v < tr.max_input)
    hm = h[mask]
    u_x, u_y = hm[..., :tr.n_bins], hm[..., tr.n_bins:2 * tr.n_bins]
    bin_x, _ = tr.compute_bins(u_x, tr.min_input, tr.max_input)
    bin_y, _ = tr.compute_bins(u_x + u_y / 1000, tr.min_output, tr.max_output)
    bins = bin_x if direction == 'forward' else bin_y
    k_out[mask] = (torch.searchsorted(bins, v[mask][..., None]) - 1).view(-1)
    return k_out


def transformer_cases():
    cases = []
    g = torch.Generator().manual_seed(1234)
    # Affine / InverseAffine / Shift as in test/test_reconstruction_transformers.py:22-28,68-70
    for name, cls in (('affine', Affine), ('inverse_affine', InverseAffine), ('shift', Shift)):
        for batch_shape, event_shape in (((5,), (3,)), ((5, 2, 3), (3, 5, 2)), ((64,), (33,))):
            tr = cls(event_shape)
            x = torch.randn(*batch_shape, *event_shape, generator=g)
            h = torch.randn(*batch_shape, *tr.parameter_shape, generator=g)
            z, ld_f = tr.forward(x, h)
            xr, ld_i = tr.inverse(z, h)
            cases.append(dict(kind=name, event_shape=event_shape, x=x, h=h, z=z, ld_f=ld_f, xr=xr, ld_i=ld_i))
    # Rational quadratic as in test/test_spline.py:92-135: n_bins, boundary and input scale vary
    for n_bins in (2, 4, 8, 16, 32):
        for boundary in (1.0, 5.0, 50.0):
            for scale in (1e-2, 1.0, 1e2):
                event_shape = (8,)
                batch_shape = (16,)
                tr = RationalQuadratic(event_shape, boundary=boundary, n_bins=n_bins)
                x = torch.randn(*batch_shape, *event_shape, generator=g) * scale
                h = torch.randn(*batch_shape, *tr.parameter_shape, generator=g)
                z, ld_f = tr.forward(x, h)
                xr, ld_i = tr.inverse(z, h)
                cases.append(dict(kind='rq', n_bins=n_bins, boundary=boundary, scale=scale,
                                  event_shape=event_shape, x=x, h=h, z=z, ld_f=ld_f, xr=xr, ld_i=ld_i,
                                  k_f=rq_bin_index(tr, x, h, 'forward'), k_i=rq_bin_index(tr, z, h, 'inverse')))
    # A larger default-parameter case (n_bins=8, boundary=50) with O(1) and O(3) logits; exact knots too
    for hs in (1.0, 3.0):
        tr = RationalQuadratic((32,), boundary=50.0, n_bins=8)
        x = torch.randn(256, 32, generator=g) * 3
        x[0, :8] = torch.tensor([-50.0, 50.0, -49.999996, 49.999996, 0.0, -60.0, 75.0, 1e-30])
        h = torch.randn(256, 32, 23, generator=g) * hs
        z, ld_f = tr.forward(x, h)
        xr, ld_i = tr.inverse(z, h)
        cases.append(dict(kind='rq', n_bins=8, boundary=50.0, scale=3.0, event_shape=(32,), x=x, h=h, z=z,
                          ld_f=ld_f, xr=xr, ld_i=ld_i, k_f=rq_bin_index(tr, x, h, 'forward'),
                          k_i=rq_bin_index(tr, z, h, 'inverse')))
    # zero parameters => identity (test/test_identity_bijections.py:56-68)
    tr = RationalQuadratic((4,), boundary=50.0, n_bins=8)
    x = torch.randn(7, 4, generator=g)
    h = torch.zeros(7, 4, 23)
    z, ld_f = tr.forward(x, h)
    xr, ld_i = tr.inverse(z, h)
    cases.append(dict(kind='rq', n_bins=8, boundary=50.0, scale=1.0, event_shape=(4,), x=x, h=h, z=z, ld_f=ld_f,
                      xr=xr, ld_i=ld_i, k_f=rq_bin_index(tr, x, h, 'forward'), k_i=rq_bin_index(tr, z, h, 'inverse')))
    return cases


PRESET_CASES = [
    # (preset, event_shape, batch_shape, kwargs)
    ('RealNVP', (3,), (1000,), {}),                       # README config (data only; fit below)
    ('NICE', (8,), (5, 2, 3), {}),
    ('RealNVP', (3, 5, 2), (5,), {}),
    ('InverseRealNVP', (8,), (7,), {}),
    ('MAF', (8,), (33,), {}),
    ('IAF', (8,), (33,), {}),
    ('CouplingRQNSF', (3, 5, 2), (5, 2), {}),
    ('MaskedAutoregressiveRQNSF', (8,), (33,), {}),
    ('InverseAutoregressiveRQNSF', (5,), (9,), {}),
    ('RealNVP', (64,), (256,), {}),                       # R64 slice
    ('NICE', (64,), (256,), {}),
    ('CouplingRQNSF', (256,), (96,), {}),                 # Q256 slice
    ('MAF', (128,), (64,), {}),                           # M128 slices
    ('IAF', (128,), (64,), {}),
    ('MaskedAutoregressiveRQNSF', (128,), (48,), {}),
    ('CouplingRQNSF', (64,), (64,), {'conditioner_kwargs': {'n_hidden': 48}}),   # wide-ish conditioner
]


def preset_cases():
    cases = []
    for n, (preset, event_shape, batch_shape, kwargs) in enumerate(PRESET_CASES):
        torch.manual_seed(100 + n)
        bij = getattr(ref_arch, preset)(event_shape, **kwargs)
        flow = Flow(bij)
        flow.eval()   # state E of SURVEY 8d: no ActNorm data init
        x = torch.randn(*batch_shape, *event_shape)
        noise = torch.randn(*batch_shape, *event_shape)
        with torch.no_grad():
            z, ld_f = bij.forward(x)
            lp = flow.log_prob(x)
            xs, ld_i = bij.inverse(noise)
            lp_s = flow.base_log_prob(noise) + ld_i        # what sample(return_log_prob=True) returns
            xr, ld_r = bij.inverse(z)
        case = dict(preset=preset, event_shape=event_shape, kwargs=kwargs,
                    state_dict={k: v.clone() for k, v in flow.state_dict().items()},
                    x=x, noise=noise, z=z, ld_f=ld_f, log_prob=lp, xs=xs, ld_i=ld_i, lp_s=lp_s, xr=xr, ld_r=ld_r)
        # state T: one training-mode forward data-initialises every ActNorm (layers.py:58-68)
        flow.train()
        with torch.no_grad():
            lp_train = flow.log_prob(x)
        flow.eval()
        case['actnorm_T'] = {k: v.clone() for k, v in flow.state_dict().items()
                             if k.endswith('.value') and int(k.split('.')[2]) in (3, 6, 8)}
        case['log_prob_T'] = lp_train
        cases.append(case)
    return cases


GRAD_CASES = [
    ('RealNVP', (8,), 64, {}),
    ('NICE', (8,), 64, {}),
    ('CouplingRQNSF', (8,), 64, {}),
    ('MAF', (8,), 64, {}),
    ('MaskedAutoregressiveRQNSF', (6,), 32, {}),
    ('RealNVP', (64,), 128, {}),
    ('CouplingRQNSF', (32,), 128, {'conditioner_kwargs': {'n_hidden': 32}}),
]


def grad_cases():
    cases = []
    for n, (preset, event_shape, batch, kwargs) in enumerate(GRAD_CASES):
        torch.manual_seed(500 + n)
        flow = Flow(getattr(ref_arch, preset)(event_shape, **kwargs))
        flow.eval()
        x = torch.randn(batch, *event_shape, requires_grad=True)
        w = torch.rand(batch) + 0.5
        sd = {k: v.clone() for k, v in flow.state_dict().items()}
        loss = flow._base_batch_loss((x, w))            # flows.py:199-224
        loss.backward()
        grads = {k: p.grad.clone() for k, p in flow.named_parameters() if p.grad is not None}
        cases.append(dict(preset=preset, event_shape=event_shape, kwargs=kwargs, state_dict=sd, x=x.detach().clone(),
                          w=w, loss=loss.detach().clone(), grad_x=x.grad.clone(), grads=grads))
    return cases


def fit_cases():
    """Loss trajectories of BaseFlow.fit's inner loop (flows.py:379-398) with full-batch, unshuffled
    steps so that they are comparable step by step (SURVEY 8d, check P5)."""
    cases = []
    for n, (preset, event_shape, n_data, lr, data_init) in enumerate((('RealNVP', (3,), 1000, 0.05, False),
                                                                      ('CouplingRQNSF', (4,), 512, 0.01, False),
                                                                      ('MAF', (4,), 512, 0.05, False),
                                                                      ('RealNVP', (3,), 1000, 0.05, True))):
        torch.manual_seed(0)
        x = torch.randn(n_data, *event_shape)
        flow = Flow(getattr(ref_arch, preset)(event_shape))
        sd0 = {k: v.clone() for k, v in flow.state_dict().items()}
        flow.train()
        if not data_init:
            # Keep the constructor's ActNorm parameters.  With a fresh data-dependent init the mean of every
            # normalised activation is exactly zero, so several gradients are pure rounding noise (~1e-9) and Adam's
            # first step (lr * g / (|g| + eps)) turns that noise into O(lr) parameter changes: the trajectory is then
            # not reproducible even between two runs of the reference on different thread counts.
            for layer in flow.bijection.layers:
                if hasattr(layer, 'first_training_batch_pass'):
                    layer.first_training_batch_pass = False
        opt = torch.optim.AdamW(flow.parameters(), lr=lr)
        w = torch.ones(n_data)
        losses = []
        for _ in range(20):
            opt.zero_grad()
            loss = flow._base_batch_loss((x, w))
            losses.append(float(loss))
            loss.backward()
            opt.step()
        flow.eval()
        with torch.no_grad():
            lp = flow.log_prob(x)
        cases.append(dict(preset=preset, event_shape=event_shape, lr=lr, x=x, state_dict0=sd0, losses=losses,
                          data_init=data_init,
                          state_dict20={k: v.clone() for k, v in flow.state_dict().items()}, log_prob20=lp))
    return cases


CONTEXT_CASES = [
    # (preset, event_shape, context_shape, batch_shape)   -- test/constants.py:5 context shapes
    ('RealNVP', (3,), (2,), (7,)),
    ('NICE', (3, 5, 2), (3,), (5, 2)),
    ('CouplingRQNSF', (8,), (3, 5, 2), (9,)),
    ('MAF', (5,), (2,), (11,)),
    ('IAF', (2,), (3, 5, 2), (6,)),
    ('MaskedAutoregressiveRQNSF', (4,), (3,), (5,)),
    ('InverseAutoregressiveRQNSF', (3,), (2,), (4,)),
]


def context_cases():
    """Context-conditioned presets (SURVEY 8f-1): x, context -> z, log_det, log_prob, inverse; gradients of the loss."""
    cases = []
    for n, (preset, event_shape, context_shape, batch_shape) in enumerate(CONTEXT_CASES):
        torch.manual_seed(900 + n)
        flow = Flow(getattr(ref_arch, preset)(event_shape, context_shape=context_shape))
        flow.eval()
        x = torch.randn(*batch_shape, *event_shape)
        c = torch.randn(*batch_shape, *context_shape)
        with torch.no_grad():
            z, ld_f = flow.bijection.forward(x, context=c)
            lp = flow.log_prob(x, context=c)
            xr, ld_r = flow.bijection.inverse(z, context=c)
        sd = {k: v.clone() for k, v in flow.state_dict().items()}
        xg = x.clone().reshape(-1, *event_shape).requires_grad_(True)
        cg = c.reshape(-1, *context_shape)
        loss = flow._base_batch_loss((xg, torch.ones(len(xg)), cg))
        loss.backward()
        grads = {k: p.grad.clone() for k, p in flow.named_parameters() if p.grad is not None and p.numel()}
        cases.append(dict(preset=preset, event_shape=event_shape, context_shape=context_shape, state_dict=sd, x=x,
                          context=c, z=z, ld_f=ld_f, log_prob=lp, xr=xr, ld_r=ld_r, loss=loss.detach().clone(),
                          grad_x=xg.grad.clone(), grads=grads))
    return cases


def main():
    torch.set_num_threads(1)   # fixed reduction order on the generating side
    save(transformer_cases(), 'transformers.pt')
    save(preset_cases(), 'presets.pt')
    save(grad_cases(), 'grads.pt')
    save(fit_cases(), 'fit.pt')
    save(context_cases(), 'context.pt')


if __name__ == '__main__':
    main()
