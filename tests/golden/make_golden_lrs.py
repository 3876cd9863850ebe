"""Golden vectors for the linear-rational-spline and Scale transformers (SURVEY 8f-3), produced by the REAL reference.

Run in the build container only (the reference lives at /root/reference and does not travel to the GPU box):

    python tests/golden/make_golden_lrs.py

Stores tests/golden/lrs.pt: transformer-level cases (inputs, parameters, outputs of forward and inverse, autograd gradients of
a fixed scalar objective), single layers outside the presets (residual conditioner, graphical coupling mask, Linear*
couplings, ElementwiseScale) and preset-level cases (CouplingLRS, MaskedAutoregressiveLRS, InverseAutoregressiveLRS: state_dict,
inputs, log_prob, samples from given noise).  Pins oracle/flow_oracle.py (tests/test_oracle_golden.py) and is the
reference-produced half of tests/test_gpu_lrs.py.
"""
import os
import sys
import warnings

import torch

REF = os.environ.get('TORCHFLOWS_REF', '/root/reference')
sys.path.insert(0, REF)
warnings.filterwarnings('ignore')

from torchflows.flows import Flow  # noqa: E402
from torchflows.bijections.finite.autoregressive import architectures as ref_arch  # noqa: E402
from torchflows.bijections.finite.autoregressive.transformers.linear.affine import Scale  # noqa: E402
from torchflows.bijections.finite.autoregressive.transformers.spline.linear_rational import LinearRational  # noqa: E402

from make_golden import save  # noqa: E402


def with_grads(tr, fn, v, h, g):
    """Outputs of tr.<fn>(v, h) and the gradients of sum(out * cz) + sum(log_det * cl) for fixed random cz, cl."""
    v = v.clone().requires_grad_(True)
    h = h.clone().requires_grad_(True)
    out, ld = getattr(tr, fn)(v, h)
    cz = torch.randn(out.shape, generator=g)
    cl = torch.randn(ld.shape, generator=g)
    ((out * cz).sum() + (ld * cl).sum()).backward()
    return dict(out=out.detach(), ld=ld.detach(), cz=cz, cl=cl, gv=v.grad.clone(), gh=h.grad.clone())


def transformer_cases():
    cases = []
    g = torch.Generator().manual_seed(4321)
    for n_bins in (4, 8, 16):
        for boundary in (5.0, 50.0):
            for scale, h_scale in ((0.3, 1.0), (1.0, 1.0), (3.0, 3.0)):
                event_shape, batch = (5,), 24
                tr = LinearRational(event_shape, n_bins=n_bins, boundary=boundary)
                x = torch.randn(batch, *event_shape, generator=g) * scale * min(boundary, 10.0) / 3
                h = torch.randn(batch, *tr.parameter_shape, generator=g) * h_scale
                fwd = with_grads(tr, 'forward', x, h, g)
                z_in = torch.randn(batch, *event_shape, generator=g) * scale * min(boundary, 10.0) / 3
                inv = with_grads(tr, 'inverse', z_in, h, g)
                cases.append(dict(kind='lrs', n_bins=n_bins, boundary=boundary, event_shape=event_shape, x=x, h=h,
                                  forward=fwd, z_in=z_in, inverse=inv))
    for event_shape, batch in (((5,), 33), ((3, 4), 20)):
        tr = Scale(event_shape)
        x = torch.randn(batch, *event_shape, generator=g)
        h = torch.randn(batch, *tr.parameter_shape, generator=g)
        cases.append(dict(kind='scale', event_shape=event_shape, x=x, h=h, forward=with_grads(tr, 'forward', x, h, g),
                          z_in=x, inverse=with_grads(tr, 'inverse', x, h, g)))
    return cases


PRESET_CASES = [
    ('CouplingLRS', (8,), (64,)),
    ('CouplingLRS', (33,), (40,)),
    ('MaskedAutoregressiveLRS', (12,), (48,)),
    ('InverseAutoregressiveLRS', (10,), (32,)),
]


def preset_cases():
    cases = []
    for n, (preset, event_shape, batch_shape) in enumerate(PRESET_CASES):
        torch.manual_seed(900 + n)
        bij = getattr(ref_arch, preset)(event_shape)
        flow = Flow(bij)
        flow.eval()
        with torch.no_grad():                      # move the conditioners off their near-identity initialisation
            for name, p in flow.named_parameters():
                if 'conditioner_transform' in name:
                    p.add_(0.3 * torch.randn_like(p))
        x = torch.randn(*batch_shape, *event_shape)
        noise = torch.randn(*batch_shape, *event_shape)
        with torch.no_grad():
            z, ld_f = bij.forward(x)
            lp = flow.log_prob(x)
            xs, ld_i = bij.inverse(noise)
            lp_s = flow.base_log_prob(noise) + ld_i
        xg = x.clone().requires_grad_(True)
        loss = flow._base_batch_loss((xg, torch.ones(batch_shape)))
        loss.backward()
        grads = {k: p.grad.clone() for k, p in flow.named_parameters() if p.grad is not None}
        cases.append(dict(preset=preset, event_shape=event_shape, state_dict={k: v.clone() for k, v in flow.state_dict().items()},
                          x=x, noise=noise, z=z, ld_f=ld_f, log_prob=lp, xs=xs, ld_i=ld_i, lp_s=lp_s,
                          loss=loss.detach().clone(), grad_x=xg.grad.clone(), grads=grads))
    return cases


def layer_cases():
    """Single layers outside the presets: residual conditioner, graphical coupling mask, Linear* couplings, ElementwiseScale."""
    from torchflows.bijections.finite.autoregressive import layers as L
    from torchflows.bijections.finite.autoregressive.conditioning.transforms import ResidualFeedForward
    specs = [
        ('RQSCoupling', (10,), dict(conditioner_transform_class=ResidualFeedForward)),
        ('LRSCoupling', (9,), dict(conditioner_transform_class=ResidualFeedForward, conditioner_kwargs=dict(n_layers=4))),
        ('AffineCoupling', (8,), dict(coupling_kwargs=dict(edge_list=[(0, 4), (1, 5), (2, 6), (0, 7)]))),
        ('RQSCoupling', (8,), dict(coupling_kwargs=dict(edge_list=[(0, 1), (2, 3), (5, 3), (5, 7)]))),
        ('LinearAffineCoupling', (6,), {}),
        ('LinearLRSCoupling', (6,), {}),
        ('ElementwiseScale', (6,), {}),
    ]
    cases = []
    for n, (name, event_shape, kwargs) in enumerate(specs):
        torch.manual_seed(700 + n)
        layer = getattr(L, name)(event_shape, **kwargs)
        layer.eval()
        with torch.no_grad():
            for p in layer.parameters():
                p.add_(0.2 * torch.randn_like(p))
        x = torch.randn(40, *event_shape)
        noise = torch.randn(40, *event_shape)
        with torch.no_grad():
            z, ld_f = layer.forward(x)
            xs, ld_i = layer.inverse(noise)
        kw = {k: v for k, v in kwargs.items() if k != 'conditioner_transform_class'}
        cases.append(dict(layer=name, event_shape=event_shape, kwargs=kw,
                          conditioner='ResidualFeedForward' if 'conditioner_transform_class' in kwargs else None,
                          state_dict={k: v.clone() for k, v in layer.state_dict().items()}, x=x, noise=noise, z=z, ld_f=ld_f,
                          xs=xs, ld_i=ld_i))
    return cases


def main():
    torch.manual_seed(0)
    save(dict(transformers=transformer_cases(), presets=preset_cases(), layers=layer_cases()), 'lrs.pt')


if __name__ == '__main__':
    main()
