"""Linear rational spline (LRS) presets as fused flow programs: CouplingLRS, MaskedAutoregressiveLRS and
InverseAutoregressiveLRS with n_bins = 8 run on the generic FP32 kernel (csrc/b2f_flow.cu) and, for the sequential
inverse, on the row-per-thread kernel (csrc/b2f_flow_rows.cuh); gradients come from the fused backward
(csrc/b2f_flow_bwd.cu).  Referees: the reference's own vectors (tests/golden/lrs), the oracle (bit-identical to the
reference in fp32, differentiated in fp64 for gradients) and the same flow forced onto the composite path (conditioner
GEMMs + stand-alone transformer kernel, the sequential direction as the reference's D-step loop)."""
import copy

import pytest
import torch

from oracle.flow_oracle import OracleFlow

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda:0')
PRESETS = ('CouplingLRS', 'MaskedAutoregressiveLRS', 'InverseAutoregressiveLRS')


def close(a, b, what, atol, rtol):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert torch.isfinite(a).all(), what
    err = (a - b).abs() - (atol + rtol * b.abs())
    assert (err <= 0).all(), f'{what}: max abs diff {(a - b).abs().max().item():.3e}, worst excess {err.max().item():.3e}'


def rel_l2(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def close_or_as_good(a, ref32, ref64, what, atol=1e-4, rtol=1e-4):
    """``a`` within atol / rtol of the fp32 referee ``ref32``, or, where the inverse spline amplifies fp32 rounding beyond
    that, at least as close to the fp64 truth ``ref64`` as twice the fp32 referee is."""
    a, r32, r64 = (t.detach().cpu().double() for t in (a, ref32, ref64))
    assert torch.isfinite(a).all(), what
    if ((a - r32).abs() <= atol + rtol * r32.abs()).all():
        return
    err, ref_err = (a - r64).abs().max().item(), (r32 - r64).abs().max().item()
    assert err <= max(atol, 2 * ref_err), f'{what}: {err:.3e} from fp64, the fp32 referee {ref_err:.3e}'


def lrs_layers(module):
    from torchflows_b200.bijections.finite.autoregressive.layers_base import AutoregressiveBijection
    from torchflows_b200.bijections.finite.autoregressive.transformers.spline.linear_rational import LinearRational
    return [m for m in module.modules() if isinstance(m, AutoregressiveBijection) and isinstance(m.transformer, LinearRational)]


def force_composite(flow):
    """A copy of ``flow`` whose LRS layers run as the composite (the second referee)."""
    other = copy.deepcopy(flow)
    for m in lrs_layers(other):
        m._fusable = False
        if hasattr(m, '_fusable_ctx'):
            m._fusable_ctx = False
    return other


def set_quirk(flow, on: bool):
    for m in lrs_layers(flow):
        if hasattr(m, 'sequential_log_det_reference_quirk'):
            m.sequential_log_det_reference_quirk = on


def make_flow(preset, D, seed=0, scale=0.3, actnorm_init=False, **kwargs):
    """A preset with random conditioner weights; ActNorm optionally data-initialised from one training-mode pass."""
    from torchflows_b200 import Flow
    import torchflows_b200.architectures as arch
    torch.manual_seed(seed)
    flow = Flow(getattr(arch, preset)(D, **kwargs))
    with torch.no_grad():
        for name, p in flow.named_parameters():
            if 'conditioner_transform' in name:
                p.add_(scale * torch.randn_like(p))
    flow = flow.to(DEV)
    if actnorm_init:
        flow.train()
        with torch.no_grad():
            flow.log_prob(2.0 * torch.randn(512, D, device=DEV))
    return flow.eval()


def kernel_is_fused():
    from torchflows_b200 import _native as N
    return N.last_flow_kernel() in (N.KERNEL_GENERIC, N.KERNEL_ROWS)


class ExactOracle(OracleFlow):
    """The oracle with the exact log-determinant in the sequential direction (minus the one-pass log-det at the result),
    i.e. what the fused program computes with sequential_log_det_reference_quirk = False and what it differentiates."""

    def _ma_sequential(self, spec, z):
        x, _ = super()._ma_sequential(spec, z)
        return x, -self._ma_one_pass(spec, x, 'forward')[1]


# ---- 1. the reference's vectors, fused -------------------------------------------------------------------------------------
@pytest.mark.parametrize('idx', range(4))
def test_reference_vectors_on_fused_programs(golden, idx):
    from torchflows_b200 import Flow
    import torchflows_b200.architectures as arch
    c = golden('lrs.pt')['presets'][idx]
    flow = Flow(getattr(arch, c['preset'])(c['event_shape']))
    flow.load_state_dict(c['state_dict'])
    flow = flow.to(DEV).eval()
    assert flow.bijection.fused_ops('forward') is not None and flow.bijection.fused_ops('inverse') is not None
    with torch.no_grad():
        lp = flow.log_prob(c['x'].to(DEV))
        assert kernel_is_fused()
        xs, lps = flow._sample_from_base(c['noise'].to(DEV), no_grad=True, return_log_prob=True)
        assert kernel_is_fused()
    close(lp, c['log_prob'], 'log_prob', 1e-4, 1e-4)
    close(xs, c['xs'], 'samples', 1e-4, 1e-4)
    close(lps, c['lp_s'], 'sample log_prob', 1e-4, 1e-4)
    x = c['x'].to(DEV).requires_grad_(True)
    loss = flow._base_batch_loss((x, torch.ones(c['x'].shape[0], device=DEV)))
    assert kernel_is_fused()
    loss.backward()
    close(loss, c['loss'], 'loss', 1e-4, 1e-4)
    assert rel_l2(x.grad, c['grad_x']) < 1e-3
    for name, p in flow.named_parameters():
        if name in c['grads']:
            assert rel_l2(p.grad, c['grads'][name]) < 2e-3, name


# ---- 2. many tiles, ragged tails ----------------------------------------------------------------------------------------
@pytest.mark.parametrize('actnorm_init', [False, True])
@pytest.mark.parametrize('B', [1, 127, 4097, 40000])
@pytest.mark.parametrize('preset,D', [('CouplingLRS', 64), ('MaskedAutoregressiveLRS', 32), ('InverseAutoregressiveLRS', 32)])
def test_many_tiles_against_oracle_and_composite(preset, D, B, actnorm_init):
    flow = make_flow(preset, D, seed=B % 97, actnorm_init=actnorm_init)
    comp = force_composite(flow)
    oracle = OracleFlow(preset, (D,), flow.state_dict(), device='cuda:0')       # the reference's ATen ops, fp32
    oracle64 = OracleFlow(preset, (D,), {k: v.double() for k, v in flow.state_dict().items()}, device='cuda:0')
    g = torch.Generator().manual_seed(B)
    x = (2.0 * torch.randn(B, D, generator=g)).to(DEV)
    noise = torch.randn(B, D, generator=g).to(DEV)
    with torch.no_grad():
        lp = flow.log_prob(x)
        assert kernel_is_fused()
        xs = flow._sample_from_base(noise, no_grad=True)
        assert kernel_is_fused()
        close(lp, oracle.log_prob(x), 'log_prob vs oracle', 1e-4, 1e-4)
        close(lp, comp.log_prob(x), 'log_prob vs composite', 1e-4, 1e-4)
        truth = oracle64.sample_from_noise(noise.double())
        close_or_as_good(xs, oracle.sample_from_noise(noise), truth, 'inverse vs oracle')
        close_or_as_good(xs, comp._sample_from_base(noise, no_grad=True), truth, 'inverse vs composite')


# ---- 3. the sequential direction ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('preset', ['MaskedAutoregressiveLRS', 'InverseAutoregressiveLRS'])
def test_sequential_direction(preset):
    D, B = 24, 3000
    flow = make_flow(preset, D, seed=5)
    comp = force_composite(flow)
    x = 1.5 * torch.randn(B, D, device=DEV)
    noise = torch.randn(B, D, device=DEV)
    with torch.no_grad():
        # reference quirk on (default): the last iteration's log-det, as the composite D-step loop reports it
        if preset == 'MaskedAutoregressiveLRS':
            xs, lps = flow._sample_from_base(noise, no_grad=True, return_log_prob=True)
            xc, lpc = comp._sample_from_base(noise, no_grad=True, return_log_prob=True)
            close(xs, xc, 'samples', 1e-4, 1e-4)
            close(lps, lpc, 'sample log_prob (quirk)', 1e-4, 1e-4)
        else:
            close(flow.log_prob(x), comp.log_prob(x), 'log_prob (quirk)', 1e-4, 1e-4)
        # quirk off: the exact log-det = minus the one-pass log-det at the result
        set_quirk(flow, False)
        bij = flow.bijection
        seq_dir, one_dir = ('inverse', 'forward') if preset == 'MaskedAutoregressiveLRS' else ('forward', 'inverse')
        v = noise if seq_dir == 'inverse' else x
        out, ld_seq = getattr(bij, seq_dir)(v)
        assert kernel_is_fused()
        back, ld_one = getattr(bij, one_dir)(out)
        close(ld_seq, -ld_one, 'exact sequential log-det', 1e-4, 1e-4)
        # round trip through the one-pass direction, against the oracle's own fp32 round trip
        oracle = OracleFlow(preset, (D,), flow.state_dict(), device='cuda:0')
        o_out, _ = getattr(oracle, seq_dir)(v)
        o_back, _ = getattr(oracle, one_dir)(o_out)
        limit = max(1e-5, 2 * (o_back - v).abs().max().item())
        assert (back - v).abs().max().item() <= limit, ((back - v).abs().max().item(), limit)


# ---- 4. gradients at scale ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('preset', PRESETS)
def test_fused_backward_against_fp64_oracle(preset):
    D, B = 16, 4096
    flow = make_flow(preset, D, seed=11, actnorm_init=True)
    set_quirk(flow, False)
    x_cpu = 1.5 * torch.randn(B, D)
    x = x_cpu.to(DEV).requires_grad_(True)
    loss = flow._base_batch_loss((x, torch.ones(B, device=DEV)))
    assert kernel_is_fused()
    loss.backward()
    sd64 = {k: v.detach().cpu().double() for k, v in flow.state_dict().items()}
    oracle = ExactOracle(preset, (D,), sd64)
    leaves = {}
    for name, p in flow.named_parameters():
        if p.grad is not None and p.numel() > 0:
            leaves[name] = sd64[name].clone().requires_grad_(True)
            oracle.sd[name] = leaves[name]
    x64 = x_cpu.double().requires_grad_(True)
    loss64 = oracle.batch_loss(x64)
    loss64.backward()
    close(loss, loss64, 'loss', 1e-4, 1e-4)
    assert rel_l2(x.grad, x64.grad) < 1e-3
    assert leaves
    for name, p in flow.named_parameters():
        if name in leaves:
            assert rel_l2(p.grad, leaves[name].grad) < 2e-3, name


# ---- 5. tails and edges ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('layer_name', ['LRSCoupling', 'LRSForwardMaskedAutoregressive', 'LRSInverseMaskedAutoregressive'])
def test_outside_the_boundary_is_identity_inside_a_program(layer_name):
    from torchflows_b200.bijections.finite.autoregressive import layers as L
    from torchflows_b200.bijections.base import BijectiveComposition
    D = 16
    torch.manual_seed(3)
    comp = BijectiveComposition([getattr(L, layer_name)((D,), transformer_kwargs={'boundary': 2.0})]).to(DEV)
    assert comp.fused_ops('forward') is not None and comp.fused_ops('inverse') is not None
    sign = torch.where(torch.rand(257, D) < 0.5, -1.0, 1.0)
    x = (sign * (2.0 + 3.0 * torch.rand(257, D))).to(DEV)          # every element at or beyond +-boundary
    with torch.no_grad():
        for direction in ('forward', 'inverse'):
            y, ld = getattr(comp, direction)(x)
            assert kernel_is_fused()
            assert torch.equal(y, x), direction
            assert torch.equal(ld, torch.zeros_like(ld)), direction


@pytest.mark.parametrize('preset', PRESETS)
def test_empty_batch(preset):
    flow = make_flow(preset, 8)
    with torch.no_grad():
        assert flow.log_prob(torch.empty(0, 8, device=DEV)).shape == (0,)
        assert flow._sample_from_base(torch.empty(0, 8, device=DEV), no_grad=True).shape == (0, 8)


@pytest.mark.parametrize('preset', PRESETS)
def test_other_bin_counts_stay_composite(preset):
    D = 8
    flow = make_flow(preset, D, transformer_kwargs={'n_bins': 4})
    assert flow.bijection.fused_ops('forward') is None and flow.bijection.fused_ops('inverse') is None
    oracle = OracleFlow(preset, (D,), flow.state_dict(), n_bins=4, device='cuda:0')
    x, noise = torch.randn(300, D, device=DEV), torch.randn(300, D, device=DEV)
    with torch.no_grad():
        close(flow.log_prob(x), oracle.log_prob(x), 'log_prob', 1e-4, 1e-4)
        close(flow._sample_from_base(noise, no_grad=True), oracle.sample_from_noise(noise), 'samples', 1e-4, 1e-4)


# ---- 6. context ----------------------------------------------------------------------------------------------------------
def test_context_conditioned_coupling_is_one_program():
    from torchflows_b200 import _native as N
    D, B = 12, 1000
    flow = make_flow('CouplingLRS', D, seed=7, context_shape=(3,))
    comp = force_composite(flow)
    x, ctx = torch.randn(B, D, device=DEV), torch.randn(B, 3, device=DEV)
    for direction in ('forward', 'inverse'):
        segs = flow.bijection._segments(direction, ctx)
        assert len(segs) == 1 and segs[0][0] == 'ops', direction
        couplings = [op for op in segs[0][1] if op.kind == N.OP_COUPLING]
        assert couplings and all(op.flags & N.FLAG_ROW_BIAS for op in couplings)
    with torch.no_grad():
        z, ld = flow.bijection.forward(x, context=ctx)
        zc, ldc = comp.bijection.forward(x, context=ctx)
        close(z, zc, 'forward', 1e-4, 1e-4)
        close(ld, ldc, 'forward log-det', 1e-4, 1e-4)
        xr, ldi = flow.bijection.inverse(z, context=ctx)
        close(xr, x, 'round trip', 1e-4, 1e-4)
        close(ldi, -ld, 'inverse log-det', 1e-4, 1e-4)
    grads = []
    for f in (flow, comp):
        xg, cg = x.clone().requires_grad_(True), ctx.clone().requires_grad_(True)
        f.zero_grad()
        loss = f._base_batch_loss((xg, torch.ones(B, device=DEV), cg))
        loss.backward()
        grads.append((float(loss), xg.grad, cg.grad, {n: p.grad.clone() for n, p in f.named_parameters() if p.grad is not None}))
    (l1, gx1, gc1, gp1), (l2, gx2, gc2, gp2) = grads
    assert abs(l1 - l2) <= 1e-4 * (1 + abs(l2))
    assert rel_l2(gx1, gx2) < 1e-3 and rel_l2(gc1, gc2) < 1e-3
    assert gp1.keys() == gp2.keys()
    for n in gp1:
        assert rel_l2(gp1[n], gp2[n]) < 2e-3, n


# ---- 7. training and sampling -------------------------------------------------------------------------------------------
@pytest.mark.parametrize('preset', ['InverseAutoregressiveLRS', 'MaskedAutoregressiveLRS'])
def test_fit_follows_composite_trajectory(preset):
    """20 Flow.fit steps (one full batch per epoch, ActNorm initialised on the first) from identical weights.  The exact
    sequential log-det on both sides: the fused backward differentiates it (the reference's last-iteration value has no
    fused gradient)."""
    D, B = 16, 2048
    flow = make_flow(preset, D, seed=13)
    set_quirk(flow, False)
    comp = force_composite(flow)
    x = 1.5 * torch.randn(B, D, device=DEV)
    losses = []
    for f in (flow, comp):
        per_step = []
        hook = f._base_batch_loss

        def recording(batch, *args, _hook=hook, _log=per_step, **kwargs):
            loss = _hook(batch, *args, **kwargs)
            if torch.is_grad_enabled():
                _log.append(float(loss.detach()))
            return loss
        f._base_batch_loss = recording
        f.fit(x, n_epochs=20, batch_size=B, shuffle=False, keep_best_weights=False)
        losses.append(per_step)
    fused, composite = losses
    assert len(fused) == len(composite) == 20
    for i, (a, b) in enumerate(zip(fused, composite)):
        assert abs(a - b) <= 1e-4 * (1 + abs(b)), (i, a, b)


@pytest.mark.parametrize('preset', PRESETS)
def test_sample_is_seeded_and_matches_forward_of_its_noise(preset):
    from torchflows_b200 import _native as N
    D, n = 16, 50000
    flow = make_flow(preset, D, seed=17)
    torch.manual_seed(123)
    s1 = flow.sample(n, no_grad=True)
    assert kernel_is_fused() and N.last_flow_kernel() != N.KERNEL_TCQ
    torch.manual_seed(123)
    s2 = flow.sample(n, no_grad=True)
    assert torch.equal(s1, s2)
    # the same draws, materialised by the library's Philox stream, pushed through the inverse directly
    torch.manual_seed(123)
    from torchflows_b200 import _program as prog
    seed, offset = prog.next_noise_stream(DEV, n * D)
    noise = torch.empty(n, D, device=DEV)
    N.check(N.lib().b2f_philox_normal(N.ptr(noise), n, D, None, None, seed, offset, N.stream_ptr(DEV)))
    with torch.no_grad():
        direct = flow._sample_from_base(noise, no_grad=True)
    close(s1.mean(0), direct.mean(0), 'sample mean', 1e-4, 1e-4)
    close(s1.std(0), direct.std(0), 'sample std', 1e-4, 1e-4)
