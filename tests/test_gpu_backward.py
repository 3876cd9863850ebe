"""The fused backward kernel (csrc/b2f_flow_bwd.cu) in every tile shape and GEMM path it can launch, against torch
autograd through the oracle in fp32 and fp64.

bwd_tile_shape() picks rows per tile TM in {32, 64}, threads NT and per-warp staging of the spline output weights from
the program's shared-memory footprint; inside a shape a spline layer takes the tensor-core GEMM path of its hidden-width
bucket (H <= 7, 15, 23, 31) or the scalar one (H > 31, `precise`, no staging).  The kernel starts either from the layer
inputs the tensor-core forward saved (B2F_FLOW_WS_FILLED) or recomputes them.  Every case asserts through
b2f_flow_backward_shape which shape launched.

Referee (as tests/test_gpu_training.py at the benchmark shapes): a gradient passes when it is within 1e-4 relative L2 of
the fp32 oracle, or else at most max(1e-4, 3x the fp32 rounding level) from the fp64 oracle.  The rounding level is the
larger distance from fp64 of two fp32 autograd runs of the oracle, on the CPU and on the GPU: one fp32 run alone can land
close to fp64 by chance on a small, heavily cancelled tensor (a MADE layer's 4 hidden biases).  dL/dx is checked
per row as well (max over rows of |row difference| / |row|), so a defect in a few rows cannot hide in the batch norm.
The loss is -sum(w * log_prob) / (B * D) without the regulariser, whose gradient would mask the data term."""
import pytest
import torch

from tests.test_gpu_lrs_fused import ExactOracle

pytestmark = pytest.mark.gpu

DEV = torch.device('cuda:0')
# every admissible forced shape: TM = 32 with 1..12 warps, TM = 64 with 1..6 warps per 32-row group
SHAPES = [(32, 32 * w) for w in range(1, 13)] + [(64, 64 * w) for w in range(1, 7)]
FUSED_KERNELS = (1, 2, 3)            # KERNEL_GENERIC, KERNEL_TC, KERNEL_ROWS
WORST = {}                           # largest forced-vs-default distance seen, reported at the end of the module


def rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def row_rel(a, b):
    n = b.norm(dim=1)
    live = n > 0
    assert (a[~live] == 0).all(), 'dL/dx of a row without loss weight is not zero'
    return ((a - b).norm(dim=1)[live] / n[live]).max().item() if live.any() else 0.0


def make_flow(preset, D, seed=0, **kwargs):
    """A preset whose elementwise and ActNorm layers are not the identity and whose conditioners are perturbed, with the
    exact log-det in the sequential direction (the one the fused backward differentiates)."""
    from torchflows_b200 import Flow
    import torchflows_b200.architectures as arch
    torch.manual_seed(seed)
    flow = Flow(getattr(arch, preset)(D, **kwargs))
    with torch.no_grad():
        for name, p in flow.named_parameters():
            if name.endswith('.value'):
                p.add_(0.3 * torch.randn_like(p))
            elif 'conditioner_transform' in name:
                p.add_((0.5 / p.shape[1] ** 0.5 if p.dim() == 2 else 0.1) * torch.randn_like(p))
    for m in flow.modules():
        if hasattr(m, 'sequential_log_det_reference_quirk'):
            m.sequential_log_det_reference_quirk = False
    return flow.to(DEV).eval()


def query_shape(flow, D, precise=False):
    from torchflows_b200 import _native as N, _program as P
    ops = flow.bijection.fused_ops('forward')
    assert ops is not None
    return N.flow_backward_shape(P.op_dicts(ops), D, N.FLOW_MODE_PRECISE if precise else 0)


def fused_grads(flow, x, w, precise=False, kernel=None, n_rows=None):
    """(loss, dL/dx, {name: dL/dparam}) from the fused program, all float64 on the CPU; n_rows as in oracle_grads."""
    from torchflows_b200 import _native as N, set_math_mode
    B, D = x.shape
    flow.zero_grad(set_to_none=True)
    xg = x.to(DEV).clone().requires_grad_(True)
    previous = set_math_mode('precise') if precise else None
    try:
        lp = flow.log_prob(xg)
        ran = N.last_flow_kernel()
        loss = -(lp * w.to(DEV)).sum() / ((n_rows or B) * D)
        loss.backward()
    finally:
        if previous is not None:
            set_math_mode(previous)
    assert ran in FUSED_KERNELS and (kernel is None or ran == kernel), ran
    assert flow.bijection.fused_ops('forward') is not None
    assert all(l._fusable for l in flow.bijection.layers if hasattr(l, '_fusable'))
    grads = {k: p.grad.detach().cpu().double() for k, p in flow.named_parameters() if p.grad is not None}
    return float(loss.detach()), xg.grad.detach().cpu().double(), grads


def oracle_grads(flow, preset, x, w, dtype, n_rows=None, device='cpu'):
    """The same loss by torch autograd through the oracle in `dtype` on `device`; n_rows: the batch size of the loss
    normaliser when x holds only the weighted rows of a larger batch."""
    names = {k for k, p in flow.named_parameters() if p.requires_grad}          # ActNorm values are frozen
    leaves = {k: v.detach().to(device).clone().to(dtype).requires_grad_(k in names) if v.is_floating_point() else v.to(device)
              for k, v in flow.state_dict().items()}
    B, D = x.shape
    o = ExactOracle(preset, (D,), {})
    o.sd = leaves
    xg = x.detach().to(device).clone().to(dtype).requires_grad_(True)
    loss = -(o.log_prob(xg) * w.to(device, dtype)).sum() / ((n_rows or B) * D)
    loss.backward()
    return float(loss.detach()), xg.grad.cpu().double(), {k: leaves[k].grad.cpu().double() for k in names
                                                          if leaves[k].grad is not None}


def referees(flow, preset, x, w, n_rows=None):
    """fp32 autograd through the oracle on the CPU and on the GPU (the same ATen ops, other kernels: two independent fp32
    roundings of one computation), and fp64 autograd on the CPU."""
    return (oracle_grads(flow, preset, x, w, torch.float32, n_rows), oracle_grads(flow, preset, x, w, torch.float64, n_rows),
            oracle_grads(flow, preset, x, w, torch.float32, n_rows, device=DEV))


def fp32_floor(a32, b32, r64, dist=None):
    """How far fp32 rounding alone takes this computation from fp64: the larger of the two fp32 oracles' distances."""
    dist = dist or rel
    return max(dist(a32, r64), dist(b32, r64))


def referee(what, ours, r32, r64, r32g):
    if r64.norm() == 0:
        assert ours.abs().max().item() < 1e-6, what
        return
    e32 = rel(ours, r32)
    if e32 < 1e-4:
        return
    e64, ref = rel(ours, r64), fp32_floor(r32, r32g, r64)
    assert e64 <= max(1e-4, 3 * ref), f'{what}: {e32:.2e} from fp32, {e64:.2e} from fp64, fp32 oracles {ref:.2e} from fp64'


def check(ours, ref32, ref64, ref32g, what=''):
    (loss, gx, g), (l32, gx32, g32), (l64, gx64, g64), (_, gx32g, g32g) = ours, ref32, ref64, ref32g
    assert abs(loss - l64) <= 1e-4 * abs(l64) + 1e-9, (what, loss, l64)
    referee(f'{what} dL/dx', gx, gx32, gx64, gx32g)
    e32 = row_rel(gx, gx32)
    if e32 >= 1e-4:
        e64, ref = row_rel(gx, gx64), fp32_floor(gx32, gx32g, gx64, row_rel)
        assert e64 <= max(1e-4, 3 * ref), f'{what} dL/dx per row: {e32:.2e} from fp32, {e64:.2e} from fp64 (oracle {ref:.2e})'
    assert len(g64) >= 4 and g64.keys() <= g.keys(), (what, sorted(g64.keys() - g.keys()))
    for k in g64:
        referee(f'{what} {k}', g[k], g32[k], g64[k], g32g[k])


def batch(B, D, seed):
    g = torch.Generator().manual_seed(seed)
    return 1.2 * torch.randn(B, D, generator=g), 0.5 + torch.rand(B, generator=g)


# ---- a. every admissible forced shape ---------------------------------------------------------------------------------
PROGRAMS = {                          # name: preset, D, precise
    'rq-mma': ('CouplingRQNSF', 64, False),
    'rq-precise': ('CouplingRQNSF', 64, True),
    'realnvp': ('RealNVP', 64, False),
    'nice': ('NICE', 48, False),
    'maf': ('MAF', 64, False),
    'made-rq': ('MaskedAutoregressiveRQNSF', 32, False),
    'iaf-seq': ('IAF', 32, False),
    'iarq-seq': ('InverseAutoregressiveRQNSF', 16, False),
    'lrs': ('CouplingLRS', 32, False),
}
B_FORCED = 229                        # ragged last tile for TM = 32 (5 rows) and TM = 64 (37 rows)


@pytest.fixture(scope='module')
def programs():
    """Per program, built once: the flow, its batch, the fp32 / fp64 oracle gradients, the default shape and its gradients."""
    cache = {}

    def get(name):
        if name not in cache:
            preset, D, precise = PROGRAMS[name]
            flow = make_flow(preset, D, seed=list(PROGRAMS).index(name) + 1)
            x, w = batch(B_FORCED, D, seed=D)
            refs = referees(flow, preset, x, w)
            cache[name] = (flow, x, w, refs, query_shape(flow, D, precise), fused_grads(flow, x, w, precise))
        return cache[name]
    yield get
    if WORST:
        print('\nworst relative L2 of a forced shape from the default shape: ' +
              ', '.join(f'{k} {v:.2e}' for k, v in sorted(WORST.items())))


@pytest.mark.parametrize('TM,NT', SHAPES)
@pytest.mark.parametrize('name', list(PROGRAMS))
def test_every_forced_shape_against_oracle_and_default_shape(programs, monkeypatch, name, TM, NT):
    """Only the reduction order differs from the default shape, so every gradient is within max(1e-5, the fp32 rounding
    level of the same computation) relative L2 of the default shape's: a reordered fp32 sum cannot be expected to agree
    more closely than that.  Worst observed on a B200 at 1000 W: 1.6e-5 (MaskedAutoregressiveRQNSF(32), the first layer's
    hidden-bias gradient, whose fp32 oracle is 3.6e-5 from fp64); below 1e-5 for every other program."""
    flow, x, w, refs, default, dgrads = programs(name)
    preset, D, precise = PROGRAMS[name]
    assert default is not None
    monkeypatch.setenv('B2F_BWD_TM', str(TM))
    monkeypatch.setenv('B2F_BWD_NT', str(NT))
    assert query_shape(flow, D, precise) == (TM, NT, default[2])
    ours = fused_grads(flow, x, w, precise)
    check(ours, *refs, what=f'{name} {TM}x{NT}')
    (_, gx32, g32), (_, gx64, g64), (_, gx32g, g32g) = refs
    pairs = [('dL/dx', ours[1], dgrads[1], fp32_floor(gx32, gx32g, gx64))] + \
            [(k, ours[2][k], dgrads[2][k], fp32_floor(g32[k], g32g[k], g64[k]) if k in g64 else 0.0) for k in dgrads[2]]
    for k, a, b, floor in pairs:
        e = rel(a, b)
        WORST[name] = max(WORST.get(name, 0.0), e)
        assert e <= max(1e-5, floor), (name, TM, NT, k, e, floor)


def test_default_shapes_of_the_forced_programs(programs):
    expect = {'rq-mma': (32, 384, 24 * 15), 'rq-precise': (64, 256, 0), 'made-rq': (32, 384, 24 * 5)}
    for name in PROGRAMS:
        flow, x, w, refs, default, ours = programs(name)
        assert default == expect.get(name, (64, 256, 0)), (name, default)
        check(ours, *refs, what=name)


# ---- b. entry modes: layer inputs saved by the tensor-core forward, or recomputed ---------------------------------------
@pytest.mark.parametrize('preset,D', [('CouplingRQNSF', 64), ('MaskedAutoregressiveRQNSF', 32)])
def test_saved_and_recomputed_layer_inputs(monkeypatch, preset, D):
    from torchflows_b200 import _native as N
    flow = make_flow(preset, D, seed=3)
    assert sum(l.__class__.__name__.startswith('Reverse') for l in flow.bijection.layers) % 2 == 0
    x, w = batch(B_FORCED, D, seed=4)
    refs = referees(flow, preset, x, w)
    saved = fused_grads(flow, x, w, kernel=N.KERNEL_TC)
    check(saved, *refs, what='saved inputs')
    monkeypatch.setenv('B2F_DISABLE_TC', '1')
    recomputed = fused_grads(flow, x, w, kernel=N.KERNEL_GENERIC)
    check(recomputed, *refs, what='recomputed inputs')


# ---- c. both sides of every tensor-core GEMM bucket, and the scalar path above it ---------------------------------------
@pytest.mark.parametrize('H', [7, 8, 15, 16, 23, 24, 31, 32, 40])
@pytest.mark.parametrize('preset', ['CouplingRQNSF', 'MaskedAutoregressiveRQNSF'])
def test_gemm_buckets(preset, H):
    D = 32
    flow = make_flow(preset, D, seed=H, conditioner_kwargs={'n_hidden': H})
    shape = query_shape(flow, D)
    assert shape is not None and shape[2] == (24 * (H + 1) if H <= 31 else 0), shape
    x, w = batch(3 * shape[0] + 5, D, seed=H)
    refs = referees(flow, preset, x, w)
    check(fused_grads(flow, x, w), *refs, what=f'H={H}')


# ---- d. the shapes default-width presets reach at large D ---------------------------------------------------------------
@pytest.mark.parametrize('preset,D,TM,NT,staged', [
    ('CouplingRQNSF', 352, 32, 256, True), ('CouplingRQNSF', 480, 32, 128, True), ('CouplingRQNSF', 608, 32, 128, False),
    ('RealNVP', 304, 32, 256, False), ('RealNVP', 608, 32, 128, False), ('MAF', 320, 32, 256, False),
    ('MAF', 640, 32, 128, False), ('MaskedAutoregressiveRQNSF', 496, 32, 256, True),
    ('MaskedAutoregressiveRQNSF', 576, 32, 128, True), ('CouplingLRS', 272, 32, 256, False),
    ('CouplingLRS', 560, 32, 128, False), ('IAF', 320, 32, 256, False), ('InverseAutoregressiveRQNSF', 128, 64, 256, False)])
def test_natural_shape_ladder(preset, D, TM, NT, staged):
    flow = make_flow(preset, D, seed=D)
    shape = query_shape(flow, D)
    assert shape is not None and shape[:2] == (TM, NT) and (shape[2] > 0) == staged, shape
    x, w = batch(3 * TM + 5, D, seed=D)
    refs = referees(flow, preset, x, w)
    check(fused_grads(flow, x, w), *refs, what=f'{preset}({D})')


# ---- e. the last partial tile in isolation ------------------------------------------------------------------------------
@pytest.mark.parametrize('forced', [None, (32, 128), (64, 192)], ids=['default', '32x128', '64x192'])
@pytest.mark.parametrize('preset,D', [('CouplingRQNSF', 16), ('MAF', 16)])
def test_last_partial_tile_in_isolation(monkeypatch, preset, D, forced):
    """Weights only on the rows of the last partial tile: every parameter gradient comes from those rows (and the padding
    rows of that tile must contribute nothing).  Weights zero on exactly those rows: the gradients of the batch truncated to
    whole tiles.  Batches of one row, TM - 1, TM + 1 and more than two tiles per SM."""
    flow = make_flow(preset, D, seed=21)
    if forced:
        monkeypatch.setenv('B2F_BWD_TM', str(forced[0]))
        monkeypatch.setenv('B2F_BWD_NT', str(forced[1]))
    TM = query_shape(flow, D)[0]
    assert forced is None or query_shape(flow, D)[:2] == forced
    for B in (1, TM - 1, TM + 1, 2 * 148 * TM + 17):
        x, w = batch(B, D, seed=B)
        full = (B // TM) * TM
        tail_w = torch.zeros(B)
        tail_w[full:] = w[full:]
        ours = fused_grads(flow, x, tail_w)
        refs = referees(flow, preset, x[full:], w[full:], n_rows=B)
        assert (ours[1][:full] == 0).all()
        check((ours[0], ours[1][full:], ours[2]), *refs, what=f'B={B} tail only')

        head_w = w.clone()
        head_w[full:] = 0.0
        ours = fused_grads(flow, x, head_w)
        assert (ours[1][full:] == 0).all()
        if full == 0:
            assert ours[0] == 0.0 and all((g == 0).all() for g in ours[2].values()), B
            continue
        trunc = fused_grads(flow, x[:full], w[:full], n_rows=B)      # same normaliser: the same per-row seeds
        assert abs(ours[0] - trunc[0]) <= 1e-6 * abs(trunc[0]), B
        assert rel(ours[1][:full], trunc[1]) <= 1e-6, B
        for k, g in trunc[2].items():
            assert rel(ours[2][k], g) <= 1e-6, (B, k, rel(ours[2][k], g))


# ---- f. context-conditioned couplings: per-row hidden biases and per-row elementwise parameters --------------------------
CONTEXT_CASES = [('RealNVP', 8, (3,)), ('CouplingRQNSF', 12, (5,))]


@pytest.fixture(scope='module')
def context_flows():
    cache = {}

    def get(case):
        if case not in cache:
            from torchflows_b200 import Flow
            import torchflows_b200.architectures as arch
            preset, D, ctx = case
            torch.manual_seed(D)
            flow = Flow(getattr(arch, preset)(D, context_shape=ctx)).to(DEV).eval()
            with torch.no_grad():
                for name, p in flow.named_parameters():
                    if 'conditioner_transform' in name:
                        p.add_(0.3 * torch.randn_like(p))
            g = torch.Generator().manual_seed(D)
            x, c = torch.randn(B_FORCED, D, generator=g).to(DEV), torch.randn(B_FORCED, *ctx, generator=g).to(DEV)
            cache[case] = (flow, x, c, context_grads(flow, x, c, fused=False))
        return cache[case]
    return get


def context_grads(flow, x, c, fused):
    from torchflows_b200 import _native as N
    for l in flow.bijection.layers:
        if hasattr(l, '_fusable_ctx'):
            l._fusable_ctx = fused
        if hasattr(l, 'fuse_context'):
            l.fuse_context = fused
    try:
        xg, cg = x.clone().requires_grad_(True), c.clone().requires_grad_(True)
        flow.zero_grad(set_to_none=True)
        z, ld = flow.bijection.forward(xg, context=cg)
        lp = flow.log_prob(xg, context=cg)
        if fused:
            assert N.last_flow_kernel() == N.KERNEL_GENERIC
        (lp.mean() + 0.1 * z.square().mean()).backward()
    finally:
        for l in flow.bijection.layers:
            if hasattr(l, '_fusable_ctx'):
                l._fusable_ctx = True
            if hasattr(l, 'fuse_context'):
                l.fuse_context = True
    return xg.grad, cg.grad, {k: p.grad.clone() for k, p in flow.named_parameters() if p.grad is not None}


@pytest.mark.parametrize('TM,NT', [(32, 64), (32, 384), (64, 64), (64, 384)])
@pytest.mark.parametrize('case', CONTEXT_CASES, ids=[p for p, _, _ in CONTEXT_CASES])
def test_context_couplings_in_forced_shapes(context_flows, monkeypatch, case, TM, NT):
    from torchflows_b200 import _native as N, _program as P
    flow, x, c, comp = context_flows(case)
    preset, D, _ = case
    monkeypatch.setenv('B2F_BWD_TM', str(TM))
    monkeypatch.setenv('B2F_BWD_NT', str(NT))
    segs = flow.bijection._segments('forward', c)
    assert [k for k, _ in segs] == ['ops']
    assert any(op.flags & N.FLAG_ROW_BIAS for op in segs[0][1] if op.kind == N.OP_COUPLING)
    assert any(op.flags & N.FLAG_ROW_BIAS for op in segs[0][1] if op.kind == N.OP_ELEMENTWISE)
    shape = N.flow_backward_shape(P.op_dicts(segs[0][1]), D)
    assert shape is not None and shape[:2] == (TM, NT), shape
    fused = context_grads(flow, x, c, fused=True)
    tol = 5e-3 if 'RQNSF' in preset else 2e-4
    assert rel(fused[0].cpu().double(), comp[0].cpu().double()) < tol, 'd/dx'
    assert rel(fused[1].cpu().double(), comp[1].cpu().double()) < tol, 'd/dcontext'
    assert fused[2].keys() == comp[2].keys()
    for k, g in comp[2].items():
        if g.norm() > 0:
            assert rel(fused[2][k].cpu().double(), g.cpu().double()) < tol, k
