"""CPU tests: package structure, lowering to flow programs, weight tile layout, C-ABI exports, data-parallel
helpers over gloo (world_size 2).  No kernel is launched here."""
import ctypes
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_import_paths_and_presets():
    from torchflows_b200 import Flow                                      # README spelling
    from torchflows_b200.architectures import RealNVP as A                # README spelling
    from torchflows_b200.flows import Flow as F2                          # reference module path
    from torchflows_b200.bijections.finite.autoregressive.architectures import (   # reference module path
        NICE, RealNVP, MAF, IAF, CouplingRQNSF, MaskedAutoregressiveRQNSF, InverseRealNVP, InverseAutoregressiveRQNSF)
    assert Flow is F2 and A is RealNVP
    expected = {  # SURVEY Appendix A.1: conditioner shapes and parameter counts
        (RealNVP, 3): 86, (RealNVP, 64): 2514, (NICE, 64): 1614, (CouplingRQNSF, 256): 112930,
        (MAF, 128): 6412, (IAF, 128): 6412, (MaskedAutoregressiveRQNSF, 128): 44044}
    for (cls, d), n in expected.items():
        bij = cls(d)
        assert sum(p.numel() for p in bij.parameters()) == n, (cls.__name__, d)
        assert len(bij.layers) == 9


def test_state_dict_layout_matches_reference(golden):
    import torchflows_b200.architectures as arch
    from torchflows_b200 import Flow
    for c in golden('presets.pt'):
        flow = Flow(getattr(arch, c['preset'])(c['event_shape'], **c['kwargs']))
        ours = flow.state_dict()
        assert list(ours.keys()) == list(c['state_dict'].keys())
        for k, v in c['state_dict'].items():
            assert ours[k].shape == v.shape, k
        flow.load_state_dict(c['state_dict'])
        # ActNorm parameters are frozen, the rest trainable (layers.py:49)
        assert not flow.bijection.layers[3].value.requires_grad and flow.bijection.layers[0].value.requires_grad


def test_made_masks_match_reference(golden):
    import torchflows_b200.architectures as arch
    for c in golden('presets.pt'):
        if c['preset'] not in ('MAF', 'IAF', 'MaskedAutoregressiveRQNSF', 'InverseAutoregressiveRQNSF'):
            continue
        bij = getattr(arch, c['preset'])(c['event_shape'])
        for i in (2, 5):
            for j in (0, 2):
                k = f'bijection.layers.{i}.conditioner_transform.sequential.{j}.mask'
                assert torch.equal(bij.layers[i].conditioner_transform.sequential[j].mask, c['state_dict'][k])
        fin = bij.layers[2]._fin_steps
        d = bij.n_dim
        assert torch.equal(fin, ((torch.arange(len(fin)) % (d - 1)) + 1).to(torch.int32))


def test_lowering_programs():
    from torchflows_b200 import _native as N
    from torchflows_b200.architectures import RealNVP, MAF, IAF, CouplingRQNSF
    bij = CouplingRQNSF(256).eval()
    fwd, inv = bij.lower('forward'), bij.lower('inverse')
    assert [o.kind for o in fwd] == [0, 1, 2, 0, 1, 2, 0, 0, 0]
    assert [o.kind for o in inv] == [0, 0, 0, 2, 1, 0, 2, 1, 0]
    assert [o.tkind for o in fwd if o.kind == 2] == [N.T_RQ_FWD] * 2 and [o.tkind for o in inv if o.kind == 2] == [N.T_RQ_INV] * 2
    # ElementwiseAffine forward is AFFINE_FWD, ActNorm forward is AFFINE_INV, and they swap in the inverse direction
    assert [o.tkind for o in fwd if o.kind == 0] == [2, 3, 3, 2, 3] and [o.tkind for o in inv if o.kind == 0] == [2, 3, 2, 2, 3]
    assert fwd[2].n_hidden == 17 and fwd[2].n_bins == 8 and fwd[2].boundary == 50.0
    assert [o.kind for o in MAF(8).eval().lower('forward')].count(N.OP_MADE) == 2
    assert [o.kind for o in MAF(8).eval().lower('inverse')].count(N.OP_MADE_SEQ) == 2
    assert [o.kind for o in IAF(8).eval().lower('forward')].count(N.OP_MADE_SEQ) == 2
    # a fresh module is in training mode: ActNorm wants a data-dependent init, so nothing is fused yet
    assert RealNVP(4).lower('forward') is None and RealNVP(4).eval().lower('forward') is not None
    # non-default conditioner depth is decided at construction: composite, not fused
    deep = RealNVP(4, conditioner_kwargs={'n_layers': 3}).eval()
    assert deep.layers[2].lower('forward') is None and deep.lower('forward') is None
    # context-conditioned couplings / elementwise layers are composites; MADE layers stay fused (the context provably
    # never reaches their outputs), ActNorm and the permutations ignore the context
    ctx = RealNVP(4, context_shape=(2,)).eval()
    assert ctx.lower('forward') is None and ctx.layers[2].lower('forward') is None and ctx.layers[3].lower('forward')
    assert MAF(4, context_shape=(2,)).eval().layers[2].lower('forward') is not None


def test_tile_layout_round_trip():
    from torchflows_b200 import _program as prog
    torch.manual_seed(0)
    for n_elem, P, H in ((128, 23, 17), (32, 2, 9), (5, 1, 4)):
        W = torch.randn(n_elem * P, H)
        T = prog.to_tile_layout(W, n_elem, P)
        PP = prog.padded(P)
        assert T.shape == (n_elem, H, PP) and T.is_contiguous()
        for e, p, j in ((0, 0, 0), (n_elem - 1, P - 1, H - 1), (n_elem // 2, P // 2, H // 2)):
            assert T[e, j, p] == W[e * P + p, j]
        assert (T[..., P:] == 0).all()
        assert torch.equal(prog.from_tile_layout(T, n_elem, P), W)


def test_c_abi_exports_every_declared_symbol():
    """The shared library loads and exports every entry point include/b2f.h declares (no compute calls here)."""
    from torchflows_b200 import _native as N
    hdr = open(os.path.join(ROOT, 'include', 'b2f.h')).read()
    names = set(re.findall(r'\b(b2f_[a-z_0-9]+)\s*\(', hdr))
    assert {'b2f_flow_apply', 'b2f_flow_backward', 'b2f_transformer_apply', 'b2f_column_stats'} <= names
    lib = ctypes.CDLL(N.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), n
    L = N.lib()
    assert L.b2f_abi_version() == 1
    assert L.b2f_params_per_element(N.T_RQ_FWD, 8) == 23 and L.b2f_padded_params(23) == 24
    assert ctypes.sizeof(N.Op) == 24 + 12 * 8
    # without a GPU a compute call fails loudly instead of falling back
    if not torch.cuda.is_available():
        with pytest.raises(N.B2FError):
            N.flow_apply([], torch.zeros(2, 2))
        from torchflows_b200 import Flow
        from torchflows_b200.architectures import NICE
        with pytest.raises(N.B2FError):
            Flow(NICE(4)).eval().log_prob(torch.zeros(3, 4))


def test_product_never_touches_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's CPU legs may use oracle/."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'torchflows_b200')):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, os.path.join(dirpath, f)
                assert 'b2f_oracle' not in src.replace('oracle/b2f_oracle.c', ''), os.path.join(dirpath, f)


def test_shard_bounds_cover_batch():
    from torchflows_b200.flows import shard_bounds
    for n in (0, 1, 7, 1024, 1031):
        for world in (1, 2, 3, 8):
            spans = [shard_bounds(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


_DP_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from torchflows_b200.flows import allreduce_gradients, shard_bounds, _allreduce_stats
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:' + sys.argv[2], rank=int(sys.argv[3]), world_size=2)
rank = dist.get_rank()
torch.manual_seed(0)
# a toy model whose loss is a mean over the global batch: DP gradient mean == single-process gradient
w = torch.nn.Parameter(torch.randn(5)); b = torch.nn.Parameter(torch.randn(1))
x = torch.randn(11, 5); y = torch.randn(11)
lo, hi = shard_bounds(11, rank, 2)
loss = ((x[lo:hi] @ w + b - y[lo:hi]) ** 2).sum() * (2 / 11)      # local sum * world / global count
loss.backward()
allreduce_gradients([w, b], 2)
w2 = torch.nn.Parameter(w.detach().clone()); b2 = torch.nn.Parameter(b.detach().clone())
((x @ w2 + b2 - y) ** 2).mean().backward()
assert torch.allclose(w.grad, w2.grad, atol=1e-6) and torch.allclose(b.grad, b2.grad, atol=1e-6)
# ActNorm statistics all-reduce: (sum, sumsq, n) of the shards add up to those of the whole batch
xs = x[lo:hi].double()
s, q, n = _allreduce_stats(xs.sum(0), (xs * xs).sum(0), torch.tensor(float(hi - lo), dtype=torch.float64))
assert torch.allclose(s, x.double().sum(0)) and torch.allclose(q, (x.double() ** 2).sum(0)) and float(n) == 11
# GradBuckets: gradients live in per-layer buckets, each bucket is all-reduced from a hook while backward is still running
from torchflows_b200.flows import GradBuckets
class Toy(torch.nn.Module):
    def __init__(self):
        super().__init__()
        torch.manual_seed(1)
        self.bijection = torch.nn.Module()
        self.bijection.layers = torch.nn.ModuleList([torch.nn.Linear(5, 7), torch.nn.Tanh(), torch.nn.Linear(7, 3)])
        self.extra = torch.nn.Parameter(torch.randn(3))
        self.frozen = torch.nn.Parameter(torch.randn(2), requires_grad=False)
    def forward(self, t):
        for layer in self.bijection.layers:
            t = layer(t)
        return t + self.extra
GradBuckets.MIN_BUCKET_BYTES = 0            # one bucket per layer even for these tiny layers
toy, ref = Toy(), Toy()
buckets = GradBuckets(toy, 2)
assert len(buckets.flats) == 3 and buckets.nbytes == 4 * sum(p.numel() for p in toy.parameters() if p.requires_grad)
for step in range(3):
    xs = torch.randn(10, 5, generator=torch.Generator().manual_seed(step))
    lo, hi = shard_bounds(10, rank, 2)
    buckets.begin_step()
    (toy(xs[lo:hi]) ** 2).sum().mul(2 / 10).backward()
    buckets.finish()
    for p in ref.parameters():
        p.grad = None
    (ref(xs) ** 2).sum().mul(1 / 10).backward()
    for (n, p), q in zip(toy.named_parameters(), ref.parameters()):
        if p.requires_grad:
            assert torch.allclose(p.grad, q.grad, atol=1e-6), (step, n)
            assert p.grad.data_ptr() == buckets.flats[buckets.bucket_of[id(p)]].data_ptr() + 4 * sum(
                r.numel() for r in buckets.params[buckets.bucket_of[id(p)]][:[id(r) for r in buckets.params[buckets.bucket_of[id(p)]]].index(id(p))])
buckets.close()
dist.destroy_process_group()
print('ok', rank)
'''


def test_data_parallel_helpers_gloo_world2(tmp_path):
    script = tmp_path / 'dp_worker.py'
    script.write_text(_DP_WORKER)
    port = str(29500 + os.getpid() % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, port, str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0 and 'ok' in o, o


def test_weight_snapshots_follow_in_place_updates():
    """BaseFlow._snapshot_weights (the keep-best-weights copy of fit, flows.py:246,429): the first call clones the
    state_dict, later calls refresh the same buffers from the live tensors; ActNorm's data-dependent initialisation is in
    place, so the live tensors stay the ones the snapshot remembers."""
    import torch
    from torchflows_b200 import Flow
    from torchflows_b200.architectures import RealNVP
    torch.manual_seed(0)
    flow = Flow(RealNVP(4))
    snap = flow._snapshot_weights()
    assert set(snap.keys()) == set(flow.state_dict().keys())
    storages = {k: v.data_ptr() for k, v in snap.items()}
    with torch.no_grad():
        for p in flow.parameters():
            p.add_(1.0)
    stale = {k: v.clone() for k, v in snap.items()}
    snap2 = flow._snapshot_weights(snap)
    assert snap2 is snap and all(v.data_ptr() == storages[k] for k, v in snap.items())
    for k, v in flow.state_dict().items():
        assert torch.equal(snap[k], v)
        if v.is_floating_point() and v.numel() and k.endswith(('weight', 'bias', 'value')):
            assert not torch.equal(stale[k], v)
    flow.load_state_dict(stale)
    for k, v in flow.state_dict().items():
        assert torch.equal(stale[k], v)


def test_composition_regularization_sums_layer_terms():
    """BijectiveComposition.regularization (bijections/base.py:234-243): l2_coef * sum of squared trainable parameters of
    the layers that ask for it, zero placeholders ignored."""
    import torch
    from torchflows_b200.architectures import RealNVP
    torch.manual_seed(0)
    bij = RealNVP(6)
    expected = 0.0
    n_reg = 0
    for layer in bij.layers:
        if getattr(layer, 'l2_regularization', False) and getattr(layer, 'l2_coef', 0.0) > 0:
            expected = expected + layer.l2_coef * sum(float((p.detach() ** 2).sum()) for p in layer.parameters() if p.requires_grad)
            n_reg += 1
    total = bij.regularization()
    assert isinstance(total, torch.Tensor) and total.dim() == 0
    assert abs(float(total.detach()) - float(expected)) <= 1e-6 * (1 + abs(float(expected)))
    if n_reg:
        total.backward()
        assert any(p.grad is not None and p.grad.abs().sum() > 0 for p in bij.parameters())


def test_philox_restatement_known_answer():
    """The numpy restatement of csrc/b2f_philox.cuh used by the GPU sampling tests reproduces the Random123 known-answer
    vector of philox4x32-10 (counter 0, key 0), so the GPU stream is pinned to the published generator."""
    import numpy as np
    from tests.test_gpu_sampling import philox4x32_10
    u = philox4x32_10(np.zeros(1, dtype=np.uint64), 0)
    assert [int(v[0]) for v in u] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]


def test_bench_dump_outputs_fixed_row_sample(tmp_path):
    """bench.py --dump-outputs: float32 .npy files within the size cap, the same seeded rows of every output in every
    run, and torch's global RNG (which keys Flow.sample's draws) untouched."""
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(1)
    rows, D = 2 * bench.DUMP_BYTES // (4 * 65), 64
    lp, xs = torch.arange(rows, dtype=torch.float64), torch.randn(rows, D, generator=g)      # log_prob holds the row index
    rng = torch.random.get_rng_state()
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'log_prob': lp, 'sample': xs})
    assert torch.equal(rng, torch.random.get_rng_state())
    a_lp, a_xs = np.load(tmp_path / 'a' / 'log_prob.npy'), np.load(tmp_path / 'a' / 'sample.npy')
    assert a_lp.dtype == a_xs.dtype == np.float32 and a_xs.shape[1] == D
    assert 0 < len(a_lp) == len(a_xs) < rows
    assert sum(f.stat().st_size for f in (tmp_path / 'a').iterdir()) <= bench.DUMP_BYTES + 1024
    assert np.array_equal(a_lp, np.load(tmp_path / 'b' / 'log_prob.npy'))
    assert np.array_equal(a_xs, np.load(tmp_path / 'b' / 'sample.npy'))
    kept = a_lp.astype(np.int64)
    assert np.all(np.diff(kept) > 0) and np.array_equal(xs.numpy()[kept], a_xs)
    small = tmp_path / 'small'
    bench.dump_outputs(str(small), {'log_prob': lp[:100], 'sample': xs[:100]})
    assert np.array_equal(np.load(small / 'sample.npy'), xs[:100].numpy())


def test_backward_tile_shape_query(monkeypatch):
    """b2f_flow_backward_shape: the tile shape (rows per tile TM, threads NT, per-warp spline-weight staging) the fused
    backward kernel launches, on the lowered programs of real presets.  Default-width presets climb a ladder of smaller
    shapes as the shared-memory footprint grows with D, until the forward budget sends the layers to the composite path;
    `precise` arithmetic turns the staging (tensor-core GEMM path) off; B2F_BWD_TM / B2F_BWD_NT force a shape when it is
    admissible and fits, and are ignored otherwise."""
    import torchflows_b200.architectures as arch
    from torchflows_b200 import _native as N, _program as P
    from torchflows_b200.bijections.finite.autoregressive.layers_base import _fits_fused_kernel
    for var in ('B2F_BWD_TM', 'B2F_BWD_NT', 'B2F_BWD_NO_MMA'):
        monkeypatch.delenv(var, raising=False)

    def program(preset, D, **kwargs):
        ops = getattr(arch, preset)(D, **kwargs).eval().fused_ops('forward')
        assert ops is not None, (preset, D)
        return P.op_dicts(ops)

    def staging(ops):        # per-warp stride of one element's output weights + bias, H = widest spline layer <= 31
        h = max([o['n_hidden'] for o in ops if o['kind'] in (N.OP_COUPLING, N.OP_MADE) and o['tkind'] == N.T_RQ_FWD
                 and o['n_hidden'] <= 31], default=0)
        return 24 * (h + 1) if h else 0

    ladder = [('CouplingRQNSF', 64, 32, 384, True), ('CouplingRQNSF', 320, 32, 384, True),
              ('CouplingRQNSF', 352, 32, 256, True), ('CouplingRQNSF', 448, 32, 256, True),
              ('CouplingRQNSF', 480, 32, 128, True), ('CouplingRQNSF', 592, 32, 128, True),
              ('CouplingRQNSF', 608, 32, 128, False),
              ('RealNVP', 288, 64, 256, False), ('RealNVP', 304, 32, 256, False), ('RealNVP', 608, 32, 128, False),
              ('MAF', 304, 64, 256, False), ('MAF', 320, 32, 256, False), ('MAF', 640, 32, 128, False),
              ('MaskedAutoregressiveRQNSF', 480, 32, 384, True), ('MaskedAutoregressiveRQNSF', 496, 32, 256, True),
              ('MaskedAutoregressiveRQNSF', 576, 32, 128, True),
              ('CouplingLRS', 16, 64, 256, False), ('CouplingLRS', 272, 32, 256, False),
              ('CouplingLRS', 560, 32, 128, False),
              ('IAF', 320, 32, 256, False), ('InverseAutoregressiveRQNSF', 128, 64, 256, False)]
    for preset, D, TM, NT, staged in ladder:
        ops = program(preset, D)
        want = (TM, NT, staging(ops) if staged else 0)
        assert (not staged) or want[2] > 0, (preset, D)
        assert N.flow_backward_shape(ops, D) == want, (preset, D, N.flow_backward_shape(ops, D), want)
    # 608 still trains fused (on the scalar spline path); at 640 the forward budget sends the layers to the composite
    assert _fits_fused_kernel(608, 19, N.OP_COUPLING, N.T_RQ_FWD, 8)
    assert not _fits_fused_kernel(640, 19, N.OP_COUPLING, N.T_RQ_FWD, 8)
    assert arch.CouplingRQNSF(640).eval().fused_ops('forward') is None

    q256 = program('CouplingRQNSF', 256)
    assert N.flow_backward_shape(q256, 256) == (32, 384, 24 * 18)
    assert N.flow_backward_shape(q256, 256, N.FLOW_MODE_PRECISE) == (64, 256, 0)
    wide_h = program('CouplingRQNSF', 64, conditioner_kwargs={'n_hidden': 32})
    assert N.flow_backward_shape(wide_h, 64) == (64, 256, 0)
    monkeypatch.setenv('B2F_BWD_NO_MMA', '1')
    assert N.flow_backward_shape(q256, 256) == (64, 256, 0)
    monkeypatch.delenv('B2F_BWD_NO_MMA')

    spline, affine = program('CouplingRQNSF', 64), program('MAF', 64)
    defaults = {id(spline): (32, 384, staging(spline)), id(affine): (64, 256, 0)}
    for ops in (spline, affine):
        assert N.flow_backward_shape(ops, 64) == defaults[id(ops)]
        for TM, NT in ((32, 32), (32, 160), (64, 64), (64, 192), (64, 384)):
            monkeypatch.setenv('B2F_BWD_TM', str(TM))
            monkeypatch.setenv('B2F_BWD_NT', str(NT))
            assert N.flow_backward_shape(ops, 64) == (TM, NT, defaults[id(ops)][2]), (TM, NT)
        for TM, NT in ((64, 32), (48, 256), (32, 416), (64, 416)):        # NT < TM, TM not a power of two, NT > 384
            monkeypatch.setenv('B2F_BWD_TM', str(TM))
            monkeypatch.setenv('B2F_BWD_NT', str(NT))
            assert N.flow_backward_shape(ops, 64) == defaults[id(ops)], (TM, NT)
    # admissible but too large for the program: 64 x 384 with staging does not fit beside CouplingRQNSF(256)'s tiles
    monkeypatch.setenv('B2F_BWD_TM', '64')
    monkeypatch.setenv('B2F_BWD_NT', '384')
    assert N.flow_backward_shape(q256, 256) == (32, 384, 24 * 18)
    monkeypatch.delenv('B2F_BWD_TM')
    monkeypatch.delenv('B2F_BWD_NT')

    # b2f_flow_backward_fits answers for one layer what the query answers at flags = 0
    for kind, tkind in ((N.OP_COUPLING, N.T_RQ_FWD), (N.OP_COUPLING, N.T_AFFINE_FWD), (N.OP_MADE, N.T_RQ_FWD),
                        (N.OP_MADE_SEQ, N.T_AFFINE_INV), (N.OP_COUPLING, N.T_LRS_FWD)):
        for H in (4, 19, 31, 32, 64, 1024):
            for D in (16, 256, 608, 640, 768, 1024, 2048, 4096):
                n_bins = 8 if tkind in (N.T_RQ_FWD, N.T_LRS_FWD) else 0
                op = [dict(kind=kind, tkind=tkind, n_hidden=H, n_bins=n_bins)]
                fits = N.flow_backward_fits(kind, tkind, H, n_bins, D)
                assert fits == (N.flow_backward_shape(op, D) is not None), (kind, tkind, H, D)
    assert N.flow_backward_shape([dict(kind=N.OP_COUPLING, tkind=N.T_RQ_FWD, n_hidden=1024, n_bins=8)], 4096) is None
