"""CPU-only tests: the C-ABI library loads and exports what the header declares, the Python mirror
matches the reference's module surface, the product path has no CPU fallback, and the multi-process
sharding logic works over gloo."""
import ctypes

import os
import re
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT, load_golden


def test_library_exports_every_declared_symbol():
    from pvraft_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'pvraft_b200.h')).read()
    declared = set(re.findall(r'PVRAFT_API\s+[\w\s\*]+?\b(pvraft_\w+)\s*\(', hdr))
    assert len(declared) >= 15
    handle = ctypes.CDLL(_lib.LIB_PATH) if os.path.exists(_lib.LIB_PATH) else _lib.lib()
    for name in declared:
        assert hasattr(handle, name), f'{name} is declared in the header but not exported'
    assert declared == set(_lib.EXPORTS), 'ctypes binding and header disagree'
    lib = _lib.lib()
    assert lib.pvraft_version() == 100
    for which, struct in enumerate([_lib.LinearArgs, _lib.CorrFeatArgs, _lib.GruArgs, _lib.FlowOutArgs, _lib.TcLinearArgs,
                                    _lib.KnnBranchArgs]):
        assert lib.pvraft_sizeof(which) == ctypes.sizeof(struct), f'struct {struct.__name__} layout drifted'


def test_argument_errors_are_reported_without_a_gpu():
    from pvraft_b200 import _lib
    lib = _lib.lib()
    rc = lib.pvraft_corr_lookup_fwd(None, None, None, None, 1, 64, 64, 3, 0.25, None, 0, None, None, None, None, None)
    assert rc == -1 and b'null' in lib.pvraft_last_error_string()
    rc = lib.pvraft_corr_lookup_fwd(16, 16, 16, 16, 1, 64, 96, 3, 0.25, 16, 0, 16, None, None, None, None)
    assert rc == -2 and b'truncate_k=96' in lib.pvraft_last_error_string()
    rc = lib.pvraft_knn_fwd(8, 8, 1, 16, 16, 33, 0, 8, None, None, None)
    assert rc == -2
    with pytest.raises(_lib.PvraftError):
        _lib.check(rc, 'knn')


def test_module_surface_matches_reference_state_dict():
    from pvraft_b200 import RSF, RSF_refine
    arr, W = load_golden('small_rsf_refine.npz')
    args = types.SimpleNamespace(corr_levels=3, base_scales=0.25, truncate_k=64)
    m = RSF_refine(args)
    sd = m.state_dict()
    assert list(sd.keys()) == list(W.keys())            # same keys, same order as the reference
    for k in W:
        assert tuple(sd[k].shape) == tuple(W[k].shape), k
    m.load_state_dict(W, strict=True)
    rsf = RSF(args)
    missing = rsf.load_state_dict(W, strict=False)       # tools/engine_refine.py:110 style
    assert not missing.missing_keys and all(k.startswith('refine_block.') for k in missing.unexpected_keys)
    for attr in ('feature_extractor', 'context_extractor', 'corr_block', 'update_block', 'refine_block'):
        assert hasattr(m, attr)
    assert len(sd) == 124 and sum(p.numel() for p in rsf.parameters()) == 192034


def test_reference_import_paths():
    from model.RAFTSceneFlow import RSF
    from model.RAFTSceneFlowRefine import RSF_refine
    from model.corr import CorrBlock
    from model.update import UpdateBlock
    from model.pointconv import knn_point
    from model.flot.gconv import SetConv
    from model.flot.graph import Graph
    import pvraft_b200
    assert RSF is pvraft_b200.RSF and RSF_refine is pvraft_b200.RSF_refine
    assert CorrBlock is pvraft_b200.CorrBlock and UpdateBlock is pvraft_b200.UpdateBlock
    assert callable(knn_point) and SetConv is pvraft_b200.SetConv and Graph is pvraft_b200.Graph


def test_no_cpu_fallback():
    from oracle import pvraft_oracle as O
    from pvraft_b200 import RSF, _lib
    args = types.SimpleNamespace(corr_levels=3, base_scales=0.25, truncate_k=32)
    m = RSF(args).eval()
    pc, pc2 = O.synthetic_clouds(1, 64)
    with torch.no_grad(), pytest.raises(_lib.PvraftError):
        m([pc, pc2], 1)
    with pytest.raises(_lib.PvraftError):                # the training path has no CPU fallback either
        m([pc, pc2], 1)


def test_product_never_imports_the_oracle():
    pat = re.compile(r'^\s*(from|import)\s+oracle|import_module\(.oracle|oracle/', re.M)
    for top in ('pvraft_b200', 'model'):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith('.py'):
                    assert not pat.search(open(os.path.join(dirpath, f)).read()), f'{f} reaches into oracle/'


def test_shard_range_covers_batch():
    from pvraft_b200.dist import shard_range
    for total in (1, 2, 7, 8, 16, 17):
        for world in (1, 2, 3, 8):
            spans = [shard_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [e - b for b, e in spans]
            assert max(sizes) - min(sizes) <= 1


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from pvraft_b200 import dist as D
    r, w, _ = D.init_from_env(backend='gloo')
    g = torch.Generator().manual_seed(0)
    xyz1 = torch.rand(5, 16, 3, generator=g)
    xyz2 = torch.rand(5, 16, 3, generator=g)
    mine = D.shard_batch([xyz1, xyz2], r, w)
    local = mine[0] * 2.0 + mine[1]                    # stands in for the per-sample forward
    full = D.gather_batch(local)
    ok = torch.equal(full, xyz1 * 2.0 + xyz2)
    t = D.max_over_ranks(1.0 + r)
    s = D.sum_over_ranks(float(mine[0].shape[0]))
    D.barrier()
    out[rank] = (ok, t, s)
    dist.destroy_process_group()


def test_two_rank_gloo_shard_gather_and_timing():
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    for r in range(world):
        ok, t, s = out[r]
        assert ok and t == 2.0 and s == 5.0


def _grad_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    from pvraft_b200 import dist as D
    r, w, _ = D.init_from_env(backend='gloo')
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.GroupNorm(1, 5), torch.nn.Linear(5, 3))   # per-sample norm, as the model
    x = torch.randn(8, 6, generator=torch.Generator().manual_seed(1))
    y = torch.randn(8, 3, generator=torch.Generator().manual_seed(2))
    lo, hi = D.shard_range(8, r, w)
    (net(x[lo:hi]) - y[lo:hi]).abs().mean().backward()          # masked-mean loss of the rank's shard (tools/loss.py:34-38)
    nbytes = D.allreduce_gradients(net.parameters())
    got = [p.grad.clone() for p in net.parameters()]
    net.zero_grad()
    (net(x) - y).abs().mean().backward()                        # the same step on the concatenated batch
    want = [p.grad for p in net.parameters()]
    out[rank] = (all(torch.allclose(a, b, rtol=1e-5, atol=1e-7) for a, b in zip(got, want)), nbytes)
    wrapped = D.ddp(net)                                        # the DDP wrapper gives the same averaged gradients
    wrapped.zero_grad()
    (wrapped(x[lo:hi]) - y[lo:hi]).abs().mean().backward()
    out[rank] = out[rank] + (all(torch.allclose(p.grad, b, rtol=1e-5, atol=1e-7) for p, b in zip(net.parameters(), want)),)
    dist.destroy_process_group()


def test_two_rank_gloo_gradient_allreduce_equals_the_full_batch():
    """SURVEY 8c item 5 (host-side logic on CPU): per-rank shard gradients, one all-reduce (sum -> mean), == the gradient of
    the concatenated batch, because every normalisation is per sample and the loss is a mean over equal shards."""
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_grad_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    for r in range(world):
        ok, nbytes, ok_ddp = out[r]
        assert ok and ok_ddp and nbytes == 4 * (6 * 5 + 5 + 5 + 5 + 5 * 3 + 3)


def test_division_by_constant_sequence_is_exact():
    """k_corr_gemm divides by sqrt(C) with q0 = x*r, q = q0 + (x - q0*s)*r, r = RN(1/s) (csrc/corr_gemm.cu: div_by_const).
    Emulated here in numpy (an fp32 FMA = the double-precision product-sum rounded once to fp32): bit-identical to the true
    fp32 division for every sampled x and every channel count the model can use."""
    rng = np.random.default_rng(0)

    def fma32(a, b, c):
        return (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(np.float32)

    for channels in (3, 32, 64, 96, 100, 128, 160, 256):
        s = np.float32(np.sqrt(np.float32(channels)))
        r = np.float32(1.0 / np.float64(s))
        x = np.concatenate([rng.standard_normal(200_000).astype(np.float32) * np.float32(v) for v in (1e-3, 1.0, 50.0, 1e4)])
        q0 = (x * r).astype(np.float32)
        q = fma32(fma32(-q0, np.full_like(x, s), x), np.full_like(x, r), q0)
        assert np.array_equal(q, (x / s).astype(np.float32)), channels


def test_derived_cache_follows_parameter_versions():
    from pvraft_b200 import ops
    w = torch.nn.Parameter(torch.ones(4))
    calls = []

    def make(t):
        calls.append(1)
        return float(t.detach().sum())

    assert ops.derived((w,), 'sum', make) == 4.0 and ops.derived((w,), 'sum', make) == 4.0 and len(calls) == 1
    with torch.no_grad():
        w.mul_(2.0)                                     # in-place update bumps the version -> re-derived
    assert ops.derived((w,), 'sum', make) == 8.0 and len(calls) == 2
    w.data = torch.full((4,), 3.0)                      # storage swap (e.g. module.to(device)) -> re-derived
    assert ops.derived((w,), 'sum', make) == 12.0 and len(calls) == 3


def test_morton_order_is_a_spatially_coherent_permutation():
    from pvraft_b200 import ops
    g = torch.Generator().manual_seed(0)
    pts = torch.rand(2, 4096, 3, generator=g) * torch.tensor([20.0, 10.0, 2.0])
    perm = ops.morton_order(pts)
    assert perm.shape == (2, 4096) and torch.equal(perm.sort(1).values, torch.arange(4096).expand(2, -1))
    ordered = torch.gather(pts, 1, perm.unsqueeze(-1).expand(-1, -1, 3))
    step_sorted = (ordered[:, 1:] - ordered[:, :-1]).norm(dim=-1).mean()
    step_input = (pts[:, 1:] - pts[:, :-1]).norm(dim=-1).mean()
    assert step_sorted < 0.25 * step_input          # consecutive rows are spatial neighbours


def test_weight_folds_equal_the_unfused_layers():
    """The two algebraic folds of the RAFT loop, against the unfused layer sequences in float64."""
    from pvraft_b200.corr import fold_corr_motion
    from pvraft_b200.update import fold_flow_head
    g = torch.Generator().manual_seed(0)
    r = lambda *s: torch.randn(*s, generator=g)
    # flow head: out_conv.0(cat([s, conv1(x)]))
    w_o0, b_o0, w_c1, b_c1 = r(64, 128, 1), r(64), r(64, 64, 1), r(64)
    s_, x = r(5, 64).double(), r(5, 64).double()
    want = torch.cat([s_, x @ w_c1[..., 0].double().T + b_c1.double()], 1) @ w_o0[..., 0].double().T + b_o0.double()
    w, b = fold_flow_head(w_o0, w_c1, b_c1, b_o0)
    got = torch.cat([s_, x], 1) @ w.double().T + b.double()
    assert float((got - want).abs().max() / want.abs().max()) < 1e-6
    # feature head + conv_corr: conv_corr(out_conv.3(a) + knn_out(k))
    w_cc, b_cc, w_out, b_out, w_kout, b_kout = r(64, 64, 1), r(64), r(64, 128, 1), r(64), r(64, 64, 1), r(64)
    a, k = r(5, 128).double(), r(5, 64).double()
    corr = a @ w_out[..., 0].double().T + b_out.double() + k @ w_kout[..., 0].double().T + b_kout.double()
    want = corr @ w_cc[..., 0].double().T + b_cc.double()
    w, b = fold_corr_motion(w_cc, b_cc, w_out, b_out, w_kout, b_kout)
    got = torch.cat([a, k], 1) @ w.double().T + b.double()
    assert float((got - want).abs().max() / want.abs().max()) < 1e-6


def test_batch_collate_matches_the_reference_class():
    """pvraft_b200.data.Batch against what the reference's class (datasets/generic.py:6-66) returned for the same three items
    (tests/golden/batch_collate.npz, made by tests/golden/make_golden.py)."""
    from pvraft_b200.data import Batch, subsample
    arr, _ = load_golden('batch_collate.npz')
    items = [{key: [arr[f'item{i}/{key}{ind}'] for ind in range(2)] for key in ('sequence', 'ground_truth')} for i in range(3)]
    mine = Batch(items)
    ref = {key: [arr[f'batch/{key}{ind}'] for ind in range(2)] for key in ('sequence', 'ground_truth')}
    for key in ('sequence', 'ground_truth'):
        for a, b in zip(mine[key], ref[key]):
            assert a.shape == b.shape and torch.equal(a, b)
    moved = mine.to('cpu')
    assert moved is mine and torch.equal(mine['sequence'][1], ref['sequence'][1])
    assert mine['sequence'][0].untyped_storage().data_ptr() == mine['ground_truth'][1].untyped_storage().data_ptr()   # one buffer
    pts = torch.arange(300.).view(100, 3)
    sub, lab = subsample(pts, 40, generator=torch.Generator().manual_seed(1), extra=(torch.arange(100),))
    assert sub.shape == (40, 3) and torch.equal(sub, pts[lab]) and len(set(lab.tolist())) == 40
