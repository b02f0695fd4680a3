"""Parity of the code path that bench.py TIMES (VERDICT r1, weak #1-#3): the RAFT loop at the BASELINE size
(N = 8192, K = 512) against the CPU oracle -- teacher-forced per iteration and free-running --, a B = 8 batch against
its own samples run one by one (dynamic work claims, 2B-batched encoder), 32 free-running iterations, and the
model-level fallback kernels that run when N is not a multiple of 128.

Tolerances (written here, measured values are printed with `-s`):
  teacher-forced corr / motion / net      <= 1e-5  (max-abs / max-abs; 2e-5 where the input is the kernel's own corr)
  teacher-forced delta_flow               <= 5e-5
  free-running flows, 8 iterations        mean-abs <= 1e-4 * mean|flow| on the oracle's adjacency (measured 6e-6; the reference's
                                          own fp32-vs-fp64 drift is 1.1e-3), <= 1e-2 with the own tie-broken adjacency (1e-3)
  free-running flows, 32 iterations       mean-abs <= 5e-4 * mean|flow| on the oracle's adjacency (measured 6.5e-5; reference
                                          fp32-vs-fp64: 1.7e-3 at |flow| ~ 3.4), <= 2e-2 with the own adjacency (1.7e-3)
  batch-of-8 vs one-by-one                mean-abs <= 2e-4 * mean|flow|   (same kernels; only the order of double-precision
                                                                          GroupNorm partial sums may differ)
"""
import contextlib
import types

import pytest
import torch

from conftest import default_weights, rel_err
from oracle import pvraft_oracle as O

pytestmark = pytest.mark.gpu
N, K, LEVELS, SCALE = 8192, 512, 3, 0.25


@pytest.fixture(scope='module')
def dev():
    return torch.device('cuda:0')


@pytest.fixture(scope='module', autouse=True)
def _cpu_threads():
    old = torch.get_num_threads()
    torch.set_num_threads(min(16, old))      # torch CPU ops collapse at 100+ threads on these op sizes
    yield
    torch.set_num_threads(old)


def make_model(dev, k=K, refine=False, weights=None):
    from pvraft_b200 import RSF, RSF_refine
    args = types.SimpleNamespace(corr_levels=LEVELS, base_scales=SCALE, truncate_k=k)
    W = weights if weights is not None else default_weights(refine=refine, args=args)
    m = (RSF_refine if refine else RSF)(args)
    m.load_state_dict(W, strict=True)
    return m.to(dev).eval(), W


def product_graph(og, b, n, dev):
    from pvraft_b200 import Graph
    k = og.k_neighbors
    nbr = (og.edges.reshape(b, n, k) - (torch.arange(b) * n).view(b, 1, 1)).to(torch.int32)
    return Graph(nbr.to(dev), og.edge_feats.reshape(b, n, k, 3).to(dev).contiguous(), k, [b * n, b * n])


@contextlib.contextmanager
def oracle_adjacency():
    """Run the product on the ORACLE's kNN adjacency.  The reference ranks neighbours by a cancellation-prone fp32 distance
    (model/flot/graph.py:53-60); where two candidates tie exactly at the 32nd place either neighbour set is valid (SURVEY H1)
    and torch.argsort's pick is unspecified.  At N=8192 a handful of rows per cloud tie, and three SetConv layers spread
    such a row's different max-pool over 32^3 > N points (measured: ~1e-3 on the correlation values), so value-level
    parity of everything downstream is checked on a common adjacency; the adjacency itself is checked separately
    (different rows must be exact ties)."""
    from pvraft_b200 import graph as G

    def from_oracle(pcloud, k):
        b, n, _ = pcloud.shape
        return product_graph(O.construct_graph(pcloud.detach().cpu(), k), b, n, pcloud.device)

    orig = G.Graph.__dict__['construct_graph']
    G.Graph.construct_graph = staticmethod(from_oracle)
    try:
        yield
    finally:
        G.Graph.construct_graph = orig


def pm(x):   # [B,C,N] -> point-major [B,N,C]
    return x.transpose(1, 2).contiguous()


@pytest.fixture(scope='module')
def config2(dev):
    """BASELINE config 2 (N=8192, iters=8, batch=2, fp32): one oracle run shared by the tests below."""
    b, iters = 2, 8
    m, W = make_model(dev)
    pc1, pc2 = O.synthetic_clouds(b, N, seed=1234)
    with torch.no_grad():
        li = O.prepare(W, pc1, pc2, K)
        trace = []
        flows = O.raft_loop(W, li, pc1, iters, LEVELS, SCALE, trace)
    return dict(b=b, iters=iters, m=m, W=W, pc1=pc1, pc2=pc2, li=li, trace=trace, flows=flows)


def test_config2_teacher_forced_loop_path(dev, config2):
    """The loop's own kernels (feature_motion_tc, UpdateBlock.forward_pm: lookup with per-sample dynamic claims, tcgen05
    layers, SetConv edge kernel) on oracle-produced state, iteration by iteration."""
    c = config2
    m, b = c['m'], c['b']
    li = c['li']
    m.corr_block.set_state(li.state.truncated_corr.to(dev), li.state.indices.to(dev), c['pc2'].to(dev))
    g = product_graph(li.graph, b, N, dev)
    pc1 = c['pc1'].to(dev)
    inp = pm(li.inp).to(dev)
    net = pm(li.net).to(dev)
    me = m.update_block.motion_encoder
    worst = dict(corr=0.0, motion=0.0, net=0.0, delta=0.0)
    with torch.no_grad():
        for it, t in enumerate(c['trace']):
            coords = t['coords'].to(dev).contiguous()
            flow = (coords - pc1).contiguous()
            corr_pm, motion = m.corr_block.feature_motion_tc(coords, flow, me, need_corr=True)
            e = rel_err(corr_pm.transpose(1, 2).cpu(), t['corr'])
            worst['corr'] = max(worst['corr'], e)
            assert e < 1e-5, (it, 'corr', e)
            want_motion = O.motion_encoder(c['W'], (t['coords'] - c['pc1']), t['corr'], 'update_block.motion_encoder')
            e = rel_err(motion.transpose(1, 2).cpu(), want_motion)
            worst['motion'] = max(worst['motion'], e)
            assert e < 2e-5, (it, 'motion', e)
            _, motion_f = m.corr_block.feature_motion_tc(coords, flow, me, need_corr=False)     # what the loop runs
            assert rel_err(motion_f.cpu(), motion.cpu()) < 2e-5
            net_new, delta = m.update_block.forward_pm(net, inp, motion_f, g)
            e = rel_err(net_new.transpose(1, 2).cpu(), t['net'])
            worst['net'] = max(worst['net'], e)
            assert e < 2e-5, (it, 'net', e)
            e = rel_err(delta.cpu(), t['delta'])
            worst['delta'] = max(worst['delta'], e)
            assert e < 5e-5, (it, 'delta', e)
            net = pm(t['net']).to(dev)                     # teacher forcing: the oracle's hidden state goes on
    print('config2 teacher-forced worst rel err:', worst)


def test_config2_build_matches_oracle_state(dev, config2):
    """Pre-loop path at N=8192: encoders (2B-batched), tcgen05 correlation GEMM, top-512 -- candidate SETS equal to the
    oracle's except at near-ties of the 512th value (3xTF32 vs fp32 summation order), values and context features 1e-5;
    the kNN adjacency differs from the oracle's argsort only where the 32nd distance ties exactly."""
    c = config2
    m, b, li = c['m'], c['b'], c['li']
    with torch.no_grad():
        _, _, _, graph_own, _, _ = m._encode([c['pc1'].to(dev), c['pc2'].to(dev)])
        with oracle_adjacency():
            xyz1, xyz2, graph, graph_ctx, net, inp = m._encode([c['pc1'].to(dev), c['pc2'].to(dev)])
    got = m.corr_block.corr_idx.long().cpu().sort(-1).values
    want = li.state.indices.sort(-1).values
    rows_differ = (got != want).any(-1).float().mean().item()
    assert rel_err(m.corr_block.truncated_corr.cpu(), li.state.truncated_corr) < 1e-5
    assert rows_differ < 0.02, rows_differ
    # three chained SetConv layers (9 GroupNorms) behind these: measured 1.7e-5
    assert rel_err(net.transpose(1, 2).cpu(), li.net) < 3e-5 and rel_err(inp.transpose(1, 2).cpu(), li.inp) < 3e-5
    nb = graph_own.nbr.long().cpu().sort(-1).values
    ref = (li.graph.edges.reshape(b, N, 32) - (torch.arange(b) * N).view(b, 1, 1)).sort(-1).values
    bad = (nb != ref).any(-1)
    d = O.pairwise_sqdist_expanded(c['pc1'])
    assert torch.equal(torch.gather(d, 2, nb).max(-1).values[bad], torch.gather(d, 2, ref).max(-1).values[bad])
    assert bad.float().mean() < 0.01
    print(f'config2 build: rows with a different candidate set {rows_differ:.2e}; adjacency rows with a tie-broken neighbour '
          f'{int(bad.sum())} of {bad.numel()}')


def _free_running(m, pc1, pc2, iters, dev):
    with torch.no_grad():
        own = m([pc1.to(dev), pc2.to(dev)], iters)            # as shipped (CUDA-graph replay for batches <= 2)
        auto, m.use_cuda_graph = m.use_cuda_graph, False      # the oracle's adjacency is computed on the host: not capturable
        try:
            with oracle_adjacency():
                common = m([pc1.to(dev), pc2.to(dev)], iters)
        finally:
            m.use_cuda_graph = auto
    return own, common


def test_config2_free_running(dev, config2):
    c = config2
    own, common = _free_running(c['m'], c['pc1'], c['pc2'], c['iters'], dev)
    assert len(own) == c['iters']
    rel_common = [float((g.cpu() - r).abs().mean() / r.abs().mean()) for g, r in zip(common, c['flows'])]
    rel_own = [float((g.cpu() - r).abs().mean() / r.abs().mean()) for g, r in zip(own, c['flows'])]
    print('config2 free-running mean-abs / mean|flow| per iteration, common adjacency:', [f'{r:.1e}' for r in rel_common])
    print('                                                     own (tie-broken) adjacency:', [f'{r:.1e}' for r in rel_own])
    assert max(rel_common) < 1e-4, rel_common    # measured 6e-6; the 2e-3 of SURVEY 8c is the reference's own fp32-vs-fp64 drift
    assert max(rel_own) < 1e-2, rel_own          # includes the reference's own tie ambiguity (see oracle_adjacency)


def test_batch8_equals_one_by_one(dev):
    """The bench batch (8 samples per launch: per-sample dynamic 4-point claims across 18/19 CTAs, a 16-sample encoder
    batch) gives every sample the flow it gets alone."""
    m, _ = make_model(dev)
    b, iters = 8, 8
    pc1, pc2 = [t.to(dev) for t in O.synthetic_clouds(b, N, seed=77)]
    with torch.no_grad():
        together = m([pc1, pc2], iters)[-1]
        alone = torch.cat([m([pc1[i:i + 1].contiguous(), pc2[i:i + 1].contiguous()], iters)[-1] for i in range(b)], 0)
    scale = float(together.abs().mean())
    per_sample = (together - alone).abs().mean((1, 2)) / scale
    print('batch-8 vs one-by-one, mean-abs / mean|flow| per sample:', [f'{float(v):.1e}' for v in per_sample],
          'max abs', float((together - alone).abs().max()))
    assert float(per_sample.max()) < 2e-4


def test_free_running_32_iterations(dev):
    """BASELINE's metric runs 32 iterations: one sample, N=8192, K=512, against the oracle."""
    m, W = make_model(dev)
    pc1, pc2 = O.synthetic_clouds(1, N, seed=4321)
    with torch.no_grad():
        want = O.rsf_forward(W, pc1, pc2, 32, LEVELS, SCALE, K)
    own, common = _free_running(m, pc1, pc2, 32, dev)
    rels = [float((g.cpu() - w).abs().mean() / w.abs().mean()) for g, w in zip(common, want)]
    rels_own = [float((g.cpu() - w).abs().mean() / w.abs().mean()) for g, w in zip(own, want)]
    print('32-iteration free-running mean-abs / mean|flow| at iterations 1, 8, 16, 32 (common adjacency):',
          [f'{rels[i]:.1e}' for i in (0, 7, 15, 31)], ' own adjacency:', [f'{rels_own[i]:.1e}' for i in (0, 7, 15, 31)],
          ' mean|flow| at 32:', float(want[-1].abs().mean()))
    assert max(rels[:8]) < 1e-4 and max(rels) < 5e-4, rels      # measured 6e-6 / 6.5e-5
    assert max(rels_own) < 2e-2, rels_own


def _ragged_cases():
    cases = []
    for n, k in ((300, 128), (1000, 256)):
        cases.append(pytest.param(n, k, None, id=f'{n}-{k}'))
        cases += [pytest.param(n, k, s, id=f'{n}-{k}-randomised{s}') for s in (-0.5, 1.7)]
    return cases


def _model_vs_oracle(m, W, pc1, pc2, k, iters, dev):
    """Free-running flows against the oracle, then teacher forcing through the reference-layout module seams
    (CorrBlock.__call__, UpdateBlock.forward) on the oracle's state, graph and hidden states, then the correlation build."""
    b, n, _ = pc1.shape
    m.reset_graphs()
    li = O.prepare(W, pc1, pc2, k)
    trace = []
    want = O.raft_loop(W, li, pc1, iters, LEVELS, SCALE, trace)
    got = m([pc1.to(dev), pc2.to(dev)], iters)
    worst = dict(flow=0.0, corr=0.0, net=0.0, delta=0.0)
    for g, w in zip(got, want):
        e = float((g.cpu() - w).abs().mean()) / float(w.abs().mean())
        worst['flow'] = max(worst['flow'], e)
        assert e < 2e-3
    m.corr_block.set_state(li.state.truncated_corr.to(dev), li.state.indices.to(dev), pc2.to(dev))
    g = product_graph(li.graph, b, n, dev)
    net = li.net.to(dev)
    for t in trace:
        coords = t['coords'].to(dev).contiguous()
        corr = m.corr_block(coords)
        worst['corr'] = max(worst['corr'], rel_err(corr.cpu(), t['corr']))
        assert rel_err(corr.cpu(), t['corr']) < 1e-5
        net2, delta = m.update_block(net, li.inp.to(dev), t['corr'].to(dev), (t['coords'] - pc1).to(dev), g)
        worst['net'] = max(worst['net'], rel_err(net2.cpu(), t['net']))
        worst['delta'] = max(worst['delta'], rel_err(delta.cpu(), t['delta']))
        assert rel_err(net2.cpu(), t['net']) < 1e-5
        assert rel_err(delta.cpu(), t['delta']) < 5e-5
        net = t['net'].to(dev)
    # the correlation build (at a ragged N: tcgen05 GEMM on zero-padded feature maps, no library GEMM)
    m._encode([pc1.to(dev), pc2.to(dev)])
    assert rel_err(m.corr_block.truncated_corr.cpu(), li.state.truncated_corr) < 1e-5
    return worst


@pytest.mark.parametrize('n,k,slope', _ragged_cases())
def test_ragged_point_count_model_level(dev, n, k, slope):
    """N % 128 != 0 (`--max_points` is a free flag, train.py:8-71): the CUDA-core kernels (k_corrfeat + motion stage,
    k_gru, k_flowout, k_linear) carry the loop and the padded tcgen05 GEMM builds the correlation; teacher-forced
    module seams and free-running flows against the oracle.  `slope`: every GroupNorm (scale, shift) redrawn, some scales
    negative, and both single-slope PReLUs set to it (O.randomised_affine); None = the default init."""
    b, iters = 2, 3
    args = types.SimpleNamespace(corr_levels=LEVELS, base_scales=SCALE, truncate_k=k)
    W = default_weights(args=args, seed=5)
    if slope is not None:
        W = O.randomised_affine(W, seed=n, slope=slope)
    m, W = make_model(dev, k=k, weights=W)
    pc1, pc2 = O.synthetic_clouds(b, n, seed=n)
    pc1, pc2 = pc1 * 0.3, pc2 * 0.3                  # denser cloud: non-empty voxel cells at this small N
    with torch.no_grad():
        worst = _model_vs_oracle(m, W, pc1, pc2, k, iters, dev)
    print(f'ragged N={n} slope={slope}: worst', {key: f'{v:.1e}' for key, v in worst.items()})


def test_tensor_core_and_cuda_core_paths_match_oracle(dev, monkeypatch):
    """The same N = 1024 model with randomised GroupNorm / PReLU parameters, once as shipped (every per-point layer on tcgen05)
    and once with ops.tc_supported answering False, which routes every layer to the CUDA-core kernels that otherwise only
    run at a ragged N.  Both against the oracle: free-running, and teacher-forced at the module seams."""
    from pvraft_b200 import ops
    b, n, k, iters = 2, 1024, 256, 3
    args = types.SimpleNamespace(corr_levels=LEVELS, base_scales=SCALE, truncate_k=k)
    W = O.randomised_affine(default_weights(args=args, seed=5), seed=n, slope=-0.5)
    m, W = make_model(dev, k=k, weights=W)
    pc1, pc2 = O.synthetic_clouds(b, n, seed=n)
    pc1, pc2 = pc1 * 0.5, pc2 * 0.5
    with torch.no_grad():
        worst = {'tcgen05': _model_vs_oracle(m, W, pc1, pc2, k, iters, dev)}
        monkeypatch.setattr(ops, 'tc_supported', lambda *a, **kw: False)
        worst['cuda-core'] = _model_vs_oracle(m, W, pc1, pc2, k, iters, dev)
    for path, w in worst.items():
        print(f'N=1024 {path} path: worst', {key: f'{v:.1e}' for key, v in w.items()})


def test_cuda_graph_recaptured_after_weight_update(dev):
    """ADVICE r1: replays must not keep using derived weight copies (tf32 splits, folded products) of old parameter values."""
    from pvraft_b200 import RSF
    args = types.SimpleNamespace(corr_levels=3, base_scales=0.25, truncate_k=128)
    torch.manual_seed(0)
    m = RSF(args).to(dev).eval()
    pc1, pc2 = [t.to(dev) for t in O.synthetic_clouds(1, 1024, seed=5)]
    with torch.no_grad():
        m.use_cuda_graph = True
        before = m([pc1, pc2], 2)[-1].clone()
        m.update_block.flow_head.out_conv[0].weight.mul_(1.5)       # in-place update (an optimizer step / load_state_dict)
        m.corr_block.out_conv[2].weight.fill_(0.1)                  # PReLU slope: a host-side derived constant
        graphed = m([pc1, pc2], 2)[-1].clone()
        m.use_cuda_graph = False
        eager = m([pc1, pc2], 2)[-1]
    assert rel_err(graphed.cpu(), eager.cpu()) < 1e-6
    assert rel_err(before.cpu(), eager.cpu()) > 1e-3


def test_chained_tensor_core_launches_equal_grid_wide_waits(dev):
    """Opt-in (PVRAFT_TC_CHAIN=1): inside the loop six of the nine tensor-core launches start per SAMPLE on the completion
    counters of the launch before them instead of waiting for its whole grid (ops.tc_linear(chain=True)): scheduling only.  The flows must equal those of
    the same launches with grid-wide waits up to the order of the double-precision GroupNorm partial sums (the bound of the
    batch-of-8 test) -- a stale or early read would show at 1e-2.  Eager launches and CUDA-graph replay, several repeats,
    a batch large enough (4 x 64 tiles over 148 SMs) for CTAs to run ahead of the previous launch's last tiles."""
    from pvraft_b200 import ops
    m, _ = make_model(dev)
    b, iters = 4, 12
    pc1, pc2 = [t.to(dev) for t in O.synthetic_clouds(b, N, seed=123)]
    was = ops._CHAIN
    runs = {}
    with torch.no_grad():
        for graph in (False, True):
            m.use_cuda_graph = graph
            try:
                ops._CHAIN = False
                m.reset_graphs()
                plain = m([pc1, pc2], iters)[-1].clone()
                ops._CHAIN = True
                m.reset_graphs()
                runs[graph] = (plain, [m([pc1, pc2], iters)[-1].clone() for _ in range(4)])
            finally:
                ops._CHAIN = was
    scale = float(runs[False][0].abs().mean())
    for graph, (plain, chained) in runs.items():
        errs = [float((c - plain).abs().mean()) / scale for c in chained]
        print(f'chained vs grid-wide waits ({"graph replay" if graph else "eager"}): mean-abs / mean|flow| =', [f'{e:.1e}' for e in errs])
        assert max(errs) < 2e-4
