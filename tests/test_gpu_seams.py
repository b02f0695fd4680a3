"""The fused forward kernels of the RAFT loop, one at a time at their `ops.*` / C-ABI seam, against a float64 restatement of
the reference formula on random inputs and random parameters.

The module-level tests compare whole outputs with one `max|err| / max|ref|` number and mostly at the default init (GroupNorm
(1, 0), PReLU 0.25), which hides whole branches: the PReLU variants of the kNN branch, the residual term of the ConvGRU
gate epilogue, the coordinate update and user-order scatter of the flow epilogue, ragged tiles.  Here every kernel meets
GroupNorm scales drawn around 0.8 with spread 0.5 (some negative), shifts ~ 0.2 N(0, 1), PReLU slopes from SLOPES (negative,
zero, the default, 1, above 1), B in {1, 3}, ragged and full tiles, and for the tensor-core layers one shape with several
128-point tiles per CTA (B = 8, N = 8192: 512 tiles on 148 SMs, both TMEM accumulators and the phase wrap in use).

Two metrics per output: `rel_err` (max-abs error over max-abs reference) and the per-channel
`max_c max_n |got - want| / max_n |want_c|`, which a wrong small channel cannot hide behind a large one.  Bounds are about 5x
the worst value measured on a B200 (1000 W power limit); `-s` prints the measured values.
"""
import pytest
import torch

from conftest import rel_err
from oracle import pvraft_oracle as O

pytestmark = pytest.mark.gpu

SLOPES = (-0.5, 0.0, 0.25, 1.0, 1.7)
TC_SHAPES = [(1, 1024), (3, 1024), (8, 8192)]
LEVELS, SCALE, K = 3, 0.25, 128


@pytest.fixture(scope='module')
def dev():
    return torch.device('cuda:0')


@pytest.fixture(scope='module', autouse=True)
def _cpu_threads():
    old = torch.get_num_threads()
    torch.set_num_threads(min(16, old))
    yield
    torch.set_num_threads(old)


def chan_err(got, want):
    """max over channels (last axis) of max|got - want| / max|want| within the channel."""
    g = got.detach().cpu().double().reshape(-1, got.shape[-1])
    w = want.detach().cpu().double().reshape(-1, want.shape[-1])
    return float(((g - w).abs().amax(0) / w.abs().amax(0).clamp_min(1e-30)).max())


def check(tag, got, want, bound, chan_bound=None):
    """rel_err below `bound`, the per-channel error below `chan_bound` (default: the same); NaN anywhere fails.
    A ReLU output channel that is zero at almost every point has a small maximum, so the fp32 rounding of its few non-zero
    entries reads large against it: those outputs get a looser per-channel bound."""
    chan_bound = bound if chan_bound is None else chan_bound
    e1, e2 = rel_err(got.detach().cpu(), want), chan_err(got, want)
    print(f'{tag}: rel {e1:.2e}  per-channel {e2:.2e}  (bounds {bound:.1e} / {chan_bound:.1e})')
    assert e1 < bound and e2 < chan_bound, (tag, e1, e2)


def rnd(g, *shape, scale=1.0, shift=0.0):
    return torch.randn(*shape, generator=g) * scale + shift


def gn_params(g, c):
    """GroupNorm (gamma, beta): gamma ~ N(0.8, 0.5) -- some negative --, beta ~ 0.2 N(0, 1)."""
    return rnd(g, c, scale=0.5, shift=0.8), rnd(g, c, scale=0.2)


def gn_sums(x):
    """[B,N,C] -> [B,8,2] float64 (sum, sum of squares) per GroupNorm group: what the producers of a layer accumulate."""
    b, n, c = x.shape
    xg = x.double().reshape(b, n, 8, c // 8)
    return torch.stack([xg.sum((1, 3)), (xg ** 2).sum((1, 3))], -1)


def gn_fp64(x, gamma, beta):
    """GroupNorm(8, C) of a point-major [B,N,C] tensor in float64 (O.group_norm on the channel-major view)."""
    return O.group_norm(x.double().transpose(1, 2), gamma.double(), beta.double()).transpose(1, 2)


def slope_t(slope):
    """The slope as the one-element fp32 parameter holds it, widened exactly."""
    return torch.tensor([slope], dtype=torch.float32).double()


def to(dev, *ts):
    return [t.to(dev).contiguous() if t is not None else None for t in ts]


# ----------------------------------------------------------------------------------------------------
# lookup state: knn_sel / moments / vox come from the lookup kernel itself (pinned bit-exact by test_gpu_parity)
# ----------------------------------------------------------------------------------------------------
_LOOKUPS = {}


def lookup_state(dev, b, n):
    key = (b, n)
    if key not in _LOOKUPS:
        from pvraft_b200 import CorrBlock
        state, coords, xyz2 = O.synthetic_state(b, n, K, seed=100 + n + b, box=3.0)
        cb = CorrBlock(num_levels=LEVELS, base_scale=SCALE, truncate_k=K).to(dev)
        cb.set_state(state.truncated_corr.to(dev), state.indices.to(torch.int32).to(dev), xyz2.to(dev))
        coords = coords.to(dev).contiguous()
        lk = cb.lookup(coords)
        torch.cuda.synchronize()
        _LOOKUPS[key] = (cb, coords, lk)
    return _LOOKUPS[key]


def knn_branch_fp64(sel, w, bias, gamma, beta, slope):
    """model/corr.py:86-92 in float64: conv 4->64 on the [B,N,32,4] selection, GroupNorm over the whole [B,64,N,32] tensor,
    PReLU, max over the 32 neighbours -> [B,N,64]."""
    t = sel.double() @ w.double().reshape(64, 4).t() + bias.double()           # [B,N,32,64]
    t = O.group_norm(t.permute(0, 3, 1, 2), gamma.double(), beta.double())      # [B,64,N,32]
    t = O.prelu(t, slope_t(slope))
    return t.amax(3).transpose(1, 2)


def knn_branch_params(g):
    w = rnd(g, 64, 4, scale=0.5)
    bias = rnd(g, 64, scale=2.0)        # channel means spread within a group: some channels mostly below zero after GN
    gamma, beta = gn_params(g, 64)
    return w, bias, gamma, beta, rnd(g, 64, 3, scale=0.5), rnd(g, 64, scale=0.3)


# ----------------------------------------------------------------------------------------------------
# A1. k_knn_branch: both PReLU variants, partial tiles
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('slope', SLOPES)
@pytest.mark.parametrize('n', [1000, 1024])
@pytest.mark.parametrize('b', [1, 3])
def test_knn_branch_fp64(dev, b, n, slope):
    """kfeat = max_e PReLU(GN(knn_conv.0(f_e))) with the GroupNorm statistics folded from the lookup's moments, and
    cflow = relu(conv_flow(flow)).  The kernel picks its variant from the host copy of the slope: the endpoint shortcut
    max(PReLU(max t), PReLU(min t)) for slope <= 1, per-candidate PReLU above.  The shortcut is exact for every slope
    (fp32 multiplication by the slope is monotone), so both variants run on the same device slope and must agree with
    float64 and with each other bit for bit.  N = 1000 ends on a partial 64-point tile."""
    from pvraft_b200 import _lib, ops
    _, _, lk = lookup_state(dev, b, n)
    g = torch.Generator().manual_seed(int(1000 * slope) + n + b)
    w, bias, gamma, beta, w_cf, b_cf = knn_branch_params(g)
    flow = rnd(g, b, n, 3, scale=0.3)
    w_d, bias_d, gamma_d, beta_d, w_cf_d, b_cf_d, flow_d = to(dev, w, bias, gamma, beta, w_cf, b_cf, flow)
    slope_d = torch.tensor([slope], dtype=torch.float32, device=dev)

    def run(host_slope, with_flow):
        a = _lib.KnnBranchArgs()
        a.knn_sel, a.moments = ops._p(lk['knn_sel']), ops._p(lk['moments'], torch.float64)
        a.w_knn, a.b_knn, a.gnk_gamma, a.gnk_beta, a.preluk = (ops._p(t) for t in (w_d, bias_d, gamma_d, beta_d, slope_d))
        a.preluk_host = host_slope
        kfeat = torch.empty(b, n, 64, dtype=torch.float32, device=dev)
        a.kfeat = ops._p(kfeat)
        cflow = None
        if with_flow:
            cflow = torch.empty(b, n, 64, dtype=torch.float32, device=dev)
            a.flow, a.cflow, a.w_cf, a.b_cf = ops._p(flow_d), ops._p(cflow), ops._p(w_cf_d), ops._p(b_cf_d)
        a.B, a.N = b, n
        ops.knn_branch(a)
        return kfeat, cflow

    want = knn_branch_fp64(lk['knn_sel'].cpu(), w, bias, gamma, beta, slope)
    natural, cflow = run(slope, True)
    check(f'knn_branch b={b} n={n} slope={slope} kfeat', natural, want, 8e-6)
    want_cf = torch.relu(flow.double() @ w_cf.double().t() + b_cf.double())
    check(f'knn_branch b={b} n={n} slope={slope} cflow', cflow, want_cf, 5e-7, 2e-4)
    other = 0.5 if slope > 1.0 else 1.7            # the other variant on the same device slope
    forced, none = run(other, False)
    assert none is None
    assert torch.equal(forced, natural), 'convex shortcut and per-candidate PReLU differ'
    if slope > 1.0:
        read_back, _ = run(float('nan'), False)     # NaN: the slope is read from the device
        assert torch.equal(read_back, natural)


# ----------------------------------------------------------------------------------------------------
# A2. correlation feature + MotionEncoder
# ----------------------------------------------------------------------------------------------------
def randomise_block(module, g, slope):
    """Every parameter of a CorrBlock / MotionEncoder redrawn: convolutions ~ N(0, 1/fan_in), biases ~ 0.5 N(0, 1),
    GroupNorm as gn_params, both PReLU slopes = slope."""
    with torch.no_grad():
        for name, p in module.named_parameters():
            if 'out_conv.1.' in name or 'knn_conv.1.' in name:
                gamma, beta = gn_params(g, p.numel())
                p.copy_(gamma if name.endswith('weight') else beta)
            elif name.endswith('out_conv.2.weight') or name.endswith('knn_conv.2.weight'):
                p.fill_(slope)
            elif name.endswith('weight'):
                p.copy_(rnd(g, *p.shape) / (p[0].numel() ** 0.5))
            else:
                p.copy_(rnd(g, *p.shape, scale=0.5))


def corr_feature_fp64(cb, vox, sel):
    """CorrBlock.__call__ (model/corr.py:44-45) in float64 on the lookup's own voxel means and kNN selection -> [B,64,N]."""
    P = {k: v.detach().cpu().double() for k, v in cb.state_dict().items()}
    x = vox[..., :LEVELS * 27].cpu().double().transpose(1, 2)
    y = O.pointwise_linear(x, P['out_conv.0.weight'], P['out_conv.0.bias'])
    y = O.prelu(O.group_norm(y, P['out_conv.1.weight'], P['out_conv.1.bias']), P['out_conv.2.weight'])
    a = O.pointwise_linear(y, P['out_conv.3.weight'], P['out_conv.3.bias'])
    kf = knn_branch_fp64(sel.cpu(), P['knn_conv.0.weight'], P['knn_conv.0.bias'], P['knn_conv.1.weight'], P['knn_conv.1.bias'],
                         float(P['knn_conv.2.weight'].reshape(-1)[0]))
    return a + O.pointwise_linear(kf.transpose(1, 2), P['knn_out.weight'], P['knn_out.bias'])


@pytest.mark.parametrize('slope', [-0.5, 0.25, 1.7])
@pytest.mark.parametrize('n', [300, 1024])
@pytest.mark.parametrize('b', [1, 3])
def test_corr_feature_and_motion_fp64(dev, b, n, slope):
    """feature_point_major with the MotionEncoder fused into k_corrfeat (every N; out_conv.0 on the CUDA cores at N = 300),
    and at N % 128 == 0 feature_motion_tc (lookup, tcgen05 layers, k_knn_branch) with need_corr True and False."""
    from pvraft_b200 import ops
    from pvraft_b200.update import MotionEncoder
    cb, coords, lk = lookup_state(dev, b, n)
    me = MotionEncoder().to(dev)
    g = torch.Generator().manual_seed(7 * n + b + int(10 * slope))
    randomise_block(cb, g, slope)
    randomise_block(me, g, slope)
    flow = rnd(g, b, n, 3, scale=0.3)
    flow_d = flow.to(dev)
    want_corr = corr_feature_fp64(cb, lk['vox'], lk['knn_sel'])                 # [B,64,N]
    Pm = {'me.' + k: v.detach().cpu().double() for k, v in me.state_dict().items()}
    want_motion = O.motion_encoder(Pm, flow.double(), want_corr, 'me').transpose(1, 2)
    want_corr = want_corr.transpose(1, 2)
    tag = f'b={b} n={n} slope={slope}'
    with torch.no_grad():
        motion = torch.empty(b, n, 64, dtype=torch.float32, device=dev)

        def attach(a, keep):
            me.fill(a, flow_d)
            a.motion = ops._p(motion)
            keep.append(motion)

        corr, _ = cb.feature_point_major(coords, motion_args=attach)
        check(f'feature_point_major {tag} corr', corr, want_corr, 5e-6)
        check(f'feature_point_major {tag} motion', motion, want_motion, 3e-6, 2e-4)
        assert torch.equal(motion[..., 61:], flow_d)
        if ops.tc_supported(n):
            corr_tc, motion_tc = cb.feature_motion_tc(coords, flow_d, me, need_corr=True)
            check(f'feature_motion_tc {tag} corr', corr_tc, want_corr, 1e-5, 2e-5)
            check(f'feature_motion_tc {tag} motion', motion_tc, want_motion, 1.6e-5, 7e-4)
            none, motion_f = cb.feature_motion_tc(coords, flow_d, me, need_corr=False)
            assert none is None
            check(f'feature_motion_tc(need_corr=False) {tag} motion', motion_f, want_motion, 1.6e-5, 7e-4)
            assert torch.equal(motion_tc[..., 61:], flow_d) and torch.equal(motion_f[..., 61:], flow_d)


# ----------------------------------------------------------------------------------------------------
# A3. tensor-core epilogues
# ----------------------------------------------------------------------------------------------------
def gru_inputs(g, b, n):
    h = torch.tanh(rnd(g, b, n, 64))
    inp = torch.relu(rnd(g, b, n, 64))
    mot = torch.relu(rnd(g, b, n, 64))
    return h, inp, mot


def gru_weights(g):
    return {f'gru.conv{k}.{p}': (rnd(g, 64, 192, 1) / 192 ** 0.5 if p == 'weight' else rnd(g, 64, scale=0.5))
            for k in 'zrq' for p in ('weight', 'bias')}


@pytest.mark.parametrize('b,n', TC_SHAPES)
@pytest.mark.parametrize('terms', ['bias', 'residual', 'both'])
def test_tc_gru_zr_fp64(dev, b, n, terms):
    """TC_GRU_ZR: [z | r] = sigmoid([h, inp, motion] W_zr^T + bias/bias2 + residual); out = z, out2 = r * h."""
    from pvraft_b200 import ops
    g = torch.Generator().manual_seed(b * n + len(terms))
    h, inp, mot = gru_inputs(g, b, n)
    wz, wr = rnd(g, 64, 192) / 192 ** 0.5, rnd(g, 64, 192) / 192 ** 0.5
    bz, br = rnd(g, 64, scale=0.5), rnd(g, 64, scale=0.5)
    res = rnd(g, b, n, 128, scale=0.7)
    use_bias, use_res = terms in ('bias', 'both'), terms in ('residual', 'both')
    pre = torch.cat([h, inp, mot], -1).double() @ torch.cat([wz, wr]).double().t()
    if use_bias:
        pre = pre + torch.cat([bz, br]).double()
    if use_res:
        pre = pre + res.double()
    want_z = torch.sigmoid(pre[..., :64])
    want_rh = torch.sigmoid(pre[..., 64:]) * h.double()
    h_d, inp_d, mot_d, wz_d, wr_d, bz_d, br_d, res_d = to(dev, h, inp, mot, wz, wr, bz, br, res)
    z = torch.empty(b, n, 64, device=dev)
    rh = torch.empty(b, n, 64, device=dev)
    ops.tc_linear([h_d, inp_d, mot_d], ops.tc_weights((wz_d, wr_d)), bz_d if use_bias else None,
                  bias2=br_d if use_bias else None, residual=res_d if use_res else None, epilogue=ops.TC_GRU_ZR,
                  out=z, out2=rh, h=h_d, cout=64)
    check(f'TC_GRU_ZR {terms} b={b} n={n} z', z, want_z, 7e-6)
    check(f'TC_GRU_ZR {terms} b={b} n={n} r*h', rh, want_rh, 7e-6)


@pytest.mark.parametrize('b,n', TC_SHAPES)
@pytest.mark.parametrize('with_residual', [False, True])
def test_tc_gru_q_fp64(dev, b, n, with_residual):
    """TC_GRU_Q: h' = (1 - z) h + z tanh([r*h, inp, motion] W_q^T + bias (+ residual))."""
    from pvraft_b200 import ops
    g = torch.Generator().manual_seed(b * n + 3 + with_residual)
    h, inp, mot = gru_inputs(g, b, n)
    rh = torch.sigmoid(rnd(g, b, n, 64)) * h
    z = torch.sigmoid(rnd(g, b, n, 64, scale=2.0))
    wq, bq = rnd(g, 64, 192) / 192 ** 0.5, rnd(g, 64, scale=0.5)
    res = rnd(g, b, n, 64, scale=0.7)
    pre = torch.cat([rh, inp, mot], -1).double() @ wq.double().t() + bq.double()
    if with_residual:
        pre = pre + res.double()
    want = (1 - z.double()) * h.double() + z.double() * torch.tanh(pre)
    h_d, rh_d, inp_d, mot_d, z_d, wq_d, bq_d, res_d = to(dev, h, rh, inp, mot, z, wq, bq, res)
    out = torch.empty(b, n, 64, device=dev)
    ops.tc_linear([rh_d, inp_d, mot_d], ops.tc_weights(wq_d), bq_d, residual=res_d if with_residual else None,
                  epilogue=ops.TC_GRU_Q, out=out, h=h_d, z=z_d, cout=64)
    check(f'TC_GRU_Q residual={with_residual} b={b} n={n}', out, want, 1.5e-5)


def gru_module(dev, W):
    from pvraft_b200.update import ConvGRU
    m = ConvGRU()
    m.load_state_dict({k[len('gru.'):]: v for k, v in W.items()})
    return m.to(dev)


def conv_gru_fp64(W, h, inp, mot):
    P = {k: v.double() for k, v in W.items()}
    x = torch.cat([inp, mot], -1).double().transpose(1, 2)
    return O.conv_gru(P, h.double().transpose(1, 2), x, 'gru').transpose(1, 2)


@pytest.mark.parametrize('b,n', TC_SHAPES)
def test_tc_gru_chain_vs_oracle(dev, b, n):
    """ConvGRU.forward_pm on the tensor cores: the TC_GRU_ZR launch feeding TC_GRU_Q, against O.conv_gru in float64."""
    g = torch.Generator().manual_seed(b + n + 11)
    h, inp, mot = gru_inputs(g, b, n)
    W = gru_weights(g)
    with torch.no_grad():
        got = gru_module(dev, W).forward_pm(*to(dev, h, inp, mot))
    check(f'ConvGRU tcgen05 b={b} n={n}', got, conv_gru_fp64(W, h, inp, mot), 1.2e-5)


def flow_head_inputs(g, b, n):
    z3 = rnd(g, b, n, 64, scale=1.3, shift=0.4)
    net = torch.tanh(rnd(g, b, n, 64))
    gamma, beta = gn_params(g, 64)
    coords1 = rnd(g, b, n, 3, scale=3.0)
    coords2 = coords1 + rnd(g, b, n, 3, scale=0.2)
    return z3, net, gamma, beta, coords1, coords2


def a3_fp64(z3, gamma, beta):
    """LeakyReLU(0.1)(GN3(z3)) in float64: the SetConv output that the flow head's first layer reads (gconv.py:82-83)."""
    return O.leaky_relu(gn_fp64(z3, gamma, beta))


@pytest.mark.parametrize('b,n', TC_SHAPES)
@pytest.mark.parametrize('alias', [True, False])
def test_tc_flow_fp64(dev, b, n, alias):
    """TC_FLOW with the GN3 prologue: delta = w3 . relu([a3, net] W^T + bias) + b3; coords2_out = coords2 + delta (in place
    when coords2_out aliases coords2, as the loop calls it); flow_out = coords2_out - coords1; flow_user[row_map[r]] =
    flow_out[r] for a random per-sample row map."""
    from pvraft_b200 import ops
    g = torch.Generator().manual_seed(b * n + 17 + alias)
    z3, net, gamma, beta, coords1, coords2 = flow_head_inputs(g, b, n)
    w, bias = rnd(g, 64, 128) / 128 ** 0.5, rnd(g, 64, scale=0.3)
    w3, b3 = rnd(g, 3, 64) / 8.0, rnd(g, 3, scale=0.1)
    perm = torch.stack([torch.randperm(n, generator=g) for _ in range(b)]) + (torch.arange(b) * n).view(b, 1)
    row_map = perm.reshape(-1).to(torch.int32)
    y = torch.relu(torch.cat([a3_fp64(z3, gamma, beta), net.double()], -1) @ w.double().t() + bias.double())
    want_delta = y @ w3.double().t() + b3.double()
    z3_d, net_d, gamma_d, beta_d, c1_d, c2_d, w_d, bias_d, w3_d, b3_d, row_map_d = to(
        dev, z3, net, gamma, beta, coords1, coords2, w, bias, w3, b3, row_map)
    c2_before = c2_d.clone()
    delta = torch.empty(b, n, 3, device=dev)
    flow_out = torch.empty(b, n, 3, device=dev)
    flow_user = torch.empty(b, n, 3, device=dev)
    c2_out = c2_d if alias else torch.empty(b, n, 3, device=dev)
    ops.tc_linear([z3_d, net_d], ops.tc_weights(w_d), bias_d, in_stats=gn_sums(z3).to(dev), in_gamma=gamma_d, in_beta=beta_d,
                  in_count=float(n) * 8.0, in_act=ops.ACT_LRELU, in_slope=0.1, epilogue=ops.TC_FLOW, out=delta, cout=64,
                  w3=w3_d, b3=b3_d, coords1=c1_d, coords2=c2_d, coords2_out=c2_out, flow_out=flow_out, flow_user=flow_user,
                  row_map=row_map_d)
    check(f'TC_FLOW alias={alias} b={b} n={n} delta', delta, want_delta, 8e-6)
    assert torch.equal(c2_out, c2_before + delta)                       # the same fp32 additions
    assert torch.equal(flow_out, c2_out - c1_d)
    if not alias:
        assert torch.equal(c2_d, c2_before), 'coords2 was written through a separate coords2_out'
    assert torch.equal(flow_user.reshape(-1, 3)[row_map_d.long()], flow_out.reshape(-1, 3))


@pytest.mark.parametrize('b,n', [(3, 1024), (8, 8192)])
@pytest.mark.parametrize('layout', ['tail', 'three_sources', 'kcat', 'cols_kpad'])
def test_tc_plain_layouts_fp64(dev, b, n, layout):
    """The plain epilogue with the operand layouts the loop uses: a 3-column tail (MotionEncoder.conv + cat flow), three
    64-channel sources, a 128 + 64 K concatenation of two weights (kcat) behind a GroupNorm + PReLU prologue on source 0 only,
    and the 81 of 96 columns of out_conv.0 (cols=81, k_pad=96; the padding columns of the source hold junk)."""
    from pvraft_b200 import ops
    g = torch.Generator().manual_seed(b * n + len(layout))
    tag = f'{layout} b={b} n={n}'
    if layout == 'tail':
        cc, cfl, flow = torch.relu(rnd(g, b, n, 64)), torch.relu(rnd(g, b, n, 64)), rnd(g, b, n, 3)
        w, bias = rnd(g, 61, 128) / 128 ** 0.5, rnd(g, 61, scale=0.3)
        want = torch.relu(torch.cat([cc, cfl], -1).double() @ w.double().t() + bias.double())
        cc_d, cfl_d, flow_d, w_d, bias_d = to(dev, cc, cfl, flow, w, bias)
        got = ops.tc_linear([cc_d, cfl_d], ops.tc_weights(w_d), bias_d, out_act=ops.ACT_RELU, tail=flow_d)
        assert got.shape == (b, n, 64)
        check(f'tc plain {tag}', got[..., :61], want, 1e-5, 1.4e-5)
        assert torch.equal(got[..., 61:], flow_d)
    elif layout == 'three_sources':
        xs = [rnd(g, b, n, 64, shift=0.1 * i) for i in range(3)]
        w, bias = rnd(g, 64, 192) / 192 ** 0.5, rnd(g, 64, scale=0.3)
        want = torch.cat(xs, -1).double() @ w.double().t() + bias.double()
        *xs_d, w_d, bias_d = to(dev, *xs, w, bias)
        got = ops.tc_linear(xs_d, ops.tc_weights(w_d), bias_d)
        check(f'tc plain {tag}', got, want, 1e-5)
    elif layout == 'kcat':
        y1, kf = rnd(g, b, n, 128, scale=2.0, shift=0.5), rnd(g, b, n, 64)
        gamma, beta = gn_params(g, 128)
        wa, wb = rnd(g, 64, 128) / 128 ** 0.5, rnd(g, 64, 64) / 8.0
        bias = rnd(g, 64, scale=0.3)
        slope = -0.5
        a = O.prelu(gn_fp64(y1, gamma, beta), slope_t(slope))
        want = a @ wa.double().t() + kf.double() @ wb.double().t() + bias.double()
        y1_d, kf_d, gamma_d, beta_d, wa_d, wb_d, bias_d = to(dev, y1, kf, gamma, beta, wa, wb, bias)
        got = ops.tc_linear([y1_d, kf_d], ops.tc_weights((wa_d, wb_d), kcat=True), bias_d, in_stats=gn_sums(y1).to(dev),
                            in_gamma=gamma_d, in_beta=beta_d, in_count=float(n) * 16.0, in_act=ops.ACT_LRELU, in_slope=slope)
        check(f'tc plain {tag}', got, want, 1e-5)
    else:
        vox = torch.rand(b, n, 96, generator=g) * 4.0
        vox[..., 81:] = rnd(g, b, n, 15, scale=100.0)              # junk behind the 81 used columns
        w, bias = rnd(g, 128, 81) / 9.0, rnd(g, 128, scale=0.3)
        want = vox[..., :81].double() @ w.double().t() + bias.double()
        stats = torch.zeros(b, 8, 2, dtype=torch.float64, device=dev)
        vox_d, w_d, bias_d = to(dev, vox, w, bias)
        got = ops.tc_linear([vox_d], ops.tc_weights(w_d, cols=81, k_pad=96), bias_d, out_stats=stats)
        check(f'tc plain {tag}', got, want, 1e-5)
        s = gn_sums(want)
        # (the kernel sums its own fp32 outputs in fp32 over 32 rows before the double atomics: measured 1.3e-6)
        assert torch.allclose(stats.cpu()[..., 1], s[..., 1], rtol=6e-6)
        assert ((stats.cpu()[..., 0] - s[..., 0]).abs() <= 6e-6 * gn_sums(want.abs())[..., 0]).all()


# ----------------------------------------------------------------------------------------------------
# A4. CUDA-core twins (N % 128 != 0 path)
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('n', [65, 300, 1024])
@pytest.mark.parametrize('b', [1, 3])
def test_cuda_core_gru(dev, b, n):
    """k_gru (GruArgs) against O.conv_gru in float64; at N = 1024 also against the tcgen05 pair it stands in for."""
    from pvraft_b200 import _lib, ops
    g = torch.Generator().manual_seed(31 * n + b)
    h, inp, mot = gru_inputs(g, b, n)
    W = gru_weights(g)
    h_d, inp_d, mot_d = to(dev, h, inp, mot)
    Wd = {k: v.to(dev).contiguous() for k, v in W.items()}
    out = torch.empty(b, n, 64, device=dev)
    a = _lib.GruArgs(ops._p(h_d), ops._p(inp_d), ops._p(mot_d), *(ops._p(Wd[f'gru.conv{k}.{p}']) for k in 'zrq' for p in ('weight', 'bias')),
                     ops._p(out), b, n)
    ops.gru(a)
    check(f'k_gru b={b} n={n}', out, conv_gru_fp64(W, h, inp, mot), 3e-6)
    if ops.tc_supported(n):
        with torch.no_grad():
            tc = gru_module(dev, W).forward_pm(h_d, inp_d, mot_d)
        assert rel_err(out.cpu(), tc.cpu()) < 5e-6


@pytest.mark.parametrize('n', [65, 300, 1024])
@pytest.mark.parametrize('b', [1, 3])
def test_cuda_core_flow_out(dev, b, n):
    """k_flowout (FlowOutArgs): GN3 prologue, conv1, out_conv and the coordinate update against float64; at N = 1024 also
    against TC_FLOW with conv1 folded into the weight (FlowHead.forward_pm)."""
    from pvraft_b200 import _lib, ops
    from pvraft_b200.update import fold_flow_head
    g = torch.Generator().manual_seed(37 * n + b)
    z3, net, gamma, beta, coords1, coords2 = flow_head_inputs(g, b, n)
    w_c1, b_c1 = rnd(g, 64, 64, 1) / 8.0, rnd(g, 64, scale=0.3)
    w_o0, b_o0 = rnd(g, 64, 128, 1) / 128 ** 0.5, rnd(g, 64, scale=0.3)
    w_o2, b_o2 = rnd(g, 3, 64, 1) / 8.0, rnd(g, 3, scale=0.1)
    c1 = net.double() @ w_c1.double().reshape(64, 64).t() + b_c1.double()
    y = torch.relu(torch.cat([a3_fp64(z3, gamma, beta), c1], -1) @ w_o0.double().reshape(64, 128).t() + b_o0.double())
    want = y @ w_o2.double().reshape(3, 64).t() + b_o2.double()
    d = dict(zip(('z3', 'net', 'gamma', 'beta', 'c1', 'c2', 'w_c1', 'b_c1', 'w_o0', 'b_o0', 'w_o2', 'b_o2'),
                 to(dev, z3, net, gamma, beta, coords1, coords2, w_c1, b_c1, w_o0, b_o0, w_o2, b_o2)))
    stats = gn_sums(z3).to(dev)
    delta, c2_out, flow_out = (torch.empty(b, n, 3, device=dev) for _ in range(3))
    a = _lib.FlowOutArgs(ops._p(d['z3']), ops._p(stats, torch.float64), ops._p(d['gamma']), ops._p(d['beta']), ops._p(d['net']),
                         ops._p(d['w_c1']), ops._p(d['b_c1']), ops._p(d['w_o0']), ops._p(d['b_o0']), ops._p(d['w_o2']),
                         ops._p(d['b_o2']), ops._p(d['c1']), ops._p(d['c2']), ops._p(delta), ops._p(c2_out), ops._p(flow_out), b, n)
    ops.flow_out(a)
    check(f'k_flowout b={b} n={n} delta', delta, want, 2.5e-6)
    assert torch.equal(c2_out, d['c2'] + delta) and torch.equal(flow_out, c2_out - d['c1'])
    if ops.tc_supported(n):
        w_eff, b_eff = fold_flow_head(d['w_o0'], d['w_c1'], d['b_c1'], d['b_o0'])
        tc = ops.tc_linear([d['z3'], d['net']], ops.tc_weights(w_eff), b_eff, in_stats=stats, in_gamma=d['gamma'],
                           in_beta=d['beta'], in_count=float(n) * 8.0, in_act=ops.ACT_LRELU, in_slope=0.1, epilogue=ops.TC_FLOW,
                           cout=64, out=torch.empty(b, n, 3, device=dev), w3=d['w_o2'].reshape(3, 64).contiguous(), b3=d['b_o2'])
        assert rel_err(delta.cpu(), tc.cpu()) < 1e-5


@pytest.mark.parametrize('n', [65, 300])
def test_cuda_core_linear_gn_minmax_ragged(dev, n):
    """k_linear in IN_GN_MINMAX mode (the SetConv fc2 input: max-pool commuted with GN + LeakyReLU, min where the folded
    scale is negative) at ragged point counts."""
    from pvraft_b200 import ops
    b, cin, cout = 3, 64, 128
    g = torch.Generator().manual_seed(n)
    xmax = rnd(g, b, n, cin, scale=1.5, shift=0.2)
    xmin = xmax - torch.rand(b, n, cin, generator=g) * 2.0
    gamma, beta = gn_params(g, cin)
    assert (gamma < 0).any()
    w, bias = rnd(g, cout, cin) / 8.0, rnd(g, cout, scale=0.3)
    stats = gn_sums(xmax)             # any statistics do: the kernel takes them as given
    cnt = float(n * cin // 8)
    mean = stats[..., 0] / cnt
    rstd = (stats[..., 1] / cnt - mean ** 2 + 1e-5).rsqrt()
    sc = (rstd.repeat_interleave(cin // 8, 1) * gamma.double()).unsqueeze(1)
    sh = beta.double() - mean.repeat_interleave(cin // 8, 1).unsqueeze(1) * sc
    t = torch.where(sc < 0, xmin.double(), xmax.double()) * sc + sh
    want = O.leaky_relu(t) @ w.double().t() + bias.double()
    xmax_d, xmin_d, gamma_d, beta_d, w_d, bias_d = to(dev, xmax, xmin, gamma, beta, w, bias)
    got = ops.linear(xmax_d, w_d, bias_d, in_mode=ops.IN_GN_MINMAX, in_min=xmin_d, in_stats=stats.to(dev), in_gamma=gamma_d,
                     in_beta=beta_d, in_count=cnt, in_act=ops.ACT_LRELU, in_slope=0.1)
    check(f'k_linear GN_MINMAX n={n}', got, want, 2.5e-6)


# ----------------------------------------------------------------------------------------------------
# A5. SetConv edge stage and the point order
# ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('c', [16, 48, 64, 96, 128])
def test_setconv_edge_fp64(dev, c):
    """y_e = P_j - P_i + W_e . e over the 32 neighbours (the point itself and repeated neighbours among them): max / min
    against float64, GroupNorm sums to 3e-8 of the sum of magnitudes, and a processing order that changes no output bit."""
    from pvraft_b200 import ops
    b, n, cin = 3, 1000, 32
    g = torch.Generator().manual_seed(c)
    fc1p = rnd(g, b, n, c, shift=0.3)
    nbr = torch.randint(0, n, (b, n, 32), generator=g)
    nbr[..., 0] = torch.arange(n)                  # the point itself (distance 0 in a kNN graph)
    nbr[..., 5] = nbr[..., 4]                      # repeated neighbours
    nbr[..., 31] = nbr[..., 1]
    nbr = nbr.to(torch.int32)
    ef = torch.rand(b, n, 32, 3, generator=g) - 0.3
    w_fc1 = rnd(g, c, cin + 3)
    nl = nbr.long()
    pj = torch.gather(fc1p.double().unsqueeze(1).expand(b, n, n, c), 2, nl.unsqueeze(-1).expand(b, n, 32, c))
    y = pj - fc1p.double().unsqueeze(2) + ef.double() @ w_fc1[:, cin:].double().t()     # [B,N,32,C]
    fc1p_d, nbr_d, ef_d, w_d = to(dev, fc1p, nbr, ef, w_fc1)
    stats = torch.zeros(b, 8, 2, dtype=torch.float64, device=dev)
    ymax, ymin = ops.setconv_edge(fc1p_d, nbr_d, ef_d, w_d, cin, stats)
    check(f'setconv_edge C={c} max', ymax, y.amax(2), 5e-7)
    check(f'setconv_edge C={c} min', ymin, y.amin(2), 5e-7)
    yg = y.reshape(b, n * 32, 8, c // 8)
    s1, s2, mag = yg.sum((1, 3)), (yg ** 2).sum((1, 3)), yg.abs().sum((1, 3))
    e1 = float(((stats[..., 0].cpu() - s1).abs() / mag).max())
    e2 = float(((stats[..., 1].cpu() - s2).abs() / s2).max())
    print(f'setconv_edge C={c} GroupNorm sums: {e1:.2e} (of sum |y|), sum of squares {e2:.2e}')
    assert e1 < 3e-8 and e2 < 3e-8
    order = torch.stack([torch.randperm(n, generator=g) for _ in range(b)]).to(torch.int32).to(dev)
    stats_o = torch.zeros_like(stats)
    ymax_o, ymin_o = ops.setconv_edge(fc1p_d, nbr_d, ef_d, w_d, cin, stats_o, order=order)
    assert torch.equal(ymax_o, ymax) and torch.equal(ymin_o, ymin)
    assert torch.allclose(stats_o, stats, rtol=1e-12, atol=0)   # (only the order of the double partial sums differs)


@pytest.mark.parametrize('n', [64, 1000, 8192])
@pytest.mark.parametrize('cloud', ['uniform', 'duplicated'])
def test_point_order_is_permutation(dev, n, cloud):
    """ops.point_order is a permutation of every sample (the SetConv edge kernel processes exactly the points it lists)."""
    from pvraft_b200 import ops
    b = 3
    g = torch.Generator().manual_seed(n)
    pts = torch.rand(b, n, 3, generator=g) * 10.0
    if cloud == 'duplicated':
        pts[:, 1::2] = pts[:, 0::2][:, :n // 2]
        pts[1] = 1.0                                 # one sample with every point equal
    perm = ops.point_order(pts.to(dev), as_int32=True)
    assert perm.dtype == torch.int32 and perm.shape == (b, n)
    assert torch.equal(perm.cpu().long().sort(-1).values, torch.arange(n).expand(b, n))


# ----------------------------------------------------------------------------------------------------
# A6. bf16 state pack
# ----------------------------------------------------------------------------------------------------
def bits_to_f32(bits):
    return torch.tensor(bits, dtype=torch.int64).to(torch.int32).view(torch.float32)


def pack(dev, vals, ids=None):
    from pvraft_b200 import ops
    m = vals.numel()
    ids = torch.zeros(m, dtype=torch.int32) if ids is None else ids
    v16, i16 = ops.corr_state_pack_bf16(vals.reshape(1, 1, m).to(dev), ids.reshape(1, 1, m).to(torch.int32).to(dev))
    return v16.reshape(-1).cpu(), i16.reshape(-1).cpu()


def test_state_pack_bf16_rounding(dev):
    """Round to nearest even, bit-exact against torch's conversion: exact halfway cases both ways, a carry into the exponent,
    FLT_MAX (rounds to inf), subnormals, signed zeros and infinities; uint16 ids past the signed 16-bit boundary."""
    crafted = [
        0x3F808000, 0x3F818000, 0xBF808000, 0xBF818000,    # exact halfway: even stays, odd rounds up (magnitude)
        0x3F808001, 0x3F807FFF, 0x3F817FFF,                # just above / below halfway
        0x3FFFFFFF, 0x3FFF8000, 0xBFFF8000, 0x7F7F8000,    # carry into the exponent (the last one to inf)
        0x7F7FFFFF, 0xFF7FFFFF,                            # +-FLT_MAX -> +-inf
        0x00000001, 0x00008000, 0x00018000, 0x007FFFFF, 0x80000001, 0x807F8000, 0x00800000,   # subnormals
        0x00000000, 0x80000000, 0x7F800000, 0xFF800000,    # +-0, +-inf
    ]
    vals = bits_to_f32(crafted)
    g = torch.Generator().manual_seed(0)
    vals = torch.cat([vals, torch.randn(100000, generator=g) * torch.exp2(torch.randint(-140, 128, (100000,), generator=g).float())])
    ids = torch.cat([torch.tensor([0, 1, 32767, 32768, 65535, 40000], dtype=torch.int32),
                     torch.randint(0, 65536, (vals.numel() - 6,), generator=g, dtype=torch.int32)])
    v16, i16 = pack(dev, vals, ids)
    want = vals.to(torch.bfloat16)
    bad = (v16.view(torch.int16) != want.view(torch.int16)).nonzero().reshape(-1)
    assert bad.numel() == 0, [(hex(int(vals[i].view(torch.int32)) & 0xFFFFFFFF), hex(int(v16[i].view(torch.int16)) & 0xFFFF),
                               hex(int(want[i].view(torch.int16)) & 0xFFFF)) for i in bad[:8]]
    assert torch.equal(i16.to(torch.int32) & 0xFFFF, ids)


def test_state_pack_bf16_nan_stays_nan(dev):
    """Every NaN packs to a NaN with its sign kept -- also one whose payload lies in the 16 bits the conversion drops, which
    truncation would turn into inf.  (torch canonicalises NaN payloads, so only NaN-ness and the sign are compared.)"""
    nan_bits = [0x7FC00000, 0x7F800001, 0x7F80FFFF, 0xFF80FFFF, 0xFF800001, 0x7FFFFFFF, 0xFFC00001, 0x7F810000]
    vals = bits_to_f32(nan_bits)
    assert vals.isnan().all()
    v16, _ = pack(dev, vals)
    got = v16.float()
    assert got.isnan().all(), [hex(int(x) & 0xFFFF) for x in v16.view(torch.int16)]
    assert torch.equal(v16.view(torch.int16) < 0, vals.view(torch.int32) < 0)
