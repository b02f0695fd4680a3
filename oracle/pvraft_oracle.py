"""CPU oracle for the PV-RAFT hot path -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

A functional (no nn.Module) fp32 restatement, on torch-CPU tensors, of the reference's
point-voxel correlation lookup + GRU update loop.  Every function cites the reference
file:line it follows (paths relative to /root/reference).  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference` leg may import
this module; the product package `pvraft_b200` never does.

Pinning: the reference ships no tests or golden vectors (SURVEY.md section 4), so this
restatement is pinned against outputs of the reference itself, imported unmodified in the
build container by `tests/golden/make_golden.py` (fixtures committed under `tests/golden/`)
and checked by `tests/test_oracle_golden.py`.

Weights are a flat dict keyed exactly like the reference `state_dict()`
(e.g. 'corr_block.out_conv.0.weight'), so a reference checkpoint can be fed in directly.

Layout conventions follow the reference: coordinates / flows [B,N,3]; feature maps [B,C,N].
"""
from __future__ import annotations

import math
from typing import Dict, List, NamedTuple, Optional, Tuple

import torch

Params = Dict[str, torch.Tensor]

KNN = 32          # model/corr.py:9 (knn=32), model/extractor.py:9 (num_neighbors=32)
RESOLUTION = 3    # model/RAFTSceneFlow.py:18 (resolution=3)
GN_GROUPS = 8     # model/corr.py:17,25 ; model/flot/gconv.py:27,30,33
GN_EPS = 1e-5     # torch.nn.GroupNorm default


# --------------------------------------------------------------------------------------
# small building blocks
# --------------------------------------------------------------------------------------
def pointwise_linear(x: torch.Tensor, w: torch.Tensor, b: Optional[torch.Tensor] = None) -> torch.Tensor:
    """1x1 convolution over the trailing point axis: x [B,Cin,*] -> [B,Cout,*].

    Restates nn.Conv1d(k=1) / nn.Conv2d(k=1) as used throughout model/corr.py:15-29,
    model/update.py:11-13,27-29,60-66 and model/flot/gconv.py:26-33.  `w` keeps the
    reference's trailing singleton kernel dims ([Cout,Cin,1] or [Cout,Cin,1,1]).
    """
    w2 = w.reshape(w.shape[0], w.shape[1])
    shp = x.shape
    y = torch.matmul(w2, x.reshape(shp[0], shp[1], -1))
    if b is not None:
        y = y + b.view(1, -1, 1)
    return y.reshape(shp[0], w2.shape[0], *shp[2:])


def group_norm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, groups: int = GN_GROUPS) -> torch.Tensor:
    """nn.GroupNorm(groups, C): per-sample, per-group biased statistics over (C/groups, *spatial)."""
    b, c = x.shape[0], x.shape[1]
    xg = x.reshape(b, groups, -1)
    mean = xg.mean(dim=2, keepdim=True)
    var = xg.var(dim=2, unbiased=False, keepdim=True)
    xn = ((xg - mean) * torch.rsqrt(var + GN_EPS)).reshape(x.shape)
    bshape = [1, c] + [1] * (x.dim() - 2)
    return xn * gamma.view(bshape) + beta.view(bshape)


def prelu(x: torch.Tensor, a: torch.Tensor) -> torch.Tensor:
    """nn.PReLU() with a single shared slope (model/corr.py:18,26)."""
    return torch.where(x >= 0, x, a.view(-1)[0] * x)


def leaky_relu(x: torch.Tensor, slope: float = 0.1) -> torch.Tensor:
    """LeakyReLU(0.1), model/flot/gconv.py:36."""
    return torch.where(x >= 0, x, slope * x)


# --------------------------------------------------------------------------------------
# kNN graph  (model/flot/graph.py:28-89) and the kNN utility (model/pointconv.py:4-39)
# --------------------------------------------------------------------------------------
class Graph(NamedTuple):
    """Mirror of model/flot/graph.py:4-25 (edges are GLOBAL row ids b*N + j, flat)."""
    edges: torch.Tensor       # int64 [B*N*k]
    edge_feats: torch.Tensor  # f32   [B*N*k, 3]  neighbour - centre
    k_neighbors: int
    size: Tuple[int, int]


def pairwise_sqdist_expanded(pc: torch.Tensor) -> torch.Tensor:
    """||a||^2 + ||b||^2 - 2 a.b in the reference's op order (model/flot/graph.py:53-57)."""
    sq = torch.sum(pc * pc, -1, keepdim=True)
    d = sq + sq.transpose(1, 2)
    return d - 2 * torch.bmm(pc, pc.transpose(1, 2))


def construct_graph(pc: torch.Tensor, k: int = KNN) -> Graph:
    """model/flot/graph.py:28-89: k nearest (incl. self) by full argsort of the N x N distance."""
    b, n, _ = pc.shape
    nbr = torch.argsort(pairwise_sqdist_expanded(pc), -1)[..., :k]          # graph.py:60
    k_eff = nbr.shape[-1]
    centre = pc.unsqueeze(2)                                                # [B,N,1,3]
    gathered = torch.gather(pc.unsqueeze(1).expand(b, n, n, 3), 2,
                            nbr.unsqueeze(-1).expand(b, n, k_eff, 3))
    edge_feats = (gathered - centre).reshape(b * n * k_eff, 3)              # graph.py:69-74
    offs = (torch.arange(b, dtype=torch.int64, device=pc.device) * n).view(b, 1, 1)   # graph.py:77-79
    edges = (nbr + offs).reshape(-1)
    return Graph(edges, edge_feats, k_eff, (b * n, b * n))


def square_distance(src: torch.Tensor, dst: torch.Tensor) -> torch.Tensor:
    """model/pointconv.py:4-25: -2 src.dst^T, then += |src|^2, += |dst|^2 (that op order)."""
    d = -2 * torch.matmul(src, dst.permute(0, 2, 1))
    d = d + torch.sum(src * src, -1).unsqueeze(2)
    d = d + torch.sum(dst * dst, -1).unsqueeze(1)
    return d


def knn_point(nsample: int, xyz: torch.Tensor, new_xyz: torch.Tensor) -> torch.Tensor:
    """model/pointconv.py:28-39: indices of the nsample smallest distances (unsorted)."""
    return torch.topk(square_distance(new_xyz, xyz), nsample, dim=-1, largest=False, sorted=False).indices


# --------------------------------------------------------------------------------------
# SetConv  (model/flot/gconv.py:21-36,58-85)
# --------------------------------------------------------------------------------------
def set_conv(P: Params, prefix: str, signal: torch.Tensor, graph: Graph) -> torch.Tensor:
    """signal [B,N,C] -> [B,N,Cout].  fc1 over [x_j - x_i, rel_xyz] on every edge, GN, LReLU,
    max over the k neighbours, then two (1x1 conv, GN, LReLU) blocks (gconv.py:58-85)."""
    b, n, c = signal.shape
    k = graph.k_neighbors
    flat = signal.reshape(b * n, c)
    edge = flat[graph.edges].reshape(b * n, k, c) - flat.unsqueeze(1)       # gconv.py:65
    x = torch.cat([edge.reshape(-1, c), graph.edge_feats], -1)              # gconv.py:66
    x = x.reshape(b, n, k, c + 3).permute(0, 3, 2, 1)                       # [B,C+3,k,N] gconv.py:67-68
    x = pointwise_linear(x, P[prefix + '.fc1.weight'])
    x = leaky_relu(group_norm(x, P[prefix + '.gn1.weight'], P[prefix + '.gn1.bias']))
    x = x.max(dim=2).values                                                 # [B,mid,N]
    x = pointwise_linear(x, P[prefix + '.fc2.weight'])
    x = leaky_relu(group_norm(x, P[prefix + '.gn2.weight'], P[prefix + '.gn2.bias']))
    x = pointwise_linear(x, P[prefix + '.fc3.weight'])
    x = leaky_relu(group_norm(x, P[prefix + '.gn3.weight'], P[prefix + '.gn3.bias']))
    return x.transpose(1, 2)                                                # [B,N,Cout]


def flot_encoder(P: Params, prefix: str, pc: torch.Tensor, graph: Optional[Graph] = None):
    """model/extractor.py:17-24 -> (feat [B,128,N], graph)."""
    if graph is None:
        graph = construct_graph(pc, KNN)
    x = set_conv(P, prefix + '.feat_conv1', pc, graph)
    x = set_conv(P, prefix + '.feat_conv2', x, graph)
    x = set_conv(P, prefix + '.feat_conv3', x, graph)
    return x.transpose(1, 2).contiguous(), graph


def flot_refine(P: Params, prefix: str, flow: torch.Tensor, graph: Graph) -> torch.Tensor:
    """model/refine.py:16-22: three SetConvs + Linear(128,3), residual on the flow."""
    x = set_conv(P, prefix + '.ref_conv1', flow, graph)
    x = set_conv(P, prefix + '.ref_conv2', x, graph)
    x = set_conv(P, prefix + '.ref_conv3', x, graph)
    x = torch.matmul(x, P[prefix + '.fc.weight'].t()) + P[prefix + '.fc.bias']
    return flow + x


# --------------------------------------------------------------------------------------
# CorrBlock  (model/corr.py:31-100)
# --------------------------------------------------------------------------------------
class CorrState(NamedTuple):
    """What CorrBlock.init_module leaves behind as module attributes (model/corr.py:38-42)."""
    truncated_corr: torch.Tensor   # [B,N,K] f32, sorted descending along K
    indices: torch.Tensor          # [B,N,K] int64 candidate index into xyz2
    truncate_xyz2: torch.Tensor    # [B,N,K,3] f32


def calculate_corr(fmap1: torch.Tensor, fmap2: torch.Tensor) -> torch.Tensor:
    """model/corr.py:95-100: fmap1^T fmap2 / sqrt(C)."""
    c = fmap1.shape[1]
    corr = torch.matmul(fmap1.transpose(1, 2), fmap2)
    return corr / torch.sqrt(torch.tensor(c).float())


def corr_init(fmap1: torch.Tensor, fmap2: torch.Tensor, xyz2: torch.Tensor, truncate_k: int) -> CorrState:
    """model/corr.py:31-42: per-row top-K of the all-pairs correlation + xyz2 of the K candidates."""
    b, n, _ = xyz2.shape
    top = torch.topk(calculate_corr(fmap1, fmap2), k=truncate_k, dim=2, sorted=True)
    idx = top.indices
    cand = torch.gather(xyz2.unsqueeze(1).expand(b, n, n, 3), 2, idx.unsqueeze(-1).expand(b, n, truncate_k, 3))
    return CorrState(top.values, idx, cand)


def voxel_cube_index(state: CorrState, coords: torch.Tensor, r: float):
    """model/corr.py:52-62.  Returns (cube_idx int64 [B,N,K] with invalid -> 0, valid bool [B,N,K]).

    round() is round-half-to-even; the division is a true fp32 division (corr.py:54).
    """
    q = torch.round((state.truncate_xyz2 - coords.unsqueeze(-2)) / r)
    valid = (torch.abs(q) <= math.floor(RESOLUTION / 2)).all(dim=-1)
    q = q + 1.0
    cube = q[..., 0] * (RESOLUTION ** 2) + q[..., 1] * RESOLUTION + q[..., 2]
    return cube.to(torch.int64) * valid, valid


def voxel_means(state: CorrState, coords: torch.Tensor, num_levels: int, base_scale: float) -> torch.Tensor:
    """model/corr.py:47-71 up to (not incl.) out_conv -> [B, num_levels*27, N].

    Per level: mean correlation of the candidates falling in each of the 27 cells
    (scatter_add of values / clamp(scatter_add of ones, 1, N)); channel = level*27 + cell.
    The reference's zero-pad "repair" (corr.py:67-69) is equivalent to always using 27 bins.
    """
    b, n, _ = coords.shape
    cells = RESOLUTION ** 3
    feats = []
    for lvl in range(num_levels):
        r = base_scale * (2 ** lvl)
        cube, valid = voxel_cube_index(state, coords, r)
        w = valid.to(state.truncated_corr.dtype)
        s = torch.zeros(b, n, cells, device=coords.device).scatter_add_(2, cube, state.truncated_corr * w)
        c = torch.zeros(b, n, cells, device=coords.device).scatter_add_(2, cube, w)
        feats.append((s / torch.clamp(c, 1, n)).transpose(1, 2))
    return torch.cat(feats, dim=1).contiguous()


def voxel_feature(P: Params, state: CorrState, coords: torch.Tensor, num_levels: int, base_scale: float,
                  prefix: str = 'corr_block') -> torch.Tensor:
    """model/corr.py:47-73 -> [B,64,N]  (out_conv = Conv1d 81->128, GN, PReLU, Conv1d 128->64)."""
    x = voxel_means(state, coords, num_levels, base_scale)
    x = pointwise_linear(x, P[prefix + '.out_conv.0.weight'], P[prefix + '.out_conv.0.bias'])
    x = prelu(group_norm(x, P[prefix + '.out_conv.1.weight'], P[prefix + '.out_conv.1.bias']),
              P[prefix + '.out_conv.2.weight'])
    return pointwise_linear(x, P[prefix + '.out_conv.3.weight'], P[prefix + '.out_conv.3.bias'])


def knn_sqdist(state: CorrState, coords: torch.Tensor) -> torch.Tensor:
    """model/corr.py:78-79: (dx*dx + dy*dy) + dz*dz, each op rounded to fp32 (no FMA)."""
    d = state.truncate_xyz2 - coords.unsqueeze(2)
    return (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]


def knn_select(state: CorrState, coords: torch.Tensor, knn: int = KNN) -> torch.Tensor:
    """model/corr.py:81: slots (0..K-1) of the knn nearest candidates, [B,N,knn] int64."""
    return torch.topk(-knn_sqdist(state, coords), k=knn, dim=2).indices


def knn_gather(state: CorrState, coords: torch.Tensor, slots: torch.Tensor) -> torch.Tensor:
    """model/corr.py:84-91 -> [B,4,N,knn] = (corr, dx, dy, dz) of the selected candidates."""
    b, n, k = slots.shape
    kc = torch.gather(state.truncated_corr, 2, slots).unsqueeze(1)
    kx = torch.gather(state.truncate_xyz2, 2, slots.unsqueeze(-1).expand(b, n, k, 3))
    kx = kx.permute(0, 3, 1, 2) - coords.transpose(1, 2).unsqueeze(-1)
    return torch.cat([kc, kx], dim=1)


def knn_feature(P: Params, state: CorrState, coords: torch.Tensor, knn: int = KNN,
                prefix: str = 'corr_block') -> torch.Tensor:
    """model/corr.py:75-93 -> [B,64,N]."""
    x = knn_gather(state, coords, knn_select(state, coords, knn))
    x = pointwise_linear(x, P[prefix + '.knn_conv.0.weight'], P[prefix + '.knn_conv.0.bias'])
    x = prelu(group_norm(x, P[prefix + '.knn_conv.1.weight'], P[prefix + '.knn_conv.1.bias']),
              P[prefix + '.knn_conv.2.weight'])
    x = x.max(dim=3).values
    return pointwise_linear(x, P[prefix + '.knn_out.weight'], P[prefix + '.knn_out.bias'])


def corr_lookup(P: Params, state: CorrState, coords: torch.Tensor, num_levels: int, base_scale: float,
                prefix: str = 'corr_block') -> torch.Tensor:
    """CorrBlock.__call__, model/corr.py:44-45."""
    return (voxel_feature(P, state, coords, num_levels, base_scale, prefix)
            + knn_feature(P, state, coords, KNN, prefix))


# --------------------------------------------------------------------------------------
# UpdateBlock  (model/update.py:8-40,57-87)
# --------------------------------------------------------------------------------------
def motion_encoder(P: Params, flow: torch.Tensor, corr: torch.Tensor, prefix: str) -> torch.Tensor:
    """model/update.py:15-21 -> [B,64,N] (61 learned channels ++ the 3 flow channels)."""
    ft = flow.transpose(1, 2)
    cor = torch.relu(pointwise_linear(corr, P[prefix + '.conv_corr.weight'], P[prefix + '.conv_corr.bias']))
    flo = torch.relu(pointwise_linear(ft, P[prefix + '.conv_flow.weight'], P[prefix + '.conv_flow.bias']))
    out = torch.relu(pointwise_linear(torch.cat([cor, flo], 1), P[prefix + '.conv.weight'], P[prefix + '.conv.bias']))
    return torch.cat([out, ft], dim=1)


def conv_gru(P: Params, h: torch.Tensor, x: torch.Tensor, prefix: str) -> torch.Tensor:
    """model/update.py:31-40."""
    hx = torch.cat([h, x], dim=1)
    z = torch.sigmoid(pointwise_linear(hx, P[prefix + '.convz.weight'], P[prefix + '.convz.bias']))
    r = torch.sigmoid(pointwise_linear(hx, P[prefix + '.convr.weight'], P[prefix + '.convr.bias']))
    q = torch.tanh(pointwise_linear(torch.cat([r * h, x], 1), P[prefix + '.convq.weight'], P[prefix + '.convq.bias']))
    return (1 - z) * h + z * q


def flow_head(P: Params, x: torch.Tensor, graph: Graph, prefix: str) -> torch.Tensor:
    """model/update.py:68-72 -> [B,3,N]."""
    a = pointwise_linear(x, P[prefix + '.conv1.weight'], P[prefix + '.conv1.bias'])
    s = set_conv(P, prefix + '.setconv', x.transpose(1, 2), graph).transpose(1, 2)
    y = torch.relu(pointwise_linear(torch.cat([s, a], 1), P[prefix + '.out_conv.0.weight'], P[prefix + '.out_conv.0.bias']))
    return pointwise_linear(y, P[prefix + '.out_conv.2.weight'], P[prefix + '.out_conv.2.bias'])


def update_block(P: Params, net: torch.Tensor, inp: torch.Tensor, corr: torch.Tensor, flow: torch.Tensor,
                 graph: Graph, prefix: str = 'update_block'):
    """model/update.py:82-87 -> (net [B,64,N], delta_flow [B,N,3])."""
    motion = motion_encoder(P, flow, corr, prefix + '.motion_encoder')
    net = conv_gru(P, net, torch.cat([inp, motion], dim=1), prefix + '.gru')
    delta = flow_head(P, net, graph, prefix + '.flow_head').transpose(1, 2).contiguous()
    return net, delta


# --------------------------------------------------------------------------------------
# RAFT loop  (model/RAFTSceneFlow.py:22-50, model/RAFTSceneFlowRefine.py:22-48)
# --------------------------------------------------------------------------------------
class LoopInputs(NamedTuple):
    state: CorrState
    net: torch.Tensor    # [B,64,N]
    inp: torch.Tensor    # [B,64,N]
    graph: Graph         # context graph of pc1 (consumed by the flow head)
    feat_graph: Graph    # feature-extractor graph of pc1 (consumed by the refiner)


def prepare(P: Params, xyz1: torch.Tensor, xyz2: torch.Tensor, truncate_k: int) -> LoopInputs:
    """Everything RSF.forward does before the loop (model/RAFTSceneFlow.py:24-35)."""
    fmap1, g1 = flot_encoder(P, 'feature_extractor', xyz1)
    fmap2, _ = flot_encoder(P, 'feature_extractor', xyz2)
    state = corr_init(fmap1, fmap2, xyz2, truncate_k)
    fct1, gctx = flot_encoder(P, 'context_extractor', xyz1)
    net, inp = torch.split(fct1, [64, 64], dim=1)
    return LoopInputs(state, torch.tanh(net), torch.relu(inp), gctx, g1)


def raft_loop(P: Params, li: LoopInputs, xyz1: torch.Tensor, num_iters: int, num_levels: int,
              base_scale: float, trace: Optional[list] = None) -> List[torch.Tensor]:
    """model/RAFTSceneFlow.py:37-46 -> list of num_iters flow predictions [B,N,3]."""
    coords1, coords2, net = xyz1, xyz1, li.net
    flows = []
    for _ in range(num_iters):
        coords2 = coords2.detach()                                              # RAFTSceneFlow.py:41 (no gradient through the query)
        corr = corr_lookup(P, li.state, coords2, num_levels, base_scale)
        flow = coords2 - coords1
        net, delta = update_block(P, net, li.inp, corr, flow, li.graph)
        if trace is not None:
            trace.append(dict(coords=coords2, corr=corr, net=net, delta=delta))
        coords2 = coords2 + delta
        flows.append(coords2 - coords1)
    return flows


def rsf_forward(P: Params, xyz1: torch.Tensor, xyz2: torch.Tensor, num_iters: int, num_levels: int = 3,
                base_scale: float = 0.25, truncate_k: int = 512) -> List[torch.Tensor]:
    """RSF.forward, model/RAFTSceneFlow.py:22-50."""
    li = prepare(P, xyz1, xyz2, truncate_k)
    return raft_loop(P, li, xyz1, num_iters, num_levels, base_scale)


def rsf_refine_forward(P: Params, xyz1: torch.Tensor, xyz2: torch.Tensor, num_iters: int, num_levels: int = 3,
                       base_scale: float = 0.25, truncate_k: int = 512) -> torch.Tensor:
    """RSF_refine.forward, model/RAFTSceneFlowRefine.py:22-48."""
    li = prepare(P, xyz1, xyz2, truncate_k)
    flows = raft_loop(P, li, xyz1, num_iters, num_levels, base_scale)
    return flot_refine(P, 'refine_block', flows[-1], li.feat_graph)


# --------------------------------------------------------------------------------------
# synthetic inputs shared by tests / bench (SURVEY.md section 8d)
# --------------------------------------------------------------------------------------
def synthetic_clouds(b: int, n: int, seed: int = 1234):
    """pc1 = 10*U[0,1)^3, pc2 = pc1 + 0.1*N(0,1) -- the BASELINE.md synthetic workload."""
    g = torch.Generator().manual_seed(seed)
    pc1 = 10.0 * torch.rand(b, n, 3, generator=g)
    pc2 = pc1 + 0.1 * torch.randn(b, n, 3, generator=g)
    return pc1, pc2


def randomised_affine(P: Params, seed: int, slope: Optional[float] = None) -> Params:
    """A copy of the weights with every GroupNorm (scale, shift) and the two single-slope PReLUs redrawn.

    The default init leaves every GroupNorm at (1, 0) and PReLU at 0.25, which hides sign and bias handling.  Restates
    `tests/golden/make_golden.py:randomise_affine`, in the same parameter order: scales ~ N(0.8, 0.5) (some negative),
    shifts ~ 0.2 N(0, 1), slopes U(0.05, 0.35) -- or `slope` for both PReLUs when given (e.g. negative, or above 1)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, p in P.items():
        p = p.detach().clone()
        if '.gn' in name or 'out_conv.1.' in name or 'knn_conv.1.' in name:
            if name.endswith('weight'):
                p = torch.randn(p.shape, generator=g) * 0.5 + 0.8
            else:
                p = torch.randn(p.shape, generator=g) * 0.2
        if name.endswith('out_conv.2.weight') and p.numel() == 1 or name.endswith('knn_conv.2.weight'):
            p = torch.rand(p.shape, generator=g) * 0.3 + 0.05
            if slope is not None:
                p = torch.full(p.shape, float(slope))
        out[name] = p.to(P[name].dtype)
    return out


def synthetic_state(b: int, n: int, k: int, seed: int = 7, box: float = 3.0, jitter: float = 0.2):
    """Kernel-level state with controllable voxel density (SURVEY.md section 8d).

    xyz2 ~ U[0,box)^3 (box=3 -> most candidates land inside the coarsest 3x3x3 cube, box=10 ->
    sparse); candidate ids are distinct per row (start + j*odd_step mod n, n a power of two, else a
    random permutation prefix); correlations ~ N(20,5) sorted descending; the query `coords` is a
    random xyz2 point + U(-jitter,jitter).  Returns (CorrState, coords [B,N,3], xyz2 [B,N,3])."""
    g = torch.Generator().manual_seed(seed)
    xyz2 = box * torch.rand(b, n, 3, generator=g)
    if n & (n - 1) == 0:
        start = torch.randint(0, n, (b, n, 1), generator=g)
        step = torch.randint(0, n // 2, (b, n, 1), generator=g) * 2 + 1
        idx = (start + torch.arange(k).view(1, 1, k) * step) % n
    else:
        idx = torch.argsort(torch.rand(b, n, n, generator=g), dim=2)[:, :, :k]
    cand = torch.gather(xyz2.unsqueeze(1).expand(b, n, n, 3), 2, idx.unsqueeze(-1).expand(b, n, k, 3))
    pick = torch.randint(0, n, (b, n), generator=g)
    coords = torch.gather(xyz2, 1, pick.unsqueeze(-1).expand(b, n, 3)) + (torch.rand(b, n, 3, generator=g) * 2 - 1) * jitter
    corr = torch.sort(torch.randn(b, n, k, generator=g) * 5 + 20, dim=2, descending=True).values
    return CorrState(corr, idx, cand.contiguous()), coords, xyz2
