"""Generate golden vectors by running the UNMODIFIED reference (mounted read-only at
/root/reference) on CPU in the build container.  The reference cannot travel to the GPU box,
so the vectors are committed next to this script (tests/golden/*.npz) and this script is the
record of how they were made.

    python tests/golden/make_golden.py            # rewrites tests/golden/*.npz

The only thing added to the reference is a shim for its one absent third-party import,
`torch_scatter.scatter_add` (model/corr.py:50), with torch-scatter's documented semantics
(sum-scatter along `dim`, output width max(index)+1).
"""
import copy
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = os.environ.get('PVRAFT_REFERENCE', '/root/reference')


def install_scatter_shim():
    mod = types.ModuleType('torch_scatter')

    def scatter_add(src, index, dim=-1, out=None, dim_size=None):
        index = index.expand_as(src)
        size = list(src.size())
        size[dim] = dim_size if dim_size is not None else (0 if index.numel() == 0 else int(index.max()) + 1)
        return torch.zeros(size, dtype=src.dtype, device=src.device).scatter_add_(dim, index, src)

    mod.scatter_add = scatter_add
    sys.modules['torch_scatter'] = mod


def np_state(sd):
    return {'w/' + k: v.detach().cpu().numpy() for k, v in sd.items()}


def clouds(b, n, seed):
    g = torch.Generator().manual_seed(seed)
    pc1 = 10.0 * torch.rand(b, n, 3, generator=g)
    pc2 = pc1 + 0.1 * torch.randn(b, n, 3, generator=g)
    return pc1, pc2


def randomise_affine(model, seed):
    """The default init leaves every GroupNorm at (1,0) and PReLU at 0.25, which hides sign and
    bias handling; draw them at random (incl. negative GroupNorm scales) for the golden model."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if ('.gn' in name or 'out_conv.1.' in name or 'knn_conv.1.' in name):
                if name.endswith('weight'):
                    p.copy_(torch.randn(p.shape, generator=g) * 0.5 + 0.8)   # some negative scales
                else:
                    p.copy_(torch.randn(p.shape, generator=g) * 0.2)
            if name.endswith('out_conv.2.weight') and p.numel() == 1 or name.endswith('knn_conv.2.weight'):
                p.copy_(torch.rand(p.shape, generator=g) * 0.3 + 0.05)


def trace_forward(model, pc1, pc2, iters):
    """Re-run RSF.forward's own statements (model/RAFTSceneFlow.py:22-50) keeping intermediates."""
    out = {}
    with torch.no_grad():
        fmap1, graph = model.feature_extractor(pc1)
        fmap2, _ = model.feature_extractor(pc2)
        model.corr_block.init_module(fmap1, fmap2, pc2)
        fct1, gctx = model.context_extractor(pc1)
        net, inp = torch.split(fct1, [64, 64], dim=1)
        net, inp = torch.tanh(net), torch.relu(inp)
        cb = model.corr_block
        out.update(fmap1=fmap1, fmap2=fmap2, fct1=fct1,
                   graph_edges=gctx.edges.reshape(pc1.shape[0], pc1.shape[1], -1),
                   graph_edge_feats=gctx.edge_feats,
                   truncated_corr=cb.truncated_corr, truncate_xyz2=cb.truncate_xyz2)
        coords1, coords2 = pc1, pc1
        for it in range(iters):
            vox = cb.get_voxel_feature(coords2)
            knn = cb.get_knn_feature(coords2)
            corr = cb(coords=coords2)
            flow = coords2 - coords1
            motion = model.update_block.motion_encoder(flow, corr)
            net, delta = model.update_block(net, inp, corr, flow, gctx)
            out[f'it{it}/coords'] = coords2
            out[f'it{it}/voxel_feature'] = vox
            out[f'it{it}/knn_feature'] = knn
            out[f'it{it}/corr'] = corr
            out[f'it{it}/motion'] = motion
            out[f'it{it}/net'] = net
            out[f'it{it}/delta'] = delta
            # index-level goldens for the first level math (model/corr.py:52-62, 78-81)
            if it == 1 or iters == 1:
                for lvl in range(cb.num_levels):
                    r = cb.base_scale * (2 ** lvl)
                    dis = torch.round((cb.truncate_xyz2 - coords2.unsqueeze(-2)) / r)
                    valid = (torch.abs(dis) <= 1).all(dim=-1)
                    dis = dis + 1
                    cube = (dis[..., 0] * 9 + dis[..., 1] * 3 + dis[..., 2]).type(torch.int64) * valid
                    out[f'it{it}/cube_idx_l{lvl}'] = cube.to(torch.int8)
                    out[f'it{it}/valid_l{lvl}'] = valid
                dist = torch.sum((cb.truncate_xyz2 - coords2.view(*coords2.shape[:2], 1, 3)) ** 2, dim=-1)
                out[f'it{it}/knn_dist'] = dist
                out[f'it{it}/knn_slots'] = torch.topk(-dist, k=cb.knn, dim=2).indices.to(torch.int16)
            coords2 = coords2 + delta
            out[f'it{it}/flow'] = coords2 - coords1
    return {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else v) for k, v in out.items()}


def batch_collate():
    """Fixture 5: the reference's collate class (datasets/generic.py:6-66) on three items of 50 points.  Loaded by file path:
    the HuggingFace `datasets` package would shadow the reference's namespace package."""
    import importlib.util
    spec = importlib.util.spec_from_file_location('ref_generic', os.path.join(REF, 'datasets', 'generic.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    g = torch.Generator().manual_seed(0)
    items = [{'sequence': [torch.rand(1, 50, 3, generator=g), torch.rand(1, 50, 3, generator=g)],
              'ground_truth': [(torch.rand(1, 50, 1, generator=g) > 0.2).float(), torch.randn(1, 50, 3, generator=g)]}
             for _ in range(3)]
    out = {}
    for key in ('sequence', 'ground_truth'):
        for ind, t in enumerate(mod.Batch(items).data[key]):
            out[f'batch/{key}{ind}'] = t.numpy()
            for i, it in enumerate(items):
                out[f'item{i}/{key}{ind}'] = it[key][ind].numpy()
    np.savez_compressed(os.path.join(HERE, 'batch_collate.npz'), **out)


def main():
    install_scatter_shim()
    sys.path.insert(0, REF)
    from model.RAFTSceneFlow import RSF
    from model.RAFTSceneFlowRefine import RSF_refine
    from model.pointconv import knn_point
    torch.set_num_threads(8)

    # ---- fixture 1: small, everything kept (B=2, N=256, K=64, 3 iterations) ----------------
    args = types.SimpleNamespace(corr_levels=3, base_scales=0.25, truncate_k=64)
    torch.manual_seed(0)
    model = RSF_refine(args).eval()
    randomise_affine(model, 11)
    pc1, pc2 = clouds(2, 256, 1234)
    tr = trace_forward(model, pc1, pc2, 3)
    with torch.no_grad():
        refined = model([pc1, pc2], 3)
    small = dict(pc1=pc1.numpy(), pc2=pc2.numpy(), refined=refined.numpy(),
                 meta=np.array([2, 256, 64, 3, 3], dtype=np.int64), base_scale=np.float32(0.25))
    small.update(tr)
    small.update(np_state(model.state_dict()))
    np.savez_compressed(os.path.join(HERE, 'small_rsf_refine.npz'), **small)

    # ---- fixture 2: default-init RSF, N=1024, K=512, 4 iters; outputs only -----------------
    args = types.SimpleNamespace(corr_levels=3, base_scales=0.25, truncate_k=512)
    torch.manual_seed(0)
    rsf = RSF(args).eval()
    pc1, pc2 = clouds(1, 1024, 77)
    tr = trace_forward(rsf, pc1, pc2, 4)
    keep = {k: v for k, v in tr.items()
            if k.split('/')[-1] in ('corr', 'net', 'delta', 'flow', 'voxel_feature', 'knn_feature', 'coords')}
    keep['truncated_corr_checksum'] = np.array([tr['truncated_corr'].astype(np.float64).sum(),
                                                np.abs(tr['truncated_corr']).astype(np.float64).sum()])
    keep['knn_slots'] = tr['it1/knn_slots']
    for lvl in range(3):
        keep[f'cube_idx_l{lvl}'] = tr[f'it1/cube_idx_l{lvl}']
    medium = dict(pc1=pc1.numpy(), pc2=pc2.numpy(), meta=np.array([1, 1024, 512, 3, 4], dtype=np.int64),
                  base_scale=np.float32(0.25), seed_note=np.array('torch.manual_seed(0); RSF(args) default init'))
    medium.update(keep)
    np.savez_compressed(os.path.join(HERE, 'medium_rsf.npz'), **medium)

    # ---- fixture 3: non power-of-two base scale + 2 levels (exercises true fp32 division) --
    args = types.SimpleNamespace(corr_levels=2, base_scales=0.3, truncate_k=32)
    torch.manual_seed(3)
    rsf = RSF(args).eval()
    randomise_affine(rsf, 5)
    pc1, pc2 = clouds(1, 128, 99)
    pc1 = pc1 * 0.3
    pc2 = pc2 * 0.3
    tr = trace_forward(rsf, pc1, pc2, 2)
    odd = dict(pc1=pc1.numpy(), pc2=pc2.numpy(), meta=np.array([1, 128, 32, 2, 2], dtype=np.int64),
               base_scale=np.float32(0.3))
    odd.update(tr)
    odd.update(np_state(rsf.state_dict()))
    np.savez_compressed(os.path.join(HERE, 'oddscale_rsf.npz'), **odd)

    # ---- fixture 4: knn_point (model/pointconv.py:28-39) ------------------------------------
    g = torch.Generator().manual_seed(5)
    xyz = torch.rand(2, 300, 3, generator=g) * 4
    q = torch.rand(2, 50, 3, generator=g) * 4
    idx = knn_point(16, xyz, q)
    np.savez_compressed(os.path.join(HERE, 'knn_point.npz'), xyz=xyz.numpy(), query=q.numpy(),
                        idx=np.sort(idx.numpy(), axis=-1).astype(np.int32))
    batch_collate()
    for f in sorted(os.listdir(HERE)):
        if f.endswith('.npz'):
            print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, 'KiB')


if __name__ == '__main__':
    main()
