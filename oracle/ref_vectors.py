"""TEST INFRASTRUCTURE ONLY -- the seeded inputs of the checks that pin the restatements to the reference's own code, and the
stored form of the reference's answers (``tests/golden/reference_ops.npz``, written by ``python -m oracle.make_golden
reference_ops`` where the reference is present).

Every function here takes the implementation as an argument: ``oracle/ref_ext.py`` or ``geotransformer.modules.ops`` of the
reference when the fixture is written, ``oracle/collate_oracle.py`` or ``oracle/geo_oracle.py`` when the tests check against it.
All outputs are stored as SHA-256 digests and compared bit for bit.
"""
import numpy as np
import torch

from geotransformer_b200.synth import make_pair
from oracle import geo_oracle as G
from oracle.fixture import digest

COLLATE_CASES = (('demo2k', 0.05), ('3dmatch20k', 0.05), ('modelnet717', 0.1))
REHASH_SIZES = (1, 2, 12, 13, 14, 28, 29, 30, 58, 59, 60, 126, 127, 128, 129, 257, 258, 542)


def collate_chain(impl, workload, voxel):
    """three grid subsamplings of pair 1 of the workload (voxel doubling), then one radius search on the last level"""
    pair = make_pair(workload, 1)
    pts = torch.from_numpy(np.concatenate([pair['ref_points'], pair['src_points']]))
    lens = torch.tensor([len(pair['ref_points']), len(pair['src_points'])])
    out = {}
    for i in range(1, 4):
        pts, lens = impl.grid_subsampling(pts, lens, voxel)
        out[f'points_{i}'], out[f'lengths_{i}'] = pts, lens
        voxel *= 2
    out['neighbors'] = impl.radius_neighbors(pts, pts, lens, lens, voxel * 1.25)
    return out


def rehash_points(impl, n):
    """one cloud of n points spread so that nearly every point has its own voxel (libstdc++ rehash thresholds)"""
    g = torch.Generator().manual_seed(0)
    for m in REHASH_SIZES:
        pts = torch.rand(m, 3, generator=g) * 100.0
        if m == n:
            return impl.grid_subsampling(pts, torch.tensor([n]), 0.5)[0]
    raise ValueError(n)


def adversarial_cases(n=60):
    """(lengths, seed, lattice, voxel) of the adversarial collate inputs: 1-point clouds and the largest batch first, then
    seeded draws of 1-4 clouds of 1-40 points, lattice step 0 / 0.05 / 0.25 and voxel 0.3 / 0.5 / 1.0"""
    cases = [([1], 0, 0.0, 0.3), ([1, 1, 1, 1], 1, 0.25, 1.0), ([40, 1, 40], 2, 0.05, 0.5), ([40, 40, 40, 40], 3, 0.25, 0.3)]
    g = torch.Generator().manual_seed(60)
    while len(cases) < n:
        k = int(torch.randint(1, 5, (1,), generator=g))
        lengths = torch.randint(1, 41, (k,), generator=g).tolist()
        seed = int(torch.randint(0, 2 ** 31 - 1, (1,), generator=g))
        lattice = (0.0, 0.05, 0.25)[int(torch.randint(0, 3, (1,), generator=g))]
        voxel = (0.3, 0.5, 1.0)[int(torch.randint(0, 3, (1,), generator=g))]
        cases.append((lengths, seed, lattice, voxel))
    return cases


def adversarial(impl, lengths, seed, lattice, voxel):
    """several ragged clouds, coordinates optionally on a coarse lattice (exact-distance ties, duplicated points): grid
    subsampling, the self search and the search of the subsampled points in the full clouds, the neighbour tables in the
    canonical order of ``geo_oracle.canonical_neighbors`` (std::sort orders exact ties arbitrarily)"""
    g = torch.Generator().manual_seed(seed)
    n = sum(lengths)
    pts = (torch.rand(n, 3, generator=g) - 0.5) * 4.0
    if lattice > 0:
        pts = torch.round(pts / lattice) * lattice
    pts = pts.contiguous()
    lens = torch.tensor(lengths)
    a, al = impl.grid_subsampling(pts, lens, voxel)
    r = voxel * 1.5
    na = impl.radius_neighbors(pts, pts, lens, lens, r)
    nq = impl.radius_neighbors(a, pts, al, lens, r)
    return {'points': a, 'lengths': al, 'self': G.canonical_neighbors(pts, pts, na), 'sub': G.canonical_neighbors(a, pts, nq)}


def boundary_2_ops(ops):
    """(label, result) of pairwise_distance / knn_partition / get_point_to_node_indices / point_to_node_partition /
    ball_query_partition / apply_transform of ``ops`` on seeded inputs"""
    res = []
    for seed, n, m in ((0, 500, 40), (1, 64, 64), (2, 2000, 7)):
        g = torch.Generator().manual_seed(seed)
        pts = torch.rand(n, 3, generator=g) * 2.0
        nodes = pts[torch.randperm(n, generator=g)[:m]].contiguous() + 0.01 * torch.randn(m, 3, generator=g)
        feats_a = torch.nn.functional.normalize(torch.randn(m, 32, generator=g), dim=1)
        feats_b = torch.nn.functional.normalize(torch.randn(n, 32, generator=g), dim=1)
        s = f'{seed}_'
        res.append((s + 'pairwise_distance', ops.pairwise_distance(nodes, pts)))
        res.append((s + 'pairwise_distance_normalized', ops.pairwise_distance(feats_a, feats_b, normalized=True)))
        for k in (1, 8, 33):
            kk = min(k, n)
            res.append((s + f'knn_{k}', ops.knn_partition(pts, nodes, kk)))
            d, i = ops.knn_partition(pts, nodes, kk, return_distance=True)
            res += [(s + f'knn_{k}_distance', d), (s + f'knn_{k}_distance_indices', i)]
        res.append((s + 'point_to_node', ops.get_point_to_node_indices(pts, nodes)))
        i, c = ops.get_point_to_node_indices(pts, nodes, return_counts=True)
        res += [(s + 'point_to_node_indices', i), (s + 'point_to_node_counts', c)]
        for limit in (4, 16):
            out = ops.point_to_node_partition(pts, nodes, limit)
            assert len(out) == 4
            res += [(s + f'partition_{limit}_{j}', t) for j, t in enumerate(out)]
            for radius in (0.05, 0.3):
                out = ops.ball_query_partition(pts, nodes, radius, limit, return_count=True)
                res += [(s + f'ball_{limit}_{radius}_{j}', t) for j, t in enumerate(out)]
        T = torch.eye(4)
        q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g))
        T[:3, :3], T[:3, 3] = q, torch.randn(3, generator=g)
        res.append((s + 'apply_transform', ops.apply_transform(pts, T)))
    return res
