"""The oracle itself (CPU): plain-C collate restatement vs the answers of the real reference build (oracle/_ref) stored in
tests/golden/reference_ops.npz, and the torch restatement of the forward vs the committed reference fixtures."""
import numpy as np
import pytest
import torch

from geotransformer_b200.synth import make_pair
from oracle import collate_oracle as co
from oracle import geo_oracle as G
from oracle import ref_vectors as V


def _stack(pair):
    pts = torch.from_numpy(np.concatenate([pair['ref_points'], pair['src_points']]))
    return pts, torch.tensor([len(pair['ref_points']), len(pair['src_points'])])


@pytest.fixture(scope='module')
def reference_digests(golden):
    gold = golden('reference_ops')
    return dict(zip(gold['digest_keys'].tolist(), gold['digests'].tolist()))


@pytest.mark.parametrize('workload,voxel', V.COLLATE_CASES)
def test_c_restatement_matches_reference_build(workload, voxel, reference_digests):
    """three grid subsamplings and a radius search: bit for bit (values AND unordered_map order) what the reference build gave"""
    got = V.collate_chain(co, workload, voxel)
    for k, t in got.items():
        assert V.digest(t) == reference_digests[f'collate.{workload}.{k}'], k


def test_grid_subsample_golden_order(golden):
    """against the committed fixture (reference output), no reference build needed"""
    gold = golden('demo2k')
    pts, lens = _stack(make_pair('demo2k', 0))
    v = 0.05
    for i in range(1, 4):
        pts, lens = co.grid_subsampling(pts, lens, v)
        assert np.array_equal(pts.numpy(), gold[f'points_{i}']) and lens.tolist() == gold[f'lengths_{i}'].tolist()
        v *= 2


def test_rehash_schedule_edge_sizes(reference_digests):
    """clouds whose voxel counts straddle the libstdc++ rehash thresholds (13/14, 29/30, 59/60, 127/128): the reference build's
    points and order"""
    for n in V.REHASH_SIZES:
        assert V.digest(V.rehash_points(co, n)) == reference_digests[f'rehash.{n}'], n


def _forward_vs_fixture(workload, cfg_name, golden, models, allow_tie_permutation=False):
    cfg, sd, _ = models(cfg_name)
    gold = golden(workload)
    pair = make_pair(workload, 0)
    data = G.collate_pair(pair, cfg, gold['neighbor_limits'].tolist())
    for i in range(1, cfg.backbone.num_stages):
        assert np.array_equal(data['points'][i].numpy(), gold[f'points_{i}'])
    for key in ('neighbors', 'subsampling', 'upsampling'):
        for i in range(len(data[key])):
            want = torch.from_numpy(gold[f'{key}_{i}'].astype(np.int64))
            q = data['points'][i + (1 if key == 'subsampling' else 0)]
            s = data['points'][i + (1 if key == 'upsampling' else 0)]
            assert torch.equal(G.canonical_neighbors(q, s, data[key][i]), G.canonical_neighbors(q, s, want))
            data[key][i] = want
    with torch.no_grad():
        out = G.forward(sd, cfg, data)
    assert np.abs(out['ref_feats_c'].numpy() - gold['ref_feats_c']).max() < 1e-5
    if allow_tie_permutation and not np.array_equal(out['ref_node_corr_indices'].numpy(), gold['ref_node_corr_indices']):
        # adjacent coarse scores within an ulp of each other may swap (make_golden.run): same set, permuted only between scores
        # equal to 1e-5 relative; the fine correspondences then come out block-permuted and compare as a set
        from oracle.fixture import corr_rows
        got = list(zip(out['ref_node_corr_indices'].tolist(), out['src_node_corr_indices'].tolist()))
        want = list(zip(gold['ref_node_corr_indices'].tolist(), gold['src_node_corr_indices'].tolist()))
        assert len(got) == len(want) and set(got) == set(want)
        pos = {pr: i for i, pr in enumerate(got)}
        perm = torch.tensor([pos[pr] for pr in want])
        assert torch.allclose(out['node_corr_scores'][perm], out['node_corr_scores'], rtol=1e-5, atol=0)
        ref = {k: torch.from_numpy(gold[k]) for k in ('ref_corr_points', 'src_corr_points', 'corr_scores')}
        assert np.abs(corr_rows(out)[1] - corr_rows(ref)[1]).max() < 1e-5
    else:
        assert np.array_equal(out['ref_node_corr_indices'].numpy(), gold['ref_node_corr_indices'])
        assert np.array_equal(out['ref_corr_points'].numpy(), gold['ref_corr_points'])
    assert np.abs(out['estimated_transform'].numpy() - gold['estimated_transform']).max() < 1e-5
    # ground-truth superpoint correspondences (matching.py:231-315) and the Evaluator (loss.py:95-159)
    assert np.array_equal(out['gt_node_corr_indices'].numpy(), gold['gt_node_corr_indices'])
    assert np.abs(out['gt_node_corr_overlaps'].numpy() - gold['gt_node_corr_overlaps']).max() < 1e-6
    metrics = G.evaluate(cfg, out, data['transform'])
    assert sorted(metrics) == gold['metric_names'].tolist()
    for name, v in zip(gold['metric_names'].tolist(), gold['metric_values']):
        assert abs(float(metrics[name]) - v) < (1e-3 if name == 'RRE' else 1e-5), name


def test_forward_restatement_matches_reference_fixture(golden, models):
    """torch restatement vs the real reference on the ModelNet-shape pair (teacher-forced neighbour tables)"""
    _forward_vs_fixture('modelnet717', 'modelnet', golden, models)


@pytest.mark.parametrize('workload,cfg_name', [('demo2k', '3dmatch'), ('kitti4k', 'kitti')])
def test_forward_restatement_matches_reference_fixture_3dmatch_kitti(workload, cfg_name, golden, models):
    """the same on pair 0 of the 3DMatch-shape and KITTI-shape workloads"""
    _forward_vs_fixture(workload, cfg_name, golden, models, allow_tie_permutation=True)


def test_evaluator_variants_match_reference_fixture(golden, models):
    """the three Evaluator variants (3DMatch / KITTI / ModelNet, loss.py:95-159) of the restatement on the demo pair vs the
    numbers the real reference Evaluators produced on the same outputs"""
    from geotransformer_b200.config import make_cfg
    cfg, sd, _ = models('3dmatch')
    gold = golden('demo2k')
    pair = make_pair('demo2k', 0)
    data = G.collate_pair(pair, cfg, gold['neighbor_limits'].tolist())
    for key in ('neighbors', 'subsampling', 'upsampling'):
        for i in range(len(data[key])):
            data[key][i] = torch.from_numpy(gold[f'{key}_{i}'].astype(np.int64))      # the reference's exact-tie order
    with torch.no_grad():
        out = G.forward(sd, cfg, data)
    assert np.array_equal(out['gt_node_corr_indices'].numpy(), gold['gt_node_corr_indices'])
    for variant, suffix in (('3dmatch', ''), ('kitti', '_kitti'), ('modelnet', '_modelnet')):
        metrics = G.evaluate(make_cfg(variant), out, data['transform'])
        assert sorted(metrics) == gold['metric_names' + suffix].tolist()
        for name, v in zip(gold['metric_names' + suffix].tolist(), gold['metric_values' + suffix]):
            assert abs(float(metrics[name]) - v) < (1e-3 if name == 'RRE' else 1e-5), (variant, name)


def test_calibration_restatement_matches_reference_fixture(golden, models):
    """calibrate_neighbors_stack_mode (utils/data.py:190-217): restatement vs the limits the real reference computed"""
    cfg, _, _ = models('3dmatch')
    keys = ('ref_points', 'src_points', 'ref_feats', 'src_feats', 'transform')
    pairs = [{k: make_pair('demo2k', i)[k] for k in keys} for i in range(3)]
    gold = golden('calibration')
    for thr in (2000, 150):
        assert np.array_equal(G.calibrate_neighbors(pairs, cfg, sample_threshold=thr), gold[f'limits_threshold_{thr}'])


def test_sinkhorn_marginals_property():
    g = torch.Generator().manual_seed(1)
    s = torch.randn(3, 20, 20, generator=g)
    rm, cm = torch.rand(3, 20, generator=g) > 0.2, torch.rand(3, 20, generator=g) > 0.2
    out = G.optimal_transport(torch.tensor(1.0), s, rm, cm, 100).exp()
    rows = out[:, :-1, :].sum(dim=2)
    assert (rows[rm] - 1).abs().max() < 1e-3


def test_procrustes_degenerate_cases():
    src = torch.randn(1, 10, 3)
    T = G.weighted_procrustes(src, src + 1.0, torch.zeros(1, 10))
    assert torch.equal(T[0], torch.eye(4))


@pytest.mark.parametrize('c,n,sigma_d,extent', [(256, 100, 0.2, 2.0), (128, 90, 4.8, 20.0)])
def test_tabulated_structure_embedding_model_vs_oracle(c, n, sigma_d, extent):
    """oracle/gse_table_model.py (the arithmetic of csrc/gse_table.cu: fp64-built table of proj(sinusoid(x)) on a 1/256 grid,
    fp16 forward differences, fp32 lerp) reproduces GeometricStructureEmbedding.forward to ~3e-6: the tabulation error is an
    order of magnitude below the 2e-5 of the split-precision tensor-core kernels it replaces"""
    import math
    from oracle.gse_table_model import structure_embedding_tabulated
    g = torch.Generator().manual_seed(n)
    pts = torch.rand(n, 3, generator=g) * extent
    sd = {'e.embedding.div_term': torch.exp(torch.arange(0, c, 2).float() * (-np.log(10000.0) / c)),
          'e.proj_d.weight': torch.randn(c, c, generator=g) / math.sqrt(c), 'e.proj_d.bias': torch.randn(c, generator=g) * 0.1,
          'e.proj_a.weight': torch.randn(c, c, generator=g) / math.sqrt(c), 'e.proj_a.bias': torch.randn(c, generator=g) * 0.1}
    want = G.structure_embedding(sd, 'e.', pts, sigma_d, 15, 3)
    got = structure_embedding_tabulated(sd, 'e.', pts, sigma_d, 15, 3)
    assert float((got - want).abs().max()) < 1e-5
    coarse = structure_embedding_tabulated(sd, 'e.', pts, sigma_d, 15, 3, inv_step=64)
    assert float((coarse - want).abs().max()) < 5e-5


def test_c_restatement_matches_reference_build_on_adversarial_small_inputs(reference_digests):
    """several ragged clouds per batch, coordinates quantised to a coarse lattice (many points per voxel, exact-distance ties,
    duplicated points), negative coordinates, 1-point clouds: grid_subsampling values AND unordered_map order bit for bit;
    radius_neighbors (self search and the sub-sampled queries against the full support, the 'subsampling' tables of the collate)
    identical rows up to the order inside exact-distance tie groups (std::sort is unstable in both) -- vs the reference build"""
    cases = V.adversarial_cases()
    assert len(cases) == 60
    for c, (lengths, seed, lattice, voxel) in enumerate(cases):
        for k, t in V.adversarial(co, lengths, seed, lattice, voxel).items():
            assert V.digest(t) == reference_digests[f'adversarial.{c}.{k}'], (c, k)


def test_boundary_2_op_restatements_match_the_real_reference(reference_digests):
    """the oracle's pairwise_distance / knn_partition / get_point_to_node_indices / point_to_node_partition /
    ball_query_partition / apply_transform are bit-identical to what geotransformer.modules.ops of the reference returned on the
    same seeded inputs (oracle/ref_vectors.py)"""
    results = V.boundary_2_ops(G)
    assert len(results) == 105
    for k, t in results:
        assert V.digest(t) == reference_digests['ops.' + k], k


def test_restatement_matches_the_real_reference_on_other_pairs(golden, models):
    """the committed full fixtures pin the restatement on pair 0 of each workload; here on further seeded pairs of all three
    models, against the compact fixtures make_golden wrote from the real reference run: collate levels and neighbour tables (up to
    tie order, then the reference's own order is restored), sampled features and matching scores, coarse correspondences (a
    permutation between scores equal to 1e-5 relative allowed), fine correspondences, transform, gt superpoint pairs, all three
    Evaluator variants -- make_golden.run's tolerances"""
    from geotransformer_b200.config import make_cfg
    from oracle import fixture
    for workload, index in (('demo2k', 1), ('demo2k', 2), ('modelnet717', 1), ('modelnet717', 3), ('kitti4k', 1)):
        gold = golden(f'check_{workload}_{index}')
        pair = make_pair(workload, index)
        cfg, sd, _ = models(pair['config'])
        data = G.collate_pair(pair, cfg, gold['neighbor_limits'].tolist())
        assert fixture.apply_reference_tables(data, gold) == [], (workload, index)
        with torch.no_grad():
            out = G.forward(sd, cfg, data)
        metrics = {v: G.evaluate(make_cfg(v), out, data['transform']) for v in fixture.VARIANTS}
        report = fixture.check_outputs(out, metrics, gold)
        assert fixture.deviations(report) == [], (workload, index, report)
