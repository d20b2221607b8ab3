"""Batched execution (several pairs per forward, SURVEY.md section 8 f-2): the reference's collate already stacks B pairs as
[ref_1..ref_B, src_1..src_B] (utils/data.py:144) but its model asserts batch_size == 1; here the batched forward must give,
per pair, what the single-pair forward gives (which the other tests pin to the reference)."""
import numpy as np
import pytest
import torch

from geotransformer_b200.model import enable_native
from geotransformer_b200.synth import make_pair
from geotransformer_b200.utils.data import registration_collate_fn_stack_mode
from oracle import geo_oracle as G

pytestmark = pytest.mark.gpu
KEYS = ('ref_points', 'src_points', 'ref_feats', 'src_feats', 'transform')
LIMITS = {'3dmatch': [38, 36, 36, 38], 'modelnet': [13, 21, 27], 'kitti': [27, 75, 147, 157, 119]}


def _pairs(workload, ids):
    return [{k: make_pair(workload, i)[k] for k in KEYS} for i in ids]


def _collate(dicts, cfg, limits):
    b = cfg.backbone
    return registration_collate_fn_stack_mode(dicts, b.num_stages, b.init_voxel_size, b.init_radius, limits)


def _pair_group_norm(x, gamma, beta, groups, cloud_rows, residual=None, slope=None):
    """torch reference: GroupNorm over the stacked (ref, src) rows of every pair separately (modules/kpconv/modules.py:46-50)"""
    B = len(cloud_rows) // 2
    off = np.concatenate([[0], np.cumsum(cloud_rows)])
    y = torch.empty_like(x)
    for p in range(B):
        rows = torch.cat([torch.arange(off[p], off[p + 1]), torch.arange(off[B + p], off[B + p + 1])])
        t = torch.nn.functional.group_norm(x[rows].double().t().unsqueeze(0), groups, gamma.double(), beta.double(), 1e-5)
        y[rows] = t.squeeze(0).t().float()
    if residual is not None:
        y = y + residual
    if slope is not None:
        y = torch.nn.functional.leaky_relu(y, slope)
    return y


@pytest.mark.parametrize('cloud_rows', [(300, 77, 500, 130, 260, 90), (2048, 2048, 2048, 2048), (40, 9, 33, 70), (1000, 129, 127, 1, 640, 383),
                                        (5000, 7000, 6500, 5100), (1434, 700)])
@pytest.mark.parametrize('c', [64, 128, 1024])
def test_group_norm_per_pair_statistics(cloud_rows, c):
    from geotransformer_b200 import functional as GF
    g = torch.Generator().manual_seed(sum(cloud_rows) + c)
    n = sum(cloud_rows)
    x = torch.randn(n, c, generator=g) * torch.linspace(0.5, 3.0, n).unsqueeze(1) + torch.linspace(-1, 1, c)
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g) * 0.1
    res = torch.randn(n, c, generator=g)
    want = _pair_group_norm(x, gamma, beta, 32, cloud_rows, residual=res, slope=0.1)
    got = GF.group_norm_batched(x.cuda(), gamma.cuda(), beta.cuda(), 32, cloud_rows, negative_slope=0.1, residual=res.cuda())
    err = (got.cpu() - want).abs().max().item()
    assert err < 2e-5, f'group_norm_batched: {err:.2e}'
    if len(cloud_rows) == 2:      # a single pair is one segment: the batched entry point is the unbatched one, bit for bit
        assert torch.equal(got, GF.group_norm(x.cuda(), gamma.cuda(), beta.cuda(), 32, negative_slope=0.1, residual=res.cuda()))
    # Linear -> GroupNorm with the statistics from the tcgen05 GEMM epilogue (tile partials folded per pair)
    k = 64
    w, b = torch.randn(c, k, generator=g) / 8.0, torch.randn(c, generator=g) * 0.1
    xin = torch.randn(n, k, generator=g)
    pre = xin.double() @ w.double().t() + b.double()
    want = _pair_group_norm(pre.float(), gamma, beta, 32, cloud_rows, slope=0.1)
    got = GF.linear_group_norm_batched(xin.cuda(), w.cuda(), b.cuda(), gamma.cuda(), beta.cuda(), 32, cloud_rows, negative_slope=0.1)
    err = (got.cpu() - want).abs().max().item()
    assert err < 5e-5, f'linear_group_norm_batched: {err:.2e}'
    if len(cloud_rows) == 2:
        assert torch.equal(got, GF.linear_group_norm(xin.cuda(), w.cuda(), b.cuda(), gamma.cuda(), beta.cuda(), 32, negative_slope=0.1))


@pytest.mark.parametrize('workload,cfg_name,ids', [('demo2k', '3dmatch', (0, 1, 2)), ('modelnet717', 'modelnet', (0, 1, 2, 3)),
                                                   ('kitti4k', 'kitti', (0, 1))])
def test_batched_collate_equals_per_pair(workload, cfg_name, ids, models):
    """stack-mode collate of B pairs == the per-pair collates placed at the cloud offsets (indices shifted, sentinel = stacked rows)"""
    cfg, sd, model = models(cfg_name)
    limits = LIMITS[cfg_name]
    dicts = _pairs(workload, ids)
    B = len(dicts)
    batch = _collate(dicts, cfg, limits)
    singles = [_collate([d], cfg, limits) for d in dicts]
    S = cfg.backbone.num_stages
    for lvl in range(S):
        lens = batch['lengths_host'][lvl]
        assert lens == [s['lengths_host'][lvl][0] for s in singles] + [s['lengths_host'][lvl][1] for s in singles]
        off = np.concatenate([[0], np.cumsum(lens)])
        for p, s in enumerate(singles):
            n_r = s['lengths_host'][lvl][0]
            assert torch.equal(batch['points'][lvl][off[p]:off[p + 1]], s['points'][lvl][:n_r])
            assert torch.equal(batch['points'][lvl][off[B + p]:off[B + p + 1]], s['points'][lvl][n_r:])
    for key, ql, sl in (('neighbors', 0, 0), ('subsampling', 1, 0), ('upsampling', 0, 1)):
        for i, table in enumerate(batch[key]):
            q_lens, s_lens = batch['lengths_host'][i + ql], batch['lengths_host'][i + sl]
            q_off, s_off = np.concatenate([[0], np.cumsum(q_lens)]), np.concatenate([[0], np.cumsum(s_lens)])
            n_s_total = int(s_off[-1])
            for p, s in enumerate(singles):
                one = s[key][i]
                nq_r, ns_r = s['lengths_host'][i + ql][0], s['lengths_host'][i + sl][0]
                ns_pair = sum(s['lengths_host'][i + sl])
                for cloud, rows, shift in ((p, slice(0, nq_r), int(s_off[p])), (B + p, slice(nq_r, None), int(s_off[B + p]) - ns_r)):
                    want = one[rows]
                    want = torch.where(want == ns_pair, torch.full_like(want, n_s_total), want + shift)
                    got = table[q_off[cloud]:q_off[cloud + 1]]
                    w = want.shape[1]
                    assert got.shape[1] >= w, f'{key}[{i}] narrower than the pair table'
                    assert torch.equal(got[:, :w], want), f'{key}[{i}] pair {p} cloud {cloud}'
                    assert bool((got[:, w:] == n_s_total).all())


def test_structure_embedding_indices_of_a_batch_in_one_launch():
    """geob200_gse_indices_batched == the per-cloud launches, bit for bit, clouds of different sizes"""
    from geotransformer_b200 import functional as GF
    g = torch.Generator().manual_seed(4)
    rows = (57, 130, 7, 321, 64, 200)
    pts = torch.rand(sum(rows), 3, generator=g).cuda() * 3.0
    tot = sum(r * r for r in rows)
    d_all, a_all = torch.empty(tot, device='cuda'), torch.empty(tot, 3, device='cuda')
    GF.gse_indices_batched(pts, rows, 0.2, 15, 3, d_all, a_all)
    o, e = 0, 0
    for r in rows:
        d, a = GF.gse_indices(pts[o:o + r].contiguous(), 0.2, 15, 3)
        assert torch.equal(d_all[e:e + r * r].view(r, r), d) and torch.equal(a_all[e:e + r * r].view(r, r, 3), a)
        o, e = o + r, e + r * r


@pytest.mark.parametrize('workload,cfg_name,ids', [('demo2k', '3dmatch', (0, 1, 2)), ('modelnet717', 'modelnet', (0, 1, 2, 3)),
                                                   ('kitti4k', 'kitti', (0, 1)), ('3dmatch20k', '3dmatch', (0, 1))])
def test_forward_batch_equals_single_pair_forward(workload, cfg_name, ids, models):
    cfg, sd, model = models(cfg_name)
    model = model.cuda().eval()
    enable_native(model)
    limits = LIMITS[cfg_name]
    dicts = _pairs(workload, ids)
    singles = [model(_collate([d], cfg, limits)) for d in dicts]
    sides = [torch.cuda.Stream() for _ in range(3)]
    outs = model.forward_batch(_collate(dicts, cfg, limits), side_streams=sides)
    torch.cuda.synchronize()
    assert len(outs) == len(dicts)
    for p, (a, b) in enumerate(zip(outs, singles)):
        for k in ('ref_points_c', 'src_points_c', 'ref_points_f', 'src_points_f', 'ref_points', 'src_points'):
            assert torch.equal(a[k], b[k]), k
        # backbone features: only the order of the GroupNorm sums differs (per-pair fold of tile partials)
        for k in ('ref_feats_f', 'src_feats_f'):
            err = (a[k] - b[k]).abs().max().item() / max(b[k].abs().max().item(), 1.0)
            assert err < 2e-5, f'pair {p} {k}: {err:.2e}'
        for k in ('ref_feats_c', 'src_feats_c'):
            assert (a[k] - b[k]).abs().max().item() < 2e-5, f'pair {p} {k}'
        assert torch.equal(a['gt_node_corr_indices'], b['gt_node_corr_indices'])
        got = set(zip(a['ref_node_corr_indices'].tolist(), a['src_node_corr_indices'].tolist()))
        want = set(zip(b['ref_node_corr_indices'].tolist(), b['src_node_corr_indices'].tolist()))
        assert len(got ^ want) <= max(2, len(want) // 50), f'pair {p}: {len(got ^ want)} coarse correspondences differ'
        if got == want and torch.equal(a['ref_node_corr_indices'], b['ref_node_corr_indices']):
            assert (a['matching_scores'] - b['matching_scores']).abs()[b['matching_scores'] > -1e11].max().item() < 2e-4
            na, nb = a['ref_corr_points'].shape[0], b['ref_corr_points'].shape[0]
            assert abs(na - nb) <= max(2, nb // 200), f'pair {p}: {na} vs {nb} fine correspondences'
            if na == nb and torch.equal(a['ref_corr_points'], b['ref_corr_points']):
                rre, rte = G.registration_error(b['estimated_transform'].cpu().numpy(), a['estimated_transform'].cpu().numpy())
                scale = max(1.0, float(b['ref_points'].abs().max()) / 2.0)
                assert rre < 0.05 and rte < 1e-3 * scale, f'pair {p}: transforms differ by {rre:.4f} deg / {rte:.5f}'


def test_engine_batch_mode_matches_stream_mode(models):
    """RegistrationEngine(batch_size=B): same transforms and metrics as one pair per forward"""
    from geotransformer_b200.engine import RegistrationEngine
    from geotransformer_b200.loss import Evaluator
    cfg, sd, model = models('3dmatch')
    model = model.cuda().eval()
    pairs = _pairs('demo2k', range(7))
    ev = Evaluator(cfg)
    one = RegistrationEngine(model, cfg, cfg.neighbor_limits, num_streams=2, evaluator=ev)
    want = one.register(pairs)
    one.close()
    eng = RegistrationEngine(model, cfg, cfg.neighbor_limits, num_streams=2, evaluator=ev, batch_size=3, side_streams=3)
    got = eng.register(pairs)            # 7 pairs = 3 + 3 + 1: also covers the trailing single pair
    eng.close()
    torch.cuda.synchronize()
    assert len(got) == 7
    for p, (a, b) in enumerate(zip(got, want)):
        assert a['num_superpoints'] == b['num_superpoints']
        if a['num_corr'] == b['num_corr']:
            rre, rte = G.registration_error(b['estimated_transform'].numpy(), a['estimated_transform'].numpy())
            assert rre < 0.05 and rte < 1e-3, f'pair {p}: {rre} deg, {rte}'
            for k in ('PIR', 'IR', 'RMSE', 'RR'):
                x, y = a['metrics'][k], b['metrics'][k]
                assert (np.isnan(x) and np.isnan(y)) or abs(x - y) < 1e-3, (p, k, x, y)
        else:
            assert abs(a['num_corr'] - b['num_corr']) <= max(3, b['num_corr'] // 100), (p, a['num_corr'], b['num_corr'])
