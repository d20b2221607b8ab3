"""Every CUDA op of the hot path against the CPU oracle (oracle/geo_oracle.py) on seeded inputs, through the C ABI.
Tolerance: 1e-4 (north star) on fp32 values -- stated per test, usually much tighter; indices bit-exact."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from geotransformer_b200 import functional as GF
from geotransformer_b200.synth import make_pair
from oracle import geo_oracle as G

pytestmark = pytest.mark.gpu


def close(a, b, tol, what=''):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    assert a.shape == b.shape, f'{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}'
    err = (a - b).abs().max().item() if a.numel() else 0.0
    scale = max(b.abs().max().item(), 1.0) if b.numel() else 1.0
    assert err <= tol * scale, f'{what}: max abs err {err:.3e} (scale {scale:.3g}) > {tol:g}'
    return err


@pytest.fixture(scope='module')
def mn(models):
    """ModelNet-shape pair collated by the oracle + deterministic weights."""
    cfg, sd, model = models('modelnet')
    pair = make_pair('modelnet717', 0)
    data = G.collate_pair(pair, cfg, [13, 21, 27])
    return cfg, sd, data


def _cuda_data(data):
    out = {}
    for k, v in data.items():
        if isinstance(v, list):
            out[k] = [x.cuda() if isinstance(x, torch.Tensor) else x for x in v]
        elif isinstance(v, torch.Tensor):
            out[k] = v.cuda()
        else:
            out[k] = v
    return out


@pytest.mark.parametrize('cin,cout,h', [(1, 64, 13), (32, 32, 21), (64, 64, 38), (128, 128, 27), (256, 256, 40)])
def test_kpconv(cin, cout, h):
    g = torch.Generator().manual_seed(cin + h)
    ns, m = 700, 333
    s_pts = torch.rand(ns, 3, generator=g)
    q_pts = s_pts[torch.randperm(ns, generator=g)[:m]] + 0.01 * torch.randn(m, 3, generator=g)
    d = torch.cdist(q_pts, s_pts)
    nbr = d.argsort(dim=1)[:, :h].contiguous()
    nbr[d.gather(1, nbr) > 0.25] = ns                     # shadow neighbours
    feats = torch.randn(ns, cin, generator=g) if cin > 1 else torch.ones(ns, 1)
    sd = {'w.weights': torch.randn(15, cin, cout, generator=g) * 0.1, 'w.bias': torch.randn(cout, generator=g) * 0.1,
          'w.kernel_points': (torch.rand(15, 3, generator=g) - 0.5) * 0.3}
    sd['w.kernel_points'][0] = 0
    want = G.kpconv(sd, 'w.', feats, q_pts, s_pts, nbr, 0.12)
    args = (feats.cuda(), q_pts.cuda(), s_pts.cuda(), nbr.cuda(), sd['w.kernel_points'].cuda(), sd['w.weights'].cuda(),
            sd['w.bias'].cuda(), 0.12)
    old = GF.KPCONV_MODE
    try:
        GF.KPCONV_MODE = 'tc'        # gather kernel + tcgen05 3xTF32 GEMM (K = 15*cin: tensor-core accumulation error grows with K)
        close(GF.kpconv(*args), want, 2e-5 if cin <= 64 else 5e-5, f'kpconv tc {cin}->{cout}')
        GF.KPCONV_MODE = 'fused'     # single fp32 CUDA-core kernel
        close(GF.kpconv(*args), want, 2e-5, f'kpconv fused {cin}->{cout}')
    finally:
        GF.KPCONV_MODE = old


@pytest.mark.parametrize('m,k,n', [(5, 7, 3), (333, 64, 32), (1000, 1536, 512), (4100, 256, 128), (64, 512, 256)])
def test_linear(m, k, n):
    g = torch.Generator().manual_seed(m)
    x, w, b = torch.randn(m, k, generator=g), torch.randn(n, k, generator=g) / math.sqrt(k), torch.randn(n, generator=g)
    tol = 1e-5 if k <= 512 else 2.5e-5     # tensor-core accumulation (see the 3xTF32 test below)
    got = GF.linear(x.cuda(), w.cuda(), b.cuda())
    close(got, F.linear(x, w, b), tol, 'linear')
    got = GF.linear(x.cuda(), w.cuda(), None, relu=True)
    close(got, F.relu(F.linear(x, w)), tol, 'linear relu')


@pytest.mark.parametrize('m,k,n', [(64, 32, 32), (647, 256, 768), (333, 64, 32), (1000, 1536, 512), (40000, 64, 128), (4100, 1024, 256),
                                   (130, 36, 48), (129, 2048, 1024)])
def test_linear_tensor_core_3xtf32_matches_fp32(m, k, n):
    """tcgen05 3xTF32 Linear (default) vs the fp32 CUDA-core kernel and torch: fp32-level agreement"""
    from geotransformer_b200 import _lib
    g = torch.Generator().manual_seed(m + k)
    x, w, b = torch.randn(m, k, generator=g), torch.randn(n, k, generator=g) / math.sqrt(k), torch.randn(n, generator=g)
    want = F.linear(x.double(), w.double(), b.double()).float()
    lib = _lib.lib()
    try:
        lib.geob200_set_linear_mode(1)
        got_tc = GF.linear(x.cuda(), w.cuda(), b.cuda())
        got_tc_relu = GF.linear(x.cuda(), w.cuda(), None, relu=True)
        lib.geob200_set_linear_mode(0)
        got_fp = GF.linear(x.cuda(), w.cuda(), b.cuda())
    finally:
        lib.geob200_set_linear_mode(1)
    # the tensor core accumulates in fp32 with truncation: the error grows ~linearly with K (about 1e-5 relative at K=2048),
    # the fp32 FMA chain of the CUDA-core kernel rounds to nearest (random walk).  Budget of the path: 1e-4.
    tol_tc = 1e-5 if k <= 512 else 2.5e-5
    close(got_fp, want, 1e-5, 'linear fp32')
    close(got_tc, want, tol_tc, 'linear 3xTF32')
    close(got_tc_relu, F.relu(F.linear(x.double(), w.double())).float(), tol_tc, 'linear 3xTF32 relu')


@pytest.mark.parametrize('m,k,n', [(640, 3840, 256), (130, 1920, 128), (3400, 1920, 128), (640, 1024, 256), (64, 512, 32)])
def test_linear_split_k(m, k, n):
    """deep-K GEMMs on few tiles run one CTA per K-slice + a fixed-order reduction: same result as the single-CTA K loop (to
    accumulation-order noise), deterministic, bias / ReLU / strided output applied by the reduction"""
    from geotransformer_b200 import _lib
    g = torch.Generator().manual_seed(m + k)
    x, w, b = torch.randn(m, k, generator=g), torch.randn(n, k, generator=g) / math.sqrt(k), torch.randn(n, generator=g)
    want = F.linear(x.double(), w.double(), b.double()).float()
    lib = _lib.lib()
    cx, cw, cb = x.cuda(), w.cuda(), b.cuda()
    try:
        lib.geob200_set_split_k(0)
        one = GF.linear(cx, cw, cb)
        lib.geob200_set_split_k(1)
        split = GF.linear(cx, cw, cb)
        split2 = GF.linear(cx, cw, cb)
        out = torch.full((m, 2 * n), 3.0, device='cuda')
        GF.linear(cx, cw, cb, relu=True, out=out[:, n:])
    finally:
        lib.geob200_set_split_k(1)
    close(one, want, 2.5e-5, 'single-CTA K loop')
    close(split, want, 2.5e-5, 'split-K')
    assert torch.equal(split, split2)
    close(out[:, n:], F.relu(want), 2.5e-5, 'split-K relu, strided out')
    assert bool((out[:, :n] == 3.0).all())


@pytest.mark.parametrize('m,k,n,groups', [(40000, 64, 128, 32), (40000, 480, 32, 32), (20011, 32, 128, 32), (24000, 64, 256, 32),
                                          (19000, 96, 128, 0)])
def test_linear_persistent_tile_loop(m, k, n, groups):
    """multi-wave GEMMs through the persistent kernel (two TMEM accumulator sets, operand ring running across tiles): bitwise
    the same output and GroupNorm statistics as one CTA per tile"""
    from geotransformer_b200 import _lib
    g = torch.Generator().manual_seed(m + k)
    x, w, b = torch.randn(m, k, generator=g), torch.randn(n, k, generator=g) / math.sqrt(k), torch.randn(n, generator=g)
    gw, gb = torch.rand(n, generator=g) + 0.5, torch.randn(n, generator=g)
    cx, cw, cb, cgw, cgb = x.cuda(), w.cuda(), b.cuda(), gw.cuda(), gb.cuda()
    lib = _lib.lib()

    def run():
        if groups:
            return GF.linear_group_norm(cx, cw, cb, cgw, cgb, groups, negative_slope=0.1)
        return GF.linear(cx, cw, cb, relu=True)
    try:
        lib.geob200_set_linear_persistent(0)
        one = run()
        lib.geob200_set_linear_persistent(1)
        per = run()
        per2 = run()
    finally:
        lib.geob200_set_linear_persistent(1)          # the default
    y = F.linear(x.double(), w.double(), b.double())
    want = F.leaky_relu(F.group_norm(y.t().unsqueeze(0), groups, gw.double(), gb.double(), 1e-5).squeeze(0).t(), 0.1).float() if groups \
        else F.relu(y).float()
    close(one, want, 3e-5, 'one CTA per tile')
    assert torch.equal(per, one), float((per - one).abs().max())
    assert torch.equal(per, per2)


def test_linear_column_slice_input():
    g = torch.Generator().manual_seed(1)
    x, w = torch.randn(50, 256, generator=g), torch.randn(64, 64, generator=g)
    got = GF.linear(x.cuda()[:, 64:128], w.cuda())
    close(got, F.linear(x[:, 64:128], w), 1e-5, 'linear slice')


@pytest.mark.parametrize('n,c', [(1434, 64), (4100, 128), (37, 512), (300, 1024)])
def test_group_norm_variants(n, c):
    g = torch.Generator().manual_seed(n)
    x = torch.randn(n, c, generator=g) * 2 + 0.5
    w, b = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g)
    res = torch.randn(n, c, generator=g)
    ref = F.group_norm(x.t().unsqueeze(0), 32, w, b, 1e-5).squeeze(0).t()
    close(GF.group_norm(x.cuda(), w.cuda(), b.cuda(), 32), ref, 1e-5, 'gn')
    close(GF.group_norm(x.cuda(), w.cuda(), b.cuda(), 32, negative_slope=0.1), F.leaky_relu(ref, 0.1), 1e-5, 'gn+lrelu')
    close(GF.group_norm(x.cuda(), w.cuda(), b.cuda(), 32, negative_slope=0.1, residual=res.cuda()),
          F.leaky_relu(ref + res, 0.1), 1e-5, 'gn+res+lrelu')
    # repeated on the same stream, through the same workspace
    close(GF.group_norm(x.cuda(), w.cuda(), b.cuda(), 32), ref, 1e-5, 'gn again')


@pytest.mark.parametrize('m,k,n,groups', [(4100, 64, 32, 32), (1434, 128, 64, 32), (333, 64, 128, 32), (20011, 32, 128, 32),
                                          (700, 256, 256, 32), (130, 512, 1024, 32), (257, 256, 2048, 32), (640, 64, 512, 8),
                                          (37, 64, 128, 32), (300, 100, 48, 4), (300, 100, 48, 1)])
def test_linear_group_norm_fused_statistics(m, k, n, groups):
    """UnaryBlock as one op: GroupNorm statistics produced by the tcgen05 GEMM epilogue (channels per group 1..64, ragged last
    row tile, several column tiles) against torch; shapes the tensor-core path rejects (groups of 12 or 48 channels) fall back to
    the stand-alone kernels"""
    g = torch.Generator().manual_seed(m + n)
    x = torch.randn(m, k, generator=g)
    w, b = torch.randn(n, k, generator=g) / math.sqrt(k), torch.randn(n, generator=g)
    gw, gb = torch.rand(n, generator=g) + 0.5, torch.randn(n, generator=g)
    res = torch.randn(m, n, generator=g)
    y = F.linear(x.double(), w.double(), b.double())
    ref = F.group_norm(y.t().unsqueeze(0), groups, gw.double(), gb.double(), 1e-5).squeeze(0).t().float()
    c = lambda t: t.cuda()
    tol = 3e-5
    close(GF.linear_group_norm(c(x), c(w), c(b), c(gw), c(gb), groups), ref, tol, 'linear+gn')
    close(GF.linear_group_norm(c(x), c(w), c(b), c(gw), c(gb), groups, negative_slope=0.1, residual=c(res)),
          F.leaky_relu(ref + res, 0.1), tol, 'linear+gn+res+lrelu')
    # interleaved with the stand-alone GroupNorm on the same stream (shared workspace) and repeated: deterministic
    plain = GF.group_norm(GF.linear(c(x), c(w), c(b)), c(gw), c(gb), groups)
    close(plain, ref, tol, 'linear, gn')
    a1 = GF.linear_group_norm(c(x), c(w), c(b), c(gw), c(gb), groups)
    a2 = GF.linear_group_norm(c(x), c(w), c(b), c(gw), c(gb), groups)
    assert torch.equal(a1, a2)
    assert float((a1 - plain).abs().max()) < 2e-5 * float(ref.abs().max())


@pytest.mark.parametrize('cin,cout,h', [(32, 32, 21), (64, 64, 38), (128, 128, 27)])
def test_kpconv_group_norm_fused(cin, cout, h):
    g = torch.Generator().manual_seed(cin + h)
    ns, m = 900, 517
    s_pts = torch.rand(ns, 3, generator=g)
    q_pts = s_pts[torch.randperm(ns, generator=g)[:m]] + 0.01 * torch.randn(m, 3, generator=g)
    d = torch.cdist(q_pts, s_pts)
    nbr = d.argsort(dim=1)[:, :h].contiguous()
    nbr[d.gather(1, nbr) > 0.25] = ns
    feats = torch.randn(ns, cin, generator=g)
    sd = {'w.weights': torch.randn(15, cin, cout, generator=g) * 0.1, 'w.bias': torch.randn(cout, generator=g) * 0.1,
          'w.kernel_points': (torch.rand(15, 3, generator=g) - 0.5) * 0.3}
    sd['w.kernel_points'][0] = 0
    gw, gb = torch.rand(cout, generator=g) + 0.5, torch.randn(cout, generator=g)
    y = G.kpconv(sd, 'w.', feats, q_pts, s_pts, nbr, 0.12)
    want = F.leaky_relu(F.group_norm(y.t().unsqueeze(0), 32, gw, gb, 1e-5).squeeze(0).t(), 0.1)
    args = (feats.cuda(), q_pts.cuda(), s_pts.cuda(), nbr.cuda(), sd['w.kernel_points'].cuda(), sd['w.weights'].cuda(),
            sd['w.bias'].cuda(), 0.12, gw.cuda(), gb.cuda(), 32)
    close(GF.kpconv_group_norm(*args), want, 1e-4, f'kpconv+gn {cin}->{cout}')


def test_maxpool_and_upsample(mn):
    cfg, sd, data = mn
    g = torch.Generator().manual_seed(0)
    x = torch.randn(data['points'][0].shape[0], 64, generator=g)
    close(GF.maxpool(x.cuda(), data['subsampling'][0].cuda()), G.maxpool(x, data['subsampling'][0]), 0, 'maxpool')
    y = torch.randn(data['points'][1].shape[0], 32, generator=g)
    skip = torch.randn(data['points'][0].shape[0], 16, generator=g)
    want = torch.cat([G.nearest_upsample(y, data['upsampling'][0]), skip], dim=1)
    close(GF.upsample_concat(y.cuda(), data['upsampling'][0].cuda(), skip.cuda()), want, 0, 'upsample_concat')


def test_backbone_blocks_modelnet(mn, models):
    """whole KPConv-FPN (15 blocks for S=3) with teacher-forced oracle collate: fine and coarse features"""
    cfg, sd, data = mn
    _, _, model = models('modelnet')
    model = model.cuda()
    with torch.no_grad():
        want = G.backbone(sd, cfg, data['features'], data)
        got = model.backbone(data['features'].cuda(), _cuda_data(data))
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        close(a, b, 1e-4, f'backbone output {i}')


def _tie_aware_index_check(got, want, dist_rows, what, ulp_tol=4):
    """indices must match; a mismatch is tolerated only where the oracle's own two candidate distances are within a few
    ulp of each other (matmul-formula distances, SURVEY.md 'hard parts')."""
    got, want = got.cpu(), want.cpu()
    bad = (got != want).nonzero()
    n_tol = 0
    for idx in bad:
        r = idx[0].item()
        a, b = dist_rows(r, got[tuple(idx)].item()), dist_rows(r, want[tuple(idx)].item())
        assert abs(a - b) <= ulp_tol * np.spacing(np.float32(max(abs(a), abs(b), 1e-30))), f'{what}: row {r} picks {got[tuple(idx)]} vs {want[tuple(idx)]} with distances {a} vs {b}'
        n_tol += 1
    return n_tol


def test_point_to_node_partition(mn):
    cfg, sd, data = mn
    n0 = int(data['lengths'][0][0])
    nc = int(data['lengths'][-1][0])
    pts, nodes = data['points'][0][:n0], data['points'][-1][:nc]
    p2n, masks, knn, knn_masks = G.point_to_node_partition(pts, nodes, 128)
    g_p2n, g_masks, g_knn, g_knn_masks = GF.point_to_node_partition(pts.cuda(), nodes.cuda(), 128)
    sq = G.pairwise_distance(nodes, pts)
    n_tol = _tie_aware_index_check(g_p2n, p2n, lambda r, m: sq[int(m), r].item(), 'point_to_node')
    if n_tol == 0:
        assert torch.equal(g_masks.cpu(), masks)
        assert torch.equal(g_knn_masks.cpu(), knn_masks)
        _tie_aware_index_check(g_knn, knn, lambda r, n: sq[r, int(n)].item() if n < n0 else 1e12, 'node_knn')


def test_point_to_node_partition_crowded_node():
    """a node owning far more points than one selection buffer (the former 4096-point cap): still the exact K nearest"""
    g = torch.Generator().manual_seed(3)
    pts = torch.cat([torch.randn(9000, 3, generator=g) * 0.05, torch.randn(300, 3, generator=g) * 0.05 + 3.0])
    nodes = torch.tensor([[0.0, 0.0, 0.0], [3.0, 3.0, 3.0], [-9.0, 0.0, 0.0]])
    p2n, masks, knn, knn_masks = G.point_to_node_partition(pts, nodes, 64)
    g_p2n, g_sizes, g_masks, g_knn, g_knn_masks = GF.point_to_node_partition(pts.cuda(), nodes.cuda(), 64, return_count=True)
    assert torch.equal(g_p2n.cpu(), p2n) and g_sizes.tolist() == [9000, 300, 0]
    assert torch.equal(g_masks.cpu(), masks) and torch.equal(g_knn_masks.cpu(), knn_masks)
    sq = G.pairwise_distance(nodes, pts)
    _tie_aware_index_check(g_knn, knn, lambda r, n: sq[r, int(n)].item() if n < pts.shape[0] else 1e12, 'node_knn')


@pytest.mark.parametrize('n,m,k', [(717, 41, 16), (9000, 37, 64), (5000, 3, 1500), (50, 7, 64)])
def test_knn_partition_and_ball_query(n, m, k):
    """Boundary 2 ops: knn_partition / ball_query_partition / get_point_to_node_indices / pairwise_distance / apply_transform
    (reference modules/ops/pointcloud_partition.py:9-57,159-175, pairwise_distance.py:4-31, transformation.py:7-60)"""
    from geotransformer_b200.modules import ops
    g = torch.Generator().manual_seed(n + k)
    pts, nodes = torch.rand(n, 3, generator=g) * 2.0, torch.rand(m, 3, generator=g) * 2.0
    sq = G.pairwise_distance(nodes, pts)
    w_d, w_idx = G.knn_partition(pts, nodes, k, return_distance=True)
    g_d, g_idx = ops.knn_partition(pts.cuda(), nodes.cuda(), k, return_distance=True)
    assert g_idx.shape == w_idx.shape == (m, min(k, n))
    _tie_aware_index_check(g_idx, w_idx, lambda r, i: sq[r, int(i)].item(), 'knn_partition')
    close(g_d ** 2, w_d ** 2, 2e-6, 'knn squared distances (matmul form: abs error ~ulp(|x|^2))')
    assert torch.equal(ops.knn_partition(pts.cuda(), nodes.cuda(), k), g_idx)
    # ball query: the mask is a threshold on the distance, compare where the oracle distance is not within float noise of it
    radius = float(w_d.median())
    w_bi, w_bm, w_bc = G.ball_query_partition(pts, nodes, radius, k, return_count=True)
    g_bi, g_bm, g_bc = ops.ball_query_partition(pts.cuda(), nodes.cuda(), radius, k, return_count=True)
    safe = (w_d - radius).abs() > 1e-4
    assert torch.equal(g_bm.cpu()[safe], w_bm[safe])
    same_idx = g_idx.cpu() == w_idx
    assert torch.equal(g_bi.cpu()[safe & same_idx], w_bi[safe & same_idx])
    assert (g_bc.cpu() - w_bc).abs().max() <= int((~safe).sum())
    # get_point_to_node_indices: POINT-first rounding of the matmul form
    w_pi, w_ps = G.get_point_to_node_indices(pts, nodes, return_counts=True)
    g_pi, g_ps = ops.get_point_to_node_indices(pts.cuda(), nodes.cuda(), return_counts=True)
    sq_pn = G.pairwise_distance(pts, nodes)
    n_tol = _tie_aware_index_check(g_pi, w_pi, lambda r, j: sq_pn[r, int(j)].item(), 'get_point_to_node_indices')
    if n_tol == 0:
        assert torch.equal(g_ps.cpu(), w_ps)
    assert torch.equal(ops.get_point_to_node_indices(pts.cuda(), nodes.cuda()), g_pi)
    # pairwise_distance (3-D points and unit features, incl. the normalized and channel_first forms)
    close(ops.pairwise_distance(nodes.cuda(), pts.cuda()), sq, 1e-6, 'pairwise_distance')
    fa, fb = F.normalize(torch.randn(m, 64, generator=g), dim=1), F.normalize(torch.randn(53, 64, generator=g), dim=1)
    close(ops.pairwise_distance(fa.cuda(), fb.cuda(), normalized=True), G.pairwise_distance(fa, fb, normalized=True), 1e-6, 'normalized')
    close(ops.pairwise_distance(fa.t().contiguous().cuda(), fb.t().contiguous().cuda(), channel_first=True), G.pairwise_distance(fa, fb), 2e-6,
          'channel_first')
    # apply_transform
    T = torch.eye(4)
    T[:3, :3] = torch.linalg.qr(torch.randn(3, 3, generator=g))[0]
    T[:3, 3] = torch.randn(3, generator=g)
    close(ops.apply_transform(pts.cuda(), T.cuda()), G.apply_transform(pts, T), 1e-6, 'apply_transform')
    close(ops.apply_transform(pts.reshape(-1, 1, 3).cuda(), T.cuda()).reshape(-1, 3), G.apply_transform(pts, T), 1e-6, 'apply_transform nd')


def test_superpoint_matching_masked_candidates_fewer_than_k():
    """valid_ref x valid_src < k <= n_ref x n_src (ADVICE r1): row count = the masked product, like the reference's
    min(k, masked numel); the deferred-count form pads with index -1 and gather_patches makes those patches empty"""
    g = torch.Generator().manual_seed(5)
    nr, ns, c, k = 40, 30, 256, 256
    fr = F.normalize(torch.randn(nr, c, generator=g), dim=1)
    fs = F.normalize(torch.randn(ns, c, generator=g), dim=1)
    rm, sm = torch.zeros(nr, dtype=torch.bool), torch.zeros(ns, dtype=torch.bool)
    rm[::4], sm[::3] = True, True                     # 10 x 10 = 100 valid pairs < 256 <= 1200
    wr, ws, wsc = G.superpoint_matching(fr, fs, rm, sm, k, True)
    gr, gs, gsc = GF.superpoint_matching(fr.cuda(), fs.cuda(), rm.cuda(), sm.cuda(), k, True)
    assert gr.shape[0] == wr.shape[0] == 100
    assert set(zip(gr.tolist(), gs.tolist())) == set(zip(wr.tolist(), ws.tolist()))
    close(gsc, wsc, 1e-5 * wsc.max().item(), 'scores')
    fr_i, fs_i, fsc, cnt = GF.superpoint_matching(fr.cuda(), fs.cuda(), rm.cuda(), sm.cuda(), k, True, defer_count=True)
    assert int(cnt.item()) == 100 and fr_i.shape[0] == k
    assert bool((fr_i[100:] == -1).all()) and bool((fs_i[100:] == -1).all()) and bool((fsc[100:] == 0).all())
    knn = torch.randint(0, 500, (nr, 64), generator=g).cuda()
    knn_m = (torch.rand(nr, 64, generator=g) > 0.2).cuda()
    pts = torch.rand(500, 3, generator=g).cuda()
    idx, msk, ppts = GF.gather_patches(fr_i, knn, knn_m, pts)
    assert bool((idx[100:] == 500).all()) and not bool(msk[100:].any()) and bool((ppts[100:] == 0).all())
    assert torch.equal(idx[:100], knn[fr_i[:100]]) and torch.equal(msk[:100], knn_m[fr_i[:100]])


def test_gse_indices_and_embedding(mn):
    cfg, sd, data = mn
    nc = int(data['lengths'][-1][0])
    pts = data['points'][-1][:nc]
    g = cfg.geotransformer
    d_want, a_want = G.embedding_indices(pts, g.sigma_d, g.sigma_a, g.angle_k)
    d_got, a_got = GF.gse_indices(pts.cuda(), g.sigma_d, g.sigma_a, g.angle_k)
    close(d_got, d_want, 2e-5, 'd_indices')
    close(a_got, a_want, 2e-5, 'a_indices')
    pre = 'transformer.embedding.'
    want = G.structure_embedding(sd, pre, pts, g.sigma_d, g.sigma_a, g.angle_k)
    wd, wa = sd[pre + 'proj_d.weight'].cuda(), sd[pre + 'proj_a.weight'].cuda()
    got = GF.gse_embed(d_got, a_got, sd[pre + 'embedding.div_term'].cuda(), wd, wa, sd[pre + 'proj_d.bias'].cuda(),
                       sd[pre + 'proj_a.bias'].cuda(), wd.t().contiguous(), wa.t().contiguous(), mode=0)
    close(got, want, 2e-5, 'structure embedding (fp32 path)')


@pytest.mark.parametrize('n', [7, 100, 271])
def test_gse_embedding_tensor_core_modes(n):
    """tcgen05 contraction: 3xTF32 (default) must be fp32-accurate, 1xTF32 within TF32 rounding; vs the oracle"""
    g = torch.Generator().manual_seed(n)
    c = 256
    pts = torch.rand(n, 3, generator=g) * 2.0
    sd = {'e.embedding.div_term': torch.exp(torch.arange(0, c, 2).float() * (-np.log(10000.0) / c)),
          'e.proj_d.weight': torch.randn(c, c, generator=g) / math.sqrt(c), 'e.proj_d.bias': torch.randn(c, generator=g) * 0.1,
          'e.proj_a.weight': torch.randn(c, c, generator=g) / math.sqrt(c), 'e.proj_a.bias': torch.randn(c, generator=g) * 0.1}
    want = G.structure_embedding(sd, 'e.', pts, 0.2, 15, 3)
    d, a = GF.gse_indices(pts.cuda(), 0.2, 15, 3)
    cu = {k: v.cuda() for k, v in sd.items()}
    args = (d, a, cu['e.embedding.div_term'], cu['e.proj_d.weight'], cu['e.proj_a.weight'], cu['e.proj_d.bias'], cu['e.proj_a.bias'],
            cu['e.proj_d.weight'].t().contiguous(), cu['e.proj_a.weight'].t().contiguous())
    close(GF.gse_embed(*args, mode=3), want, 2e-5, 'structure embedding 3xFP16')
    close(GF.gse_embed(*args, mode=4), want, 2e-5, 'structure embedding 3xFP16, CTA-pair multicast')
    close(GF.gse_embed(*args, mode=1), want, 2e-5, 'structure embedding 3xTF32')
    close(GF.gse_embed(*args, mode=2), want, 2e-3, 'structure embedding 1xTF32')
    close(GF.gse_embed(*args, mode=0), want, 2e-5, 'structure embedding fp32')


def test_gse_embedding_fp16_split_is_scale_invariant():
    """the 3xFP16 path pre-scales the weights by a power of two: tiny and huge weights keep fp32-level accuracy"""
    g = torch.Generator().manual_seed(5)
    c, n = 256, 60
    pts = torch.rand(n, 3, generator=g)
    for wscale in (1e-4, 1.0, 300.0):
        sd = {'e.embedding.div_term': torch.exp(torch.arange(0, c, 2).float() * (-np.log(10000.0) / c)),
              'e.proj_d.weight': torch.randn(c, c, generator=g) * wscale, 'e.proj_d.bias': torch.randn(c, generator=g) * wscale,
              'e.proj_a.weight': torch.randn(c, c, generator=g) * wscale, 'e.proj_a.bias': torch.randn(c, generator=g) * wscale}
        want = G.structure_embedding(sd, 'e.', pts, 0.2, 15, 3)
        d, a = GF.gse_indices(pts.cuda(), 0.2, 15, 3)
        cu = {k: v.cuda() for k, v in sd.items()}
        got = GF.gse_embed(d, a, cu['e.embedding.div_term'], cu['e.proj_d.weight'], cu['e.proj_a.weight'], cu['e.proj_d.bias'],
                           cu['e.proj_a.bias'], cu['e.proj_d.weight'].t().contiguous(), cu['e.proj_a.weight'].t().contiguous(), mode=3)
        err = (got.cpu() - want).abs().max().item() / want.abs().max().item()
        assert err < 2e-5, f'weight scale {wscale}: relative error {err:.2e}'


def _gse_case(c, n, extent, seed):
    g = torch.Generator().manual_seed(seed)
    pts = torch.rand(n, 3, generator=g) * extent
    sd = {'e.embedding.div_term': torch.exp(torch.arange(0, c, 2).float() * (-np.log(10000.0) / c)),
          'e.proj_d.weight': torch.randn(c, c, generator=g) / math.sqrt(c), 'e.proj_d.bias': torch.randn(c, generator=g) * 0.1,
          'e.proj_a.weight': torch.randn(c, c, generator=g) / math.sqrt(c), 'e.proj_a.bias': torch.randn(c, generator=g) * 0.1}
    cu = {k: v.cuda() for k, v in sd.items()}
    return pts, sd, cu


def _gse_table(cu, **kw):
    return GF.gse_table(cu['e.embedding.div_term'], cu['e.proj_d.weight'].t().contiguous(), cu['e.proj_a.weight'].t().contiguous(),
                        cu['e.proj_d.bias'], cu['e.proj_a.bias'], 15, **kw)


@pytest.mark.parametrize('c,n,sigma_d,extent', [(256, 7, 0.2, 2.0), (256, 100, 0.2, 2.0), (256, 271, 0.2, 3.0), (128, 40, 4.8, 20.0),
                                                (128, 173, 4.8, 60.0)])
def test_gse_embedding_tabulated_projections(c, n, sigma_d, extent):
    """mode 5 (csrc/gse_table.cu): proj_d / proj_a tabulated over the scalar index, 4 lookups per (i, j) -- vs the oracle.  Also
    with a table that covers only half of the distance range (the rest takes the direct evaluation inside the kernel) and with a
    4x coarser grid (error grows with step^2, still inside the tolerance)."""
    pts, sd, cu = _gse_case(c, n, extent, 100 + n)
    want = G.structure_embedding(sd, 'e.', pts, sigma_d, 15, 3)
    d, a = GF.gse_indices(pts.cuda(), sigma_d, 15, 3)
    args = (d, a, cu['e.embedding.div_term'], cu['e.proj_d.weight'], cu['e.proj_a.weight'], cu['e.proj_d.bias'], cu['e.proj_a.bias'],
            cu['e.proj_d.weight'].t().contiguous(), cu['e.proj_a.weight'].t().contiguous())
    close(GF.gse_embed(*args, mode=5, table=_gse_table(cu)), want, 1e-5, 'structure embedding, tabulated projections')
    close(GF.gse_embed(*args, mode=5, table=_gse_table(cu, d_max=float(d.max()) * 0.5)), want, 2e-5,
          'structure embedding, table covering half of the distance range')
    close(GF.gse_embed(*args, mode=5, table=_gse_table(cu, inv_step=64)), want, 3e-5, 'structure embedding, table step 1/64')
    with pytest.raises(RuntimeError):
        GF.gse_embed(*args, mode=5)                      # no table given


def test_gse_embedding_tabulated_is_scale_invariant():
    """one power-of-two scale per table keeps the fp16 differences in range: tiny and huge weights keep fp32-level accuracy"""
    for wscale in (1e-4, 1.0, 300.0):
        pts, sd, cu = _gse_case(256, 60, 1.0, 5)
        for k in list(sd):
            if 'proj' in k:
                sd[k] = sd[k] * wscale
        cu = {k: v.cuda() for k, v in sd.items()}
        want = G.structure_embedding(sd, 'e.', pts, 0.2, 15, 3)
        d, a = GF.gse_indices(pts.cuda(), 0.2, 15, 3)
        got = GF.gse_embed(d, a, cu['e.embedding.div_term'], cu['e.proj_d.weight'], cu['e.proj_a.weight'], cu['e.proj_d.bias'],
                           cu['e.proj_a.bias'], None, None, mode=5, table=_gse_table(cu))
        err = (got.cpu() - want).abs().max().item() / want.abs().max().item()
        assert err < 1e-5, f'weight scale {wscale}: relative error {err:.2e}'


def test_gse_table_follows_the_weights():
    """GeometricStructureEmbedding.table(): rebuilt when a projection parameter changes in place (load_state_dict)"""
    from geotransformer_b200.modules.geotransformer import GeometricStructureEmbedding
    prev = GF.GSE_MODE
    GF.GSE_MODE = 5
    try:
        torch.manual_seed(3)
        emb = GeometricStructureEmbedding(256, 0.2, 15, 3).cuda()
        pts = torch.rand(50, 3).cuda()
        t1 = emb.table()
        e1 = emb(pts).clone()
        assert emb.table() is t1
        with torch.no_grad():
            emb.proj_a.bias.add_(1.0)
        assert emb.table() is not t1
        close(emb(pts), e1 + 1.0, 2e-6, 'embedding after an in-place bias update')
    finally:
        GF.GSE_MODE = prev


def test_gse_embedding_generic_channels():
    """hidden_dim 128 (KITTI) goes through the generic contraction"""
    g = torch.Generator().manual_seed(9)
    n, c = 40, 128
    pts = torch.rand(n, 3, generator=g) * 20
    sd = {'e.embedding.div_term': torch.exp(torch.arange(0, c, 2).float() * (-np.log(10000.0) / c)),
          'e.proj_d.weight': torch.randn(c, c, generator=g) / math.sqrt(c), 'e.proj_d.bias': torch.randn(c, generator=g) * 0.1,
          'e.proj_a.weight': torch.randn(c, c, generator=g) / math.sqrt(c), 'e.proj_a.bias': torch.randn(c, generator=g) * 0.1}
    want = G.structure_embedding(sd, 'e.', pts, 4.8, 15, 3)
    d, a = GF.gse_indices(pts.cuda(), 4.8, 15, 3)
    cu = {k: v.cuda() for k, v in sd.items()}
    got = GF.gse_embed(d, a, cu['e.embedding.div_term'], cu['e.proj_d.weight'], cu['e.proj_a.weight'], cu['e.proj_d.bias'],
                       cu['e.proj_a.bias'], cu['e.proj_d.weight'].t().contiguous(), cu['e.proj_a.weight'].t().contiguous(), mode=0)
    close(got, want, 2e-5, 'structure embedding C=128')
    # tensor-core path for hidden 128: the 3xFP16 tcgen05 kernel instantiated for N = 128 (two angle + two distance chunks per tile)
    for nn in (40, 173):
        pts = torch.rand(nn, 3, generator=g) * 20
        want = G.structure_embedding(sd, 'e.', pts, 4.8, 15, 3)
        d, a = GF.gse_indices(pts.cuda(), 4.8, 15, 3)
        got = GF.gse_embed(d, a, cu['e.embedding.div_term'], cu['e.proj_d.weight'], cu['e.proj_a.weight'], cu['e.proj_d.bias'],
                           cu['e.proj_a.bias'], cu['e.proj_d.weight'].t().contiguous(), cu['e.proj_a.weight'].t().contiguous(), mode=3)
        close(got, want, 3e-5, f'structure embedding C=128, tcgen05 3xFP16 (n={nn})')


def test_transformer_layers(mn, models):
    cfg, sd, data = mn
    _, _, model = models('modelnet')
    model = model.cuda()
    nc = int(data['lengths'][-1][0])
    pts_r, pts_s = data['points'][-1][:nc], data['points'][-1][nc:]
    g = torch.Generator().manual_seed(4)
    fr, fs = torch.randn(pts_r.shape[0], 512, generator=g), torch.randn(pts_s.shape[0], 512, generator=g)
    taps = {}
    with torch.no_grad():
        want_r, want_s = G.geometric_transformer(sd, cfg, pts_r, pts_s, fr, fs, taps=taps)
        # one self layer and one cross layer in isolation first
        e0 = taps['ref_embeddings']
        x = torch.randn(pts_r.shape[0], 256, generator=g)
        mem = torch.randn(pts_s.shape[0], 256, generator=g)
        lp = 'transformer.transformer.layers.0.'
        w_self = G.rpe_self_layer(sd, lp, x, e0, 4)
        g_self, _ = model.transformer.transformer.layers[0](x.cuda(), x.cuda(), e0.cuda())
        close(g_self, w_self, 2e-5, 'rpe self layer')
        lp = 'transformer.transformer.layers.1.'
        w_cross = G.cross_layer(sd, lp, x, mem, 4)
        g_cross, _ = model.transformer.transformer.layers[1](x.cuda(), mem.cuda())
        close(g_cross, w_cross, 2e-5, 'cross layer')
        got_r, got_s = model.transformer(pts_r.cuda(), pts_s.cuda(), fr.cuda(), fs.cuda())
    close(got_r, want_r, 1e-4, 'transformer ref feats')
    close(got_s, want_s, 1e-4, 'transformer src feats')
    close(GF.l2_normalize(got_r), F.normalize(want_r, p=2, dim=1), 1e-4, 'normalised ref feats')


@pytest.mark.parametrize('n,m,c,h,with_e', [(37, 53, 256, 4, True), (130, 130, 256, 4, True), (64, 201, 128, 4, True),
                                            (33, 65, 256, 4, False), (320, 317, 256, 4, False), (5, 3, 128, 2, True),
                                            (40, 70, 256, 8, True), (19, 23, 64, 4, True), (70, 41, 128, 1, False), (323, 323, 256, 4, True),
                                            (100, 100, 128, 1, True), (48, 16, 128, 2, True)])
def test_attention_paths_vs_torch(n, m, c, h, with_e):
    """softmax((q.k + qp.E + qb)/sqrt(d)) v : streaming (lanes <-> channels) and single-kernel paths against fp64 torch;
    q/k/v are column slices of wider buffers like the fused projections"""
    g = torch.Generator().manual_seed(n * 7 + m)
    d = c // h
    qkv_q = torch.randn(n, 3 * c, generator=g)
    qkv_k = torch.randn(m, 3 * c, generator=g)
    q, k, v = qkv_q[:, :c], qkv_k[:, c:2 * c], qkv_k[:, 2 * c:]
    qp = torch.randn(n, h, c, generator=g) * 0.2 if with_e else None
    qb = torch.randn(n, h, generator=g) if with_e else None
    E = torch.randn(n, m, c, generator=g) if with_e else None
    qd, kd, vd = q.double(), k.double(), v.double()
    s = torch.einsum('nhd,mhd->hnm', qd.view(n, h, d), kd.view(m, h, d))
    if with_e:
        s = s + torch.einsum('nhc,nmc->hnm', qp.double(), E.double()) + qb.double().t()[:, :, None]
    p = torch.softmax(s / math.sqrt(d), dim=-1)
    want = torch.einsum('hnm,mhd->nhd', p, vd.view(m, h, d)).reshape(n, c).float()
    cq, ck = qkv_q.cuda(), qkv_k.cuda()
    args = (cq[:, :c], ck[:, c:2 * c], ck[:, 2 * c:], h)
    kw = dict(qp=None if qp is None else qp.cuda(), qb=None if qb is None else qb.cuda(), embed=None if E is None else E.cuda())
    got_stream = GF.attention(*args, **kw)          # self-attention: TMA-staged E stream (attention_tma.cu); cross: cp.async path
    got_single = GF.attention(*args, streaming=False, **kw)
    close(got_stream, want, 2e-5, 'attention (default path)')
    close(got_single, want, 2e-5, 'attention (single-kernel path)')
    from geotransformer_b200 import _lib as L
    L.lib().geob200_set_attention_tma(0)
    try:
        got_cpasync = GF.attention(*args, **kw)
    finally:
        L.lib().geob200_set_attention_tma(1)
    close(got_cpasync, want, 2e-5, 'attention (lanes<->channels cp.async streaming path)')
    out = torch.full((n, 2 * c), 7.0, device='cuda')                 # strided output, untouched columns stay
    GF.attention(*args, out=out[:, c:], **kw)
    assert torch.equal(out[:, c:], got_stream) and bool((out[:, :c] == 7.0).all())


def test_superpoint_matching_separated_features():
    """well separated unit features: indices and order must match exactly (SURVEY.md: K9 in isolation)"""
    g = torch.Generator().manual_seed(11)
    nr, ns, c = 150, 170, 256
    fr = F.normalize(torch.randn(nr, c, generator=g), dim=1)
    fs = F.normalize(torch.randn(ns, c, generator=g), dim=1)
    rm, sm = torch.rand(nr, generator=g) > 0.1, torch.rand(ns, generator=g) > 0.1
    wr, ws, wsc = G.superpoint_matching(fr, fs, rm, sm, 256, True)
    gr, gs, gsc = GF.superpoint_matching(fr.cuda(), fs.cuda(), rm.cuda(), sm.cuda(), 256, True)
    close(gsc, wsc, 1e-5 / max(wsc.max().item(), 1e-9) * wsc.max().item(), 'corr scores')
    same = (gr.cpu() == wr) & (gs.cpu() == ws)
    # entries may swap only between near-equal scores
    for i in (~same).nonzero().flatten().tolist():
        assert abs(gsc[i].item() - wsc[i].item()) <= 1e-6 * wsc[i].item()
    assert same.float().mean() > 0.98
    assert set(zip(gr.tolist(), gs.tolist())) == set(zip(wr.tolist(), ws.tolist())) or same.float().mean() > 0.98
    # fewer candidates than requested
    wr2, ws2, _ = G.superpoint_matching(fr[:5], fs[:7], None or torch.ones(5, dtype=torch.bool), torch.ones(7, dtype=torch.bool), 256, True)
    gr2, gs2, _ = GF.superpoint_matching(fr[:5].cuda(), fs[:7].cuda(), None, None, 256, True)
    assert gr2.shape[0] == 35 and torch.equal(gr2.cpu(), wr2) and torch.equal(gs2.cpu(), ws2)


@pytest.mark.parametrize('k', [64, 128])
def test_patch_scores_and_sinkhorn(k):
    g = torch.Generator().manual_seed(k)
    p, nf, c = 24, 900, 256
    fr, fs = torch.randn(nf, c, generator=g) * 0.5, torch.randn(nf + 10, c, generator=g) * 0.5
    ri = torch.randint(0, nf + 1, (p, k), generator=g)          # nf = sentinel
    si = torch.randint(0, nf + 11, (p, k), generator=g)
    rm, sm = ri < nf, si < nf + 10
    rm[3] = False                                               # a fully masked patch side
    rpad, spad = torch.cat([fr, torch.zeros(1, c)]), torch.cat([fs, torch.zeros(1, c)])
    want = torch.einsum('bnd,bmd->bnm', rpad[ri], spad[si]) / c ** 0.5
    got = GF.patch_scores(fr.cuda(), fs.cuda(), ri.cuda(), si.cuda())
    close(got, want, 1e-5, 'patch scores')
    alpha = torch.tensor(1.0)
    want_ot = G.optimal_transport(alpha, want, rm, sm, 100)
    got_ot = GF.sinkhorn(got, rm.cuda(), sm.cuda(), alpha.cuda(), 100)
    fin = torch.isfinite(want_ot) & (want_ot > -1e11)
    assert torch.equal(torch.isfinite(got_ot.cpu()) & (got_ot.cpu() > -1e11), fin)
    err = (got_ot.cpu()[fin] - want_ot[fin]).abs().max().item()
    assert err <= 1e-4, f'sinkhorn log-assignment max abs err {err:.3e}'
    # marginals of the valid block: rows of exp(out) sum to ~1 for valid rows (property test, any size)
    pr = got_ot.exp().cpu()
    rows = pr[:, :-1, :].sum(dim=2)
    ok = rm & (sm.sum(dim=1, keepdim=True) > 0)
    assert (rows[ok] - 1).abs().max() < 1e-3


@pytest.mark.parametrize('k', [5, 39, 40, 71, 72, 131, 200])
def test_sinkhorn_kernel_variants(k):
    """register-resident kernels (K+1 <= 40 / 72 / 132) and the generic shared-memory kernel against the oracle"""
    g = torch.Generator().manual_seed(k)
    p = 7
    scores = torch.randn(p, k, k, generator=g) * 3.0
    rm, cm = torch.rand(p, k, generator=g) > 0.2, torch.rand(p, k, generator=g) > 0.2
    rm[:, 0] = True
    cm[:, 0] = True
    rm[2] = False
    alpha = torch.tensor(0.7)
    want = G.optimal_transport(alpha, scores, rm, cm, 100)
    got = GF.sinkhorn(scores.cuda(), rm.cuda(), cm.cuda(), alpha.cuda(), 100).cpu()
    fin = torch.isfinite(want) & (want > -1e11)
    assert torch.equal(torch.isfinite(got) & (got > -1e11), fin)
    err = (got[fin] - want[fin]).abs().max().item()
    assert err <= 1e-4, f'k={k}: sinkhorn log-assignment max abs err {err:.3e}'


def test_weighted_procrustes_and_edge_cases():
    g = torch.Generator().manual_seed(2)
    b, n = 9, 50
    src = torch.randn(b, n, 3, generator=g)
    from geotransformer_b200.synth import _rodrigues
    Rs = torch.stack([torch.from_numpy(_rodrigues(np.random.default_rng(i).normal(size=3), 0.3 * i)).float() for i in range(b)])
    t = torch.randn(b, 3, generator=g)
    ref = src @ Rs.transpose(1, 2) + t[:, None, :] + 0.01 * torch.randn(b, n, 3, generator=g)
    w = torch.rand(b, n, generator=g)
    w[0] = 0                                                   # degenerate: all-zero weights -> identity
    ref[1] = src[1] * torch.tensor([1.0, 1.0, -1.0])           # reflection: det fix must kick in
    want = G.weighted_procrustes(src, ref, w)
    got = GF.weighted_procrustes(src.cuda(), ref.cuda(), w.cuda())
    close(got[0], torch.eye(4), 0, 'zero-weight transform is the identity')
    close(got, want, 1e-4, 'weighted procrustes')
    R = got[:, :3, :3].cpu().double()
    assert (R @ R.transpose(1, 2) - torch.eye(3, dtype=torch.double)).abs().max() < 1e-5      # R in O(3)
    assert (torch.det(R[2:]) - 1).abs().max() < 1e-5                                           # proper rotations


def test_local_global_registration_pipeline(models):
    """LGR on oracle-made assignment matrices: correspondences identical (order too), transform within 1e-4"""
    cfg, sd, model = models('3dmatch')
    g = torch.Generator().manual_seed(8)
    p, k = 40, 64
    from geotransformer_b200.synth import _rodrigues
    R = torch.from_numpy(_rodrigues(np.array([0.3, -0.5, 0.8]), 0.4)).float()
    t = torch.tensor([0.2, -0.1, 0.3])
    src = torch.rand(p, k, 3, generator=g)
    perm = torch.stack([torch.randperm(k, generator=g) for _ in range(p)])
    ref = torch.gather(src, 1, perm[:, :, None].expand(-1, -1, 3)) @ R.t() + t + 0.003 * torch.randn(p, k, 3, generator=g)
    # ref[p,i] corresponds to src[p,perm[p,i]]
    rm, sm = torch.rand(p, k, generator=g) > 0.15, torch.rand(p, k, generator=g) > 0.15
    logits = torch.randn(p, k, k, generator=g) * 0.5
    logits[torch.arange(p)[:, None], torch.arange(k)[None, :], perm] += 6.0
    logits[5] = -3.0 + 0.01 * torch.randn(k, k, generator=g)       # a patch with (almost) no confident matches
    ot = G.optimal_transport(torch.tensor(1.0), logits, rm, sm, 100)
    taps = {}
    w_rc, w_sc, w_cs, w_T = G.local_global_registration(cfg, ref, src, rm, sm, ot[:, :-1, :-1], taps=taps)
    lgr = model.fine_matching
    rc, sc, cs, T, det = lgr(ref.cuda(), src.cuda(), rm.cuda(), sm.cuda(), ot.cuda(), None, return_details=True)
    assert rc.shape == w_rc.shape, f'{rc.shape[0]} correspondences vs {w_rc.shape[0]}'
    close(rc, w_rc, 0, 'ref corr points')
    close(sc, w_sc, 0, 'src corr points')
    close(cs, w_cs, 1e-5, 'corr scores')
    assert torch.equal(det['corr_patch'].cpu().long(), taps['corr_batch_indices'])
    assert int(det['best'].item()) >= 0
    close(T, w_T, 1e-4, 'estimated transform')
    gt = torch.eye(4); gt[:3, :3] = R; gt[:3, 3] = t
    close(T, gt, 5e-3, 'estimated transform vs ground truth')
