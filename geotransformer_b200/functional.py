"""Thin torch-tensor wrappers over the C ABI (``include/geob200.h``).

PyTorch is used here only for device memory and the current stream; every computation is a hand-written
sm_100a kernel inside ``libgeob200.so``.  All functions require CUDA tensors and raise ``RuntimeError`` otherwise
(there is no CPU path in the product).
"""
import math

import torch

from . import _lib as L

_f32, _i64, _u8, _i32 = torch.float32, torch.int64, torch.uint8, torch.int32

# mode of the structure-embedding contraction (see geob200_gse_embed): 0 fp32 CUDA cores, 1 tcgen05 3xTF32, 2 1xTF32,
# 3 3xFP16 (fp32-accurate like 3xTF32 at half the tensor-pipe time), 4 3xFP16 on CTA pairs,
# 5 tabulated projections (geob200_gse_embed_table: no contraction at all; default -- 6.4x faster than mode 3 and 3x closer to
# the oracle, profiles/r02_gse_table_check.txt).  Mode 5 needs the ``table`` of the weights (``gse_table``; the modules build and
# cache it); the functional ops called WITHOUT a table and without an explicit mode run the tcgen05 contraction (mode 3).
GSE_MODE = int(__import__('os').environ.get('GEOB200_GSE_MODE', '5'))
# tabulation grid of mode 5: step 1 / GSE_TABLE_INV_STEP index units (power of two), distance indices up to GSE_TABLE_D_MAX
# (larger ones are evaluated directly inside the kernel: correct, slow)
GSE_TABLE_INV_STEP = int(__import__('os').environ.get('GEOB200_GSE_TABLE_INV_STEP', '256'))
GSE_TABLE_D_MAX = float(__import__('os').environ.get('GEOB200_GSE_TABLE_D_MAX', '96'))

# Optional per-op CUDA-event timing on the launching stream (bench.py sets EVENTS = {} to collect
# {op name: [(start_event, end_event), ...]}; None = off, zero overhead).
EVENTS = None


class _timed:
    def __init__(self, name):
        self.name = name

    def __enter__(self):
        if EVENTS is not None:
            self.s = torch.cuda.Event(enable_timing=True)
            self.e = torch.cuda.Event(enable_timing=True)
            self.s.record()
        return self

    def __exit__(self, *a):
        if EVENTS is not None:
            self.e.record()
            EVENTS.setdefault(self.name, []).append((self.s, self.e))
        return False


def _f(t, name):
    L.require_cuda(t, name, _f32)
    return t


def _detach(t):
    return t.detach() if t is not None and t.requires_grad else t


# ------------------------------------------------------------------------------------------------ backbone

# KPConv formulation: 'tc' = gather kernel + tcgen05 3xTF32 GEMM (default where the shape allows), 'fused' = single fp32 kernel
KPCONV_MODE = 'tc'


def kpconv(s_feats, q_points, s_points, neighbor_indices, kernel_points, weights, bias, sigma, weights_t=None):
    """weights_t: optional cached (c_out, 15*c_in) transpose of the weights for the tensor-core path"""
    s_feats, weights, bias = _detach(s_feats), _detach(weights), _detach(bias)
    _f(s_feats, 's_feats'); _f(q_points, 'q_points'); _f(s_points, 's_points')
    L.require_cuda(neighbor_indices, 'neighbor_indices', _i64)
    m, h = neighbor_indices.shape
    ns = s_points.shape[0]
    k, cin, cout = weights.shape
    out = torch.empty((m, cout), dtype=_f32, device=s_feats.device)
    lib = L.lib()
    if (KPCONV_MODE == 'tc' and cin % 32 == 0 and cout % 16 == 0 and cout >= 32 and (cout <= 128 or cout % 128 == 0) and m >= 64):
        if weights_t is None:
            weights_t = weights.reshape(k * cin, cout).t().contiguous()
        ws = L.workspace(lib.geob200_kpconv_tc_workspace_bytes(m, ns, cin), s_feats.device, 'kpconv_tc')
        L.check(lib.geob200_kpconv_tc(s_feats.data_ptr(), q_points.data_ptr(), s_points.data_ptr(), neighbor_indices.data_ptr(), m, ns,
                                      h, kernel_points.data_ptr(), k, weights_t.data_ptr(), L.ptr(bias), cin, cout, float(sigma),
                                      out.data_ptr(), ws.data_ptr(), ws.numel(), L.stream_ptr()), 'kpconv_tc')
        return out
    ws = L.workspace(lib.geob200_kpconv_workspace_bytes(ns), s_feats.device, 'kpconv')
    L.check(lib.geob200_kpconv(s_feats.data_ptr(), q_points.data_ptr(), s_points.data_ptr(),
                               neighbor_indices.data_ptr(), m, ns, h, kernel_points.data_ptr(), k,
                               weights.data_ptr(), L.ptr(bias), cin, cout, float(sigma), out.data_ptr(),
                               ws.data_ptr(), ws.numel(), L.stream_ptr()), 'kpconv')
    return out


def linear(x, weight, bias=None, relu=False, out=None):
    """y = x @ weight.T + bias; x may be a column slice of a wider row-major tensor (stride(1) == 1)."""
    x, weight, bias = _detach(x), _detach(weight), _detach(bias)
    if not x.is_cuda or x.dtype != _f32 or x.stride(1) != 1:
        raise RuntimeError('linear: x must be a float32 CUDA tensor with unit inner stride')
    L.require_cuda(weight, 'weight', _f32)
    m, k = x.shape
    n = weight.shape[0]
    if out is None:
        out = torch.empty((m, n), dtype=_f32, device=x.device)
    L.check(L.lib().geob200_linear(x.data_ptr(), x.stride(0), weight.data_ptr(), L.ptr(bias), out.data_ptr(),
                                   out.stride(0), m, n, k, int(relu), L.stream_ptr()), 'linear')
    return out


def group_norm(x, weight, bias, groups, eps=1e-5, negative_slope=None, residual=None):
    x, weight, bias = _detach(x), _detach(weight), _detach(bias)
    _f(x, 'x')
    n, c = x.shape
    lib = L.lib()
    ws = L.workspace(lib.geob200_group_norm_workspace_bytes(n, c, groups, 1), x.device, 'group_norm')
    y = torch.empty_like(x)
    L.check(lib.geob200_group_norm(x.data_ptr(), n, c, groups, weight.data_ptr(), bias.data_ptr(), float(eps),
                                   L.ptr(residual), int(negative_slope is not None),
                                   float(negative_slope or 0.0), y.data_ptr(), ws.data_ptr(), ws.numel(),
                                   L.stream_ptr()), 'group_norm')
    return y


def linear_group_norm(x, weight, bias, gn_weight, gn_bias, groups, eps=1e-5, negative_slope=None, residual=None):
    """UnaryBlock: leaky(GroupNorm(x @ weight.T + bias) + residual); statistics from the GEMM epilogue on the tcgen05 path"""
    x, weight, bias, gn_weight, gn_bias = _detach(x), _detach(weight), _detach(bias), _detach(gn_weight), _detach(gn_bias)
    if not x.is_cuda or x.dtype != _f32 or x.stride(1) != 1:
        raise RuntimeError('linear_group_norm: x must be a float32 CUDA tensor with unit inner stride')
    L.require_cuda(weight, 'weight', _f32)
    m, k = x.shape
    n = weight.shape[0]
    lib = L.lib()
    pre = scratch((m, n), x.device, 'pre_norm')
    y = torch.empty((m, n), dtype=_f32, device=x.device)
    ws = L.workspace(lib.geob200_group_norm_workspace_bytes(m, n, groups, 1), x.device, 'group_norm')
    L.check(lib.geob200_linear_group_norm(x.data_ptr(), x.stride(0), weight.data_ptr(), L.ptr(bias), m, n, k, groups,
                                          gn_weight.data_ptr(), gn_bias.data_ptr(), float(eps), L.ptr(residual),
                                          int(negative_slope is not None), float(negative_slope or 0.0), pre.data_ptr(),
                                          y.data_ptr(), ws.data_ptr(), ws.numel(), L.stream_ptr()), 'linear_group_norm')
    return y


def kpconv_group_norm(s_feats, q_points, s_points, neighbor_indices, kernel_points, weights, bias, sigma, gn_weight, gn_bias, groups,
                      eps=1e-5, negative_slope=0.1, weights_t=None):
    """ConvBlock / conv part of ResidualBlock: leaky(GroupNorm(KPConv(...)))"""
    m, h = neighbor_indices.shape
    k, cin, cout = weights.shape
    if not (KPCONV_MODE == 'tc' and cin % 32 == 0 and cout % 16 == 0 and cout >= 32 and (cout <= 128 or cout % 128 == 0) and m >= 64):
        x = kpconv(s_feats, q_points, s_points, neighbor_indices, kernel_points, weights, bias, sigma, weights_t=weights_t)
        return group_norm(x, gn_weight, gn_bias, groups, eps, negative_slope=negative_slope)
    s_feats, weights, bias, gn_weight, gn_bias = _detach(s_feats), _detach(weights), _detach(bias), _detach(gn_weight), _detach(gn_bias)
    _f(s_feats, 's_feats'); _f(q_points, 'q_points'); _f(s_points, 's_points')
    L.require_cuda(neighbor_indices, 'neighbor_indices', _i64)
    ns = s_points.shape[0]
    dev = s_feats.device
    if weights_t is None:
        weights_t = weights.reshape(k * cin, cout).t().contiguous()
    lib = L.lib()
    pre = scratch((m, cout), dev, 'pre_norm')
    y = torch.empty((m, cout), dtype=_f32, device=dev)
    gws = L.workspace(lib.geob200_group_norm_workspace_bytes(m, cout, groups, 1), dev, 'group_norm')
    ws = L.workspace(lib.geob200_kpconv_tc_workspace_bytes(m, ns, cin), dev, 'kpconv_tc')
    L.check(lib.geob200_kpconv_group_norm(s_feats.data_ptr(), q_points.data_ptr(), s_points.data_ptr(), neighbor_indices.data_ptr(),
                                          m, ns, h, kernel_points.data_ptr(), k, weights_t.data_ptr(), L.ptr(bias), cin, cout,
                                          float(sigma), groups, gn_weight.data_ptr(), gn_bias.data_ptr(), float(eps),
                                          int(negative_slope is not None), float(negative_slope or 0.0), pre.data_ptr(),
                                          y.data_ptr(), gws.data_ptr(), gws.numel(), ws.data_ptr(), ws.numel(), L.stream_ptr()),
            'kpconv_group_norm')
    return y


def _cloud_rows(cloud_rows):
    import ctypes
    return (ctypes.c_int64 * len(cloud_rows))(*[int(r) for r in cloud_rows])


def group_norm_batched(x, weight, bias, groups, cloud_rows, eps=1e-5, negative_slope=None, residual=None):
    """GroupNorm with per-PAIR statistics for rows in stack order [ref_1..ref_B, src_1..src_B] (``cloud_rows``: 2B host ints)"""
    x, weight, bias = _detach(x), _detach(weight), _detach(bias)
    _f(x, 'x')
    n, c = x.shape
    np_ = len(cloud_rows) // 2
    lib = L.lib()
    ws = L.workspace(lib.geob200_group_norm_workspace_bytes(n, c, groups, np_), x.device, 'group_norm')
    y = torch.empty_like(x)
    L.check(lib.geob200_group_norm_batched(x.data_ptr(), n, c, groups, weight.data_ptr(), bias.data_ptr(), float(eps), L.ptr(residual),
                                           int(negative_slope is not None), float(negative_slope or 0.0), y.data_ptr(), ws.data_ptr(),
                                           ws.numel(), L.stream_ptr(), np_, _cloud_rows(cloud_rows)), 'group_norm_batched')
    return y


def linear_group_norm_batched(x, weight, bias, gn_weight, gn_bias, groups, cloud_rows, eps=1e-5, negative_slope=None, residual=None):
    """linear_group_norm with per-pair GroupNorm statistics (see group_norm_batched)"""
    x, weight, bias, gn_weight, gn_bias = _detach(x), _detach(weight), _detach(bias), _detach(gn_weight), _detach(gn_bias)
    m, k = x.shape
    n = weight.shape[0]
    np_ = len(cloud_rows) // 2
    lib = L.lib()
    pre = scratch((m, n), x.device, 'pre_norm')
    y = torch.empty((m, n), dtype=_f32, device=x.device)
    ws = L.workspace(lib.geob200_group_norm_workspace_bytes(m, n, groups, np_), x.device, 'group_norm')
    L.check(lib.geob200_linear_group_norm_batched(x.data_ptr(), x.stride(0), weight.data_ptr(), L.ptr(bias), m, n, k, groups,
                                                  gn_weight.data_ptr(), gn_bias.data_ptr(), float(eps), L.ptr(residual),
                                                  int(negative_slope is not None), float(negative_slope or 0.0), pre.data_ptr(),
                                                  y.data_ptr(), ws.data_ptr(), ws.numel(), L.stream_ptr(), np_, _cloud_rows(cloud_rows)),
            'linear_group_norm_batched')
    return y


def maxpool(x, neighbor_indices):
    x = _detach(x)
    _f(x, 'x'); L.require_cuda(neighbor_indices, 'neighbor_indices', _i64)
    m, h = neighbor_indices.shape
    y = torch.empty((m, x.shape[1]), dtype=_f32, device=x.device)
    L.check(L.lib().geob200_maxpool(x.data_ptr(), neighbor_indices.data_ptr(), m, x.shape[0], h, x.shape[1],
                                    y.data_ptr(), L.stream_ptr()), 'maxpool')
    return y


def upsample_concat(x, upsample_indices, skip=None):
    """[nearest_upsample(x, upsample_indices) | skip]; ``upsample_indices`` (M, H) -- only column 0 is used."""
    x = _detach(x)
    _f(x, 'x')
    if not upsample_indices.is_cuda or upsample_indices.dtype != _i64:
        raise RuntimeError('upsample_indices must be an int64 CUDA tensor')
    m = upsample_indices.shape[0]
    stride = upsample_indices.stride(0) if upsample_indices.ndim == 2 else 1
    c1 = x.shape[1]
    c2 = 0 if skip is None else skip.shape[1]
    y = torch.empty((m, c1 + c2), dtype=_f32, device=x.device)
    L.check(L.lib().geob200_upsample_concat(x.data_ptr(), upsample_indices.data_ptr(), stride, x.shape[0],
                                            L.ptr(skip), m, c1, c2, y.data_ptr(), L.stream_ptr()), 'upsample_concat')
    return y


def nearest_upsample(x, upsample_indices):
    return upsample_concat(x, upsample_indices, None)


# ------------------------------------------------------------------------------------------------ partition

def point_to_node_partition(points, nodes, point_limit, return_count=False):
    _f(points, 'points'); _f(nodes, 'nodes')
    n, m = points.shape[0], nodes.shape[0]
    dev = points.device
    p2n = torch.empty((n,), dtype=_i64, device=dev)
    node_masks = torch.empty((m,), dtype=torch.bool, device=dev)
    node_sizes = torch.empty((m,), dtype=_i32, device=dev)
    knn = torch.empty((m, point_limit), dtype=_i64, device=dev)
    knn_masks = torch.empty((m, point_limit), dtype=torch.bool, device=dev)
    L.check(L.lib().geob200_point_to_node_partition(points.data_ptr(), n, nodes.data_ptr(), m, point_limit,
                                                    p2n.data_ptr(), node_masks.data_ptr(), node_sizes.data_ptr(),
                                                    knn.data_ptr(), knn_masks.data_ptr(), None,
                                                    L.stream_ptr()), 'point_to_node_partition')
    if return_count:
        return p2n, node_sizes.long(), node_masks, knn, knn_masks
    return p2n, node_masks, knn, knn_masks


def knn_partition(points, nodes, k, return_distance=False):
    """reference ``pointcloud_partition.py:35-57``: (n_nodes, k) nearest point indices per node [and their distances]"""
    _f(points, 'points'); _f(nodes, 'nodes')
    n, m = points.shape[0], nodes.shape[0]
    k = min(int(k), n)
    idx = torch.empty((m, k), dtype=_i64, device=points.device)
    d2 = torch.empty((m, k), dtype=_f32, device=points.device) if return_distance else None
    L.check(L.lib().geob200_knn_partition(points.data_ptr(), n, nodes.data_ptr(), m, k, idx.data_ptr(), L.ptr(d2), L.stream_ptr()),
            'knn_partition')
    if return_distance:
        return d2.sqrt_(), idx
    return idx


def pairwise_distance(x, y, normalized=False, channel_first=False):
    """reference ``pairwise_distance.py:4-31`` for 2-D (or batched 3-D) inputs"""
    if channel_first:
        x, y = x.transpose(-1, -2), y.transpose(-1, -2)
    if x.ndim == 3:
        return torch.stack([pairwise_distance(a, b, normalized) for a, b in zip(x, y)])
    x, y = x.contiguous(), y.contiguous()
    _f(x, 'x'); _f(y, 'y')
    if x.ndim != 2 or y.ndim != 2 or x.shape[1] != y.shape[1]:
        raise RuntimeError('pairwise_distance: x (N, C) and y (M, C) expected')
    out = torch.empty((x.shape[0], y.shape[0]), dtype=_f32, device=x.device)
    L.check(L.lib().geob200_pairwise_distance(x.data_ptr(), x.shape[0], y.data_ptr(), y.shape[0], x.shape[1], int(normalized),
                                              out.data_ptr(), L.stream_ptr()), 'pairwise_distance')
    return out


def point_to_node_indices(points, nodes, return_counts=False):
    """reference ``pointcloud_partition.py:9-32`` (get_point_to_node_indices)"""
    _f(points, 'points'); _f(nodes, 'nodes')
    idx = torch.empty((points.shape[0],), dtype=_i64, device=points.device)
    sizes = torch.empty((nodes.shape[0],), dtype=_i32, device=points.device) if return_counts else None
    L.check(L.lib().geob200_point_to_node_indices(points.data_ptr(), points.shape[0], nodes.data_ptr(), nodes.shape[0], idx.data_ptr(),
                                                  L.ptr(sizes), L.stream_ptr()), 'get_point_to_node_indices')
    return (idx, sizes.long()) if return_counts else idx


def apply_transform(points, transform):
    """reference ``ops/transformation.py:7-60`` (points only) for a single (4, 4) transform: Q = P R^T + t"""
    _f(transform, 'transform')
    p = points.reshape(-1, 3).contiguous()
    _f(p, 'points')
    out = torch.empty_like(p)
    L.check(L.lib().geob200_apply_transform(p.data_ptr(), p.shape[0], transform.data_ptr(), out.data_ptr(), L.stream_ptr()),
            'apply_transform')
    return out.reshape(points.shape)


def gather_rows(table, indices):
    """index_select on a zero-padded table: rows with index >= len(table) come back as zeros."""
    table = _detach(table)
    _f(table, 'table'); L.require_cuda(indices, 'indices', _i64)
    c = table.shape[1]
    out = torch.empty((*indices.shape, c), dtype=_f32, device=table.device)
    L.check(L.lib().geob200_gather_rows(table.data_ptr(), table.shape[0], c, indices.data_ptr(), indices.numel(),
                                        out.data_ptr(), L.stream_ptr()), 'gather_rows')
    return out


# ------------------------------------------------------------------------------------------------ transformer

def gse_indices(points, sigma_d, sigma_a, angle_k, out=None):
    """``out``: optional (d, a) contiguous float buffers of n*n and n*n*angle_k elements to write into"""
    _f(points, 'points')
    n = points.shape[0]
    if out is not None:
        d, a = out[0].view(n, n), out[1].view(n, n, angle_k)
    else:
        d = torch.empty((n, n), dtype=_f32, device=points.device)
        a = torch.empty((n, n, angle_k), dtype=_f32, device=points.device)
    factor_a = 180.0 / (sigma_a * math.pi)
    L.check(L.lib().geob200_gse_indices(points.data_ptr(), n, float(sigma_d), float(factor_a), angle_k, d.data_ptr(),
                                        a.data_ptr(), L.stream_ptr()), 'gse_indices')
    return d, a


def gse_indices_batched(points, cloud_rows, sigma_d, sigma_a, angle_k, d_out, a_out):
    """get_embedding_indices of several stacked clouds in ONE launch; d_out (sum n^2,), a_out (sum n^2, angle_k) receive the
    clouds' index arrays one after the other (the layout ``gse_embed_flat`` consumes)"""
    _f(points, 'points')
    factor_a = 180.0 / (sigma_a * math.pi)
    L.check(L.lib().geob200_gse_indices_batched(points.data_ptr(), len(cloud_rows), _cloud_rows(cloud_rows), float(sigma_d), float(factor_a),
                                                angle_k, d_out.data_ptr(), a_out.data_ptr(), L.stream_ptr()), 'gse_indices_batched')
    return d_out, a_out


def scratch(shape, device, tag):
    """View of a grow-only per-(device, stream, tag) float buffer: for big intermediates whose size changes from pair to
    pair (the N x N x C structure embedding), so that the caching allocator never has to cudaMalloc inside the timed loop.
    The result aliases the buffer: it is only valid until the next call with the same tag on the same stream."""
    numel = 1
    for s in shape:
        numel *= int(s)
    key = (device.index if device.index is not None else torch.cuda.current_device(), L.stream_ptr(), tag)
    buf = _SCRATCH.get(key)
    if buf is None or buf.numel() < numel:
        buf = torch.empty(int(numel * 1.3) + 1024, dtype=_f32, device=device)
        _SCRATCH[key] = buf
    return buf[:numel].view(*shape)


_SCRATCH = {}
_ARANGE = {}


def scratch_arange(n, device, tag='arange'):
    """arange(n) int64 from a cached, read-only per-device table (no launch, no allocation in steady state)."""
    key = device.index if device.index is not None else torch.cuda.current_device()
    buf = _ARANGE.get(key)
    if buf is None or buf.numel() < n:
        buf = torch.arange(max(int(n) * 2, 4096), dtype=_i64, device=device)
        torch.cuda.current_stream(device).synchronize()      # other streams may read it right away
        _ARANGE[key] = buf
    return buf[:n]


class GseTable:
    """Tabulated proj_d(sinusoid(x)) / proj_a(sinusoid(x)) (``geob200_gse_table_build``): the device blob and the grid it was
    built on."""
    __slots__ = ('blob', 'channels', 'inv_step', 'd_max', 'a_max')

    def __init__(self, blob, channels, inv_step, d_max, a_max):
        self.blob, self.channels, self.inv_step, self.d_max, self.a_max = blob, channels, inv_step, d_max, a_max


def gse_table(div_term, wd_t, wa_t, bd, ba, sigma_a, inv_step=None, d_max=None):
    """Tabulate the two projections of GeometricStructureEmbedding for the given weights (wd_t / wa_t: transposed nn.Linear
    weights (in, out)).  Angle indices lie in [0, 180 / sigma_a]; distance indices above ``d_max`` fall back to the direct
    evaluation inside ``gse_embed*``.  Returns after the build has COMPLETED, so any stream may use the table."""
    for t, name in ((div_term, 'div_term'), (wd_t, 'wd_t'), (wa_t, 'wa_t'), (bd, 'bd'), (ba, 'ba')):
        L.require_cuda(t, name, _f32)
    c = int(wd_t.shape[0])
    inv_step = GSE_TABLE_INV_STEP if inv_step is None else int(inv_step)
    d_max = GSE_TABLE_D_MAX if d_max is None else float(d_max)
    a_max = 180.0 / float(sigma_a) + 0.25
    lib = L.lib()
    nbytes = lib.geob200_gse_table_bytes(c, inv_step, d_max, a_max)
    if nbytes == 0:
        raise RuntimeError(f'gse_table: bad grid (channels {c}, inv_step {inv_step}, d_max {d_max}, a_max {a_max})')
    blob = torch.empty(nbytes, dtype=_u8, device=wd_t.device)
    L.check(lib.geob200_gse_table_build(div_term.data_ptr(), wd_t.data_ptr(), wa_t.data_ptr(), bd.data_ptr(), ba.data_ptr(), c,
                                        inv_step, d_max, a_max, blob.data_ptr(), nbytes, L.stream_ptr()), 'gse_table_build')
    torch.cuda.current_stream(wd_t.device).synchronize()
    return GseTable(blob, c, inv_step, d_max, a_max)


def _gse_embed_table(d_indices, a_indices, n_rows, div_term, wd, wa, bd, ba, table, out):
    c = wd.shape[0]
    if table is None or table.channels != c:
        raise RuntimeError('gse_embed mode 5 (tabulated projections) needs the GseTable of these weights (functional.gse_table)')
    with _timed('gse_embed'):
        L.check(L.lib().geob200_gse_embed_table(d_indices.data_ptr(), a_indices.data_ptr(), int(n_rows), c, table.blob.data_ptr(),
                                                table.blob.numel(), table.inv_step, table.d_max, table.a_max, div_term.data_ptr(),
                                                wd.data_ptr(), wa.data_ptr(), bd.data_ptr(), ba.data_ptr(), out.data_ptr(),
                                                L.stream_ptr()), 'gse_embed_table')
    return out


def _gse_mode(mode, table):
    """explicit mode wins (mode 5 without a table is an error, raised by ``_gse_embed_table``); the default is GSE_MODE, except
    that the tabulated mode without a table means the caller has none: tensor-core contraction"""
    if mode is not None:
        return mode
    return 3 if (GSE_MODE == 5 and table is None) else GSE_MODE


def gse_embed_flat(d_indices, a_indices, n_rows, div_term, wd, wa, bd, ba, wd_t, wa_t, out, mode=None, table=None):
    """structure embedding of ``n_rows`` (anchor, point) pairs given as flat index arrays -- the (i, j) pairs of SEVERAL clouds
    concatenated (d (n_rows,), a (n_rows, k)) -> out (n_rows, C): one launch for a whole batch of clouds."""
    c = wd.shape[0]
    mode = _gse_mode(mode, table)
    if mode == 5 and c in (128, 256):
        return _gse_embed_table(d_indices, a_indices, n_rows, div_term, wd, wa, bd, ba, table, out)
    if c == 128 and mode != 0:
        mode = 3                     # hidden_dim 128 (KITTI): the 3xFP16 tcgen05 kernel has an N = 128 instantiation
    elif c != 256:
        mode = 0                     # other widths: fp32 CUDA-core kernel
    lib = L.lib()
    ws = L.workspace(lib.geob200_gse_embed_workspace_bytes(1, c), d_indices.device, 'gse')
    with _timed('gse_embed'):
        L.check(lib.geob200_gse_embed_pairs(d_indices.data_ptr(), a_indices.data_ptr(), int(n_rows), c, div_term.data_ptr(),
                                            wd_t.data_ptr(), wa_t.data_ptr(), wd.data_ptr(), wa.data_ptr(), bd.data_ptr(),
                                            ba.data_ptr(), out.data_ptr(), int(mode), ws.data_ptr(), ws.numel(), L.stream_ptr()),
                'gse_embed_pairs')
    return out


def gse_embed(d_indices, a_indices, div_term, wd, wa, bd, ba, wd_t, wa_t, mode=None, out=None, table=None):
    n = d_indices.shape[0]
    c = wd.shape[0]
    mode = _gse_mode(mode, table)
    emb = torch.empty((n, n, c), dtype=_f32, device=d_indices.device) if out is None else out
    if mode == 5 and c in (128, 256):
        return _gse_embed_table(d_indices, a_indices, n * n, div_term, wd, wa, bd, ba, table, emb)
    if c == 128 and mode != 0:
        mode = 3                     # hidden_dim 128 (KITTI): the 3xFP16 tcgen05 kernel has an N = 128 instantiation
    elif c != 256:
        mode = 0                     # other widths: fp32 CUDA-core kernel
    lib = L.lib()
    ws = L.workspace(lib.geob200_gse_embed_workspace_bytes(n, c), d_indices.device, 'gse')
    with _timed('gse_embed'):
        L.check(lib.geob200_gse_embed(d_indices.data_ptr(), a_indices.data_ptr(), n, c, div_term.data_ptr(),
                                      wd_t.data_ptr(), wa_t.data_ptr(), wd.data_ptr(), wa.data_ptr(), bd.data_ptr(),
                                      ba.data_ptr(), emb.data_ptr(), int(mode), ws.data_ptr(), ws.numel(), L.stream_ptr()),
                'gse_embed')
    return emb


def _rows(t, name):
    if not t.is_cuda or t.dtype != _f32 or t.ndim != 2 or t.stride(1) != 1:
        raise RuntimeError(f'{name} must be a 2-D float32 CUDA tensor with unit inner stride')
    return t


def attention(q, k, v, heads, qp=None, qb=None, embed=None, out=None, streaming=True):
    """q, k, v may be column slices of a fused projection buffer (row stride != channels).  streaming=False forces the
    single-kernel path (the only one for channel counts other than 128 / 256)."""
    _rows(q, 'q'); _rows(k, 'k'); _rows(v, 'v')
    n, c = q.shape
    m = k.shape[0]
    if out is None:
        out = torch.empty((n, c), dtype=_f32, device=q.device)
    lib = L.lib()
    ws = L.workspace(lib.geob200_attention_workspace_bytes(n, m, heads), q.device, tag='attention') if streaming else None
    L.check(lib.geob200_attention(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0),
                                  L.ptr(qp), L.ptr(qb), L.ptr(embed), n, m, c, heads, out.data_ptr(), out.stride(0),
                                  L.ptr(ws), 0 if ws is None else ws.numel(), L.stream_ptr()), 'attention')
    return out


def head_project(q, wp_t, bp, heads):
    """qp[n,h,:] = Wp[h*d:(h+1)*d, :]^T q[n,h*d:(h+1)*d]  and  qb[n,h] = q_h . bp_h   (proj_p moved onto q)."""
    _rows(q, 'q')
    n, c = q.shape
    d = c // heads
    qp = torch.empty((n, heads, c), dtype=_f32, device=q.device)
    qb = torch.empty((n, heads), dtype=_f32, device=q.device)
    lib = L.lib()
    # batched over heads: x = q[:, h*d:(h+1)*d] (ldx=row stride, stride d), W' = wp_t[:, h*d:(h+1)*d] (ldw=c, stride d),
    # y = qp[:, h, :] (ldy=heads*c, stride c)
    L.check(lib.geob200_linear_batched(q.data_ptr(), q.stride(0), d, wp_t.data_ptr(), c, d, None, 0, qp.data_ptr(), heads * c, c,
                                       n, c, d, heads, 0, L.stream_ptr()), 'head_project')
    L.check(lib.geob200_head_bias(q.data_ptr(), q.stride(0), bp.data_ptr(), n, c, heads, qb.data_ptr(), L.stream_ptr()), 'head_bias')
    return qp, qb


def add_layernorm(a, b, weight, bias, eps=1e-5, out=None):
    weight, bias = _detach(weight), _detach(bias)
    L.require_cuda(a, 'a', _f32)
    if b is not None:
        L.require_cuda(b, 'b', _f32)
    n, c = a.shape
    y = torch.empty_like(a) if out is None else out
    if not y.is_contiguous():
        raise RuntimeError('add_layernorm: out must be contiguous')
    L.check(L.lib().geob200_add_layernorm(a.data_ptr(), L.ptr(b), weight.data_ptr(), bias.data_ptr(), n, c, float(eps),
                                          y.data_ptr(), L.stream_ptr()), 'add_layernorm')
    return y


def l2_normalize(x):
    _f(x, 'x')
    y = torch.empty_like(x)
    L.check(L.lib().geob200_l2_normalize(x.data_ptr(), x.shape[0], x.shape[1], y.data_ptr(), L.stream_ptr()), 'l2_normalize')
    return y


# ------------------------------------------------------------------------------------------------ matching

def superpoint_matching(ref_feats, src_feats, ref_masks, src_masks, num_correspondences, dual_normalization=True, defer_count=False):
    """reference ``superpoint_matching.py:13-50``.  The number of rows is min(k, #valid ref x #valid src): it is read back
    from the device (one small D2H) unless ``defer_count`` -- then the full-capacity tensors (padding rows: index -1, score 0,
    which ``gather_patches`` turns into empty patches) and the device count are returned and the caller trims later."""
    _f(ref_feats, 'ref_feats'); _f(src_feats, 'src_feats')
    dev = ref_feats.device
    nr, ns, c = ref_feats.shape[0], src_feats.shape[0], ref_feats.shape[1]
    if ref_masks is None:
        ref_masks = torch.ones((nr,), dtype=torch.bool, device=dev)
    if src_masks is None:
        src_masks = torch.ones((ns,), dtype=torch.bool, device=dev)
    lib = L.lib()
    ws = L.workspace(lib.geob200_superpoint_matching_workspace_bytes(nr, ns), dev)
    k = int(num_correspondences)
    ri = torch.empty((k,), dtype=_i64, device=dev)
    si = torch.empty((k,), dtype=_i64, device=dev)
    sc = torch.empty((k,), dtype=_f32, device=dev)
    cnt = torch.empty((1,), dtype=_i32, device=dev)
    L.check(lib.geob200_superpoint_matching(ref_feats.data_ptr(), src_feats.data_ptr(), nr, ns, c, ref_masks.data_ptr(),
                                            src_masks.data_ptr(), k, int(dual_normalization), ri.data_ptr(),
                                            si.data_ptr(), sc.data_ptr(), cnt.data_ptr(), ws.data_ptr(), ws.numel(),
                                            L.stream_ptr()), 'superpoint_matching')
    if defer_count:
        return ri, si, sc, cnt
    kk = int(cnt.item())
    return ri[:kk], si[:kk], sc[:kk]


def gather_patches(corr_indices, node_knn_indices, node_knn_masks, points):
    p, k = corr_indices.shape[0], node_knn_indices.shape[1]
    dev = points.device
    idx = torch.empty((p, k), dtype=_i64, device=dev)
    msk = torch.empty((p, k), dtype=torch.bool, device=dev)
    pts = torch.empty((p, k, 3), dtype=_f32, device=dev)
    L.check(L.lib().geob200_gather_patches(corr_indices.data_ptr(), p, node_knn_indices.data_ptr(),
                                           node_knn_masks.data_ptr(), k, points.data_ptr(), points.shape[0],
                                           idx.data_ptr(), msk.data_ptr(), pts.data_ptr(), L.stream_ptr()), 'gather_patches')
    return idx, msk, pts


def patch_scores(ref_feats, src_feats, ref_knn_indices, src_knn_indices):
    ref_feats, src_feats = _detach(ref_feats), _detach(src_feats)
    p, k = ref_knn_indices.shape
    out = torch.empty((p, k, k), dtype=_f32, device=ref_feats.device)
    L.check(L.lib().geob200_patch_scores(ref_feats.data_ptr(), ref_feats.shape[0], src_feats.data_ptr(),
                                         src_feats.shape[0], ref_feats.shape[1], ref_knn_indices.data_ptr(),
                                         src_knn_indices.data_ptr(), p, k, out.data_ptr(), L.stream_ptr()), 'patch_scores')
    return out


def sinkhorn(scores, row_masks, col_masks, alpha, num_iterations, inf=1e12):
    scores, alpha = _detach(scores), _detach(alpha)
    _f(scores, 'scores')
    p, k, k2 = scores.shape
    if k != k2:
        raise RuntimeError('sinkhorn: the B200 kernel handles square patch score matrices')
    dev = scores.device
    if row_masks is None:
        row_masks = torch.ones((p, k), dtype=torch.bool, device=dev)
    if col_masks is None:
        col_masks = torch.ones((p, k), dtype=torch.bool, device=dev)
    out = torch.empty((p, k + 1, k + 1), dtype=_f32, device=dev)
    L.check(L.lib().geob200_sinkhorn(scores.data_ptr(), row_masks.data_ptr(), col_masks.data_ptr(), alpha.data_ptr(), p, k,
                                     int(num_iterations), float(inf), out.data_ptr(), L.stream_ptr()), 'sinkhorn')
    return out


def local_global_registration(ref_knn_points, src_knn_points, ref_knn_masks, src_knn_masks, score_mat, k, acceptance_radius,
                              mutual, confidence_threshold, correspondence_threshold, num_refinement_steps,
                              return_details=False, defer_count=False, transform_out=None):
    """``defer_count``: no host read-back -- returns the full-capacity correspondence tensors and the device count
    ``(ref_c, src_c, scores, T, n)``; rows ``[:n]`` are valid.  ``transform_out``: (16,) float view to write T into."""
    p, kk = ref_knn_masks.shape
    ld = score_mat.shape[1]
    dev = score_mat.device
    lib = L.lib()
    cap = p * kk * k * (1 if mutual else 2)
    ref_c = torch.empty((cap, 3), dtype=_f32, device=dev)
    src_c = torch.empty((cap, 3), dtype=_f32, device=dev)
    sc = torch.empty((cap,), dtype=_f32, device=dev)
    cp = torch.empty((cap,), dtype=_i32, device=dev)
    n = torch.empty((1,), dtype=_i32, device=dev)
    T = torch.empty((4, 4), dtype=_f32, device=dev) if transform_out is None else transform_out
    pT = torch.empty((p, 4, 4), dtype=_f32, device=dev)
    pin = torch.empty((p,), dtype=_i32, device=dev)
    best = torch.empty((1,), dtype=_i32, device=dev)
    ws = L.workspace(lib.geob200_lgr_workspace_bytes(p, kk, k), dev)
    L.check(lib.geob200_local_global_registration(
        ref_knn_points.data_ptr(), src_knn_points.data_ptr(), ref_knn_masks.data_ptr(), src_knn_masks.data_ptr(),
        score_mat.data_ptr(), p, kk, ld, k, float(acceptance_radius), int(mutual), float(confidence_threshold),
        int(correspondence_threshold), int(num_refinement_steps), ref_c.data_ptr(), src_c.data_ptr(), sc.data_ptr(),
        cp.data_ptr(), n.data_ptr(), T.data_ptr(), pT.data_ptr(), pin.data_ptr(), best.data_ptr(), ws.data_ptr(),
        ws.numel(), L.stream_ptr()), 'local_global_registration')
    if defer_count:
        return ref_c, src_c, sc, T, n
    c = int(n.item())    # the one D2H of the stage: the number of correspondences sizes the returned tensors
    if return_details:
        return ref_c[:c], src_c[:c], sc[:c], T, dict(corr_patch=cp[:c], patch_transforms=pT, patch_inliers=pin, best=best)
    return ref_c[:c], src_c[:c], sc[:c], T


def weighted_procrustes(src_points, ref_points, weights=None, weight_thresh=0.0, eps=1e-5):
    b, n = src_points.shape[0], src_points.shape[1]
    T = torch.empty((b, 4, 4), dtype=_f32, device=src_points.device)
    L.check(L.lib().geob200_weighted_procrustes(src_points.data_ptr(), ref_points.data_ptr(), L.ptr(weights), b, n,
                                                float(weight_thresh), float(eps), T.data_ptr(), L.stream_ptr()),
            'weighted_procrustes')
    return T


def node_correspondences(ref_nodes, src_nodes, ref_knn_points, src_knn_points, transform, pos_radius, ref_masks=None,
                         src_masks=None, ref_knn_masks=None, src_knn_masks=None):
    """Ground-truth superpoint pairs (reference matching.py:231-315).  Asynchronous: returns full-capacity
    ``(indices (M*N,2), overlaps (M*N,), count (1,) int32)``; rows ``[:count]`` are valid (see ``finish_node_correspondences``)."""
    for t, name in ((ref_nodes, 'ref_nodes'), (src_nodes, 'src_nodes'), (ref_knn_points, 'ref_knn_points'),
                    (src_knn_points, 'src_knn_points'), (transform, 'transform')):
        _f(t, name)
    m, n, k = ref_nodes.shape[0], src_nodes.shape[0], ref_knn_points.shape[1]
    if src_knn_points.shape[1] != k or tuple(transform.shape) != (4, 4):
        raise ValueError('node_correspondences: patches must share K and transform must be (4, 4)')
    for t, shape, name in ((ref_masks, (m,), 'ref_masks'), (src_masks, (n,), 'src_masks'),
                           (ref_knn_masks, (m, k), 'ref_knn_masks'), (src_knn_masks, (n, k), 'src_knn_masks')):
        if t is not None:
            L.require_cuda(t, name, torch.bool)
            if tuple(t.shape) != shape:
                raise ValueError('node_correspondences: %s must have shape %s' % (name, shape))
    dev = ref_nodes.device
    lib = L.lib()
    ws = L.workspace(lib.geob200_node_correspondences_workspace_bytes(m, n, k), dev, tag='node_corr')
    cap = (m * n + 65535) // 65536 * 65536          # rounded: same block sizes from pair to pair (no allocator churn)
    idx = torch.empty((cap, 2), dtype=_i64, device=dev)
    ov = torch.empty((cap,), dtype=_f32, device=dev)
    cnt = torch.empty((1,), dtype=_i32, device=dev)
    L.check(lib.geob200_node_correspondences(ref_nodes.data_ptr(), src_nodes.data_ptr(), ref_knn_points.data_ptr(),
                                             src_knn_points.data_ptr(), L.ptr(ref_masks), L.ptr(src_masks),
                                             L.ptr(ref_knn_masks), L.ptr(src_knn_masks), m, n, k, transform.data_ptr(),
                                             float(pos_radius), idx.data_ptr(), ov.data_ptr(), cnt.data_ptr(), ws.data_ptr(),
                                             ws.numel(), L.stream_ptr()), 'node_correspondences')
    return idx, ov, cnt


def finish_node_correspondences(idx, ov, cnt):
    c = int(cnt.item())
    return idx[:c], ov[:c]


EVAL_MODES = {'3dmatch': 0, 'kitti': 1, 'modelnet': 2}


def evaluate(gt_node_corr_indices, gt_node_corr_overlaps, ref_node_corr_indices, src_node_corr_indices, ref_corr_points,
             src_corr_points, gt_transform, est_transform, src_points, mode, acceptance_overlap, acceptance_radius,
             rmse_threshold=0.0, rre_threshold=0.0, rte_threshold=0.0, out=None, n_gt=None, n_node_corr=None, n_corr=None):
    """Evaluator.forward (reference experiments/<exp>/loss.py:95-159) as one launch; returns a device tensor
    ``[PIR, IR, RRE, RTE, RMSE, RR, #corr, #gt_node_corr]``.  ``n_gt / n_node_corr / n_corr``: optional device int32 counts
    of valid rows when the index / point tensors are full-capacity buffers (no host read-back in between)."""
    dev = est_transform.device
    if out is None:
        out = torch.empty((8,), dtype=_f32, device=dev)
    for t, name in ((ref_corr_points, 'ref_corr_points'), (src_corr_points, 'src_corr_points'), (gt_transform, 'transform'),
                    (est_transform, 'estimated_transform'), (src_points, 'src_points'), (gt_node_corr_overlaps, 'overlaps')):
        _f(t, name)
    for t, name in ((gt_node_corr_indices, 'gt_node_corr_indices'), (ref_node_corr_indices, 'ref_node_corr_indices'),
                    (src_node_corr_indices, 'src_node_corr_indices')):
        L.require_cuda(t, name, _i64)
    L.check(L.lib().geob200_evaluate_counts(gt_node_corr_indices.data_ptr(), gt_node_corr_overlaps.data_ptr(),
                                            gt_node_corr_indices.shape[0], L.ptr(n_gt), float(acceptance_overlap),
                                            ref_node_corr_indices.data_ptr(), src_node_corr_indices.data_ptr(),
                                            ref_node_corr_indices.shape[0], L.ptr(n_node_corr), ref_corr_points.data_ptr(),
                                            src_corr_points.data_ptr(), ref_corr_points.shape[0], L.ptr(n_corr),
                                            float(acceptance_radius), gt_transform.data_ptr(),
                                            est_transform.data_ptr(), src_points.data_ptr(), src_points.shape[0], int(mode),
                                            float(rmse_threshold), float(rre_threshold), float(rte_threshold), out.data_ptr(),
                                            L.stream_ptr()), 'evaluate')
    return out
