"""ctypes mirror of the native stage drivers (``csrc/native.cu``, structs in ``include/geob200.h``).

``NativeModel`` snapshots the parameter pointers of a ``GeoTransformer`` module (plus the derived weight layouts: the
tensor-core KPConv transposes, fused q|k|v and k|v projections, ``proj_p`` transposes) into the C structs and runs the
backbone and the transformer with ONE C call each.  Same kernels, same order as the module path: results are bitwise
identical (tests/test_gpu_native.py); only the host cost changes (~340 Python ops per pair -> ~40).
"""
import ctypes

import torch

from . import _lib as L

MAX_STAGES = 6
P, I64, I32, F32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float


class LinearT(ctypes.Structure):
    _fields_ = [('weight', P), ('bias', P), ('c_in', I64), ('c_out', I64)]


class NormT(ctypes.Structure):
    _fields_ = [('gamma', P), ('beta', P)]


class KPConvT(ctypes.Structure):
    _fields_ = [('weights', P), ('weights_t', P), ('bias', P), ('kernel_points', P), ('c_in', I64), ('c_out', I64), ('sigma', F32)]


class ResBlockT(ctypes.Structure):
    _fields_ = [('has_unary1', I32), ('has_shortcut', I32), ('strided', I32), ('reserved', I32), ('c_in', I64),
                ('unary1', LinearT), ('norm1', NormT), ('conv', KPConvT), ('norm_conv', NormT), ('unary2', LinearT), ('norm2', NormT),
                ('shortcut', LinearT), ('norm_sc', NormT)]


class BackboneT(ctypes.Structure):
    _fields_ = [('num_stages', I32), ('finest_decoder', I32), ('groups', I32), ('init_dim', I32), ('conv1', KPConvT), ('norm1', NormT),
                ('blocks', ResBlockT * (1 + 3 * (MAX_STAGES - 1))), ('decoders', LinearT * MAX_STAGES), ('decoder_norms', NormT * MAX_STAGES)]


class TLayerT(ctypes.Structure):
    _fields_ = [('is_self', I32), ('reserved', I32), ('w_qkv', P), ('b_qkv', P), ('w_q', P), ('b_q', P), ('w_kv', P), ('b_kv', P),
                ('wp_t', P), ('bp', P), ('att_linear', LinearT), ('att_norm', NormT), ('expand', LinearT), ('squeeze', LinearT),
                ('out_norm', NormT)]


def _ptr(t):
    return None if t is None else t.data_ptr()


class NativeModel:
    """Holds the C descriptors of one model on one device.  Rebuild it if parameters are re-assigned (pointers are snapshotted)."""

    def __init__(self, model):
        self.model = model
        self._keep = []                     # derived tensors must outlive the structs
        self.device = next(model.parameters()).device
        self.backbone = self._build_backbone(model.backbone)
        self.layers, self.num_layers = self._build_transformer(model.transformer.transformer)
        self.hidden = model.transformer.in_proj.out_features
        self.heads = model.transformer.transformer.layers[0].attention.attention.num_heads

    # -- descriptors ---------------------------------------------------------------------------------------------
    def _lin(self, mlp):
        return LinearT(_ptr(mlp.weight), _ptr(mlp.bias), mlp.in_features, mlp.out_features)

    def _norm(self, gn):
        return NormT(_ptr(gn.norm.weight), _ptr(gn.norm.bias))

    def _kp(self, kp):
        w = kp.weights.detach()
        wt = w.reshape(-1, w.shape[2]).t().contiguous() if w.shape[1] % 32 == 0 else None
        if wt is not None:
            self._keep.append(wt)
        return KPConvT(_ptr(w), _ptr(wt), _ptr(kp.bias), _ptr(kp.kernel_points), w.shape[1], w.shape[2], float(kp.sigma))

    def _res(self, blk):
        r = ResBlockT()
        r.c_in, r.strided = blk.in_channels, int(blk.strided)
        r.has_unary1 = int(not isinstance(blk.unary1, torch.nn.Identity))
        if r.has_unary1:
            r.unary1, r.norm1 = self._lin(blk.unary1.mlp), self._norm(blk.unary1.norm)
        r.conv, r.norm_conv = self._kp(blk.KPConv), self._norm(blk.norm_conv)
        r.unary2, r.norm2 = self._lin(blk.unary2.mlp), self._norm(blk.unary2.norm)
        r.has_shortcut = int(not isinstance(blk.unary_shortcut, torch.nn.Identity))
        if r.has_shortcut:
            r.shortcut, r.norm_sc = self._lin(blk.unary_shortcut.mlp), self._norm(blk.unary_shortcut.norm)
        return r

    def _build_backbone(self, bb):
        b = BackboneT()
        b.num_stages, b.finest_decoder = bb.num_stages, bb.finest_decoder
        b.groups = bb.encoder1_1.norm.num_groups
        b.init_dim = bb.encoder1_1.out_channels
        b.conv1, b.norm1 = self._kp(bb.encoder1_1.KPConv), self._norm(bb.encoder1_1.norm)
        b.blocks[0] = self._res(bb.encoder1_2)
        i = 1
        for lvl in range(2, bb.num_stages + 1):
            for j in (1, 2, 3):
                b.blocks[i] = self._res(getattr(bb, f'encoder{lvl}_{j}'))
                i += 1
        for d, lvl in enumerate(range(bb.num_stages - 1, bb.finest_decoder - 1, -1)):
            dec = getattr(bb, f'decoder{lvl}')
            b.decoders[d] = self._lin(dec.mlp)
            if lvl != bb.finest_decoder:
                b.decoder_norms[d] = self._norm(dec.norm)
        self._dec_channels = [getattr(bb, f'decoder{lvl}').mlp.out_features
                              for lvl in range(bb.num_stages - 1, bb.finest_decoder - 1, -1)]
        self._coarse_channels = getattr(bb, f'encoder{bb.num_stages}_3').out_channels
        return b

    def _build_transformer(self, tr):
        arr = (TLayerT * len(tr.layers))()
        for i, (blk, layer) in enumerate(zip(tr.blocks, tr.layers)):
            mha = layer.attention.attention
            t = TLayerT()
            t.is_self = int(blk == 'self')
            cat = lambda names, attr: torch.cat([getattr(getattr(mha, n), attr).detach() for n in names], dim=0).contiguous()
            if t.is_self:
                wqkv, bqkv = cat(('proj_q', 'proj_k', 'proj_v'), 'weight'), cat(('proj_q', 'proj_k', 'proj_v'), 'bias')
                wpt = mha.proj_p.weight.detach().t().contiguous()
                self._keep += [wqkv, bqkv, wpt]
                t.w_qkv, t.b_qkv, t.wp_t, t.bp = _ptr(wqkv), _ptr(bqkv), _ptr(wpt), _ptr(mha.proj_p.bias)
            else:
                wkv, bkv = cat(('proj_k', 'proj_v'), 'weight'), cat(('proj_k', 'proj_v'), 'bias')
                self._keep += [wkv, bkv]
                t.w_q, t.b_q, t.w_kv, t.b_kv = _ptr(mha.proj_q.weight), _ptr(mha.proj_q.bias), _ptr(wkv), _ptr(bkv)
            att, ffn = layer.attention, layer.output
            t.att_linear = LinearT(_ptr(att.linear.weight), _ptr(att.linear.bias), att.linear.in_features, att.linear.out_features)
            t.att_norm = NormT(_ptr(att.norm.weight), _ptr(att.norm.bias))
            t.expand = LinearT(_ptr(ffn.expand.weight), _ptr(ffn.expand.bias), ffn.expand.in_features, ffn.expand.out_features)
            t.squeeze = LinearT(_ptr(ffn.squeeze.weight), _ptr(ffn.squeeze.bias), ffn.squeeze.in_features, ffn.squeeze.out_features)
            t.out_norm = NormT(_ptr(ffn.norm.weight), _ptr(ffn.norm.bias))
            arr[i] = t
        return arr, len(tr.layers)

    # -- stage calls ---------------------------------------------------------------------------------------------
    def backbone_forward(self, feats, data_dict):
        """KPConvFPN.forward: returns feats_list [fine ... coarse] like the module."""
        lib = L.lib()
        S = self.backbone.num_stages
        pts, nb, sub, up = data_dict['points'], data_dict['neighbors'], data_dict['subsampling'], data_dict['upsampling']
        dev = feats.device
        rows = (I64 * S)(*[p.shape[0] for p in pts])
        parr = (P * S)(*[p.data_ptr() for p in pts])
        narr, nw = (P * S)(*[t.data_ptr() for t in nb]), (I64 * S)(*[t.shape[1] for t in nb])
        sarr, sw = (P * S)(*[t.data_ptr() for t in sub]), (I64 * S)(*[t.shape[1] for t in sub])
        uarr, uw = (P * S)(*[t.data_ptr() for t in up]), (I64 * S)(*[t.shape[1] for t in up])
        outs = [torch.empty((pts[-1].shape[0], self._coarse_channels), dtype=torch.float32, device=dev)]
        for d, lvl in enumerate(range(S - 1, self.backbone.finest_decoder - 1, -1)):
            outs.append(torch.empty((pts[lvl - 1].shape[0], self._dec_channels[d]), dtype=torch.float32, device=dev))
        oarr = (P * len(outs))(*[o.data_ptr() for o in outs])
        ws_bytes = lib.geob200_backbone_workspace_bytes(ctypes.byref(self.backbone), rows)
        ws = L.workspace(ws_bytes, dev, 'native_backbone')
        n_pairs = int(data_dict.get('batch_size', 1))
        gn_bytes = lib.geob200_backbone_gn_workspace_bytes(ctypes.byref(self.backbone), rows, n_pairs)
        gn = L.workspace(gn_bytes, dev, 'group_norm')
        carr = marr = None
        if n_pairs > 1:
            # batch of pairs in stack order [ref_1..ref_B, src_1..src_B]: per-pair GroupNorm statistics need the cloud rows
            lens = data_dict['lengths_host']
            keep = [(I64 * (2 * n_pairs))(*[int(v) for v in lens[l]]) for l in range(S)]
            carr = (P * S)(*[ctypes.cast(k, P).value for k in keep])
            # widest subsampling row per cloud: the strided blocks' maxpool sees each pair at its own table width
            cmax = torch.empty((S - 1, 2 * n_pairs), dtype=torch.int32, device=dev)
            for l in range(S - 1):
                L.check(lib.geob200_cloud_max_count(sub[l].data_ptr(), sub[l].shape[0], pts[l].shape[0], sub[l].shape[1], n_pairs, keep[l + 1],
                                                    cmax[l].data_ptr(), L.stream_ptr()), 'cloud_max_count')
            marr = (P * S)(*([cmax[l].data_ptr() for l in range(S - 1)] + [None]))
        L.check(lib.geob200_backbone_forward_batched(ctypes.byref(self.backbone), feats.data_ptr(), parr, rows, narr, nw, sarr, sw, uarr, uw,
                                                     oarr, gn.data_ptr(), gn.numel(), ws.data_ptr(), ws.numel(), L.stream_ptr(), n_pairs,
                                                     carr, marr), 'backbone_forward_batched')
        outs.reverse()
        return outs

    def transformer_forward_batched(self, x, cloud_rows, embeddings):
        """RPEConditionalTransformer over a batch of pairs: x rows in stack order [ref_1..ref_B, src_1..src_B],
        ``cloud_rows`` their 2B row counts (host ints), ``embeddings`` the 2B structure embeddings (device tensors)."""
        lib = L.lib()
        nc = len(cloud_rows)
        rows = (I64 * nc)(*[int(r) for r in cloud_rows])
        earr = (P * nc)(*[e.data_ptr() for e in embeddings])
        out = torch.empty_like(x)
        ws_bytes = lib.geob200_transformer_batched_workspace_bytes(nc // 2, rows, self.hidden, self.heads, self.num_layers)
        ws = L.workspace(ws_bytes, x.device, 'native_transformer')
        L.check(lib.geob200_transformer_forward_batched(self.layers, self.num_layers, self.hidden, self.heads, x.data_ptr(), nc // 2, rows,
                                                        earr, out.data_ptr(), ws.data_ptr(), ws.numel(), L.stream_ptr()),
                'transformer_forward_batched')
        return out

    def transformer_forward(self, x, n0, emb0, emb1):
        """RPEConditionalTransformer.forward_stacked"""
        lib = L.lib()
        n1 = x.shape[0] - n0
        out = torch.empty_like(x)
        ws_bytes = lib.geob200_transformer_workspace_bytes(n0, n1, self.hidden, self.heads, self.num_layers)
        ws = L.workspace(ws_bytes, x.device, 'native_transformer')
        L.check(lib.geob200_transformer_forward(self.layers, self.num_layers, self.hidden, self.heads, x.data_ptr(), n0, n1, emb0.data_ptr(),
                                                emb1.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel(), L.stream_ptr()),
                'transformer_forward')
        return out
