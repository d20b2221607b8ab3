"""TEST INFRASTRUCTURE ONLY -- packs the stage-boundary tensors of one forward (the real reference's, when run by
oracle/make_golden.py in the build container; the pinned restatement oracle/geo_oracle.py's, when a -m gpu parity test runs
it live at BASELINE.json's full sizes) into the flat dict layout of tests/golden/*.npz, so that fixture-based and live
parity tests share one checker (tests/test_gpu_e2e.py::check_forward)."""
import hashlib

import numpy as np
import torch


def sample_rows(t, n=64):
    t = t.detach()
    idx = np.unique(np.linspace(0, t.shape[0] - 1, num=min(n, t.shape[0])).astype(np.int64))
    return idx, t[idx].numpy()


def pack(data, taps, out, node_corr_scores, limits):
    """data: collated dict (CPU tensors); taps: geo_oracle.forward taps; out: output_dict the fixture is made of."""
    g = {}
    for i, (p, l) in enumerate(zip(data['points'], data['lengths'])):
        if i > 0:
            g[f'points_{i}'] = p.numpy()
        g[f'lengths_{i}'] = l.numpy()
    for key in ('neighbors', 'subsampling', 'upsampling'):
        for i, t in enumerate(data[key]):
            g[f'{key}_{i}'] = t.numpy().astype(np.uint16 if int(t.max()) < 65536 else np.int32)   # sentinel = number of support rows
    for k in ('feats_c', 'feats_f', 'ref_embeddings'):
        t = taps[k]
        idx, rows = sample_rows(t.reshape(t.shape[0], -1) if k != 'ref_embeddings' else t.reshape(-1, t.shape[-1]), 96)
        g[k + '_rows'], g[k + '_sample'] = idx, rows
        g[k + '_sum'] = np.array([t.double().sum().item(), t.double().abs().sum().item()])
    for k in ('ref_feats_c', 'src_feats_c', 'estimated_transform', 'corr_scores', 'ref_corr_points', 'src_corr_points',
              'ref_node_corr_indices', 'src_node_corr_indices'):
        g[k] = out[k].detach().numpy()
    g['gt_node_corr_indices'] = out['gt_node_corr_indices'].numpy()
    g['gt_node_corr_overlaps'] = out['gt_node_corr_overlaps'].numpy()
    g['node_corr_scores'] = node_corr_scores.numpy()
    idx, rows = sample_rows(out['matching_scores'].reshape(out['matching_scores'].shape[0], -1), 16)
    g['matching_scores_rows'], g['matching_scores_sample'] = idx, rows
    for k in ('ref_node_knn_indices', 'src_node_knn_indices'):
        g[k] = taps[k].numpy().astype(np.int32)
    g['neighbor_limits'] = np.array(limits)
    return g


# ---- compact form of one checked pair (tests/golden/check_<workload>_<pair>.npz): what make_golden.run compares, small enough
# to store for several pairs.  Collate outputs as SHA-256 digests plus the rows in which the reference's neighbour tables differ
# from the restatement's (order inside exact-distance ties), float outputs as fixed strided element samples.
CHECK_FLOATS = ('ref_feats_c', 'src_feats_c', 'ref_feats_f', 'src_feats_f', 'matching_scores')
CORR_KEYS = ('ref_corr_points', 'src_corr_points', 'corr_scores')
VARIANTS = ('3dmatch', 'kitti', 'modelnet')
TABLES = (('neighbors', 0, 0), ('subsampling', 1, 0), ('upsampling', 0, 1))


def digest(t):
    """SHA-256 of dtype, shape and bytes of a CPU tensor"""
    a = np.ascontiguousarray(t.numpy())
    h = hashlib.sha256(f'{a.dtype.str}{a.shape}'.encode())
    h.update(a.tobytes())
    return h.hexdigest()


def _elements(t, n=512):
    flat = t.detach().reshape(-1)
    idx = np.unique(np.linspace(0, flat.shape[0] - 1, num=min(n, flat.shape[0])).astype(np.int64))
    return idx, flat[idx].numpy()


def corr_rows(out):
    """fine correspondences as rows [ref point, src point, score] (float64), in output order and sorted lexicographically"""
    r = torch.cat([out['ref_corr_points'], out['src_corr_points'], out['corr_scores'][:, None]], dim=1).double().numpy()
    return r, r[np.lexsort(r.T[::-1])]


def pack_check(data, own_tables, ref_out, metrics, limits):
    """data: the reference's collated dict; own_tables: {key: [table per level]} of the restatement; metrics: {variant: {name: value}}"""
    g = {'neighbor_limits': np.array(limits)}
    for i, (p, l) in enumerate(zip(data['points'], data['lengths'])):
        g[f'points_{i}.digest'], g[f'lengths_{i}'] = np.array(digest(p)), l.numpy()
    for key, _, _ in TABLES:
        for i, (mine, ref) in enumerate(zip(own_tables[key], data[key])):
            rows = (mine != ref).any(dim=1).nonzero().reshape(-1)
            g[f'{key}_{i}.digest'] = np.array(digest(ref))
            g[f'{key}_{i}.patch_rows'], g[f'{key}_{i}.patch'] = rows.numpy().astype(np.int32), ref[rows].numpy().astype(np.int32)
    for k in CHECK_FLOATS:
        g[k + '.shape'] = np.array(ref_out[k].shape, dtype=np.int64)
        g[k + '.index'], g[k + '.sample'] = _elements(ref_out[k])
    for k in ('estimated_transform', 'ref_node_corr_indices', 'src_node_corr_indices', 'gt_node_corr_indices', 'gt_node_corr_overlaps'):
        g[k] = ref_out[k].detach().numpy()
    ordered, as_set = corr_rows(ref_out)
    g['corr.count'] = np.array(ordered.shape[0])
    g['corr.index'], g['corr.ordered'] = sample_rows(torch.from_numpy(ordered), 128)
    g['corr.sorted'] = as_set[g['corr.index']]
    for v, m in metrics.items():
        g['metric_names_' + v] = np.array(sorted(m))
        g['metric_values_' + v] = np.array([m[k] for k in sorted(m)], dtype=np.float64)
    return g


def apply_reference_tables(data, gold):
    """checks the restatement's collate against the stored digests and replaces its neighbour tables by the reference's own
    (restatement rows + the stored rows that differ only in the order inside exact-distance ties); returns mismatches"""
    from oracle import geo_oracle
    bad = []
    for i, p in enumerate(data['points']):
        if digest(p) != str(gold[f'points_{i}.digest']) or data['lengths'][i].tolist() != gold[f'lengths_{i}'].tolist():
            bad.append(f'points_{i}')
    for key, qi, si in TABLES:
        for i, mine in enumerate(data[key]):
            ref = mine.clone()
            rows = torch.from_numpy(gold[f'{key}_{i}.patch_rows'].astype(np.int64))
            ref[rows] = torch.from_numpy(gold[f'{key}_{i}.patch'].astype(np.int64))
            q, s = data['points'][i + qi], data['points'][i + si]
            if digest(ref) != str(gold[f'{key}_{i}.digest']) or not torch.equal(
                    geo_oracle.canonical_neighbors(q, s, mine), geo_oracle.canonical_neighbors(q, s, ref)):
                bad.append(f'{key}_{i}')
            data[key][i] = ref
    return bad


def check_outputs(o, metrics, gold):
    """make_golden.run's restatement-vs-reference report on the compact form: max abs differences (or False / 'SHAPE') per key"""
    report = {}
    want = list(zip(gold['ref_node_corr_indices'].tolist(), gold['src_node_corr_indices'].tolist()))
    got = list(zip(o['ref_node_corr_indices'].tolist(), o['src_node_corr_indices'].tolist()))
    perm = None
    if got != want:
        # coarse scores within 1e-5 relative of each other may swap places: accept such a permutation and compare under it
        pos = {pr: i for i, pr in enumerate(got)}
        report['node_corr_set'] = len(pos) == len(want) and set(pos) == set(want)
        if report['node_corr_set']:
            perm = torch.tensor([pos[pr] for pr in want])
            sc = o['node_corr_scores']
            report['node_corr_permuted_between_equal_scores'] = bool(torch.allclose(sc[perm], sc, rtol=1e-5, atol=0))
    for k in CHECK_FLOATS:
        t = o[k] if (perm is None or k != 'matching_scores') else o[k][perm]
        if list(t.shape) != gold[k + '.shape'].tolist():
            report[k] = 'SHAPE'
            continue
        report[k] = float(np.abs(t.detach().reshape(-1).numpy()[gold[k + '.index']] - gold[k + '.sample']).max())
    report['estimated_transform'] = float(np.abs(o['estimated_transform'].numpy() - gold['estimated_transform']).max())
    ordered, as_set = corr_rows(o)
    if ordered.shape[0] != int(gold['corr.count']):
        report['corr'] = 'SHAPE'
    else:
        # the fine correspondences come out patch after patch: under a coarse permutation only the set is comparable
        report['corr_set'] = float(np.abs(as_set[gold['corr.index']] - gold['corr.sorted']).max())
        if perm is None:
            report['corr'] = float(np.abs(ordered[gold['corr.index']] - gold['corr.ordered']).max())
    report['gt_node_corr_indices'] = bool(np.array_equal(o['gt_node_corr_indices'].numpy(), gold['gt_node_corr_indices']))
    if o['gt_node_corr_overlaps'].shape != gold['gt_node_corr_overlaps'].shape:
        report['gt_node_corr_overlaps'] = 'SHAPE'
    else:
        report['gt_node_corr_overlaps'] = float(np.abs(o['gt_node_corr_overlaps'].numpy() - gold['gt_node_corr_overlaps']).max())
    for v in VARIANTS:
        names = gold['metric_names_' + v].tolist()
        report[f'metric_{v}_names'] = sorted(metrics[v]) == names
        for name, value in zip(names, gold['metric_values_' + v]):
            report[f'metric_{v}_{name}'] = abs(float(metrics[v][name]) - float(value))
    return report


def deviations(report):
    """keys of a report beyond the tolerances of make_golden.run (1e-5; RRE, an acos of an fp32 3x3 product: 1e-3)"""
    return [k for k, v in report.items() if v == 'SHAPE' or v is False or
            (isinstance(v, float) and v > (1e-3 if k.endswith('RRE') else 1e-5))]
