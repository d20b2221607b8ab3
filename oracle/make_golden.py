"""TEST INFRASTRUCTURE ONLY -- generates the committed fixtures under tests/golden/ by running the REAL reference
(imported from /root/reference through oracle/ref_harness.py, CPU) and checks the restatement oracle/geo_oracle.py
against it.  Run in the build container:   python -m oracle.make_golden

Fixtures (compressed npz, a few MB in total):
  tests/golden/<workload>.npz        reference outputs at the stage boundaries of SURVEY.md section 8a for the
                                     deterministic pair synth.make_pair(workload, 0) and the deterministic weights
                                     weights.synthetic_state_dict(model, 7351)
The big tensors are stored as strided row samples + float64 checksums (row index arrays are stored alongside).
"""
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from geotransformer_b200.config import make_cfg                     # noqa: E402
from geotransformer_b200.model import create_model                  # noqa: E402
from geotransformer_b200.synth import make_pair                     # noqa: E402
from geotransformer_b200.weights import synthetic_state_dict        # noqa: E402
from oracle import fixture, geo_oracle, ref_ext, ref_harness        # noqa: E402

GOLD = os.environ.get('GEOB200_GOLDEN_OUT') or os.path.join(ROOT, 'tests', 'golden')    # override: regenerate elsewhere and compare
LIMITS = {'demo2k': [38, 36, 36, 38], 'modelnet717': [13, 21, 27], 'kitti4k': [27, 75, 147, 157, 119]}


def run(workload, index=0, write=True):
    """reference run + restatement check on pair ``index`` of the workload; ``write``: pack the fixture (pair 0 is the committed one)"""
    pair = make_pair(workload, index)
    cfg = make_cfg(pair['config'])
    limits = cfg.neighbor_limits or LIMITS[workload]
    torch.manual_seed(0)
    sd = synthetic_state_dict(create_model(cfg), 7351)

    rcfg, rcreate = ref_harness.load_experiment(pair['config'])
    from geotransformer.utils.data import registration_collate_fn_stack_mode
    ref_model = rcreate(rcfg).eval()
    ref_model.load_state_dict(sd, strict=True)
    dd = {k: pair[k] for k in ('ref_points', 'src_points', 'ref_feats', 'src_feats', 'transform')}
    t0 = time.time()
    data = registration_collate_fn_stack_mode([dd], rcfg.backbone.num_stages, rcfg.backbone.init_voxel_size,
                                              rcfg.backbone.init_radius, limits)
    data = {k: ([x.clone() if isinstance(x, torch.Tensor) else x for x in v] if isinstance(v, list) else
                (v.clone() if isinstance(v, torch.Tensor) else v)) for k, v in data.items()}
    t1 = time.time()
    with torch.no_grad():
        ref_out = ref_model(data)
    t2 = time.time()
    print(f'[{workload}] reference collate {t1 - t0:.2f}s forward {t2 - t1:.2f}s; '
          f'levels {[int(p.shape[0]) for p in data["points"]]} corr {ref_out["ref_corr_points"].shape[0]}')

    # ---- the restatement must reproduce the reference on CPU
    odata = geo_oracle.collate_pair(pair, cfg, limits, impl=ref_ext)
    for i in range(cfg.backbone.num_stages):
        assert torch.equal(odata['points'][i], data['points'][i]) and torch.equal(odata['neighbors'][i], data['neighbors'][i])
    odata2 = geo_oracle.collate_pair(pair, cfg, limits)          # plain-C restatement of the ext
    for i in range(cfg.backbone.num_stages):
        assert torch.equal(odata2['points'][i], data['points'][i]), f'grid order differs at level {i}'
    # Neighbour tables: identical up to the order inside EXACT-distance tie groups (the barycentre of a 2-point voxel
    # is equidistant to both points; the reference orders such ties by an unstable std::sort, the restatement by index)
    n_tie_rows = 0
    for key, qi, si in (('neighbors', 0, 0), ('subsampling', 1, 0), ('upsampling', 0, 1)):
        for i, (a, b) in enumerate(zip(odata2[key], data[key])):
            q, s = data['points'][i + qi], data['points'][i + si]
            ca, cb = geo_oracle.canonical_neighbors(q, s, a), geo_oracle.canonical_neighbors(q, s, b)
            assert torch.equal(ca, cb), f'{key}[{i}] differs beyond tie order'
            n_tie_rows += int((a != b).any(dim=1).sum())
    print(f'[{workload}] neighbour tables equal up to exact-tie order ({n_tie_rows} rows with a swapped tie)')
    own_tables = {key: list(odata2[key]) for key in ('neighbors', 'subsampling', 'upsampling')}
    odata2 = {k: v for k, v in odata2.items()}
    for key in ('neighbors', 'subsampling', 'upsampling'):
        odata2[key] = data[key]                                   # teacher-force the reference's tie order downstream
    taps = {}
    with torch.no_grad():
        o = geo_oracle.forward(sd, cfg, odata2, taps=taps)
    report = {}
    for k in ('ref_feats_c', 'src_feats_c', 'ref_feats_f', 'src_feats_f', 'matching_scores', 'estimated_transform',
              'ref_corr_points', 'src_corr_points', 'corr_scores'):
        a, b = o[k], ref_out[k]
        report[k] = (tuple(a.shape) == tuple(b.shape)) and float((a - b).abs().max()) if a.shape == b.shape else 'SHAPE'
    for k in ('ref_node_corr_indices', 'src_node_corr_indices'):
        report[k] = bool(torch.equal(o[k], ref_out[k]))
    if not (report['ref_node_corr_indices'] and report['src_node_corr_indices']):
        # adjacent coarse scores can sit within an ulp of each other (SURVEY.md 'hard parts': min relative gap 2e-6 with
        # random weights) while the restatement's features differ from the reference's by 1e-7: accept a permutation
        # between scores that agree to 1e-5 relative and compare the per-patch tensors under it
        pos = {pr: i for i, pr in enumerate(zip(o['ref_node_corr_indices'].tolist(), o['src_node_corr_indices'].tolist()))}
        want = list(zip(ref_out['ref_node_corr_indices'].tolist(), ref_out['src_node_corr_indices'].tolist()))
        assert len(pos) == len(want) and set(pos) == set(want), 'coarse correspondence SETS differ'
        perm = torch.tensor([pos[pr] for pr in want])
        sc = o['node_corr_scores']
        assert torch.allclose(sc[perm], sc, rtol=1e-5, atol=0), 'coarse correspondences permuted between DIFFERENT scores'
        moved = int((perm != torch.arange(len(want))).sum())
        print(f'[{workload}] {moved} coarse correspondences swapped between scores equal to 1e-5 relative')
        a, b = o['matching_scores'][perm], ref_out['matching_scores']
        report['matching_scores'] = float((a - b).abs().max())
        report['ref_node_corr_indices'] = report['src_node_corr_indices'] = True
        # the fine correspondences come out patch after patch, i.e. block-permuted with the coarse order: compare them as a SET
        # (rows [ref point, src point, score] sorted lexicographically)

        def rows(out):
            r = torch.cat([out['ref_corr_points'], out['src_corr_points'], out['corr_scores'][:, None]], dim=1).double().numpy()
            return r[np.lexsort(r.T[::-1])]
        ra, rb = rows(o), rows(ref_out)
        same = ra.shape == rb.shape and float(np.abs(ra - rb).max()) if ra.shape == rb.shape else 'SHAPE'
        report['ref_corr_points'] = report['src_corr_points'] = report['corr_scores'] = same
    # ground-truth superpoint correspondences and the Evaluator (loss.py:95-159)
    report['gt_node_corr_indices'] = bool(torch.equal(o['gt_node_corr_indices'], ref_out['gt_node_corr_indices']))
    report['gt_node_corr_overlaps'] = float((o['gt_node_corr_overlaps'] - ref_out['gt_node_corr_overlaps']).abs().max())
    evaluator = ref_harness.load_evaluator(pair['config'], rcfg)
    with torch.no_grad():
        ref_metrics = {k: float(v) for k, v in evaluator(ref_out, data).items()}
    o_metrics = {k: float(v) for k, v in geo_oracle.evaluate(cfg, o, data['transform']).items()}
    assert set(ref_metrics) == set(o_metrics), (ref_metrics, o_metrics)
    for k in ref_metrics:
        report['metric_' + k] = abs(ref_metrics[k] - o_metrics[k])
    # the other two Evaluator variants (KITTI: no RMSE, RR from RRE/RTE; ModelNet: RMSE of T_est x - T_gt x) on the same outputs
    other_metrics, o_metrics_all = {}, {pair['config']: o_metrics}
    for other in ('3dmatch', 'kitti', 'modelnet'):
        if other == pair['config']:
            continue
        ocfg_ref, _ = ref_harness.load_experiment(other)
        with torch.no_grad():
            rm = {k: float(v) for k, v in ref_harness.load_evaluator(other, ocfg_ref)(ref_out, data).items()}
        om = {k: float(v) for k, v in geo_oracle.evaluate(make_cfg(other), o, data['transform']).items()}
        assert set(rm) == set(om), (rm, om)
        for k in rm:
            report[f'metric_{other}_{k}'] = abs(rm[k] - om[k])
        other_metrics[other] = rm
        o_metrics_all[other] = om
    print(f'[{workload}] reference metrics:', ref_metrics)
    print(f'[{workload}] oracle-vs-reference max abs diff:', report)
    bad = [k for k, v in report.items() if v == 'SHAPE' or v is False or
           (isinstance(v, float) and v > (1e-3 if k.endswith('RRE') else 1e-5))]   # RRE: acos of an fp32 3x3 product
    assert not bad, f'oracle restatement deviates from the reference: {bad}'

    if not write:
        # compact fixture of this pair for tests/test_oracle.py, and its replay on the restatement's output
        g = fixture.pack_check(data, own_tables, ref_out, dict(other_metrics, **{pair['config']: ref_metrics}), limits)
        bad = fixture.deviations(fixture.check_outputs(o, o_metrics_all, g))
        assert not bad, f'replay of the compact fixture deviates: {bad}'
        os.makedirs(GOLD, exist_ok=True)
        path = os.path.join(GOLD, f'check_{workload}_{index}.npz')
        np.savez_compressed(path, **g)
        print(f'[{workload}] pair {index}: restatement == reference; wrote {path} ({os.path.getsize(path) / 1e3:.0f} kB)')
        return
    # ---- fixtures
    g = fixture.pack(data, taps, ref_out, o['node_corr_scores'], limits)
    g['metric_names'] = np.array(sorted(ref_metrics))
    g['metric_values'] = np.array([ref_metrics[k] for k in sorted(ref_metrics)], dtype=np.float64)
    for other, rm in other_metrics.items():
        g['metric_names_' + other] = np.array(sorted(rm))
        g['metric_values_' + other] = np.array([rm[k] for k in sorted(rm)], dtype=np.float64)
    os.makedirs(GOLD, exist_ok=True)
    path = os.path.join(GOLD, workload + '.npz')
    np.savez_compressed(path, **g)
    print(f'[{workload}] wrote {path} ({os.path.getsize(path) / 1e6:.2f} MB)')


def run_calibration():
    """neighbour-limit calibration (utils/data.py:190-217) of the real reference over three demo pairs"""
    ref_harness.load_experiment('3dmatch')
    from geotransformer.utils.data import calibrate_neighbors_stack_mode, registration_collate_fn_stack_mode
    cfg = make_cfg('3dmatch')
    b = cfg.backbone
    keys = ('ref_points', 'src_points', 'ref_feats', 'src_feats', 'transform')
    pairs = [{k: make_pair('demo2k', i)[k] for k in keys} for i in range(3)]
    g = {}
    for thr in (2000, 150):
        want = calibrate_neighbors_stack_mode(pairs, registration_collate_fn_stack_mode, b.num_stages, b.init_voxel_size, b.init_radius,
                                              sample_threshold=thr)
        got = geo_oracle.calibrate_neighbors(pairs, cfg, sample_threshold=thr)
        got_ref_ext = geo_oracle.calibrate_neighbors(pairs, cfg, sample_threshold=thr, impl=ref_ext)
        assert np.array_equal(want, got) and np.array_equal(want, got_ref_ext), (want, got, got_ref_ext)
        g[f'limits_threshold_{thr}'] = np.asarray(want)
        print(f'[calibration] sample_threshold {thr}: limits {want.tolist()} (oracle equal)')
    np.savez_compressed(os.path.join(GOLD, 'calibration.npz'), **g)


def run_reference_ops():
    """the reference's C++ collate ops (oracle/_ref) and its Boundary-2 torch ops on the seeded inputs of oracle/ref_vectors.py,
    checked LIVE against the restatements, stored as tests/golden/reference_ops.npz for tests/test_oracle.py"""
    from oracle import collate_oracle
    from oracle import ref_vectors as V
    assert ref_ext.available(), 'needs oracle/_ref (make -C oracle ref)'
    digests = {}
    for w, voxel in V.COLLATE_CASES:
        want, got = V.collate_chain(ref_ext, w, voxel), V.collate_chain(collate_oracle, w, voxel)
        for k, t in want.items():
            assert torch.equal(t, got[k]), (w, k)
            digests[f'collate.{w}.{k}'] = V.digest(t)
    for n in V.REHASH_SIZES:
        t = V.rehash_points(ref_ext, n)
        assert torch.equal(t, V.rehash_points(collate_oracle, n)), n
        digests[f'rehash.{n}'] = V.digest(t)
    cases = V.adversarial_cases()
    for c, (lengths, seed, lattice, voxel) in enumerate(cases):
        want, got = V.adversarial(ref_ext, lengths, seed, lattice, voxel), V.adversarial(collate_oracle, lengths, seed, lattice, voxel)
        for k, t in want.items():
            assert torch.equal(t, got[k]), (c, k)
            digests[f'adversarial.{c}.{k}'] = V.digest(t)
    # Boundary-2 ops of the reference package, in this process (ref_harness patches Tensor.cuda: nothing after this uses CUDA)
    ref_harness.install()
    from geotransformer.modules import ops as R
    mine = dict(V.boundary_2_ops(geo_oracle))
    for k, t in V.boundary_2_ops(R):
        assert torch.equal(t, mine[k]), k
        digests['ops.' + k] = V.digest(t)
    path = os.path.join(GOLD, 'reference_ops.npz')
    np.savez_compressed(path, digest_keys=np.array(list(digests)), digests=np.array(list(digests.values())))
    print(f'[reference_ops] {len(cases)} adversarial cases, {len(mine)} op results: restatement == reference; wrote {path} '
          f'({os.path.getsize(path) / 1e3:.0f} kB)')


if __name__ == '__main__':
    assert ref_harness.available(), 'needs /root/reference'
    # `check:<workload>:<pair index>` = compare the restatement with the reference on ANOTHER pair of the workload, write nothing
    for w in (sys.argv[1:] or ['demo2k', 'modelnet717', 'kitti4k', 'calibration', 'reference_ops']):
        if w.startswith('check:'):
            _, name, idx = w.split(':')
            run(name, int(idx), write=False)
        elif w == 'reference_ops':
            run_reference_ops()
        else:
            run_calibration() if w == 'calibration' else run(w)
