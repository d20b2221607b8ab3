#!/usr/bin/env python
"""Benchmark of the registration hot path (BASELINE.json metric: point-cloud pairs/sec on 3DMatch-shape synthetic pairs).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload 3dmatch20k] [--dump-outputs DIR]

A step = one pass of the hot path (stack-mode collate -> KPConv-FPN -> geometric transformer -> superpoint matching ->
Sinkhorn -> local-to-global registration -> Evaluator) over --pairs-per-step (64) synthetic pairs per rank, registered by
geotransformer_b200.engine.RegistrationEngine: --batch (8) pairs per forward, --streams (2) forwards in flight (weak scaling:
pair i of rank r is synth.make_pair(workload, r + i*W); at 8 GPUs two steps are BASELINE config 5's 1024 pairs).
Prints ONE JSON line (see the task contract):
  value     pairs/s with the raw pairs already resident in HBM when the timed region starts
  e2e       pairs/s through the public API with HOST (pinned) inputs: H2D + collate + forward + D2H of transform + metrics
  roofline  the dominant kernel family by GPU-time share (tcgen05 3xTF32 GEMMs), algorithmic FLOPs / CUDA-event time, with the
            measured TF32 dense peak and the committed ncu DRAM traffic; beside it roofline_gse_embed (the structure embedding:
            an HBM row with the default tabulated projections, a tensor row with --gse-mode 3) and roofline_attention (HBM)
  config    the STATIC workload description, identical in both arms; run_info = what was measured during the run
  cpu_baseline    the reference's CPU path on this box's host cores, bounded sample (N=1 only): 16-thread and 1-thread numbers
  gpu_eager_port  host collate + the pinned torch restatement executed as eager ops on this GPU (what a drop-in user sees today)
--impl reference times the CPU path alone (the reference's own C++ collate ops + the oracle port of the forward) on the same
config, each of its steps a bounded sample (one pair) of the configured step.
"""
import argparse
import json
import os

import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'point-cloud pairs/sec (3DMatch-shape synth)'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='3dmatch20k')
    ap.add_argument('--gse-mode', type=int, default=None)
    ap.add_argument('--linear-persistent', type=int, default=None, help='1/0: persistent tile loop of the tcgen05 GEMM')
    ap.add_argument('--batch', type=int, default=8, help='pairs per forward (GeoTransformer.forward_batch); 1 = one pair per forward')
    ap.add_argument('--streams', type=int, default=None,
                    help='forwards in flight per GPU (one CUDA stream + host thread each); default 2 in batch mode, 4 with --batch 1')
    ap.add_argument('--pairs-per-step', type=int, default=None, help='pairs per GPU and step (default 4 x batch x streams = 64)')
    ap.add_argument('--attention-tma', type=int, default=None, help='1/0: TMA-staged self-attention kernels (default 1)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned for each of its pairs as DIR/<name>.npy (rank 0), so that two '
                         'builds run with the same arguments can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes what the GPU path computed: use it with --impl ours')
    return args


def dist_env():
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    return rank, world, local


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons DURING the timed region (profiling recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': float(self.rows[0][1]), 'reasons': reasons}


def load_peaks():
    """(bf16 dense TF/s BURST -- the roofline kernels are timed alone --, sustained, HBM GB/s, source)"""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('bf16_tflops'), d.get('bf16_tflops_sustained', d.get('bf16_tflops')), d.get('hbm_gbs'), 'measured'
    return 1690.0, 1400.0, 6650.0, 'fallback (B200_PROFILING.md)'


def measure_tf32_peak(dev):
    """Dense TF32 tensor throughput of this GPU, measured the way MEASURED_PEAKS.json's bf16 figure was (torch.matmul 8192^3,
    best of 10, CUDA events) with fp32 operands and allow_tf32=True.  A library GEMM as a yardstick only -- not on the product path."""
    try:
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        n = 8192
        a = torch.randn(n, n, device=dev)
        b = torch.randn(n, n, device=dev)
        c = torch.empty(n, n, device=dev)
        best = float('inf')
        for i in range(13):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b, out=c)
            e1.record()
            e1.synchronize()
            if i >= 3:
                best = min(best, e0.elapsed_time(e1))
        torch.backends.cuda.matmul.allow_tf32 = prev
        del a, b, c
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    except Exception:
        return None


def attention_roofline(dev, n_sp, clouds, channels, heads, peak_hbm, traffic):
    """HBM roofline of the self-attention (the E stream, N^2 C 4 bytes per cloud and layer, is its only large operand): one
    layer over `clouds` clouds of n_sp superpoints through geob200_attention_batched (q.k pass + TMA-staged E stream + P.v pass),
    CUDA events around the three launches, L2 flushed between repetitions.  achieved = E bytes / time of ALL three launches."""
    try:
        import ctypes
        from geotransformer_b200 import _lib as L

        class Item(ctypes.Structure):
            _fields_ = [(n, ctypes.c_void_p) for n in ('q', 'k', 'v', 'qp', 'qb', 'embed', 'out')] + [('n_query', ctypes.c_int64), ('n_key', ctypes.c_int64)]
        C, H, N = channels, heads, n_sp
        rows = clouds * N
        qkv = torch.randn(rows, 3 * C, device=dev)
        qp = torch.randn(rows, H, C, device=dev) * 0.2
        qb = torch.randn(rows, H, device=dev)
        E = torch.randn(clouds, N, N, C, device=dev)
        out = torch.empty(rows, C, device=dev)
        items = (Item * clouds)()
        for c in range(clouds):
            o = c * N
            items[c] = Item(qkv[o:].data_ptr(), qkv[o:, C:].data_ptr(), qkv[o:, 2 * C:].data_ptr(), qp[o:].data_ptr(), qb[o:].data_ptr(),
                            E[c].data_ptr(), out[o:].data_ptr(), N, N)
        lib = L.lib()
        ws = torch.empty(lib.geob200_attention_batched_workspace_bytes(items, clouds, H) + 1024, dtype=torch.uint8, device=dev)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        ts = []
        for i in range(13):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            L.check(lib.geob200_attention_batched(items, clouds, 3 * C, 3 * C, 3 * C, C, C, H, ws.data_ptr(), ws.numel(), st), 'attention')
            e1.record()
            e1.synchronize()
            if i >= 3:
                ts.append(e0.elapsed_time(e1))
        ts.sort()
        ms = ts[len(ts) // 2]
        e_bytes = float(clouds) * N * N * C * 4
        ach = e_bytes / (ms * 1e-3) / 1e9
        return {'kernel': 'self-attention layer: att_qk_kernel + att_stream_kernel (TMA-staged E stream) + att_pv_kernel', 'bound': 'hbm',
                'achieved': ach, 'peak': peak_hbm, 'unit': 'GB/s', 'frac': ach / peak_hbm, 'traffic': traffic.get('att_stream_bytes_per_launch'),
                'algorithmic_bytes_per_launch': e_bytes, 'ms_per_layer': ms, 'clouds': clouds, 'superpoints_per_cloud': N,
                'timing': 'CUDA events around the three launches of one layer (median of 10, L2 flushed), kernels alone on the GPU, after the timed regions',
                'note': 'achieved counts the E bytes only and divides by the time of ALL three launches; the streaming kernel alone moves '
                        'E at 5.35 TB/s = 0.81 of the peak (ncu, profiles/r02_top_kernels_ncu_selected.csv)'}
    except Exception as ex:
        return {'kernel': 'self-attention', 'bound': 'hbm', 'achieved': None, 'note': f'failed: {type(ex).__name__}: {ex}'}


def gse_contraction_roofline(dev, emb_mod, n_sp, clouds, peak_tf, peak_src, traffic):
    """Tensor roofline of the structure embedding IN ITS CONTRACTION FORM (tcgen05 3xFP16 kernel, GSE mode 3 -- the dense
    contraction north_star names), timed alone on a batch-sized problem after the timed regions: the default path does not run it
    any more (tabulated projections, roofline_gse_embed), the number stays in the line for comparison.  Same call sequence as
    tests/gse_table_check.py."""
    try:
        from geotransformer_b200 import functional as GF
        C = emb_mod.proj_d.out_features
        if C not in (128, 256):
            return None
        g = torch.Generator().manual_seed(11)
        pts = (torch.rand(clouds * n_sp, 3, generator=g) * 3.0).to(dev)
        rows = clouds * n_sp * n_sp
        d_all, a_all = torch.empty(rows, device=dev), torch.empty(rows, 3, device=dev)
        E = torch.empty(rows, C, device=dev)
        GF.gse_indices_batched(pts, [n_sp] * clouds, emb_mod.sigma_d, emb_mod.sigma_a, emb_mod.angle_k, d_all, a_all)
        wd, wa = emb_mod.proj_d.weight.detach(), emb_mod.proj_a.weight.detach()
        rest = (emb_mod.embedding.div_term, wd, wa, emb_mod.proj_d.bias.detach(), emb_mod.proj_a.bias.detach(), wd.t().contiguous(),
                wa.t().contiguous(), E)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        ts = []
        for i in range(6):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            GF.gse_embed_flat(d_all, a_all, rows, *rest, mode=3)
            e1.record()
            e1.synchronize()
            if i:
                ts.append(e0.elapsed_time(e1))
        ts.sort()
        ms = ts[len(ts) // 2]
        flops = 2.0 * rows * 4 * C * C
        ach = flops / (ms * 1e-3) / 1e12
        return {'kernel': f'gse_embed_f16_kernel<{C}> (structure embedding as a tcgen05 3xFP16 contraction; NOT on the default path)', 'bound': 'tensor',
                'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach / peak_tf, 'traffic': traffic.get('gse_embed_bytes_per_launch'),
                'ms_per_launch': ms, 'flops_per_launch': flops, 'clouds': clouds, 'superpoints_per_cloud': n_sp,
                'timing': 'CUDA events around the launch (median of 5, L2 flushed), kernel alone on the GPU, after the timed regions',
                'peak_source': f'{peak_src} bf16 dense BURST (MEASURED_PEAKS.json; the kernel is timed alone)'}
    except Exception as ex:
        return {'kernel': 'gse_embed_f16_kernel', 'bound': 'tensor', 'achieved': None, 'note': f'failed: {type(ex).__name__}: {ex}'}


def load_traffic():
    """per-launch DRAM traffic of the roofline kernels from the committed ncu --set full capture (profiles/r02_dram_traffic.json)"""
    p = os.path.join(ROOT, 'profiles', 'r02_dram_traffic.json')
    return json.load(open(p)) if os.path.exists(p) else {}


def make_inputs(workload, n_pairs, rank, world):
    from geotransformer_b200.synth import make_pair
    pairs = []
    from geotransformer_b200.distributed import pair_ids
    for pid in pair_ids(n_pairs, rank, world):
        p = make_pair(workload, pid)
        pairs.append({k: p[k] for k in ('ref_points', 'src_points', 'ref_feats', 'src_feats', 'transform')})
    return pairs


def cpu_threads():
    """Intra-op threads for the CPU reference path.  Measured on the B200 host (128 vCPU): the forward of one demo-size
    pair takes 1.3 s with 1 thread, 0.1 s with 16, 0.5 s with 64 and 116 s with 128 (oversubscription on the thousands of
    tiny ATen ops) -- so the baseline uses min(cores, 16), the fastest setting, and reports that number as `cores`."""
    return max(1, min(os.cpu_count() or 1, 16))


def _stats(xs):
    a = np.sort(np.asarray(xs, dtype=np.float64))
    q = lambda p: float(a[min(len(a) - 1, int(round(p * (len(a) - 1))))])
    return {'median': q(0.5), 'p10': q(0.1), 'p90': q(0.9), 'n': int(len(a))}


def gpu_eager_port(workload, n_pairs, device):
    """What a drop-in user of the reference sees today on this GPU (SURVEY.md 8d, engine/single_tester.py:52-58): collate on the
    host CPU (the reference runs it in DataLoader workers), then the model forward as EAGER torch ops on the GPU.
    /root/reference is not on the GPU box, so the forward is the pinned torch restatement (oracle/geo_oracle.py, bit-identical
    to the reference on CPU) executed with device tensors -- cuBLAS / ATen kernels, allow_tf32 off as in the reference.
    Returns a dict for the bench line (never raises)."""
    try:
        from geotransformer_b200.config import make_cfg
        from geotransformer_b200.model import create_model
        from geotransformer_b200.synth import make_pair, WORKLOADS
        from geotransformer_b200.weights import synthetic_state_dict
        from oracle import geo_oracle as G, collate_oracle, ref_ext
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
        cfg = make_cfg(WORKLOADS[workload][0])
        sd = {k: v.to(device) for k, v in synthetic_state_dict(create_model(cfg), 7351).items()}
        impl = ref_ext if ref_ext.available() else collate_oracle
        limits = cfg.neighbor_limits or [27, 75, 147, 157, 119][:cfg.backbone.num_stages]
        sync = (lambda: torch.cuda.synchronize(device)) if torch.device(device).type == 'cuda' else (lambda: None)
        t_col, t_fwd = [], []
        for i in range(n_pairs + 1):                    # first pair = warm-up (cuBLAS handles, allocator)
            pair = make_pair(workload, 2000 + i)
            t0 = time.perf_counter()
            data = G.collate_pair(pair, cfg, limits, impl=impl)
            t1 = time.perf_counter()
            data = {k: ([x.to(device) if isinstance(x, torch.Tensor) else x for x in v] if isinstance(v, list) else
                        (v.to(device) if isinstance(v, torch.Tensor) else v)) for k, v in data.items()}
            sync()
            t2 = time.perf_counter()
            with torch.no_grad(), torch.device(device):
                out = G.forward(sd, cfg, data)
                G.evaluate(cfg, out, data['transform'])
            sync()
            t3 = time.perf_counter()
            if i > 0:
                t_col.append(t1 - t0)
                t_fwd.append(t3 - t1)                   # H2D of the collated dict + forward + metrics
        tot = float(np.sum(t_col) + np.sum(t_fwd))
        return {'value': n_pairs / tot, 'unit': 'pairs/s', 'kind': 'gpu_eager_port',
                'forward_only_pairs_per_s': n_pairs / float(np.sum(t_fwd)),
                'collate_s': _stats(t_col), 'h2d_forward_metrics_s': _stats(t_fwd),
                'sample': f'{n_pairs} pair(s) of {workload} after 1 warm-up pair; host-CPU collate ({"reference C++" if impl is ref_ext else "C port"}, '
                          f'1 thread, in line) + eager torch forward of the pinned restatement on {device}, allow_tf32=False'}
    except Exception as ex:
        return {'value': None, 'unit': 'pairs/s', 'kind': 'gpu_eager_port', 'sample': f'failed: {type(ex).__name__}: {ex}'}


def cpu_reference_pairs_per_s(workload, n_pairs, threads, return_times=False):
    """The reference's CPU path: its own C++ collate ops (oracle/_ref) when built, else the plain-C port; the model forward is
    the torch-CPU restatement (a port, pinned bit-for-bit to the reference).  Returns (pairs/s, seconds, description)."""
    from geotransformer_b200.config import make_cfg
    from geotransformer_b200.model import create_model
    from geotransformer_b200.synth import make_pair, WORKLOADS
    from geotransformer_b200.weights import synthetic_state_dict
    from oracle import geo_oracle as G, collate_oracle, ref_ext
    torch.set_num_threads(threads)
    cfg = make_cfg(WORKLOADS[workload][0])
    sd = synthetic_state_dict(create_model(cfg), 7351)
    impl = ref_ext if ref_ext.available() else collate_oracle
    limits = cfg.neighbor_limits or [27, 75, 147, 157, 119][:cfg.backbone.num_stages]
    t_collate = t_fwd = 0.0
    per_pair = []
    for i in range(n_pairs):
        pair = make_pair(workload, 1000 + i)
        t0 = time.perf_counter()
        data = G.collate_pair(pair, cfg, limits, impl=impl)
        t1 = time.perf_counter()
        with torch.no_grad():
            out = G.forward(sd, cfg, data)
            G.evaluate(cfg, out, pair['transform'])
        t2 = time.perf_counter()
        t_collate += t1 - t0
        t_fwd += t2 - t1
        per_pair.append(t2 - t0)
    total = t_collate + t_fwd
    kind = 'reference C++ collate + port forward' if impl is ref_ext else 'port'
    desc = f'{n_pairs} pair(s) of {workload}: collate {t_collate:.1f}s + forward {t_fwd:.1f}s ({kind}; one reference search per table)'
    if return_times:
        return n_pairs / total, total, desc, per_pair, kind
    return n_pairs / total, total, desc


def step_shape(args):
    """(pairs per forward, forwards in flight, pairs per GPU and step) of the GPU arm for these flags"""
    batch = max(1, args.batch)
    lanes = max(1, args.streams if args.streams is not None else (2 if batch > 1 else 4))
    per_step = max(1, args.pairs_per_step if args.pairs_per_step is not None else (4 * batch * lanes if batch > 1 else lanes))
    return batch, lanes, per_step


def workload_config(args, world):
    """The STATIC description of the workload: identical in the GPU arm and in the --impl reference arm (which times a bounded
    sample of it per step, see its ``step_sample``); everything measured during the run goes into ``run_info`` instead."""
    from geotransformer_b200.config import make_cfg
    from geotransformer_b200.synth import WORKLOADS
    cfg_name, _, kw, _ = WORKLOADS[args.workload]
    batch, lanes, per_step = step_shape(args)
    return {'workload': args.workload, 'pairs_per_step_per_gpu': per_step, 'pairs_per_forward': batch, 'forwards_in_flight': lanes,
            'points_per_cloud': int(kw['n']), 'sinkhorn_iterations': make_cfg(cfg_name).model.num_sinkhorn_iterations,
            'parallelism': f'pairs sharded over {world} GPU(s), one all_gather of metric rows',
            'l2': 'a different pair every step; per-pair working set (~0.5 GB incl. 2x75 MB embeddings) exceeds the 126 MB L2',
            'weights': 'random init (synthetic_state_dict seed 7351)'}


def dump_outputs(out_dir, results):
    """What RegistrationEngine.register returned for the pairs of one step, stacked per field in pair order (float32 / float64)"""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {'estimated_transform': np.stack([r['estimated_transform'].numpy() for r in results]).astype(np.float32),
              'num_corr': np.array([r['num_corr'] for r in results], dtype=np.float64),
              'num_superpoints': np.array([r['num_superpoints'] for r in results], dtype=np.float64)}
    for name in ('PIR', 'IR', 'RRE', 'RTE', 'RMSE', 'RR'):
        arrays['metric_' + name] = np.array([r['metrics'][name] for r in results], dtype=np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def main():
    args = parse()
    rank, world, local = dist_env()
    assert world == args.gpus or world == 1, f'WORLD_SIZE={world} but --gpus {args.gpus}'

    if args.impl == 'reference':
        if rank != 0:
            return
        threads = cpu_threads()
        # bounded sample per step: 1 pair of the workload (~3 s of CPU work on 16 threads)
        steps, warm = args.steps, args.warmup
        for _ in range(warm):
            cpu_reference_pairs_per_s(args.workload, 1, threads)
        v, secs, desc, per_pair, kind = cpu_reference_pairs_per_s(args.workload, steps, threads, return_times=True)
        v1, _, desc1 = cpu_reference_pairs_per_s(args.workload, 1, 1)          # the same path on ONE thread, one pair
        line = {'metric': METRIC, 'value': v, 'unit': 'pairs/s', 'n_gpus': args.gpus, 'steps': steps, 'warmup': warm,
                'ms_per_step': 1000.0 * secs / steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
                'config': workload_config(args, args.gpus),
                'step_sample': f'each step of this arm is a BOUNDED SAMPLE of the configured step: 1 pair of the workload on the host cores '
                               f'(CPU path, rank 0 only; {steps} timed / {warm} warm-up pairs); the unit (pairs/s) is the same',
                'cpu_baseline': {'value': v, 'unit': 'pairs/s', 'cores': threads, 'kind': kind, 'sample': desc,
                                 'seconds_per_pair': _stats(per_pair),
                                 'one_thread': {'value': v1, 'unit': 'pairs/s', 'cores': 1, 'sample': desc1},
                                 'host_cpus': os.cpu_count(),
                                 'threads_note': 'min(cores, 16) intra-op threads is the fastest setting measured on the 128-vCPU host '
                                                 '(more threads oversubscribe the thousands of tiny ATen ops); the 1-thread number is printed beside it'},
                'e2e': {'value': v, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
                'gpu_launches': 0}
        print(json.dumps(line))
        return

    assert torch.cuda.is_available(), 'bench.py needs a GPU (the product has no CPU path)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        import torch.distributed as dist
        # NCCL may print its version banner on stdout (NCCL_DEBUG=VERSION): keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=dev)
            warm = torch.zeros(1, device=dev)
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    from geotransformer_b200 import functional as GF, _lib
    from geotransformer_b200.distributed import gather_metric_rows, max_over_ranks
    from geotransformer_b200.config import make_cfg
    from geotransformer_b200.model import create_model
    from geotransformer_b200.synth import WORKLOADS
    from geotransformer_b200.weights import synthetic_state_dict

    if args.gse_mode is not None:
        GF.GSE_MODE = args.gse_mode
    if args.linear_persistent is not None:
        _lib.lib().geob200_set_linear_persistent(int(args.linear_persistent))
    if args.attention_tma is not None:
        _lib.lib().geob200_set_attention_tma(int(args.attention_tma))
    cfg = make_cfg(WORKLOADS[args.workload][0])
    limits = cfg.neighbor_limits or [27, 75, 147, 157, 119][:cfg.backbone.num_stages]
    model = create_model(cfg)
    model.load_state_dict(synthetic_state_dict(model, 7351), strict=True)
    model = model.to(dev).eval()
    from geotransformer_b200.model import enable_native
    enable_native(model)

    from geotransformer_b200.engine import RegistrationEngine
    BATCH, LANES, S = step_shape(args)          # pairs per forward, forwards in flight, pairs per GPU and step
    W, K = args.warmup, args.steps
    pairs = make_inputs(args.workload, (W + K) * S, rank, world)
    # host staging (pinned) and device-resident copies: one pinned slab and one device slab per key, the pairs are views
    slab_h = {k: torch.from_numpy(np.stack([p[k] for p in pairs])).pin_memory() for k in pairs[0]}
    slab_d = {k: v.to(dev) for k, v in slab_h.items()}
    pinned = [{k: slab_h[k][i] for k in slab_h} for i in range(len(pairs))]
    resident = [{k: slab_d[k][i] for k in slab_d} for i in range(len(pairs))]
    h2d_bytes = sum(v.numel() * v.element_size() for v in pinned[0].values()) * S
    from geotransformer_b200.loss import Evaluator
    evaluator = Evaluator(cfg)          # PIR/IR/RRE/RTE/RMSE/RR on the device, inside the timed region (one launch per pair)
    engine = RegistrationEngine(model, cfg, limits, num_streams=LANES, device=dev, evaluator=evaluator, pin_cpu=True, batch_size=BATCH)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(source, n0, n, sink=None):
        """n steps of S pairs each (the engine keeps S pairs in flight and pulls the next pair as a stream frees up);
        CUDA events on the current stream, which the engine's streams fork from / join into"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = engine.register(source[n0 * S:(n0 + n) * S], start_event=e0)
        timed.results = res
        if sink is not None:
            sink.extend(res)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if os.environ.get('GEOB_BENCH_DEBUG'):
            print(f'[rank {rank}] {n} steps x {S} pairs: {ms:.1f} ms', file=sys.stderr, flush=True)
        per_rank = [ms]
        if world > 1:                     # after the timed region: every rank's own time, so that a straggler is attributable
            t = torch.tensor([ms], device=dev)
            gathered = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(gathered, t)
            per_rank = [float(g.item()) for g in gathered]
        timed.per_rank = per_rank
        return max_over_ranks(ms, dev, world)

    def segs():
        return torch.cuda.memory_stats(dev).get('segment.all.allocated', 0)

    # One large cached block per lane for torch's caching allocator to carve later requests from (its free lists are per stream,
    # the lanes allocate under their own streams): the timed pairs are not the warm-up pairs, and a batch a few percent larger than
    # any seen before regrows a scratch buffer -- without a cached block to split that is a cudaMalloc (a device-wide
    # synchronisation) inside the first timed region (reported below as cuda_mallocs).
    try:
        for lane_stream in engine.streams:
            with torch.cuda.stream(lane_stream):
                pool = torch.empty(6 << 30, dtype=torch.uint8, device=dev)
                del pool
        torch.cuda.synchronize()
    except Exception:                      # not enough free memory: keep going, the counter will show the mallocs
        pass
    timed(resident, 0, W)
    timed(pinned, 0, W)
    seg0 = segs()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib = _lib.lib()
    l0 = lib.geob200_launch_count()
    GF.EVENTS = {}
    ms_res = timed(resident, W, K)
    per_rank_res = timed.per_rank
    last_step = timed.results[-S:]
    mallocs_res = segs() - seg0
    launches = (lib.geob200_launch_count() - l0)
    events = GF.EVENTS
    GF.EVENTS = None
    results = []
    seg_a = segs()
    ms_e2e = timed(pinned, W, K, sink=results)
    per_rank_e2e = timed.per_rank
    mallocs_e2e = segs() - seg_a
    # roofline pass: the dominant kernel timed ALONE (one pair in flight, so no other stream shares the SMs), same workload
    solo = RegistrationEngine(model, cfg, limits, num_streams=1, device=dev, evaluator=evaluator, batch_size=BATCH)
    GF.EVENTS = {}
    barrier()
    n_solo = min(K * S, max(8, 2 * BATCH))
    lib.geob200_linear_profile_enable(1)          # CUDA events around every tcgen05 GEMM launch of these pairs
    solo.register(resident[W * S:W * S + n_solo])
    barrier()
    import ctypes
    cap = 400 * max(n_solo, 8)
    shp, gms = (ctypes.c_int64 * (3 * cap))(), (ctypes.c_float * cap)()
    n_gemm = int(lib.geob200_linear_profile_read(cap, shp, gms))
    lib.geob200_linear_profile_enable(0)
    gemm = [(int(shp[3 * i]), int(shp[3 * i + 1]), int(shp[3 * i + 2]), float(gms[i])) for i in range(n_gemm)]
    events_solo = GF.EVENTS
    GF.EVENTS = None
    solo.close()
    sampler.stop_flag = True
    engine.close()
    tf32_peak = measure_tf32_peak(dev) if rank == 0 else None

    # metric rows (RRE, RTE, nCorr, pair id, PIR, IR, RMSE, RR) gathered with ONE collective (SURVEY.md 8e)
    rows = []
    for j, out in enumerate(results):
        m = out['metrics']
        rows.append([m['RRE'], m['RTE'], float(out['num_corr']), float(rank + (W * S + j) * world), m['PIR'], m['IR'], m['RMSE'],
                     m['RR']])
    rows_t = torch.tensor(rows, dtype=torch.float32, device=dev)
    rows_t = gather_metric_rows(rows_t, world)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # roofline of the dominant kernel: structure-embedding contraction, 2*N^2*(1+k)*C^2 FLOPs per launch
    C = cfg.geotransformer.hidden_dim
    gse = events.get('gse_embed', [])
    gse_ms = [s.elapsed_time(e) for s, e in gse]
    gse_solo_ms = [s.elapsed_time(e) for s, e in events_solo.get('gse_embed', [])]
    n_c = [r['num_superpoints'][0] for r in results] + [r['num_superpoints'][1] for r in results]
    mean_n2 = float(np.mean([n * n for n in n_c])) if n_c else 0.0
    clouds_per_launch = 2 * BATCH if BATCH > 1 else 1          # batch mode: ONE structure-embedding launch covers all clouds of the batch
    flops = 2.0 * mean_n2 * 4 * C * C * clouds_per_launch
    peak_tf, peak_tf_sustained, peak_hbm, peak_src = load_peaks()
    traffic = load_traffic()
    avg_ms = float(np.mean(gse_solo_ms)) if gse_solo_ms else None
    achieved = flops / (avg_ms * 1e-3) / 1e12 if avg_ms else None
    avg_ms_concurrent = float(np.mean(gse_ms)) if gse_ms else None
    mode_name = {0: 'fp32 CUDA cores', 1: 'tcgen05 3xTF32', 2: 'tcgen05 1xTF32', 3: 'tcgen05 3xFP16 (fp32-accurate split)',
                 4: 'tcgen05 3xFP16 split, CTA-pair TMA multicast of B',
                 5: 'tabulated projections (4 lookups + 3 max + 1 add per row and channel; no contraction)'}[GF.GSE_MODE]
    common = {'avg_ms_per_launch': avg_ms, 'launches_timed': len(gse_solo_ms), 'clouds_per_launch': clouds_per_launch,
              'avg_ms_per_launch_with_other_streams_active': avg_ms_concurrent,
              'timing': 'CUDA events around the launch, one pair in flight (kernel alone on the GPU), same workload, after the timed regions',
              'share_of_gpu_time': (avg_ms / clouds_per_launch * 2.0) / (ms_res / (K * S)) if avg_ms else None, 'mode': mode_name}
    if GF.GSE_MODE == 5:
        # no contraction left: the kernel writes E once (rows x C fp32) and reads 16 B of indices per row from HBM; the node
        # reads (4 lookups x 6 B per channel and row) are served by L2 (hot part of the table: ~15 MB)
        rows = mean_n2 * clouds_per_launch
        e_bytes = rows * (C * 4 + 16)
        gbps = e_bytes / (avg_ms * 1e-3) / 1e9 if avg_ms else None
        roofline_gse = {'kernel': 'table_embed_kernel (structure embedding through tabulated projections, csrc/gse_table.cu)', 'bound': 'hbm',
                        'achieved': gbps, 'peak': peak_hbm, 'unit': 'GB/s', 'frac': (gbps / peak_hbm) if gbps else None, 'traffic': None,
                        'algorithmic_bytes_per_launch': e_bytes, 'l2_node_bytes_per_launch': rows * 4 * C * 6,
                        'l2_node_read_GBps': (rows * 4 * C * 6 / (avg_ms * 1e-3) / 1e9) if avg_ms else None,
                        'contraction_flops_replaced_per_launch': flops,
                        'peak_source': f'{peak_src} HBM copy bandwidth (MEASURED_PEAKS.json)',
                        'note': 'HBM roofline = the compulsory write of E; the kernel is bound by the L2 reads of the table nodes '
                                '(6 x the E bytes), see l2_node_read_GBps', **common}
    else:
        roofline_gse = {'kernel': 'gse_embed (structure-embedding contraction)', 'bound': 'tensor', 'achieved': achieved, 'peak': peak_tf,
                        'unit': 'TFLOP/s', 'frac': (achieved / peak_tf) if achieved else None, 'traffic': traffic.get('gse_embed_bytes_per_launch'),
                        'flops_per_launch': flops, 'peak_source': f'{peak_src} bf16 dense BURST (MEASURED_PEAKS.json; the kernel is timed alone)',
                        **common}

    # dominant kernel by share of the step's GPU time: linear_tc_kernel (every nn.Linear and the KPConv contraction; ~80 launches
    # per pair, shapes M=40 000..320, K=32..3840, N=32..1024).  ALGORITHMIC flops = 2*M*N*K of the fp32 product the reference
    # computes (the kernel executes 3 TF32 MMAs per product term for fp32 accuracy); times = CUDA events around each launch.
    g_flops = sum(2.0 * m * n * k for m, n, k, _ in gemm)
    g_ms = sum(t for _, _, _, t in gemm)
    g_bytes = sum(4.0 * (m * k + n * k + m * n) for m, n, k, _ in gemm)
    big = sorted(gemm, key=lambda r: -r[3])[:3]
    by_shape = {}
    for m, n, k, t in gemm:
        key = (n, k)
        e = by_shape.setdefault(key, [0, 0.0, 0.0, 0])
        e[0] += 1; e[1] += t; e[2] += 2.0 * m * n * k; e[3] = max(e[3], m)
    shape_table = [{'n': n, 'k': k, 'launches': c, 'max_m': mm, 'ms_per_pair': round(t / max(n_solo, 1), 4), 'tflops': round(fl / (t * 1e-3) / 1e12, 1)}
                   for (n, k), (c, t, fl, mm) in sorted(by_shape.items(), key=lambda kv: -kv[1][1])[:12]]
    roofline = {'kernel': 'linear_tc_kernel (tcgen05 3xTF32 GEMM: all nn.Linear + KPConv contraction)', 'bound': 'tensor',
                'achieved': (g_flops / (g_ms * 1e-3) / 1e12) if g_ms else None, 'peak': peak_tf, 'unit': 'TFLOP/s',
                'frac': (g_flops / (g_ms * 1e-3) / 1e12 / peak_tf) if g_ms else None,
                'traffic': traffic.get('linear_tc_bytes_per_launch'), 'traffic_note': traffic.get('note'),
                'algorithmic_bytes_per_launch': (g_bytes / n_gemm) if n_gemm else None,
                'tf32_dense_peak_measured': tf32_peak,
                'frac_of_3xtf32_ceiling': (g_flops / (g_ms * 1e-3) / 1e12 / (tf32_peak / 3.0)) if (g_ms and tf32_peak) else None,
                'launches_timed': n_gemm, 'launches_per_pair': n_gemm / max(n_solo, 1), 'ms_per_pair': g_ms / max(n_solo, 1),
                'flops_per_pair': g_flops / max(n_solo, 1), 'algorithmic_bytes_per_pair': g_bytes / max(n_solo, 1),
                'achieved_GBps': (g_bytes / (g_ms * 1e-3) / 1e9) if g_ms else None, 'hbm_peak_GBps': peak_hbm,
                'slowest_launches_m_n_k_ms': [[m, n, k, round(t, 4)] for m, n, k, t in big], 'time_by_weight_shape': shape_table,
                'share_of_gpu_time': (g_ms / max(n_solo, 1)) / (ms_res / (K * S)) if g_ms else None,
                'timing': 'CUDA events around every launch, one pair in flight (kernel alone on the GPU), same workload, after the timed regions',
                'note': 'the ~80 GEMMs of one forward (every nn.Linear + the KPConv contractions), each over the stacked rows of all pairs of the '
                        'batch; the wide / deep shapes run at 125-133 TFLOP/s (shared-memory-bandwidth ceiling of the 3xTF32 formulation, DESIGN.md 5a), '
                        'the narrow (N = 32, 64) and the M = 5 100 transformer shapes pull the family average down: see time_by_weight_shape; '
                        'share_of_gpu_time = its time per pair (kernel alone) / wall time per pair of the timed region',
                'peak_source': f'{peak_src} bf16 dense BURST (MEASURED_PEAKS.json; launches timed alone); tf32_dense_peak_measured = torch.matmul fp32 '
                               f'8192^3 with allow_tf32, best of 10, this run; the kernel executes 3 TF32 MMAs per product term'}

    roofline_att = None
    roofline_gse_tc = None
    if rank == 0 and C in (128, 256) and n_c:
        roofline_att = attention_roofline(dev, int(np.mean(n_c)), 2 * BATCH, C, cfg.geotransformer.num_heads, peak_hbm, traffic)
        if GF.GSE_MODE == 5:
            roofline_gse_tc = gse_contraction_roofline(dev, model.transformer.embedding, int(np.mean(n_c)), 2 * BATCH, peak_tf, peak_src, traffic)

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            threads = cpu_threads()
            cpu_reference_pairs_per_s(args.workload, 1, threads)              # warm-up pair (thread pool, allocator)
            v, secs, desc, per_pair, kind = cpu_reference_pairs_per_s(args.workload, 3, threads, return_times=True)
            v1, _, desc1 = cpu_reference_pairs_per_s(args.workload, 1, 1)
            cpu = {'value': v, 'unit': 'pairs/s', 'cores': threads, 'kind': kind, 'sample': desc, 'seconds_per_pair': _stats(per_pair),
                   'one_thread': {'value': v1, 'unit': 'pairs/s', 'cores': 1, 'sample': desc1}, 'host_cpus': os.cpu_count()}
        except Exception as ex:   # the baseline must never take the bench line down
            cpu = {'value': None, 'unit': 'pairs/s', 'cores': os.cpu_count(), 'kind': 'port', 'sample': f'failed: {ex}'}
    eager = gpu_eager_port(args.workload, 3, dev) if (world == 1 and not args.no_cpu_baseline) else None

    total_pairs = K * S * world
    line = {
        'metric': METRIC, 'value': total_pairs / (ms_res * 1e-3), 'unit': 'pairs/s', 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms_res / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': workload_config(args, world),
        'run_info': {'superpoints_per_cloud': int(np.mean(n_c)) if n_c else None,
                     'host_threads_pinned_to_gpu_numa_node': bool(engine.pinned_cpu)},
        'e2e': {'value': total_pairs / (ms_e2e * 1e-3), 'unit': 'pairs/s', 'ms_per_step': ms_e2e / K,
                'h2d_bytes_per_step': int(h2d_bytes), 'd2h_bytes_per_step': 96 * S},
        'gpu_launches': int(launches), 'gpu_launches_per_pair': launches / max(K * S, 1),
        'cuda_mallocs': {'timed_region_resident': int(mallocs_res), 'timed_region_e2e': int(mallocs_e2e)},
        'per_rank_ms': {'value': per_rank_res, 'e2e': per_rank_e2e}, 'roofline': roofline, 'roofline_gse_embed': roofline_gse, 'roofline_gse_contraction_tcgen05': roofline_gse_tc, 'roofline_attention': roofline_att, 'cpu_baseline': cpu, 'gpu_eager_port': eager, 'clocks': sampler.summary(),
        'quality': {'median_rre_deg': float(rows_t[:, 0].median()), 'median_rte': float(rows_t[:, 1].median()),
                    'mean_correspondences': float(rows_t[:, 2].mean()), 'pairs': int(rows_t.shape[0]),
                    'mean_PIR': float(rows_t[:, 4].nanmean()), 'mean_IR': float(rows_t[:, 5].nanmean()),
                    'registration_recall': float(rows_t[:, 7].mean()),
                    'note': 'random-init weights: the numbers show the metric path runs, not registration quality'},
    }
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
