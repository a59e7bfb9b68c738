"""Bucketed codebooks (--nuql_use_buckets) on ResNet-50's quantized kernels: CUDA-event timings of

  * the weight-quant phase (per-bucket min/max + codebook quantize) per-layer vs 'channel' vs 'split'-256,
  * the codebook gradient (cluster / both modes) and the quantile init, for each of the three,
  * ms/step of the resnet50_nuq4_dst_b256 learner with and without --nuql_use_buckets --nuql_bucket_type channel,
    the two learners alive side by side and their timed windows alternated,

at 4 and 8 bits, with algorithmic bytes over time against the HBM data-sheet peak (7.7 TB/s).  The 94 MB of ResNet-50
kernels fit the 126 MB L2, as they do inside the training step: the phase numbers are L2-resident rates, like the step's.

  python tools/bench_nuq_buckets.py --out profiles/bench_nuq_buckets.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pocketflow_b200 import graph as G  # noqa: E402
from pocketflow_b200 import ops  # noqa: E402
from pocketflow_b200.flags import FLAGS  # noqa: E402

HBM_PEAK = 7.7e12


def card():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm',
                              '--format=csv,noheader'], capture_output=True, text=True, timeout=10)
        if out.returncode == 0:
            name, power, clk = [c.strip() for c in out.stdout.strip().split(',')]
            info.update(name=name, power_limit=power, sm_max_clock=clk)
    except (OSError, ValueError, subprocess.SubprocessError):
        info['power_limit'] = 'unavailable'
    return info


def resnet50_kernel_shapes():
    """shapes of the kernels the non-uniform learner quantizes on ResNet-50 (first and last layer excluded)"""
    import bench
    mod = bench.setup_flags('resnet50_nuq4_dst_b256', 2)
    from pocketflow_b200.learners.nonuniform_quantization.utils import NonUniformQuantization
    mh = mod.ModelHelper()
    g = G.Graph()
    with g.as_default():
        with G.variable_scope('data'):
            im, _ = mh.build_dataset_train().get_next()
        with G.variable_scope('model'):
            mh.forward_train(im)
            nq = NonUniformQuantization(g, 256, False, 'quantile', 'split')
            shapes = [tuple(op.vars['kernel'].shape) for op in nq.search_matmul_op(False)]
    FLAGS.reset()
    return shapes


def timed(fn, iters, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def phase_rows(shapes, bits, iters):
    rng = np.random.RandomState(bits)
    srcs = [torch.from_numpy((rng.randn(*s) * np.sqrt(2.0 / max(1, int(np.prod(s[:-1]))))).astype(np.float32)).cuda()
            for s in shapes]
    dsts = [torch.empty_like(s) for s in srcs]
    grads = [torch.randn_like(s) for s in srcs]
    numel = sum(s.numel() for s in srcs)
    rows = []
    for mode, btype in (('per-layer', None), ('channel', 'channel'), ('split-256', 'split')):
        use_b = btype is not None
        sizes = [(1 << bits) * (ops.nuq_bucket_layout(s.shape, btype, 256)[0] if use_b else 1) for s in srcs]
        offs = np.concatenate([[0], np.cumsum([(n + 3) // 4 * 4 for n in sizes])]).astype(np.int64)
        base = torch.zeros(int(offs[-1]) + 4, dtype=torch.float32, device='cuda')
        views = [base[o:o + n] for o, n in zip(offs, sizes)]
        if use_b:
            views = [v.view(1 << bits, -1) for v in views]
        gbase = torch.zeros_like(base)
        kw = dict(use_buckets=True, bucket_type=btype, bucket_size=256) if use_b else {}
        q = ops.CodebookWeightQuantizer(srcs, dsts, bits, cluster_views=views, cluster_base=base, **kw)
        qi = ops.CodebookWeightQuantizer(srcs, dsts, bits, keep_index=True, cluster_views=views, cluster_base=base, **kw)
        t_init = timed(q.quantile_init, 3, warmup=1)
        t_fwd = timed(q.forward, iters)
        qi.forward()
        t_grad = timed(lambda: qi.cluster_grad(grads, gbase), iters)
        cb = 4 * sum(sizes)
        nb = sum(int(s['ncols']) for s in q.uq.segs)
        # algorithmic bytes: min/max reads w; quantize reads w, writes qw (+ the codebooks); the gradient reads g and
        # the uint8 index once and writes the codebook gradients
        fwd_bytes = 12 * numel + cb
        grad_bytes = 5 * numel + cb
        rows.append(dict(bits=bits, mode=mode, buckets=nb, codebook_bytes=cb,
                         quant_phase_ms=t_fwd, quant_phase_bytes=fwd_bytes,
                         quant_phase_share_of_hbm_peak=fwd_bytes / (t_fwd * 1e-3) / HBM_PEAK,
                         cluster_grad_ms=t_grad, cluster_grad_bytes=grad_bytes,
                         cluster_grad_share_of_hbm_peak=grad_bytes / (t_grad * 1e-3) / HBM_PEAK,
                         quantile_init_ms=t_init))
        print('[nuq-buckets] %d bits %-9s quant %.3f ms  grad %.3f ms  init %.2f ms' % (bits, mode, t_fwd, t_grad, t_init),
              file=sys.stderr)
        del q, qi, base, gbase, views
    return numel, rows


def step_rows(batch, steps, warmup, rounds):
    import bench
    from pocketflow_b200.learners.learner_utils import create_learner
    lrns = {}
    for name, over in (('per-layer', {}), ('channel', dict(nuql_use_buckets=True, nuql_bucket_type='channel'))):
        mod = bench.setup_flags('resnet50_nuq4_dst_b256', batch)
        for k, v in over.items():
            setattr(FLAGS, k, v)
        lrn = create_learner(None, mod.ModelHelper())
        ex = lrn.sess_train
        lrn.iterator_train.prefill()
        allreduce = lrn.grad_allreduce()
        lrn.feed(ex, lrn.iterator_train)
        ex.run_step(lrn.lrn_rate(0), allreduce)
        ex.capture(allreduce)
        for _ in range(warmup):
            ex.run_step(lrn.lrn_rate(0), allreduce)
        torch.cuda.synchronize()
        lrns[name] = lrn
        print('[nuq-buckets] built %s learner, %.1f GB allocated' % (name, torch.cuda.memory_allocated() / 2 ** 30),
              file=sys.stderr)
    ms = {k: [] for k in lrns}
    for _ in range(rounds):
        for name, lrn in lrns.items():
            ex = lrn.sess_train
            ms[name].append(timed(lambda: ex.run_step(lrn.lrn_rate(0), lrn.grad_allreduce()), steps, warmup=2))
    return {k: dict(ms_per_step=v, median=float(np.median(v))) for k, v in ms.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--batch', type=int, default=256)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--rounds', type=int, default=4)
    ap.add_argument('--no-step', action='store_true')
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_nuq_buckets.py measures the device: no CUDA device found')
    torch.cuda.set_device(0)
    t0 = time.time()
    result = dict(tool='tools/bench_nuq_buckets.py', card=card(), hbm_peak_bytes_per_s=HBM_PEAK,
                  working_set='ResNet-50 quantized kernels (L2-resident, as in the training step)')
    shapes = resnet50_kernel_shapes()
    result['kernels'] = len(shapes)
    result['phases'] = []
    for bits in (4, 8):
        numel, rows = phase_rows(shapes, bits, args.iters)
        result['weights'] = numel
        result['phases'] += rows
    if not args.no_step:
        result['step'] = dict(workload='resnet50_nuq4_dst_b256', batch=args.batch, steps_per_window=args.steps,
                              rounds=args.rounds, **step_rows(args.batch, args.steps, args.warmup, args.rounds))
        s = result['step']
        result['step']['channel_over_per_layer'] = s['channel']['median'] / s['per-layer']['median']
    result['card_after'] = card()
    result['wall_s'] = time.time() - t0
    txt = json.dumps(result, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(txt)


if __name__ == '__main__':
    main()
