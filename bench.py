#!/usr/bin/env python
"""bench.py — images/sec of one compression-aware training step (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--workload NAME] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is one pass of the hot path over one batch of synthetic input: teacher forward (eval mode),
weight + activation fake-quant, student forward, hard + distillation cross-entropy, backward (STE),
gradient all-reduce (N > 1), fused optimizer.  Nothing is skipped inside the timed region.

  value : images/s with the batch already resident in HBM (CUDA-graph replay of the device step),
          CUDA events on the launching stream, barrier + synchronize on both sides, max over ranks.
  e2e   : the same metric through the learner's public `train_step()` — pinned-host -> device copy of
          every batch inside the timed region and a device -> host read of the step's losses.
  roofline      : the conv stack (fwd+dgrad+wgrad), the one dense contraction: achieved TFLOP/s from
                  an instrumented eager step (CUDA events per launch group) vs the measured bf16 peak.
  roofline_hbm  : the activation fake-quant kernel, achieved GB/s (8 B/element) vs measured HBM peak.
  cpu_baseline  : the oracle step (oracle/step_oracle.py: un-fused PyTorch-CPU fp32, all host cores)
                  on a bounded sample of the same workload (TF 1.x cannot run in this image).
`--impl reference` times that CPU path alone (rank 0 only) and prints the same line.
`--dump-outputs DIR` writes what the last timed step handed its caller (see dump_outputs); inputs and initial weights are
seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'images_per_sec_compression_aware_training_step'

WORKLOADS = {
    # name: (net module, resnet_size, learner, flag overrides, description)
    'resnet50_uq8_dst_b256': ('resnet_at_ilsvrc12', 50, 'uniform', dict(batch_size=256, enbl_dst=True,
                              uql_weight_bits=8, uql_activation_bits=8, uql_use_buckets=True, uql_bucket_type='channel'),
                              'ResNet-50 v2 / synthetic 224x224x3, UniformQuantLearner W8(per-channel)A8 + distillation'),
    'resnet20_uq8_dst_b256': ('resnet_at_cifar10', 20, 'uniform', dict(batch_size=256, enbl_dst=True,
                              uql_weight_bits=8, uql_activation_bits=8, uql_use_buckets=True, uql_bucket_type='channel'),
                              'ResNet-20 v2 / synthetic CIFAR-10 32x32x3, UniformQuantLearner W8(per-channel)A8 + distillation'),
    'resnet50_ws50_dst_b256': ('resnet_at_ilsvrc12', 50, 'weight-sparse', dict(batch_size=256, enbl_dst=True,
                               ws_prune_ratio=0.5, ws_prune_ratio_prtl='uniform'),
                               'ResNet-50 v2 / synthetic 224x224x3, WeightSparseLearner 50% + distillation'),
    'resnet20_ws50_dst_b256': ('resnet_at_cifar10', 20, 'weight-sparse', dict(batch_size=256, enbl_dst=True,
                               ws_prune_ratio=0.5, ws_prune_ratio_prtl='uniform'),
                               'ResNet-20 v2 / synthetic CIFAR-10, WeightSparseLearner 50% + distillation'),
    'resnet50_nuq4_dst_b256': ('resnet_at_ilsvrc12', 50, 'non-uniform', dict(batch_size=256, enbl_dst=True,
                               nuql_weight_bits=4), 'ResNet-50 v2 / synthetic 224x224x3, NonUniformQuantLearner 4-bit codebook + distillation'),
    'mobilenet_cpg50_b256': ('mobilenet_at_ilsvrc12', 0, 'chn-pruned-gpu', dict(batch_size=256, cpg_prune_ratio=0.5),
                             'MobileNet-v1 / synthetic 224x224x3, ChannelPrunedGpuLearner masked step at 0.5 channel ratio'),
    'lenet_uq8_b128': ('lenet_at_cifar10', 0, 'uniform', dict(batch_size=128, uql_weight_bits=8),
                       'LeNet-5 / synthetic CIFAR-10, UniformQuantLearner 8-bit (configs[0], plumbing)'),
}
DEFAULT_WORKLOAD = os.environ.get('PF_BENCH_WORKLOAD', 'resnet50_uq8_dst_b256')    # the driver passes no --workload


def setup_flags(workload, batch_override=None, world=1):
    import importlib
    from pocketflow_b200.flags import FLAGS
    FLAGS.reset()
    net, size, learner, over, _ = WORKLOADS[workload]
    mod = importlib.import_module('pocketflow_b200.nets.' + net)
    if learner == 'uniform':
        importlib.import_module('pocketflow_b200.learners.uniform_quantization.learner')
    elif learner == 'weight-sparse':
        importlib.import_module('pocketflow_b200.learners.weight_sparsification.learner')
    elif learner == 'non-uniform':
        importlib.import_module('pocketflow_b200.learners.nonuniform_quantization.learner')
    elif learner == 'chn-pruned-gpu':
        importlib.import_module('pocketflow_b200.learners.channel_pruning_gpu.learner')
    importlib.import_module('pocketflow_b200.learners.distillation_helper')
    # each net module re-declares its own defaults (lrn_rate_init, loss_w_dcy, ...): re-apply them
    importlib.reload(importlib.import_module('pocketflow_b200.datasets.' +
                                             ('ilsvrc12_dataset' if 'ilsvrc12' in net else 'cifar10_dataset')))
    mod = importlib.reload(mod)
    if size:
        FLAGS.resnet_size = size
    FLAGS.learner = learner
    for k, v in over.items():
        setattr(FLAGS, k, v)
    if batch_override:
        FLAGS.batch_size = batch_override
    FLAGS.enbl_multi_gpu = world > 1
    FLAGS.summ_step = 10 ** 9
    FLAGS.save_step = 10 ** 9
    return mod


def conv_flops_per_image(ex):
    """2*M*N*K per conv/dense pass; fwd + wgrad + dgrad (no dgrad into the input images)."""
    fwd = dgrad = 0
    for op in ex.ops:
        if op.type in ('Conv2D', 'MatMul'):
            y = op.output
            k = op.vars['kernel']
            m = int(np.prod(y.shape[:-1]))
            f = 2.0 * m * k.numel
            fwd += f
            if op.inputs[0].op.type != 'Placeholder':
                dgrad += f
    n = ex.logits_t.shape[0]
    return fwd / n, (2 * fwd + dgrad) / n


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([c.strip() for c in out.stdout.strip().split(',')])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = [float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[4:8]) if v.lower().startswith('active')})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(self.rows)}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d['hbm_gbs'], d['bf16_tflops'], d.get('bf16_tflops_sustained', d['bf16_tflops']), 'measured'
    return 6650.0, 1590.0, 1400.0, 'fallback'


DUMP_LIMIT_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 16


def dump_outputs(out_dir, losses, state):
    """<out_dir>/loss.<term>.npy for every loss term of the step and <out_dir>/var.<variable>.npy for every model variable
    after it ('/' -> '.', ':' -> '_'), float32.  A variable larger than the per-variable share of DUMP_LIMIT_BYTES (at
    most DUMP_SAMPLE elements) is written as the 1-D sample of its flattened entries at sorted indices drawn by
    np.random.default_rng(0): the same entries in every run of the same workload."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {'loss.' + k: np.asarray(v, np.float32) for k, v in losses.items()}
    per_var = max(1, min(DUMP_SAMPLE, (DUMP_LIMIT_BYTES // 4 - len(arrays)) // max(len(state), 1)))
    for name, v in state.items():
        a = np.asarray(v, np.float32)
        if a.size > per_var:
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, per_var, replace=False))]
        arrays['var.' + name.replace('/', '.').replace(':', '_')] = a
    for n, a in arrays.items():
        np.save(os.path.join(out_dir, n + '.npy'), a)


def build_learner(workload, world, batch_override=None):
    mod = setup_flags(workload, batch_override, world)
    from pocketflow_b200.learners.learner_utils import create_learner
    lrn = create_learner(None, mod.ModelHelper())
    if hasattr(lrn, 'choose_channels'):
        # config 4 times the steady-state masked step: a SHORT run of the layer-wise channel selection (2 proximal +
        # 2 fine-tune iterations per layer instead of cpg_nb_iters_layer = 1000) yields the 50 % input-channel masks
        lrn.init_from_full()
        lrn.choose_channels(nb_iters_layer=2)
    return lrn


# ------------------------------------------------------------------------------ CPU reference arm
def host_threads():
    """Threads this process may actually use: min(affinity mask, cgroup CPU quota, 32).  The GPU boxes expose 128
    logical cores through the affinity mask while the container's CFS quota is a small fraction of that; 128 OpenMP
    threads spinning on a few cores' worth of quota made one oracle step take minutes."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:                      # cgroup v2: "<quota> <period>" or "max <period>"
            q, per = f.read().split()[:2]
            if q != 'max':
                n = min(n, max(1, int(int(q) / int(per))))
    except (OSError, ValueError):
        try:
            with open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us') as f, open('/sys/fs/cgroup/cpu/cpu.cfs_period_us') as g_:
                q, per = int(f.read()), int(g_.read())
                if q > 0:
                    n = min(n, max(1, q // per))
        except (OSError, ValueError):
            pass
    return max(1, min(n, 32))


def cpu_oracle_rate(workload, sample_batch, steps, threads, budget_s=30.0):
    """images/s of the un-fused PyTorch-CPU oracle step on a bounded sample (batch `sample_batch`): one warm-up
    step, then up to `steps` timed steps, fewer when they would not fit `budget_s` seconds (at least one).
    Returns (images/s, seconds per step, timed steps)."""
    import torch
    from oracle.step_oracle import StepOracle
    from pocketflow_b200 import graph as G
    from pocketflow_b200.flags import FLAGS
    torch.set_num_threads(threads)
    mod = setup_flags(workload, sample_batch, 1)
    net, size, learner, over, _ = WORKLOADS[workload]
    mh = mod.ModelHelper()
    from pocketflow_b200.learners.distillation_helper import DistillationHelper
    g = G.Graph()
    with g.as_default():
        with G.variable_scope('data'):
            it = mh.build_dataset_train()
            im, lab = it.get_next()
        tl = None
        if FLAGS.enbl_dst:
            with G.variable_scope('distilled_model'):
                tl = mh.forward_eval(im)
        with G.variable_scope('model'):
            out = mh.forward_train(im)
            tv = [v for v in g.variables.values() if v.name.startswith('model/') and v.trainable]
            loss, _ = mh.calc_loss(lab, out, tv)
            if tl is not None:
                loss += DistillationHelper.calc_loss(out, tl)
    wq = aq = None
    opt = dict(kind='momentum', slots={})
    if learner == 'uniform':
        from pocketflow_b200.learners.uniform_quantization.utils import UniformQuantization
        uq = UniformQuantization(g, FLAGS.uql_bucket_size, FLAGS.uql_use_buckets, FLAGS.uql_bucket_type)
        mm = uq.search_matmul_op(FLAGS.uql_quantize_all_layers)
        aa = uq.search_activation_op()
        uq.insert_quant_op_for_weights({o.name: FLAGS.uql_weight_bits for o in mm})
        uq.insert_quant_op_for_activations({o.name: FLAGS.uql_activation_bits for o in aa})
        wq, aq = uq.weight_quant_spec(), uq.act_quant_spec()
        opt = dict(kind='adam', slots={})
    sops = [o for o in g.ops if 'distilled' not in o.name]
    teacher = None
    tstate = None
    rng = np.random.default_rng(1)
    if tl is not None:
        tops = [o for o in g.ops if 'distilled' in o.name or o.type == 'Placeholder']
        teacher = StepOracle(tops, tl, im)
        tstate = {v.name: v.initializer(rng, v.shape) for v in g.variables.values() if v.name.startswith('distilled')}
    orc = StepOracle(sops, out, im, lab, loss, wq, aq, teacher)
    state = {v.name: v.initializer(rng, v.shape) for v in g.variables.values() if v.name.startswith('model/')}
    masks = None
    images, labels = it.next_batch()
    img, lb = images.numpy(), labels.numpy()
    tw = time.perf_counter()
    orc.step(state, img, lb, opt, 1e-3, teacher_state=tstate, masks=masks)       # warm-up
    tw = time.perf_counter() - tw
    steps = max(1, min(steps, int(budget_s / max(tw, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps):
        _, state, _ = orc.step(state, img, lb, opt, 1e-3, teacher_state=tstate, masks=masks)
    dt = time.perf_counter() - t0
    return sample_batch * steps / dt, dt / steps, steps


def cpu_oracle_rate_bounded(workload, sample_batch, steps, threads, budget_s, hard_timeout_s):
    """cpu_oracle_rate in a child process with a hard wall-clock limit (a contended host must not stall the bench).
    Returns (images/s | None, seconds per step | None, timed steps, note)."""
    import subprocess
    cmd = [sys.executable, os.path.abspath(__file__), '--cpu-leg', workload, str(sample_batch), str(steps), str(threads),
           str(budget_s)]
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=hard_timeout_s, env=dict(os.environ, CUDA_VISIBLE_DEVICES=''))
        for ln in reversed(out.stdout.strip().split('\n')):
            if ln.startswith('{'):
                r = json.loads(ln)
                return r['rate'], r['sec'], r['steps'], 'ok'
        return None, None, 0, 'cpu leg failed: %s' % out.stderr.strip().split('\n')[-1][:200]
    except subprocess.TimeoutExpired:
        return None, None, 0, 'cpu leg exceeded %d s of wall clock on this host (warm-up + 1 step of batch %d)' % (
            hard_timeout_s, sample_batch)


def cpu_sample_batch(args):
    """Mini-batch of the CPU legs: the workload's own batch where a step fits the time budget (CIFAR / LeNet), 16 for the
    224x224 networks (a batch-2 sample would handicap the CPU: its GEMMs do not fill 16 cores)."""
    if args.cpu_batch:
        return args.cpu_batch
    full = WORKLOADS[args.workload][3]['batch_size']
    return min(full, 16 if ('resnet50' in args.workload or 'mobilenet' in args.workload) else 64)


def kernel_source_stamp():
    """sha1 over the conv kernel sources: profiles/*_conv_traffic.json carries the stamp of the binary it was measured
    with, and a stale file is refused (the GPU box has no .git to ask for a commit id)."""
    import hashlib
    h = hashlib.sha1()
    d = os.path.join(ROOT, 'pocketflow_b200', 'csrc')
    for fn in ('pf_conv_tc.cu', 'pf_conv_tma.cu', 'pf_conv_tc.cuh', 'pf_tma.cuh', 'pf_tc_common.cuh'):
        with open(os.path.join(d, fn), 'rb') as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def run_reference(args, rank):
    if rank != 0:
        return
    cores = host_threads()
    sb = cpu_sample_batch(args)
    rate, sec, steps, note = cpu_oracle_rate_bounded(args.workload, sb, args.steps, cores, 150.0, 290)
    if rate is None:
        emit({'impl': 'reference', 'unavailable': note})
        return
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': rate, 'unit': 'images/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': 1, 'steps_requested': args.steps, 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': args.workload, 'description': WORKLOADS[args.workload][4], 'sample_batch': sb,
                   'note': 'TensorFlow 1.x (the reference runtime) is not installable in this image; this is the '
                           'oracle restatement of the reference step, un-fused, PyTorch-CPU fp32'},
        'cpu_baseline': {'value': rate, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d steps of batch %d (bounded sample of the batch-%d workload)' % (
                             steps, sb, WORKLOADS[args.workload][3]['batch_size'])},
        'e2e': {'value': rate, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


# ------------------------------------------------------------------------------ GPU arm
_RESULT_FD = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Native libraries (NCCL's version banner, ...) write to file
    descriptor 1 directly, so fd 1 is pointed at stderr for the whole run and the result line goes to a saved copy
    of the original stdout."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + '\n').encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    if len(sys.argv) >= 7 and sys.argv[1] == '--cpu-leg':
        wl, sb, st, th, bud = sys.argv[2], int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5]), float(sys.argv[6])
        rate, sec, nst = cpu_oracle_rate(wl, sb, st, th, bud)
        print(json.dumps({'rate': rate, 'sec': sec, 'steps': nst}), flush=True)
        return
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=None, help='override the per-GPU batch (smoke runs only)')
    ap.add_argument('--cpu-batch', type=int, default=None)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the losses of the last timed step and the model variables after it to DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to --impl b200')
    quiet_stdout()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3
    os.environ.setdefault('NCCL_DEBUG', 'WARN')      # keep NCCL's chatter off stdout: ONE JSON line
    os.environ.setdefault('NCCL_DEBUG_FILE', '/tmp/pf_nccl_%h_%p.log')   # (the version banner goes to a file)
    import torch
    import torch.distributed as dist
    from pocketflow_b200 import ops
    from pocketflow_b200.flags import FLAGS
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local_rank)
    lrn = build_learner(args.workload, world, args.batch)
    ex = lrn.sess_train
    B = FLAGS.batch_size
    allreduce = lrn.grad_allreduce()
    if world > 1:
        from pocketflow_b200.utils.multi_gpu_wrapper import MultiGpuWrapper as mgw
        mgw.broadcast_global_variables([ex.store.P, ex.store.O])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    lr = lrn.lrn_rate(0)
    lrn.iterator_train.prefill()      # synthetic batches live in pinned host memory before any timing
    # ---- untimed: one eager step (counts launches), capture, warm-up
    lrn.feed(ex, lrn.iterator_train)
    ops.launch_count_reset()
    ex.run_step(lr, allreduce)
    torch.cuda.synchronize()
    launches_per_step = ops.launch_count()
    graph_ok = False
    if not args.no_graph:
        try:
            ex.capture(allreduce)
            graph_ok = True
        except Exception as e:  # noqa: BLE001  (e.g. a collective that refuses capture)
            print('[bench] CUDA-graph capture failed (%s); running eagerly' % e, file=sys.stderr)
            ex._graph = None
    for _ in range(args.warmup):
        ex.run_step(lr, allreduce)
    # ---- timed region 1: device-resident batch
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        ex.run_step(lr, allreduce)
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device='cuda')
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    # ---- timed region 2: end to end through the public API (H2D of every batch, D2H of the losses)
    for _ in range(2):
        lrn.train_step()
        ex.fetch_losses()
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(args.steps):
        lrn.train_step()
        losses = ex.fetch_losses()
    t1.record()
    barrier()
    sampler.stop_flag = True
    ms2 = torch.tensor([t0.elapsed_time(t1)], device='cuda')
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    e2e_ms = float(ms2.item())
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, losses, ex.store.state_dict())
    # ---- instrumented eager step: per-group device time for the roofline
    hbm_peak, tf_peak, tf_sust, peak_kind = peaks()
    prof = ex.profile_step(lr, allreduce)
    fwd_pi, train_pi = conv_flops_per_image(ex)
    conv_ms = sum(prof.get(k, 0.0) for k in ('conv_fwd', 'conv_dgrad', 'conv_wgrad', 'conv_prep'))
    teacher_fwd = fwd_pi if ex.teacher is not None else 0.0
    conv_flops = (train_pi + teacher_fwd) * B
    conv_tflops = conv_flops / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
    step_ms_eager = sum(prof.values())
    # HBM-bound companion: the BN(+ReLU)(+activation fake-quant) apply pass — 4 B per element read (fp32 conv output)
    # plus what it writes: split-bf16 operand planes or fp32 (4 B), ONE bf16 plane of quantizer levels (2 B, + the
    # per-pixel channel sums), the fp32 copy as well where another consumer needs it; teacher + student
    aq_bytes = 0
    for e in ([ex] + ([ex.teacher] if ex.teacher is not None else [])):
        for op in e.ops:
            if op.type != 'FusedBatchNorm':
                continue
            n_el = op.output.numel
            lv = getattr(e, 'act_lv', {}).get(op)
            has_planes = op in getattr(e, 'xplanes', {})
            out_b = (2 if lv is not None else 4) if has_planes else 4
            if has_planes and e.bn_need_f32.get(op, False):
                out_b += 4
            aq_bytes += n_el * (4 + out_b) + (4 * n_el // op.output.shape[-1] * lv['nseg'] if lv is not None else 0)
    aq_elems = aq_bytes / 8.0
    aq_ms = prof.get('bn_apply', 0.0)
    conv_traffic, traffic_src = None, 'no ncu launch list of this binary under profiles/ (run tools/gpu_launchlist.sh)'
    try:
        tj = json.load(open(os.path.join(ROOT, 'profiles', 'r2_ncu_conv_traffic.json')))
        if tj.get('workload') != args.workload or B != tj.get('batch'):
            traffic_src = 'profiles/r2_ncu_conv_traffic.json is for another workload / batch'
        elif tj.get('kernel_source_stamp') != kernel_source_stamp():
            traffic_src = 'profiles/r2_ncu_conv_traffic.json is stale (kernel sources changed since it was measured)'
        else:
            conv_traffic = tj['conv_dram_bytes_per_step']
            traffic_src = 'ncu launch list of this binary (kernel source stamp %s), profiles/r2_ncu_conv_traffic.json' % tj['kernel_source_stamp']
    except Exception:  # noqa: BLE001
        pass
    # MMA multiplicity per pass (tensor-core work issued per algorithmic product)
    n_lv_w = len(getattr(ex, 'w_lv', {}))
    n_lv_a = len(getattr(ex, 'act_lv', {}))
    n_tc = len(ex.tc)
    if rank == 0:
        value = B * world * args.steps / (ms_total * 1e-3)
        e2e_value = B * world * args.steps / (e2e_ms * 1e-3)
        line = {
            'metric': METRIC, 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': args.workload, 'description': WORKLOADS[args.workload][4],
                       'batch_per_gpu': B, 'global_batch': B * world, 'parallelism': 'dp%d' % world,
                       'conv_path': ('tcgen05 + TMEM, persistent warp-specialised kernels, operands fed by TMA (im2col-mode '
                                     'tensor maps for the NHWC operand, tiled maps for weights / dy) where channel counts are '
                                     'multiples of 64, cp.async elsewhere: %d of %d conv/dense layers (+ the stem through '
                                     'space-to-depth planes); exact-fp32 CUDA-core kernels for the rest.  MMAs per k-slice: '
                                     'student fwd 1 on %d layers (integer quantizer levels x levels, exact in bf16; 3 on the '
                                     'others), wgrad 2 on %d layers (levels x split-bf16 dy), dgrad 3, teacher fwd 3 '
                                     '(split-bf16 x split-bf16 = fp32-equivalent product)'
                                     % (n_tc, sum(1 for o in ex.ops if o.type in ('Conv2D', 'MatMul')), n_lv_w, n_lv_a))
                       if ex.tc or ex.im2col else 'fp32 CUDA-core implicit GEMM (pf_conv.cu)',
                       'l2': 'per-step working set (GBs of activations) >> 126 MB L2; no explicit flush',
                       'cuda_graph': graph_ok,
                       'input_pipeline': 'e2e: batch i+1 is copied host->device (pinned memory, copy stream) while step i '
                                         'runs, then moved into the graph input buffers device-to-device; one H2D per step'},
            'e2e': {'value': e2e_value, 'unit': 'images/s', 'h2d_bytes_per_step': int(lrn.h2d_bytes),
                    'd2h_bytes_per_step': int(getattr(ex, 'last_d2h_bytes', 0)), 'ms_per_step': e2e_ms / args.steps},
            'gpu_launches': int(launches_per_step * args.steps),
            'launches_per_step': int(launches_per_step),
            'roofline': {'bound': 'tensor',
                         'kernel': 'conv stack: conv_tma_kernel (fwd, dgrad) + conv_tma_wgrad_kernel (+ conv_tc_persist_kernel for '
                                   'the stem and strided dgrad)',
                         'achieved': conv_tflops, 'peak': tf_sust, 'unit': 'TFLOP/s',
                         'frac': conv_tflops / tf_sust, 'traffic': conv_traffic,
                         'traffic_source': traffic_src,
                         'traffic_note': 'achieved counts ALGORITHMIC flops (2*M*N*K per conv pass: student fwd, teacher fwd, '
                                         'dgrad, wgrad) over the conv kernels\' summed device time in ONE EAGER INSTRUMENTED '
                                         'step (CUDA events per launch group; `value` comes from the graph replay); the tensor '
                                         'cores issue 1 / 3 / 3 / 2 MMAs per product on those passes (9 units per 4 passes '
                                         'against 12 for all-split-bf16), so frac <= 4/9 by construction',
                         'peak_kind': peak_kind + ' bf16 sustained',
                         'flops_per_step': conv_flops, 'ms_per_step': conv_ms,
                         'share_of_step': conv_ms / step_ms_eager if step_ms_eager else None},
            'roofline_hbm': {'bound': 'hbm', 'kernel': 'bn_apply_kernel / bn_apply_levels_kernel (BN + ReLU + activation fake-quant -> operand planes / levels)',
                             'achieved': (8.0 * aq_elems / (aq_ms * 1e-3) / 1e9) if aq_ms > 0 else None,
                             'peak': hbm_peak, 'unit': 'GB/s',
                             'frac': (8.0 * aq_elems / (aq_ms * 1e-3) / 1e9 / hbm_peak) if aq_ms > 0 else None,
                             'traffic': None, 'peak_kind': peak_kind, 'bytes_per_step': int(aq_bytes), 'ms_per_step': aq_ms,
                             'note': 'algorithmic bytes: 4 B/element read + 4 B (split planes or fp32) or 2 B (one plane of '
                                     'quantizer levels) written'},
            'step_breakdown_ms': {k: round(v, 4) for k, v in sorted(prof.items())},
            'losses_last_step': {k: float(v) for k, v in losses.items()},
            'clocks': sampler.summary(),
        }
        if not args.no_cpu_baseline and world == 1:
            cores = host_threads()
            sb = cpu_sample_batch(args)
            try:
                rate, sec, nst, note = cpu_oracle_rate_bounded(args.workload, sb, 2, cores, 30.0, 150)
                line['cpu_baseline'] = {'value': rate, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                                        'sample': ('%d step(s) of batch %d of the same graph (bounded sample, %.1f s '
                                                   'per step), oracle/step_oracle.py' % (nst, sb, sec)) if rate else note}
            except Exception as e:  # noqa: BLE001
                line['cpu_baseline'] = {'value': None, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                                        'sample': 'failed: %s' % e}
        emit(line)
    if world > 1:
        dist.barrier()


if __name__ == '__main__':
    main()
