"""Bucketed codebooks (--nuql_use_buckets) on the device: pf_nuq_bucket_weight_quant / _quantile_init / _cluster_grad
against the numpy oracle (tests/nuq_bucket_oracle.py), then the non-uniform learner with split and channel buckets in
its three optimisation modes against the step oracle, on the tensor-core path (ResNet-50, MobileNet), through save /
--exec_mode eval in both checkpoint formats, and across a bit-width change."""
import numpy as np
import pytest
import torch

import nuq_bucket_oracle as B
from oracle import step_oracle
from oracle.step_oracle import StepOracle
from pocketflow_b200 import ops
from pocketflow_b200.flags import FLAGS

pytestmark = pytest.mark.gpu
F32 = np.float32
DEV = 'cuda:0'


def rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-30)


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def he(rng, shape):
    fan_in = int(np.prod(shape[:-1])) if len(shape) > 1 else 1
    return (rng.randn(*shape) * np.sqrt(2.0 / fan_in)).astype(F32)


# conv, dense, depthwise, ncols not a multiple of any tile width (1000, 130), numel % bucket_size != 0, tiny tensors
SHAPES = [(3, 3, 16, 32), (1, 1, 64, 1000), (3, 3, 32, 1), (5, 5, 3, 7), (64, 10), (3, 3, 128, 130), (7,)]


def quantizer(ws, bits, bucket_type, bucket_size, keep_index=True, gap=0):
    """codebook tables as [k, ncols] views of one flat buffer (like the parameter store), `gap` floats between them"""
    src = [cu(w) for w in ws]
    dst = [torch.empty_like(s) for s in src]
    sizes, offs, tot = [], [], 16
    for w in ws:
        ncols, _, _ = ops.nuq_bucket_layout(w.shape, bucket_type, bucket_size)
        sizes.append((1 << bits, ncols))
        offs.append(tot)
        tot += ((1 << bits) * ncols + 3) // 4 * 4 + gap             # views 16-byte aligned, like the parameter store
    base = torch.zeros(tot + 16, dtype=torch.float32, device=DEV)
    views = [base[o:o + k * n].view(k, n) for o, (k, n) in zip(offs, sizes)]
    q = ops.CodebookWeightQuantizer(src, dst, bits, keep_index=keep_index, cluster_views=views, cluster_base=base,
                                    use_buckets=True, bucket_type=bucket_type, bucket_size=bucket_size)
    return q, src, dst, base, views, offs


@pytest.mark.parametrize('bucket_type,bucket_size', [('channel', 256), ('split', 256), ('split', 100)])
@pytest.mark.parametrize('bits', [1, 2, 3, 4, 5, 6, 7, 8])
def test_bucket_quantile_init_and_quantize_bit_exact(bucket_type, bucket_size, bits):
    rng = np.random.RandomState(bits * 10 + len(bucket_type) + bucket_size)
    ws = [he(rng, s) for s in SHAPES]
    ws[3][..., 2] = 0.25                                                 # a constant bucket (alpha = 1e-10)
    ws[4] = (rng.randint(-3, 4, size=ws[4].shape) * 0.25).astype(F32)     # exact ties
    q, src, dst, base, views, _ = quantizer(ws, bits, bucket_type, bucket_size)
    q.quantile_init()
    q.forward()
    idx = q.idx.cpu().numpy()
    for i, w in enumerate(ws):
        rq, rc, ridx, _, _ = B.nonuniform_bucket_quantize(w, bits, bucket_type, bucket_size)
        assert np.array_equal(views[i].cpu().numpy(), rc), 'codebooks %d %s' % (i, w.shape)
        assert np.array_equal(dst[i].cpu().numpy(), rq), 'quantized %d %s' % (i, w.shape)
        o = q.idx_offsets[i]
        assert np.array_equal(idx[o:o + w.size], ridx.reshape(-1)[:w.size].astype(np.uint8)), 'index %d' % i
    assert q.bucket_storage_bits() == B.bucket_storage_bits([w.shape for w in ws], bucket_type, bucket_size)


@pytest.mark.parametrize('bits', [2, 4, 8])
def test_depthwise_channel_bucket_is_the_per_layer_codebook(bits):
    """[3, 3, C, 1] in channel mode is ONE bucket: the same bits as the per-layer quantizer"""
    rng = np.random.RandomState(bits)
    ws = [he(rng, (3, 3, 64, 1)), he(rng, (3, 3, 1024, 1))]
    qb, _, dst_b, _, views, _ = quantizer(ws, bits, 'channel', 256)
    qb.quantile_init()
    qb.forward()
    src = [cu(w) for w in ws]
    dst_l = [torch.empty_like(s) for s in src]
    ql = ops.CodebookWeightQuantizer(src, dst_l, bits)
    ql.quantile_init()
    ql.forward()
    for i in range(len(ws)):
        assert np.array_equal(views[i].cpu().numpy()[:, 0], ql.clusters.cpu().numpy()[i, :1 << bits])
        assert np.array_equal(dst_b[i].cpu().numpy(), dst_l[i].cpu().numpy())


@pytest.mark.parametrize('bucket_type,bucket_size', [('channel', 256), ('split', 256), ('split', 100)])
@pytest.mark.parametrize('bits', [2, 4, 8])
def test_bucket_codebook_gradient(bucket_type, bucket_size, bits):
    """dL/dc[j, b] = alpha_b * sum over the bucket's real rows with idx = j, within the per-layer test's bar; nothing
    written outside the codebooks; a second run is bit-identical"""
    rng = np.random.RandomState(20 + bits)
    shapes = SHAPES + [(3, 3, 512, 64)]                                  # 4608 rows per channel bucket: row-split tiles
    ws = [he(rng, s) for s in shapes]
    q, src, dst, base, views, offs = quantizer(ws, bits, bucket_type, bucket_size, gap=4)
    q.quantile_init()
    q.forward()
    gs = [rng.randn(*s).astype(F32) for s in shapes]
    gdev = [cu(g) for g in gs]
    gbase = torch.full_like(base, 7.0)
    q.cluster_grad(gdev, gbase)
    gb = gbase.cpu().numpy()
    keep = np.ones(gb.size, bool)
    for i, (w, g) in enumerate(zip(ws, gs)):
        _, rc, ridx, alpha, _ = B.nonuniform_bucket_quantize(w, bits, bucket_type, bucket_size)
        _, gc = B.nuq_bucket_grads(g, ridx, 1 << bits, alpha, bucket_type, bucket_size)
        got = gb[offs[i]:offs[i] + gc.size].reshape(gc.shape)
        n = max(1, w.size // gc.shape[1])
        assert np.abs(got - gc).max() <= 2e-6 * max(np.abs(gc).max(), 1e-20) * np.sqrt(n), i
        keep[offs[i]:offs[i] + gc.size] = False
    assert np.all(gb[keep] == 7.0)                                       # nothing written outside the codebooks
    q.cluster_grad(gdev, gbase)
    assert np.array_equal(gbase.cpu().numpy(), gb)                       # deterministic


def test_set_bits_refits_the_leading_rows():
    """RL bit search: tables sized for 8 bits; set_bits(3) + quantile_init() re-fit rows 0..7 exactly and zero the rest"""
    rng = np.random.RandomState(5)
    ws = [he(rng, s) for s in [(3, 3, 16, 32), (64, 10), (3, 3, 32, 1)]]
    q, src, dst, base, views, _ = quantizer(ws, 8, 'channel', 256)
    q.quantile_init()
    q.forward()
    for bits in (3, 1, 6):
        q.set_bits(bits)
        q.quantile_init()
        q.forward()
        for i, w in enumerate(ws):
            rq, rc, _, _, _ = B.nonuniform_bucket_quantize(w, bits, 'channel', 256)
            v = views[i].cpu().numpy()
            assert np.array_equal(v[:1 << bits], rc) and np.all(v[1 << bits:] == 0)
            assert np.array_equal(dst[i].cpu().numpy(), rq)
    with pytest.raises(ValueError):
        q.set_bits(9)


def test_over_limit_bucket_is_refused_before_any_launch():
    src = [torch.zeros(3, 3, 2048, 1, device=DEV)]
    with pytest.raises(ValueError, match='16384'):
        ops.CodebookWeightQuantizer(src, [torch.empty_like(src[0])], 4, use_buckets=True, bucket_type='channel')


# ---------------------------------------------------------------------------------------------------- learner
def make(bucket_type, **flags):
    from test_learners_gpu import make as make_lrn
    return make_lrn('non-uniform', nuql_use_buckets=True, nuql_bucket_type=bucket_type, **flags)


def bucketed_oracle(monkeypatch, ex, lrn):
    """the step oracle with the bucketed codebook quantizer of the learner's spec"""
    wq = ex.weight_quant
    monkeypatch.setattr(step_oracle, 'codebook_quant', lambda w, c: B.codebook_quant_bucketed(
        w, c, wq['bucket_type'], wq['bucket_size']))
    teacher = StepOracle(ex.teacher.ops, ex.teacher.logits_t, lrn.images) if ex.teacher is not None else None
    return StepOracle(ex.ops, ex.logits_t, lrn.images, lrn.labels, ex.loss, wq, ex.act_quant, teacher)


@pytest.mark.parametrize('mode', ['weights', 'cluster', 'both'])
@pytest.mark.parametrize('bucket_type', ['split', 'channel'])
def test_bucketed_learner_step_matches_oracle(monkeypatch, bucket_type, mode):
    monkeypatch.setenv('PF_CONV_PATH', 'fp32')
    lrn = make(bucket_type, nuql_weight_bits=4, enbl_dst=True, nuql_opt_mode=mode)
    ex = lrn.sess_train
    assert ex.wq.use_buckets and ex.weight_quant['bucket_type'] == bucket_type
    state, tstate = ex.store.state_dict(), ex.teacher.store.state_dict()
    cnames = [op.vars['clusters'].name for op in ex.wq_ops]
    assert all(n.endswith('/nonuniform_bucket_quantize/clusters:0') for n in cnames)
    trainable = [v.name for v in lrn.trainable_vars]
    frozen = {'weights': cnames, 'cluster': [n for n in trainable if n not in cnames], 'both': []}[mode]
    for op, cn in zip(ex.wq_ops, cnames):
        _, c_ref, _, _, _ = B.nonuniform_bucket_quantize(state[op.vars['kernel'].name], 4, bucket_type, 256)
        assert np.array_equal(state[cn], c_ref), cn                       # quantile init: exact order statistics
    orc = bucketed_oracle(monkeypatch, ex, lrn)
    images, labels = lrn.iterator_train.next_batch()
    ex.buf[lrn.images].copy_(images)
    ex.buf[lrn.labels].copy_(labels)
    ex.run_step(lrn.lrn_rate(0))
    got = ex.fetch_losses()
    for op, cn in zip(ex.wq_ops, cnames):
        v = op.vars['kernel']
        q_ref, _, _, _, _ = B.nonuniform_bucket_quantize(state[v.name], 4, bucket_type, 256, state[cn])
        assert np.array_equal(ex.store.view(v, ex.QW).cpu().numpy(), q_ref), v.name
    ref, new_state, grads = orc.step(state, images.numpy(), labels.numpy(), dict(kind='adam', slots={}), lrn.lrn_rate(0),
                                     teacher_state=tstate, frozen=frozen)
    for k in ('ce', 'l2', 'dst_loss', 'loss'):
        assert rel(got[k], ref[k]) <= 1e-5, (k, got[k], ref[k])
    after = ex.store.state_dict()
    for n in frozen:
        assert np.array_equal(after[n], state[n]), n
    if mode != 'weights':
        for op, cn in zip(ex.wq_ops, cnames):
            g_dev = ex.store.view(op.vars['clusters'], ex.G).cpu().numpy()
            # the segment sums of the device's own gradient w.r.t. the quantized kernel, then the oracle's autograd
            v = op.vars['kernel']
            _, _, ridx, alpha, _ = B.nonuniform_bucket_quantize(state[v.name], 4, bucket_type, 256, state[cn])
            _, gc = B.nuq_bucket_grads(ex.store.view(v, ex.G).cpu().numpy(), ridx, 16, alpha, bucket_type, 256)
            assert np.abs(g_dev - gc).max() <= 2e-6 * max(np.abs(gc).max(), 1e-20) * np.sqrt(ridx.shape[0]), cn
            assert np.abs(g_dev - grads[cn]).max() <= 1e-4 * max(np.abs(grads[cn]).max(), 1e-12), cn
    lr = lrn.lrn_rate(0)
    for n in [n for n in trainable if n not in frozen and 'batch_normalization' not in n]:
        assert np.abs((after[n] - state[n]) - (new_state[n] - state[n])).max() <= 2e-2 * lr + 1e-12, n


def _check_quantized_kernels(ex, state, bucket_type, bits=4):
    """QW of the last step against the oracle on the variables that step started from"""
    for op in ex.wq_ops:
        v = op.vars['kernel']
        q_ref, _, _, _, _ = B.nonuniform_bucket_quantize(state[v.name], bits, bucket_type, 256,
                                                         state[op.vars['clusters'].name])
        assert np.array_equal(ex.store.view(v, ex.QW).cpu().numpy(), q_ref), v.name


def test_bucketed_learner_on_tensor_core_path_resnet50():
    """channel buckets on ResNet-50 (the benchmark's NUQ network) at batch 2 on the default tensor-core path"""
    import bench
    from pocketflow_b200.learners.learner_utils import create_learner
    mod = bench.setup_flags('resnet50_nuq4_dst_b256', 2)
    FLAGS.nuql_use_buckets, FLAGS.nuql_bucket_type = True, 'channel'
    lrn = create_learner(None, mod.ModelHelper())
    ex = lrn.sess_train
    assert ex.wq.use_buckets and len(ex.tc) >= 8
    state = ex.store.state_dict()
    for op in ex.wq_ops[:6]:
        _, c_ref, _, _, _ = B.nonuniform_bucket_quantize(state[op.vars['kernel'].name], 4, 'channel', 256)
        assert np.array_equal(state[op.vars['clusters'].name], c_ref)
    cn = [op.vars['clusters'].name for op in ex.wq_ops]
    losses = []
    for _ in range(2):
        prev = ex.store.state_dict()
        lrn.train_step()
        losses.append(ex.fetch_losses()['loss'])
    assert all(np.isfinite(losses))
    _check_quantized_kernels(ex, prev, 'channel')
    after = ex.store.state_dict()
    assert all(np.array_equal(after[n], state[n]) for n in cn)              # 'weights' mode: codebooks frozen


def test_bucketed_learner_on_mobilenet_with_depthwise_codebooks():
    from test_learners_gpu import make_mobilenet
    import importlib
    importlib.import_module('pocketflow_b200.learners.nonuniform_quantization.learner')
    lrn = make_mobilenet('non-uniform', nuql_use_buckets=True, nuql_bucket_type='split', nuql_weight_bits=4,
                         nuql_opt_mode='both', enbl_dst=False)
    ex = lrn.sess_train
    assert any(op.type == 'DepthwiseConv2dNative' for op in ex.wq_ops)
    before = ex.store.state_dict()
    lrn.train_step()
    assert np.isfinite(ex.fetch_losses()['loss'])
    _check_quantized_kernels(ex, before, 'split')
    after = ex.store.state_dict()
    moved = [op.vars['clusters'].name for op in ex.wq_ops if not np.array_equal(after[op.vars['clusters'].name],
                                                                                  before[op.vars['clusters'].name])]
    assert len(moved) == len(ex.wq_ops)                                    # 'both': every codebook is trained


@pytest.mark.parametrize('fmt', ['npz', 'tf'])
def test_bucketed_codebooks_survive_save_and_exec_mode_eval(tmp_path, fmt):
    from pocketflow_b200.datasets.abstract_dataset import POOL_SIZE
    flags = dict(nuql_weight_bits=4, nuql_opt_mode='cluster', summ_step=10 ** 9, save_step=10 ** 9, ckpt_format=fmt,
                 nuql_save_quant_model_path=str(tmp_path / 'ckpt' / 'model.ckpt'))
    lrn = make('channel', **flags)
    lrn.train(nb_iters=4)
    trained = lrn.sess_train.store.state_dict()
    score = float(lrn.evaluate(nb_iters=POOL_SIZE))
    del lrn
    fresh = make('channel', exec_mode='eval', **flags)
    restored = float(fresh.evaluate(nb_iters=POOL_SIZE))
    assert rel(restored, score) <= 1e-6, (restored, score)
    st = fresh.sess_train.store.state_dict()
    for op in fresh.sess_train.wq_ops:
        n = op.vars['clusters'].name
        assert st[n].shape == (16, op.vars['kernel'].shape[-1]) and np.array_equal(st[n], trained[n]), n
