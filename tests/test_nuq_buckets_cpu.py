"""Bucketed codebooks (--nuql_use_buckets) without a device: the oracle against the reference's own __bucket_quantize
(tests/golden/ref_executed_nuq_bucket_v1.json), a hand-derived 2-bucket case, the graph edit's `clusters` variables,
the refused configurations, the host work tables, and the step oracle's autograd form against the numpy oracle."""
import hashlib
import importlib
import json
import os
import sys

import numpy as np
import pytest
import torch

from pocketflow_b200 import graph as G
from pocketflow_b200 import ops
from pocketflow_b200.flags import FLAGS

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, 'golden'))
import nuq_bucket_oracle as B  # noqa: E402
from make_golden_nuq_bucket import make_input  # noqa: E402

F32 = np.float32


def _sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def test_oracle_matches_the_reference_bucket_quantize_bit_for_bit():
    with open(os.path.join(HERE, 'golden', 'ref_executed_nuq_bucket_v1.json')) as f:
        gold = json.load(f)['cases']
    assert len(gold) == 60
    seen = set()
    for g in gold:
        x = make_input(g['index'], tuple(g['shape']), g['bucket_type'], g['bucket_size'], g['kind'])
        q, c, idx, alpha, beta = B.nonuniform_bucket_quantize(x, g['bits'], g['bucket_type'], g['bucket_size'])
        assert _sha(q) == g['sha256'], g
        assert list(c.shape) == g['clusters_shape'] and _sha(c) == g['clusters_sha256'], g
        assert B.bucket_storage_bits([g['shape']], g['bucket_type'], g['bucket_size']) == g['bucket_storage'], g
        seen.add((g['bucket_type'], g['bits'], g['kind']))
    assert {b for _, b, _ in seen} == {1, 2, 4, 8} and {k for _, _, k in seen} == {'normal', 'constant', 'ties'}


def test_two_bucket_known_answer():
    """A [4, 2] dense kernel, channel buckets, 1 bit.  Column 0 = (0, 1, 2, 3): alpha = 3 + 1e-10 = 3 in fp32, x_n =
    (0, 1/3, 2/3, 1); percentiles 33.3 / 66.7 of 4 rows -> descending ranks rint(3 * 2/3) = 2 and rint(3 * 1/3) = 1 ->
    1/3 and 2/3.  Column 1 = (10, 10, 10, 14): alpha = 4, x_n = (0, 0, 0, 1) -> centroids 0 and 0; every element takes
    centroid 0 (first index on ties), so q = 0 * sign(x_n + 1e-6) and the column becomes beta = 10."""
    w = np.array([[0, 10], [1, 10], [2, 10], [3, 14]], F32)
    q, c, idx, alpha, beta = B.nonuniform_bucket_quantize(w, 1, 'channel', 256)
    assert np.array_equal(alpha, np.array([3, 4], F32)) and np.array_equal(beta, np.array([0, 10], F32))
    assert np.array_equal(c, np.array([[F32(1) / F32(3), 0], [F32(2) / F32(3), 0]], F32))
    assert np.array_equal(idx, np.array([[0, 0], [0, 0], [1, 0], [1, 0]]))
    third = F32(3) * (F32(1) / F32(3))
    assert np.array_equal(q, np.array([[third, 10], [third, 10], [F32(3) * (F32(2) / F32(3)), 10],
                                       [F32(3) * (F32(2) / F32(3)), 10]], F32))
    # split buckets of 4 over 6 elements: 2 strided buckets (flat i -> bucket i % 2), two padding copies of w[-1]
    x = np.arange(6, dtype=F32)
    xb, ncols, padded = B.bucket_view(x, 'split', 4)
    assert ncols == 2 and padded == 2 and np.array_equal(xb, np.array([[0, 1], [2, 3], [4, 5], [5, 5]], F32))
    assert ops.nuq_bucket_layout((6,), 'split', 4) == (2, 8, 4)
    # the codebook gradient sums over real rows only: the padding copies of bucket 0 carry no gradient
    qx, c, idx, alpha, _ = B.nonuniform_bucket_quantize(x, 1, 'split', 4)
    _, gc = B.nuq_bucket_grads(np.ones(6, F32), idx, 2, alpha, 'split', 4)
    assert gc.sum(axis=0).tolist() == [float(alpha[0]) * 3, float(alpha[1]) * 3]


def _graph(net, bucket_type, bucket_size=256, cap=None, bits=4):
    FLAGS.reset()
    importlib.import_module('pocketflow_b200.learners.nonuniform_quantization.learner')
    from pocketflow_b200.learners.nonuniform_quantization.utils import NonUniformQuantization
    if net == 'resnet20':
        mod = importlib.import_module('pocketflow_b200.nets.resnet_at_cifar10')
        FLAGS.resnet_size = 20
    else:
        mod = importlib.import_module('pocketflow_b200.nets.mobilenet_at_ilsvrc12')
    mh = mod.ModelHelper()
    g = G.Graph()
    with g.as_default():
        with G.variable_scope('data'):
            im, _ = mh.build_dataset_train().get_next()
        with G.variable_scope('model'):
            mh.forward_train(im)
            before = set(g.variables)
            nq = NonUniformQuantization(g, bucket_size, True, 'quantile', bucket_type, codebook_bits_cap=cap)
            ops_ = nq.search_matmul_op(False)
            nq.insert_quant_op_for_weights({o.name: bits for o in ops_})
    return g, nq, ops_, sorted(set(g.variables) - before)


@pytest.mark.parametrize('net', ['resnet20', 'mobilenet'])
@pytest.mark.parametrize('bucket_type', ['split', 'channel'])
def test_graph_edit_creates_one_bucket_codebook_table_per_quantized_op(net, bucket_type):
    """<model scope>/<op>/nonuniform_bucket_quantize/clusters, shape [2^bits, bucket_num], for EVERY quantized op —
    depthwise included — and the reference's bucket storage (64 bits per bucket)."""
    g, nq, ops_, new = _graph(net, bucket_type)
    assert len(new) == len(ops_) > 0
    if net == 'mobilenet':
        assert any(o.type == 'DepthwiseConv2dNative' for o in ops_)
    storage = 0
    for o in ops_:
        v = o.vars['clusters']
        shape = o.vars['kernel'].shape
        ncols = shape[-1] if bucket_type == 'channel' else -(-int(np.prod(shape)) // 256)
        assert v.name == 'model/' + o.name.split('/', 1)[1] + '/nonuniform_bucket_quantize/clusters:0' and v.name in new
        assert v.trainable and v.shape == (16, ncols), (v.name, v.shape)
        if o.type == 'DepthwiseConv2dNative' and bucket_type == 'channel':
            assert ncols == 1                                       # [3, 3, C, 1] -> one bucket
        storage += 64 * ncols
    assert nq.bucket_storage == storage == B.bucket_storage_bits([o.vars['kernel'].shape for o in ops_], bucket_type, 256)
    spec = nq.weight_quant_spec()
    assert spec['use_buckets'] is True and spec['bucket_type'] == bucket_type and spec['bucket_size'] == 256
    assert spec['kind'] == 'nonuniform' and spec['bits'] == [4] * len(ops_)
    FLAGS.reset()


def test_codebook_tables_sized_for_the_bit_search_cap():
    _, _, ops_, _ = _graph('resnet20', 'channel', cap=6)
    assert all(o.vars['clusters'].shape == (64, o.vars['kernel'].shape[-1]) for o in ops_)
    FLAGS.reset()


def test_unbucketed_spec_is_unchanged():
    FLAGS.reset()
    importlib.import_module('pocketflow_b200.learners.nonuniform_quantization.learner')
    from pocketflow_b200.learners.nonuniform_quantization.utils import NonUniformQuantization
    nq = NonUniformQuantization(G.Graph(), 256, False, 'quantile', 'split')
    nq.quantized_matmul_ops, nq.weight_bits = ['op'], [4]
    assert set(nq.weight_quant_spec()) == {'kind', 'ops', 'bits', 'init_style', 'train_clusters'}


def test_refused_configurations_raise_value_error():
    FLAGS.reset()
    importlib.import_module('pocketflow_b200.learners.nonuniform_quantization.learner')
    from pocketflow_b200.learners.nonuniform_quantization.utils import NonUniformQuantization
    # the reference's bucketed uniform init calls __uniform_init with the wrong arguments: it cannot run
    with pytest.raises(ValueError, match='uniform'):
        NonUniformQuantization(G.Graph(), 256, True, 'uniform', 'channel')
    NonUniformQuantization(G.Graph(), 256, False, 'uniform', 'channel')             # unbucketed: unchanged
    # a bucket taller than the quantile init sorts: at the graph edit, before anything reaches the device
    assert ops.nuq_bucket_layout((3, 3, 1024, 1), 'channel', 256) == (1, 9216, 9216)
    with pytest.raises(ValueError, match='16384'):
        ops.nuq_bucket_layout((3, 3, 2048, 1), 'channel', 256)
    with pytest.raises(ValueError, match='16384'):
        ops.nuq_bucket_layout((100000,), 'split', 16385)
    with pytest.raises(ValueError, match='16384'):
        _graph('resnet20', 'split', bucket_size=20000)
    FLAGS.reset()


@pytest.mark.parametrize('bits', [1, 4, 8])
def test_work_tables_cover_every_element_once(bits):
    shapes = [(3, 3, 64, 64), (3, 3, 16, 1), (64, 10), (1, 1, 256, 1000), (7,)]
    for btype, bsz in (('channel', 256), ('split', 256), ('split', 100)):
        segs = np.zeros(len(shapes), dtype=ops.UQ_SEG)
        for i, s in enumerate(shapes):
            ncols, padded, _ = ops.nuq_bucket_layout(s, btype, bsz)
            segs[i]['numel'], segs[i]['padded'], segs[i]['ncols'], segs[i]['bits'] = int(np.prod(s)), padded, ncols, bits
        wq = ops.nuq_bucket_quant_works(segs)
        assert np.all((1 << bits) * wq['ncol_tile'] <= max(ops.NUQ_BUCKET_TILE_FLOATS, 32 << bits))
        assert np.all(wq['ncol_tile'] <= ops.NUQ_BUCKET_MAX_TILE)
        assert np.all((1 << bits) * wq['ncol_tile'] <= ops.NUQ_BUCKET_TILE_FLOATS)
        wg, tiles = ops.nuq_bucket_grad_works(segs)
        for table in (wq, wg):
            for i, seg in enumerate(segs):
                cover = np.zeros(int(seg['padded']), np.int32)
                for w in table[table['seg'] == i]:
                    r = np.arange(w['start'], w['start'] + w['count'])[:, None]
                    cover[(r * seg['ncols'] + w['c0'] + np.arange(w['ncol_tile'])[None, :]).reshape(-1)] += 1
                assert np.all(cover == 1)
        assert np.all(tiles['ncol_tile'] <= ops.NUQ_BUCKET_GRAD_TILE)
        assert tiles['count'].sum() == len(wg) and np.array_equal(np.cumsum(tiles['count'])[:-1], tiles['start'][1:])
        for t in tiles:
            sub = wg[t['start']:t['start'] + t['count']]
            assert np.all(sub['seg'] == t['seg']) and np.all(sub['c0'] == t['c0'])


@pytest.mark.parametrize('bucket_type,bucket_size', [('channel', 256), ('split', 64), ('split', 256)])
def test_step_oracle_bucketed_forward_is_the_numpy_oracle(bucket_type, bucket_size):
    rng = np.random.RandomState(7)
    for shape in [(3, 3, 8, 16), (64, 10), (3, 3, 16, 1)]:
        w = rng.randn(*shape).astype(F32)
        for bits in (2, 4):
            q_ref, c, _, _, _ = B.nonuniform_bucket_quantize(w, bits, bucket_type, bucket_size)
            q = B.codebook_quant_bucketed(torch.from_numpy(w), torch.from_numpy(c), bucket_type, bucket_size)
            assert np.array_equal(q.detach().numpy(), q_ref), (shape, bits)
    # autograd: the codebook gradient is the per-bucket segment sum of g * alpha
    w = rng.randn(5, 5, 3, 7).astype(F32)
    q_ref, c, idx, alpha, _ = B.nonuniform_bucket_quantize(w, 2, bucket_type, bucket_size)
    ct = torch.from_numpy(c).requires_grad_(True)
    wt = torch.from_numpy(w).requires_grad_(True)
    g = rng.randn(*w.shape).astype(F32)
    (B.codebook_quant_bucketed(wt, ct, bucket_type, bucket_size) * torch.from_numpy(g)).sum().backward()
    gx, gc = B.nuq_bucket_grads(g, idx, 4, alpha, bucket_type, bucket_size)
    assert np.abs(ct.grad.numpy() - gc).max() <= 1e-5 * max(np.abs(gc).max(), 1e-12)
    assert np.abs(wt.grad.numpy() - gx).max() <= 1e-6 * np.abs(gx).max()
