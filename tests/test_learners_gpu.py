"""Learner-level GPU tests through the plugin surface (create_learner / train_step / prune / evaluate):
WeightSparseLearner (masks bit-exact vs the oracle inside a real training loop, pruned weights stay
zero), NonUniformQuantLearner (codebook init + step loss vs the oracle), FullPrecLearner, checkpoints."""
import os

import numpy as np
import pytest
import torch

from oracle import pf_oracle as O
from oracle.step_oracle import StepOracle
from pocketflow_b200.flags import FLAGS

pytestmark = pytest.mark.gpu
F32 = np.float32


def rel(a, b):
    return abs(float(a) - float(b)) / max(abs(float(b)), 1e-30)


def make(learner, **flags):
    FLAGS.reset()
    from pocketflow_b200.nets import resnet_at_cifar10 as R
    from pocketflow_b200.learners.learner_utils import create_learner
    import pocketflow_b200.learners.weight_sparsification.learner  # noqa: F401  (flag definitions)
    import pocketflow_b200.learners.nonuniform_quantization.learner  # noqa: F401
    import pocketflow_b200.learners.uniform_quantization.learner  # noqa: F401
    import pocketflow_b200.learners.channel_pruning_gpu.learner  # noqa: F401
    FLAGS.resnet_size, FLAGS.batch_size, FLAGS.learner = 8, 16, learner
    for k, v in flags.items():
        setattr(FLAGS, k, v)
    return create_learner(None, R.ModelHelper())


def test_create_learner_names():
    from pocketflow_b200.learners.learner_utils import create_learner
    FLAGS.reset()
    FLAGS.learner = 'bogus'
    with pytest.raises(ValueError):
        create_learner(None, None)
    FLAGS.learner = 'uniform-tf'
    with pytest.raises(ValueError):
        create_learner(None, None)


def test_weight_sparse_learner_masks_bit_exact_in_training_loop():
    lrn = make('weight-sparse', ws_prune_ratio=0.6, ws_prune_ratio_prtl='uniform', enbl_dst=False)
    ex = lrn.sess_train
    names = [v.name for v in lrn.maskable_vars]
    assert len(names) == 11 and all('kernel' in n for n in names)       # 10 convs + dense of ResNet-8
    lrn.nb_iters_train = 40                                             # t_b = 4, t_e = 20
    ref_bkup = {v.name: ex.store.view(v).cpu().numpy().copy() for v in lrn.maskable_vars}
    ref_mask = {n: np.ones_like(b) for n, b in ref_bkup.items()}
    for it in range(24):
        lrn.train_step()
        if (it + 1) % 4 == 0:
            w_now = {v.name: ex.store.view(v).cpu().numpy().copy() for v in lrn.maskable_vars}
            ratios = lrn.prune()
            step = ex.step_count
            assert ratios[0] == O.ws_prune_ratio_dyn(step, 40, 0.6)
            for v, r in zip(lrn.maskable_vars, ratios):
                nv, nb, nm, thr = O.ws_build_mask(w_now[v.name], ref_bkup[v.name], ref_mask[v.name], r)
                ref_bkup[v.name], ref_mask[v.name] = nb, nm
                assert np.array_equal(ex.store.view(v, ex.MASK).cpu().numpy(), nm), (it, v.name)     # bit-exact
                assert np.array_equal(ex.store.view(v, ex.BKUP).cpu().numpy(), nb)
                assert np.array_equal(ex.store.view(v).cpu().numpy(), nv)
            assert float(ex.S1.abs().max()) == 0.0                      # momentum slots re-initialised
        else:
            # between mask updates pruned weights stay exactly zero (gradient masked in the fused optimizer)
            for v in lrn.maskable_vars:
                w = ex.store.view(v).cpu().numpy()
                assert np.all(w[ref_mask[v.name] == 0] == 0)
    loss, pr = lrn.evaluate()
    assert abs(pr - 0.6) < 0.01 and np.isfinite(loss)
    assert O.calc_prune_ratio([ex.store.view(v).cpu().numpy() for v in lrn.maskable_vars]) == F32(pr)


def test_weight_sparse_heurist_protocol():
    lrn = make('weight-sparse', ws_prune_ratio=0.5, ws_prune_ratio_prtl='heurist')
    n = np.array([v.numel for v in lrn.maskable_vars], dtype=np.float64)
    r = np.array([x[1] for x in lrn.var_names_n_prune_ratios])
    np.testing.assert_allclose(r, O.ws_heurist_ratios(n, 0.5), rtol=1e-12)
    assert abs((r * n).sum() / n.sum() - 0.5) < 1e-12


@pytest.mark.parametrize('mode', ['weights', 'cluster', 'both'])
def test_nonuniform_learner_step_matches_oracle(monkeypatch, mode):
    """NonUniformQuantLearner, the three optimisation modes (learners/nonuniform_quantization/learner.py:252-270): the
    codebooks are trainable `clusters` variables of the model scope; 'weights' freezes them, 'cluster' trains ONLY them
    (gradient = alpha * segment sum of the kernel gradient over each centroid's members), 'both' trains everything.
    Quantile init exact, quantized kernels bit-exact, losses 1e-5, codebook / kernel updates vs the oracle step."""
    monkeypatch.setenv('PF_CONV_PATH', 'fp32')
    lrn = make('non-uniform', nuql_weight_bits=4, enbl_dst=True, nuql_opt_mode=mode)
    ex = lrn.sess_train
    assert isinstance(ex.wq, __import__('pocketflow_b200.ops', fromlist=['x']).CodebookWeightQuantizer)
    state, tstate = ex.store.state_dict(), ex.teacher.store.state_dict()
    cnames = [op.vars['clusters'].name for op in ex.wq_ops]
    assert all(n.startswith('model/') and n.endswith('/Conv2D/nonuniform_quantize/clusters:0') for n in cnames)
    trainable = [v.name for v in lrn.trainable_vars]
    assert set(cnames) <= set(trainable)
    frozen = {'weights': cnames, 'cluster': [n for n in trainable if n not in cnames], 'both': []}[mode]
    teacher = StepOracle(ex.teacher.ops, ex.teacher.logits_t, lrn.images)
    orc = StepOracle(ex.ops, ex.logits_t, lrn.images, lrn.labels, ex.loss, ex.weight_quant, ex.act_quant, teacher)
    for op, cn in zip(ex.wq_ops, cnames):
        _, c_ref, _ = O.nonuniform_quantize(state[op.vars['kernel'].name], 4)
        assert np.array_equal(state[cn], c_ref)                           # quantile init: exact order statistics
    images, labels = lrn.iterator_train.next_batch()
    ex.buf[lrn.images].copy_(images)
    ex.buf[lrn.labels].copy_(labels)
    ex.run_step(lrn.lrn_rate(0))
    got = ex.fetch_losses()
    for op, cn in zip(ex.wq_ops, cnames):
        v = op.vars['kernel']
        q_ref, _, _ = O.nonuniform_quantize(state[v.name], 4, state[cn])
        assert np.array_equal(ex.store.view(v, ex.QW).cpu().numpy(), q_ref)
    ref, new_state, grads = orc.step(state, images.numpy(), labels.numpy(), dict(kind='adam', slots={}), lrn.lrn_rate(0),
                                     teacher_state=tstate, frozen=frozen)
    for k in ('ce', 'l2', 'dst_loss', 'loss'):
        assert rel(got[k], ref[k]) <= 1e-5, (k, got[k], ref[k])
    # the l2 term counts the codebooks in every mode ("clusters should be not included for regularization", :219)
    wd = sum(float(c) * float((state[v.name].astype(np.float64) ** 2).sum()) / 2 for v, c in ex.loss.l2.items())
    assert rel(got['l2'], wd) <= 1e-5 and any(v.name in cnames for v in ex.loss.l2)
    after = ex.store.state_dict()
    for n in frozen:
        assert np.array_equal(after[n], state[n]), n                      # outside the optimizer's var_list
    if mode != 'weights':
        # codebook gradients: device (G buffer) vs autograd through gather, 1e-4 of the layer's largest entry
        for op, cn in zip(ex.wq_ops, cnames):
            g_dev = ex.store.view(op.vars['clusters'], ex.G).cpu().numpy()
            assert np.abs(g_dev - grads[cn]).max() <= 1e-4 * max(np.abs(grads[cn]).max(), 1e-12), cn
    # first Adam step: every updated entry moves by ~lr in the direction of its gradient
    lr = lrn.lrn_rate(0)
    moved = [n for n in trainable if n not in frozen and 'batch_normalization' not in n]
    for n in moved:
        d_dev, d_ref = after[n] - state[n], new_state[n] - state[n]
        assert np.abs(d_dev - d_ref).max() <= 2e-2 * lr + 1e-12, n


def test_full_prec_learner_and_checkpoint_roundtrip(tmp_path):
    lrn = make('full-prec', save_path=str(tmp_path / 'models' / 'model.ckpt'))
    ex = lrn.sess_train
    losses = []
    for _ in range(8):
        lrn.train_step()
        losses.append(ex.fetch_losses()['loss'])
    assert np.all(np.isfinite(losses))
    from pocketflow_b200.learners.abstract_learner import save_checkpoint, load_checkpoint, latest_checkpoint
    fn = save_checkpoint(FLAGS.save_path, ex.store.state_dict(), ex.step_count)
    assert latest_checkpoint(os.path.dirname(FLAGS.save_path)) == fn
    sd = load_checkpoint(fn)
    before = ex.store.P.clone()
    ex.store.P.zero_()
    ex.store.load_state_dict(sd)
    assert torch.equal(ex.store.P, before)
    assert np.isfinite(lrn.evaluate())


def test_uniform_learner_trains_and_evaluates(tmp_path):
    lrn = make('uniform', uql_weight_bits=8, uql_use_buckets=True, enbl_dst=True, summ_step=5, save_step=10 ** 9,
               uql_save_quant_model_path=str(tmp_path / 'uql' / 'model.ckpt'))
    lrn.train(nb_iters=6)            # includes the CUDA-graph-free eager loop, logging, final save + evaluate
    r = lrn.sess_train.fetch_losses()
    assert np.isfinite(r['loss']) and lrn.sess_train.step_count == 6


def make_mobilenet(learner, **flags):
    FLAGS.reset()
    import importlib
    import pocketflow_b200.datasets.ilsvrc12_dataset as D
    importlib.reload(D)
    from pocketflow_b200.nets import mobilenet_at_ilsvrc12 as M
    importlib.reload(M)
    from pocketflow_b200.learners.learner_utils import create_learner
    import pocketflow_b200.learners.channel_pruning_gpu.learner  # noqa: F401
    FLAGS.batch_size, FLAGS.learner, FLAGS.nb_classes = 2, learner, 1001
    for k, v in flags.items():
        setattr(FLAGS, k, v)
    return create_learner(None, M.ModelHelper())


@pytest.mark.parametrize('conv_path', ['fp32', 'tc'])
def test_mobilenet_channel_pruned_gpu_learner_step(monkeypatch, conv_path):
    """Config 4 steady state: MobileNet-v1, input-channel masks on the 13 interior pointwise kernels (chosen by a short
    run of the selection phase), masked Momentum step; loss vs the oracle step with the same masks; pruned channels
    stay zero.  Both the exact-fp32 and the (default) tensor-core conv path."""
    monkeypatch.setenv('PF_CONV_PATH', conv_path)
    lrn = make_mobilenet('chn-pruned-gpu', cpg_prune_ratio=0.5)
    ex = lrn.sess_train
    assert len(lrn.maskable_vars) == 15 and sum(v.numel for v in lrn.maskable_vars) == 4165472
    assert all(v.name.startswith('pruned_model/') for v in lrn.maskable_vars)
    assert lrn.prune_ratios[0] == 0.0 and lrn.prune_ratios[-1] == 0.0 and lrn.prune_ratios[5] == 0.5
    lrn.init_from_full()
    lrn.choose_channels(nb_iters_layer=2)
    masks = {v.name: ex.store.view(v, ex.MASK).cpu().numpy().copy() for v in lrn.maskable_vars}
    for v in lrn.maskable_vars[1:-1]:
        m = masks[v.name]
        per_cin = m.reshape(-1, m.shape[2], m.shape[3]).max(axis=(0, 2))
        assert abs(per_cin.mean() - 0.5) < 0.02                           # half of the input channels kept
        assert np.all(ex.store.view(v).cpu().numpy()[m == 0] == 0)
    orc = StepOracle(ex.ops, ex.logits_t, lrn.images, lrn.labels, ex.loss)
    state = ex.store.state_dict()
    images, labels = lrn.iterator_train.next_batch()
    ex.buf[lrn.images].copy_(images)
    ex.buf[lrn.labels].copy_(labels)
    lr = lrn.lrn_rate(0)
    ex.run_step(lr)
    got = ex.fetch_losses()
    ref, new_state, grads = orc.step(state, images.numpy(), labels.numpy(), dict(kind='momentum', slots={}, momentum=0.9),
                                     lr, masks=masks)
    # the 3 -> 32 stem's weight gradient (tc path: g = 2 pixels per GEMM row on the tensor cores, diagonal blocks folded)
    stem = ex.ops[[o.type for o in ex.ops].index('Conv2D')].vars['kernel']
    g_dev, g_ref = ex.store.view(stem, ex.G).cpu().numpy().reshape(-1), grads[stem.name].reshape(-1)
    cos = float(np.dot(g_dev, g_ref) / (np.linalg.norm(g_dev) * np.linalg.norm(g_ref) + 1e-30))
    # (the deepest gradient of the net: 27 layers of ReLU6 boundaries behind it at batch 2; the kernel itself is checked
    # against float64 in tests/test_tc_gpu.py::test_small_cout_wgrad_by_pixel_pairing)
    assert cos >= (0.999 if conv_path == 'fp32' else 0.995) and abs(np.linalg.norm(g_dev) / np.linalg.norm(g_ref) - 1.0) <= 2e-2, cos
    if conv_path == 'tc':
        assert 'pair' in ex.im2col[ex.ops[[o.type for o in ex.ops].index('Conv2D')]]
    # split-bf16 operands carry 16 mantissa bits: 2e-6 per convolution, 28 of them in a row at batch 2 (measured 2e-5 on
    # the cross-entropy with half of the channels masked); the exact-fp32 path holds 1e-5
    bar = 1e-5 if conv_path == 'fp32' else 3e-5
    for k in ('ce', 'l2', 'loss'):
        assert rel(got[k], ref[k]) <= bar, (k, got[k], ref[k])
    for v in lrn.maskable_vars[1:-1]:
        assert np.all(ex.store.view(v).cpu().numpy()[masks[v.name] == 0] == 0)


@pytest.mark.parametrize('conv_path', ['fp32', 'tc'])
def test_channel_selection_phase_matches_the_oracle(monkeypatch, tmp_path, conv_path):
    """SURVEY §8 f4 — the layer-wise channel selection (learners/channel_pruning_gpu/learner.py:445-518) of ONE MobileNet
    layer, iteration by iteration against the oracle's restatement driven on the same mini-batches: regression loss
    and its weight gradient, the proximal step (threshold, surviving channels), the lr / percentile schedule, the
    mask, the masked-Adam layer fine-tuning, the pruned model's BN moving statistics."""
    from oracle.step_oracle import cpg_layer_regression
    monkeypatch.setenv('PF_CONV_PATH', conv_path)
    layers, nb_iters = (3, 4), 3
    ratios = ['0'] * 15
    for idx in layers:
        ratios[idx] = '0.5'
    (tmp_path / 'ratios.txt').write_text(','.join(ratios) + '\n')
    lrn = make_mobilenet('chn-pruned-gpu', cpg_prune_ratio_type='list', cpg_prune_ratio_file=str(tmp_path / 'ratios.txt'),
                         cpg_lrn_rate_pgd_init=1e-7)
    ex = lrn.sess_train
    lrn.init_from_full()
    g = lrn.graph_train
    ops_full = [op for op in g.ops if op.name.startswith('model/')]
    ops_prnd = [op for op in g.ops if op.name.startswith('pruned_model/')]
    orc_f = StepOracle(ops_full, lrn.logits_full, lrn.images)
    orc_p = StepOracle(ops_prnd, ex.logits_t, lrn.images)
    st_f, st_p = lrn.store_full.state_dict(), ex.store.state_dict()
    pool = lrn.iterator_train
    pool.prefill()
    # ---- the oracle's run of the same loop (layer 3 first: layer 4 then sees a pruned input, as in a real run)
    ref_log, mask_ref, batch = [], {}, 0
    for idx in layers:
        conv_f, conv_p = lrn.conv_ops_full[idx], lrn.conv_ops_prnd[idx]
        kname = conv_p.vars['kernel'].name
        lr, prev = 1e-7, 0.0
        for it in range(nb_iters):
            images = pool.pool[batch % len(pool.pool)][0].numpy()
            batch += 1
            loss, grad, stats = cpg_layer_regression(orc_f, orc_p, st_f, st_p, images, conv_f, conv_p)
            perctl = 0.5 * 100.0 * (it + 1) / nb_iters
            st_p[kname], norms, thr = O.cpg_prox_step(st_p[kname], grad, lr, perctl)
            st_p.update(stats)
            ref_log.append(('prune', loss, lr, perctl, thr))
            lr = lr * 1.4 if loss < prev else lr * 0.7
            prev = loss
        mask_ref[kname] = O.cpg_channel_mask(st_p[kname])
        m_, v_, b1p, b2p = np.zeros_like(st_p[kname]), np.zeros_like(st_p[kname]), F32(0.9), F32(0.999)
        for it in range(nb_iters):
            images = pool.pool[batch % len(pool.pool)][0].numpy()
            batch += 1
            loss, grad, stats = cpg_layer_regression(orc_f, orc_p, st_f, st_p, images, conv_f, conv_p)
            st_p[kname], m_, v_ = O.adam_step(st_p[kname], m_, v_, grad * mask_ref[kname], 1e-2, b1p, b2p)
            st_p.update(stats)
            b1p, b2p = F32(b1p * F32(0.9)), F32(b2p * F32(0.999))
            ref_log.append(('finetune', loss))
    # ---- the learner's
    lrn.choose_channels(nb_iters_layer=nb_iters)
    got_log = lrn.selection_log
    assert len(got_log) == len(ref_log) == 2 * nb_iters * len(layers)
    bar = 1e-5 if conv_path == 'fp32' else 5e-5
    scale = max(r[1] for r in ref_log)
    assert scale > 0
    for gl, rl in zip(got_log, ref_log):
        assert gl[0] == rl[0]
        assert abs(gl[3] - rl[1]) <= (bar if gl[0] == 'prune' else 10 * bar) * abs(rl[1]) + 1e-9 * scale, (gl, rl)
        if gl[0] == 'prune':
            assert rel(gl[4], rl[2]) <= 1e-12 and rel(gl[5], rl[3]) <= 1e-12           # lr / percentile schedule
    new = ex.store.state_dict()
    for idx in layers:
        var = lrn.conv_ops_prnd[idx].vars['kernel']
        w, mask = ex.store.view(var).cpu().numpy(), ex.store.view(var, ex.MASK).cpu().numpy()
        assert np.array_equal(mask, mask_ref[var.name])                                # the SAME channels survive
        assert abs(mask.reshape(-1, mask.shape[2], mask.shape[3]).max(axis=(0, 2)).mean() - 0.5) < 0.02
        assert np.all(w[mask == 0] == 0)
        assert np.abs(w - st_p[var.name]).max() <= 2e-3 * np.abs(st_p[var.name]).max()  # after 3 Adam steps at lr 1e-2
    for k, v in st_p.items():
        if 'moving_' in k:
            # (layers behind the re-trained kernels see weights that differ by the Adam steps' 1e-3: same bar here)
            assert np.abs(new[k] - v).max() <= 1e-3 * np.abs(v).max() + 1e-7, k
    # the other layers are untouched and unmasked
    for j, v in enumerate(lrn.maskable_vars):
        if j not in layers:
            assert float(ex.store.view(v, ex.MASK).min()) == 1.0
            assert np.array_equal(new[v.name], st_p[v.name])


@pytest.mark.parametrize('learner,path_flag,extra', [
    ('full-prec', 'save_path', {}),
    ('weight-sparse', 'ws_save_path', dict(ws_prune_ratio=0.5, ws_prune_ratio_prtl='uniform', ws_mask_update_step=2)),
    ('uniform', 'uql_save_quant_model_path', dict(uql_weight_bits=8, uql_use_buckets=True)),
    ('non-uniform', 'nuql_save_quant_model_path', dict(nuql_weight_bits=4)),
    ('chn-pruned-gpu', 'cpg_save_path', dict(cpg_prune_ratio=0.5, cpg_nb_iters_layer=2)),
])
def test_exec_mode_eval_restores_the_saved_model(tmp_path, learner, path_flag, extra):
    """--exec_mode eval (nets/*_run.py:62-64): evaluate() restores the latest checkpoint first — a freshly built learner
    must score the TRAINED model, not its seed initialisation.  Both passes average the same 8 pooled batches."""
    from pocketflow_b200.datasets.abstract_dataset import POOL_SIZE
    flags = dict(extra, summ_step=10 ** 9, save_step=10 ** 9)
    flags[path_flag] = str(tmp_path / 'ckpt' / 'model.ckpt')
    lrn = make(learner, **flags)
    lrn.nb_iters_train = 6
    lrn.train(nb_iters=6)                                               # ends with save + evaluate
    first = lambda r: float(r[0] if isinstance(r, tuple) else r)
    trained = first(lrn.evaluate(nb_iters=POOL_SIZE))
    del lrn
    flags['exec_mode'] = 'eval'
    fresh = make(learner, **flags)
    restored = first(fresh.evaluate(nb_iters=POOL_SIZE))
    assert rel(restored, trained) <= 1e-6, (restored, trained)
    # and the default iteration count is the reference's ceil(nb_smpls_eval / batch_size_eval)
    assert fresh.eval_nb_iters() == int(np.ceil(FLAGS.nb_smpls_eval / FLAGS.batch_size_eval))


def test_exec_mode_eval_without_a_checkpoint_raises(tmp_path):
    flags = dict(exec_mode='eval', save_path=str(tmp_path / 'none' / 'model.ckpt'))
    lrn = make('full-prec', **flags)
    with pytest.raises(ValueError):
        lrn.evaluate()


def test_restore_refuses_a_checkpoint_of_another_scope(tmp_path):
    from pocketflow_b200.learners.abstract_learner import save_checkpoint
    lrn = make('full-prec', save_path=str(tmp_path / 'm' / 'model.ckpt'))
    state = {('other/' + k): v for k, v in lrn.sess_train.store.state_dict().items()}
    save_checkpoint(FLAGS.save_path, state, 1)
    with pytest.raises(ValueError):
        lrn.restore_model(FLAGS.save_path)


@pytest.mark.parametrize('conv_path', ['fp32', 'tc'])
def test_weight_sparse_layerwise_regression_matches_the_oracle(monkeypatch, conv_path):
    """The layer-wise regression stage of the pruning-ratio search (learners/weight_sparsification/pr_optimizer.py:
    283-314, :542-548) on ResNet-8 (its conv3-style adds are fused into the conv epilogues here): every core op in turn,
    Adam on its kernel with masked gradients of l2_loss(out_pruned - out_full), both networks in inference mode —
    against the oracle driven on the same mini-batches."""
    from oracle.step_oracle import cpg_layer_regression
    monkeypatch.setenv('PF_CONV_PATH', conv_path)
    lrn = make('weight-sparse', ws_prune_ratio=0.5, ws_prune_ratio_prtl='uniform', enbl_dst=True, ws_lrn_rate_rg=3e-3)
    ex = lrn.sess_train
    nb = 2
    lrn.pr_prune([0.5] * len(lrn.maskable_vars))
    st_full = dict(lrn._pr_full_state)
    st_p = ex.store.state_dict()
    masks = {v.name: ex.store.view(v, ex.MASK).cpu().numpy().copy() for v in lrn.maskable_vars}
    assert all(abs(m.mean() - 0.5) < 0.05 for m in masks.values())
    core = lrn.pr_core_ops()
    assert len(core) == len(lrn.maskable_vars) == 11
    assert any(op in ex.fused_add for op in core) == (conv_path == 'tc')    # residual adds fused into tcgen05 epilogues
    orc = StepOracle(ex.ops, ex.logits_t, lrn.images)
    pool = lrn.iterator_train
    pool.prefill()
    ref, batch = [], 0
    for op in core:
        kname = op.vars['kernel'].name
        m_, v_, b1p, b2p = np.zeros_like(st_p[kname]), np.zeros_like(st_p[kname]), F32(0.9), F32(0.999)
        ref.append([])
        for _ in range(nb):
            images = pool.pool[batch % len(pool.pool)][0].numpy()
            batch += 1
            loss, grad, _ = cpg_layer_regression(orc, orc, st_full, st_p, images, op, op, training=False)
            st_p[kname], m_, v_ = O.adam_step(st_p[kname], m_, v_, grad * masks[kname], 3e-3, b1p, b2p)
            b1p, b2p = F32(b1p * F32(0.9)), F32(b2p * F32(0.999))
            ref[-1].append(loss)
    got = lrn.pr_regress_layers(nb)
    bar = 1e-5 if conv_path == 'fp32' else 5e-5
    scale = max(max(r) for r in ref)
    for g_l, r_l, op in zip(got, ref, core):
        for a, b in zip(g_l, r_l):
            # (fused-add layers recover the conv difference from two differences: an absolute floor of 1e-6 of the scale)
            assert abs(a - b) <= bar * abs(b) + 1e-6 * scale, (op.name, a, b)
    new = ex.store.state_dict()
    for v in lrn.maskable_vars:
        w = new[v.name]
        assert np.all(w[masks[v.name] == 0] == 0)                           # pruned weights stay pruned
        assert np.abs(w - st_p[v.name]).max() <= 2e-3 * np.abs(st_p[v.name]).max() + 1e-6, v.name
    for k in new:
        if 'moving_' in k or 'batch_normalization' in k:
            assert np.array_equal(new[k], lrn._pr_full_state[k] if k in lrn._pr_full_state else new[k])   # inference mode: BN untouched
