"""Non-Uniform Quantization Learner (/root/reference/learners/nonuniform_quantization/learner.py:33-520),
'weights' optimisation mode: a 2^b-entry codebook per layer, quantile-initialised AFTER the weights
are in place (learner.py:127-129), frozen; weights trained with Adam through the STE."""
import os
from timeit import default_timer as timer

import numpy as np

from ... import graph as G
from ...engine import Executor
from ...flags import FLAGS, DEFINE_integer, DEFINE_boolean, DEFINE_string
from ...utils.multi_gpu_wrapper import MultiGpuWrapper as mgw
from ...utils.lrn_rate_utils import piecewise_constant
from ..abstract_learner import AbstractLearner, latest_checkpoint, load_checkpoint, save_checkpoint
from ..distillation_helper import DistillationHelper
from .utils import NonUniformQuantization
from .bit_optimizer import BitOptimizer

DEFINE_string('nuql_opt_mode', 'weights', 'the variables to optimize: [clusters, weights, both]')
DEFINE_string('nuql_init_style', 'quantile', 'the initialization of quantization points: [quantile, uniform]')
DEFINE_integer('nuql_weight_bits', 4, 'Number of bits to use for quantizing weights')
DEFINE_integer('nuql_activation_bits', 32, 'Number of bits to use for quantizing activations')
DEFINE_boolean('nuql_use_buckets', False, 'Use bucketing or not')
DEFINE_integer('nuql_bucket_size', 256, 'Number of bucket size')
DEFINE_string('nuql_bucket_type', 'split', 'bucket type: [split, channel]')
DEFINE_integer('nuql_quant_epochs', 60, 'To be determined by datasets')
DEFINE_boolean('nuql_quantize_all_layers', False, 'If False, leaving first and last layers unquantized')
DEFINE_boolean('nuql_enbl_rl_agent', False, 'enable the RL agent')
DEFINE_string('nuql_save_quant_model_path', './nuql_quant_models/model.ckpt', 'dir to save quantization model')


def setup_bnds_decay_rates(model_name, dataset_name):
    """learner.py:52-73; the lenet crash is patched like in the uniform learner (SURVEY A.6-1)."""
    batch_size = FLAGS.batch_size if not FLAGS.enbl_multi_gpu else FLAGS.batch_size * mgw.size()
    nb_batches_per_epoch = int(FLAGS.nb_smpls_train / batch_size)
    mgw_size = int(mgw.size()) if FLAGS.enbl_multi_gpu else 1
    init_lr = FLAGS.lrn_rate_init * FLAGS.batch_size * mgw_size / FLAGS.batch_size_norm \
        if FLAGS.enbl_multi_gpu else FLAGS.lrn_rate_init
    if dataset_name == 'cifar_10':
        # (the NUQ constants differ from the UQ ones: epochs 40/80, rates 1e-4..1e-6 — pinned against the reference
        # function by tests/test_oracle_kat.py, which caught the UQ values having been carried over here)
        bnds = [nb_batches_per_epoch * 40, nb_batches_per_epoch * 80]
        decay_rates = [1e-4, 1e-5, 1e-6]
    elif dataset_name == 'ilsvrc_12':
        if model_name.startswith('resnet'):
            bnds = [nb_batches_per_epoch * 5, nb_batches_per_epoch * 20]
            decay_rates = [5e-4, 5e-5, 5e-6]
        else:
            bnds = [nb_batches_per_epoch * 5, nb_batches_per_epoch * 30]
            decay_rates = [1e-4, 1e-5, 1e-6]
    else:
        raise ValueError('Unrecognized dataset name')
    finetune_steps = nb_batches_per_epoch * FLAGS.nuql_quant_epochs
    init_lr = init_lr if FLAGS.enbl_warm_start else FLAGS.lrn_rate_init
    return init_lr, bnds, decay_rates, finetune_steps


class NonUniformQuantLearner(AbstractLearner):
    # pylint: disable=too-many-instance-attributes
    def __init__(self, sm_writer, model_helper):
        super(NonUniformQuantLearner, self).__init__(sm_writer, model_helper)
        # learner.py:254-268 tests for 'cluster' / 'both' / 'weights' (the flag's help text says 'clusters'; that
        # spelling ends in the reference's ValueError too)
        if FLAGS.nuql_opt_mode not in ('weights', 'cluster', 'both'):
            raise ValueError('Unknown optimization mode')
        if FLAGS.enbl_dst:
            self.helper_dst = DistillationHelper(sm_writer, model_helper, self.mpi_comm)
        self.statistics = {}
        self._rl_initial_state = None
        if FLAGS.nuql_enbl_rl_agent and FLAGS.nuql_opt_mode != 'weights':
            raise NotImplementedError('--nuql_enbl_rl_agent searches bit-widths in the \'weights\' optimisation mode only')
        self.__build_train()
        if FLAGS.nuql_enbl_rl_agent:
            # the step is compiled with the flag bit-widths; the search drives that step with per-roll-out bit-widths
            # and leaves the best allocation in place (learner.py:95-116)
            self.auto_barrier()
            bit_optimizer = BitOptimizer(self.dataset_name, self.weights, self.statistics, tuner=self,
                                         barrier_fn=self.auto_barrier)
            self.optimal_w_bit_list, self.optimal_a_bit_list = bit_optimizer.run()
            self.rl_restore()
            self.rl_set_bits(self.optimal_w_bit_list, self.optimal_a_bit_list)
            self.auto_barrier()

    def train(self, nb_iters=None):
        total = self.finetune_steps if nb_iters is None else nb_iters
        ex = self.sess_train
        if FLAGS.enbl_warm_start:
            # use the latest model for warm start, THEN fit the codebooks to it (learner.py:124-129); the pre-trained
            # checkpoint holds no codebooks (saver_train is built before the graph is quantized, :209)
            self.restore_model(FLAGS.save_path, optional=('/clusters',))
            self.cluster_init()
        if FLAGS.enbl_multi_gpu:
            mgw.broadcast_global_variables([ex.store.P, ex.store.O])
        time_prev = timer()
        for idx_iter in range(total):
            self.train_step()
            if (idx_iter + 1) % FLAGS.summ_step == 0 and self.is_primary_worker():
                r = ex.fetch_losses()
                speed = FLAGS.batch_size * FLAGS.summ_step / (timer() - time_prev) * (mgw.size() if FLAGS.enbl_multi_gpu else 1)
                print('iter #%d: lr = %e | model_loss = %.4f | loss = %.4f | acc_top1 = %.4f | speed = %.2f pics / sec'
                      % (idx_iter + 1, self.lrn_rate(idx_iter), r['model_loss'], r['loss'], r['acc_top1'], speed))
                time_prev = timer()
            # save & evaluate the model at certain steps (learner.py:148-153)
            if (idx_iter + 1) % FLAGS.save_step == 0:
                self.__save_model()
                self.evaluate()
                self.auto_barrier()
        self.__save_model()
        self.evaluate()

    def __save_model(self):
        if not self.is_primary_worker():
            return
        ex = self.sess_train
        # the codebooks are variables of the model scope and travel with its checkpoints, as in the reference
        print('quantized model saved to ' + save_checkpoint(FLAGS.nuql_save_quant_model_path, ex.store.state_dict(),
                                                            ex.step_count))

    def train_step(self):
        ex = self.sess_train
        self.h2d_bytes = self.feed(ex, self.iterator_train)
        ex.run_step(self.lrn_rate(ex.step_count), self.grad_allreduce())

    def evaluate(self, nb_iters=None):
        if not self.is_primary_worker():
            return None
        self.restore_for_eval(FLAGS.nuql_save_quant_model_path)
        ex = self.sess_train
        out = []
        for _ in range(self.eval_nb_iters(nb_iters)):
            self.feed(ex, self.eval_iterator())
            ex.forward_eval_loss()
            out.append(ex.fetch_losses()['loss'])
        if FLAGS.nuql_use_buckets:
            self.__show_bucket_storage(self.bucket_storage)
        return float(np.mean(out))

    def __show_bucket_storage(self, bucket_storage):
        """learner.py:470-476: the per-bucket alpha / beta against the quantized weights' own bits"""
        bits = FLAGS.nuql_weight_bits if not FLAGS.nuql_enbl_rl_agent else FLAGS.nuql_equivalent_bits
        weight_storage = sum(self.statistics['num_weights']) * bits
        print('bucket storage: %d bit / %.3f kb | weight storage: %d bit / %.3f kb | ratio: %.3f'
              % (bucket_storage, bucket_storage / (8. * 1024.), weight_storage, weight_storage / (8. * 1024.),
                 bucket_storage * 1. / weight_storage))

    # ------------------------------------------------------------------ what the RL bit search drives
    def rl_restore(self):
        """Back to the pre-trained weights with a fresh optimizer (bit_optimizer.py:200-206): the latest checkpoint under
        --save_path if there is one, else the state this learner was built with."""
        ex = self.sess_train
        if self._rl_initial_state is None:
            ckpt_dir = os.path.dirname(FLAGS.save_path)
            fn = latest_checkpoint(ckpt_dir) if os.path.isdir(ckpt_dir) else None
            self._rl_initial_state = load_checkpoint(fn) if fn is not None else ex.store.state_dict()
        ex.store.load_state_dict(self._rl_initial_state, strict=False)
        ex.reset_optimizer_state()
        if FLAGS.enbl_multi_gpu:
            mgw.broadcast_global_variables([ex.store.P, ex.store.O])

    def rl_set_bits(self, w_bits, a_bits):
        """New bit-widths, then the codebooks re-fitted to the (restored) weights: a layer's codebook has 2^bits entries"""
        self.sess_train.set_quant_bits(w_bits, a_bits)
        self.cluster_init()

    def rl_finetune(self, nb_steps, disp_steps):
        for t_step in range(nb_steps):
            self.train_step()
            if disp_steps and (t_step + 1) % disp_steps == 0 and self.is_primary_worker():
                r = self.sess_train.fetch_losses()
                print('iter #%d: model_loss = %.4f | loss = %.4f | acc_top1 = %.4f'
                      % (t_step + 1, r['model_loss'], r['loss'], r['acc_top1']))
        self.sess_train.step_count = 0

    def rl_evaluate(self):
        """(loss, top-1, top-5) averaged over nb_smpls_eval // batch_size_eval mini-batches"""
        ex = self.sess_train
        rows = []
        bs = self.iterator_train.batch_size if FLAGS.data_dir_local else FLAGS.batch_size_eval
        for _ in range(max(1, FLAGS.nb_smpls_eval // bs)):
            self.feed(ex, self.eval_iterator())
            ex.forward_eval_loss()
            r = ex.fetch_losses()
            rows.append((r['loss'], r['acc_top1'], r['acc_top5']))
        loss, top1, top5 = [float(v) for v in np.mean(np.array(rows, np.float64), axis=0)]
        return loss, top1, top5

    def cluster_init(self):
        """ops['cluster_init'] (learner.py:127-129, 297-298): run AFTER the weights are restored."""
        self.sess_train.wq.quantile_init()

    def __build_train(self):
        self.graph_train = G.Graph()
        with self.graph_train.as_default():
            with G.variable_scope(self.data_scope):
                self.iterator_train = self.build_dataset_train()
                images, labels = self.iterator_train.get_next()
            self.images, self.labels = images, labels
            logits_dst = self.helper_dst.calc_logits(None, images) if FLAGS.enbl_dst else None
            with G.variable_scope(self.model_scope):
                logits = self.forward_train(images)
                self.weights = [v for v in self.trainable_vars if 'kernel' in v.name or 'weight' in v.name]
                if not FLAGS.nuql_quantize_all_layers:
                    self.weights = self.weights[1:-1]
                self.statistics['num_weights'] = [v.numel for v in self.weights]
                nq = NonUniformQuantization(self.graph_train, FLAGS.nuql_bucket_size, FLAGS.nuql_use_buckets,
                                            FLAGS.nuql_init_style, FLAGS.nuql_bucket_type,
                                            codebook_bits_cap=FLAGS.nuql_w_bit_max if FLAGS.nuql_enbl_rl_agent else None)
                matmul_ops = nq.search_matmul_op(FLAGS.nuql_quantize_all_layers)
                act_ops = nq.search_activation_op()
                self.statistics['nb_matmuls'], self.statistics['nb_activations'] = len(matmul_ops), len(act_ops)
                w_bits = [FLAGS.nuql_weight_bits] * len(matmul_ops)
                a_bits = [FLAGS.nuql_activation_bits] * len(act_ops)
                self.optimal_w_bit_list, self.optimal_a_bit_list = w_bits, a_bits
                nq.insert_quant_op_for_weights({op.name: b for op, b in zip(matmul_ops, w_bits)})
                nq.insert_quant_op_for_activations({op.name: b for op, b in zip(act_ops, a_bits)})
                self.bucket_storage = nq.bucket_storage
                # "Strictly speaking, clusters should be not included for regularization" (learner.py:219-220): they are
                loss, metrics = self.calc_loss(labels, logits, self.trainable_vars)
                if FLAGS.enbl_dst:
                    loss += self.helper_dst.calc_loss(logits, logits_dst)
                # the variables the optimizer updates (learner.py:252-268): the codebooks ('cluster'), everything else
                # ('weights') or all trainable variables ('both')
                clusters = [v for v in self.trainable_vars if 'clusters' in v.name]
                rest = [v for v in self.trainable_vars if v not in clusters]
                frozen = {'weights': clusters, 'cluster': rest, 'both': []}[FLAGS.nuql_opt_mode]
        init_lr, bnds, decay_rates, self.finetune_steps = setup_bnds_decay_rates(self.model_name, self.dataset_name)
        self.lrn_rate = piecewise_constant(list(bnds), [init_lr * d for d in decay_rates])
        world = mgw.size() if FLAGS.enbl_multi_gpu else 1
        teacher = None
        if FLAGS.enbl_dst:
            teacher = Executor(self.graph_train, images, logits_dst, self.device, train=False, seed=2)
            self.helper_dst.restore(teacher.store)
        wq_spec = nq.weight_quant_spec()
        if wq_spec is not None:
            wq_spec['train_clusters'] = FLAGS.nuql_opt_mode in ('cluster', 'both')
        self.sess_train = Executor(self.graph_train, images, logits, self.device, train=True, loss=loss, labels=labels,
                                   optimizer=dict(kind='adam'), weight_quant=wq_spec,
                                   act_quant=nq.act_quant_spec(), teacher=teacher, seed=1, grad_scale=1.0 / world,
                                   frozen=frozen)
        if teacher is not None:
            teacher.buf[images] = self.sess_train.buf[images]
            self.sess_train.share_im2col_from(teacher)
        self.cluster_init()
