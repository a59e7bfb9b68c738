"""Util functions for Non-Uniform Quantization — graph-editing surface of the reference
(/root/reference/learners/nonuniform_quantization/utils.py:31-476).  Weights go through the codebook
quantizer (pf_nuq_weight_quant), activations through the UNIFORM quantizer (utils.py:58-85)."""
import numpy as np

from ...ops import nuq_bucket_layout
from ..uniform_quantization.utils import prefix_filter


class NonUniformQuantization:
    # pylint: disable=too-many-instance-attributes
    def __init__(self, sess, bucket_size=0, use_buckets=False, init_style='quantile', bucket_type='split',
                 codebook_bits_cap=None):
        """codebook_bits_cap: size the codebook variables for this many bits (the RL bit search changes a layer's
        bit-width at run time; its codebook then uses the first 2^bits entries)."""
        self.sess = sess
        self.codebook_bits_cap = codebook_bits_cap
        self.use_buckets = use_buckets
        self.bucket_size = bucket_size
        self.bucket_type = bucket_type
        self.init_style = init_style
        self.matmul_ops, self.activation_ops = [], []
        self.quantized_matmul_ops, self.quantized_activation_ops = [], []
        self.weight_bits, self.activation_bits = [], []
        self.bucket_storage = 0
        if self.bucket_size < 0:
            raise ValueError("Bucket size must be a postive integer")
        if self.bucket_type not in ('split', 'channel'):
            raise ValueError("Unrecognized bucket type, must be 'weight' or 'channel'.")
        if self.init_style not in ('quantile', 'uniform'):
            raise ValueError("Unrecognized Initialization Mode.")
        if self.use_buckets and self.init_style == 'uniform':
            # __bucket_quantize calls __uniform_init(x_normalized, k) (utils.py:225) against its signature
            # __uniform_init(nb_clusters, bucket_num=0) (:368): the reference cannot run this combination
            raise ValueError('--nuql_init_style uniform with --nuql_use_buckets is broken in the reference '
                             '(__uniform_init is called with the wrong arguments, SURVEY A.6-6); use quantile')
        self.support_act_types = ['Relu', 'Relu6', 'Crelu', 'Elu', 'Selu', 'Softplus', 'Softsign', 'Sigmoid', 'Tanh']
        self.support_mul_types = ['Conv2D', 'MatMul', 'DepthwiseConv2dNative']

    def search_matmul_op(self, quantize_all_layers):
        is_student_fn = lambda x: 'distilled' not in x.name
        for op in self.sess.get_operations():
            if op.type in self.support_mul_types and is_student_fn(op):
                self.matmul_ops.append(op)
        if not quantize_all_layers:
            self.matmul_ops = self.matmul_ops[1:-1]
        return self.matmul_ops

    def search_activation_op(self):
        is_student_fn = lambda x: 'distilled' not in x.name
        for op in self.sess.get_operations():
            if op.type in self.support_act_types and is_student_fn(op):
                self.activation_ops.append(op)
        return self.activation_ops

    def insert_quant_op_for_weights(self, w_bit_dict):
        """Marks the ops and creates each one's codebook variable — tf.get_variable('clusters', initializer=init_c) under
        variable_scope(prefix + '/nonuniform_quantize') inside the learner's model scope (utils.py:180, :297): a
        TRAINABLE variable of 2^bits quantization points on [0, 1], named like the reference's so that checkpoints
        interchange.  Its value is set by the learner's cluster_init (quantiles of the restored weights)."""
        g = self.sess
        for op in self.matmul_ops:
            bits = int(w_bit_dict[op.name])
            self.quantized_matmul_ops.append(op)
            self.weight_bits.append(bits)
            if self.use_buckets:
                # __bucket_quantize: a [k, bucket_num] `clusters` variable under <prefix>/nonuniform_bucket_quantize
                # (utils.py:209, :324) for EVERY quantized op, depthwise included; bucket_storage as :487-494
                ncols, _, _ = nuq_bucket_layout(op.vars['kernel'].shape, self.bucket_type, self.bucket_size)
                name = g.scope_prefix() + prefix_filter(op.name) + '/nonuniform_bucket_quantize/clusters'
                op.vars['clusters'] = g.get_variable(name, (2 ** max(bits, self.codebook_bits_cap or 0), ncols),
                                                     lambda rng, shape: np.zeros(shape, np.float32), trainable=True)
                self.bucket_storage += ncols * 32 * 2
            elif op.type != 'DepthwiseConv2dNative' and bits <= 8:
                name = g.scope_prefix() + prefix_filter(op.name) + '/nonuniform_quantize/clusters'
                op.vars['clusters'] = g.get_variable(name, (2 ** max(bits, self.codebook_bits_cap or 0),), lambda rng, shape: np.zeros(shape, np.float32),
                                                     trainable=True)

    def insert_quant_op_for_activations(self, act_bit_dict):
        for op in self.activation_ops:
            if op.type not in ('Relu', 'Relu6'):
                raise NotImplementedError("The activation_fn needs to include %s manually" % op.type)
            self.quantized_activation_ops.append(op)
            self.activation_bits.append(int(act_bit_dict[op.name]))

    def weight_quant_spec(self):
        if not self.quantized_matmul_ops:
            return None
        spec = dict(kind='nonuniform', ops=self.quantized_matmul_ops, bits=self.weight_bits,
                    init_style=self.init_style, train_clusters=False)
        if self.use_buckets:
            spec.update(use_buckets=True, bucket_type=self.bucket_type, bucket_size=self.bucket_size)
        return spec

    def act_quant_spec(self):
        if not self.quantized_activation_ops:
            return None
        return dict(ops=self.quantized_activation_ops, bits=self.activation_bits)
