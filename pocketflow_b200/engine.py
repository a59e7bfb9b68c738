"""Executor: lowers a `graph.Graph` to launches of libpf_b200.so kernels (forward, backward,
gradient reduction, optimizer) and replays them through a CUDA graph.

This is the stand-in for `sess.run(train_op)` into TensorFlow's executor
(/root/reference/learners/uniform_quantization/learner.py:114-152): one call = one training step
on one GPU.  State layout (B200, 180 GB HBM): all trainable parameters, their gradients and the
optimizer slots live in FLAT fp32 buffers so that (a) the data-parallel gradient reduction is one
collective over one buffer (SURVEY §8e) and (b) the optimizer / mask / weight-decay work is a
handful of launches instead of ~110 per step.
"""
import contextlib
import os
from collections import OrderedDict

import numpy as np
import torch

from . import ops

F32 = np.float32
MATMUL_TYPES = ('Conv2D', 'MatMul', 'DepthwiseConv2dNative')
ACT_TYPES = {'Relu': 1, 'Relu6': 2}


def _align4(n):
    return (n + 3) // 4 * 4


class ParamStore:
    """Flat storage for the trainable variables of one model scope (+ separate non-trainable store).

    Order: maskable variables first, then by weight-decay coefficient, so that the optimizer runs
    over at most a few contiguous ranges."""

    def __init__(self, variables, device, wd_of=None, maskable=None, seed=1, frozen=None):
        """frozen: trainable variables the optimizer must NOT update (they still count in the weight-decay loss and
        receive gradients): the codebooks in the non-uniform learner's 'weights' mode, everything but the codebooks in
        its 'cluster' mode (learners/nonuniform_quantization/learner.py:252-268).  They form their own ranges."""
        self.device = device
        wd_of = wd_of or {}
        maskable = set(maskable or [])
        frozen = set(frozen or [])
        train = [v for v in variables if v.trainable]
        other = [v for v in variables if not v.trainable]
        key = lambda v: (0 if v in maskable else 1, 1 if v in frozen else 0, -float(wd_of.get(v, 0.0)))
        order = sorted(range(len(train)), key=lambda i: (key(train[i]), i))
        self.train_vars = [train[i] for i in order]
        self.other_vars = other
        self.offset, self.ranges = {}, []      # ranges: (start, end, masked, wd)
        self.frozen_ranges = set()             # (start, end) of the ranges the optimizer skips
        pos = 0
        cur = None

        def close(cur, pos):
            self.ranges.append((cur[0], pos, cur[2], cur[3]))
            if cur[4]:
                self.frozen_ranges.add((cur[0], pos))
        for v in self.train_vars:
            k = (v in maskable, float(wd_of.get(v, 0.0)), v in frozen)
            if cur is None or cur[2:] != k:
                if cur is not None:
                    close(cur, pos)
                cur = (pos, None) + k
            self.offset[v] = pos
            pos += _align4(v.numel)
        if cur is not None:
            close(cur, pos)
        self.n_train = max(pos, 4)
        self.n_masked = max([e for (s, e, m, w) in self.ranges if m] + [0])
        opos = 0
        for v in other:
            self.offset[v] = opos
            opos += _align4(v.numel)
        self.n_other = max(opos, 4)
        self.P = torch.zeros(self.n_train, dtype=torch.float32, device=device)
        self.O = torch.zeros(self.n_other, dtype=torch.float32, device=device)
        self.listeners = []                     # called after every bulk (re)load of the parameters
        self.init(seed)

    def init(self, seed):
        rng = np.random.default_rng(seed)
        hp = np.zeros(self.n_train, F32)
        for v in sorted(self.train_vars, key=lambda v: v.name):
            hp[self.offset[v]:self.offset[v] + v.numel] = v.initializer(rng, v.shape).reshape(-1)
        ho = np.zeros(self.n_other, F32)
        for v in self.other_vars:
            ho[self.offset[v]:self.offset[v] + v.numel] = v.initializer(rng, v.shape).reshape(-1)
        self.P.copy_(torch.from_numpy(hp))
        self.O.copy_(torch.from_numpy(ho))
        for f in self.listeners:
            f()

    def view(self, v, flat=None):
        buf = flat if flat is not None else (self.P if v.trainable else self.O)
        o = self.offset[v]
        return buf[o:o + v.numel].view(v.shape)

    def state_dict(self):
        d = OrderedDict()
        for v in self.train_vars + self.other_vars:
            d[v.name] = self.view(v).detach().cpu().numpy().copy()
        return d

    def load_state_dict(self, d, strict=True, require=None, optional=()):
        """Copy the variables `d` names into the store.  Returns (trainable variables found, trainable variables).
        strict: every variable must be present.  require ('any' | 'all' | None) applies to the TRAINABLE variables of a
        non-strict load: a checkpoint of another net / scope matches nothing and must not pass for a restore;
        variables whose name contains one of the `optional` substrings are not required."""
        found = 0
        for v in self.train_vars + self.other_vars:
            if v.name in d:
                a = np.asarray(d[v.name], F32)
                if a.size != v.numel:
                    raise ValueError('checkpoint variable %s has %d elements, the model\'s has %d'
                                     % (v.name, a.size, v.numel))
                self.view(v).copy_(torch.from_numpy(a.reshape(v.shape)))
                found += 1 if v.trainable else 0
            elif strict:
                raise KeyError('missing variable in checkpoint: ' + v.name)
        needed = [v for v in self.train_vars if not any(o in v.name for o in optional)]
        total = len(needed)
        found = sum(1 for v in needed if v.name in d)
        if require is not None and total > 0:
            if found == 0 or (require == 'all' and found < total):
                missing = [v.name for v in needed if v.name not in d][:5]
                raise ValueError('checkpoint matches %d of the model\'s %d trainable variables (e.g. missing %s; the '
                                 'checkpoint holds %s ...)' % (found, total, missing, sorted(d)[:3]))
        for f in self.listeners:
            f()
        return found, total


class Executor:
    """Forward (+ backward + update) of one graph on one GPU."""

    def __init__(self, graph, images, logits, device, store=None, train=True, loss=None, labels=None,
                 optimizer=None, weight_quant=None, act_quant=None, maskable=None, teacher=None,
                 seed=1, exact_ste=True, grad_scale=1.0, scope=None, conv_path=None, fuse_add=True,
                 update_moving_stats=True, frozen=None):
        self.g, self.device, self.train = graph, device, train
        # fuse_add=False: every Conv2D output is materialised on its own (the channel-pruning learner regresses conv
        # outputs of a pruned model onto those of the full model, learners/channel_pruning_gpu/learner.py:339-354);
        # update_moving_stats=False: training-mode BN without the moving-average update ops (the FULL model of that
        # learner runs forward_train but only the pruned model's update ops are ever executed, :283-286)
        self.fuse_add, self.update_moving_stats = bool(fuse_add), bool(update_moving_stats)
        self.images, self.logits_t, self.labels_t = images, logits, labels
        self.loss, self.teacher = loss, teacher
        self.optimizer = optimizer or {}
        self.exact_ste, self.grad_scale = exact_ste, float(grad_scale)
        # 'tc': tcgen05 split-bf16 conv where the shape allows (Cin, Cout multiples of 16), exact-fp32
        # CUDA-core kernels elsewhere; 'fp32': exact-fp32 everywhere (the on-device reference)
        import os as _os
        self.conv_path = conv_path or _os.environ.get('PF_CONV_PATH', 'tc')
        self.ops = self._reachable_ops(logits)
        variables = []
        for op in self.ops:
            for v in op.vars.values():
                if v not in variables:
                    variables.append(v)
        self.variables = variables
        wd_of = dict(loss.l2) if loss is not None else {}
        self.wd_of = wd_of
        self.maskable = [v for v in (maskable or []) if v in variables]
        # an inference-only executor that owns its parameters (the distillation teacher): the split-bf16 weight
        # copies are prepared once and refreshed only when the store is (re)loaded
        self.static_weights = (not train) and store is None
        self._static_ready = False
        self.store = store or ParamStore(variables, device, wd_of, self.maskable, seed, frozen=frozen)
        if self.static_weights:
            self.store.listeners.append(self._invalidate_static)
        self.weight_quant, self.act_quant = weight_quant, act_quant
        self.prof = None
        # multi-stream overlap inside one step (captured into the CUDA graph as parallel branches): the teacher's
        # forward runs beside the student's, and the weight-gradient kernels run beside dgrad + BN-backward, so that
        # tensor-bound and HBM-bound kernels share the GPU (a BN kernel's CTAs fit next to a persistent conv CTA)
        self.overlap = _os.environ.get('PF_OVERLAP', '1') != '0' and device.type == 'cuda'
        self.side = torch.cuda.Stream(device=device) if self.overlap else None
        self.side2 = torch.cuda.Stream(device=device) if self.overlap else None
        self._shares_cols = False
        self._side_active = False
        self.cols_event = None          # recorded after this executor's im2col (shared columns)
        self.cols_wait = None           # event to wait for before reading shared columns
        self._plan()
        self._graph = None
        self.step_count = 0

    def _invalidate_static(self):
        """Parameters were (re)loaded: refresh the prepared weight copies now (a captured CUDA graph that contains
        this executor's forward does not re-run the preparation)."""
        self._static_ready = False
        if hasattr(self, 'tc'):
            self.prepare_static_weights()

    def prepare_static_weights(self):
        for op in self.ops:
            if op in self.im2col:
                im, wk = self.im2col[op], self.kernel_of(op)
                self._stem_weights(im, wk)
            elif op in self.tc:
                self.tc[op].prepare(self.kernel_of(op))
        self._static_ready = True

    def _stem_weights(self, im, wk):
        """fp32 kernel of the first layer -> the (re-arranged / padded) matrix its tensor-core conv multiplies by"""
        k = wk.shape[-1]
        if im['mode'] == 's2d':
            ops.gather_rows(wk, im['fwd_map'], im['wpad'], k)
        else:
            ops.add(wk.reshape(-1), None, im['wpad'][:wk.numel()])       # rows >= R*S*C stay zero
        im['tw'].prepare(im['wpad'])

    # ------------------------------------------------------------------ planning
    def _reachable_ops(self, out):
        seen, order = set(), []

        def visit(t):
            if t.op in seen:
                return
            seen.add(t.op)
            for i in t.op.inputs:
                visit(i)
            order.append(t.op)
        import sys
        sys.setrecursionlimit(max(10000, sys.getrecursionlimit()))
        visit(out)
        pos = {op: i for i, op in enumerate(self.g.ops)}
        return sorted(order, key=lambda o: pos[o])

    def _consumers(self, t):
        return [c for c in t.consumers if c in self._opset]

    def _plan(self):
        dev = self.device
        self._opset = set(self.ops)
        st = self.store
        # PF_POISON=1 (debugging): every scratch / activation buffer starts as NaN, so that a read of memory no kernel
        # has written this step shows up in the losses instead of depending on what the allocator recycled
        poison = os.environ.get('PF_POISON', '0') == '1'
        E = (lambda shape: torch.full(shape, float('nan'), dtype=torch.float32, device=dev)) if poison else \
            (lambda shape: torch.empty(shape, dtype=torch.float32, device=dev))
        self.buf, self.alias = {}, {}
        self.fused_act, self.fused_into = {}, {}
        # ---- fusion: BN -> Relu/Relu6 and Conv/MatMul(bias) -> Relu with a single consumer
        for op in self.ops:
            if op.type in ACT_TYPES:
                src = op.inputs[0].op
                if src.type in ('FusedBatchNorm', 'Conv2D', 'MatMul') and len(self._consumers(src.output)) == 1:
                    if src.type == 'FusedBatchNorm' or op.type == 'Relu':
                        self.fused_act[src] = ACT_TYPES[op.type]
                        self.fused_into[op] = src
                        continue
                raise NotImplementedError('activation %s is not preceded by a fusable producer' % op.name)
        # ---- quantization marks
        self.wq_ops = list(self.weight_quant['ops']) if self.weight_quant else []
        self.aq_ops = list(self.act_quant['ops']) if self.act_quant else []
        self.aq_index = {op: i for i, op in enumerate(self.aq_ops)}
        self.aq_slots = torch.zeros(max(len(self.aq_ops), 1), 2, dtype=torch.int32, device=dev)
        self.aq_out = {}           # relu op -> out-of-place quantized buffer (producer is not BN)
        # quantized weights live in a flat buffer with the same offsets as the parameters
        self.QW = torch.zeros(st.n_train, dtype=torch.float32, device=dev) if self.wq_ops else None
        self.wq = None
        if self.wq_ops:
            kvars = [op.vars['kernel'] for op in self.wq_ops]
            srcs = [st.view(v) for v in kvars]
            dsts = [st.view(v, self.QW) for v in kvars]
            wq = self.weight_quant
            if wq.get('kind', 'uniform') == 'uniform':
                self.wq = ops.UniformWeightQuantizer(srcs, dsts, wq['bits'], wq.get('use_buckets', False),
                                                     wq.get('bucket_type', 'channel'), wq.get('bucket_size', 256))
            else:
                # codebooks: the reference's trainable `clusters` variables when the graph carries them (then they
                # live in the parameter store), else a private table of the quantizer
                cvars = [op.vars.get('clusters') for op in self.wq_ops]
                self.train_clusters = bool(wq.get('train_clusters', False)) and self.train
                if wq.get('use_buckets', False):
                    # per-bucket codebooks: always the [k, ncols] `clusters` variables of the graph edit.  They are
                    # consumed through QW like every codebook (the integer-level conv operands are uniform-only)
                    self.wq = ops.CodebookWeightQuantizer(srcs, dsts, wq['bits'], keep_index=self.train_clusters,
                                                          cluster_views=[st.view(c) for c in cvars], cluster_base=st.P,
                                                          use_buckets=True, bucket_type=wq['bucket_type'],
                                                          bucket_size=wq['bucket_size'])
                elif all(c is not None for c in cvars):
                    self.wq = ops.CodebookWeightQuantizer(srcs, dsts, wq['bits'], keep_index=self.train_clusters,
                                                          cluster_views=[st.view(c) for c in cvars], cluster_base=st.P)
                else:
                    if self.train_clusters:
                        raise ValueError('training the codebooks needs `clusters` variables on the quantized ops')
                    self.wq = ops.CodebookWeightQuantizer(srcs, dsts, wq['bits'])
        self.qvars = {op: op.vars['kernel'] for op in self.wq_ops}
        # ---- tensors
        for op in self.ops:
            t = op.output
            if op.type == 'Placeholder':
                self.buf[t] = E(t.shape)
                self.buf[t].zero_()
            elif op.type in ('Reshape', 'Identity'):
                self.alias[t] = op.inputs[0]
            elif op in self.fused_into:
                self.alias[t] = op.inputs[0]
            else:
                self.buf[t] = E(t.shape)
            if op in self.aq_index and self.fused_into.get(op) is not None and \
                    self.fused_into[op].type != 'FusedBatchNorm':
                self.aq_out[op] = E(t.shape)
        # ---- per-op scratch
        self.bn = {}
        self.tc = {}
        self.tc_wgrad = set()
        self.im2col = {}
        self.pool_argmax = {}
        max_ws, max_wt, max_bnws = 4, 4, 4
        self.desc = {}
        for op in self.ops:
            if op.type == 'FusedBatchNorm':
                c = op.output.shape[-1]
                self.bn[op] = dict(mean=E((c,)), var=E((c,)), rstd=E((c,)))
                max_bnws = max(max_bnws, 5 * c * ops.BN_MAX_SPLITS)
            if op.type in ('Conv2D', 'MatMul'):
                x, y = op.inputs[0], op.output
                if op.type == 'Conv2D':
                    n, h, w, c = x.shape
                    _, p, q, k = y.shape
                    (kh, kw), (sh, sw), (pt, pl) = op.attrs['ksize'], op.attrs['strides'], op.attrs['pad']
                    d = ops.conv_desc(n, h, w, c, k, kh, kw, p, q, sh, sw, pt, pl)
                else:
                    n, c = x.shape
                    k = y.shape[1]
                    d = ops.conv_desc(n, 1, 1, c, k, 1, 1, 1, 1, 1, 1, 0, 0)
                self.desc[op] = d
                if self.conv_path == 'tc' and op.type == 'Conv2D' and not ops.conv2d_tc_supported(d) \
                        and k % 16 == 0 and c % 16 != 0 and x.op.type == 'Placeholder':
                    # first layer (Cin = 3): explicit im2col into kpad channels, then a 1x1 tensor-core conv
                    kdim = kh * kw * c
                    kpad = (kdim + 15) // 16 * 16
                    d1 = ops.conv_desc(n, p, q, kpad, k, 1, 1, p, q, 1, 1, 0, 0)
                    # columns directly in operand planes when every consumer is a tensor-core kernel
                    as_planes = (not self.train) or ops.conv2d_tc_wgrad_supported(d1)
                    mode = 'im2col'
                    # fewer than 64 output channels (MobileNet's 3 -> 32 stem): the tensor-core wgrad wants Cout % 64 == 0,
                    # so g = 64 / Cout pixels share one GEMM row — cols [pixels, kpad] and dy [pixels, k] are read as
                    # [pixels / g, g kpad] and [pixels / g, g k]; the weight gradient is the sum of the g diagonal
                    # kpad x k blocks of the (g kpad) x (g k) result (the exact-fp32 CUDA-core wgrad of this layer took
                    # 4.3 of MobileNet's 23 ms: profiles/r2_ncu_launchlist_mobilenet_step_v1.txt)
                    pair = None
                    if self.train and not as_planes and k in (16, 32) and (kpad * (64 // k)) % 64 == 0 \
                            and (p * q) % (64 // k) == 0:
                        g_ = 64 // k
                        dp = ops.conv_desc(n, 1, p * q // g_, kpad * g_, k * g_, 1, 1, 1, p * q // g_, 1, 1, 0, 0)
                        if ops.conv2d_tc_wgrad_supported(dp):
                            pair, as_planes = dict(g=g_, d=dp), True
                    if sh == 2 and sw == 2 and 4 * c <= 16 and os.environ.get('PF_STEM_S2D', '1') != '0':
                        # stride-2 stem: space-to-depth instead of im2col — a stride-1 conv over 16 channels that the
                        # tensor-core kernels gather themselves (no 2 GB column matrix)
                        r2, s2, fwd_map, bwd_map = ops.s2d_weight_maps(kh, kw, c, 16)
                        d2 = ops.conv_desc(n, p + r2 - 1, q + s2 - 1, 16, k, r2, s2, p, q, 1, 1, 0, 0)
                        if ops.conv2d_tc_supported(d2) and ((not self.train) or ops.conv2d_tc_wgrad_supported(d2)):
                            mode, d1, as_planes, kpad = 's2d', d2, True, r2 * s2 * 16
                    self.im2col[op] = dict(kdim=kdim, kpad=kpad, d1=d1, compute=True, planes=as_planes, mode=mode,
                                           cols=ops.Planes(n * d1.h * d1.w * d1.c, dev) if as_planes else E((n * p * q, kpad)),
                                           wpad=torch.zeros(kpad * k, dtype=torch.float32, device=dev),
                                           tw=ops.TcWeights(d1, dev, need_dgrad=False))
                    if mode == 's2d':
                        self.im2col[op]['fwd_map'] = torch.from_numpy(fwd_map).to(dev)
                        self.im2col[op]['bwd_map'] = torch.from_numpy(bwd_map).to(dev)
                    if self.train:
                        self.im2col[op]['dwpad'] = torch.zeros(kpad * k, dtype=torch.float32, device=dev)
                        if pair is not None and mode == 'im2col':
                            pair['dw'] = torch.zeros(pair['g'] * kpad * pair['g'] * k, dtype=torch.float32, device=dev)
                            self.im2col[op]['pair'] = pair
                            max_ws = max(max_ws, ops.conv2d_tc_wgrad_planes_workspace_floats(pair['d']))
                            self._stem_dy = max(getattr(self, '_stem_dy', 8), n * p * q * k)
                        if ops.conv2d_tc_wgrad_supported(d1):
                            max_ws = max(max_ws, ops.conv2d_tc_wgrad_planes_workspace_floats(d1))
                            self._stem_dy = max(getattr(self, '_stem_dy', 8), n * p * q * k)
                        max_ws = max(max_ws, ops.conv2d_wgrad_workspace_floats(d1))
                if self.conv_path == 'tc' and ops.conv2d_tc_supported(d):
                    self.tc[op] = ops.TcWeights(d, dev, need_dgrad=self.train and x.op.type != 'Placeholder')
                if self.train:
                    if op in self.tc and ops.conv2d_tc_wgrad_supported(d):
                        self.tc_wgrad.add(op)
                        max_ws = max(max_ws, ops.conv2d_tc_wgrad_planes_workspace_floats(d))
                    max_ws = max(max_ws, ops.conv2d_wgrad_workspace_floats(d))
                    max_wt = max(max_wt, op.vars['kernel'].numel)
            if op.type == 'DepthwiseConv2dNative':
                x, y = op.inputs[0], op.output
                n, h, w, c = x.shape
                _, p, q, _ = y.shape
                (kh, kw), (sh, sw), (pt, pl) = op.attrs['ksize'], op.attrs['strides'], op.attrs['pad']
                self.desc[op] = ops.conv_desc(n, h, w, c, c, kh, kw, p, q, sh, sw, pt, pl)
                if self.train:
                    max_ws = max(max_ws, ops.dwconv_wgrad_workspace_floats(self.desc[op]))
            if op.type == 'MaxPool':
                x, y = op.inputs[0], op.output
                n, h, w, c = x.shape
                _, p, q, _ = y.shape
                (kh, kw), (sh, sw), (pt, pl) = op.attrs['ksize'], op.attrs['strides'], op.attrs['pad']
                self.desc[op] = ops.conv_desc(n, h, w, c, c, kh, kw, p, q, sh, sw, pt, pl)
                if self.train:
                    self.pool_argmax[op] = torch.empty(y.shape, dtype=torch.uint8, device=dev)
        # ---- residual Add fused into the epilogue of the tcgen05 conv that produces one of its inputs:
        # the conv writes conv(x) + shortcut straight into the Add's buffer (one pass instead of three)
        self.fused_add = {}        # conv op -> (add op, other input tensor)
        self.add_fused = set()
        for op in self.ops:
            if op.type != 'Add' or not self.fuse_add:
                continue
            for i, x_t in enumerate(op.inputs):
                src, other = x_t.op, op.inputs[1 - i]
                if src.type == 'Conv2D' and src in self.tc and x_t not in self.alias and src not in self.fused_act \
                        and 'bias' not in src.vars and len(self._consumers(x_t)) == 1 \
                        and self.g.ops.index(other.op) < self.g.ops.index(src):
                    self.fused_add[src] = (op, other)
                    self.add_fused.add(op)
                    self.buf[x_t] = self.buf[op.output]       # the conv output IS the add output
                    break
        # ---- split-bf16 operand planes (tensor-core path): the BN-apply / activation-quantizer that produces a conv
        # input writes it directly in the operand format of the tcgen05 kernels (x = hi + lo, two bf16 planes);
        # the fp32 copy is only written when some other consumer needs it
        self.xplanes, self.bn_need_f32 = {}, {}
        max_x = max_dy = 8
        for op in self.ops:
            if op in self.tc and op not in self.im2col:
                r = self._root(op.inputs[0])
                if r is not None and r.op.type == 'FusedBatchNorm' and r.numel % 8 == 0:
                    if r.op not in self.xplanes:
                        self.xplanes[r.op] = ops.Planes(r.numel, dev)
                        self.bn_need_f32[r.op] = False
                elif self.train:
                    max_x = max(max_x, op.inputs[0].numel)
        for bn_op in self.xplanes:
            ts = [bn_op.output] + [c.output for c in self._consumers(bn_op.output) if c in self.fused_into]
            for t in ts:
                for c in self._consumers(t):
                    if c in self.fused_into and self.fused_into[c] is bn_op:
                        continue
                    if not (c in self.tc and c not in self.im2col and (not self.train or c in self.tc_wgrad)):
                        self.bn_need_f32[bn_op] = True
        # ---- integer-level operands (TMA-fed kernels, SURVEY §7 hard part 1b): a <= 8-bit fake-quantized tensor is
        # exactly scale * level, and the levels are exact in bf16 — one operand plane instead of hi + lo, one MMA per
        # k-slice instead of three (two against a split gradient).  Activation side: the fused BN + ReLU + fake-quant
        # pass writes levels + a device header + per-pixel channel sums when EVERY consumer of its planes is a TMA-fed
        # kernel.  Weight side: the preparation launch derives the levels from the unquantized kernel with the
        # quantizer's own op chain; needs per-layer / per-output-channel buckets and the input's channel sums.
        self.act_lv, self.w_lv = {}, {}
        use_lv = os.environ.get('PF_TC_LEVELS', '1') != '0' and self.train and dev.type == 'cuda'
        if use_lv and self.aq_ops:
            cons = {}
            for op in self.ops:
                if op in self.tc and op not in self.im2col:
                    r = self._root(op.inputs[0])
                    if r is not None and r.op in self.xplanes:
                        cons.setdefault(r.op, []).append(op)
            for bn_op, users in cons.items():
                act = self.fused_act.get(bn_op, 0)
                relu_op = self._consumers(bn_op.output)[0] if act else None
                c = bn_op.output.shape[-1]
                if relu_op not in self.aq_index or not bn_op.attrs['training'] or c < 16 or (c & (c - 1)):
                    continue
                if all(ops.conv2d_tc_tma_supported(self.desc[u], 0) and u in self.tc_wgrad
                       and ops.conv2d_tc_tma_supported(self.desc[u], 2) for u in users):
                    m = bn_op.output.numel // c
                    nseg = (c + 127) // 128
                    self.act_lv[bn_op] = dict(hdr=torch.zeros(2, dtype=torch.int32, device=dev),
                                              csum=E((m * nseg,)), nseg=nseg)
            wq = self.weight_quant
            if self.wq is not None and isinstance(self.wq, ops.UniformWeightQuantizer) and \
                    (not wq.get('use_buckets', False) or wq.get('bucket_type', 'channel') == 'channel'):
                nbk = self.wq.n_buckets
                for i, op in enumerate(self.wq_ops):
                    if op not in self.tc or op in self.im2col or op.type != 'Conv2D':
                        continue
                    r = self._root(op.inputs[0])
                    if r is None or r.op not in self.act_lv or not 1 <= self.wq.bits[i] <= 8:
                        continue
                    b0, ncols = int(self.wq.segs[i]['bucket0']), int(self.wq.segs[i]['ncols'])
                    sc = self.wq.scales
                    self.w_lv[op] = dict(index=i, ncols=ncols, alpha=sc[b0:b0 + ncols], beta=sc[nbk + b0:nbk + b0 + ncols],
                                         ralpha=sc[2 * nbk + b0:2 * nbk + b0 + ncols])
        # one launch refreshes the split-bf16 copies of all (trainable) conv kernels
        self.tc_batch = None
        if self.tc and not self.static_weights:
            tc_ops = [op for op in self.ops if op in self.tc]
            levels = {}
            for j, op in enumerate(tc_ops):
                if op in self.w_lv:
                    lv = self.w_lv[op]
                    levels[j] = (self.store.view(op.vars['kernel']), lv['alpha'], lv['beta'], lv['ralpha'], lv['ncols'],
                                 self.wq.bits[lv['index']])
                    lv['batch_index'] = j
            self.tc_batch = ops.TcWeightsBatch([(self.tc[op], self.kernel_of(op)) for op in tc_ops], dev, levels)
        self._lv_on = False            # set per forward(): levels only in training-mode passes
        if self.labels_t is not None and self.labels_t not in self.buf:
            self.buf[self.labels_t] = torch.zeros(self.labels_t.shape, dtype=torch.float32, device=dev)
        self.bn_ws = E((max_bnws,))
        n_rows = self.logits_t.shape[0]
        self.loss_out = torch.zeros(8, dtype=torch.float32, device=dev)
        self.row_ws = E((4 * n_rows,))
        if self.train:
            self.G = torch.zeros(st.n_train, dtype=torch.float32, device=dev)
            self.S1 = torch.zeros(st.n_train, dtype=torch.float32, device=dev)
            self.S2 = torch.zeros(st.n_train, dtype=torch.float32, device=dev) \
                if self.optimizer.get('kind') == 'adam' else None
            self.hp = torch.zeros(4, dtype=torch.float32, device=dev)
            # per-step scalars (lr, Adam beta powers) travel through a RING of pinned slots: the async upload of step
            # i must have executed before the host rewrites its slot (a single slot let step i pick up step i+1's
            # beta powers whenever the host ran ahead of the GPU)
            self.hp_ring = torch.zeros(16, 4, dtype=torch.float32).pin_memory() if dev.type == 'cuda' else torch.zeros(16, 4)
            self.hp_events, self._hp_i = [None] * 16, 0
            self.wgrad_ws = E((max_ws,))
            self.wgrad_ws2 = E((max_ws,)) if self.overlap else None
            self.wt_ws = E((max_wt,))
            self.l2_out = torch.zeros(4, dtype=torch.float32, device=dev)
            self.l2_ws = E((ops.L2_PARTIALS,))
            self.gbuf, self.galias = {}, {}
            self.relu_scratch = {}
            # d(out)/d(in) of a residual Add is the identity, so an input can SHARE the Add output's gradient buffer
            # (no copy kernel):
            #  - an input consumed only by the Add (the conv3 / projection branch) is a pure reader of it;
            #  - the identity shortcut x (also consumed by the next BN) turns the buffer into an in-place
            #    accumulator: x's other consumers add their dx into it.  That is safe when every reader of the Add
            #    output's gradient runs (in backward order) before every such writer, i.e. comes LATER in forward
            #    order — checked below.
            pos = {op: i for i, op in enumerate(self.ops)}
            add_alias = {}

            def root_of(t):
                while t in add_alias or t in self.alias:
                    t = add_alias[t] if t in add_alias else self.alias[t]
                return t
            for op in self.ops:
                if op.type != 'Add':
                    continue
                for x_t in op.inputs:
                    root = x_t
                    while root in self.alias:
                        root = self.alias[root]
                    if root.op.type == 'Placeholder' or root in add_alias or root is op.output:
                        continue
                    single = len(self._consumers(x_t)) == 1
                    chain_single = True
                    tt = x_t
                    while tt in self.alias:
                        tt = self.alias[tt]
                        chain_single = chain_single and len(self._consumers(tt)) == 1
                    if single and chain_single:
                        add_alias[root] = op.output
                        continue
                    if x_t in self.alias:
                        continue
                    # readers of g(Add out): ops whose output gradient lives in that buffer
                    key = root_of(op.output)
                    readers = [o for o in self.ops if o.type != 'Placeholder' and o is not op and root_of(o.output) is key]
                    writers = [c for c in self._consumers(x_t) if c is not op]
                    if all(pos[r] > pos[w] for r in readers for w in writers) and all(pos[w] < pos[op] for w in writers):
                        add_alias[root] = op.output
            for op in self.ops:
                t = op.output
                if op.type == 'Placeholder':
                    continue
                if t in self.alias:
                    self.galias[t] = self.alias[t]
                elif t in add_alias:
                    self.galias[t] = add_alias[t]
                else:
                    self.gbuf[t] = E(t.shape)
                if op.type in ('Conv2D', 'MatMul') and op in self.fused_act:
                    self.relu_scratch[op] = E(t.shape)
            # ---- dy operand planes.  For every tensor-core conv, the LAST op that writes the gradient of its output
            # before the conv's own backward runs; when that is a BatchNorm backward, it also emits the gradient as
            # split-bf16 planes (dgrad + wgrad operands) instead of a separate split pass.  If the BN is the only
            # writer and the conv the only reader, the fp32 copy is dropped and the planes live in its memory.
            grad_writers = {}
            for op in self.ops:
                if op.type in ('Placeholder', 'Reshape', 'Identity') or op in self.fused_into:
                    continue
                ins = op.inputs if op.type == 'Add' else op.inputs[:1]
                for x_t in ins:
                    if x_t.op.type == 'Placeholder':
                        continue
                    k = self.gkey(x_t)
                    if op.type == 'Add' and k is self.gkey(op.output):
                        continue
                    grad_writers.setdefault(k, []).append(op)
            self.bn_gplanes, self.bn_gplanes_only, self.conv_dy_planes = {}, {}, {}
            for op in self.ops:
                if op not in self.tc_wgrad or op in self.fused_act or 'bias' in op.vars or op.output.numel % 8:
                    if op in self.tc_wgrad:
                        max_dy = max(max_dy, op.output.numel)
                    continue
                k = self.gkey(op.output)
                later = [w for w in grad_writers.get(k, []) if pos[w] > pos[op]]
                lw = min(later, key=lambda w: pos[w]) if later else None
                if lw is None or lw.type != 'FusedBatchNorm' or lw.inputs[0].numel != op.output.numel:
                    max_dy = max(max_dy, op.output.numel)
                    continue
                if lw not in self.bn_gplanes:
                    readers = [o for o in self.ops if o.type != 'Placeholder' and self.gkey(o.output) is k]
                    only = len(grad_writers[k]) == 1 and readers == [op]
                    self.bn_gplanes_only[lw] = only
                    self.bn_gplanes[lw] = ops.Planes(op.output.numel, dev,
                                                     self.gbuf[k].view(-1).view(torch.bfloat16) if only else None)
                self.conv_dy_planes[op] = self.bn_gplanes[lw]
            # split-K partials of every tensor-core wgrad get their own buffer; ONE reduction launch at the end of the
            # backward pass sums them into the flat gradient buffer (fixed order: deterministic)
            self.wg_part, red_items = {}, []
            for op in self.ops:
                if op in self.tc_wgrad:
                    splits = ops.conv2d_tc_wgrad_splits(self.desc[op])
                    if splits > 1:
                        gk = st.view(op.vars['kernel'], self.G)
                        self.wg_part[op] = E((splits * gk.numel(),))
                        red_items.append((self.wg_part[op], gk, splits))
            self._red_items = red_items
            self.wg_reduce = ops.TcWgradReduceBatch(red_items, dev) if red_items else None
            max_dy = max(max_dy, getattr(self, '_stem_dy', 8))
            self.x_scratch = ops.Planes(max_x, dev)
            self.dy_scratch = ops.Planes(max_dy, dev)
            if self.maskable:
                self.MASK = torch.ones(st.n_masked, dtype=torch.float32, device=dev)
                self.BKUP = st.P[:st.n_masked].clone()
                mv = self.maskable
                # (the builder takes device pointers: planning-only executors on the CPU — tests — do without)
                self.mask_builder = ops.MaskBuilder([st.view(v) for v in mv],
                                                    [st.view(v, self.BKUP) for v in mv],
                                                    [st.view(v, self.MASK) for v in mv]) if dev.type == 'cuda' else None
            else:
                self.MASK = None
            if self.exact_ste and self.wq is not None and isinstance(self.wq, ops.UniformWeightQuantizer):
                self._ste_grads = [st.view(v, self.G) for v in [op.vars['kernel'] for op in self.wq_ops]]
            else:
                self._ste_grads = None
            self.beta1_power = F32(self.optimizer.get('beta1', 0.9))
            self.beta2_power = F32(self.optimizer.get('beta2', 0.999))

    # ------------------------------------------------------------------ profiling (bench.py roofline)
    class _Timed:
        def __init__(self, ex, cat):
            self.ex, self.cat = ex, cat

        def __enter__(self):
            if self.ex.prof is not None:
                self.a = torch.cuda.Event(enable_timing=True)
                self.a.record()

        def __exit__(self, *exc):
            if self.ex.prof is not None:
                b = torch.cuda.Event(enable_timing=True)
                b.record()
                self.ex.prof.setdefault(self.cat, []).append((self.a, b))

    def timed(self, cat):
        return Executor._Timed(self, cat)

    def profile_step(self, lr, allreduce=None):
        """One EAGER step with every launch group bracketed by CUDA events on the launching stream.
        Returns {category: milliseconds}.  (Not the timed region: the benchmark replays a CUDA graph.)"""
        self.prof = {}
        if self.teacher is not None:
            self.teacher.prof = self.prof
        self.set_hyper(lr)
        self.device_step(allreduce)
        torch.cuda.synchronize()
        out = {k: sum(a.elapsed_time(b) for a, b in v) for k, v in self.prof.items()}
        self.prof = None
        if self.teacher is not None:
            self.teacher.prof = None
        self.advance_optimizer_state()
        return out

    # ------------------------------------------------------------------ helpers
    def T(self, t):
        """Buffer that holds tensor t as seen by its consumers."""
        shape = t.shape
        while t in self.alias:
            op = t.op
            if op in self.aq_out:
                return self.aq_out[op].view(shape)
            t = self.alias[t]
        b = self.buf[t]
        return b if b.shape == shape else b.view(shape)

    def _root(self, t):
        """The tensor whose buffer holds t (following Reshape / fused-activation aliases); None when t is
        held by an out-of-place quantized buffer."""
        while t in self.alias:
            if t.op in self.aq_out:
                return None
            t = self.alias[t]
        return t

    def planes_of(self, t):
        r = self._root(t)
        return self.xplanes.get(r.op) if r is not None else None

    def _act_lv_of(self, t):
        """level-operand record of the BN that produced tensor t's planes (None: plain split-bf16 planes)"""
        r = self._root(t)
        return self.act_lv.get(r.op) if r is not None else None

    def _tc_act(self, t):
        lv, xp = self._act_lv_of(t), self.planes_of(t)
        return ops.tc_act(xp, lv['hdr'], lv['csum'], lv['nseg']) if lv is not None else ops.tc_act(xp)

    def _tc_wt(self, op):
        tw = self.tc[op]
        lv = self.w_lv.get(op) if self._lv_on else None
        if lv is not None and self.wq.bits[lv['index']] <= 8:
            return ops.tc_wt(tw.f_hi, None, lv['alpha'], lv['beta'], lv['ncols'] > 1, self.wq.bits[lv['index']])
        return ops.tc_wt(tw.f_hi, tw.f_lo)

    def raw(self, t):
        while t in self.alias:
            t = self.alias[t]
        return self.buf[t]

    def gkey(self, t):
        while t in self.galias:
            t = self.galias[t]
        return t

    def grad_target(self, t):
        """(buffer, accumulate) for writing a contribution to dL/dt."""
        k = self.gkey(t)
        acc = k in self._gwritten
        self._gwritten.add(k)
        return self.gbuf[k], acc

    def grad_of(self, t):
        k = self.gkey(t)
        return self.gbuf[k] if k in self._gwritten else None

    def kernel_of(self, op):
        v = op.vars['kernel']
        if op in self.qvars:
            return self.store.view(v, self.QW)
        return self.store.view(v)

    # ------------------------------------------------------------------ forward
    def forward(self, training=None, upto=None):
        """upto: stop after this op has run (its output buffer is the result wanted)."""
        st = self.store
        training = self.train if training is None else training
        if self.aq_ops:
            ops.minmax_reset(self.aq_slots)
        if self.wq is not None:
            with self.timed('weight_quant'):
                self.wq.forward()
        if self.static_weights and not self._static_ready:
            self.prepare_static_weights()
        self._lv_on = bool(training and (self.act_lv or self.w_lv))
        if self.tc_batch is not None:
            with self.timed('conv_prep'):
                self.tc_batch.prepare(levels=self._lv_on)
        prev = None
        for op in self.ops:
            if prev is not None and prev is upto:
                return None
            prev = op
            ty = op.type
            if ty in ('Placeholder', 'Reshape', 'Identity'):
                continue
            if ty in ('Conv2D', 'MatMul'):
                bias = st.view(op.vars['bias']) if 'bias' in op.vars else None
                if op in self.im2col:
                    im = self.im2col[op]
                    wk = self.kernel_of(op)
                    with self.timed('conv_prep'):
                        if im['compute']:
                            if im['mode'] == 's2d':
                                pt_, pl_ = op.attrs['pad']
                                ops.s2d_planes(self.T(op.inputs[0]), pt_, pl_, im['d1'].h, im['d1'].w, im['d1'].c, im['cols'])
                            elif im['planes']:
                                ops.im2col_planes(self.desc[op], self.T(op.inputs[0]), im['kpad'], im['cols'])
                            else:
                                ops.im2col(self.desc[op], self.T(op.inputs[0]), im['kpad'], im['cols'])
                            if self.cols_event is not None:
                                self.cols_event.record()
                        elif self.cols_wait is not None:
                            torch.cuda.current_stream().wait_event(self.cols_wait)
                        if not self.static_weights:
                            self._stem_weights(im, wk)
                    with self.timed('conv_fwd'):
                        if im['planes']:
                            ops.conv2d_tc_fwd_planes(im['d1'], im['cols'], im['tw'], bias, op in self.fused_act,
                                                     self.buf[op.output])
                        else:
                            ops.conv2d_tc_fwd(im['d1'], im['cols'], im['tw'], bias, op in self.fused_act,
                                              self.buf[op.output])
                elif op in self.tc:
                    if not self.static_weights and self.tc_batch is None:
                        with self.timed('conv_prep'):
                            self.tc[op].prepare(self.kernel_of(op))
                    res = self.T(self.fused_add[op][1]) if op in self.fused_add else None
                    xp = self.planes_of(op.inputs[0])
                    with self.timed('conv_fwd'):
                        if xp is not None and self._lv_on and self._act_lv_of(op.inputs[0]) is not None:
                            ops.conv2d_tc_fwd_ex(self.desc[op], self._tc_act(op.inputs[0]), self._tc_wt(op), bias,
                                                 op in self.fused_act, self.buf[op.output], res)
                        elif xp is not None:
                            ops.conv2d_tc_fwd_planes(self.desc[op], xp, self.tc[op], bias, op in self.fused_act,
                                                     self.buf[op.output], res)
                        else:
                            ops.conv2d_tc_fwd(self.desc[op], self.T(op.inputs[0]), self.tc[op], bias,
                                              op in self.fused_act, self.buf[op.output], res)
                else:
                    with self.timed('conv_fwd'):
                        ops.conv2d_fwd(self.desc[op], self.T(op.inputs[0]), self.kernel_of(op), bias,
                                       op in self.fused_act, self.buf[op.output])
            elif ty == 'DepthwiseConv2dNative':
                with self.timed('dwconv'):
                    ops.dwconv_fwd(self.desc[op], self.T(op.inputs[0]), self.kernel_of(op), self.buf[op.output])
            elif ty == 'FusedBatchNorm':
                x, y = self.T(op.inputs[0]), self.buf[op.output]
                c = y.shape[-1]
                m = y.numel() // c
                b = self.bn[op]
                gamma, beta = st.view(op.vars['gamma']), st.view(op.vars['beta'])
                mm, mv = st.view(op.vars['moving_mean']), st.view(op.vars['moving_variance'])
                act = self.fused_act.get(op, 0)
                relu_op = self._consumers(op.output)[0] if act else None
                slot = self.aq_slots[self.aq_index[relu_op]] if relu_op in self.aq_index else None
                pl = self.xplanes.get(op)
                need_f32 = pl is None or self.bn_need_f32[op]
                # with an activation quantizer the BN pass writes fp32 (+ range) and the quantizer writes the planes
                pl_bn = pl if slot is None else None
                y_bn = y if (need_f32 or slot is not None) else None
                bn_mom = op.attrs['momentum'] if self.update_moving_stats else 1.0
                if op.attrs['training'] and training and slot is not None:
                    # the statistics pass also yields the range of act(bn(x)); one fused BN + fake-quant pass
                    with self.timed('bn_stats'):
                        ops.bn_train_stats_range(x, m, c, op.attrs['epsilon'], bn_mom, b['mean'], b['var'],
                                                 b['rstd'], mm, mv, gamma, beta, act, slot, self.bn_ws)
                    with self.timed('bn_apply'):
                        bits = self.act_quant['bits'][self.aq_index[relu_op]]
                        if self._lv_on and op in self.act_lv:
                            lv = self.act_lv[op]
                            ops.bn_apply_quant_levels(x, m, c, b['mean'], b['rstd'], gamma, beta, act, slot, bits,
                                                      y if need_f32 else None, pl, lv['hdr'], lv['csum'])
                        else:
                            ops.bn_apply_quant(x, m, c, b['mean'], b['rstd'], gamma, beta, act, slot, bits,
                                               y if need_f32 else None, pl)
                    slot = None                                    # quantized already
                elif op.attrs['training'] and training:
                    with self.timed('bn_stats'):
                        ops.bn_train_stats(x, m, c, op.attrs['epsilon'], bn_mom, b['mean'], b['var'],
                                           b['rstd'], mm, mv, self.bn_ws)
                    with self.timed('bn_apply'):
                        ops.bn_apply(x, m, c, b['mean'], b['rstd'], gamma, beta, act, y_bn, slot, pl_bn)
                else:
                    with self.timed('bn_apply'):
                        ops.bn_apply_eval(x, m, c, mm, mv, op.attrs['epsilon'], gamma, beta, act, y_bn, slot, pl_bn)
                if slot is not None:
                    with self.timed('act_quant'):
                        ops.act_quant(y, y if need_f32 else None, slot, self.act_quant['bits'][self.aq_index[relu_op]], pl)
            elif ty in ACT_TYPES:
                src = self.fused_into[op]
                if op in self.aq_index and src.type != 'FusedBatchNorm':
                    y = self.buf[src.output]
                    slot = self.aq_slots[self.aq_index[op]]
                    with self.timed('act_quant'):
                        ops.act_minmax(y, slot)
                        ops.act_quant(y, self.aq_out[op], slot, self.act_quant['bits'][self.aq_index[op]])
            elif ty == 'MaxPool':
                with self.timed('pool'):
                    ops.maxpool_fwd(self.desc[op], self.T(op.inputs[0]), self.buf[op.output], self.pool_argmax.get(op))
            elif ty == 'Mean':
                x = op.inputs[0]
                n, h, w, c = x.shape
                with self.timed('pool'):
                    ops.global_avgpool_fwd(self.T(x), n, h * w, c, self.buf[op.output])
            elif ty == 'Add':
                if op in self.add_fused:
                    continue                               # computed by the producing conv's epilogue
                with self.timed('add_fwd'):
                    ops.add(self.T(op.inputs[0]), self.T(op.inputs[1]), self.buf[op.output])
            elif ty == 'Softmax':
                ops.softmax_fwd(self.T(op.inputs[0]), self.buf[op.output])
            else:
                raise NotImplementedError('op type %s' % ty)
        return self.T(self.logits_t)

    # ------------------------------------------------------------------ gradient buckets of the data-parallel step
    def _bucket_plan(self):
        """The flat gradient buffer is summed over the workers in TWO all-reduces instead of one (SURVEY §8e): the
        kernels of the LAST layers — about half of the first (weight-decayed) range of the parameter store, which is laid
        out in forward order — are complete long before the backward pass ends (stage 4 + the dense layer of ResNet-50
        hold 2/3 of its parameters and take ~10 % of its backward time), so their all-reduce runs on a communication
        stream underneath the rest of the backward pass.  Returns None when the split does not apply."""
        if hasattr(self, '_bk'):
            return self._bk
        self._bk = None
        st = self.store
        if os.environ.get('PF_AR_BUCKETS', '2') == '1' or not self.overlap or getattr(self, 'train_clusters', False) \
                or not st.ranges:
            return None
        s0, e0 = st.ranges[0][0], st.ranges[0][1]
        pos = {op: i for i, op in enumerate(self.ops)}
        owners = sorted((st.offset[v], v.numel, pos[op]) for op in self.ops for v in op.vars.values()
                        if v.trainable and s0 <= st.offset[v] < e0)
        if len(owners) < 4 or any(b[2] < a[2] for a, b in zip(owners, owners[1:])):
            return None                                    # store order is not the forward order: no valid split
        acc, cut = 0, None
        for i in range(len(owners) - 1, 0, -1):
            acc += owners[i][1]
            if acc >= 0.5 * (e0 - s0) and owners[i][2] > owners[i - 1][2]:
                cut = i
                break
        if cut is None:
            return None
        split, bpos = owners[cut][0], owners[cut][2]
        off = lambda t: (t.data_ptr() - self.G.data_ptr()) // 4
        hi = [it for it in self._red_items if off(it[1]) >= split]
        lo = [it for it in self._red_items if off(it[1]) < split]
        ste_hi = ste_lo = None
        if self._ste_grads is not None:
            ste_hi = [i for i, g in enumerate(self._ste_grads) if off(g) >= split]
            ste_lo = [i for i, g in enumerate(self._ste_grads) if off(g) < split]
        self._bk = dict(split=split, end=e0, pos=bpos, stream=torch.cuda.Stream(device=self.device),
                        red_hi=ops.TcWgradReduceBatch(hi, self.device) if hi else None,
                        red_lo=ops.TcWgradReduceBatch(lo, self.device) if lo else None, ste_hi=ste_hi, ste_lo=ste_lo)
        return self._bk

    def _bucket_hi(self, bk, allreduce):
        """the last layers' gradients are final: reduce their split-K partials, apply their STE, start their all-reduce —
        all on the communication stream, behind what the main and the weight-gradient streams have enqueued so far"""
        cs, main = bk['stream'], torch.cuda.current_stream()
        cs.wait_stream(main)
        if self._side_active:
            cs.wait_stream(self.side2)
        with torch.cuda.stream(cs):
            if bk['red_hi'] is not None:
                bk['red_hi'].reduce()
            if bk['ste_hi']:
                self.wq.ste_backward_(self._ste_grads, bk['ste_hi'])
            allreduce(self.G[bk['split']:bk['end']])

    # ------------------------------------------------------------------ loss + backward
    def loss_and_backward(self, allreduce=None):
        """allreduce (data-parallel step): callable summing a contiguous range of the flat gradient buffer over the
        workers on the current stream; called for every range of the buffer before this method returns."""
        st = self.store
        L = self.loss
        self._gwritten = set()
        self._side_active = self.overlap and self.prof is None
        bk = self._bucket_plan() if (allreduce is not None and self._side_active) else None
        bk_fired = False
        op_pos = {op: i for i, op in enumerate(self.ops)} if bk is not None else None
        labels = self.T(self.labels_t)
        ce_logits = L.ce[1]
        teacher_logits, w_dst, T_dst = None, 0.0, 1.0
        if L.dst is not None:
            teacher_logits = self.teacher.T(self.teacher.logits_t)
            w_dst, T_dst = L.dst[2], L.dst[3]
        gl, _ = self.grad_target(ce_logits)
        ops.softmax_ce(self.T(ce_logits), labels, teacher_logits, T_dst, w_dst, gl.view(ce_logits.shape),
                       self.loss_out[:4], self.row_ws)
        for op in reversed(self.ops):
            if bk is not None and not bk_fired and op_pos[op] < bk['pos']:
                bk_fired = True
                self._bucket_hi(bk, allreduce)
            ty = op.type
            if ty == 'Placeholder':
                continue
            gy = self.grad_of(op.output)
            if gy is None:
                continue
            if ty in ('Reshape', 'Identity') or op in self.fused_into:
                continue                                   # gradient buffer is shared with the input
            if ty in ('Conv2D', 'MatMul'):
                d = self.desc[op]
                x_t = op.inputs[0]
                y = self.buf[op.output]
                m, k = y.numel() // y.shape[-1], y.shape[-1]
                if op in self.fused_act:
                    dz = self.relu_scratch[op]
                    ops.relu_bwd(gy, y, dz, self.fused_act[op])
                    gy = dz
                if 'bias' in op.vars:
                    ops.colsum(gy, m, k, st.view(op.vars['bias'], self.G))
                with self.timed('conv_wgrad'):
                    if op in self.im2col:
                        im = self.im2col[op]
                        gk = st.view(op.vars['kernel'], self.G)
                        if im['planes']:
                            gp = ops.Planes(op.output.numel, self.device, self.dy_scratch.buf)
                            ops.split_bf16(gy, gp)
                            self._stem_wgrad_planes(im, gp)
                        elif ops.conv2d_tc_wgrad_supported(im['d1']):
                            ops.conv2d_tc_wgrad(im['d1'], im['cols'], gy, self.wgrad_ws, im['dwpad'])
                        else:
                            ops.conv2d_wgrad(im['d1'], im['cols'], gy, self.wgrad_ws, im['dwpad'])
                        if im['mode'] == 's2d':
                            ops.gather_rows(im['dwpad'], im['bwd_map'], gk, gk.shape[-1])
                        else:
                            ops.add(im['dwpad'][:gk.numel()], None, gk.reshape(-1))
                    elif op in self.tc_wgrad and self._side_active and self.planes_of(x_t) is not None \
                            and self.conv_dy_planes.get(op) is not None:
                        # both operands exist as planes: the weight gradient runs on the side stream, beside the
                        # dgrad / BN-backward chain that continues on the main stream
                        gp = self.conv_dy_planes[op]
                        self.side2.wait_stream(torch.cuda.current_stream())
                        with torch.cuda.stream(self.side2):
                            part = self.wg_part.get(op)
                            dw = None if part is not None else st.view(op.vars['kernel'], self.G)
                            if self._lv_on and self._act_lv_of(x_t) is not None:
                                ops.conv2d_tc_wgrad_ex(d, self._tc_act(x_t), ops.tc_act(gp),
                                                       part if part is not None else self.wgrad_ws2, dw)
                            else:
                                ops.conv2d_tc_wgrad_planes(d, self.planes_of(x_t), gp,
                                                           part if part is not None else self.wgrad_ws2, dw)
                    elif op in self.tc_wgrad:
                        # operands in split-bf16 planes: native (written by BN-apply / BN-backward) or split here
                        xp = self.planes_of(x_t)
                        if xp is None:
                            xp = ops.Planes(x_t.numel, self.device, self.x_scratch.buf)
                            ops.split_bf16(self.T(x_t), xp)
                        gp = self.conv_dy_planes.get(op)
                        if gp is None:
                            gp = ops.Planes(op.output.numel, self.device, self.dy_scratch.buf)
                            ops.split_bf16(gy, gp)
                        part = self.wg_part.get(op)
                        dw = None if part is not None else st.view(op.vars['kernel'], self.G)
                        if self._lv_on and self._act_lv_of(x_t) is not None:
                            ops.conv2d_tc_wgrad_ex(d, self._tc_act(x_t), ops.tc_act(gp),
                                                   part if part is not None else self.wgrad_ws, dw)
                        else:
                            ops.conv2d_tc_wgrad_planes(d, xp, gp, part if part is not None else self.wgrad_ws, dw)
                    else:
                        gp = None
                        ops.conv2d_wgrad(d, self.T(x_t), gy, self.wgrad_ws, st.view(op.vars['kernel'], self.G))
                if x_t.op.type != 'Placeholder':
                    gx, acc = self.grad_target(x_t)
                    with self.timed('conv_dgrad'):
                        if op in self.tc_wgrad and op not in self.im2col:
                            ops.conv2d_tc_dgrad_planes(d, gp, self.tc[op], acc, gx)
                        elif op in self.tc:
                            ops.conv2d_tc_dgrad(d, gy, self.tc[op], acc, gx)
                        else:
                            ops.conv2d_dgrad(d, gy, self.kernel_of(op), self.wt_ws, acc, gx)
            elif ty == 'DepthwiseConv2dNative':
                d = self.desc[op]
                x_t = op.inputs[0]
                with self.timed('dwconv'):
                    ops.dwconv_wgrad(d, self.T(x_t), gy, self.wgrad_ws, st.view(op.vars['kernel'], self.G))
                    if x_t.op.type != 'Placeholder':
                        gx, acc = self.grad_target(x_t)
                        ops.dwconv_dgrad(d, gy, self.kernel_of(op), acc, gx)
            elif ty == 'FusedBatchNorm':
                x_t = op.inputs[0]
                y = self.buf[op.output]
                c = y.shape[-1]
                m = y.numel() // c
                b = self.bn[op]
                gx, acc = self.grad_target(x_t)
                gp = self.bn_gplanes.get(op)
                only = gp is not None and self.bn_gplanes_only[op]
                assert not (only and acc)
                with self.timed('bn_bwd'):
                    ops.bn_bwd(gy, self.T(x_t), m, c, b['mean'], b['rstd'], st.view(op.vars['gamma']),
                               st.view(op.vars['beta']), self.fused_act.get(op, 0),
                               st.view(op.vars['gamma'], self.G), st.view(op.vars['beta'], self.G),
                               None if only else gx, acc, self.bn_ws, gp)
            elif ty == 'MaxPool':
                x_t = op.inputs[0]
                gx, acc = self.grad_target(x_t)
                with self.timed('pool'):
                    ops.maxpool_bwd(self.desc[op], gy, self.pool_argmax[op], gx, acc)
            elif ty == 'Mean':
                x_t = op.inputs[0]
                n, h, w, c = x_t.shape
                gx, acc = self.grad_target(x_t)
                with self.timed('pool'):
                    ops.global_avgpool_bwd(gy, n, h * w, c, gx, acc)
            elif ty == 'Add':
                for x_t in op.inputs:
                    if self.gkey(x_t) is self.gkey(op.output):
                        continue                           # gradient buffer shared with the output (plan-time alias)
                    gx, acc = self.grad_target(x_t)
                    with self.timed('add_bwd'):
                        ops.add(gy, None, gx, acc)
            elif ty == 'Softmax':
                x_t = op.inputs[0]
                gx, acc = self.grad_target(x_t)
                assert not acc
                ops.softmax_bwd(gy, self.buf[op.output], gx)
            else:
                raise NotImplementedError('backward of %s' % ty)
        if self._side_active:
            torch.cuda.current_stream().wait_stream(self.side2)
        if bk is not None and bk_fired:
            # the rest of the buffer: [0, split) of the first range and everything behind it (BN scales / offsets, ...)
            if bk['red_lo'] is not None:
                bk['red_lo'].reduce()
            if bk['ste_lo']:
                self.wq.ste_backward_(self._ste_grads, bk['ste_lo'])
            allreduce(self.G[:bk['split']])
            if bk['end'] < self.G.numel():
                allreduce(self.G[bk['end']:])
            torch.cuda.current_stream().wait_stream(bk['stream'])
            return
        if self.wg_reduce is not None:
            with self.timed('conv_wgrad'):
                self.wg_reduce.reduce()
        if self._ste_grads is not None:
            self.wq.ste_backward_(self._ste_grads)
        if getattr(self, 'train_clusters', False):
            # codebook gradients from the gradients w.r.t. the quantized kernels (which stay, unchanged, as the kernels'
            # own gradients: the straight-through estimator of utils.py:303-306)
            with self.timed('weight_quant'):
                self.wq.cluster_grad([st.view(op.vars['kernel'], self.G) for op in self.wq_ops], self.G)

    def _stem_wgrad_planes(self, im, gp):
        """weight gradient of the first layer from its column planes and the dy planes, into im['dwpad']"""
        if 'pair' in im:
            pr = im['pair']
            ops.conv2d_tc_wgrad_planes(pr['d'], im['cols'], gp, self.wgrad_ws, pr['dw'])
            ops.fold_diag_blocks(pr['dw'], pr['g'], im['kpad'], im['d1'].k, im['dwpad'])
        else:
            ops.conv2d_tc_wgrad_planes(im['d1'], im['cols'], gp, self.wgrad_ws, im['dwpad'])

    @contextlib.contextmanager
    def standalone_forward(self):
        """forward() calls outside device_step (layer-wise regression passes): an executor that shares the first layer's
        im2col columns with the distillation teacher normally lets the teacher's forward fill them — here it fills
        them itself."""
        saved = {op: im['compute'] for op, im in self.im2col.items()}
        for im in self.im2col.values():
            im['compute'] = True
        try:
            yield self
        finally:
            for op, c in saved.items():
                self.im2col[op]['compute'] = c

    def layer_wgrad(self, op, gy, dw):
        """dW of ONE Conv2D / MatMul for an externally supplied gradient `gy` of its output, after a training-mode
        forward() of this executor: the weight gradient of the layer-wise regression loss of the channel-pruning
        learner (learners/channel_pruning_gpu/learner.py:370, :391 — compute_gradients(reg_loss_i, [kernel_i])).
        Same kernels as the step's own backward; `dw` is an fp32 tensor of the kernel's shape."""
        d, x_t = self.desc[op], op.inputs[0]
        # own dy planes: the step's dy_scratch is only sized for the layers whose gradient is split in a separate pass
        lw = getattr(self, '_lw_planes', None)
        if lw is None or lw.numel < op.output.numel:
            lw = self._lw_planes = ops.Planes(op.output.numel, self.device)
        with self.timed('conv_wgrad'):
            if op in self.im2col:
                im = self.im2col[op]
                if im['planes']:
                    gp = ops.Planes(op.output.numel, self.device, lw.buf)
                    ops.split_bf16(gy, gp)
                    self._stem_wgrad_planes(im, gp)
                elif ops.conv2d_tc_wgrad_supported(im['d1']):
                    ops.conv2d_tc_wgrad(im['d1'], im['cols'], gy, self.wgrad_ws, im['dwpad'])
                else:
                    ops.conv2d_wgrad(im['d1'], im['cols'], gy, self.wgrad_ws, im['dwpad'])
                if im['mode'] == 's2d':
                    ops.gather_rows(im['dwpad'], im['bwd_map'], dw, dw.shape[-1])
                else:
                    ops.add(im['dwpad'][:dw.numel()], None, dw.reshape(-1))
            elif op in self.tc_wgrad:
                xp = self.planes_of(x_t)
                if xp is None:
                    xp = ops.Planes(x_t.numel, self.device, self.x_scratch.buf)
                    ops.split_bf16(self.T(x_t), xp)
                gp = ops.Planes(op.output.numel, self.device, lw.buf)
                ops.split_bf16(gy, gp)
                if self._lv_on and self._act_lv_of(x_t) is not None:
                    ops.conv2d_tc_wgrad_ex(d, self._tc_act(x_t), ops.tc_act(gp), self.wgrad_ws, dw)
                else:
                    ops.conv2d_tc_wgrad_planes(d, xp, gp, self.wgrad_ws, dw)
            else:
                ops.conv2d_wgrad(d, self.T(x_t), gy, self.wgrad_ws, dw)

    def forward_eval_loss(self):
        """Evaluation pass: BN in inference mode, quantizers active, losses/metrics only."""
        if self.teacher is not None:
            self.teacher.forward()
        self.forward(training=False)
        L = self.loss
        teacher_logits, w_dst, T_dst = None, 0.0, 1.0
        if L.dst is not None:
            teacher_logits = self.teacher.T(self.teacher.logits_t)
            w_dst, T_dst = L.dst[2], L.dst[3]
        scratch = self.gbuf[self.gkey(L.ce[1])]
        ops.softmax_ce(self.T(L.ce[1]), self.T(self.labels_t), teacher_logits, T_dst, w_dst,
                       scratch.view(L.ce[1].shape), self.loss_out[:4], self.row_ws)
        self.l2_value()

    def l2_value(self):
        first = True
        for (s, e, masked, wd) in self.store.ranges:
            if wd != 0.0:
                ops.l2_loss(self.store.P[s:e], wd, self.l2_out, self.l2_ws, accumulate=not first)
                first = False
        if first:
            self.l2_out.zero_()

    def apply_gradients(self):
        st, o = self.store, self.optimizer
        for (s, e, masked, wd) in st.ranges:
            if e <= s or (s, e) in st.frozen_ranges:
                continue
            if o['kind'] == 'momentum':
                mask = self.MASK[s:e] if (masked and self.MASK is not None) else None
                ops.momentum_step(st.P[s:e], self.S1[s:e], self.G[s:e], mask, self.hp, o.get('momentum', 0.9), wd,
                                  self.grad_scale)
            else:
                ops.adam_step(st.P[s:e], self.S1[s:e], self.S2[s:e], self.G[s:e], self.hp, o.get('beta1', 0.9),
                              o.get('beta2', 0.999), o.get('eps', 1e-8), wd, self.grad_scale)

    def share_im2col_from(self, other):
        """The teacher and the student read the same image batch: reuse the teacher's im2col of the first
        layer (it runs first inside device_step) instead of recomputing it."""
        for op, im in self.im2col.items():
            for op2, im2 in other.im2col.items():
                if op.inputs[0] is op2.inputs[0] and im['kpad'] == im2['kpad'] and im['planes'] == im2['planes'] \
                        and im['mode'] == im2['mode'] \
                        and all(op.attrs[a] == op2.attrs[a] for a in ('ksize', 'strides', 'pad')):
                    im['cols'] = im2['cols']
                    im['compute'] = False
                    self._shares_cols = True

    # ------------------------------------------------------------------ one training step
    def device_step(self, allreduce=None):
        """Everything that runs on the GPU for one step (CUDA-graph capturable)."""
        par = self.overlap and self.prof is None and self.teacher is not None
        if par:
            main = torch.cuda.current_stream()
            self.side.wait_stream(main)
            if self._shares_cols:
                self.teacher.cols_event = self.cols_wait = torch.cuda.Event()
            with torch.cuda.stream(self.side):
                self.teacher.forward()
            self.forward()
            main.wait_stream(self.side)
            self.teacher.cols_event = self.cols_wait = None
        else:
            if self.teacher is not None:
                self.teacher.forward()
            self.forward()
        self.loss_and_backward(allreduce)
        if allreduce is not None and not (self._side_active and self._bucket_plan() is not None):
            with self.timed('allreduce'):
                allreduce(self.G)
        with self.timed('optimizer'):
            self.l2_value()
            self.apply_gradients()

    def set_hyper(self, lr):
        i = self._hp_i % self.hp_ring.shape[0]
        self._hp_i += 1
        if self.hp_events[i] is not None:
            self.hp_events[i].synchronize()            # slot's previous upload has executed (16 steps ago: no wait)
        slot = self.hp_ring[i]
        slot[0] = float(lr)
        slot[1] = float(self.beta1_power)
        slot[2] = float(self.beta2_power)
        self.hp.copy_(slot, non_blocking=True)
        if self.hp.device.type == 'cuda':
            ev = torch.cuda.Event()
            ev.record()
            self.hp_events[i] = ev

    def advance_optimizer_state(self):
        if self.optimizer.get('kind') == 'adam':
            self.beta1_power = F32(self.beta1_power * F32(self.optimizer.get('beta1', 0.9)))
            self.beta2_power = F32(self.beta2_power * F32(self.optimizer.get('beta2', 0.999)))
        self.step_count += 1

    def reset_optimizer_slots(self):
        """tf.variables_initializer(optimizer.variables()) — run after every mask update
        (weight_sparsification/learner.py:128,217)."""
        self.S1.zero_()
        if self.S2 is not None:
            self.S2.zero_()

    def reset_optimizer_state(self):
        """A fresh optimizer: zero slots, Adam's beta powers and the step counter back to their initial values."""
        self.reset_optimizer_slots()
        self.beta1_power = F32(self.optimizer.get('beta1', 0.9))
        self.beta2_power = F32(self.optimizer.get('beta2', 0.999))
        self.step_count = 0

    def set_quant_bits(self, w_bits=None, a_bits=None):
        """New bit-widths for the quantized layers / activations.  The reference feeds them through placeholders on
        every sess.run (uniform_quantization/learner.py:330-337); here they are launch arguments (the weight
        quantizer's segment table, the activation kernels' `bits`), so a captured step graph is dropped and the next
        steps run eagerly until `capture` is called again."""
        if w_bits is not None:
            if self.wq is None:
                raise ValueError('this executor has no weight quantizer')
            self.wq.set_bits(list(w_bits))
            self.weight_quant['bits'] = list(w_bits)
            if self.tc_batch is not None and self.w_lv:
                self.tc_batch.set_bits({lv['batch_index']: self.wq.bits[lv['index']] for lv in self.w_lv.values()})
        if a_bits is not None:
            if len(a_bits) != len(self.aq_ops):
                raise ValueError('one bit-width per quantized activation expected (%d)' % len(self.aq_ops))
            if any(int(b) < 1 or int(b) > 32 for b in a_bits):
                raise ValueError('bit-widths must be in [1, 32]')
            if self.act_quant:
                self.act_quant['bits'] = [int(b) for b in a_bits]
        self._graph = None

    def capture(self, allreduce=None):
        """Capture device_step into a CUDA graph (after one eager warm-up on a side stream)."""
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.device_step(allreduce)
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self.device_step(allreduce)
        return self._graph

    def run_step(self, lr, allreduce=None):
        self.set_hyper(lr)
        if self._graph is not None:
            self._graph.replay()
        else:
            self.device_step(allreduce)
        self.advance_optimizer_state()

    def fetch_losses(self):
        """(hard CE, distillation, l2, total, top1, top5) of the last step — one small D2H read."""
        dev_vals = torch.cat([self.loss_out[:4], self.l2_out[:1]])
        self.last_d2h_bytes = dev_vals.numel() * dev_vals.element_size()      # what this call reads back
        o = dev_vals.cpu().numpy()
        hard, dst, top1, top5, l2 = [F32(x) for x in o]
        total = F32(F32(hard + l2) + dst)
        return dict(model_loss=F32(hard + l2), dst_loss=dst, l2=l2, ce=hard, loss=total, acc_top1=top1,
                    acc_top5=top5)
