"""Golden values of the bucketed codebook quantizer produced by the REFERENCE'S OWN code: NonUniformQuantization.
__bucket_quantize with __split_bucket, __channel_bucket, __scale, __quantile_init, __build_bucket_norm_quant_point,
__inv_scale and __updt_bucket_storage (learners/nonuniform_quantization/utils.py:196-243, 309-366, 388-494), executed
from a checkout of the reference on numpy-backed stub tensors (TensorFlow 1.x is not a dependency), like the unbucketed
case of make_golden_from_reference.py.

  python tests/golden/make_golden_nuq_bucket.py <reference checkout>   ->  tests/golden/ref_executed_nuq_bucket_v1.json

Every tensor op maps one-to-one onto the numpy float32 op (each individually rounded, no FMA); tf.map_fn over the
buckets and tf.transpose are real.  tf.contrib.distributions.percentile is the oracle's 'nearest' rule
(oracle/pf_oracle.py:percentile_nearest), the one assumption shared with the unbucketed golden values."""
import builtins
import hashlib
import importlib.util
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, 'ref_executed_nuq_bucket_v1.json')
sys.path.insert(0, ROOT)
from oracle import pf_oracle as ORC  # noqa: E402


class Dim(object):
    def __init__(self, v):
        self.value = int(v)


class T(object):
    """numpy-backed tensor"""

    def __init__(self, a):
        self.a = np.asarray(a, dtype=np.float32)

    shape = property(lambda self: tuple(self.a.shape))

    def get_shape(self):
        return [Dim(d) for d in self.a.shape]

    def __getitem__(self, i):
        return T(self.a[i])

    @staticmethod
    def _v(o):
        return o.a if isinstance(o, T) else np.float32(o)

    def __add__(self, o):
        return T(self.a + T._v(o))

    def __radd__(self, o):
        return T(T._v(o) + self.a)

    def __sub__(self, o):
        return T(self.a - T._v(o))

    def __rsub__(self, o):
        return T(T._v(o) - self.a)

    def __mul__(self, o):
        return T(self.a * T._v(o))

    def __rmul__(self, o):
        return T(T._v(o) * self.a)

    def __truediv__(self, o):
        return T(self.a / T._v(o))


class Ctx(object):
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


def make_tf(created):
    tf = types.ModuleType('tensorflow')
    tf.float32, tf.int32, tf.int64 = np.float32, 'int32', 'int64'
    tf.variable_scope = lambda *a, **k: Ctx()
    tf.get_variable_scope = lambda: types.SimpleNamespace(name='scope')
    tf.constant = lambda value=0, dtype=None: T(value) if dtype is np.float32 else 0
    tf.cast = lambda x, dt=None: int(x) if dt == 'int64' else (x if isinstance(x, T) else T(np.float32(x)))
    tf.reshape = lambda t, shape: T(t.a.reshape([d.value if isinstance(d, Dim) else int(d) for d in shape]))
    tf.ones = lambda n, dtype=None: [1] * int(n) if dtype == 'int64' else T(np.ones(int(n), np.float32))
    tf.concat = lambda ts, axis=0: ([int(v) for part in ts for v in part] if isinstance(ts[0], list)
                                    else T(np.concatenate([t.a for t in ts], axis=axis)))
    tf.reduce_max = lambda w, axis=None: T(np.max(w.a, axis=axis))
    tf.reduce_min = lambda w, axis=None: T(np.min(w.a, axis=axis))
    tf.stop_gradient = lambda x: x
    tf.range = lambda n: list(range(int(n)))
    tf.map_fn = lambda fn, elems, dtype=None: T(np.stack([np.asarray(T._v(fn(e)), np.float32) for e in elems]))
    tf.expand_dims = lambda x, axis: T(np.expand_dims(x.a, axis))
    tf.tile = lambda x, reps: T(np.tile(x.a, reps))
    tf.transpose = lambda x, perm=None: T(np.transpose(x.a, perm))
    tf.argmin = lambda x, axis=-1: np.argmin(x.a, axis=axis)
    tf.gather = lambda c, idx: T(c.a[idx])
    tf.sign = lambda x: T(np.sign(x.a))
    tf.abs = lambda x: T(np.abs(x.a))

    def get_variable(name, validate_shape=True, initializer=None, trainable=True):
        created.append(np.array(initializer.a, np.float32))
        return T(created[-1])
    tf.get_variable = get_variable
    contrib = types.ModuleType('tensorflow.contrib')
    contrib.graph_editor = types.SimpleNamespace()
    contrib.distributions = types.SimpleNamespace(
        percentile=lambda x, q, axis=None: T(ORC.percentile_nearest(x.a, float(q), axis=axis)))
    tf.contrib = contrib
    return tf, contrib


def load_reference(ref, stubs):
    saved = {k: sys.modules.get(k) for k in stubs}
    sys.modules.update(stubs)
    try:
        spec = importlib.util.spec_from_file_location('ref_nuq_utils_bucket',
                                                      os.path.join(ref, 'learners/nonuniform_quantization/utils.py'))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def cases():
    """(shape, bits, bucket_type, bucket_size, kind); kind: 'normal' | 'constant' (one constant bucket, alpha = 1e-10)
    | 'ties' (values on a coarse grid: equal order statistics and centroid distances)"""
    out = []
    for shape in [(3, 3, 8, 16), (64, 10), (3, 3, 16, 1), (5, 5, 3, 7)]:        # conv, dense, depthwise, odd conv
        for bits in (1, 2, 4, 8):
            out.append((shape, bits, 'channel', 256, 'normal'))
            out.append((shape, bits, 'split', 256, 'normal'))          # 1152 / 640 / 144 / 525 elements
            out.append((shape, bits, 'split', 100, 'normal'))          # numel % bucket_size != 0
    for shape, btype, bsz in [((3, 3, 8, 16), 'channel', 256), ((64, 10), 'split', 64), ((3, 3, 4, 1), 'split', 256)]:
        for bits in (2, 4):
            out.append((shape, bits, btype, bsz, 'constant'))
            out.append((shape, bits, btype, bsz, 'ties'))
    return out


def make_input(ci, shape, btype, bsz, kind):
    rng = np.random.default_rng(6000 + ci)
    x = (rng.standard_normal(shape) * rng.choice([1e-2, 1.0, 9.0])).astype(np.float32)
    if kind == 'ties':
        x = (rng.integers(-3, 4, size=shape) * 0.25).astype(np.float32)
    elif kind == 'constant':
        flat = x.reshape(-1)
        ncols = shape[-1] if btype == 'channel' else -(-flat.size // bsz)
        flat[0::ncols] = flat[0]                                        # bucket 0 holds one value
        if btype == 'split' and flat.size % bsz:
            flat[-1] = flat[0]                                          # ... its padding copies too
    return x


def main():
    if len(sys.argv) != 2:
        raise SystemExit('usage: python tests/golden/make_golden_nuq_bucket.py <PocketFlow reference checkout>')
    ref = sys.argv[1]
    created = []
    tf, contrib = make_tf(created)
    mod = load_reference(ref, {'tensorflow': tf, 'tensorflow.contrib': contrib,
                               'tensorflow.contrib.graph_editor': contrib.graph_editor})
    quant = getattr(mod.NonUniformQuantization, '_NonUniformQuantization__bucket_quantize')
    fake_sess = types.SimpleNamespace(graph=types.SimpleNamespace(gradient_override_map=lambda m: Ctx()))
    gold = {'source': '__bucket_quantize of learners/nonuniform_quantization/utils.py executed on numpy stub tensors',
            'cases': []}
    _print = builtins.print
    builtins.print = lambda *a, **k: None                               # the reference prints "Quantized: ..."
    try:
        for ci, (shape, bits, btype, bsz, kind) in enumerate(cases()):
            x = make_input(ci, shape, btype, bsz, kind)
            obj = mod.NonUniformQuantization(fake_sess, bsz, True, 'quantile', btype)
            del created[:]
            q = quant(obj, T(x), bits, 'weight', 'p')
            out = np.ascontiguousarray(q.a, np.float32)
            assert out.shape == tuple(shape) and len(created) == 1
            clusters = np.ascontiguousarray(created[0], np.float32)
            gold['cases'].append(dict(index=ci, seed=6000 + ci, shape=list(shape), bits=bits, bucket_type=btype,
                                      bucket_size=bsz, kind=kind, clusters_shape=list(clusters.shape),
                                      sha256=hashlib.sha256(out.tobytes()).hexdigest(),
                                      clusters_sha256=hashlib.sha256(clusters.tobytes()).hexdigest(),
                                      bucket_storage=int(obj.bucket_storage), distinct=int(len(np.unique(out)))))
    finally:
        builtins.print = _print
    with open(OUT, 'w') as f:
        json.dump(gold, f, indent=1)
    print('wrote %s: %d cases' % (OUT, len(gold['cases'])))


if __name__ == '__main__':
    main()
