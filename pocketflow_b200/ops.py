"""Host-side operator layer over the C ABI (include/pf_b200.h).

Holds PyTorch CUDA tensors (device memory, streams) and calls libpf_b200.so through ctypes.  Each
class/function names the reference op chain it replaces.  Pure host logic (bucket layouts, work
tables, percentile ranks) lives in functions that need no GPU, so it is unit-tested on CPU.
"""
import ctypes
import os

import numpy as np
import torch

from . import lib as _lib

UQ_SEG = np.dtype([('src', 'u8'), ('dst', 'u8'), ('numel', 'i8'), ('padded', 'i8'),
                   ('ncols', 'i4'), ('bucket0', 'i4'), ('bits', 'i4'), ('reserved', 'i4')])
WORK = np.dtype([('seg', 'i4'), ('kind', 'i4'), ('start', 'i8'), ('count', 'i4'),
                 ('c0', 'i4'), ('ncol_tile', 'i4'), ('reserved', 'i4')])
WS_SEG = np.dtype([('w', 'u8'), ('bkup', 'u8'), ('mask', 'u8'), ('numel', 'i8')])
assert UQ_SEG.itemsize == 48 and WORK.itemsize == 32 and WS_SEG.itemsize == 32

CHUNK = 8192            # elements per CTA work item of the elementwise multi-tensor kernels
WS_WORKSPACE_U32 = 264  # PF_WS_WORKSPACE_U32_PER_SEG
L2_PARTIALS = 1024      # PF_L2_PARTIALS


# ----------------------------------------------------------------------------- host-only helpers
def uq_bucket_layout(shape, use_buckets, bucket_type, bucket_size):
    """(ncols, padded) of a weight tensor: bucket id of flat element i is i % ncols.

    Mirrors __channel_bucket / __split_bucket (learners/uniform_quantization/utils.py:247-289)."""
    numel = int(np.prod(shape))
    if not use_buckets:
        return 1, numel
    if bucket_type == 'channel':
        return int(shape[-1]), numel
    if bucket_type == 'split':
        if bucket_size <= 0:
            raise ValueError('Bucket size must be a postive integer')
        multiple, rest = divmod(numel, bucket_size)
        if rest:
            multiple += 1
        return multiple, multiple * bucket_size
    raise ValueError("Unrecognized bucket type, must be 'weight' or 'channel'.")


def flat_works(numels, chunk=CHUNK):
    """kind-0 work items: chunks [start, start+count) of each tensor (start % 4 == 0)."""
    rows = []
    for s, n in enumerate(numels):
        for start in range(0, int(n), chunk):
            rows.append((s, 0, start, min(chunk, int(n) - start), 0, 0, 0))
    return np.array(rows, dtype=WORK) if rows else np.zeros(0, dtype=WORK)


def minmax_works(segs):
    """Work table of pf_uq_weight_minmax: flat chunks for per-layer ranges, column tiles x row
    ranges of the [padded/ncols, ncols] view for bucketed ranges."""
    rows = []
    for s, seg in enumerate(segs):
        ncols, numel, padded = int(seg['ncols']), int(seg['numel']), int(seg['padded'])
        if ncols == 1:
            for start in range(0, numel, CHUNK):
                rows.append((s, 0, start, min(CHUNK, numel - start), 0, 0, 0))
            continue
        tile = min(ncols, 1024 if ncols % 4 == 0 else 256)
        nrows = padded // ncols
        rows_per = max(64, (2 * CHUNK) // tile)
        for c0 in range(0, ncols, tile):
            tc = min(tile, ncols - c0)
            for r0 in range(0, nrows, rows_per):
                rows.append((s, 1, r0, min(rows_per, nrows - r0), c0, tc, 0))
    return np.array(rows, dtype=WORK) if rows else np.zeros(0, dtype=WORK)


NUQ_BUCKET_TILE_FLOATS = 8192   # PF_NUQ_BUCKET_TILE_FLOATS: codebook slice of one quantize work item
NUQ_BUCKET_MAX_TILE = 1024      # PF_NUQ_BUCKET_MAX_TILE
NUQ_BUCKET_MAX_ROWS = 16384     # PF_NUQ_BUCKET_MAX_ROWS: tallest bucket the quantile init sorts in shared memory
NUQ_BUCKET_GRAD_TILE = 32       # PF_NUQ_BUCKET_GRAD_TILE


def nuq_bucket_layout(shape, bucket_type, bucket_size):
    """(ncols, padded, rows) of a weight under bucketed codebooks: the [rows, ncols] view of __split_bucket /
    __channel_bucket (learners/nonuniform_quantization/utils.py:435-476).  A ValueError for buckets taller than the
    quantile init can sort (only reachable with a large --nuql_bucket_size, or channel buckets of a huge kernel)."""
    ncols, padded = uq_bucket_layout(shape, True, bucket_type, bucket_size)
    rows = padded // ncols
    if rows > NUQ_BUCKET_MAX_ROWS:
        raise ValueError('bucketed codebooks: a bucket of %d rows (weight %s, %s buckets) exceeds the %d rows the '
                         'quantile init supports' % (rows, tuple(shape), bucket_type, NUQ_BUCKET_MAX_ROWS))
    return ncols, padded, rows


def nuq_bucket_quant_works(segs):
    """kind-1 column tiles of pf_nuq_bucket_weight_quant: a tile's codebook slice (2^bits x tile floats) fits
    NUQ_BUCKET_TILE_FLOATS; about 16K elements per work item."""
    rows = []
    for s, seg in enumerate(segs):
        ncols, padded, nc = int(seg['ncols']), int(seg['padded']), 1 << int(seg['bits'])
        tile = min(ncols, NUQ_BUCKET_MAX_TILE, max(32, NUQ_BUCKET_TILE_FLOATS // nc))
        nrows = padded // ncols
        rows_per = max(1, 16384 // tile)
        for c0 in range(0, ncols, tile):
            for r0 in range(0, nrows, rows_per):
                rows.append((s, 1, r0, min(rows_per, nrows - r0), c0, min(tile, ncols - c0), 0))
    return np.array(rows, dtype=WORK) if rows else np.zeros(0, dtype=WORK)


def nuq_bucket_grad_works(segs, rows_per=256):
    """(work, tiles) of pf_nuq_bucket_cluster_grad: NUQ_BUCKET_GRAD_TILE columns x rows_per rows per work item; tile t
    lists its contiguous work items in start/count."""
    work, tiles = [], []
    for s, seg in enumerate(segs):
        ncols, padded = int(seg['ncols']), int(seg['padded'])
        nrows = padded // ncols
        for c0 in range(0, ncols, NUQ_BUCKET_GRAD_TILE):
            tc = min(NUQ_BUCKET_GRAD_TILE, ncols - c0)
            first = len(work)
            for r0 in range(0, nrows, rows_per):
                work.append((s, 1, r0, min(rows_per, nrows - r0), c0, tc, 0))
            tiles.append((s, 1, first, len(work) - first, c0, tc, 0))
    return np.array(work, dtype=WORK), np.array(tiles, dtype=WORK)


def percentile_rank_desc(n, q):
    """Index into the descending sort gathered by tf.contrib.distributions.percentile
    (interpolation='nearest'): clip(int32(rint((n-1)*(1-q/100))), 0, n-1) in float64."""
    idx = int(np.rint((float(n) - 1.0) * (1.0 - float(q) / 100.0)))
    return min(max(idx, 0), n - 1)


def ws_rank_desc(n, prune_ratio):
    """Rank used by WeightSparseLearner.__build_masks: q = float32(ratio)*100 in float32
    (learners/weight_sparsification/learner.py:284)."""
    return percentile_rank_desc(n, np.float32(np.float32(prune_ratio) * np.float32(100.0)))


def decode_ordered(u):
    """numpy inverse of the ordered-uint float encoding used by the min/max slots."""
    u = np.asarray(u).astype(np.uint32)
    bits = np.where(u & 0x80000000, u & 0x7FFFFFFF, ~u).astype(np.uint32)
    return bits.view(np.float32)


# ----------------------------------------------------------------------------- device plumbing
def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _upload(arr, device):
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.uint8).copy()).to(device)


def _check_f32(*ts):
    for t in ts:
        if t is None:
            continue
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
            raise ValueError('expected a contiguous float32 CUDA tensor')
        if t.data_ptr() % 16:
            raise ValueError('tensor storage must be 16-byte aligned')


def launch_count():
    return int(_lib.load().pf_launch_count())


def launch_count_reset():
    _lib.load().pf_launch_count_reset()


# ----------------------------------------------------------------------------- a1/a3 weights
class UniformWeightQuantizer:
    """Multi-tensor weight fake-quantizer: ONE min/max launch + ONE quantize launch for all layers.

    Stands in for UniformQuantization.insert_quant_op_for_weights' per-layer
    __uniform_quantize(mode='weight') (learners/uniform_quantization/utils.py:81-113, 163-199)."""

    def __init__(self, srcs, dsts, bits, use_buckets=False, bucket_type='channel', bucket_size=256):
        self.L = _lib.load()
        if len(srcs) != len(dsts):
            raise ValueError('srcs/dsts length mismatch')
        _check_f32(*srcs)
        _check_f32(*dsts)
        if bucket_size < 0:
            raise ValueError('Bucket size must be a postive integer')
        if bucket_type not in ('split', 'channel'):
            raise ValueError("Unrecognized bucket type, must be 'weight' or 'channel'.")
        self.srcs, self.dsts = list(srcs), list(dsts)
        self.device = srcs[0].device if srcs else torch.device('cuda')
        segs = np.zeros(len(srcs), dtype=UQ_SEG)
        b0 = 0
        for i, (s, d) in enumerate(zip(srcs, dsts)):
            ncols, padded = uq_bucket_layout(tuple(s.shape), use_buckets, bucket_type, bucket_size)
            segs[i] = (s.data_ptr(), d.data_ptr(), s.numel(), padded, ncols, b0, 8, 0)
            b0 += (ncols + 3) // 4 * 4
        self.segs = segs
        self.n_buckets = max(b0, 4)
        self.bucket_counts = [int(s['ncols']) for s in segs]
        self.mn = torch.empty(self.n_buckets, dtype=torch.int32, device=self.device)
        self.mx = torch.empty(self.n_buckets, dtype=torch.int32, device=self.device)
        self.scales = torch.empty(3 * self.n_buckets, dtype=torch.float32, device=self.device)
        self.work_mm = minmax_works(segs)
        self.work_q = flat_works([int(s['numel']) for s in segs])
        self.work_mm_dev = _upload(self.work_mm, self.device)
        self.work_q_dev = _upload(self.work_q, self.device)
        self.grad_segs_dev = None
        self.set_bits(bits)

    def set_bits(self, bits):
        bits = [int(b) for b in (bits if hasattr(bits, '__len__') else [bits] * len(self.srcs))]
        if len(bits) != len(self.srcs):
            raise ValueError('one bit-width per tensor expected')
        if any(b < 1 or b > 32 for b in bits):
            raise ValueError('bit-widths must be in [1, 32]')
        self.bits = bits
        self.segs['bits'] = bits
        self.segs_dev = _upload(self.segs, self.device)
        self.grad_segs_dev = None
        self.__dict__.pop('_grad_subsets', None)

    def reset_ranges(self):
        st = _stream()
        _lib.check(self.L.pf_fill_u32(_p(self.mn), self.n_buckets, 0xFFFFFFFF, st), 'pf_fill_u32')
        _lib.check(self.L.pf_fill_u32(_p(self.mx), self.n_buckets, 0, st), 'pf_fill_u32')

    def minmax(self):
        self.reset_ranges()
        _lib.check(self.L.pf_uq_weight_minmax(_p(self.segs_dev), _p(self.work_mm_dev), len(self.work_mm),
                                              _p(self.mn), _p(self.mx), _stream()), 'pf_uq_weight_minmax')
        _lib.check(self.L.pf_uq_weight_scales(_p(self.mn), _p(self.mx), self.n_buckets, _p(self.scales), _stream()),
                   'pf_uq_weight_scales')

    def quantize(self):
        _lib.check(self.L.pf_uq_weight_quant(_p(self.segs_dev), _p(self.work_q_dev), len(self.work_q),
                                             _p(self.scales), self.n_buckets, _stream()), 'pf_uq_weight_quant')

    def forward(self):
        if not self.srcs:
            return
        self.minmax()
        self.quantize()

    def ste_backward_(self, grads, indices=None):
        """In-place STE chain on the gradients w.r.t. the quantized weights (a3).  indices: only these tensors (the
        gradient buckets of the data-parallel step finish at different times)."""
        _check_f32(*grads)
        if indices is not None:
            key = tuple(indices)
            cache = self.__dict__.setdefault('_grad_subsets', {})
            ent = cache.get(key)
            if ent is None or ent[0] != [grads[i].data_ptr() for i in indices]:
                gs = self.segs[list(indices)].copy()
                gs['src'] = [grads[i].data_ptr() for i in indices]
                gs['dst'] = gs['src']
                work = flat_works([int(s['numel']) for s in gs])
                ent = cache[key] = ([grads[i].data_ptr() for i in indices], _upload(gs, self.device),
                                    _upload(work, self.device), len(work))
            _lib.check(self.L.pf_uq_weight_ste_bwd(_p(ent[1]), _p(ent[2]), ent[3], _p(self.scales), self.n_buckets,
                                                   _stream()), 'pf_uq_weight_ste_bwd')
            return
        if self.grad_segs_dev is None or self._grad_ptrs != [g.data_ptr() for g in grads]:
            gs = self.segs.copy()
            gs['src'] = [g.data_ptr() for g in grads]
            gs['dst'] = gs['src']
            self.grad_segs_dev = _upload(gs, self.device)
            self._grad_ptrs = [g.data_ptr() for g in grads]
        _lib.check(self.L.pf_uq_weight_ste_bwd(_p(self.grad_segs_dev), _p(self.work_q_dev), len(self.work_q),
                                               _p(self.scales), self.n_buckets, _stream()), 'pf_uq_weight_ste_bwd')

    def ranges(self):
        """Per tensor (min, max) arrays decoded from the slots (host copy; tests/diagnostics)."""
        mn = decode_ordered(self.mn.cpu().numpy().view(np.uint32))
        mx = decode_ordered(self.mx.cpu().numpy().view(np.uint32))
        out = []
        for s in self.segs:
            b0, nc = int(s['bucket0']), int(s['ncols'])
            out.append((mn[b0:b0 + nc].copy(), mx[b0:b0 + nc].copy()))
        return out

    def bucket_storage_bits(self):
        """2*32 bits per bucket (utils.py:299-306)."""
        return sum(self.bucket_counts) * 32 * 2


# ----------------------------------------------------------------------------- a2 activations
def act_range_reset(minmax):
    L = _lib.load()
    st = _stream()
    _lib.check(L.pf_fill_u32(_p(minmax), 1, 0xFFFFFFFF, st), 'pf_fill_u32')
    _lib.check(L.pf_fill_u32(ctypes.c_void_p(minmax.data_ptr() + 4), 1, 0, st), 'pf_fill_u32')


def act_minmax(x, minmax):
    """Accumulate the per-tensor range of x into minmax (int32[2], ordered-uint)."""
    _check_f32(x)
    _lib.check(_lib.load().pf_uq_act_minmax(_p(x), x.numel(), _p(minmax), _stream()), 'pf_uq_act_minmax')


def act_quant(x, y, minmax, bits, planes=None):
    """y = Q(x); `planes` = Planes to (also) receive y in the tensor-core operand format (y may then be None)."""
    _check_f32(x, y)
    if not 1 <= int(bits) <= 32:
        raise ValueError('bit-widths must be in [1, 32]')
    if planes is None:
        _lib.check(_lib.load().pf_uq_act_quant(_p(x), _p(y), x.numel(), _p(minmax), int(bits), _stream()),
                   'pf_uq_act_quant')
    else:
        _lib.check(_lib.load().pf_uq_act_quant_planes(_p(x), _p(y), _p(planes.hi), _p(planes.lo), x.numel(), _p(minmax),
                                                      int(bits), _stream()), 'pf_uq_act_quant_planes')


def act_fake_quant(x, bits, out=None, minmax=None):
    """Q(x) with per-tensor range — __uniform_quantize(mode='activation') (utils.py:51-79)."""
    if out is None:
        out = torch.empty_like(x)
    if minmax is None:
        minmax = torch.empty(2, dtype=torch.int32, device=x.device)
    act_range_reset(minmax)
    act_minmax(x, minmax)
    act_quant(x, out, minmax, bits)
    return out


# ----------------------------------------------------------------------------- a5 masks
class MaskBuilder:
    """Multi-tensor magnitude-mask build — WeightSparseLearner.__build_masks
    (learners/weight_sparsification/learner.py:260-294)."""

    def __init__(self, ws, bkups, masks):
        self.L = _lib.load()
        _check_f32(*ws)
        _check_f32(*bkups)
        _check_f32(*masks)
        self.ws, self.bkups, self.masks = list(ws), list(bkups), list(masks)
        self.device = ws[0].device
        segs = np.zeros(len(ws), dtype=WS_SEG)
        for i, (w, b, m) in enumerate(zip(ws, bkups, masks)):
            if not (w.numel() == b.numel() == m.numel()):
                raise ValueError('w/bkup/mask size mismatch')
            segs[i] = (w.data_ptr(), b.data_ptr(), m.data_ptr(), w.numel())
        self.segs = segs
        self.segs_dev = _upload(segs, self.device)
        self.work = flat_works([w.numel() for w in ws])
        self.work_dev = _upload(self.work, self.device)
        self.workspace = torch.zeros(len(ws) * WS_WORKSPACE_U32, dtype=torch.int32, device=self.device)
        self.thr = torch.zeros(len(ws), dtype=torch.float32, device=self.device)
        self.ranks = torch.zeros(len(ws), dtype=torch.int64, device=self.device)

    def build(self, prune_ratios):
        """prune_ratios: one (dynamic) float32 ratio per tensor."""
        ranks = [ws_rank_desc(w.numel(), r) for w, r in zip(self.ws, prune_ratios)]
        self.ranks.copy_(torch.tensor(ranks, dtype=torch.int64), non_blocking=False)
        _lib.check(self.L.pf_ws_mask_build(_p(self.segs_dev), len(self.ws), _p(self.work_dev), len(self.work),
                                           _p(self.ranks), _p(self.workspace), _p(self.thr), _stream()),
                   'pf_ws_mask_build')
        return ranks


def select_desc(tensors, queries):
    """Exact order statistics: queries = [(tensor_index, rank_desc)], returns a float32 CUDA tensor.
    Used by the codebook quantile init (learners/nonuniform_quantization/utils.py:349-366)."""
    L = _lib.load()
    _check_f32(*tensors)
    dev = tensors[0].device
    segs = np.zeros(len(tensors), dtype=WS_SEG)
    for i, t in enumerate(tensors):
        segs[i] = (0, t.data_ptr(), 0, t.numel())
    qseg = np.array([q[0] for q in queries], dtype=np.int32)
    ranks = torch.tensor([int(q[1]) for q in queries], dtype=torch.int64, device=dev)
    work = flat_works([tensors[q[0]].numel() for q in queries])
    ws = torch.zeros(len(queries) * WS_WORKSPACE_U32, dtype=torch.int32, device=dev)
    out = torch.empty(len(queries), dtype=torch.float32, device=dev)
    segs_dev, qseg_dev, work_dev = _upload(segs, dev), _upload(qseg, dev), _upload(work, dev)
    _lib.check(L.pf_select_desc(_p(segs_dev), _p(qseg_dev), len(queries), _p(work_dev), len(work),
                                _p(ranks), _p(ws), _p(out), _stream()), 'pf_select_desc')
    torch.cuda.current_stream().synchronize()   # tables above go out of scope
    return out


# ----------------------------------------------------------------------------- a6/a9 optimizers
def momentum_step(w, acc, g, mask, hp, momentum, wd=0.0, grad_scale=1.0):
    """g*mask + MomentumOptimizer.apply_gradients on a flat range
    (learners/weight_sparsification/learner.py:201-212, 314-332).  hp[0] = lr (device)."""
    _check_f32(w, acc, g, mask, hp)
    _lib.check(_lib.load().pf_momentum_step(_p(w), _p(acc), _p(g), _p(mask), w.numel(), _p(hp),
                                            float(momentum), float(wd), float(grad_scale), _stream()),
               'pf_momentum_step')


def adam_step(w, m, v, g, hp, beta1=0.9, beta2=0.999, eps=1e-8, wd=0.0, grad_scale=1.0):
    """tf.train.AdamOptimizer step on a flat range (uniform_quantization/learner.py:244).
    hp = [lr, beta1_power, beta2_power] (device)."""
    _check_f32(w, m, v, g, hp)
    _lib.check(_lib.load().pf_adam_step(_p(w), _p(m), _p(v), _p(g), w.numel(), _p(hp), float(beta1),
                                        float(beta2), float(eps), float(wd), float(grad_scale), _stream()),
               'pf_adam_step')


# ----------------------------------------------------------------------------- a7/a8 losses
def softmax_ce(logits, labels, teacher=None, tempr=4.0, w_dst=4.0, dlogits=None, out=None, row_ws=None):
    """hard CE (+ distillation CE) forward and d/dlogits.  Returns (out[4], dlogits):
    out = [hard, dst, top-1 accuracy, top-5 accuracy]."""
    _check_f32(logits, labels, teacher)
    n, k = logits.shape
    if labels.shape != logits.shape or (teacher is not None and teacher.shape != logits.shape):
        raise ValueError('labels/teacher must match logits shape')
    if dlogits is None:
        dlogits = torch.empty_like(logits)
    if out is None:
        out = torch.empty(4, dtype=torch.float32, device=logits.device)
    if row_ws is None:
        row_ws = torch.empty(4 * n, dtype=torch.float32, device=logits.device)
    _lib.check(_lib.load().pf_softmax_ce_fwd_bwd(_p(logits), _p(labels), _p(teacher), n, k, float(tempr),
                                                 float(w_dst), _p(dlogits), _p(out), _p(row_ws), _stream()),
               'pf_softmax_ce_fwd_bwd')
    return out, dlogits


def l2_loss(v, scale, out, partial_ws, accumulate=False):
    """out[0] (+)= scale * sum(v^2)/2 — tf.nn.l2_loss terms (nets/resnet_at_cifar10.py:105-107)."""
    _check_f32(v, out, partial_ws)
    _lib.check(_lib.load().pf_l2_loss(_p(v), v.numel(), float(scale), int(bool(accumulate)), _p(out),
                                      _p(partial_ws), _stream()), 'pf_l2_loss')


# ----------------------------------------------------------------------------- a11 codebooks
class CodebookWeightQuantizer:
    """Multi-tensor codebook quantizer, per-layer range —
    NonUniformQuantization.__nonuni_quantize (learners/nonuniform_quantization/utils.py:168-194).

    The codebooks are either a private [tensors, 256] table (`clusters`), or — `cluster_views` — 1-D views of ONE flat
    buffer `cluster_base` that the caller owns: the reference's trainable `clusters` variables (utils.py:297), which then
    sit among the model's parameters (optimizer, weight decay, checkpoints, broadcast all apply to them).

    use_buckets (NonUniformQuantization.__bucket_quantize, utils.py:196-243): one codebook per 'split' / 'channel'
    bucket, ranges per bucket through the bucketed UniformWeightQuantizer.  The codebooks of a tensor are then a
    [2^bits, ncols] row-major table — a view of cluster_base (the reference's [k, bucket_num] `clusters` variable), or
    a private buffer when no views are given."""

    def __init__(self, srcs, dsts, bits, keep_index=False, cluster_views=None, cluster_base=None, use_buckets=False,
                 bucket_type='split', bucket_size=256):
        self.L = _lib.load()
        _check_f32(*srcs)
        _check_f32(*dsts)
        self.use_buckets = bool(use_buckets)
        if self.use_buckets:
            for s in srcs:
                nuq_bucket_layout(tuple(s.shape), bucket_type, bucket_size)     # bucket height, before any launch
        # per-layer or per-bucket ranges + tables
        self.uq = UniformWeightQuantizer(srcs, dsts, bits, self.use_buckets, bucket_type, bucket_size)
        if any(b > 8 for b in self.uq.bits):
            raise ValueError('codebook bit-widths must be <= 8')
        self.srcs, self.dsts = list(srcs), list(dsts)
        self.device = self.uq.device
        self.ncols = [int(s['ncols']) for s in self.uq.segs]
        self.cluster_views, self.cluster_base, self.cluster_off = None, None, None
        if cluster_views is None and self.use_buckets:
            sizes = [(1 << b) * nc for b, nc in zip(self.uq.bits, self.ncols)]
            offs = np.concatenate([[0], np.cumsum([(n + 3) // 4 * 4 for n in sizes])]).astype(np.int64)
            cluster_base = torch.zeros(max(int(offs[-1]), 4), dtype=torch.float32, device=self.device)
            cluster_views = [cluster_base[o:o + n].view(-1, nc) for o, n, nc in zip(offs, sizes, self.ncols)]
        if cluster_views is not None:
            _check_f32(cluster_base, *cluster_views)
            offs = []
            for v, b, nc in zip(cluster_views, self.uq.bits, self.ncols):
                off = (v.data_ptr() - cluster_base.data_ptr()) // 4
                if v.numel() < (1 << b) * nc or v.numel() % nc or off < 0 or off + v.numel() > cluster_base.numel():
                    raise ValueError('codebook views must hold at least 2^bits x buckets floats inside cluster_base')
                offs.append(off)
            self.cluster_views, self.cluster_base = list(cluster_views), cluster_base
            self.cluster_off = torch.tensor(offs, dtype=torch.int64, device=self.device)
            self.clusters = None
        else:
            self.clusters = torch.zeros(len(srcs), 256, dtype=torch.float32, device=self.device)
        self.idx = None
        if keep_index:
            offs, tot = [], 0
            for s in srcs:
                offs.append(tot)
                tot += (s.numel() + 15) // 16 * 16
            self.idx = torch.zeros(tot, dtype=torch.uint8, device=self.device)
            self.idx_base = torch.tensor(offs, dtype=torch.int64, device=self.device)
            self.idx_offsets = offs
        self._grad_tables = None
        if self.use_buckets:
            self._bucket_tables()

    def _bucket_tables(self):
        """Work tables of the bucketed kernels for the current bit-widths."""
        segs = self.uq.segs
        self.work_bq = nuq_bucket_quant_works(segs)
        self.work_bg, self.tiles_bg = nuq_bucket_grad_works(segs)
        self.work_bq_dev = _upload(self.work_bq, self.device)
        self.work_bg_dev = _upload(self.work_bg, self.device)
        self.tiles_bg_dev = _upload(self.tiles_bg, self.device)
        self.kmax = max([1 << b for b in self.uq.bits] or [1])
        self.max_rows = max([int(s['padded']) // int(s['ncols']) for s in segs] or [1])
        ranks = np.zeros((max(len(segs), 1), 256), np.int32)
        for i, s in enumerate(segs):
            k, rows = 1 << int(s['bits']), int(s['padded']) // int(s['ncols'])
            ranks[i, :k] = [percentile_rank_desc(rows, (j + 1) * 100 / (k + 1)) for j in range(k)]
        self.ranks_dev = _upload(ranks, self.device)

    def quantile_values(self):
        """clusters_j = percentile(x_n, (j+1)*100/(k+1)) (utils.py:349-366), [tensors][k] as numpy.  x -> x_n is
        monotone non-decreasing in fp32, so the order statistic is selected on the raw weights (exact radix select)
        and normalised afterwards with the same fp32 ops."""
        self.uq.minmax()
        queries = []
        for i, s in enumerate(self.srcs):
            k = 1 << self.uq.bits[i]
            for j in range(k):
                queries.append((i, percentile_rank_desc(s.numel(), (j + 1) * 100 / (k + 1))))
        vals = select_desc(self.srcs, queries).cpu().numpy()
        rng = self.uq.ranges()
        out, pos = [], 0
        for i in range(len(self.srcs)):
            k = 1 << self.uq.bits[i]
            mn, mx = rng[i][0][0], rng[i][1][0]
            alpha = np.float32(np.float32(mx - mn) + np.float32(1e-10))
            out.append(((vals[pos:pos + k] - mn).astype(np.float32) / alpha).astype(np.float32))
            pos += k
        return out

    def set_bits(self, bits):
        """New bit-widths (the RL bit search): a codebook keeps its place and uses its first 2^bits entries (per-bucket
        codebooks: the first 2^bits rows of the [k, ncols] table); call quantile_init() afterwards."""
        bits = [int(b) for b in (bits if hasattr(bits, '__len__') else [bits] * len(self.srcs))]
        if any(b < 1 or b > 8 for b in bits):
            raise ValueError('codebook bit-widths must be in [1, 8]')
        if self.cluster_views is not None and any(v.numel() < (1 << b) * nc
                                                  for v, b, nc in zip(self.cluster_views, bits, self.ncols)):
            raise ValueError('a codebook variable is smaller than 2^bits')
        self.uq.set_bits(bits)
        self._grad_tables = None
        if self.use_buckets:
            self._bucket_tables()

    def quantile_init(self):
        if self.use_buckets:
            # __quantile_init(axis=0) per bucket, on the device, straight into the codebook tables
            self.uq.minmax()
            for v, b, nc in zip(self.cluster_views, self.uq.bits, self.ncols):
                if v.numel() > (1 << b) * nc:
                    v.zero_()                               # rows past 2^bits stay 0 (no weight-decay term)
            _lib.check(self.L.pf_nuq_bucket_quantile_init(_p(self.uq.segs_dev), len(self.srcs), _p(self.uq.scales),
                                                          self.uq.n_buckets, _p(self.ranks_dev), self.max_rows,
                                                          _p(self.cluster_base), _p(self.cluster_off), _stream()),
                       'pf_nuq_bucket_quantile_init')
            return
        vals = self.quantile_values()
        if self.cluster_views is not None:
            for v, c in zip(self.cluster_views, vals):
                v.zero_()                                   # entries past 2^bits stay 0 (no weight-decay term)
                v[:c.size].copy_(torch.from_numpy(c))
            return
        c = np.zeros((len(self.srcs), 256), np.float32)
        for i, v in enumerate(vals):
            c[i, :v.size] = v
        self.clusters.copy_(torch.from_numpy(c))

    def forward(self):
        self.uq.minmax()
        idx_base = _p(self.idx_base) if self.idx is not None else None
        if self.use_buckets:
            _lib.check(self.L.pf_nuq_bucket_weight_quant(_p(self.uq.segs_dev), _p(self.work_bq_dev), len(self.work_bq),
                                                         _p(self.uq.scales), self.uq.n_buckets, _p(self.cluster_base),
                                                         _p(self.cluster_off), _p(self.idx), idx_base, _stream()),
                       'pf_nuq_bucket_weight_quant')
        elif self.cluster_views is not None:
            _lib.check(self.L.pf_nuq_weight_quant_ex(_p(self.uq.segs_dev), _p(self.uq.work_q_dev), len(self.uq.work_q),
                                                     _p(self.uq.scales), self.uq.n_buckets, _p(self.cluster_base),
                                                     _p(self.cluster_off), _p(self.idx), idx_base, _stream()),
                       'pf_nuq_weight_quant_ex')
        else:
            _lib.check(self.L.pf_nuq_weight_quant(_p(self.uq.segs_dev), _p(self.uq.work_q_dev), len(self.uq.work_q),
                                                  _p(self.uq.scales), self.uq.n_buckets, _p(self.clusters),
                                                  _p(self.idx), idx_base, _stream()), 'pf_nuq_weight_quant')

    def cluster_grad(self, grads, grad_base):
        """dL/dc_j = alpha * sum_{idx = j} g (learner.py:252-261 through utils.py:303-306, :433): `grads` = the gradients
        w.r.t. the QUANTIZED tensors (one per src), results written to grad_base + the codebooks' offsets (grad_base has
        the layout of cluster_base).  Needs keep_index and store-resident codebooks."""
        if self.idx is None or self.cluster_off is None:
            raise ValueError('cluster_grad needs keep_index=True and cluster_views')
        _check_f32(grad_base, *grads)
        ptrs = [g.data_ptr() for g in grads]
        if self.use_buckets:
            # dL/dc[j, b] = alpha_b * sum_{idx = j} g over the bucket's rows (padding rows excluded)
            if self._grad_tables is None or self._grad_tables[0] != ptrs:
                gs = self.uq.segs.copy()
                gs['src'] = ptrs
                gs['dst'] = ptrs
                self._grad_tables = (ptrs, _upload(gs, self.device),
                                     torch.empty(max(len(self.work_bg), 1) * self.kmax * NUQ_BUCKET_GRAD_TILE,
                                                 dtype=torch.float32, device=self.device))
            _, gsegs, partial = self._grad_tables
            _lib.check(self.L.pf_nuq_bucket_cluster_grad(_p(gsegs), _p(self.work_bg_dev), len(self.work_bg),
                                                         _p(self.tiles_bg_dev), len(self.tiles_bg), self.kmax,
                                                         _p(self.idx), _p(self.idx_base), _p(self.uq.scales),
                                                         _p(partial), _p(grad_base), _p(self.cluster_off), _stream()),
                       'pf_nuq_bucket_cluster_grad')
            return
        if self._grad_tables is None or self._grad_tables[0] != ptrs:
            gs = self.uq.segs.copy()
            gs['src'] = ptrs
            gs['dst'] = ptrs
            first = np.zeros(len(self.srcs) + 1, np.int32)
            for w in self.uq.work_q:
                first[int(w['seg']) + 1] += 1
            first = np.cumsum(first).astype(np.int32)
            self._grad_tables = (ptrs, _upload(gs, self.device), _upload(first, self.device),
                                 torch.empty(max(len(self.uq.work_q), 1) * 256, dtype=torch.float32, device=self.device))
        _, gsegs, first_dev, partial = self._grad_tables
        _lib.check(self.L.pf_nuq_cluster_grad(_p(gsegs), len(self.srcs), _p(self.uq.work_q_dev), len(self.uq.work_q),
                                              _p(first_dev), _p(self.idx), _p(self.idx_base), _p(self.uq.scales),
                                              _p(partial), _p(grad_base), _p(self.cluster_off), _stream()),
                   'pf_nuq_cluster_grad')

    def bucket_storage_bits(self):
        """Extra storage of the per-bucket alpha and beta, 64 bits per bucket (__updt_bucket_storage, utils.py:487-494);
        the per-layer quantizer counts none."""
        return self.uq.bucket_storage_bits() if self.use_buckets else 0


# ----------------------------------------------------------------------------- a4 conv / a13 layers
BN_MAX_SPLITS = 1024


def conv_desc(n, h, w, c, k, r, s, p, q, sh, sw, pt, pl):
    return _lib.ConvDesc(n, h, w, c, k, r, s, p, q, sh, sw, pt, pl)


def im2col(d, x, kpad, cols):
    _lib.check(_lib.load().pf_im2col(ctypes.byref(d), _p(x), int(kpad), _p(cols), _stream()), 'pf_im2col')


def conv2d_fwd(d, x, w, bias, relu, y):
    _lib.check(_lib.load().pf_conv2d_fwd(ctypes.byref(d), _p(x), _p(w), _p(bias), int(bool(relu)), _p(y), _stream()),
               'pf_conv2d_fwd')


def conv2d_dgrad(d, dy, w, wt_ws, accumulate, dx):
    _lib.check(_lib.load().pf_conv2d_dgrad(ctypes.byref(d), _p(dy), _p(w), _p(wt_ws), int(bool(accumulate)), _p(dx),
                                           _stream()), 'pf_conv2d_dgrad')


def conv2d_wgrad_workspace_floats(d):
    return int(_lib.load().pf_conv2d_wgrad_workspace_bytes(ctypes.byref(d))) // 4


def conv2d_wgrad(d, x, dy, ws, dw):
    _lib.check(_lib.load().pf_conv2d_wgrad(ctypes.byref(d), _p(x), _p(dy), _p(ws), _p(dw), _stream()),
               'pf_conv2d_wgrad')


def bn_train_stats(x, m, c, eps, momentum, mean, var, rstd, mov_mean, mov_var, ws):
    _lib.check(_lib.load().pf_bn_train_stats(_p(x), m, c, float(eps), float(momentum), _p(mean), _p(var), _p(rstd),
                                             _p(mov_mean), _p(mov_var), _p(ws), _stream()), 'pf_bn_train_stats')


def bn_train_stats_range(x, m, c, eps, momentum, mean, var, rstd, mov_mean, mov_var, gamma, beta, act, minmax, ws):
    """batch statistics + range of act(bn(x)) (for the activation quantizer) in the same pass over x"""
    _lib.check(_lib.load().pf_bn_train_stats_range(_p(x), m, c, float(eps), float(momentum), _p(mean), _p(var), _p(rstd),
                                                   _p(mov_mean), _p(mov_var), _p(gamma), _p(beta), int(act), _p(minmax),
                                                   _p(ws), _stream()), 'pf_bn_train_stats_range')


def bn_apply_eval(x, m, c, mov_mean, mov_var, eps, gamma, beta, act, y, minmax=None, planes=None):
    """inference-mode BN (+act) in one launch, to fp32 and/or operand planes"""
    _lib.check(_lib.load().pf_bn_apply_eval(_p(x), m, c, _p(mov_mean), _p(mov_var), float(eps), _p(gamma), _p(beta), int(act),
                                            _p(y), _p(planes.hi if planes is not None else None),
                                            _p(planes.lo if planes is not None else None), _p(minmax), _stream()),
               'pf_bn_apply_eval')


def bn_apply_quant(x, m, c, mean, rstd, gamma, beta, act, rng, bits, y=None, planes=None):
    """Q(act(bn(x))) with a known range, to fp32 and/or operand planes"""
    _lib.check(_lib.load().pf_bn_apply_quant(_p(x), m, c, _p(mean), _p(rstd), _p(gamma), _p(beta), int(act), _p(rng),
                                             int(bits), _p(y), _p(planes.hi if planes is not None else None),
                                             _p(planes.lo if planes is not None else None), _stream()), 'pf_bn_apply_quant')


def bn_apply_quant_levels(x, m, c, mean, rstd, gamma, beta, act, rng, bits, y, planes, hdr, csum):
    """Q(act(bn(x))) as a pf_tc_act: integer levels (or hi / lo planes) + device header + channel sums"""
    _lib.check(_lib.load().pf_bn_apply_quant_levels(_p(x), m, c, _p(mean), _p(rstd), _p(gamma), _p(beta), int(act), _p(rng),
                                                    int(bits), _p(y), _p(planes.hi), _p(planes.lo), _p(hdr), _p(csum), _stream()),
               'pf_bn_apply_quant_levels')


def bn_eval_prepare(mov_var, c, eps, rstd):
    _lib.check(_lib.load().pf_bn_eval_prepare(_p(mov_var), c, float(eps), _p(rstd), _stream()), 'pf_bn_eval_prepare')


def bn_apply(x, m, c, mean, rstd, gamma, beta, act, y, minmax=None, planes=None):
    if planes is None:
        _lib.check(_lib.load().pf_bn_apply(_p(x), m, c, _p(mean), _p(rstd), _p(gamma), _p(beta), int(act), _p(y),
                                           _p(minmax), _stream()), 'pf_bn_apply')
    else:
        _lib.check(_lib.load().pf_bn_apply_planes(_p(x), m, c, _p(mean), _p(rstd), _p(gamma), _p(beta), int(act), _p(y),
                                                  _p(planes.hi), _p(planes.lo), _p(minmax), _stream()),
                   'pf_bn_apply_planes')


def bn_bwd(dy, x, m, c, mean, rstd, gamma, beta, act, dgamma, dbeta, dx, accumulate, ws, planes=None):
    if planes is None:
        _lib.check(_lib.load().pf_bn_bwd(_p(dy), _p(x), m, c, _p(mean), _p(rstd), _p(gamma), _p(beta), int(act),
                                         _p(dgamma), _p(dbeta), _p(dx), int(bool(accumulate)), _p(ws), _stream()),
                   'pf_bn_bwd')
    else:
        _lib.check(_lib.load().pf_bn_bwd_planes(_p(dy), _p(x), m, c, _p(mean), _p(rstd), _p(gamma), _p(beta), int(act),
                                                _p(dgamma), _p(dbeta), _p(dx), int(bool(accumulate)), _p(planes.hi),
                                                _p(planes.lo), _p(ws), _stream()), 'pf_bn_bwd_planes')


def add(a, b, out, accumulate=False):
    _lib.check(_lib.load().pf_add(_p(a), _p(b), a.numel(), int(bool(accumulate)), _p(out), _stream()), 'pf_add')


def fold_diag_blocks(src, g, m, n, dst):
    _lib.check(_lib.load().pf_fold_diag_blocks(_p(src), int(g), int(m), int(n), _p(dst), _stream()), 'pf_fold_diag_blocks')


def relu_bwd(dy, y, dx, act=1, accumulate=False):
    _lib.check(_lib.load().pf_relu_bwd(_p(dy), _p(y), y.numel(), int(act), int(bool(accumulate)), _p(dx), _stream()),
               'pf_relu_bwd')


def colsum(a, m, c, out):
    _lib.check(_lib.load().pf_colsum(_p(a), m, c, _p(out), _stream()), 'pf_colsum')


def maxpool_fwd(d, x, y, argmax=None):
    _lib.check(_lib.load().pf_maxpool_fwd(ctypes.byref(d), _p(x), _p(y), _p(argmax), _stream()), 'pf_maxpool_fwd')


def maxpool_bwd(d, dy, argmax, dx, accumulate=False):
    _lib.check(_lib.load().pf_maxpool_bwd(ctypes.byref(d), _p(dy), _p(argmax), int(bool(accumulate)), _p(dx),
                                          _stream()), 'pf_maxpool_bwd')


def global_avgpool_fwd(x, n, hw, c, y):
    _lib.check(_lib.load().pf_global_avgpool_fwd(_p(x), n, hw, c, _p(y), _stream()), 'pf_global_avgpool_fwd')


def global_avgpool_bwd(dy, n, hw, c, dx, accumulate=False):
    _lib.check(_lib.load().pf_global_avgpool_bwd(_p(dy), n, hw, c, int(bool(accumulate)), _p(dx), _stream()),
               'pf_global_avgpool_bwd')


def softmax_fwd(x, y):
    _lib.check(_lib.load().pf_softmax_fwd(_p(x), x.shape[0], x.shape[1], _p(y), _stream()), 'pf_softmax_fwd')


def softmax_bwd(dy, y, dx):
    _lib.check(_lib.load().pf_softmax_bwd(_p(dy), _p(y), y.shape[0], y.shape[1], _p(dx), _stream()), 'pf_softmax_bwd')


def minmax_reset(slots):
    """slots: int32 [n, 2] -> every pair = (0xFFFFFFFF, 0)."""
    _lib.check(_lib.load().pf_minmax_reset(_p(slots), slots.numel() // 2, _stream()), 'pf_minmax_reset')


# ----------------------------------------------------------------------------- a4 on tensor cores
def conv2d_tc_supported(d):
    return bool(_lib.load().pf_conv2d_tc_supported(ctypes.byref(d)))


class TcWeights:
    """Split-bf16, K-major copies of one conv kernel for the tcgen05 path (fwd and dgrad operands)."""

    def __init__(self, d, device, need_dgrad=True):
        L = _lib.load()
        self.d = d
        nf = int(L.pf_conv2d_tc_weight_elems(ctypes.byref(d), 0))
        self.f_hi = torch.zeros(nf, dtype=torch.bfloat16, device=device)
        self.f_lo = torch.zeros(nf, dtype=torch.bfloat16, device=device)
        self.d_hi = self.d_lo = None
        if need_dgrad:
            nd = int(L.pf_conv2d_tc_weight_elems(ctypes.byref(d), 1))
            self.d_hi = torch.zeros(nd, dtype=torch.bfloat16, device=device)
            self.d_lo = torch.zeros(nd, dtype=torch.bfloat16, device=device)

    def prepare(self, w):
        _lib.check(_lib.load().pf_conv2d_tc_prep_weight(ctypes.byref(self.d), _p(w), _p(self.f_hi), _p(self.f_lo),
                                                        _p(self.d_hi), _p(self.d_lo), _stream()),
                   'pf_conv2d_tc_prep_weight')


TC_PREP_SEG = np.dtype([('w', np.uint64), ('fwd_hi', np.uint64), ('fwd_lo', np.uint64), ('dgrad_hi', np.uint64),
                        ('dgrad_lo', np.uint64), ('rs', np.int32), ('c', np.int32), ('k', np.int32),
                        ('kpad_f', np.int32), ('kpad_d', np.int32), ('q_bits', np.int32), ('q_alpha', np.uint64),
                        ('q_beta', np.uint64), ('q_ralpha', np.uint64), ('q_ncols', np.int32), ('reserved', np.int32)],
                       align=True)
assert TC_PREP_SEG.itemsize == 96


class TcWeightsBatch:
    """One launch that refreshes the split-bf16 copies of MANY conv kernels (pf_conv2d_tc_prep_weights_multi)."""

    def __init__(self, items, device, levels=None):
        """items: list of (TcWeights, fp32 HWIO weight tensor [R,S,C,K]).
        levels: {item index: (unquantized weight tensor, alpha, beta, ralpha device views at the tensor's first bucket,
        ncols, bits)} — those kernels are prepared as integer levels from the UNQUANTIZED weights (pf_tc_prep_seg)."""
        segs = np.zeros(len(items), dtype=TC_PREP_SEG)
        rows = []
        self.levels = dict(levels or {})
        for i, (tw, w) in enumerate(items):
            r, s_, c, k = w.shape if w.dim() == 4 else (1, 1) + tuple(w.shape)
            segs[i] = (w.data_ptr(), tw.f_hi.data_ptr(), tw.f_lo.data_ptr(),
                       tw.d_hi.data_ptr() if tw.d_hi is not None else 0, tw.d_lo.data_ptr() if tw.d_lo is not None else 0,
                       r * s_, c, k, tw.f_hi.numel() // k, (tw.d_hi.numel() // c) if tw.d_hi is not None else 0, 0, 0, 0, 0, 0, 0)
        self.segs_plain = segs.copy()
        for i, (tw, w) in enumerate(items):
            r, s_, c, k = w.shape if w.dim() == 4 else (1, 1) + tuple(w.shape)
            if i in self.levels:
                w0, al, be, ra, ncols, bits = self.levels[i]
                if ncols not in (1, k) or not 1 <= int(bits) <= 8:
                    raise ValueError('weight levels need per-layer or per-output-channel buckets and 1..8 bits')
                segs[i]['w'], segs[i]['q_bits'], segs[i]['q_ncols'] = w0.data_ptr(), int(bits), int(ncols)
                segs[i]['q_alpha'], segs[i]['q_beta'], segs[i]['q_ralpha'] = al.data_ptr(), be.data_ptr(), ra.data_ptr()
            for k0 in range(0, r * s_ * c, 32):                 # 32 x 64 tiles of the [R*S*Cin, Cout] matrix
                for co0 in range(0, k, 64):
                    rows.append((i, 0, k0, 0, co0, 0, 0))
        self.keep = items
        self.segs = segs
        self.device = device
        self.work = np.array(rows, dtype=WORK) if rows else np.zeros(0, dtype=WORK)
        self.segs_dev = torch.from_numpy(segs.view(np.uint8).copy()).to(device)
        self.segs_plain_dev = torch.from_numpy(self.segs_plain.view(np.uint8).copy()).to(device) if self.levels else self.segs_dev
        self.work_dev = torch.from_numpy(self.work.view(np.uint8)).to(device)

    def set_bits(self, bits_of):
        """{item index: bits} for the level-prepared kernels (the RL bit search changes them between roll-outs);
        above 8 bits a kernel goes back to split-bf16 planes of its quantized values"""
        for i, b in bits_of.items():
            if i in self.levels:
                if 1 <= int(b) <= 8:
                    self.segs[i]['q_bits'], self.segs[i]['w'] = int(b), self.levels[i][0].data_ptr()
                else:
                    self.segs[i]['q_bits'], self.segs[i]['w'] = 0, self.segs_plain[i]['w']
        self.segs_dev = torch.from_numpy(self.segs.view(np.uint8).copy()).to(self.device)

    def prepare(self, levels=True):
        """levels=False: every kernel as split-bf16 planes of the tensors given at construction (evaluation passes)"""
        segs = self.segs_dev if levels else self.segs_plain_dev
        _lib.check(_lib.load().pf_conv2d_tc_prep_weights_multi(_p(segs), _p(self.work_dev), len(self.work),
                                                               _stream()), 'pf_conv2d_tc_prep_weights_multi')


def conv2d_tc_fwd(d, x, tw, bias, relu, y, residual=None):
    _lib.check(_lib.load().pf_conv2d_tc_fwd(ctypes.byref(d), _p(x), _p(tw.f_hi), _p(tw.f_lo), _p(bias),
                                            int(bool(relu)), _p(residual), _p(y), _stream()), 'pf_conv2d_tc_fwd')


def conv2d_tc_dgrad(d, dy, tw, accumulate, dx):
    _lib.check(_lib.load().pf_conv2d_tc_dgrad(ctypes.byref(d), _p(dy), _p(tw.d_hi), _p(tw.d_lo),
                                              int(bool(accumulate)), _p(dx), _stream()), 'pf_conv2d_tc_dgrad')


def conv2d_tc_wgrad_supported(d):
    return bool(_lib.load().pf_conv2d_tc_wgrad_supported(ctypes.byref(d)))


def conv2d_tc_wgrad_workspace_floats(d):
    return int(_lib.load().pf_conv2d_tc_wgrad_workspace_bytes(ctypes.byref(d))) // 4


def conv2d_tc_wgrad(d, x, dy, ws, dw):
    _lib.check(_lib.load().pf_conv2d_tc_wgrad(ctypes.byref(d), _p(x), _p(dy), _p(ws), _p(dw), _stream()),
               'pf_conv2d_tc_wgrad')


class Planes:
    """A tensor in the operand format of the tensor-core kernels: x = hi + lo, two bf16 planes with the layout of
    the fp32 tensor.  `buf` (optional) = one bf16 buffer of >= 2*numel elements to carve the planes from."""

    def __init__(self, numel, device, buf=None):
        assert numel % 8 == 0
        if buf is None:
            buf = torch.empty(2 * numel, dtype=torch.bfloat16, device=device)
            if os.environ.get('PF_POISON', '0') == '1':
                buf.fill_(float('nan'))
        assert buf.dtype == torch.bfloat16 and buf.numel() >= 2 * numel
        self.numel, self.buf = numel, buf
        self.hi, self.lo = buf[:numel], buf[numel:2 * numel]


def split_bf16(src, planes):
    """fp32 -> (hi, lo) bf16 planes."""
    _lib.check(_lib.load().pf_split_bf16(_p(src), _p(planes.hi), _p(planes.lo), src.numel(), _stream()), 'pf_split_bf16')


def conv2d_tc_fwd_planes(d, xp, tw, bias, relu, y, residual=None):
    _lib.check(_lib.load().pf_conv2d_tc_fwd_planes(ctypes.byref(d), _p(xp.hi), _p(xp.lo), _p(tw.f_hi), _p(tw.f_lo), _p(bias),
                                                   int(bool(relu)), _p(residual), _p(y), _stream()),
               'pf_conv2d_tc_fwd_planes')


def conv2d_tc_dgrad_planes(d, dyp, tw, accumulate, dx):
    _lib.check(_lib.load().pf_conv2d_tc_dgrad_planes(ctypes.byref(d), _p(dyp.hi), _p(dyp.lo), _p(tw.d_hi), _p(tw.d_lo),
                                                     int(bool(accumulate)), _p(dx), _stream()), 'pf_conv2d_tc_dgrad_planes')


def conv2d_tc_wgrad_planes_workspace_floats(d):
    return int(_lib.load().pf_conv2d_tc_wgrad_planes_workspace_bytes(ctypes.byref(d))) // 4


TC_REDUCE_SEG = np.dtype([('partial', np.uint64), ('out', np.uint64), ('n', np.int64), ('splits', np.int32),
                          ('reserved', np.int32)], align=True)


def conv2d_tc_wgrad_splits(d):
    return int(_lib.load().pf_conv2d_tc_wgrad_splits(ctypes.byref(d)))


class TcWgradReduceBatch:
    """Deferred split-K reduction of many weight gradients in one launch."""

    def __init__(self, items, device):
        """items: list of (partials tensor [splits*n], out tensor [n], splits)."""
        segs = np.zeros(len(items), dtype=TC_REDUCE_SEG)
        for i, (part, out, splits) in enumerate(items):
            segs[i] = (part.data_ptr(), out.data_ptr(), out.numel(), splits, 0)
        self.keep = items
        self.work = flat_works([o.numel() for _, o, _ in items], 1 << 14)
        self.segs_dev = torch.from_numpy(segs.view(np.uint8)).to(device)
        self.work_dev = torch.from_numpy(self.work.view(np.uint8)).to(device)

    def reduce(self):
        _lib.check(_lib.load().pf_conv2d_tc_wgrad_reduce_multi(_p(self.segs_dev), _p(self.work_dev), len(self.work),
                                                               _stream()), 'pf_conv2d_tc_wgrad_reduce_multi')


def conv2d_tc_wgrad_planes(d, xp, dyp, ws, dw):
    _lib.check(_lib.load().pf_conv2d_tc_wgrad_planes(ctypes.byref(d), _p(xp.hi), _p(xp.lo), _p(dyp.hi), _p(dyp.lo), _p(ws),
                                                     _p(dw), _stream()), 'pf_conv2d_tc_wgrad_planes')


# ---- TMA-fed kernels, operands as quantizer levels (include/pf_b200.h: pf_tc_act / pf_tc_wt)
ACT_HDR = np.dtype([('scale', np.float32), ('nplanes', np.int32)])


def conv2d_tc_set_feed(mode):
    """1: TMA kernels where eligible (default), 0: cp.async kernels everywhere, -1: PF_TC_FEED environment default."""
    _lib.check(_lib.load().pf_conv2d_tc_set_feed(int(mode)), 'pf_conv2d_tc_set_feed')


def conv2d_tc_tma_supported(d, which):
    """which: 0 fwd, 1 dgrad, 2 wgrad"""
    return bool(_lib.load().pf_conv2d_tc_tma_supported(ctypes.byref(d), int(which)))


def tc_act(planes, hdr=None, csum=None, nseg=0, single=False):
    """pf_tc_act of a Planes object (+ the producer's device header / channel sums); single: only plane0 is valid"""
    return _lib.TcAct(planes.hi.data_ptr(), 0 if single else planes.lo.data_ptr(), hdr.data_ptr() if hdr is not None else 0,
                      csum.data_ptr() if csum is not None else 0, int(nseg), 0)


def tc_wt(p0, p1=None, alpha=None, beta=None, per_channel=False, bits=0):
    return _lib.TcWt(p0.data_ptr(), p1.data_ptr() if p1 is not None else 0, alpha.data_ptr() if alpha is not None else 0,
                     beta.data_ptr() if beta is not None else 0, int(bool(per_channel)), int(bits))


def conv2d_tc_fwd_ex(d, act, wt, bias, relu, y, residual=None):
    _lib.check(_lib.load().pf_conv2d_tc_fwd_ex(ctypes.byref(d), ctypes.byref(act), ctypes.byref(wt), _p(bias), int(bool(relu)),
                                               _p(residual), _p(y), _stream()), 'pf_conv2d_tc_fwd_ex')


def conv2d_tc_dgrad_ex(d, act, wt, accumulate, dx):
    _lib.check(_lib.load().pf_conv2d_tc_dgrad_ex(ctypes.byref(d), ctypes.byref(act), ctypes.byref(wt), int(bool(accumulate)),
                                                 _p(dx), _stream()), 'pf_conv2d_tc_dgrad_ex')


def conv2d_tc_wgrad_ex(d, x_act, dy_act, ws, dw):
    _lib.check(_lib.load().pf_conv2d_tc_wgrad_ex(ctypes.byref(d), ctypes.byref(x_act), ctypes.byref(dy_act), _p(ws), _p(dw),
                                                 _stream()), 'pf_conv2d_tc_wgrad_ex')


def s2d_planes(x, pad_t, pad_l, hp, wp, cpad, planes):
    """space-to-depth of a stride-2 first layer's input [n,h,w,c] into operand planes [n,hp,wp,cpad]"""
    n, h, w, c = x.shape
    _lib.check(_lib.load().pf_s2d_planes(_p(x), n, h, w, c, int(pad_t), int(pad_l), int(hp), int(wp), int(cpad),
                                         _p(planes.hi), _p(planes.lo), _stream()), 'pf_s2d_planes')


def gather_rows(src, idx, dst, row_len):
    """dst[j] = src[idx[j]] (zero row where idx[j] < 0); rows of `row_len` floats"""
    _lib.check(_lib.load().pf_gather_rows(_p(src), _p(idx), idx.numel(), int(row_len), _p(dst), _stream()), 'pf_gather_rows')


def s2d_weight_maps(r, s, c, cpad):
    """Row maps between the HWIO kernel [r,s,c,K] of a stride-2 conv and its space-to-depth form [r2,s2,cpad,K]:
    fwd[j] = source row of s2d row j (-1: zero), bwd[i] = s2d row holding the gradient of source row i."""
    r2, s2 = (r + 1) // 2, (s + 1) // 2
    fwd = -np.ones(r2 * s2 * cpad, np.int32)
    bwd = np.zeros(r * s * c, np.int32)
    for rr in range(r):
        for ss in range(s):
            for cc in range(c):
                j = ((rr // 2) * s2 + (ss // 2)) * cpad + ((rr % 2) * 2 + (ss % 2)) * c + cc
                i = (rr * s + ss) * c + cc
                fwd[j], bwd[i] = i, j
    return r2, s2, fwd, bwd


def im2col_planes(d, x, kpad, planes):
    _lib.check(_lib.load().pf_im2col_planes(ctypes.byref(d), _p(x), int(kpad), _p(planes.hi), _p(planes.lo), _stream()),
               'pf_im2col_planes')


# ----------------------------------------------------------------------------- depthwise conv
def dwconv_fwd(d, x, w, y):
    _lib.check(_lib.load().pf_dwconv_fwd(ctypes.byref(d), _p(x), _p(w), _p(y), _stream()), 'pf_dwconv_fwd')


def dwconv_dgrad(d, dy, w, accumulate, dx):
    _lib.check(_lib.load().pf_dwconv_dgrad(ctypes.byref(d), _p(dy), _p(w), int(bool(accumulate)), _p(dx), _stream()),
               'pf_dwconv_dgrad')


def dwconv_wgrad_workspace_floats(d):
    return int(_lib.load().pf_dwconv_wgrad_workspace_bytes(ctypes.byref(d))) // 4


def dwconv_wgrad(d, x, dy, ws, dw):
    _lib.check(_lib.load().pf_dwconv_wgrad(ctypes.byref(d), _p(x), _p(dy), _p(ws), _p(dw), _stream()),
               'pf_dwconv_wgrad')


def preprocess_images(crops_u8, desc, out, mean=(123.68, 116.78, 103.94)):
    """ILSVRC-12 preprocessing of a packed mini-batch on the device (pf_preprocess_images): crops_u8 = uint8 CUDA buffer
    holding every decoded crop back to back, desc = uint8 CUDA view of n pf_img_desc records
    (datasets/ilsvrc12_dataset.py:IMG_DESC), out = fp32 [n, out_h, out_w, 3]."""
    L = _lib.load()
    _check_f32(out)
    if crops_u8.dtype != torch.uint8 or desc.dtype != torch.uint8 or not crops_u8.is_cuda or not desc.is_cuda:
        raise ValueError('expected uint8 CUDA buffers for the crops and the descriptor table')
    n, out_h, out_w, c = out.shape
    if c != 3 or desc.numel() != n * 40:
        raise ValueError('out must be [n, h, w, 3] with one 40-byte descriptor per image')
    _lib.check(L.pf_preprocess_images(_p(crops_u8), _p(desc), n, out_h, out_w, float(mean[0]), float(mean[1]),
                                      float(mean[2]), _p(out), _stream()), 'pf_preprocess_images')
    return out



# ----------------------------------------------------------------------------- f4 channel selection (pf_cpg.cu)
def cpg_diff_l2(a, b, diff, loss, partial_ws):
    """diff = a - b, loss[0] = sum(diff^2) / 2 — tf.nn.l2_loss of two conv outputs
    (learners/channel_pruning_gpu/learner.py:352); partial_ws: L2_PARTIALS floats."""
    _check_f32(a, b, diff, loss, partial_ws)
    if a.numel() != b.numel() or a.numel() != diff.numel():
        raise ValueError('cpg_diff_l2: size mismatch')
    _lib.check(_lib.load().pf_cpg_diff_l2(_p(a), _p(b), a.numel(), _p(diff), _p(loss), _p(partial_ws), _stream()),
               'pf_cpg_diff_l2')


def _rs_cin_cout(w):
    if w.dim() == 4:
        return w.shape[0] * w.shape[1], w.shape[2], w.shape[3]
    if w.dim() == 2:
        return 1, w.shape[0], w.shape[1]
    raise ValueError('kernel must be [R,S,Cin,Cout] or [Cin,Cout]')


def cpg_group_norms(w, g, lr, norms):
    """norms[c] = sqrt(sum_{r,s,k} (w - lr*g)^2) (learner.py:378-379); g None: norm of w itself (:256)."""
    _check_f32(w, g, norms)
    rs, cin, cout = _rs_cin_cout(w)
    _lib.check(_lib.load().pf_cpg_group_norms(_p(w), _p(g), float(lr), rs, cin, cout, _p(norms), _stream()),
               'pf_cpg_group_norms')


def cpg_prox_step(w, g, lr, prune_perctl, norms=None):
    """One proximal (group soft-threshold) step of the channel selection, in place on w (learner.py:375-383):
    w' = w - lr g ; n_c = ||w'[:, :, c, :]|| ; t = percentile(n, prune_perctl) ('nearest') ; w = w' max(1 - t/n_c, 0).
    Returns the threshold (device tensor [1])."""
    rs, cin, cout = _rs_cin_cout(w)
    if norms is None:
        norms = torch.empty(cin, dtype=torch.float32, device=w.device)
    lr = float(np.float32(lr))
    cpg_group_norms(w, g, lr, norms)
    # the percentile is fed through a float32 placeholder (learner.py:365) and widened to double by percentile()
    thr = select_desc([norms], [(0, percentile_rank_desc(cin, np.float32(prune_perctl)))])
    _lib.check(_lib.load().pf_cpg_prox_apply(_p(w), _p(g), float(lr), _p(norms), _p(thr), rs, cin, cout, _stream()),
               'pf_cpg_prox_apply')
    return thr


def cpg_channel_mask(w, mask, norms=None):
    """mask = tile(||w[:, :, c, :]|| > 0) (learner.py:256-259)."""
    _check_f32(w, mask)
    rs, cin, cout = _rs_cin_cout(w)
    if norms is None:
        norms = torch.empty(cin, dtype=torch.float32, device=w.device)
    cpg_group_norms(w, None, 0.0, norms)
    _lib.check(_lib.load().pf_cpg_channel_mask(_p(norms), rs, cin, cout, _p(mask), _stream()), 'pf_cpg_channel_mask')
    return norms


def mul(a, b, out):
    _check_f32(a, b, out)
    _lib.check(_lib.load().pf_mul(_p(a), _p(b), a.numel(), _p(out), _stream()), 'pf_mul')
