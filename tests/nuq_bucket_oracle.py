"""CPU oracle of the bucketed codebook quantizer (--nuql_use_buckets): NonUniformQuantization.__bucket_quantize with
__split_bucket / __channel_bucket, __scale, __quantile_init(axis=0), __build_bucket_norm_quant_point, __inv_scale
(the reference's learners/nonuniform_quantization/utils.py:196-243, 309-366, 388-476), restated on the building blocks
of oracle/pf_oracle.py, plus the torch-autograd form the step oracle uses for it.

TEST INFRASTRUCTURE ONLY, like oracle/: imported by tests and tools, never by pocketflow_b200.  Its numpy restatement is
pinned bit-for-bit against the reference's own __bucket_quantize, executed on numpy-backed stub tensors
(tests/golden/make_golden_nuq_bucket.py -> tests/golden/ref_executed_nuq_bucket_v1.json)."""
import numpy as np
import torch

from oracle import pf_oracle as O

F32 = np.float32


def bucket_view(x, bucket_type, bucket_size):
    """[rows, ncols] view, ncols and the number of padding copies (__split_bucket / __channel_bucket)."""
    if bucket_type == 'split':
        return O.split_bucket(x, bucket_size)
    if bucket_type == 'channel':
        return O.channel_bucket(x)
    raise ValueError("Unrecognized bucket type, must be 'weight' or 'channel'.")


def nonuniform_bucket_quantize(x, bits, bucket_type, bucket_size, clusters=None):
    """__bucket_quantize, 'weight' mode.  Returns (qx with x's shape, clusters [k, ncols], idx [rows, ncols], alpha
    [ncols], beta [ncols]).  clusters: the codebook table (its first 2^bits rows are used), quantile-initialised when
    None.  Ties: argmin takes the first centroid (tf.argmin)."""
    x = np.ascontiguousarray(x, dtype=F32)
    xb, ncols, padded = bucket_view(x, bucket_type, bucket_size)
    xn, alpha, beta = O.uq_scale(xb, 0)
    k = int(2 ** bits)
    if clusters is None:
        clusters = O.nuq_quantile_init(xn, k, axis=0)                      # [k, ncols]
    c = np.asarray(clusters, F32)[:k]
    d = np.abs((xn[:, None, :] - c[None, :, :]).astype(F32))            # [rows, k, ncols]
    idx = np.argmin(d, axis=1)
    q = (c[idx, np.arange(ncols)[None, :]] * np.sign((xn + F32(1e-6)).astype(F32))).astype(F32)
    qx = O.uq_inv_scale(q, alpha, beta).reshape(-1)
    if padded:
        qx = qx[:-padded]
    return qx.reshape(x.shape), np.asarray(clusters, F32), idx, alpha, beta


def nuq_bucket_grads(g, idx, k, alpha, bucket_type, bucket_size):
    """STE of the bucketed quantizer (utils.py:345-346, Mul->Add, Sign->Identity) for the gradient g w.r.t. the
    quantized weight: d/dc[j, b] = sum_{rows r with idx[r, b] = j} g_q[r, b], g_q = g * alpha_b; the padding copies are
    sliced off the output (:233-234) and receive no gradient.  Returns (g w.r.t. the weight, gc [k, ncols])."""
    g = np.ascontiguousarray(g, dtype=F32)
    gb, ncols, padded = bucket_view(g, bucket_type, bucket_size)
    gb = gb.copy()
    if padded:
        gb.reshape(-1)[-padded:] = 0
    gq = (gb * alpha).astype(F32)
    gx = (gq / alpha).astype(F32).reshape(-1)
    gc = np.zeros((k, ncols), dtype=np.float64)
    np.add.at(gc, (np.asarray(idx), np.broadcast_to(np.arange(ncols), idx.shape)), gq.astype(np.float64))
    return gx[:g.size].reshape(g.shape), gc.astype(F32)


def bucket_storage_bits(shapes, bucket_type, bucket_size):
    """__updt_bucket_storage (utils.py:487-494): 2 x 32 bits per bucket."""
    return sum(O.bucket_storage_bits(bucket_view(np.zeros(s, F32), bucket_type, bucket_size)[1]) for s in shapes)


def codebook_quant_bucketed(w, clusters, bucket_type, bucket_size):
    """torch autograd form of nonuniform_bucket_quantize for the step oracle, with the STE of the per-layer
    oracle.step_oracle.codebook_quant: the upstream gradient reaches both the gathered centroid (a segment sum into
    its bucket's codebook) and, through Sign-as-Identity, x_n.  All rows of `clusters` are centroids."""
    shape = w.shape
    n = w.numel()
    if bucket_type == 'channel':
        xb = w.reshape(-1, shape[-1])
    else:
        flat = w.reshape(-1)
        rest = n % bucket_size
        if rest:
            flat = torch.cat([flat, torch.ones(bucket_size - rest) * flat[-1]])
        xb = flat.reshape(bucket_size, -1)
    with torch.no_grad():
        w_max, w_min = xb.max(dim=0).values, xb.min(dim=0).values
    alpha = w_max - w_min + torch.tensor(1e-10)
    beta = w_min
    xn = (xb - beta) / alpha
    c = clusters if torch.is_tensor(clusters) else torch.as_tensor(clusters, dtype=torch.float32)
    with torch.no_grad():
        idx = torch.argmin(torch.abs(xn.unsqueeze(1) - c.unsqueeze(0)), dim=1)
        sgn = torch.sign(xn + 1e-6)
    q = c.gather(0, idx) * sgn + (xn - xn.detach())
    return (alpha * q + beta).reshape(-1)[:n].reshape(shape)
