// pf_nuq.cu — codebook (non-uniform) weight quantization, multi-tensor.
//
// Replaces NonUniformQuantization.__nonuni_quantize / __build_norm_quant_point
// (/root/reference/learners/nonuniform_quantization/utils.py:168-194, 284-307), which materialises
// tile(x, [...,2^b]) (a x16 temporary at 4 bits: 1.5 GB on ResNet-50), abs(sub), argmin, gather,
// mul(sign) and the inverse scale as separate TF kernels.  Here the codebook of a tensor sits in
// shared memory and the nearest-centroid search runs in registers: 8 B/element of HBM traffic
// (+1 B/element when the centroid index is kept for the codebook gradient).
#include "pf_common.cuh"

namespace {
constexpr int kThreads = 256;

// c: centroid j at c[j * cs] (cs = 1 for a per-layer codebook, the tile width for a slice of per-bucket codebooks)
__device__ __forceinline__ float nuq_one(float w, float alpha, float beta, float ralpha,
                                         const float* __restrict__ c, int nc, uint8_t* idx_out, int cs = 1) {
  const float xn = pf_div_r(__fsub_rn(w, beta), alpha, ralpha);
  float best = fabsf(__fsub_rn(xn, c[0]));
  int bi = 0;
  for (int j = 1; j < nc; ++j) {
    const float d = fabsf(__fsub_rn(xn, c[j * cs]));
    if (d < best) {  // strict: first index wins on ties (tf.argmin)
      best = d;
      bi = j;
    }
  }
  if (idx_out) *idx_out = (uint8_t)bi;
  const float t = __fadd_rn(xn, 1e-6f);
  const float sgn = t > 0.f ? 1.f : (t < 0.f ? -1.f : 0.f);
  return __fadd_rn(__fmul_rn(alpha, __fmul_rn(c[bi * cs], sgn)), beta);
}

__global__ void __launch_bounds__(kThreads)
nuq_quant_kernel(const pf_uq_seg* __restrict__ segs, const pf_work* __restrict__ work,
                 const float* __restrict__ scales, int n_buckets,
                 const float* __restrict__ clusters, const int64_t* __restrict__ cluster_off,
                 uint8_t* __restrict__ idx_out, const int64_t* __restrict__ idx_base) {
  __shared__ float sc[256];
  const pf_work w = work[blockIdx.x];
  const pf_uq_seg s = segs[w.seg];
  const int nc = 1 << s.bits;
  // the codebook of this tensor: at cluster_off[seg] floats from `clusters` (codebooks that live among the model's
  // trainable variables), or at seg * 256 (a [segments, 256] table)
  const float* cb = clusters + (cluster_off ? (size_t)cluster_off[w.seg] : (size_t)w.seg * 256);
  if ((int)threadIdx.x < nc) sc[threadIdx.x] = cb[threadIdx.x];
  __syncthreads();
  const float alpha = __ldg(scales + s.bucket0), mn = __ldg(scales + n_buckets + s.bucket0);
  const float ra = __ldg(scales + 2 * n_buckets + s.bucket0);
  uint8_t* io = idx_out ? idx_out + idx_base[w.seg] : nullptr;
  const int64_t end = w.start + w.count;
  for (int64_t i = w.start + (int64_t)threadIdx.x * 4; i < end; i += kThreads * 4) {
    if (i + 3 < end) {
      float4 v = pf_ld4(s.src + i);
      uint8_t id[4];
      v.x = nuq_one(v.x, alpha, mn, ra, sc, nc, io ? &id[0] : nullptr);
      v.y = nuq_one(v.y, alpha, mn, ra, sc, nc, io ? &id[1] : nullptr);
      v.z = nuq_one(v.z, alpha, mn, ra, sc, nc, io ? &id[2] : nullptr);
      v.w = nuq_one(v.w, alpha, mn, ra, sc, nc, io ? &id[3] : nullptr);
      pf_st_stream(s.dst + i, v);
      if (io) *reinterpret_cast<uchar4*>(io + i) = make_uchar4(id[0], id[1], id[2], id[3]);
    } else {
      for (int64_t j = i; j < end; ++j) s.dst[j] = nuq_one(s.src[j], alpha, mn, ra, sc, nc, io ? io + j : nullptr);
    }
  }
}

// ---- codebook gradient (cluster / both optimisation modes): the gather's backward is a segment sum,
//   dL/dc_j = alpha * sum_{i: idx_i = j} g_i        (g = dL/d(quantized weight); inverse scale alpha*q + beta)
// Deterministic two-stage reduction: every CTA sums its chunk per centroid in registers (16 centroids per pass, the
// chunk is re-read from L2 for codebooks with more), block-reduces, and writes partial[work][j]; the final kernel adds
// the partials of a tensor in work order and applies alpha.
constexpr int kNcPass = 16;

__global__ void __launch_bounds__(kThreads)
nuq_cluster_grad_partial_kernel(const pf_uq_seg* __restrict__ segs, const pf_work* __restrict__ work,
                                const uint8_t* __restrict__ idx, const int64_t* __restrict__ idx_base,
                                float* __restrict__ partial) {
  __shared__ float sh[kThreads / 32][kNcPass];
  const pf_work w = work[blockIdx.x];
  const pf_uq_seg s = segs[w.seg];
  const int nc = 1 << s.bits;
  const uint8_t* io = idx + idx_base[w.seg];
  const float* g = s.src;                       // the gradient w.r.t. the quantized tensor
  const int64_t end = w.start + w.count;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int j0 = 0; j0 < nc; j0 += kNcPass) {
    float acc[kNcPass];
#pragma unroll
    for (int j = 0; j < kNcPass; ++j) acc[j] = 0.f;
    for (int64_t i = w.start + threadIdx.x; i < end; i += kThreads) {
      const int id = (int)io[i] - j0;
      const float gv = g[i];
#pragma unroll
      for (int j = 0; j < kNcPass; ++j) acc[j] += (id == j) ? gv : 0.f;
    }
#pragma unroll
    for (int j = 0; j < kNcPass; ++j) {
      const float t = pf_warp_sum(acc[j]);
      if (lane == 0) sh[warp][j] = t;
    }
    __syncthreads();
    if (threadIdx.x < kNcPass && j0 + (int)threadIdx.x < nc) {
      float t = 0.f;
#pragma unroll
      for (int wv = 0; wv < kThreads / 32; ++wv) t += sh[wv][threadIdx.x];
      partial[(size_t)blockIdx.x * 256 + j0 + threadIdx.x] = t;
    }
    __syncthreads();
  }
}

// one CTA per tensor: sum the partials of its work items (a contiguous range of the work table) in order
__global__ void __launch_bounds__(256)
nuq_cluster_grad_final_kernel(const pf_uq_seg* __restrict__ segs, const int32_t* __restrict__ work_first,
                              const float* __restrict__ partial, const float* __restrict__ scales,
                              float* __restrict__ grad_base, const int64_t* __restrict__ cluster_off) {
  const int seg = blockIdx.x;
  const pf_uq_seg s = segs[seg];
  const int nc = 1 << s.bits;
  const int j = threadIdx.x;
  if (j >= nc) return;
  float t = 0.f;
  for (int wi = work_first[seg]; wi < work_first[seg + 1]; ++wi) t += partial[(size_t)wi * 256 + j];
  grad_base[cluster_off[seg] + j] = __fmul_rn(t, __ldg(scales + s.bucket0));     // * alpha
}

// ---- bucketed codebooks (__bucket_quantize, utils.py:196-243, 309-347): one codebook per bucket = per column of the
// [padded/ncols, ncols] view, stored as the [2^bits, ncols] row-major `clusters` variable (centroid j of bucket b at
// base + off[seg] + j*ncols + b).  Work items are kind-1 column tiles; a CTA stages its tile's codebook slice and
// scales in shared memory, reads rows as contiguous runs of ncol_tile floats, and never writes the padding.
constexpr int kBucketSmemFloats = PF_NUQ_BUCKET_TILE_FLOATS + 3 * PF_NUQ_BUCKET_MAX_TILE;

__global__ void __launch_bounds__(kThreads)
nuq_bucket_quant_kernel(const pf_uq_seg* __restrict__ segs, const pf_work* __restrict__ work,
                        const float* __restrict__ scales, int n_buckets, const float* __restrict__ cbase,
                        const int64_t* __restrict__ cluster_off, uint8_t* __restrict__ idx_out,
                        const int64_t* __restrict__ idx_base) {
  extern __shared__ float smem[];
  const pf_work w = work[blockIdx.x];
  const pf_uq_seg s = segs[w.seg];
  const int nc = 1 << s.bits, tc = w.ncol_tile;
  float* sc = smem;                 // [nc][tc]
  float* sa = smem + nc * tc;       // alpha, beta, RN(1/alpha) of the tile's buckets
  float* sb = sa + tc;
  float* sr = sb + tc;
  const float* cb = cbase + cluster_off[w.seg] + w.c0;
  for (int e = threadIdx.x; e < nc * tc; e += kThreads) {
    const int j = e / tc;
    sc[e] = __ldg(cb + (int64_t)j * s.ncols + (e - j * tc));
  }
  for (int c = threadIdx.x; c < tc; c += kThreads) {
    const int b = s.bucket0 + w.c0 + c;
    sa[c] = __ldg(scales + b);
    sb[c] = __ldg(scales + n_buckets + b);
    sr[c] = __ldg(scales + 2 * n_buckets + b);
  }
  __syncthreads();
  uint8_t* io = idx_out ? idx_out + idx_base[w.seg] : nullptr;
  const int n = w.count * tc;
  for (int e = threadIdx.x; e < n; e += kThreads) {
    const int rr = e / tc, c = e - rr * tc;
    const int64_t i = (w.start + rr) * (int64_t)s.ncols + w.c0 + c;
    if (i >= s.numel) break;        // i grows with e: the rest of this thread's elements are padding too
    s.dst[i] = nuq_one(s.src[i], sa[c], sb[c], sr[c], sc + c, nc, io ? io + i : nullptr, tc);
  }
}

// one CTA per bucket slot: gather the column (padding rows read as src[numel-1]), bitonic-sort its ordered-uint keys
// ascending in shared memory, pick the descending ranks of the 2^bits percentiles and normalise them with the fp32
// chain of the forward (x -> x_n is monotone non-decreasing, so the order statistic of w is that of x_n)
__global__ void __launch_bounds__(kThreads)
nuq_bucket_quantile_kernel(const pf_uq_seg* __restrict__ segs, int n_seg, const float* __restrict__ scales,
                           int n_buckets, const int32_t* __restrict__ ranks, float* __restrict__ cbase,
                           const int64_t* __restrict__ cluster_off) {
  extern __shared__ uint32_t keys[];
  const int g = blockIdx.x;
  int lo = 0, hi = n_seg - 1;       // last tensor whose first slot is <= g
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (segs[mid].bucket0 <= g) lo = mid; else hi = mid - 1;
  }
  const pf_uq_seg s = segs[lo];
  const int b = g - s.bucket0;
  if (b < 0 || b >= s.ncols) return;    // alignment slot between two tensors
  const int rows = (int)(s.padded / s.ncols);
  int P = 1;
  while (P < rows) P <<= 1;
  for (int r = threadIdx.x; r < P; r += kThreads) {
    uint32_t k = 0xFFFFFFFFu;           // sorts behind every real key
    if (r < rows) {
      const int64_t i = (int64_t)r * s.ncols + b;
      k = pf_enc(__ldg(s.src + (i < s.numel ? i : s.numel - 1)));
    }
    keys[r] = k;
  }
  __syncthreads();
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int t = threadIdx.x; t < (P >> 1); t += kThreads) {
        const int a = ((t & ~(j - 1)) << 1) | (t & (j - 1));
        const uint32_t x = keys[a], y = keys[a + j];
        if ((x > y) == ((a & k) == 0)) {
          keys[a] = y;
          keys[a + j] = x;
        }
      }
      __syncthreads();
    }
  }
  const int nc = 1 << s.bits;
  const float alpha = __ldg(scales + s.bucket0 + b), beta = __ldg(scales + n_buckets + s.bucket0 + b);
  const float ra = __ldg(scales + 2 * n_buckets + s.bucket0 + b);
  for (int j = threadIdx.x; j < nc; j += kThreads) {
    const float v = pf_dec(keys[rows - 1 - ranks[lo * 256 + j]]);
    cbase[cluster_off[lo] + (int64_t)j * s.ncols + b] = pf_div_r(__fsub_rn(v, beta), alpha, ra);
  }
}

// codebook gradient per bucket, dL/dc[j,b] = alpha_b * sum_{r < valid rows, idx[r,b] = j} g[r,b].  Stage 1: a work item
// = PF_NUQ_BUCKET_GRAD_TILE columns x a row range; thread (column, row group) sums 16 centroids per pass in registers,
// the row groups are added in fixed order -> partial[work][kmax][tile].  Stage 2: one CTA per column tile adds the
// partials of its row ranges (contiguous work items) in order and applies alpha.
constexpr int kGradTile = PF_NUQ_BUCKET_GRAD_TILE;
constexpr int kGradGroups = kThreads / kGradTile;

__global__ void __launch_bounds__(kThreads)
nuq_bucket_grad_partial_kernel(const pf_uq_seg* __restrict__ gsegs, const pf_work* __restrict__ work,
                               const uint8_t* __restrict__ idx, const int64_t* __restrict__ idx_base, int kmax,
                               float* __restrict__ partial) {
  __shared__ float sh[kGradGroups][kNcPass][kGradTile];
  const pf_work w = work[blockIdx.x];
  const pf_uq_seg s = gsegs[w.seg];
  const int nc = 1 << s.bits;
  const uint8_t* io = idx + idx_base[w.seg];
  const int c = threadIdx.x % kGradTile, rg = threadIdx.x / kGradTile;
  const int64_t rend = w.start + w.count;
  for (int j0 = 0; j0 < nc; j0 += kNcPass) {
    float acc[kNcPass];
#pragma unroll
    for (int j = 0; j < kNcPass; ++j) acc[j] = 0.f;
    if (c < w.ncol_tile) {
      for (int64_t r = w.start + rg; r < rend; r += kGradGroups) {
        const int64_t i = r * s.ncols + w.c0 + c;
        if (i >= s.numel) break;        // padding rows carry no gradient
        const int id = (int)io[i] - j0;
        const float gv = s.src[i];
#pragma unroll
        for (int j = 0; j < kNcPass; ++j) acc[j] += (id == j) ? gv : 0.f;
      }
    }
#pragma unroll
    for (int j = 0; j < kNcPass; ++j) sh[rg][j][c] = acc[j];
    __syncthreads();
    for (int e = threadIdx.x; e < kNcPass * kGradTile; e += kThreads) {
      const int j = e / kGradTile, cc = e % kGradTile;
      if (j0 + j < nc && cc < w.ncol_tile) {
        float t = 0.f;
#pragma unroll
        for (int q = 0; q < kGradGroups; ++q) t += sh[q][j][cc];
        partial[((size_t)blockIdx.x * kmax + j0 + j) * kGradTile + cc] = t;
      }
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kThreads)
nuq_bucket_grad_final_kernel(const pf_uq_seg* __restrict__ segs, const pf_work* __restrict__ tiles,
                             const float* __restrict__ partial, int kmax, const float* __restrict__ scales,
                             float* __restrict__ grad_base, const int64_t* __restrict__ cluster_off) {
  const pf_work t = tiles[blockIdx.x];    // start/count: its row-range work items
  const pf_uq_seg s = segs[t.seg];
  const int nc = 1 << s.bits;
  for (int e = threadIdx.x; e < nc * kGradTile; e += kThreads) {
    const int j = e / kGradTile, c = e % kGradTile;
    if (c >= t.ncol_tile) continue;
    float acc = 0.f;
    for (int64_t wi = t.start; wi < t.start + t.count; ++wi) acc += partial[((size_t)wi * kmax + j) * kGradTile + c];
    grad_base[cluster_off[t.seg] + (int64_t)j * s.ncols + t.c0 + c] =
        __fmul_rn(acc, __ldg(scales + s.bucket0 + t.c0 + c));     // * alpha_b
  }
}
}  // namespace

extern "C" {

int pf_nuq_weight_quant(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                        const float* scales_dev, int n_buckets,
                        const float* clusters_dev, uint8_t* idx_out_dev,
                        const int64_t* idx_base_dev, void* stream) {
  PF_REQUIRE(n_work >= 0, "pf_nuq_weight_quant: n_work < 0");
  if (n_work == 0) return PF_OK;
  PF_REQUIRE(segs_dev && work_dev && scales_dev && clusters_dev,
             "pf_nuq_weight_quant: null pointer");
  PF_REQUIRE((idx_out_dev == nullptr) == (idx_base_dev == nullptr),
             "pf_nuq_weight_quant: idx_out and idx_base must be given together");
  nuq_quant_kernel<<<n_work, kThreads, 0, (cudaStream_t)stream>>>(
      segs_dev, work_dev, scales_dev, n_buckets, clusters_dev, nullptr, idx_out_dev, idx_base_dev);
  PF_CHECK_LAUNCH("pf_nuq_weight_quant");
  return PF_OK;
}

int pf_nuq_weight_quant_ex(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                           const float* scales_dev, int n_buckets, const float* clusters_base_dev,
                           const int64_t* cluster_off_dev, uint8_t* idx_out_dev, const int64_t* idx_base_dev,
                           void* stream) {
  PF_REQUIRE(n_work >= 0, "pf_nuq_weight_quant_ex: n_work < 0");
  if (n_work == 0) return PF_OK;
  PF_REQUIRE(segs_dev && work_dev && scales_dev && clusters_base_dev && cluster_off_dev,
             "pf_nuq_weight_quant_ex: null pointer");
  PF_REQUIRE((idx_out_dev == nullptr) == (idx_base_dev == nullptr),
             "pf_nuq_weight_quant_ex: idx_out and idx_base must be given together");
  nuq_quant_kernel<<<n_work, kThreads, 0, (cudaStream_t)stream>>>(
      segs_dev, work_dev, scales_dev, n_buckets, clusters_base_dev, cluster_off_dev, idx_out_dev, idx_base_dev);
  PF_CHECK_LAUNCH("pf_nuq_weight_quant_ex");
  return PF_OK;
}

int pf_nuq_cluster_grad(const pf_uq_seg* gsegs_dev, int n_seg, const pf_work* work_dev, int n_work,
                        const int32_t* work_first_dev, const uint8_t* idx_dev, const int64_t* idx_base_dev,
                        const float* scales_dev, float* partial_ws_dev, float* grad_base_dev,
                        const int64_t* cluster_off_dev, void* stream) {
  PF_REQUIRE(n_seg >= 0 && n_work >= 0, "pf_nuq_cluster_grad: negative count");
  if (n_seg == 0 || n_work == 0) return PF_OK;
  PF_REQUIRE(gsegs_dev && work_dev && work_first_dev && idx_dev && idx_base_dev && scales_dev && partial_ws_dev &&
                 grad_base_dev && cluster_off_dev, "pf_nuq_cluster_grad: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  nuq_cluster_grad_partial_kernel<<<n_work, kThreads, 0, st>>>(gsegs_dev, work_dev, idx_dev, idx_base_dev, partial_ws_dev);
  PF_CHECK_LAUNCH("pf_nuq_cluster_grad(partial)");
  nuq_cluster_grad_final_kernel<<<n_seg, 256, 0, st>>>(gsegs_dev, work_first_dev, partial_ws_dev, scales_dev, grad_base_dev,
                                                      cluster_off_dev);
  PF_CHECK_LAUNCH("pf_nuq_cluster_grad(final)");
  return PF_OK;
}

int pf_nuq_bucket_weight_quant(const pf_uq_seg* segs_dev, const pf_work* work_dev, int n_work,
                               const float* scales_dev, int n_buckets, const float* clusters_base_dev,
                               const int64_t* cluster_off_dev, uint8_t* idx_out_dev, const int64_t* idx_base_dev,
                               void* stream) {
  PF_REQUIRE(n_work >= 0, "pf_nuq_bucket_weight_quant: n_work < 0");
  if (n_work == 0) return PF_OK;
  PF_REQUIRE(segs_dev && work_dev && scales_dev && clusters_base_dev && cluster_off_dev,
             "pf_nuq_bucket_weight_quant: null pointer");
  PF_REQUIRE((idx_out_dev == nullptr) == (idx_base_dev == nullptr),
             "pf_nuq_bucket_weight_quant: idx_out and idx_base must be given together");
  nuq_bucket_quant_kernel<<<n_work, kThreads, kBucketSmemFloats * sizeof(float), (cudaStream_t)stream>>>(
      segs_dev, work_dev, scales_dev, n_buckets, clusters_base_dev, cluster_off_dev, idx_out_dev, idx_base_dev);
  PF_CHECK_LAUNCH("pf_nuq_bucket_weight_quant");
  return PF_OK;
}

int pf_nuq_bucket_quantile_init(const pf_uq_seg* segs_dev, int n_seg, const float* scales_dev, int n_buckets,
                                const int32_t* ranks_dev, int max_rows, float* clusters_base_dev,
                                const int64_t* cluster_off_dev, void* stream) {
  PF_REQUIRE(n_seg >= 0 && n_buckets >= 0, "pf_nuq_bucket_quantile_init: negative count");
  if (n_seg == 0 || n_buckets == 0) return PF_OK;
  PF_REQUIRE(segs_dev && scales_dev && ranks_dev && clusters_base_dev && cluster_off_dev,
             "pf_nuq_bucket_quantile_init: null pointer");
  PF_REQUIRE(max_rows >= 1 && max_rows <= PF_NUQ_BUCKET_MAX_ROWS,
             "pf_nuq_bucket_quantile_init: buckets of %d rows (at most %d)", max_rows, PF_NUQ_BUCKET_MAX_ROWS);
  int P = 1;
  while (P < max_rows) P <<= 1;
  const size_t smem = (size_t)P * sizeof(uint32_t);
  PF_CUDA(cudaFuncSetAttribute(nuq_bucket_quantile_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nuq_bucket_quantile_kernel<<<n_buckets, kThreads, smem, (cudaStream_t)stream>>>(
      segs_dev, n_seg, scales_dev, n_buckets, ranks_dev, clusters_base_dev, cluster_off_dev);
  PF_CHECK_LAUNCH("pf_nuq_bucket_quantile_init");
  return PF_OK;
}

int pf_nuq_bucket_cluster_grad(const pf_uq_seg* gsegs_dev, const pf_work* work_dev, int n_work,
                               const pf_work* tiles_dev, int n_tiles, int kmax, const uint8_t* idx_dev,
                               const int64_t* idx_base_dev, const float* scales_dev, float* partial_ws_dev,
                               float* grad_base_dev, const int64_t* cluster_off_dev, void* stream) {
  PF_REQUIRE(n_work >= 0 && n_tiles >= 0, "pf_nuq_bucket_cluster_grad: negative count");
  if (n_work == 0 || n_tiles == 0) return PF_OK;
  PF_REQUIRE(kmax >= 1 && kmax <= 256, "pf_nuq_bucket_cluster_grad: kmax must be in [1, 256]");
  PF_REQUIRE(gsegs_dev && work_dev && tiles_dev && idx_dev && idx_base_dev && scales_dev && partial_ws_dev &&
                 grad_base_dev && cluster_off_dev, "pf_nuq_bucket_cluster_grad: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  nuq_bucket_grad_partial_kernel<<<n_work, kThreads, 0, st>>>(gsegs_dev, work_dev, idx_dev, idx_base_dev, kmax,
                                                              partial_ws_dev);
  PF_CHECK_LAUNCH("pf_nuq_bucket_cluster_grad(partial)");
  nuq_bucket_grad_final_kernel<<<n_tiles, kThreads, 0, st>>>(gsegs_dev, tiles_dev, partial_ws_dev, kmax, scales_dev,
                                                             grad_base_dev, cluster_off_dev);
  PF_CHECK_LAUNCH("pf_nuq_bucket_cluster_grad(final)");
  return PF_OK;
}

}  // extern "C"
