// Element-wise training stages of the U-Net family directly on the 16-bit CP8 planes the tensor-core convolutions read and write
// (bf16 training mode; reference modules: libdl/nn_models/unet_cnns.py:30-104):
//   double_conv:  y = Conv2d(x)  ->  BatchNorm2d (train mode: batch mean / biased variance, running statistics updated)  ->  ReLU
//                 forward   stats = (mean, var) of y per channel;  a = max(0, (y - mean) * rstd * gamma + beta)
//                 backward  g' = g * [a > 0];  s1 = sum g', s2 = sum g' * xhat;  dy = gamma * rstd * (g' - s1/N - xhat * s2/N)
//                           d gamma = s2, d beta = s1, d conv-bias = sum dy
//   MaxPool2d(2) backward (gradient to the first maximum of the window in row-major order, ATen semantics) with the skip connection's
//                 gradient added in the same pass
//   nn.Upsample(x2, bilinear, align_corners=True) + pad backward (the adjoint of mpa_upsample2x_cp8)
// so that between two convolutions of a training step no nchw<->CP8 converter and no fp32 NCHW tensor exists (before: cp8_to_nchw ->
// bn_stats -> bn_apply -> nchw_to_cp8 forward, cp8_to_nchw -> two reductions -> bn_bwd_apply -> nchw_to_cp8 backward, 11 + 9 launches per
// convolution, 2 x 4 bytes per element and direction instead of 2).  All sums are formed in fp32; the per-channel reductions run on a
// (chunk, slice) grid with an ordered merge (bit-reproducible), only the (mathematically zero) conv-bias gradient meets in atomics.
// Eval-mode backward (BatchNorm frozen at its running statistics) has its own one-pass kernel below: dy = gamma * rstd * g'.
#include "common.cuh"
#include "cp8.cuh"

namespace mpa {

constexpr int kUT = 256;          // threads per block of every kernel here

// 4 MB of partial sums per device + (in front of them) the arrival counter of the "last block finishes the reduction" pattern: the block
// (one per chunk plane, <= 64 chunks = 512 channels) of the "last block finishes the reduction" pattern: the slice block of a chunk that
// arrives last merges that chunk's partials (one warp per channel) and resets the counter, so a per-channel reduction is ONE launch (the
// separate final kernels were 36 launches of ~5 us per SAUnet:L training step).  Kernels of one stream run in order: one set is enough.
static float* unet_scratch() {
  static float* ptr[64] = {nullptr};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (!ptr[dev]) {
    float* p = nullptr;
    if (cudaMalloc(&p, sizeof(float) * ((1u << 20) + 64)) != cudaSuccess) return nullptr;
    if (cudaMemset(p, 0, sizeof(float) * 64) != cudaSuccess) return nullptr;
    ptr[dev] = p;
  }
  return ptr[dev] + 64;
}
// counter: one per chunk plane (blockIdx.x); the last of the gridDim.y slice blocks of a chunk finishes that chunk's channels
__device__ __forceinline__ bool last_block_done(unsigned* counter) {
  __shared__ bool last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) last = atomicAdd(counter, 1u) == gridDim.y - 1;
  __syncthreads();
  if (last) __threadfence();
  return last;
}

// v[e] <- sum over the block of v[e], e < N (every thread gets the result); sh: kUT/32 * N floats
template <int N>
__device__ __forceinline__ void block_sum_n(float (&v)[N], float* sh) {
#pragma unroll
  for (int e = 0; e < N; ++e) v[e] = warp_sum(v[e]);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) {
#pragma unroll
    for (int e = 0; e < N; ++e) sh[(threadIdx.x >> 5) * N + e] = v[e];
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < N; ++e) {
    float r = 0.f;
#pragma unroll
    for (int w = 0; w < kUT / 32; ++w) r += sh[w * N + e];
    v[e] = r;
  }
}

// pixel i of the flattened (b, t, f) index -> 16-byte offset inside a CP8 buffer with `ncs` chunk planes per item
struct Cp8Geo {
  int T, F, TP, P, pf, pt;
  __device__ __forceinline__ size_t at(unsigned i, int ncs, int ck) const {
    const unsigned row = i / (unsigned)F, f = i - row * (unsigned)F;
    const unsigned b = row / (unsigned)T, t = row - b * (unsigned)T;
    return (((size_t)b * ncs + ck) * TP + pt + t) * P + pf + f;
  }
  // the same pixel in phase-split planes (s phase sets of NCk chunk planes per item, pitch P2): bin f -> phase f % s, column f / s
  __device__ __forceinline__ size_t at_split(unsigned i, int NCk, int ck, int s, int P2) const {
    const unsigned row = i / (unsigned)F, f = i - row * (unsigned)F;
    const unsigned b = row / (unsigned)T, t = row - b * (unsigned)T;
    return ((((size_t)b * s + f % s) * NCk + ck) * TP + pt + t) * P2 + pf + f / s;
  }
};

__device__ __forceinline__ float bn_val(float y, float mean, float rstd, float w, float b) { return (y - mean) * rstd * w + b; }

__device__ __forceinline__ void chan_merge(float& n, float& mean, float& m2, float ns, float ms, float qs) {
  if (ns <= 0.f) return;
  const float nn = n + ns, delta = ms - mean;
  mean += delta * (ns / nn);
  m2 += qs + delta * delta * (n * ns / nn);
  n = nn;
}
struct BnStatsFinal {
  const float* pivot;      // [C] or null: per-channel offset subtracted before summing (the producing convolution's bias)
  float* stats;            // [2C] mean | biased variance
  float *run_mean, *run_var;
  float momentum;
  long long* nbt;
};
// one warp per channel: lane l merges slices l, l+32, ... in order, the 32 lane results are merged by a shuffle tree (fixed order).
// Also the running-statistics update of nn.BatchNorm2d (momentum m; unbiased variance).
__device__ __forceinline__ void bn_stats_merge(const float* __restrict__ partial, float* __restrict__ stats, unsigned n_tot, int C, int S, int c,
                                               float* __restrict__ run_mean, float* __restrict__ run_var, float momentum) {
  const int lane = threadIdx.x & 31;
  float n = 0.f, mean = 0.f, m2 = 0.f;
  float2 pv[16];                                   // S <= 512: all of this lane's slices are requested before the (dependent) merges
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int s = lane + 32 * i;
    pv[i] = s < S ? __ldcg(reinterpret_cast<const float2*>(partial) + (size_t)c * S + s) : make_float2(0.f, 0.f);   // L2: written by other CTAs
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int s = lane + 32 * i;
    if (s < S) {
      const float ns = (float)((unsigned)((unsigned long long)n_tot * (s + 1) / S) - (unsigned)((unsigned long long)n_tot * s / S));
      chan_merge(n, mean, m2, ns, pv[i].x, pv[i].y);
    }
  }
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const float n2 = __shfl_xor_sync(0xffffffffu, n, o), me2 = __shfl_xor_sync(0xffffffffu, mean, o), q2 = __shfl_xor_sync(0xffffffffu, m2, o);
    // both partners apply the same merge (lower lane's triple first), so all lanes agree
    float an = n, am = mean, aq = m2, bn = n2, bm = me2, bq = q2;
    if (lane & o) { an = n2; am = me2; aq = q2; bn = n; bm = mean; bq = m2; }
    chan_merge(an, am, aq, bn, bm, bq);
    n = an; mean = am; m2 = aq;
  }
  if (lane == 0) {
    const float var = m2 / (float)n_tot;
    stats[c] = mean;
    stats[C + c] = var;
    if (run_mean) {
      run_mean[c] = (1.f - momentum) * run_mean[c] + momentum * mean;
      run_var[c] = (1.f - momentum) * run_var[c] + momentum * (var * ((float)n_tot / fmaxf((float)n_tot - 1.f, 1.f)));
    }
  }
}

// ---- BatchNorm batch statistics -------------------------------------------------------------------------------------------------------
// grid (chunk, slice): per channel of the chunk the slice's mean and sum of squared deviations (two passes over the slice, the second one
// from L1/L2), merged in slice order by the final kernel with Chan's update
template <int FMT>
__global__ void __launch_bounds__(kUT) bn_stats_partial_cp8_kernel(const uint4* __restrict__ y, float* __restrict__ partial, unsigned n, Cp8Geo g,
                                                                   int ncs, int S, BnStatsFinal f) {
  const int ck = blockIdx.x, s = blockIdx.y;
  const unsigned i0 = (unsigned)((unsigned long long)n * s / S), i1 = (unsigned)((unsigned long long)n * (s + 1) / S);
  // ONE pass: sums of the deviations from a per-channel pivot (the convolution's bias: y - bias is the raw filter response, whose mean is
  // within a few standard deviations of zero) and of their squares; slice mean = pivot + sum d / n, slice M2 = sum d^2 - (sum d)^2 / n.
  // With ~2k values per slice the cancellation costs ~1e-7 * (mean_d / std)^2 of the variance; the slices are then merged with Chan's
  // update, which is robust.  (The two-pass form read every plane twice: 0.3 ms per SAUnet:L step.)
  float piv[8], a[16];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    piv[e] = f.pivot ? f.pivot[ck * 8 + e] : 0.f;
    a[e] = a[8 + e] = 0.f;
  }
  for (unsigned i = i0 + threadIdx.x; i < i1; i += kUT) {
    float v[8];
    unpack8<FMT>(y[g.at(i, ncs, ck)], v);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float d = v[e] - piv[e];
      a[e] += d;
      a[8 + e] = fmaf(d, d, a[8 + e]);
    }
  }
  __shared__ float sh16[kUT / 32 * 16];
  block_sum_n<16>(a, sh16);
  const float cnt = (float)(i1 - i0);
  float mean[8], q[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float md = cnt > 0.f ? a[e] / cnt : 0.f;
    mean[e] = piv[e] + md;
    q[e] = fmaxf(a[8 + e] - a[e] * md, 0.f);
  }
  if (threadIdx.x < 8) {
    const int e = threadIdx.x;
    partial[((size_t)(ck * 8 + e) * S + s) * 2] = mean[e];
    partial[((size_t)(ck * 8 + e) * S + s) * 2 + 1] = q[e];
  }
  unsigned* counter = reinterpret_cast<unsigned*>(partial) - 64 + ck;
  if (!last_block_done(counter)) return;
  bn_stats_merge(partial, f.stats, n, gridDim.x * 8, S, ck * 8 + (threadIdx.x >> 5), f.run_mean, f.run_var, f.momentum);     // 8 warps = 8 channels
  if (threadIdx.x == 0) {
    if (f.nbt && ck == 0) f.nbt[0] += 1;
    *counter = 0u;
  }
}

// ---- forward apply: a = relu(bn(y)) ---------------------------------------------------------------------------------------------------
// grid (pixel blocks of one item-chunk plane, B * NCk); 4 pixels per thread
template <int FMT>
__global__ void __launch_bounds__(kUT) bn_relu_apply_cp8_kernel(const uint4* __restrict__ y, uint4* __restrict__ out, const float* __restrict__ stats,
                                                                const float* __restrict__ w, const float* __restrict__ bias, float eps, int C, int NCk,
                                                                int T, int F, int TP, int P, int pf, int pt, int ncs_y, int ncs_out, int out_split,
                                                                int P2) {
  const int ck = blockIdx.y % NCk, b = blockIdx.y / NCk;
  float mean[8], rstd[8], wc[8], bc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = ck * 8 + e;
    mean[e] = stats[c];
    rstd[e] = rsqrtf(stats[C + c] + eps);
    wc[e] = w[c];
    bc[e] = bias[c];
  }
  const unsigned n = (unsigned)T * F;
  const size_t by = (((size_t)b * ncs_y + ck) * TP + pt) * P + pf, bo = (((size_t)b * ncs_out + ck) * TP + pt) * P + pf;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const unsigned i = (blockIdx.x * 4 + k) * kUT + threadIdx.x;
    if (i >= n) break;
    const unsigned t = i / (unsigned)F, f = i - t * (unsigned)F;
    float v[8];
    unpack8<FMT>(y[by + (size_t)t * P + f], v);
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = fmaxf(bn_val(v[e], mean[e], rstd[e], wc[e], bc[e]), 0.f);
    if (out_split)
      out[((((size_t)b * out_split + f % out_split) * NCk + ck) * TP + pt + t) * P2 + pf + f / out_split] = pack8<FMT>(v);
    else
      out[bo + (size_t)t * P + f] = pack8<FMT>(v);
  }
}

struct BnBwdFinal {
  float *sums2c, *dw, *db, *conv_gb;
};
// ---- backward: the two per-channel sums ----------------------------------------------------------------------------------------------
template <int FMT>
__global__ void __launch_bounds__(kUT) bn_relu_bwd_partial_cp8_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y,
                                                                      const float* __restrict__ stats, const float* __restrict__ w,
                                                                      const float* __restrict__ bias, float eps, float* __restrict__ partial,
                                                                      unsigned n, Cp8Geo geo, int C, int ncs_g, int ncs_y, int S, BnBwdFinal f,
                                                                      int g_split, int Pg) {
  __shared__ float sh[kUT / 32 * 16];
  const int ck = blockIdx.x, s = blockIdx.y;
  const unsigned i0 = (unsigned)((unsigned long long)n * s / S), i1 = (unsigned)((unsigned long long)n * (s + 1) / S);
  float mean[8], rstd[8], wc[8], bc[8], acc[16];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = ck * 8 + e;
    mean[e] = stats[c];
    rstd[e] = rsqrtf(stats[C + c] + eps);
    wc[e] = w[c];
    bc[e] = bias[c];
    acc[e] = acc[8 + e] = 0.f;
  }
  for (unsigned i = i0 + threadIdx.x; i < i1; i += kUT) {
    float gv[8], yv[8];
    unpack8<FMT>(g[g_split ? geo.at_split(i, gridDim.x, ck, g_split, Pg) : geo.at(i, ncs_g, ck)], gv);
    unpack8<FMT>(y[geo.at(i, ncs_y, ck)], yv);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float gp = bn_val(yv[e], mean[e], rstd[e], wc[e], bc[e]) > 0.f ? gv[e] : 0.f;
      acc[e] += gp;
      acc[8 + e] = fmaf(gp, (yv[e] - mean[e]) * rstd[e], acc[8 + e]);
    }
  }
  block_sum_n<16>(acc, sh);
  if (threadIdx.x < 16) {
    const int e = threadIdx.x & 7, which = threadIdx.x >> 3;
    partial[(size_t)(which * C + ck * 8 + e) * S + s] = acc[threadIdx.x];
  }
  unsigned* counter = reinterpret_cast<unsigned*>(partial) - 64 + ck;
  if (!last_block_done(counter)) return;
  // sums2c[k] = sum_s partial[k][s] (lane-strided, then a shuffle tree: fixed order) for the 16 rows of this chunk, two per warp;
  // d beta = s1, d gamma = s2; the conv-bias gradient is zeroed for the apply kernel's atomics
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int which = r, e = threadIdx.x >> 5;
    const int k = which * C + ck * 8 + e;
    float t = 0.f;
    for (int sl = threadIdx.x & 31; sl < S; sl += 32) t += __ldcg(&partial[(size_t)k * S + sl]);
    t = warp_sum(t);
    if ((threadIdx.x & 31) == 0) {
      f.sums2c[k] = t;
      if (which == 0) {
        f.db[k] = t;
        if (f.conv_gb) f.conv_gb[k] = 0.f;
      } else {
        f.dw[k - C] = t;
      }
    }
  }
  if (threadIdx.x == 0) *counter = 0u;
}

// ---- backward apply: dy (CP8) and the conv-bias gradient ------------------------------------------------------------------------------
template <int FMT>
__global__ void __launch_bounds__(kUT) bn_relu_bwd_apply_cp8_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y, uint4* __restrict__ dy,
                                                                    const float* __restrict__ stats, const float* __restrict__ w,
                                                                    const float* __restrict__ bias, const float* __restrict__ sums, float eps,
                                                                    float inv_n, float* __restrict__ conv_gb, int C, int NCk, int T, int F, int TP,
                                                                    int P, int pf, int pt, int ncs_g, int ncs_y, int ncs_dy, int g_split, int Pg) {
  __shared__ float sh[kUT / 32 * 8];
  const int ck = blockIdx.y % NCk, b = blockIdx.y / NCk;
  float mean[8], rstd[8], wc[8], bc[8], m1[8], m2[8], tot[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = ck * 8 + e;
    mean[e] = stats[c];
    rstd[e] = rsqrtf(stats[C + c] + eps);
    wc[e] = w[c];
    bc[e] = bias[c];
    m1[e] = sums[c] * inv_n;
    m2[e] = sums[C + c] * inv_n;
    tot[e] = 0.f;
  }
  const unsigned n = (unsigned)T * F;
  const size_t bg = (((size_t)b * ncs_g + ck) * TP + pt) * P + pf, by = (((size_t)b * ncs_y + ck) * TP + pt) * P + pf,
               bd = (((size_t)b * ncs_dy + ck) * TP + pt) * P + pf;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const unsigned i = (blockIdx.x * 4 + k) * kUT + threadIdx.x;
    if (i >= n) break;
    const unsigned t = i / (unsigned)F, f = i - t * (unsigned)F;
    const size_t o = (size_t)t * P + f;
    float gv[8], yv[8], r[8];
    unpack8<FMT>(g[g_split ? ((((size_t)b * g_split + f % g_split) * NCk + ck) * TP + pt + t) * Pg + pf + f / g_split : bg + o], gv);
    unpack8<FMT>(y[by + o], yv);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float gp = bn_val(yv[e], mean[e], rstd[e], wc[e], bc[e]) > 0.f ? gv[e] : 0.f;
      r[e] = wc[e] * rstd[e] * (gp - m1[e] - (yv[e] - mean[e]) * rstd[e] * m2[e]);
      tot[e] += r[e];
    }
    dy[bd + o] = pack8<FMT>(r);
  }
  if (conv_gb) {
    block_sum_n<8>(tot, sh);
    if (threadIdx.x < 8) atomicAdd(&conv_gb[ck * 8 + threadIdx.x], tot[threadIdx.x]);
  }
}

// ---- backward with frozen statistics (eval-mode BatchNorm: running mean / variance, nothing depends on the batch) ------------------
// g' = g * [a > 0];  dy = gamma * rstd * g' (one pass, written as CP8);  d gamma = sum g' * xhat, d beta = sum g', d conv-bias = sum dy.
// Same (chunk, slice) grid and ordered last-block merge as the batch-statistics backward; the conv-bias gradient is a third ordered sum
// here (it is not zero: the statistics do not follow the convolution's bias).
template <int FMT>
__global__ void __launch_bounds__(kUT) bn_relu_bwd_frozen_cp8_kernel(const uint4* __restrict__ g, const uint4* __restrict__ y, uint4* __restrict__ dy,
                                                                     const float* __restrict__ stats, const float* __restrict__ w,
                                                                     const float* __restrict__ bias, float eps, float* __restrict__ partial,
                                                                     unsigned n, Cp8Geo geo, int C, int ncs_g, int ncs_y, int ncs_dy, int S,
                                                                     BnBwdFinal f, int g_split, int Pg) {
  __shared__ float sh[kUT / 32 * 24];
  const int ck = blockIdx.x, s = blockIdx.y;
  const unsigned i0 = (unsigned)((unsigned long long)n * s / S), i1 = (unsigned)((unsigned long long)n * (s + 1) / S);
  float mean[8], rstd[8], wc[8], bc[8], acc[24];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int c = ck * 8 + e;
    mean[e] = stats[c];
    rstd[e] = rsqrtf(stats[C + c] + eps);
    wc[e] = w[c];
    bc[e] = bias[c];
    acc[e] = acc[8 + e] = acc[16 + e] = 0.f;
  }
  for (unsigned i = i0 + threadIdx.x; i < i1; i += kUT) {
    float gv[8], yv[8], r[8];
    unpack8<FMT>(g[g_split ? geo.at_split(i, gridDim.x, ck, g_split, Pg) : geo.at(i, ncs_g, ck)], gv);
    unpack8<FMT>(y[geo.at(i, ncs_y, ck)], yv);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float gp = bn_val(yv[e], mean[e], rstd[e], wc[e], bc[e]) > 0.f ? gv[e] : 0.f;
      r[e] = wc[e] * rstd[e] * gp;
      acc[e] += gp;
      acc[8 + e] = fmaf(gp, (yv[e] - mean[e]) * rstd[e], acc[8 + e]);
      acc[16 + e] += r[e];
    }
    dy[geo.at(i, ncs_dy, ck)] = pack8<FMT>(r);
  }
  block_sum_n<24>(acc, sh);
  if (threadIdx.x < 24) {
    const int e = threadIdx.x & 7, which = threadIdx.x >> 3;
    partial[(size_t)(which * C + ck * 8 + e) * S + s] = acc[threadIdx.x];
  }
  unsigned* counter = reinterpret_cast<unsigned*>(partial) - 64 + ck;
  if (!last_block_done(counter)) return;
  // the 24 rows of this chunk (s1 | s2 | sum dy per channel), three per warp, each summed lane-strided + shuffle tree (fixed order)
#pragma unroll
  for (int which = 0; which < 3; ++which) {
    const int c = ck * 8 + (threadIdx.x >> 5);
    const int k = which * C + c;
    float t = 0.f;
    for (int sl = threadIdx.x & 31; sl < S; sl += 32) t += __ldcg(&partial[(size_t)k * S + sl]);
    t = warp_sum(t);
    if ((threadIdx.x & 31) == 0) {
      if (which == 0) f.db[c] = t;
      else if (which == 1) f.dw[c] = t;
      else if (f.conv_gb) f.conv_gb[c] = t;
    }
  }
  if (threadIdx.x == 0) *counter = 0u;
}

// ---- MaxPool2d(2) backward + skip-gradient add ----------------------------------------------------------------------------------------
// thread = one pixel-chunk of the un-pooled level: out = addend + [this pixel is the first maximum of its window] * g_pool[window]
template <int FMT>
__global__ void __launch_bounds__(kUT) maxpool2x2_bwd_cp8_kernel(const uint4* __restrict__ a, const uint4* __restrict__ g_pool,
                                                                 const uint4* __restrict__ addend, uint4* __restrict__ out, int NCk, int T, int F,
                                                                 int TP, int P, int pf, int pt, int ncs_a, int ncs_add, int ncs_out, int To, int Fo,
                                                                 int TPo, int Po, int pfo, int pto, int ncs_gp) {
  const int ck = blockIdx.y % NCk, b = blockIdx.y / NCk;
  const unsigned i = blockIdx.x * kUT + threadIdx.x;
  if (i >= (unsigned)T * F) return;
  const int t = (int)(i / (unsigned)F), f = (int)(i - (unsigned)t * F);
  float r[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) r[e] = 0.f;
  if (addend) unpack8<FMT>(addend[(((size_t)b * ncs_add + ck) * TP + pt + t) * P + pf + f], r);
  const int wt = t >> 1, wf = f >> 1;
  if (wt < To && wf < Fo) {
    const size_t wb = (((size_t)b * ncs_a + ck) * TP + pt + 2 * wt) * P + pf + 2 * wf;
    float v[4][8], gp[8];
    unpack8<FMT>(a[wb], v[0]);
    unpack8<FMT>(a[wb + 1], v[1]);
    unpack8<FMT>(a[wb + P], v[2]);
    unpack8<FMT>(a[wb + P + 1], v[3]);
    unpack8<FMT>(g_pool[(((size_t)b * ncs_gp + ck) * TPo + pto + wt) * Po + pfo + wf], gp);
    const int me = (t & 1) * 2 + (f & 1);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      int am = 0;
      float best = v[0][e];
#pragma unroll
      for (int j = 1; j < 4; ++j)
        if (v[j][e] > best) { best = v[j][e]; am = j; }      // strict '>': the first maximum wins
      if (am == me) r[e] += gp[e];
    }
  }
  out[(((size_t)b * ncs_out + ck) * TP + pt + t) * P + pf + f] = pack8<FMT>(r);
}

// ---- bilinear x2 (align_corners) + pad, backward: thread = one pixel-chunk of the LOW level gathers its taps from the fine gradient ----
template <int FMT>
__global__ void __launch_bounds__(kUT) upsample2x_bwd_cp8_kernel(const uint4* __restrict__ g_up, uint4* __restrict__ g_low, int NCk, int Tl, int Fl,
                                                                 int TPl, int Pl, int pfl, int ptl, int ncs_low, int Ts, int Fs, int TPs, int Ps,
                                                                 int pfs, int pts, int ncs_up) {
  const int ck = blockIdx.y % NCk, b = blockIdx.y / NCk;
  const unsigned i = blockIdx.x * kUT + threadIdx.x;
  if (i >= (unsigned)Tl * Fl) return;
  const int y = (int)(i / (unsigned)Fl), x = (int)(i - (unsigned)y * Fl);
  const int Tu = 2 * Tl, Fu = 2 * Fl;
  const int top = (Ts - Tu) / 2, left = (Fs - Fu) / 2;
  const float ry = Tu > 1 ? (float)(Tl - 1) / (float)(Tu - 1) : 0.f;
  const float rx = Fu > 1 ? (float)(Fl - 1) / (float)(Fu - 1) : 0.f;
  const int hu_lo = ry > 0.f ? max(0, (int)floorf((y - 1) / ry)) : 0;
  const int hu_hi = ry > 0.f ? min(Tu - 1, (int)ceilf((y + 1) / ry)) : Tu - 1;
  const int wu_lo = rx > 0.f ? max(0, (int)floorf((x - 1) / rx)) : 0;
  const int wu_hi = rx > 0.f ? min(Fu - 1, (int)ceilf((x + 1) / rx)) : Fu - 1;
  float acc[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) acc[e] = 0.f;
  const size_t gb = (((size_t)b * ncs_up + ck) * TPs + pts + top) * Ps + pfs + left;
  for (int hu = hu_lo; hu <= hu_hi; ++hu) {
    const float sy = ry * hu;                      // the forward's source coordinate (mpa_upsample2x_cp8)
    const int y0 = (int)sy, y1 = min(y0 + 1, Tl - 1);
    const float ly = sy - y0;
    float wy = 0.f;
    if (y0 == y) wy += 1.f - ly;
    if (y1 == y) wy += ly;
    if (wy == 0.f) continue;
    for (int wu = wu_lo; wu <= wu_hi; ++wu) {
      const float sx = rx * wu;
      const int x0 = (int)sx, x1 = min(x0 + 1, Fl - 1);
      const float lx = sx - x0;
      float wx = 0.f;
      if (x0 == x) wx += 1.f - lx;
      if (x1 == x) wx += lx;
      if (wx == 0.f) continue;
      float gv[8];
      unpack8<FMT>(g_up[gb + (size_t)hu * Ps + wu], gv);
      const float wgt = wy * wx;
#pragma unroll
      for (int e = 0; e < 8; ++e) acc[e] = fmaf(wgt, gv[e], acc[e]);
    }
  }
  g_low[(((size_t)b * ncs_low + ck) * TPl + ptl + y) * Pl + pfl + x] = pack8<FMT>(acc);
}

static inline int slices_for(long long n_pix, int NCk) {
  long long S = (148LL * 8 + NCk - 1) / NCk, by_work = (n_pix + 2047) / 2048;
  S = S < by_work ? S : by_work;
  return (int)(S < 1 ? 1 : (S > 512 ? 512 : S));
}

}  // namespace mpa

using namespace mpa;

#define UNET_CP8_COMMON(name)                                                                                                         \
  MPA_CHECK_ARCH();                                                                                                                   \
  MPA_REQUIRE(B > 0 && C > 0 && C % 8 == 0 && T > 0 && F > 0 && pitch >= pf + F && pt >= 0 && (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16), \
              name ": bad argument (C must be a multiple of 8; 16-bit formats only)");                                               \
  MPA_REQUIRE((long long)B* T* F < (1LL << 31), name ": tensor too large")

extern "C" {

int mpa_bn_stats_cp8(const void* y_cp8, float* stats, const float* pivot, int B, int C, int T, int F, int pitch, int pf, int pt, int ncs, int fmt,
                     float* running_mean, float* running_var, float momentum, long long* num_batches_tracked, void* stream) {
  UNET_CP8_COMMON("bn_stats_cp8");
  MPA_REQUIRE(y_cp8 && stats && (!running_mean == !running_var), "bn_stats_cp8: null pointer");
  float* scratch = unet_scratch();
  MPA_REQUIRE(scratch, "bn_stats_cp8: scratch allocation failed");
  const int NCk = C / 8;
  if (ncs <= 0) ncs = NCk;
  const unsigned n = (unsigned)B * T * F;
  const int S = slices_for(n, NCk);
  MPA_REQUIRE((size_t)C * S * 2 <= (1u << 20) && NCk <= 64, "bn_stats_cp8: too many channels (<= 512)");
  const Cp8Geo g{T, F, T + 2 * pt, pitch, pf, pt};
  cudaStream_t st = (cudaStream_t)stream;
  const BnStatsFinal f{pivot, stats, running_mean, running_var, momentum, num_batches_tracked};
  if (fmt == MPA_FMT_BF16)
    bn_stats_partial_cp8_kernel<MPA_FMT_BF16><<<dim3(NCk, S), kUT, 0, st>>>((const uint4*)y_cp8, scratch, n, g, ncs, S, f);
  else
    bn_stats_partial_cp8_kernel<MPA_FMT_F16><<<dim3(NCk, S), kUT, 0, st>>>((const uint4*)y_cp8, scratch, n, g, ncs, S, f);
  MPA_CHECK_LAUNCH("bn_stats_cp8");
  return MPA_OK;
}

int mpa_bn_relu_apply_cp8(const void* y_cp8, void* out_cp8, const float* stats, const float* weight, const float* bias, float eps, int B, int C,
                          int T, int F, int pitch, int pf, int pt, int ncs_y, int ncs_out, int out_split, int out_pitch, int fmt, void* stream) {
  UNET_CP8_COMMON("bn_relu_apply_cp8");
  MPA_REQUIRE(y_cp8 && out_cp8 && stats && weight && bias, "bn_relu_apply_cp8: null pointer");
  MPA_REQUIRE(out_split == 0 || (out_split > 1 && F % out_split == 0 && out_pitch >= pf + F / out_split), "bn_relu_apply_cp8: bad phase split");
  const int NCk = C / 8;
  if (ncs_y <= 0) ncs_y = NCk;
  if (ncs_out <= 0) ncs_out = NCk;
  const dim3 grid(ceil_div((long long)T * F, 4 * kUT), B * NCk);
  if (fmt == MPA_FMT_BF16)
    bn_relu_apply_cp8_kernel<MPA_FMT_BF16><<<grid, kUT, 0, (cudaStream_t)stream>>>((const uint4*)y_cp8, (uint4*)out_cp8, stats, weight, bias, eps, C,
                                                                                  NCk, T, F, T + 2 * pt, pitch, pf, pt, ncs_y, ncs_out, out_split, out_pitch);
  else
    bn_relu_apply_cp8_kernel<MPA_FMT_F16><<<grid, kUT, 0, (cudaStream_t)stream>>>((const uint4*)y_cp8, (uint4*)out_cp8, stats, weight, bias, eps, C,
                                                                                 NCk, T, F, T + 2 * pt, pitch, pf, pt, ncs_y, ncs_out, out_split, out_pitch);
  MPA_CHECK_LAUNCH("bn_relu_apply_cp8");
  return MPA_OK;
}

int mpa_bn_relu_bwd_cp8(const void* g_cp8, const void* y_cp8, void* dy_cp8, const float* stats, const float* weight, const float* bias, float eps,
                        float* g_weight, float* g_bias, float* g_conv_bias, int B, int C, int T, int F, int pitch, int pf, int pt, int ncs_g,
                        int ncs_y, int ncs_dy, int g_split, int g_pitch, int fmt, void* stream) {
  UNET_CP8_COMMON("bn_relu_bwd_cp8");
  MPA_REQUIRE(g_cp8 && y_cp8 && dy_cp8 && stats && weight && bias && g_weight && g_bias, "bn_relu_bwd_cp8: null pointer");
  MPA_REQUIRE(g_split == 0 || (g_split > 1 && F % g_split == 0 && g_pitch >= pf + F / g_split), "bn_relu_bwd_cp8: bad phase split");
  float* scratch = unet_scratch();
  MPA_REQUIRE(scratch, "bn_relu_bwd_cp8: scratch allocation failed");
  const int NCk = C / 8;
  if (ncs_g <= 0) ncs_g = NCk;
  if (ncs_y <= 0) ncs_y = NCk;
  if (ncs_dy <= 0) ncs_dy = NCk;
  const unsigned n = (unsigned)B * T * F;
  const int S = slices_for(n, NCk);
  MPA_REQUIRE((size_t)2 * C * S + 2 * C <= (1u << 20) && NCk <= 64, "bn_relu_bwd_cp8: too many channels (<= 512)");
  float* sums = scratch + (size_t)2 * C * S;
  const Cp8Geo geo{T, F, T + 2 * pt, pitch, pf, pt};
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid_a(ceil_div((long long)T * F, 4 * kUT), B * NCk);
  const BnBwdFinal f{sums, g_weight, g_bias, g_conv_bias};
  if (fmt == MPA_FMT_BF16)
    bn_relu_bwd_partial_cp8_kernel<MPA_FMT_BF16><<<dim3(NCk, S), kUT, 0, st>>>((const uint4*)g_cp8, (const uint4*)y_cp8, stats, weight, bias, eps,
                                                                              scratch, n, geo, C, ncs_g, ncs_y, S, f, g_split, g_pitch);
  else
    bn_relu_bwd_partial_cp8_kernel<MPA_FMT_F16><<<dim3(NCk, S), kUT, 0, st>>>((const uint4*)g_cp8, (const uint4*)y_cp8, stats, weight, bias, eps,
                                                                             scratch, n, geo, C, ncs_g, ncs_y, S, f, g_split, g_pitch);
  MPA_CHECK_LAUNCH("bn_relu_bwd_sums_cp8");
  const float inv_n = 1.f / (float)n;
  if (fmt == MPA_FMT_BF16)
    bn_relu_bwd_apply_cp8_kernel<MPA_FMT_BF16><<<grid_a, kUT, 0, st>>>((const uint4*)g_cp8, (const uint4*)y_cp8, (uint4*)dy_cp8, stats, weight, bias,
                                                                      sums, eps, inv_n, g_conv_bias, C, NCk, T, F, T + 2 * pt, pitch, pf, pt, ncs_g,
                                                                      ncs_y, ncs_dy, g_split, g_pitch);
  else
    bn_relu_bwd_apply_cp8_kernel<MPA_FMT_F16><<<grid_a, kUT, 0, st>>>((const uint4*)g_cp8, (const uint4*)y_cp8, (uint4*)dy_cp8, stats, weight, bias,
                                                                     sums, eps, inv_n, g_conv_bias, C, NCk, T, F, T + 2 * pt, pitch, pf, pt, ncs_g,
                                                                     ncs_y, ncs_dy, g_split, g_pitch);
  MPA_CHECK_LAUNCH("bn_relu_bwd_apply_cp8");
  return MPA_OK;
}

int mpa_bn_relu_bwd_frozen_cp8(const void* g_cp8, const void* y_cp8, void* dy_cp8, const float* stats, const float* weight, const float* bias,
                               float eps, float* g_weight, float* g_bias, float* g_conv_bias, int B, int C, int T, int F, int pitch, int pf, int pt,
                               int ncs_g, int ncs_y, int ncs_dy, int g_split, int g_pitch, int fmt, void* stream) {
  UNET_CP8_COMMON("bn_relu_bwd_frozen_cp8");
  MPA_REQUIRE(g_cp8 && y_cp8 && dy_cp8 && stats && weight && bias && g_weight && g_bias, "bn_relu_bwd_frozen_cp8: null pointer");
  MPA_REQUIRE(g_split == 0 || (g_split > 1 && F % g_split == 0 && g_pitch >= pf + F / g_split), "bn_relu_bwd_frozen_cp8: bad phase split");
  float* scratch = unet_scratch();
  MPA_REQUIRE(scratch, "bn_relu_bwd_frozen_cp8: scratch allocation failed");
  const int NCk = C / 8;
  if (ncs_g <= 0) ncs_g = NCk;
  if (ncs_y <= 0) ncs_y = NCk;
  if (ncs_dy <= 0) ncs_dy = NCk;
  const unsigned n = (unsigned)B * T * F;
  const int S = slices_for(n, NCk);
  MPA_REQUIRE((size_t)3 * C * S <= (1u << 20) && NCk <= 64, "bn_relu_bwd_frozen_cp8: too many channels (<= 512)");
  const Cp8Geo geo{T, F, T + 2 * pt, pitch, pf, pt};
  const BnBwdFinal f{nullptr, g_weight, g_bias, g_conv_bias};
  cudaStream_t st = (cudaStream_t)stream;
  if (fmt == MPA_FMT_BF16)
    bn_relu_bwd_frozen_cp8_kernel<MPA_FMT_BF16><<<dim3(NCk, S), kUT, 0, st>>>((const uint4*)g_cp8, (const uint4*)y_cp8, (uint4*)dy_cp8, stats, weight,
                                                                             bias, eps, scratch, n, geo, C, ncs_g, ncs_y, ncs_dy, S, f, g_split, g_pitch);
  else
    bn_relu_bwd_frozen_cp8_kernel<MPA_FMT_F16><<<dim3(NCk, S), kUT, 0, st>>>((const uint4*)g_cp8, (const uint4*)y_cp8, (uint4*)dy_cp8, stats, weight,
                                                                            bias, eps, scratch, n, geo, C, ncs_g, ncs_y, ncs_dy, S, f, g_split, g_pitch);
  MPA_CHECK_LAUNCH("bn_relu_bwd_frozen_cp8");
  return MPA_OK;
}

int mpa_maxpool2x2_bwd_cp8(const void* a_cp8, const void* g_pool_cp8, const void* addend_cp8, void* out_cp8, int B, int C, int T, int F, int pitch,
                           int pf, int pt, int ncs_a, int ncs_add, int ncs_out, int pitch_o, int pf_o, int pt_o, int ncs_gp, int fmt,
                           void* stream) {
  UNET_CP8_COMMON("maxpool2x2_bwd_cp8");
  MPA_REQUIRE(a_cp8 && g_pool_cp8 && out_cp8 && T >= 2 && F >= 2 && pitch_o >= pf_o + F / 2 && pt_o >= 0, "maxpool2x2_bwd_cp8: bad argument");
  const int NCk = C / 8, To = T / 2, Fo = F / 2;
  if (ncs_a <= 0) ncs_a = NCk;
  if (ncs_add <= 0) ncs_add = NCk;
  if (ncs_out <= 0) ncs_out = NCk;
  if (ncs_gp <= 0) ncs_gp = NCk;
  const dim3 grid(ceil_div((long long)T * F, kUT), B * NCk);
  if (fmt == MPA_FMT_BF16)
    maxpool2x2_bwd_cp8_kernel<MPA_FMT_BF16><<<grid, kUT, 0, (cudaStream_t)stream>>>(
        (const uint4*)a_cp8, (const uint4*)g_pool_cp8, (const uint4*)addend_cp8, (uint4*)out_cp8, NCk, T, F, T + 2 * pt, pitch, pf, pt, ncs_a, ncs_add,
        ncs_out, To, Fo, To + 2 * pt_o, pitch_o, pf_o, pt_o, ncs_gp);
  else
    maxpool2x2_bwd_cp8_kernel<MPA_FMT_F16><<<grid, kUT, 0, (cudaStream_t)stream>>>(
        (const uint4*)a_cp8, (const uint4*)g_pool_cp8, (const uint4*)addend_cp8, (uint4*)out_cp8, NCk, T, F, T + 2 * pt, pitch, pf, pt, ncs_a, ncs_add,
        ncs_out, To, Fo, To + 2 * pt_o, pitch_o, pf_o, pt_o, ncs_gp);
  MPA_CHECK_LAUNCH("maxpool2x2_bwd_cp8");
  return MPA_OK;
}

int mpa_upsample2x_bwd_cp8(const void* g_up_cp8, void* g_low_cp8, int B, int C, int Tl, int Fl, int pitch_l, int pf_l, int pt_l, int ncs_low,
                           int Ts, int Fs, int pitch_s, int pf_s, int pt_s, int ncs_up, int fmt, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(g_up_cp8 && g_low_cp8 && B > 0 && C > 0 && C % 8 == 0 && Tl > 0 && Fl > 0 && Ts >= 2 * Tl && Fs >= 2 * Fl &&
                  pitch_l >= pf_l + Fl && pitch_s >= pf_s + Fs && (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16),
              "upsample2x_bwd_cp8: bad argument");
  const int NCk = C / 8;
  if (ncs_low <= 0) ncs_low = NCk;
  if (ncs_up <= 0) ncs_up = NCk;
  const dim3 grid(ceil_div((long long)Tl * Fl, kUT), B * NCk);
  if (fmt == MPA_FMT_BF16)
    upsample2x_bwd_cp8_kernel<MPA_FMT_BF16><<<grid, kUT, 0, (cudaStream_t)stream>>>((const uint4*)g_up_cp8, (uint4*)g_low_cp8, NCk, Tl, Fl,
                                                                                   Tl + 2 * pt_l, pitch_l, pf_l, pt_l, ncs_low, Ts, Fs, Ts + 2 * pt_s,
                                                                                   pitch_s, pf_s, pt_s, ncs_up);
  else
    upsample2x_bwd_cp8_kernel<MPA_FMT_F16><<<grid, kUT, 0, (cudaStream_t)stream>>>((const uint4*)g_up_cp8, (uint4*)g_low_cp8, NCk, Tl, Fl,
                                                                                  Tl + 2 * pt_l, pitch_l, pf_l, pt_l, ncs_low, Ts, Fs, Ts + 2 * pt_s,
                                                                                  pitch_s, pf_s, pt_s, ncs_up);
  MPA_CHECK_LAUNCH("upsample2x_bwd_cp8");
  return MPA_OK;
}

}  // extern "C"
