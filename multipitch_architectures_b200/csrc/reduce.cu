// Per-channel reductions over (batch, pixels) of NCHW fp32 tensors — bias gradients, BatchNorm batch statistics and the two
// sums of the BatchNorm backward — spread over the whole GPU: a (channel, slice) grid writes partial results, a second tiny
// kernel combines the slices of a channel in a FIXED order (bit-reproducible; no atomics).  The partials live in a small
// per-device scratch buffer owned by the library (allocated once, 4 MB).
#include "common.cuh"

namespace mpa {

constexpr int kRedThreads = 256;
constexpr int kRedMaxSlices = 64;
constexpr size_t kRedScratchFloats = 1u << 20;

static float* reduce_scratch() {
  static float* ptr[64] = {nullptr};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (!ptr[dev]) {
    float* p = nullptr;
    if (cudaMalloc(&p, kRedScratchFloats * sizeof(float)) != cudaSuccess) return nullptr;
    ptr[dev] = p;
  }
  return ptr[dev];
}

static inline int pick_slices(long long n_per_channel, int C) {
  long long want = (148LL * 8 + C - 1) / C;                  // about 8 blocks per SM in total
  long long max_by_work = (n_per_channel + 2047) / 2048;     // at least ~2k elements per block
  long long s = want < max_by_work ? want : max_by_work;
  if (s < 1) s = 1;
  if (s > kRedMaxSlices) s = kRedMaxSlices;
  return (int)s;
}

__device__ __forceinline__ float block_sum_red(float v, float* sh) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
#pragma unroll
  for (int i = 0; i < kRedThreads / 32; ++i) r += sh[i];
  return r;
}

// slice [i0, i1) of the flattened (b, hw) index of channel c
__device__ __forceinline__ void slice_range(long long n, int S, int s, long long& i0, long long& i1) {
  i0 = n * s / S;
  i1 = n * (s + 1) / S;
}
__device__ __forceinline__ size_t nchw_index(long long i, int c, int C, int HW) {
  const long long b = i / HW;
  return ((size_t)b * C + c) * HW + (size_t)(i - b * HW);
}

// mode 0: partial[c][s] = sum x.   mode 1 (BatchNorm backward): partial[c][s] = sum g', partial2 = sum g' * xhat,
//         g' = dy * (out > 0) when relu.
__global__ void __launch_bounds__(kRedThreads) channel_partial_kernel(const float* __restrict__ x, const float* __restrict__ out_act,
                                                                      const float* __restrict__ dy, const float* __restrict__ stats, float eps,
                                                                      float* __restrict__ partial, int B, int C, int HW, int S, int mode, int relu,
                                                                      int vec) {
  __shared__ float sh[kRedThreads / 32];
  const int c = blockIdx.x, s = blockIdx.y;
  long long i0, i1;
  slice_range((long long)B * HW, S, s, i0, i1);
  float a1 = 0.f, a2 = 0.f;
  if (vec) {
    // HW % 4 == 0 and 16-byte aligned tensors: 16-byte loads, one index division per 4 elements (slices in units of 4 elements)
    const int HW4 = HW >> 2;
    long long j0, j1;
    slice_range((long long)B * HW4, S, s, j0, j1);
    const float4* x4 = reinterpret_cast<const float4*>(x);
    if (mode == 0) {
#pragma unroll 2
      for (long long j = j0 + threadIdx.x; j < j1; j += kRedThreads) {
        const long long b = j / HW4;
        const float4 v = x4[(b * C + c) * HW4 + (j - b * HW4)];
        a1 += (v.x + v.y) + (v.z + v.w);
      }
    } else {
      const float4* dy4 = reinterpret_cast<const float4*>(dy);
      const float4* oa4 = reinterpret_cast<const float4*>(out_act);
      const float mean = stats[c], rstd = rsqrtf(stats[C + c] + eps);
#pragma unroll 2
      for (long long j = j0 + threadIdx.x; j < j1; j += kRedThreads) {
        const long long b = j / HW4;
        const size_t idx = (size_t)((b * C + c) * HW4 + (j - b * HW4));
        float4 g = dy4[idx];
        const float4 xv = x4[idx];
        if (relu) {
          const float4 o = oa4[idx];
          if (!(o.x > 0.f)) g.x = 0.f;
          if (!(o.y > 0.f)) g.y = 0.f;
          if (!(o.z > 0.f)) g.z = 0.f;
          if (!(o.w > 0.f)) g.w = 0.f;
        }
        a1 += (g.x + g.y) + (g.z + g.w);
        a2 += (g.x * (xv.x - mean) * rstd + g.y * (xv.y - mean) * rstd) + (g.z * (xv.z - mean) * rstd + g.w * (xv.w - mean) * rstd);
      }
    }
  } else if (mode == 0) {
    for (long long i = i0 + threadIdx.x; i < i1; i += kRedThreads) a1 += x[nchw_index(i, c, C, HW)];
  } else {
    const float mean = stats[c], rstd = rsqrtf(stats[C + c] + eps);
    for (long long i = i0 + threadIdx.x; i < i1; i += kRedThreads) {
      const size_t idx = nchw_index(i, c, C, HW);
      float g = dy[idx];
      if (relu && !(out_act[idx] > 0.f)) g = 0.f;
      a1 += g;
      a2 += g * (x[idx] - mean) * rstd;
    }
  }
  a1 = block_sum_red(a1, sh);
  if (mode == 1) a2 = block_sum_red(a2, sh);
  if (threadIdx.x == 0) {
    partial[(size_t)c * S + s] = a1;
    if (mode == 1) partial[(size_t)(C + c) * S + s] = a2;
  }
}
// out[k] = sum_s partial[k][s] in slice order; k over n_rows (C or 2C); optional second copy (dw / db of the BatchNorm backward)
__global__ void channel_final_kernel(const float* __restrict__ partial, float* __restrict__ out, float* __restrict__ out2, int n_rows, int S) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n_rows) return;
  float t = 0.f;
  for (int s = 0; s < S; ++s) t += partial[(size_t)k * S + s];
  out[k] = t;
  if (out2) out2[k] = t;
}

// Per-channel sums of a 16-bit CP8 tensor (bias gradient of a tensor-core convolution whose output gradient never leaves the CP8 layout):
// grid (chunk, slice); a thread adds the 8 channels of its pixels in fp32, the block's 8 sums go to partial[(chunk*8 + e)][slice]
template <int FMT>
__global__ void __launch_bounds__(kRedThreads) channel_partial_cp8_kernel(const uint4* __restrict__ g, float* __restrict__ partial, int B, int T, int F,
                                                                          int TP, int P, int pf, int pt, int ncs, int S) {
  __shared__ float sh[kRedThreads / 32];
  const int ck = blockIdx.x, s = blockIdx.y;
  const unsigned n = (unsigned)B * T * F;
  const unsigned i0 = (unsigned)((unsigned long long)n * s / S), i1 = (unsigned)((unsigned long long)n * (s + 1) / S);
  float a[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) a[e] = 0.f;
  for (unsigned i = i0 + threadIdx.x; i < i1; i += kRedThreads) {
    const unsigned row = i / F, f = i - row * F;
    const unsigned b = row / T, t = row - b * T;
    const uint4 u = g[(((size_t)b * ncs + ck) * TP + pt + t) * P + pf + f];
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (FMT == MPA_FMT_BF16) {
        a[2 * e] += __uint_as_float(w[e] << 16);
        a[2 * e + 1] += __uint_as_float(w[e] & 0xFFFF0000u);
      } else {
        const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&w[e]));
        a[2 * e] += f2.x;
        a[2 * e + 1] += f2.y;
      }
    }
  }
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float r = block_sum_red(a[e], sh);
    if (threadIdx.x == 0) partial[(size_t)(ck * 8 + e) * S + s] = r;
  }
}

// BatchNorm batch statistics: per slice (n, mean, M2) with a two-pass mean / squared deviation inside the slice, merged in slice
// order with Chan's parallel-variance update (robust against |mean| >> std; biased variance = M2 / n as nn.BatchNorm2d normalises)
__global__ void __launch_bounds__(kRedThreads) bn_stats_partial_kernel(const float* __restrict__ x, float* __restrict__ partial, int B, int C, int HW,
                                                                       int S) {
  __shared__ float sh[kRedThreads / 32];
  const int c = blockIdx.x, s = blockIdx.y;
  long long i0, i1;
  slice_range((long long)B * HW, S, s, i0, i1);
  float a = 0.f;
  for (long long i = i0 + threadIdx.x; i < i1; i += kRedThreads) a += x[nchw_index(i, c, C, HW)];
  const float n = (float)(i1 - i0);
  const float mean = n > 0.f ? block_sum_red(a, sh) / n : 0.f;
  float q = 0.f;
  for (long long i = i0 + threadIdx.x; i < i1; i += kRedThreads) {
    const float d = x[nchw_index(i, c, C, HW)] - mean;
    q += d * d;
  }
  q = block_sum_red(q, sh);
  if (threadIdx.x == 0) {
    partial[((size_t)c * S + s) * 2] = mean;
    partial[((size_t)c * S + s) * 2 + 1] = q;
  }
}
__global__ void bn_stats_final_kernel(const float* __restrict__ partial, float* __restrict__ stats, int B, int C, int HW, int S) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const long long n_tot = (long long)B * HW;
  float n = 0.f, mean = 0.f, m2 = 0.f;
  for (int s = 0; s < S; ++s) {
    const float ns = (float)(n_tot * (s + 1) / S - n_tot * s / S);
    if (ns <= 0.f) continue;
    const float ms = partial[((size_t)c * S + s) * 2], qs = partial[((size_t)c * S + s) * 2 + 1];
    const float delta = ms - mean, nn = n + ns;
    mean += delta * (ns / nn);
    m2 += qs + delta * delta * (n * ns / nn);
    n = nn;
  }
  stats[c] = mean;
  stats[C + c] = m2 / (float)n_tot;
}

// *found = 1 when any of x[0, n) is an inf or a NaN (the loss-scale overflow check over the flat gradient of fp16 training; the caller
// cleared the flag).  vec: x is 16-byte aligned — float4 loads over the first n / 4 * 4 elements, the ragged tail element by element.
__global__ void __launch_bounds__(kRedThreads) nonfinite_kernel(const float* __restrict__ x, long long n, int vec, int* __restrict__ found) {
  const long long tid = blockIdx.x * (long long)blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
  const long long n4 = vec ? n >> 2 : 0;
  bool bad = false;
  const float4* x4 = reinterpret_cast<const float4*>(x);
  for (long long i = tid; i < n4; i += stride) {
    const float4 v = x4[i];
    bad |= !isfinite(v.x) | !isfinite(v.y) | !isfinite(v.z) | !isfinite(v.w);
  }
  for (long long i = n4 * 4 + tid; i < n; i += stride) bad |= !isfinite(x[i]);
  if (__syncthreads_or(bad) && threadIdx.x == 0) *found = 1;
}

// Shared with backward.cu / backward_unet.cu -------------------------------------------------------------------------------
int channel_sum_launch(const float* x, float* out, int B, int C, int HW, cudaStream_t st) {
  float* scratch = reduce_scratch();
  if (!scratch) { set_error("channel_sum: scratch allocation failed"); return MPA_ERR_CUDA; }
  const int S = pick_slices((long long)B * HW, C);
  if ((size_t)C * S > kRedScratchFloats) { set_error("channel_sum: too many channels (%d)", C); return MPA_ERR_ARG; }
  const int vec = (HW % 4 == 0) && (((uintptr_t)x & 15) == 0);
  channel_partial_kernel<<<dim3(C, S), kRedThreads, 0, st>>>(x, nullptr, nullptr, nullptr, 0.f, scratch, B, C, HW, S, 0, 0, vec);
  channel_final_kernel<<<ceil_div(C, 128), 128, 0, st>>>(scratch, out, nullptr, C, S);
  return MPA_OK;
}
int channel_sum_cp8_launch(const uint4* g, float* out, int B, int C, int T, int F, int TP, int P, int pf, int pt, int ncs, int fmt, cudaStream_t st) {
  float* scratch = reduce_scratch();
  if (!scratch) { set_error("channel_sum_cp8: scratch allocation failed"); return MPA_ERR_CUDA; }
  if ((long long)B * T * F >= (1LL << 31)) { set_error("channel_sum_cp8: tensor too large"); return MPA_ERR_ARG; }
  const int NCk = (C + 7) / 8;
  // few chunk planes: more slices than pick_slices allows (about 8 CTAs per SM in total, at least ~2k pixels per CTA)
  long long S_ = (148LL * 8 + NCk - 1) / NCk, by_work = ((long long)B * T * F + 2047) / 2048;
  S_ = S_ < by_work ? S_ : by_work;
  const int S = (int)(S_ < 1 ? 1 : (S_ > 512 ? 512 : S_));
  if ((size_t)NCk * 8 * S > kRedScratchFloats) { set_error("channel_sum_cp8: too many channels (%d)", C); return MPA_ERR_ARG; }
  if (fmt == MPA_FMT_BF16)
    channel_partial_cp8_kernel<MPA_FMT_BF16><<<dim3(NCk, S), kRedThreads, 0, st>>>(g, scratch, B, T, F, TP, P, pf, pt, ncs, S);
  else
    channel_partial_cp8_kernel<MPA_FMT_F16><<<dim3(NCk, S), kRedThreads, 0, st>>>(g, scratch, B, T, F, TP, P, pf, pt, ncs, S);
  channel_final_kernel<<<ceil_div(C, 128), 128, 0, st>>>(scratch, out, nullptr, C, S);
  return MPA_OK;
}
int bn_bwd_sums_launch(const float* x, const float* out_act, const float* dy, const float* stats, float eps, float* sums2c, float* dw, float* db,
                       int B, int C, int HW, int relu, cudaStream_t st) {
  float* scratch = reduce_scratch();
  if (!scratch) { set_error("bn_relu_bwd: scratch allocation failed"); return MPA_ERR_CUDA; }
  const int S = pick_slices((long long)B * HW, C);
  if ((size_t)2 * C * S > kRedScratchFloats) { set_error("bn_relu_bwd: too many channels (%d)", C); return MPA_ERR_ARG; }
  const int vec = (HW % 4 == 0) && ((((uintptr_t)x | (uintptr_t)dy | (uintptr_t)out_act) & 15) == 0);
  channel_partial_kernel<<<dim3(C, S), kRedThreads, 0, st>>>(x, out_act, dy, stats, eps, scratch, B, C, HW, S, 1, relu, vec);
  // sums2c = [s1 | s2]; db = s1, dw = s2
  channel_final_kernel<<<ceil_div(C, 128), 128, 0, st>>>(scratch, sums2c, db, C, S);
  channel_final_kernel<<<ceil_div(C, 128), 128, 0, st>>>(scratch + (size_t)C * S, sums2c + C, dw, C, S);
  return MPA_OK;
}
int bn_stats_launch(const float* x, float* stats, int B, int C, int HW, cudaStream_t st) {
  float* scratch = reduce_scratch();
  if (!scratch) { set_error("bn_stats: scratch allocation failed"); return MPA_ERR_CUDA; }
  const int S = pick_slices((long long)B * HW, C);
  if ((size_t)2 * C * S > kRedScratchFloats) { set_error("bn_stats: too many channels (%d)", C); return MPA_ERR_ARG; }
  bn_stats_partial_kernel<<<dim3(C, S), kRedThreads, 0, st>>>(x, scratch, B, C, HW, S);
  bn_stats_final_kernel<<<ceil_div(C, 128), 128, 0, st>>>(scratch, stats, B, C, HW, S);
  return MPA_OK;
}

}  // namespace mpa

using namespace mpa;

extern "C" {

int mpa_nonfinite_check_f32(const float* x, long long n, int* found_inf, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && found_inf && n > 0, "nonfinite_check: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(found_inf, 0, sizeof(int), st);
  const int vec = ((uintptr_t)x & 15) == 0;
  long long blocks = ((vec ? n / 4 : n) + kRedThreads - 1) / kRedThreads;
  blocks = blocks < 1 ? 1 : (blocks > 148LL * 8 ? 148LL * 8 : blocks);        // a grid-stride loop over about 8 blocks per SM
  nonfinite_kernel<<<(int)blocks, kRedThreads, 0, st>>>(x, n, vec, found_inf);
  MPA_CHECK_LAUNCH("nonfinite_check");
  return MPA_OK;
}

int mpa_channel_sum_f32(const float* x, float* out, int B, int C, int HW, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && B > 0 && C > 0 && HW > 0, "channel_sum: bad argument");
  int rc = channel_sum_launch(x, out, B, C, HW, (cudaStream_t)stream);
  if (rc != MPA_OK) return rc;
  MPA_CHECK_LAUNCH("channel_sum");
  return MPA_OK;
}

}  // extern "C"
