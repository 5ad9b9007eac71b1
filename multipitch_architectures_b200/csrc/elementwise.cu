// HBM-bound stages of the patch-wise networks: LayerNorm(+log compression), pooling, bilinear upsample +
// concat, BatchNorm statistics/apply, BCE loss.  fp32 NCHW.  All kernels are grid-stride / row-per-block with
// coalesced accesses along F (the contiguous axis).
#include "common.cuh"
#include <cuda_fp16.h>

namespace mpa {

__device__ __forceinline__ float block_sum(float v, float* sh) {
  v = warp_sum(v);
  int w = threadIdx.x >> 5, l = threadIdx.x & 31, nw = (blockDim.x + 31) >> 5;
  __syncthreads();
  if (l == 0) sh[w] = v;
  __syncthreads();
  float r = (threadIdx.x < nw) ? sh[threadIdx.x] : 0.f;
  if (w == 0) {
    r = warp_sum(r);
    if (l == 0) sh[0] = r;
  }
  __syncthreads();
  return sh[0];
}

// one block per (b,t) row; the row is the C x F slab x[b, :, t, :]
template <int MAXV>
__global__ void __launch_bounds__(128) layernorm_cf_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                           const float* __restrict__ bsh, float* __restrict__ out,
                                                           int C, int T, int F, float eps, float gamma_log) {
  __shared__ float sh[8];
  int b = blockIdx.x / T, t = blockIdx.x % T;
  const int n = C * F;
  const float* xr = x + ((size_t)b * C * T + t) * F;
  float* orow = out + ((size_t)b * C * T + t) * F;
  float v[MAXV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int e = threadIdx.x + i * 128;
    float val = 0.f;
    if (e < n) {
      int c = e / F, f = e - c * F;
      val = xr[(size_t)c * T * F + f];
      if (gamma_log > 0.f) val = logf(__fadd_rn(1.f, __fmul_rn(gamma_log, val)));
      s += val;
    }
    v[i] = val;
  }
  float mean = block_sum(s, sh) / n;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int e = threadIdx.x + i * 128;
    if (e < n) {
      float d = v[i] - mean;
      q += d * d;
    }
  }
  float rstd = rsqrtf(block_sum(q, sh) / n + eps);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int e = threadIdx.x + i * 128;
    if (e < n) {
      int c = e / F, f = e - c * F;
      orow[(size_t)c * T * F + f] = (v[i] - mean) * rstd * w[e] + bsh[e];
    }
  }
}

// The same row LayerNorm written straight into the 16-bit CP8 planes the first convolution reads (C <= 8: one chunk; channels >= C hold
// zeros): the fp32 NCHW copy of the normalised input and its converter pass (2 x 100 MB per CNN:XS training step) disappear.  The row is
// staged in shared memory as [F][8] 16-bit so that every pixel leaves as one 16-byte store.
template <int MAXV>
__global__ void __launch_bounds__(128) layernorm_cf_cp8_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                               const float* __restrict__ bsh, uint4* __restrict__ out, int C, int T, int F, int TP,
                                                               int P, int pf, int pt, float eps, float gamma_log, int fmt) {
  extern __shared__ __align__(16) uint16_t row16[];      // [F][8]
  __shared__ float sh[8];
  const int b = blockIdx.x / T, t = blockIdx.x % T;
  const int n = C * F;
  const float* xr = x + ((size_t)b * C * T + t) * F;
  float v[MAXV];
  float s = 0.f;
  for (int i = threadIdx.x; i < F * 4; i += 128) reinterpret_cast<uint32_t*>(row16)[i] = 0u;
  // (c, f) of element e = threadIdx.x + 128 i advance incrementally: the kernel was issue-bound (ncu: 65 % of the issue slots, 0.9 TB/s)
  // on one integer division per element and loop
  const int c_first = threadIdx.x / F, f_first = threadIdx.x - c_first * F, dc = 128 / F, df = 128 - dc * F;
  int c = c_first, f = f_first;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int e = threadIdx.x + i * 128;
    float val = 0.f;
    if (e < n) {
      val = xr[(size_t)c * T * F + f];
      if (gamma_log > 0.f) val = logf(__fadd_rn(1.f, __fmul_rn(gamma_log, val)));
      s += val;
    }
    v[i] = val;
    c += dc; f += df;
    if (f >= F) { f -= F; ++c; }
  }
  const float mean = block_sum(s, sh) / n;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int e = threadIdx.x + i * 128;
    if (e < n) {
      const float d = v[i] - mean;
      q += d * d;
    }
  }
  const float rstd = rsqrtf(block_sum(q, sh) / n + eps);      // (block_sum's barriers order the zero fill before the writes below)
  c = c_first; f = f_first;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int e = threadIdx.x + i * 128;
    if (e < n) {
      const float r = (v[i] - mean) * rstd * w[e] + bsh[e];
      row16[f * 8 + c] = fmt == MPA_FMT_BF16 ? __bfloat16_as_ushort(__float2bfloat16(r)) : __half_as_ushort(__float2half_rn(r));
    }
    c += dc; f += df;
    if (f >= F) { f -= F; ++c; }
  }
  __syncthreads();
  uint4* orow = out + ((size_t)b * TP + pt + t) * P + pf;
  for (int f = threadIdx.x; f < F; f += 128) orow[f] = reinterpret_cast<const uint4*>(row16)[f];
}

// frame-major: frames [C][N][F]; output rows s in [0, lead+N+trail); pad rows -> bias
template <int MAXV>
__global__ void __launch_bounds__(128) layernorm_frames_kernel(const float* __restrict__ frames, const float* __restrict__ w,
                                                               const float* __restrict__ bsh, float* __restrict__ out_f32,
                                                               uint16_t* __restrict__ out_cp8, int C, int N, int F, int lead,
                                                               int trail, int pitch, int pf, float eps, float gamma_log, int fmt) {
  __shared__ float sh[8];
  const int s = blockIdx.x;
  const int NT = lead + N + trail;
  const int n = C * F;
  const int src = s - lead;
  const bool real = (src >= 0 && src < N);
  float v[MAXV];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int e = threadIdx.x + i * 128;
    float val = 0.f;
    if (real && e < n) {
      int c = e / F, f = e - c * F;
      val = frames[((size_t)c * N + src) * F + f];
      if (gamma_log > 0.f) val = logf(__fadd_rn(1.f, __fmul_rn(gamma_log, val)));
      sum += val;
    }
    v[i] = val;
  }
  float mean = block_sum(sum, sh) / n;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int e = threadIdx.x + i * 128;
    if (e < n) {
      float d = v[i] - mean;
      q += d * d;
    }
  }
  float rstd = rsqrtf(block_sum(q, sh) / n + eps);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    int e = threadIdx.x + i * 128;
    if (e < n) {
      int c = e / F, f = e - c * F;
      float r = (v[i] - mean) * rstd * w[e] + bsh[e];
      if (out_f32) out_f32[((size_t)c * NT + s) * F + f] = r;
      if (out_cp8) {
        const size_t at = ((size_t)s * pitch + pf + f) * 8 + c;
        if (fmt == MPA_FMT_F16X3) {
          // split precision: hi plane, then the lo plane [NT][pitch][8] right behind it
          const __half hi = __float2half_rn(r);
          out_cp8[at] = __half_as_ushort(hi);
          out_cp8[(size_t)NT * pitch * 8 + at] = __half_as_ushort(__float2half_rn(r - __half2float(hi)));
        } else {
          out_cp8[at] = fmt == MPA_FMT_BF16 ? __bfloat16_as_ushort(__float2bfloat16(r)) : __half_as_ushort(__float2half_rn(r));
        }
      }
    }
  }
}

__global__ void maxpool_time_kernel(const float* __restrict__ x, const float* __restrict__ res, float* __restrict__ out,
                                    long long total, int T, int F, int k) {
  const int h = k / 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f = (int)(i % F);
    long long r = i / F;
    int t = (int)(r % T);
    long long plane = r / T;
    const float* xp = x + plane * T * F + f;
    int lo = max(0, t - h), hi = min(T - 1, t + h);
    float m = -INFINITY;
    for (int tt = lo; tt <= hi; ++tt) m = fmaxf(m, xp[(size_t)tt * F]);
    if (res) m += res[i];
    out[i] = m;
  }
}

// F % 4 == 0: four neighbouring bins per thread, 16-byte loads / stores
__global__ void maxpool_time_vec4_kernel(const float4* __restrict__ x, const float4* __restrict__ res, float4* __restrict__ out, long long total4,
                                         int T, int F4, int k) {
  const int h = k / 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F4);
    const long long r = i / F4;
    const int t = (int)(r % T);
    const float4* xp = x + (r - t) * F4 + f;
    const int lo = max(0, t - h), hi = min(T - 1, t + h);
    float4 m = xp[(size_t)lo * F4];
    for (int tt = lo + 1; tt <= hi; ++tt) {
      const float4 v = xp[(size_t)tt * F4];
      m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
    }
    if (res) {
      const float4 q = res[i];
      m.x += q.x; m.y += q.y; m.z += q.z; m.w += q.w;
    }
    out[i] = m;
  }
}

// out = dropout(maxpool_time(x)) + res  — the CNN block's MaxPool -> Dropout (-> residual add) in one pass (basic_cnns.py:376-377, 415-417);
// the mask is the one mpa_dropout_f32 draws for the same (seed, offset): counter i/4, lane i%4 of the element index
__global__ void maxpool_time_dropout_vec4_kernel(const float4* __restrict__ x, const float4* __restrict__ res, float4* __restrict__ out,
                                                 long long total4, int T, int F4, int k, DropoutArgs d) {
  const int h = k / 2;
  const unsigned long long offset = dropout_offset(d);
  const float scale = 1.f / (1.f - d.p);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F4);
    const long long r = i / F4;
    const int t = (int)(r % T);
    const float4* xp = x + (r - t) * F4 + f;
    const int lo = max(0, t - h), hi = min(T - 1, t + h);
    float4 m = xp[(size_t)lo * F4];
    for (int tt = lo + 1; tt <= hi; ++tt) {
      const float4 v = xp[(size_t)tt * F4];
      m.x = fmaxf(m.x, v.x); m.y = fmaxf(m.y, v.y); m.z = fmaxf(m.z, v.z); m.w = fmaxf(m.w, v.w);
    }
    const uint4 bits = dropout_bits(i, d.seed, offset);
    // __fmul_rn: the product is rounded before the residual is added, exactly like the separate dropout and add kernels (no FMA contraction)
    m.x = __fmul_rn(m.x, dropout_factor(bits.x, d.p, scale)); m.y = __fmul_rn(m.y, dropout_factor(bits.y, d.p, scale));
    m.z = __fmul_rn(m.z, dropout_factor(bits.z, d.p, scale)); m.w = __fmul_rn(m.w, dropout_factor(bits.w, d.p, scale));
    if (res) {
      const float4 q = res[i];
      m.x += q.x; m.y += q.y; m.z += q.z; m.w += q.w;
    }
    out[i] = m;
  }
}

__global__ void maxpool2d_kernel(const float* __restrict__ x, float* __restrict__ out, long long total, int H, int W,
                                 int Ho, int Wo, int kh, int kw, int sh, int sw) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int wo = (int)(i % Wo);
    long long r = i / Wo;
    int ho = (int)(r % Ho);
    long long plane = r / Ho;
    const float* xp = x + plane * H * W + (size_t)(ho * sh) * W + wo * sw;
    float m = -INFINITY;
    for (int a = 0; a < kh; ++a)
      for (int b = 0; b < kw; ++b) m = fmaxf(m, xp[a * W + b]);
    out[i] = m;
  }
}

__global__ void upsample_concat_kernel(const float* __restrict__ low, const float* __restrict__ skip, float* __restrict__ out,
                                       long long total, int Cl, int Hl, int Wl, int Cs, int Hs, int Ws) {
  const int Ct = Cs + Cl;
  const int Hu = 2 * Hl, Wu = 2 * Wl;
  const int dY = Hs - Hu, dX = Ws - Wu;
  const int top = dY / 2, left = dX / 2;
  const float ry = (Hu > 1) ? (float)(Hl - 1) / (float)(Hu - 1) : 0.f;
  const float rx = (Wu > 1) ? (float)(Wl - 1) / (float)(Wu - 1) : 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int w = (int)(i % Ws);
    long long r = i / Ws;
    int h = (int)(r % Hs);
    r /= Hs;
    int c = (int)(r % Ct);
    int b = (int)(r / Ct);
    float v;
    if (c < Cs) {
      v = skip[(((size_t)b * Cs + c) * Hs + h) * Ws + w];
    } else {
      int hu = h - top, wu = w - left;
      if (hu < 0 || hu >= Hu || wu < 0 || wu >= Wu) {
        v = 0.f;
      } else {
        // torch area_pixel_compute_source_index(align_corners=True): src = scale * dst
        float sy = ry * hu, sx = rx * wu;
        int y0 = (int)sy, x0 = (int)sx;
        int y1 = min(y0 + 1, Hl - 1), x1 = min(x0 + 1, Wl - 1);
        float ly = sy - y0, lx = sx - x0;
        const float* lp = low + ((size_t)b * Cl + (c - Cs)) * Hl * Wl;
        float v00 = lp[y0 * Wl + x0], v01 = lp[y0 * Wl + x1], v10 = lp[y1 * Wl + x0], v11 = lp[y1 * Wl + x1];
        v = (1.f - ly) * ((1.f - lx) * v00 + lx * v01) + ly * ((1.f - lx) * v10 + lx * v11);
      }
    }
    out[i] = v;
  }
}

__global__ void bn_apply_kernel(const float* __restrict__ x, const float* __restrict__ stats, const float* __restrict__ w,
                                const float* __restrict__ b, float* __restrict__ out, long long total, int C, int HW, float eps,
                                int act, float act_param) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int c = (int)((i / HW) % C);
    float v = (x[i] - stats[c]) * rsqrtf(stats[C + c] + eps) * w[c] + b[c];
    out[i] = apply_act(v, act, act_param);
  }
}

// HW % 4 == 0 and 16-byte aligned tensors: 4 neighbouring elements share their channel — 16-byte accesses, one index division per 4
__global__ void bn_apply_vec4_kernel(const float4* __restrict__ x, const float* __restrict__ stats, const float* __restrict__ w,
                                     const float* __restrict__ b, float4* __restrict__ out, long long total4, int C, int HW4, float eps, int act,
                                     float act_param) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)((i / HW4) % C);
    const float mean = stats[c], rstd = rsqrtf(stats[C + c] + eps), wc = w[c], bc = b[c];
    const float4 v = x[i];
    float4 o;
    o.x = apply_act((v.x - mean) * rstd * wc + bc, act, act_param);
    o.y = apply_act((v.y - mean) * rstd * wc + bc, act, act_param);
    o.z = apply_act((v.z - mean) * rstd * wc + bc, act, act_param);
    o.w = apply_act((v.w - mean) * rstd * wc + bc, act, act_param);
    out[i] = o;
  }
}

// out = act(x + bias[c]) on NCHW (in place allowed): the second pass of a split-K product whose slices met in atomics
__global__ void bias_act_kernel(const float* __restrict__ x, const float* __restrict__ bias, float* __restrict__ out, long long total, int C, int HW,
                                int act, float act_param) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)((i / HW) % C);
    out[i] = apply_act(x[i] + (bias ? bias[c] : 0.f), act, act_param);
  }
}

// grad_mul (optional, device memory): the gradient is multiplied by *grad_mul (the loss scale of fp16 training); the loss is not
__global__ void __launch_bounds__(256) bce_kernel(const float* __restrict__ yp, const float* __restrict__ yt, float* __restrict__ loss_sum,
                                                  float* __restrict__ grad, long long n, const float* __restrict__ grad_mul) {
  __shared__ float sh[8];
  float acc = 0.f;
  const float inv_n = 1.f / (float)n;
  const float gm = grad_mul ? *grad_mul : 1.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    float p = yp[i], t = yt[i];
    float lp = fmaxf(logf(p), -100.f), l1p = fmaxf(logf(1.f - p), -100.f);
    acc -= t * lp + (1.f - t) * l1p;
    if (grad) {
      // d/dp of the clamped loss: the clamp kills the gradient where log < -100 (torch: p clamped via eps 1e-12)
      float g = (p - t) / fmaxf(p * (1.f - p), 1e-12f);
      grad[i] = g * inv_n * gm;
    }
  }
  float tot = block_sum(acc, sh);
  if (threadIdx.x == 0) atomicAdd(loss_sum, tot * inv_n);
}

// X[b][c][t][f] = log(1 + gamma * in[c][(i0+b)*stride + t][f])   (dataset_context.__getitem__, hcqt_datasets.py:67-75,105-106)
__global__ void gather_patches_kernel(const float* __restrict__ in, float* __restrict__ out, long long total, int C, int NT, int F,
                                      int i0, int T, int stride, float gamma) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f = (int)(i % F);
    long long r = i / F;
    int t = (int)(r % T);
    r /= T;
    int c = (int)(r % C);
    int b = (int)(r / C);
    float v = in[((size_t)c * NT + (size_t)(i0 + b) * stride + t) * F + f];
    out[i] = gamma > 0.f ? logf(__fadd_rn(1.f, __fmul_rn(gamma, v))) : v;     // 1 + gamma*x rounded twice, as the reference's tensor expression
  }
}

// adjoint of gather_patches_kernel: one thread per input element sums the patches that read it (patch order), then applies
// d log(1 + gamma*x) / dx = gamma / (1 + gamma*x)
__global__ void gather_patches_bwd_kernel(const float* __restrict__ g_out, const float* __restrict__ in, float* __restrict__ g_in, long long total,
                                          int C, int NT, int F, int i0, int n, int T, int stride, float gamma) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F);
    const int r = (int)((i / F) % NT);
    const int c = (int)(i / ((long long)F * NT));
    // patch p covers frames [(i0+p)*stride, (i0+p)*stride + T)
    const int p0 = max(0, (r - T + 1 <= 0 ? 0 : (r - T + stride) / stride) - i0);
    const int p1 = min(n - 1, r / stride - i0);
    float acc = 0.f;
    for (int p = p0; p <= p1; ++p) acc += g_out[(((size_t)p * C + c) * T + (r - (i0 + p) * stride)) * F + f];
    if (gamma > 0.f && acc != 0.f) acc *= gamma / __fadd_rn(1.f, __fmul_rn(gamma, in[i]));
    g_in[i] = acc;
  }
}

static inline int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  long long cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace mpa

using namespace mpa;

extern "C" {

int mpa_layernorm_cf_f32(const float* x, const float* ln_w, const float* ln_b, float* out, int B, int C, int T, int F,
                         float eps, float gamma_log, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && ln_w && ln_b && out && B > 0 && C > 0 && T > 0 && F > 0, "layernorm_cf: bad argument");
  MPA_REQUIRE(C * F <= 128 * 16, "layernorm_cf: C*F=%d exceeds the 2048-element row limit", C * F);
  cudaStream_t st = (cudaStream_t)stream;
  if (C * F <= 128 * 11)
    layernorm_cf_kernel<11><<<B * T, 128, 0, st>>>(x, ln_w, ln_b, out, C, T, F, eps, gamma_log);
  else
    layernorm_cf_kernel<16><<<B * T, 128, 0, st>>>(x, ln_w, ln_b, out, C, T, F, eps, gamma_log);
  MPA_CHECK_LAUNCH("layernorm_cf");
  return MPA_OK;
}

int mpa_layernorm_cf_cp8(const float* x, const float* ln_w, const float* ln_b, void* out_cp8, int B, int C, int T, int F, int pitch, int pf,
                         int pt, float eps, float gamma_log, int fmt, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && ln_w && ln_b && out_cp8 && B > 0 && C > 0 && C <= 8 && T > 0 && F > 0 && pitch >= pf + F && pt >= 0 &&
                  (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16) && C * F <= 128 * 11,
              "layernorm_cf_cp8: bad argument (C <= 8, C*F <= 1408, 16-bit formats)");
  layernorm_cf_cp8_kernel<11><<<B * T, 128, (size_t)F * 16, (cudaStream_t)stream>>>(x, ln_w, ln_b, (uint4*)out_cp8, C, T, F, T + 2 * pt, pitch, pf,
                                                                                   pt, eps, gamma_log, fmt);
  MPA_CHECK_LAUNCH("layernorm_cf_cp8");
  return MPA_OK;
}

int mpa_layernorm_frames(const float* frames, const float* ln_w, const float* ln_b, float* out_f32, void* out_cp8, int C,
                         int N, int F, int lead, int trail, int cp8_pitch, int cp8_pf, float eps, float gamma_log, int fmt,
                         void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(frames && ln_w && ln_b && (out_f32 || out_cp8) && C > 0 && N > 0 && F > 0 && lead >= 0 && trail >= 0,
              "layernorm_frames: bad argument");
  MPA_REQUIRE(C * F <= 128 * 11, "layernorm_frames: C*F=%d exceeds 1408", C * F);
  MPA_REQUIRE(!out_cp8 || (C <= 8 && cp8_pitch >= F + cp8_pf), "layernorm_frames: CP8 output needs C<=8 and pitch>=F+pf");
  layernorm_frames_kernel<11><<<lead + N + trail, 128, 0, (cudaStream_t)stream>>>(
      frames, ln_w, ln_b, out_f32, (uint16_t*)out_cp8, C, N, F, lead, trail, cp8_pitch, cp8_pf, eps, gamma_log, fmt);
  MPA_CHECK_LAUNCH("layernorm_frames");
  return MPA_OK;
}

int mpa_gather_patches_f32(const float* in, float* out, int C, int NT, int F, int i0, int n, int T, int stride, float gamma_log,
                           void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(in && out && C > 0 && F > 0 && n > 0 && T > 0 && stride > 0 && i0 >= 0, "gather_patches: bad argument");
  MPA_REQUIRE((long long)(i0 + n - 1) * stride + T <= NT, "gather_patches: patch range exceeds the %d input frames", NT);
  long long total = (long long)n * C * T * F;
  gather_patches_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(in, out, total, C, NT, F, i0, T, stride, gamma_log);
  MPA_CHECK_LAUNCH("gather_patches");
  return MPA_OK;
}

int mpa_gather_patches_bwd_f32(const float* g_out, const float* in, float* g_in, int C, int NT, int F, int i0, int n, int T, int stride,
                               float gamma_log, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(g_out && g_in && (in || gamma_log <= 0.f) && C > 0 && F > 0 && n > 0 && T > 0 && stride > 0 && i0 >= 0,
              "gather_patches_bwd: bad argument");
  MPA_REQUIRE((long long)(i0 + n - 1) * stride + T <= NT, "gather_patches_bwd: patch range exceeds the %d input frames", NT);
  long long total = (long long)C * NT * F;
  gather_patches_bwd_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(g_out, in, g_in, total, C, NT, F, i0, n, T, stride,
                                                                                    gamma_log);
  MPA_CHECK_LAUNCH("gather_patches_bwd");
  return MPA_OK;
}

int mpa_maxpool_time_f32(const float* x, const float* res, float* out, int B, int C, int T, int F, int k, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && B > 0 && C > 0 && T > 0 && F > 0 && k >= 1 && (k & 1), "maxpool_time: bad argument");
  long long total = (long long)B * C * T * F;
  if (F % 4 == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)res & 15) == 0) {
    long long g = (total / 4 + 255) / 256;
    maxpool_time_vec4_kernel<<<(unsigned)(g > 148LL * 64 ? 148LL * 64 : g), 256, 0, (cudaStream_t)stream>>>(
        (const float4*)x, (const float4*)res, (float4*)out, total / 4, T, F / 4, k);
    MPA_CHECK_LAUNCH("maxpool_time_vec4");
    return MPA_OK;
  }
  maxpool_time_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, res, out, total, T, F, k);
  MPA_CHECK_LAUNCH("maxpool_time");
  return MPA_OK;
}

int mpa_maxpool_time_dropout_f32(const float* x, const float* res, float* out, int B, int C, int T, int F, int k, float p,
                                 unsigned long long seed, unsigned long long offset, const long long* step_dev, unsigned long long step_mul,
                                 void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && B > 0 && C > 0 && T > 0 && F > 0 && k >= 1 && (k & 1) && p >= 0.f && p < 1.f, "maxpool_time_dropout: bad argument");
  MPA_REQUIRE(F % 4 == 0 && ((uintptr_t)x & 15) == 0 && ((uintptr_t)out & 15) == 0 && ((uintptr_t)res & 15) == 0,
              "maxpool_time_dropout: F must be a multiple of 4 and the tensors 16-byte aligned");
  const long long total = (long long)B * C * T * F;
  long long g = (total / 4 + 255) / 256;
  DropoutArgs d{p, seed, offset, step_dev, step_mul};
  maxpool_time_dropout_vec4_kernel<<<(unsigned)(g > 148LL * 64 ? 148LL * 64 : g), 256, 0, (cudaStream_t)stream>>>(
      (const float4*)x, (const float4*)res, (float4*)out, total / 4, T, F / 4, k, d);
  MPA_CHECK_LAUNCH("maxpool_time_dropout");
  return MPA_OK;
}

int mpa_maxpool2d_f32(const float* x, float* out, int B, int C, int H, int W, int kh, int kw, int sh, int sw, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && B > 0 && C > 0 && H >= kh && W >= kw && kh > 0 && kw > 0 && sh > 0 && sw > 0, "maxpool2d: bad argument");
  int Ho = (H - kh) / sh + 1, Wo = (W - kw) / sw + 1;
  long long total = (long long)B * C * Ho * Wo;
  maxpool2d_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, out, total, H, W, Ho, Wo, kh, kw, sh, sw);
  MPA_CHECK_LAUNCH("maxpool2d");
  return MPA_OK;
}

int mpa_upsample2x_concat_f32(const float* low, const float* skip, float* out, int B, int Cl, int Hl, int Wl, int Cs,
                              int Hs, int Ws, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(low && skip && out && B > 0 && Cl > 0 && Cs > 0 && Hs >= 2 * Hl && Ws >= 2 * Wl, "upsample2x_concat: bad argument");
  long long total = (long long)B * (Cs + Cl) * Hs * Ws;
  upsample_concat_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(low, skip, out, total, Cl, Hl, Wl, Cs, Hs, Ws);
  MPA_CHECK_LAUNCH("upsample2x_concat");
  return MPA_OK;
}

int mpa_bn_stats_f32(const float* x, float* stats, int B, int C, int HW, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && stats && B > 0 && C > 0 && HW > 0, "bn_stats: bad argument");
  {
    int rc = bn_stats_launch(x, stats, B, C, HW, (cudaStream_t)stream);
    if (rc != MPA_OK) return rc;
  }
  MPA_CHECK_LAUNCH("bn_stats");
  return MPA_OK;
}

int mpa_bn_apply_f32(const float* x, const float* stats, const float* w, const float* b, float* out, int B, int C, int HW,
                     float eps, int act, float act_param, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && stats && w && b && out && B > 0 && C > 0 && HW > 0, "bn_apply: bad argument");
  long long total = (long long)B * C * HW;
  if (HW % 4 == 0 && ((((uintptr_t)x | (uintptr_t)out) & 15) == 0))
    bn_apply_vec4_kernel<<<grid_for(total / 4, 256), 256, 0, (cudaStream_t)stream>>>((const float4*)x, stats, w, b, (float4*)out, total / 4, C, HW / 4,
                                                                                      eps, act, act_param);
  else
    bn_apply_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, stats, w, b, out, total, C, HW, eps, act, act_param);
  MPA_CHECK_LAUNCH("bn_apply");
  return MPA_OK;
}

int mpa_bias_act_f32(const float* x, const float* bias, float* out, int B, int C, int HW, int act, float act_param, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && B > 0 && C > 0 && HW > 0, "bias_act: bad argument");
  const long long total = (long long)B * C * HW;
  bias_act_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, bias, out, total, C, HW, act, act_param);
  MPA_CHECK_LAUNCH("bias_act");
  return MPA_OK;
}

int mpa_bce_fwd_bwd_f32(const float* y_pred, const float* y_true, float* loss_sum, float* grad_pred, long long n, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(y_pred && y_true && loss_sum && n > 0, "bce: bad argument");
  cudaMemsetAsync(loss_sum, 0, sizeof(float), (cudaStream_t)stream);
  bce_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(y_pred, y_true, loss_sum, grad_pred, n, nullptr);
  MPA_CHECK_LAUNCH("bce");
  return MPA_OK;
}

int mpa_bce_fwd_bwd_scaled_f32(const float* y_pred, const float* y_true, float* loss_sum, float* grad_pred, long long n, const float* loss_scale,
                               void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(y_pred && y_true && loss_sum && grad_pred && loss_scale && n > 0, "bce_scaled: bad argument");
  cudaMemsetAsync(loss_sum, 0, sizeof(float), (cudaStream_t)stream);
  bce_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(y_pred, y_true, loss_sum, grad_pred, n, loss_scale);
  MPA_CHECK_LAUNCH("bce_scaled");
  return MPA_OK;
}

}  // extern "C"
