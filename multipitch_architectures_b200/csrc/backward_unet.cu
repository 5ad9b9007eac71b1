// Backward kernels of the U-Net / SAUnet family (training configuration 5, SURVEY.md 8a N4/N5/N8/N9), fp32 NCHW.
// Reference semantics: train-mode BatchNorm2d (batch statistics, biased variance) + ReLU, MaxPool2d floor mode with
// first-arg-max routing, bilinear x2 (align_corners=True) + pad + concat, and the batch-axis transformer encoder layer
// (unet_cnns.py:30-159) exactly as autograd differentiates the reference modules.
#include "common.cuh"

namespace mpa {

static inline int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  long long cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

__device__ __forceinline__ float block_sum256(float v, float* sh) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) r += sh[i];
  return r;
}

// ---- BatchNorm2d(train) + ReLU backward -------------------------------------------------------------------------
// pass 2: dx = w * rstd * (dy' - s1/N - xhat * s2/N)
__global__ void bn_relu_bwd_apply_kernel(const float* __restrict__ x, const float* __restrict__ out, const float* __restrict__ dy,
                                         const float* __restrict__ stats, const float* __restrict__ w, const float* __restrict__ sums, float eps,
                                         float* __restrict__ dx, long long total, int C, int HW, float inv_n, int relu) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)((i / HW) % C);
    const float rstd = rsqrtf(stats[C + c] + eps);
    const float xh = (x[i] - stats[c]) * rstd;
    float g = dy[i];
    if (relu && !(out[i] > 0.f)) g = 0.f;
    dx[i] = w[c] * rstd * (g - sums[c] * inv_n - xh * sums[C + c] * inv_n);
  }
}

// HW % 4 == 0 and 16-byte aligned tensors: 16-byte accesses, one index division per 4 elements (same arithmetic per element)
__global__ void bn_relu_bwd_apply_vec4_kernel(const float4* __restrict__ x, const float4* __restrict__ out, const float4* __restrict__ dy,
                                              const float* __restrict__ stats, const float* __restrict__ w, const float* __restrict__ sums,
                                              float eps, float4* __restrict__ dx, long long total4, int C, int HW4, float inv_n, int relu) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total4; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)((i / HW4) % C);
    const float mean = stats[c], rstd = rsqrtf(stats[C + c] + eps), wc = w[c], s1 = sums[c], s2 = sums[C + c];
    const float4 xv = x[i];
    float4 g = dy[i];
    if (relu) {
      const float4 o = out[i];
      if (!(o.x > 0.f)) g.x = 0.f;
      if (!(o.y > 0.f)) g.y = 0.f;
      if (!(o.z > 0.f)) g.z = 0.f;
      if (!(o.w > 0.f)) g.w = 0.f;
    }
    float4 r;
    r.x = wc * rstd * (g.x - s1 * inv_n - (xv.x - mean) * rstd * s2 * inv_n);
    r.y = wc * rstd * (g.y - s1 * inv_n - (xv.y - mean) * rstd * s2 * inv_n);
    r.z = wc * rstd * (g.z - s1 * inv_n - (xv.z - mean) * rstd * s2 * inv_n);
    r.w = wc * rstd * (g.w - s1 * inv_n - (xv.w - mean) * rstd * s2 * inv_n);
    dx[i] = r;
  }
}

// ---- BatchNorm2d(eval: running statistics) + ReLU backward: dx = w * rstd * dy' (nothing depends on the batch) ------------------
__global__ void bn_relu_bwd_frozen_apply_kernel(const float* __restrict__ out, const float* __restrict__ dy, const float* __restrict__ stats,
                                                const float* __restrict__ w, float eps, float* __restrict__ dx, long long total, int C, int HW,
                                                int relu) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)((i / HW) % C);
    float g = dy[i];
    if (relu && !(out[i] > 0.f)) g = 0.f;
    dx[i] = w[c] * rsqrtf(stats[C + c] + eps) * g;
  }
}

// ---- MaxPool2d backward, any kernel / stride, no padding, floor mode; first arg-max in row-major window order ---------
__global__ void maxpool2d_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g_out, float* __restrict__ g_in, long long total, int H,
                                     int W, int Ho, int Wo, int kh, int kw, int sh, int sw) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int w = (int)(i % W);
    long long r = i / W;
    const int h = (int)(r % H);
    const long long plane = r / H;
    const float* xp = x + plane * H * W;
    const float mine = xp[h * W + w];
    float acc = 0.f;
    const int ho_lo = max(0, (h - kh + sh) / sh), ho_hi = min(Ho - 1, h / sh);
    const int wo_lo = max(0, (w - kw + sw) / sw), wo_hi = min(Wo - 1, w / sw);
    for (int ho = ho_lo; ho <= ho_hi; ++ho) {
      if (h < ho * sh || h >= ho * sh + kh) continue;
      for (int wo = wo_lo; wo <= wo_hi; ++wo) {
        if (w < wo * sw || w >= wo * sw + kw) continue;
        bool win = true;
        for (int a = 0; a < kh && win; ++a)
          for (int b = 0; b < kw; ++b) {
            const int hh = ho * sh + a, ww = wo * sw + b;
            const float v = xp[hh * W + ww];
            const bool earlier = (hh < h) || (hh == h && ww < w);
            if (hh == h && ww == w) continue;
            if (earlier ? (v >= mine) : (v > mine)) {
              win = false;
              break;
            }
          }
        if (win) acc += g_out[(plane * Ho + ho) * Wo + wo];
      }
    }
    g_in[i] = acc;
  }
}

// ---- unet_up_concat_padding backward: g_cat [B,Cs+Cl,Hs,Ws] -> g_skip [B,Cs,Hs,Ws] (+=), g_low [B,Cl,Hl,Wl] ----------
__global__ void upconcat_bwd_skip_kernel(const float* __restrict__ g_cat, float* __restrict__ g_skip, long long total, int Cs, int Ct, int HW,
                                         int accumulate) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(i % HW);
    long long r = i / HW;
    const int c = (int)(r % Cs);
    const long long b = r / Cs;
    const float g = g_cat[((size_t)b * Ct + c) * HW + p];
    g_skip[i] = accumulate ? g_skip[i] + g : g;
  }
}
__global__ void upconcat_bwd_low_kernel(const float* __restrict__ g_cat, float* __restrict__ g_low, long long total, int Cl, int Hl, int Wl, int Cs,
                                        int Hs, int Ws) {
  const int Ct = Cs + Cl, Hu = 2 * Hl, Wu = 2 * Wl;
  const int top = (Hs - Hu) / 2, left = (Ws - Wu) / 2;
  const float ry = Hu > 1 ? (float)(Hl - 1) / (float)(Hu - 1) : 0.f;
  const float rx = Wu > 1 ? (float)(Wl - 1) / (float)(Wu - 1) : 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % Wl);
    long long r = i / Wl;
    const int y = (int)(r % Hl);
    r /= Hl;
    const int c = (int)(r % Cl);
    const long long b = r / Cl;
    const float* gp = g_cat + ((size_t)b * Ct + Cs + c) * Hs * Ws;
    // up-sampled rows hu whose source interval touches low row y: source = ry*hu in (y-1, y+1)
    const int hu_lo = ry > 0.f ? max(0, (int)floorf((y - 1) / ry)) : 0;
    const int hu_hi = ry > 0.f ? min(Hu - 1, (int)ceilf((y + 1) / ry)) : Hu - 1;
    const int wu_lo = rx > 0.f ? max(0, (int)floorf((x - 1) / rx)) : 0;
    const int wu_hi = rx > 0.f ? min(Wu - 1, (int)ceilf((x + 1) / rx)) : Wu - 1;
    float acc = 0.f;
    for (int hu = hu_lo; hu <= hu_hi; ++hu) {
      const float sy = ry * hu;
      const int y0 = (int)sy, y1 = min(y0 + 1, Hl - 1);
      const float ly = sy - y0;
      float wy = 0.f;
      if (y0 == y) wy += 1.f - ly;
      if (y1 == y) wy += ly;
      if (wy == 0.f) continue;
      for (int wu = wu_lo; wu <= wu_hi; ++wu) {
        const float sx = rx * wu;
        const int x0 = (int)sx, x1 = min(x0 + 1, Wl - 1);
        const float lx = sx - x0;
        float wx = 0.f;
        if (x0 == x) wx += 1.f - lx;
        if (x1 == x) wx += lx;
        if (wx != 0.f) acc = fmaf(wy * wx, gp[(size_t)(hu + top) * Ws + wu + left], acc);
      }
    }
    g_low[i] = acc;
  }
}

// ---- generic fp32 GEMMs for the encoder-layer backward: C[M,N] (+)= op(A) * op(B) -------------------------------------
// mode 0: C = A[M,K] * B[K,N]     (NN)      mode 1: C = A[K,M]^T * B[K,N]   (TN)
__global__ void __launch_bounds__(256) gemm_generic_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ C, int M,
                                                           int N, int K, int mode, int accumulate) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4] = {};
  // split-K over blockIdx.z: the slices are combined with atomicAdd (C pre-zeroed unless accumulating)
  const int kchunk = (((K + (int)gridDim.z - 1) / (int)gridDim.z) + 15) / 16 * 16;
  const int k_begin = blockIdx.z * kchunk, k_end = min(K, k_begin + kchunk);
  for (int k0 = k_begin; k0 < k_end; k0 += 16) {
    for (int e = threadIdx.x; e < 64 * 16; e += 256) {
      if (mode == 0) {
        const int kk = e & 15, r = e >> 4;
        const int m = m0 + r, k = k0 + kk;
        As[kk][r] = (m < M && k < k_end) ? A[(size_t)m * K + k] : 0.f;
      } else {
        const int r = e & 63, kk = e >> 6;
        const int m = m0 + r, k = k0 + kk;
        As[kk][r] = (m < M && k < k_end) ? A[(size_t)k * M + m] : 0.f;
      }
      const int r = e & 63, kk = e >> 6;
      const int n = n0 + r, k = k0 + kk;
      Bs[kk][r] = (n < N && k < k_end) ? Bm[(size_t)k * N + n] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      const size_t idx = (size_t)m * N + n;
      if (gridDim.z > 1) atomicAdd(&C[idx], acc[i][j]);
      else C[idx] = accumulate ? C[idx] + acc[i][j] : acc[i][j];
    }
  }
}

// column sums: out[n] = sum_m A[m,n].  grid (column blocks of 32, row slices): few-column matrices (E = 128 columns, B*S = 1300 rows) ran on 4
// CTAs; the row slices meet in atomics (out pre-zeroed) when there is more than one
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ A, float* __restrict__ out, int M, int N) {
  const int n = blockIdx.x * 32 + (threadIdx.x & 31);
  const int slice = threadIdx.x >> 5;
  __shared__ float sh[8][33];
  const int per = (M + gridDim.y - 1) / gridDim.y;
  const int m0 = blockIdx.y * per, m1 = min(M, m0 + per);
  float s = 0.f;
  if (n < N)
    for (int m = m0 + slice; m < m1; m += 8) s += A[(size_t)m * N + n];
  sh[slice][threadIdx.x & 31] = s;
  __syncthreads();
  if (slice == 0 && n < N) {
    float t = 0.f;
    for (int i = 0; i < 8; ++i) t += sh[i][threadIdx.x & 31];
    if (gridDim.y > 1) atomicAdd(&out[n], t);
    else out[n] = t;
  }
}

// LayerNorm(E) backward per token: y = LN(u) * w + b.  g_u (may alias g_y), and per-CTA partial dw/db via atomics.
__global__ void __launch_bounds__(128) ln_bwd_kernel(const float* __restrict__ u, const float* __restrict__ g_y, const float* __restrict__ w,
                                                     float* __restrict__ g_u, float* __restrict__ g_w, float* __restrict__ g_b, int E, float eps) {
  __shared__ float sh[4];
  const long long tok = blockIdx.x;
  float v[8], g[8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int e = threadIdx.x + i * 128;
    v[i] = e < E ? u[tok * E + e] : 0.f;
    s += v[i];
  }
  const float mean = block_sum256(s, sh) / E;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int e = threadIdx.x + i * 128;
    if (e < E) {
      const float d = v[i] - mean;
      q += d * d;
    }
  }
  const float rstd = rsqrtf(block_sum256(q, sh) / E + eps);
  float a1 = 0.f, a2 = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int e = threadIdx.x + i * 128;
    g[i] = 0.f;
    if (e < E) {
      const float xh = (v[i] - mean) * rstd;
      const float gy = g_y[tok * E + e];
      atomicAdd(&g_w[e], gy * xh);
      atomicAdd(&g_b[e], gy);
      g[i] = gy * w[e];
      a1 += g[i];
      a2 += g[i] * xh;
      v[i] = xh;
    }
  }
  a1 = block_sum256(a1, sh) / E;
  a2 = block_sum256(a2, sh) / E;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int e = threadIdx.x + i * 128;
    if (e < E) g_u[tok * E + e] = rstd * (g[i] - a1 - v[i] * a2);
  }
}

// batch-axis attention backward; one block per (s, head).  qkv [(b*S+s)][3E], g_o [(b*S+s)][E] -> g_qkv.
// The B x B score matrix of one (token position, head) lives in shared memory; every stage is a data-parallel pass over (b1, b2) pairs or
// (b, k) outputs with a fixed summation order — no atomics, bit-reproducible:
//   P = softmax_b2(Q K^T / sqrt(hd));  dP = dO V^T;  dS = P * (dP - rowsum(P * dP)) / sqrt(hd);  dQ = dS K;  dK = dS^T Q;  dV = P^T dO.
__global__ void __launch_bounds__(256) batch_axis_attention_bwd_kernel(const float* __restrict__ qkv, const float* __restrict__ g_o,
                                                                       float* __restrict__ g_qkv, int B, int S, int E, int H) {
  extern __shared__ float sm[];
  const int hd = E / H;
  const int s = blockIdx.x / H, h = blockIdx.x % H;
  float* Q = sm;                       // [B][hd]
  float* Km = Q + (size_t)B * hd;
  float* V = Km + (size_t)B * hd;
  float* dO = V + (size_t)B * hd;
  float* P = dO + (size_t)B * hd;      // [B][B] probabilities
  float* dS = P + (size_t)B * B;       // [B][B] dP, then dS
  float* rowv = dS + (size_t)B * B;    // [B]
  const int nt = blockDim.x;
  for (int e = threadIdx.x; e < B * hd; e += nt) {
    const int b = e / hd, d = e - b * hd;
    const float* row = qkv + ((size_t)b * S + s) * 3 * E + h * hd + d;
    Q[e] = row[0];
    Km[e] = row[E];
    V[e] = row[2 * E];
    dO[e] = g_o[((size_t)b * S + s) * E + h * hd + d];
  }
  __syncthreads();
  const float sc = rsqrtf((float)hd);
  for (int e = threadIdx.x; e < B * B; e += nt) {
    const int b1 = e / B, b2 = e - b1 * B;
    float d = 0.f, dp = 0.f;
    for (int k = 0; k < hd; ++k) {
      d = fmaf(Q[b1 * hd + k], Km[b2 * hd + k], d);
      dp = fmaf(dO[b1 * hd + k], V[b2 * hd + k], dp);
    }
    P[e] = d * sc;
    dS[e] = dp;
  }
  __syncthreads();
  for (int b1 = threadIdx.x; b1 < B; b1 += nt) {
    float mx = -INFINITY;
    for (int b2 = 0; b2 < B; ++b2) mx = fmaxf(mx, P[b1 * B + b2]);
    float den = 0.f;
    for (int b2 = 0; b2 < B; ++b2) {
      const float pr = expf(P[b1 * B + b2] - mx);
      P[b1 * B + b2] = pr;
      den += pr;
    }
    float dot = 0.f;     // sum_b2 P * dP
    for (int b2 = 0; b2 < B; ++b2) {
      const float pr = P[b1 * B + b2] / den;
      P[b1 * B + b2] = pr;
      dot = fmaf(pr, dS[b1 * B + b2], dot);
    }
    rowv[b1] = dot;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < B * B; e += nt) dS[e] = P[e] * (dS[e] - rowv[e / B]) * sc;
  __syncthreads();
  for (int e = threadIdx.x; e < B * hd; e += nt) {
    const int b = e / hd, k = e - b * hd;
    float dq = 0.f, dk = 0.f, dv = 0.f;
    for (int o = 0; o < B; ++o) {
      dq = fmaf(dS[b * B + o], Km[o * hd + k], dq);
      dk = fmaf(dS[o * B + b], Q[o * hd + k], dk);
      dv = fmaf(P[o * B + b], dO[o * hd + k], dv);
    }
    float* row = g_qkv + ((size_t)b * S + s) * 3 * E + h * hd + k;
    row[0] = dq;
    row[E] = dk;
    row[2 * E] = dv;
  }
}

// tokens <-> NCHW helpers for gradients: g_tok[(b*S+s)*E+e] = g_nchw[b,e,s]   and the transpose (optionally accumulating)
__global__ void nchw_to_tok_kernel(const float* __restrict__ x, float* __restrict__ tok, long long total, int E, int S) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int e = (int)(i % E);
    const long long r = i / E;
    const int s = (int)(r % S);
    const long long b = r / S;
    tok[i] = x[((size_t)b * E + e) * S + s];
  }
}
__global__ void tok_to_nchw_kernel(const float* __restrict__ tok, float* __restrict__ x, long long total, int E, int S) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int s = (int)(i % S);
    const long long r = i / S;
    const int e = (int)(r % E);
    const long long b = r / E;
    x[i] = tok[((size_t)b * S + s) * E + e];
  }
}

// CrossEntropyLoss(mean) * scale over K classes, target class = number of active labels of the item (PUnet degree-of-polyphony
// head: n_target = sum(labels, -1).long(), RETRAIN4_exp195f...rerun1.py:343-345).  One warp per item.  grad_mul (optional, device
// memory): the gradient is multiplied by *grad_mul (the loss scale of fp16 training); the loss is not.
__global__ void __launch_bounds__(128) ce_count_kernel(const float* __restrict__ logits, const float* __restrict__ y_true, float* __restrict__ loss_sum,
                                                       float* __restrict__ grad, int B, int K, int P, float scale, const float* __restrict__ grad_mul) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  float cnt = 0.f;
  for (int i = lane; i < P; i += 32) cnt += y_true[(size_t)b * P + i];
  cnt = warp_sum(cnt);
  int cls = (int)cnt;                       // .long() truncates
  cls = cls < 0 ? 0 : (cls >= K ? K - 1 : cls);
  float mx = -INFINITY;
  for (int k = lane; k < K; k += 32) mx = fmaxf(mx, logits[(size_t)b * K + k]);
  mx = warp_max(mx);
  float den = 0.f;
  for (int k = lane; k < K; k += 32) den += expf(logits[(size_t)b * K + k] - mx);
  den = warp_sum(den);
  const float lse = mx + logf(den);
  if (lane == 0) atomicAdd(loss_sum, (lse - logits[(size_t)b * K + cls]) * scale / B);
  if (grad) {
    const float gm = grad_mul ? *grad_mul : 1.f;
    for (int k = lane; k < K; k += 32)
      grad[(size_t)b * K + k] = (expf(logits[(size_t)b * K + k] - lse) - (k == cls ? 1.f : 0.f)) * scale / B * gm;
  }
}

}  // namespace mpa

using namespace mpa;

extern "C" {

int mpa_bn_relu_bwd_f32(const float* x, const float* out, const float* dy, const float* stats, const float* w, float* dx, float* dw, float* db,
                        float* scratch2c, int B, int C, int HW, float eps, int relu, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && dy && stats && w && dx && dw && db && scratch2c && B > 0 && C > 0 && HW > 0, "bn_relu_bwd: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  {
    int rc = bn_bwd_sums_launch(x, out, dy, stats, eps, scratch2c, dw, db, B, C, HW, relu, st);
    if (rc != MPA_OK) return rc;
  }
  MPA_CHECK_LAUNCH("bn_relu_bwd_reduce");
  const long long total = (long long)B * C * HW;
  if (HW % 4 == 0 && ((((uintptr_t)x | (uintptr_t)out | (uintptr_t)dy | (uintptr_t)dx) & 15) == 0))
    bn_relu_bwd_apply_vec4_kernel<<<grid_for(total / 4, 256), 256, 0, st>>>((const float4*)x, (const float4*)out, (const float4*)dy, stats, w, scratch2c,
                                                                             eps, (float4*)dx, total / 4, C, HW / 4, 1.f / ((float)B * HW), relu);
  else
    bn_relu_bwd_apply_kernel<<<grid_for(total, 256), 256, 0, st>>>(x, out, dy, stats, w, scratch2c, eps, dx, total, C, HW, 1.f / ((float)B * HW), relu);
  MPA_CHECK_LAUNCH("bn_relu_bwd_apply");
  return MPA_OK;
}

int mpa_bn_relu_bwd_frozen_f32(const float* x, const float* out, const float* dy, const float* stats, const float* w, float* dx, float* dw, float* db,
                               float* d_conv_bias, float* scratch2c, int B, int C, int HW, float eps, int relu, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && dy && stats && w && dx && dw && db && scratch2c && B > 0 && C > 0 && HW > 0, "bn_relu_bwd_frozen: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  {
    // d beta = sum dy', d gamma = sum dy' * xhat with xhat formed from the running statistics
    int rc = bn_bwd_sums_launch(x, out, dy, stats, eps, scratch2c, dw, db, B, C, HW, relu, st);
    if (rc != MPA_OK) return rc;
  }
  MPA_CHECK_LAUNCH("bn_relu_bwd_frozen_reduce");
  const long long total = (long long)B * C * HW;
  bn_relu_bwd_frozen_apply_kernel<<<grid_for(total, 256), 256, 0, st>>>(out, dy, stats, w, eps, dx, total, C, HW, relu);
  MPA_CHECK_LAUNCH("bn_relu_bwd_frozen_apply");
  if (d_conv_bias) {
    int rc = channel_sum_launch(dx, d_conv_bias, B, C, HW, st);
    if (rc != MPA_OK) return rc;
    MPA_CHECK_LAUNCH("bn_relu_bwd_frozen_conv_bias");
  }
  return MPA_OK;
}

int mpa_maxpool2d_bwd_f32(const float* x, const float* g_out, float* g_in, int B, int C, int H, int W, int kh, int kw, int sh, int sw, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && g_out && g_in && B > 0 && C > 0 && H >= kh && W >= kw && kh > 0 && kw > 0 && sh > 0 && sw > 0, "maxpool2d_bwd: bad argument");
  const int Ho = (H - kh) / sh + 1, Wo = (W - kw) / sw + 1;
  const long long total = (long long)B * C * H * W;
  maxpool2d_bwd_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, g_out, g_in, total, H, W, Ho, Wo, kh, kw, sh, sw);
  MPA_CHECK_LAUNCH("maxpool2d_bwd");
  return MPA_OK;
}

int mpa_upsample2x_concat_bwd_f32(const float* g_cat, float* g_skip, int accumulate_skip, float* g_low, int B, int Cl, int Hl, int Wl, int Cs,
                                  int Hs, int Ws, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(g_cat && g_skip && g_low && B > 0 && Cl > 0 && Cs > 0 && Hs >= 2 * Hl && Ws >= 2 * Wl, "upsample2x_concat_bwd: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  long long t1 = (long long)B * Cs * Hs * Ws;
  upconcat_bwd_skip_kernel<<<grid_for(t1, 256), 256, 0, st>>>(g_cat, g_skip, t1, Cs, Cs + Cl, Hs * Ws, accumulate_skip);
  MPA_CHECK_LAUNCH("upconcat_bwd_skip");
  long long t2 = (long long)B * Cl * Hl * Wl;
  upconcat_bwd_low_kernel<<<grid_for(t2, 256), 256, 0, st>>>(g_cat, g_low, t2, Cl, Hl, Wl, Cs, Hs, Ws);
  MPA_CHECK_LAUNCH("upconcat_bwd_low");
  return MPA_OK;
}

int mpa_gemm_f32(const float* A, const float* Bm, float* C, int M, int N, int K, int mode, int accumulate, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(A && Bm && C && M > 0 && N > 0 && K > 0 && (mode == 0 || mode == 1), "gemm: bad argument");
  {
    const int blocks = ceil_div(N, 64) * ceil_div(M, 64);
    int ks = 1;
    if (blocks < 148 && K >= 512) {
      ks = 296 / blocks;
      if (ks > K / 128) ks = K / 128;
      if (ks > 32) ks = 32;
      if (ks < 1) ks = 1;
    }
    if (ks > 1 && !accumulate) cudaMemsetAsync(C, 0, sizeof(float) * (size_t)M * N, (cudaStream_t)stream);
    gemm_generic_kernel<<<dim3(ceil_div(N, 64), ceil_div(M, 64), ks), 256, 0, (cudaStream_t)stream>>>(A, Bm, C, M, N, K, mode, accumulate);
  }
  MPA_CHECK_LAUNCH("gemm_generic");
  return MPA_OK;
}

int mpa_colsum_f32(const float* A, float* out, int M, int N, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(A && out && M > 0 && N > 0, "colsum: bad argument");
  const int cb = ceil_div(N, 32);
  int slices = cb >= 148 ? 1 : ceil_div(296, cb);
  if (slices > ceil_div(M, 64)) slices = ceil_div(M, 64);
  if (slices > 1) cudaMemsetAsync(out, 0, sizeof(float) * N, (cudaStream_t)stream);
  colsum_kernel<<<dim3(cb, slices), 256, 0, (cudaStream_t)stream>>>(A, out, M, N);
  MPA_CHECK_LAUNCH("colsum");
  return MPA_OK;
}

int mpa_layernorm_tok_bwd_f32(const float* u, const float* g_y, const float* w, float* g_u, float* g_w, float* g_b, long long n_tok, int E, float eps,
                              void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(u && g_y && w && g_u && g_w && g_b && n_tok > 0 && E > 0 && E <= 1024, "layernorm_tok_bwd: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(g_w, 0, sizeof(float) * E, st);
  cudaMemsetAsync(g_b, 0, sizeof(float) * E, st);
  ln_bwd_kernel<<<(unsigned)n_tok, 128, 0, st>>>(u, g_y, w, g_u, g_w, g_b, E, eps);
  MPA_CHECK_LAUNCH("ln_bwd");
  return MPA_OK;
}

int mpa_batch_axis_attention_bwd_f32(const float* qkv, const float* g_o, float* g_qkv, int B, int S, int E, int num_heads, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(qkv && g_o && g_qkv && B > 0 && S > 0 && E > 0 && num_heads > 0 && E % num_heads == 0, "attention_bwd: bad argument");
  const int hd = E / num_heads;
  const size_t smem = ((size_t)4 * B * hd + (size_t)2 * B * B + B) * sizeof(float);
  MPA_REQUIRE(smem <= 48 * 1024, "attention_bwd: batch %d too large for the shared-memory tile", B);
  batch_axis_attention_bwd_kernel<<<S * num_heads, 256, smem, (cudaStream_t)stream>>>(qkv, g_o, g_qkv, B, S, E, num_heads);
  MPA_CHECK_LAUNCH("attention_bwd");
  return MPA_OK;
}

int mpa_nchw_tokens_f32(const float* src, float* dst, int B, int E, int S, int to_tokens, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(src && dst && B > 0 && E > 0 && S > 0, "nchw_tokens: bad argument");
  const long long total = (long long)B * E * S;
  if (to_tokens)
    nchw_to_tok_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, total, E, S);
  else
    tok_to_nchw_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(src, dst, total, E, S);
  MPA_CHECK_LAUNCH("nchw_tokens");
  return MPA_OK;
}

int mpa_ce_count_fwd_bwd_f32(const float* logits, const float* y_true, float* loss_sum, float* grad_logits, int B, int K, int P, float scale,
                             int accumulate_loss, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(logits && y_true && loss_sum && B > 0 && K > 0 && P > 0, "ce_count: bad argument");
  if (!accumulate_loss) cudaMemsetAsync(loss_sum, 0, sizeof(float), (cudaStream_t)stream);
  ce_count_kernel<<<ceil_div(B, 4), 128, 0, (cudaStream_t)stream>>>(logits, y_true, loss_sum, grad_logits, B, K, P, scale, nullptr);
  MPA_CHECK_LAUNCH("ce_count");
  return MPA_OK;
}

int mpa_ce_count_fwd_bwd_scaled_f32(const float* logits, const float* y_true, float* loss_sum, float* grad_logits, int B, int K, int P, float scale,
                                    int accumulate_loss, const float* loss_scale, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(logits && y_true && loss_sum && grad_logits && loss_scale && B > 0 && K > 0 && P > 0, "ce_count_scaled: bad argument");
  if (!accumulate_loss) cudaMemsetAsync(loss_sum, 0, sizeof(float), (cudaStream_t)stream);
  ce_count_kernel<<<ceil_div(B, 4), 128, 0, (cudaStream_t)stream>>>(logits, y_true, loss_sum, grad_logits, B, K, P, scale, loss_scale);
  MPA_CHECK_LAUNCH("ce_count_scaled");
  return MPA_OK;
}

}  // extern "C"
