// Element-wise training stages of the CNN blocks directly on the 16-bit CP8 planes the tensor-core convolutions read and write:
//   forward   z  = Dropout(MaxPool((3,1), stride 1, pad (1,0))(a))                 (basic_cnns.py:172-175, 376-377)
//   backward  ga = act'(a) * sum_t [first arg-max of window t == .] * mask * g[t]
//   bias gradient = per-channel sum of ga
// so that no nchw<->CP8 converter runs between two convolutions of a training step.  The planes hold the same 16-bit values the fp32
// NCHW kernels of elementwise.cu / backward.cu see behind the converters, every sum is formed in fp32 in the same order and rounded
// once on the store, and the dropout mask uses the SAME convention (Philox counter i/4, lane i%4 of the NCHW element index
// i = ((b*C + c)*T + t)*F + f) — outputs are bit-identical to the converter path (tests/test_gpu_training.py).
// One thread owns 4 neighbouring bins x 8 channels (forward) or x 4 channels (backward, to stay clear of register spills): one Philox
// draw per channel serves its 4 bins.  Both kernels walk down a segment of the T rows of their column with the window in registers, so
// every row is loaded once: forward reads a and writes z, backward reads a and g and writes ga.  Measured (profiles/README.md): forward
// 124 us, backward 230 us for 256 x 20 x 75 x 216 (the backward is bound by the compare / select arithmetic of the arg-max routing).
#include "common.cuh"
#include "cp8.cuh"

namespace mpa {

int channel_sum_cp8_launch(const uint4* g, float* out, int B, int C, int T, int F, int TP, int P, int pf, int pt, int ncs, int fmt,
                           cudaStream_t st);   // reduce.cu

// Dropout keep factors of the 8 channels ck*8 .. ck*8+7 at the 4 pixels (t, 4q .. 4q+3): one Philox draw per channel (the 4 lanes of a
// draw are the 4 neighbouring bins — F % 4 == 0 makes the NCHW element index of bin 4q a multiple of 4).  Padded channels (>= C) keep 1.
__device__ __forceinline__ void dropout_quad8(float fac[4][8], long long i_quad /* element index of channel ck*8 at (t, 4q) */, long long plane,
                                              int c_real /* C - ck*8 */, float p, float scale, unsigned long long seed,
                                              unsigned long long offset) {
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    if (e < c_real) {
      const uint4 r = dropout_bits((i_quad + (long long)e * plane) >> 2, seed, offset);
      fac[0][e] = dropout_factor(r.x, p, scale);
      fac[1][e] = dropout_factor(r.y, p, scale);
      fac[2][e] = dropout_factor(r.z, p, scale);
      fac[3][e] = dropout_factor(r.w, p, scale);
    } else {
      fac[0][e] = fac[1][e] = fac[2][e] = fac[3][e] = 1.f;
    }
  }
}

template <int FMT>
__device__ __forceinline__ void max8(uint4& c, const uint4& u) {
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    if (FMT == MPA_FMT_BF16)
      reinterpret_cast<__nv_bfloat162*>(&c)[e] = __hmax2(reinterpret_cast<__nv_bfloat162*>(&c)[e], reinterpret_cast<const __nv_bfloat162*>(&u)[e]);
    else
      reinterpret_cast<__half2*>(&c)[e] = __hmax2(reinterpret_cast<__half2*>(&c)[e], reinterpret_cast<const __half2*>(&u)[e]);
  }
}

constexpr int kCp8Threads = 128;

// thread = 4 neighbouring bins x 8 channels (64 contiguous bytes per row) of one chunk plane, walking down a segment of the T rows with
// the previous / current / next row in registers: every row is loaded once (plus one halo row at each end of a segment).
// total = B * NCk * segs * F/4
template <int FMT>
__global__ void __launch_bounds__(kCp8Threads) pool3_dropout_cp8_kernel(const uint4* __restrict__ a, uint4* __restrict__ out, long long total, int C,
                                                                        int NCk, int segs, int T, int F4, int TP, int P, int pf, int pt,
                                                                        DropoutArgs d, int out_split, int P2) {
  const long long i = blockIdx.x * (long long)kCp8Threads + threadIdx.x;
  if (i >= total) return;
  const int q = (int)(i % F4);
  long long r = i / F4;
  const int sg = (int)(r % segs);
  r /= segs;
  const int ck = (int)(r % NCk);
  const long long b = r / NCk;
  const int seg = (T + segs - 1) / segs;
  const int r0 = sg * seg, r1 = min(T, r0 + seg);
  if (r0 >= r1) return;
  const size_t base = (((size_t)b * NCk + ck) * TP + pt) * P + pf + 4 * q;
  const bool drop = d.p > 0.f;
  const unsigned long long d_off = drop ? dropout_offset(d) : 0ull;
  const float d_scale = drop ? 1.f / (1.f - d.p) : 1.f;
  const int F = 4 * F4;
  const long long plane = (long long)T * F;
  const long long i_col = (b * C + ck * 8) * plane + 4 * q;
  uint4 prev[4], cur[4], next[4];
#pragma unroll
  for (int x = 0; x < 4; ++x) {
    cur[x] = a[base + (size_t)r0 * P + x];
    prev[x] = r0 > 0 ? a[base + (size_t)(r0 - 1) * P + x] : cur[x];      // outside [0, T): a copy of a valid row is max-neutral
  }
  for (int t = r0; t < r1; ++t) {
#pragma unroll
    for (int x = 0; x < 4; ++x) next[x] = t + 1 < T ? a[base + (size_t)(t + 1) * P + x] : cur[x];
    uint4 c[4];
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      c[x] = cur[x];
      max8<FMT>(c[x], prev[x]);
      max8<FMT>(c[x], next[x]);
    }
    if (drop) {
      float fac[4][8];
      dropout_quad8(fac, i_col + (long long)t * F, plane, C - ck * 8, d.p, d_scale, d.seed, d_off);
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        float m[8];
        unpack8<FMT>(c[x], m);
#pragma unroll
        for (int e = 0; e < 8; ++e) m[e] = __fmul_rn(m[e], fac[x][e]);
        c[x] = pack8<FMT>(m);
      }
    }
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      if (out_split) {
        // phase-split hand-over to a stride-(1, s) convolution: bin f -> phase set f % s (s * NCk chunk planes per item), column f / s
        const int f = 4 * q + x, ph = f % out_split;
        out[((((size_t)b * out_split + ph) * NCk + ck) * TP + pt + t) * P2 + pf + f / out_split] = c[x];
      } else {
        out[base + (size_t)t * P + x] = c[x];
      }
      prev[x] = cur[x];
      cur[x] = next[x];
    }
  }
}

template <int FMT>
__device__ __forceinline__ float elem2(const uint2& u, int e) {       // channel e (0..3, compile-time) of half a packed pixel
  const uint32_t w = (e >> 1) == 0 ? u.x : u.y;
  if (FMT == MPA_FMT_BF16) return (e & 1) ? __uint_as_float(w & 0xFFFF0000u) : __uint_as_float(w << 16);
  const __half2 h = *reinterpret_cast<const __half2*>(&w);
  return (e & 1) ? __high2float(h) : __low2float(h);
}
template <int FMT>
__device__ __forceinline__ uint2 pack4(const float v[4]) {
  uint32_t w[2];
#pragma unroll
  for (int e = 0; e < 2; ++e) {
    if (FMT == MPA_FMT_BF16) {
      const __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
      w[e] = *reinterpret_cast<const uint32_t*>(&h);
    } else {
      const __half2 h = __floats2half2_rn(v[2 * e], v[2 * e + 1]);
      w[e] = *reinterpret_cast<const uint32_t*>(&h);
    }
  }
  return make_uint2(w[0], w[1]);
}

// thread = 4 neighbouring bins x 4 channels (half a chunk: 8-byte loads, the two halves of a pixel sit in neighbouring threads) of one
// chunk plane, walking down a segment of the T rows with the window's 3 activation rows (packed 16-bit) and the 3 pending gradient sums
// (fp32) in registers — the register version of maxpool_time_bwd_col_kernel<3>.  total = B * NCk * segs * F/4 * 2; a segment re-reads
// one halo window above and below.
template <int FMT>
__global__ void __launch_bounds__(kCp8Threads) pool3_bwd_dropout_cp8_kernel(const uint2* __restrict__ a, const uint2* __restrict__ g_p,
                                                                            uint2* __restrict__ g_a, long long total, int C, int NCk, int segs, int T,
                                                                            int F4, int TP, int P, int pf, int pt, int act, float act_param,
                                                                            DropoutArgs d, int g_split, int Pg) {
  const long long i = blockIdx.x * (long long)kCp8Threads + threadIdx.x;
  if (i >= total) return;
  const int half = (int)(i & 1);
  long long r = i >> 1;
  const int q = (int)(r % F4);
  r /= F4;
  const int sg = (int)(r % segs);
  r /= segs;
  const int ck = (int)(r % NCk);
  const long long b = r / NCk;
  // output rows [r0, r1) of this segment; windows r0-1 .. r1 contribute to them
  const int seg = (T + segs - 1) / segs;
  const int r0 = sg * seg, r1 = min(T, r0 + seg);
  if (r0 >= r1) return;
  const size_t base = ((((size_t)b * NCk + ck) * TP + pt) * P + pf + 4 * q) * 2 + half;      // in 8-byte units; next bin: + 2, next row: + 2 P
  const size_t P2 = 2 * (size_t)P;
  const bool drop = d.p > 0.f;
  const unsigned long long d_off = drop ? dropout_offset(d) : 0ull;
  const float d_scale = drop ? 1.f / (1.f - d.p) : 1.f;
  const int F = 4 * F4;
  const long long plane = (long long)T * F;
  const int c_first = ck * 8 + half * 4;
  const long long i_col = (b * C + c_first) * plane + 4 * q;
  const uint2 zero2 = make_uint2(0u, 0u);

  uint2 win[3][4];                 // win[j][x] = activation row w - 1 + j of window w, bin 4q + x
  float acc[3][4][4];              // pending gradient of those rows [row][bin][channel]
  bool valid[3];
  int w = r0 >= 1 ? r0 - 1 : 0;    // first window of the segment (for r0 >= 1 only its contribution to row r0 matters)
#pragma unroll
  for (int j = 0; j < 3; ++j) {
    const int row = w - 1 + j;
    valid[j] = row >= 0 && row < T;
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      win[j][x] = valid[j] ? a[base + (size_t)row * P2 + 2 * x] : zero2;
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[j][x][e] = 0.f;
    }
  }
  const int w_last = min(T - 1, r1);
  // gradient wrt the pool output: same planes as `a`, or (g_split = s) the phase-split planes a stride-(1, s) convolution's data gradient wrote
  size_t gbase[4], grow = P2;
#pragma unroll
  for (int x = 0; x < 4; ++x) {
    gbase[x] = base + 2 * x;
    if (g_split) {
      const int f = 4 * q + x, ph = f % g_split;
      gbase[x] = (((((size_t)b * g_split + ph) * NCk + ck) * TP + pt) * Pg + pf + f / g_split) * 2 + half;
      grow = 2 * (size_t)Pg;
    }
  }
  uint2 graw[4];
#pragma unroll
  for (int x = 0; x < 4; ++x) graw[x] = g_p[gbase[x] + (size_t)w * grow];
  for (; w <= w_last; ++w) {
    // the next rows are requested before this window's arithmetic
    uint2 gnext[4], anext[4];
    const bool more_g = w + 1 <= w_last, more_a = w + 2 < T;
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      gnext[x] = more_g ? g_p[gbase[x] + (size_t)(w + 1) * grow] : zero2;
      anext[x] = more_a ? a[base + (size_t)(w + 2) * P2 + 2 * x] : zero2;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float fac[4] = {1.f, 1.f, 1.f, 1.f};
      if (drop && c_first + e < C) {         // one Philox draw per channel serves its 4 bins; padded channels carry zeros anyway
        const uint4 rb = dropout_bits((i_col + (long long)e * plane + (long long)w * F) >> 2, d.seed, d_off);
        fac[0] = dropout_factor(rb.x, d.p, d_scale);
        fac[1] = dropout_factor(rb.y, d.p, d_scale);
        fac[2] = dropout_factor(rb.z, d.p, d_scale);
        fac[3] = dropout_factor(rb.w, d.p, d_scale);
      }
#pragma unroll
      for (int x = 0; x < 4; ++x) {
        float g = elem2<FMT>(graw[x], e);
        if (drop) g = __fmul_rn(g, fac[x]);
        const float a0 = elem2<FMT>(win[0][x], e), a1 = elem2<FMT>(win[1][x], e), a2 = elem2<FMT>(win[2][x], e);
        // strict '>': the first maximum of the window wins (ATen semantics); rows outside [0, T) never win
        int am = valid[0] ? 0 : 1;
        float best = valid[0] ? a0 : a1;
        if (valid[0] && a1 > best) { best = a1; am = 1; }
        if (valid[2] && a2 > best) am = 2;
        acc[0][x][e] += am == 0 ? g : 0.f;
        acc[1][x][e] += am == 1 ? g : 0.f;
        acc[2][x][e] += am == 2 ? g : 0.f;
      }
    }
    // row w - 1 has now seen its three windows (w - 2, w - 1, w); after the last window of the tensor row T - 1 is final as well
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int done = w - 1 + j;
      if (done >= r0 && done < r1 && (j == 0 || w == T - 1)) {
#pragma unroll
        for (int x = 0; x < 4; ++x) {
          float o[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float mine = elem2<FMT>(win[j][x], e);
            float dd = 1.f;
            if (act == MPA_ACT_LRELU) dd = mine >= 0.f ? 1.f : act_param;
            else if (act == MPA_ACT_RELU) dd = mine > 0.f ? 1.f : 0.f;
            o[e] = acc[j][x][e] * dd;
          }
          g_a[base + (size_t)done * P2 + 2 * x] = pack4<FMT>(o);
        }
      }
    }
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      win[0][x] = win[1][x]; win[1][x] = win[2][x]; win[2][x] = anext[x];
      graw[x] = gnext[x];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        acc[0][x][e] = acc[1][x][e]; acc[1][x][e] = acc[2][x][e]; acc[2][x][e] = 0.f;
      }
    }
    valid[0] = valid[1]; valid[1] = valid[2]; valid[2] = more_a;
  }
}


// ---- LayerNorm([C,F]) on the network input, one thread per pixel (basic_cnns.py:371,411; unet_cnns.py:364) ------------------------------
// The row kernels of elementwise.cu / backward.cu give one CTA to one (item, frame) row and reach ~1 TB/s (11 strided scalars per thread,
// 2-byte gathers of the 16-bit gradient, the row statistics recomputed in the backward).  Here a thread owns one bin f of a row with all
// C <= 8 channels: C coalesced fp32 loads in, ONE 16-byte CP8 pixel out (forward) / in (gradient); a CTA walks over a range of rows two at
// a time (both rows' loads in flight before the first reduction) and the forward leaves (mean, rstd) per row for the parameter gradient.
constexpr int kLnPixThreads = 256;

// sums of two values over the 8 warps of the CTA; `sh` = 16 floats not touched since the last barrier
__device__ __forceinline__ void block_sum2_8w(float& a, float& b, float* sh) {
  a = warp_sum(a);
  b = warp_sum(b);
  if ((threadIdx.x & 31) == 0) {
    sh[threadIdx.x >> 5] = a;
    sh[8 + (threadIdx.x >> 5)] = b;
  }
  __syncthreads();
  a = ((sh[0] + sh[1]) + (sh[2] + sh[3])) + ((sh[4] + sh[5]) + (sh[6] + sh[7]));
  b = ((sh[8] + sh[9]) + (sh[10] + sh[11])) + ((sh[12] + sh[13]) + (sh[14] + sh[15]));
}

template <int FMT>
__global__ void __launch_bounds__(kLnPixThreads, 4) layernorm_pix_cp8_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                                          const float* __restrict__ bsh, uint4* __restrict__ out,
                                                                          float2* __restrict__ stats, int rows, int rpb, int C, int T, int F, int TP,
                                                                          int P, int pf, int pt, float eps, float gamma_log) {
  __shared__ float sh[32];       // two regions: the barrier of the second reduction of a row pair frees the first region again
  const int f = threadIdx.x;
  const bool on = f < F;
  float wc[8], bc[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    wc[c] = (on && c < C) ? w[c * F + f] : 0.f;
    bc[c] = (on && c < C) ? bsh[c * F + f] : 0.f;
  }
  const float inv_n = 1.f / (float)(C * F);
  const size_t cs = (size_t)T * F;
  const int r0 = blockIdx.x * rpb, r1 = min(rows, r0 + rpb);
  for (int r = r0; r < r1; r += 2) {
    const bool two = r + 1 < r1;
    const int ba = r / T, ta = r - ba * T, rb = two ? r + 1 : r, bb = rb / T, tb = rb - bb * T;
    const float* xa = x + ((size_t)ba * C * T + ta) * F + f;
    const float* xb = x + ((size_t)bb * C * T + tb) * F + f;
    float va[8], vb[8], sa = 0.f, sb = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      va[c] = (on && c < C) ? xa[c * cs] : 0.f;
      vb[c] = (on && c < C) ? xb[c * cs] : 0.f;
    }
    if (gamma_log > 0.f) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        if (on && c < C) {
          va[c] = logf(__fadd_rn(1.f, __fmul_rn(gamma_log, va[c])));
          vb[c] = logf(__fadd_rn(1.f, __fmul_rn(gamma_log, vb[c])));
        }
      }
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      sa += va[c];
      sb += vb[c];
    }
    block_sum2_8w(sa, sb, sh);
    const float ma = sa * inv_n, mb = sb * inv_n;
    float qa = 0.f, qb = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      if (on && c < C) {
        const float da = va[c] - ma, db = vb[c] - mb;
        qa = fmaf(da, da, qa);
        qb = fmaf(db, db, qb);
      }
    }
    block_sum2_8w(qa, qb, sh + 16);
    const float ra = rsqrtf(qa * inv_n + eps), rbs = rsqrtf(qb * inv_n + eps);
    if (on) {
      float oa[8], ob[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        oa[c] = c < C ? fmaf((va[c] - ma) * ra, wc[c], bc[c]) : 0.f;
        ob[c] = c < C ? fmaf((vb[c] - mb) * rbs, wc[c], bc[c]) : 0.f;
      }
      out[((size_t)ba * TP + pt + ta) * P + pf + f] = pack8<FMT>(oa);
      if (two) out[((size_t)bb * TP + pt + tb) * P + pf + f] = pack8<FMT>(ob);
    }
    if (stats && threadIdx.x == 0) {
      stats[r] = make_float2(ma, ra);
      if (two) stats[r + 1] = make_float2(mb, rbs);
    }
  }
}

// gw[c,f] += sum_rows g * (x - mean) * rstd, gb[c,f] += sum_rows g over the CTA's rows; g = the CP8 planes the first convolution's data
// gradient wrote, (mean, rstd) from the forward.  12 atomics per thread and CTA (gw / gb zeroed by the launcher).
template <int FMT>
__global__ void __launch_bounds__(kLnPixThreads, 4) layernorm_pix_param_grad_cp8_kernel(const float* __restrict__ x, const uint4* __restrict__ g,
                                                                                     const float2* __restrict__ stats, float* __restrict__ gw,
                                                                                     float* __restrict__ gb, int rows, int rpb, int C, int T, int F,
                                                                                     int TP, int P, int pf, int pt, float gamma_log) {
  const int f = threadIdx.x;
  if (f >= F) return;
  float aw[8], ab[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) aw[c] = ab[c] = 0.f;
  const size_t cs = (size_t)T * F;
  const int r0 = blockIdx.x * rpb, r1 = min(rows, r0 + rpb);
#pragma unroll 2
  for (int r = r0; r < r1; ++r) {
    const int b = r / T, t = r - b * T;
    const float2 st = stats[r];
    const float* xr = x + ((size_t)b * C * T + t) * F + f;
    float gv[8], xv[8];
    unpack8<FMT>(g[((size_t)b * TP + pt + t) * P + pf + f], gv);
#pragma unroll
    for (int c = 0; c < 8; ++c) xv[c] = c < C ? xr[c * cs] : 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      if (c < C) {
        float v = xv[c];
        if (gamma_log > 0.f) v = logf(__fadd_rn(1.f, __fmul_rn(gamma_log, v)));
        aw[c] = fmaf(gv[c], (v - st.x) * st.y, aw[c]);
        ab[c] += gv[c];
      }
    }
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    if (c < C) {
      atomicAdd(&gw[c * F + f], aw[c]);
      atomicAdd(&gb[c * F + f], ab[c]);
    }
  }
}

// LayerNorm([C,F]) backward to the input, with the parameter gradients of the same rows in the same pass (gradients wrt the network input:
// saliency maps, eval-mode backward).  Per (b,t) row, with v the LayerNorm input (log(1 + gamma_log * x) when the compression is fused),
// xhat = (v - mean) * rstd and gh = g * w over the C*F elements:
//   dv = rstd * (gh - mean(gh) - xhat * mean(gh * xhat)),  dx = dv (* gamma_log / (1 + gamma_log * x)),  gw += g * xhat,  gb += g
// Layout of layernorm_pix_param_grad_cp8_kernel: a thread owns bin f with all C <= 8 channels, the two row means are one CTA reduction.
// G16 = MPA_FMT_* + 1: g is in the CP8 planes the first convolution's data gradient wrote and (mean, rstd) come from the forward's stats;
// G16 = 0: g is fp32 NCHW and the row statistics are re-reduced (two-pass, as the forward kernels do).  dx fp32 NCHW (overwritten).
template <int G16>
__global__ void __launch_bounds__(kLnPixThreads, 2) layernorm_pix_input_grad_kernel(const float* __restrict__ x, const float* __restrict__ g32,
                                                                                 const uint4* __restrict__ g16, const float2* __restrict__ stats,
                                                                                 const float* __restrict__ w, float* __restrict__ dx,
                                                                                 float* __restrict__ gw, float* __restrict__ gb, int rows, int rpb,
                                                                                 int C, int T, int F, int TP, int P, int pf, int pt, float eps,
                                                                                 float gamma_log) {
  __shared__ float sh[32];       // two regions, used alternately: a reduction's barrier frees the region the one before it read
  int region = 0;
  const int f = threadIdx.x;
  const bool on = f < F;
  float wc[8], aw[8], ab[8];
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    wc[c] = (on && c < C) ? w[c * F + f] : 0.f;
    aw[c] = ab[c] = 0.f;
  }
  const float inv_n = 1.f / (float)(C * F);
  const size_t cs = (size_t)T * F;
  const int r0 = blockIdx.x * rpb, r1 = min(rows, r0 + rpb);
  for (int r = r0; r < r1; ++r) {
    const int b = r / T, t = r - b * T;
    const size_t row = ((size_t)b * C * T + t) * F + f;
    float v[8], gv[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      v[c] = (on && c < C) ? x[row + c * cs] : 0.f;
      if constexpr (G16 == 0) gv[c] = (on && c < C) ? g32[row + c * cs] : 0.f;
    }
    if constexpr (G16 != 0) {
      if (on) {
        unpack8<G16 - 1>(g16[((size_t)b * TP + pt + t) * P + pf + f], gv);
      } else {
#pragma unroll
        for (int c = 0; c < 8; ++c) gv[c] = 0.f;
      }
    }
    if (gamma_log > 0.f) {
#pragma unroll
      for (int c = 0; c < 8; ++c)
        if (on && c < C) v[c] = logf(__fadd_rn(1.f, __fmul_rn(gamma_log, v[c])));
    }
    float mean, rstd;
    if (stats) {
      const float2 st = stats[r];
      mean = st.x;
      rstd = st.y;
    } else {
      float s = 0.f, unused = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) s += v[c];
      block_sum2_8w(s, unused, sh + 16 * (region++ & 1));
      mean = s * inv_n;
      float q = 0.f;
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        if (on && c < C) {
          const float d = v[c] - mean;
          q = fmaf(d, d, q);
        }
      }
      block_sum2_8w(q, unused, sh + 16 * (region++ & 1));
      rstd = rsqrtf(q * inv_n + eps);
    }
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const float gh = gv[c] * wc[c];          // zero outside the row (wc = 0 there)
      s1 += gh;
      s2 = fmaf(gh, (v[c] - mean) * rstd, s2);
    }
    block_sum2_8w(s1, s2, sh + 16 * (region++ & 1));
    const float m1 = s1 * inv_n, m2 = s2 * inv_n;
    if (on) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        if (c < C) {
          const float xh = (v[c] - mean) * rstd;
          float d = rstd * (gv[c] * wc[c] - m1 - xh * m2);
          if (gamma_log > 0.f) d *= gamma_log / __fadd_rn(1.f, __fmul_rn(gamma_log, x[row + c * cs]));
          dx[row + c * cs] = d;
          aw[c] = fmaf(gv[c], xh, aw[c]);
          ab[c] += gv[c];
        }
      }
    }
  }
  if (!on) return;
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    if (c < C) {
      atomicAdd(&gw[c * F + f], aw[c]);
      atomicAdd(&gb[c * F + f], ab[c]);
    }
  }
}

static inline int ln_rows_per_block(int rows, int ctas_per_sm) {
  int rpb = ceil_div(rows, 148 * ctas_per_sm);
  rpb = (rpb + 1) & ~1;
  return rpb < 2 ? 2 : rpb;
}

}  // namespace mpa

using namespace mpa;

extern "C" {

int mpa_pool3_dropout_split_cp8(const void* a_cp8, void* out_cp8, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, float p,
                                unsigned long long seed, unsigned long long offset, const long long* step_dev, unsigned long long step_mul,
                                int out_split, int out_pitch, void* stream);

int mpa_pool3_dropout_cp8(const void* a_cp8, void* out_cp8, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, float p,
                          unsigned long long seed, unsigned long long offset, const long long* step_dev, unsigned long long step_mul,
                          void* stream) {
  return mpa_pool3_dropout_split_cp8(a_cp8, out_cp8, B, C, T, F, pitch, pf, pt, fmt, p, seed, offset, step_dev, step_mul, 0, 0, stream);
}

int mpa_pool3_dropout_split_cp8(const void* a_cp8, void* out_cp8, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, float p,
                                unsigned long long seed, unsigned long long offset, const long long* step_dev, unsigned long long step_mul,
                                int out_split, int out_pitch, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(out_split == 0 || (out_split > 1 && F % out_split == 0 && out_pitch >= pf + F / out_split), "pool3_dropout_cp8: bad phase split");
  MPA_REQUIRE(a_cp8 && out_cp8 && B > 0 && C > 0 && T > 0 && F > 0 && F % 4 == 0 && pitch >= pf + F && pt >= 0 && p >= 0.f && p < 1.f &&
                  (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16),
              "pool3_dropout_cp8: bad argument (F must be a multiple of 4)");
  const int NCk = (C + 7) / 8;
  // enough threads to fill the GPU: split the T rows into segments (each segment re-reads 2 halo rows)
  const long long cols = (long long)B * NCk * (F / 4);
  int segs = ceil_div(148LL * 8 * kCp8Threads, cols);
  segs = segs < 1 ? 1 : (segs > ceil_div(T, 8) ? ceil_div(T, 8) : segs);
  const long long total = cols * segs;
  const int grid = ceil_div(total, kCp8Threads);
  const DropoutArgs d{p, seed, offset, step_dev, step_mul};
  if (fmt == MPA_FMT_BF16)
    pool3_dropout_cp8_kernel<MPA_FMT_BF16><<<grid, kCp8Threads, 0, (cudaStream_t)stream>>>((const uint4*)a_cp8, (uint4*)out_cp8, total, C, NCk, segs,
                                                                                          T, F / 4, T + 2 * pt, pitch, pf, pt, d, out_split, out_pitch);
  else
    pool3_dropout_cp8_kernel<MPA_FMT_F16><<<grid, kCp8Threads, 0, (cudaStream_t)stream>>>((const uint4*)a_cp8, (uint4*)out_cp8, total, C, NCk, segs,
                                                                                         T, F / 4, T + 2 * pt, pitch, pf, pt, d, out_split, out_pitch);
  MPA_CHECK_LAUNCH("pool3_dropout_cp8");
  return MPA_OK;
}

int mpa_pool3_bwd_dropout_split_cp8(const void* a_cp8, const void* g_out_cp8, void* g_a_cp8, int B, int C, int T, int F, int pitch, int pf, int pt,
                                    int fmt, int act, float act_param, float p, unsigned long long seed, unsigned long long offset,
                                    const long long* step_dev, unsigned long long step_mul, int g_split, int g_pitch, void* stream);

int mpa_pool3_bwd_dropout_cp8(const void* a_cp8, const void* g_out_cp8, void* g_a_cp8, int B, int C, int T, int F, int pitch, int pf, int pt,
                              int fmt, int act, float act_param, float p, unsigned long long seed, unsigned long long offset,
                              const long long* step_dev, unsigned long long step_mul, void* stream) {
  return mpa_pool3_bwd_dropout_split_cp8(a_cp8, g_out_cp8, g_a_cp8, B, C, T, F, pitch, pf, pt, fmt, act, act_param, p, seed, offset, step_dev,
                                         step_mul, 0, 0, stream);
}

int mpa_pool3_bwd_dropout_split_cp8(const void* a_cp8, const void* g_out_cp8, void* g_a_cp8, int B, int C, int T, int F, int pitch, int pf, int pt,
                                    int fmt, int act, float act_param, float p, unsigned long long seed, unsigned long long offset,
                                    const long long* step_dev, unsigned long long step_mul, int g_split, int g_pitch, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(g_split == 0 || (g_split > 1 && F % g_split == 0 && g_pitch >= pf + F / g_split), "pool3_bwd_dropout_cp8: bad phase split");
  MPA_REQUIRE(a_cp8 && g_out_cp8 && g_a_cp8 && B > 0 && C > 0 && T > 0 && F > 0 && F % 4 == 0 && pitch >= pf + F && pt >= 0 && p >= 0.f &&
                  p < 1.f && (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16),
              "pool3_bwd_dropout_cp8: bad argument (F must be a multiple of 4)");
  const int NCk = (C + 7) / 8;
  // enough threads to fill the GPU: split the T rows into segments (each segment re-reads 2 halo rows)
  const long long cols = (long long)B * NCk * (F / 4);
  int segs = ceil_div(148LL * 8 * kCp8Threads, cols * 2);
  segs = segs < 1 ? 1 : (segs > ceil_div(T, 8) ? ceil_div(T, 8) : segs);
  const long long total = cols * segs * 2;
  const int grid = ceil_div(total, kCp8Threads);
  const DropoutArgs d{p, seed, offset, step_dev, step_mul};
  if (fmt == MPA_FMT_BF16)
    pool3_bwd_dropout_cp8_kernel<MPA_FMT_BF16><<<grid, kCp8Threads, 0, (cudaStream_t)stream>>>(
        (const uint2*)a_cp8, (const uint2*)g_out_cp8, (uint2*)g_a_cp8, total, C, NCk, segs, T, F / 4, T + 2 * pt, pitch, pf, pt, act, act_param, d,
        g_split, g_pitch);
  else
    pool3_bwd_dropout_cp8_kernel<MPA_FMT_F16><<<grid, kCp8Threads, 0, (cudaStream_t)stream>>>(
        (const uint2*)a_cp8, (const uint2*)g_out_cp8, (uint2*)g_a_cp8, total, C, NCk, segs, T, F / 4, T + 2 * pt, pitch, pf, pt, act, act_param, d,
        g_split, g_pitch);
  MPA_CHECK_LAUNCH("pool3_bwd_dropout_cp8");
  return MPA_OK;
}

int mpa_channel_sum_cp8(const void* g_cp8, float* out, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, int ncs, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(g_cp8 && out && B > 0 && C > 0 && T > 0 && F > 0 && pitch >= pf + F && pt >= 0 && (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16),
              "channel_sum_cp8: bad argument");
  if (ncs <= 0) ncs = (C + 7) / 8;
  int rc = channel_sum_cp8_launch((const uint4*)g_cp8, out, B, C, T, F, T + 2 * pt, pitch, pf, pt, ncs, fmt, (cudaStream_t)stream);
  if (rc != MPA_OK) return rc;
  MPA_CHECK_LAUNCH("channel_sum_cp8");
  return MPA_OK;
}

// LayerNorm([C,F]) -> CP8 planes with one thread per pixel; stats (optional) [B*T] (mean, rstd) for mpa_layernorm_cf_param_grad_cp8_stats
int mpa_layernorm_cf_cp8_stats(const float* x, const float* ln_w, const float* ln_b, void* out_cp8, float* stats, int B, int C, int T, int F,
                               int pitch, int pf, int pt, float eps, float gamma_log, int fmt, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && ln_w && ln_b && out_cp8 && B > 0 && C > 0 && C <= 8 && T > 0 && F > 0 && F <= kLnPixThreads && pitch >= pf + F && pt >= 0 &&
                  (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16) && (long long)B * T < (1ll << 31),
              "layernorm_cf_cp8_stats: bad argument (C <= 8, F <= 256, 16-bit formats)");
  const int rows = B * T, rpb = ln_rows_per_block(rows, 4), grid = ceil_div(rows, rpb);
  if (fmt == MPA_FMT_BF16)
    layernorm_pix_cp8_kernel<MPA_FMT_BF16><<<grid, kLnPixThreads, 0, (cudaStream_t)stream>>>(x, ln_w, ln_b, (uint4*)out_cp8, (float2*)stats, rows, rpb,
                                                                                            C, T, F, T + 2 * pt, pitch, pf, pt, eps, gamma_log);
  else
    layernorm_pix_cp8_kernel<MPA_FMT_F16><<<grid, kLnPixThreads, 0, (cudaStream_t)stream>>>(x, ln_w, ln_b, (uint4*)out_cp8, (float2*)stats, rows, rpb,
                                                                                           C, T, F, T + 2 * pt, pitch, pf, pt, eps, gamma_log);
  MPA_CHECK_LAUNCH("layernorm_cf_cp8_stats");
  return MPA_OK;
}

int mpa_layernorm_cf_param_grad_cp8_stats(const float* x, const void* g_cp8, const float* stats, float* g_w, float* g_b, int B, int C, int T, int F,
                                          int pitch, int pf, int pt, int fmt, float gamma_log, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && g_cp8 && stats && g_w && g_b && B > 0 && C > 0 && C <= 8 && T > 0 && F > 0 && F <= kLnPixThreads && pitch >= pf + F &&
                  pt >= 0 && (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16) && (long long)B * T < (1ll << 31),
              "layernorm_cf_param_grad_cp8_stats: bad argument (C <= 8, F <= 256, 16-bit formats)");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(g_w, 0, sizeof(float) * (size_t)C * F, st);
  cudaMemsetAsync(g_b, 0, sizeof(float) * (size_t)C * F, st);
  const int rows = B * T, rpb = ln_rows_per_block(rows, 4), grid = ceil_div(rows, rpb);
  if (fmt == MPA_FMT_BF16)
    layernorm_pix_param_grad_cp8_kernel<MPA_FMT_BF16><<<grid, kLnPixThreads, 0, st>>>(x, (const uint4*)g_cp8, (const float2*)stats, g_w, g_b, rows, rpb,
                                                                                     C, T, F, T + 2 * pt, pitch, pf, pt, gamma_log);
  else
    layernorm_pix_param_grad_cp8_kernel<MPA_FMT_F16><<<grid, kLnPixThreads, 0, st>>>(x, (const uint4*)g_cp8, (const float2*)stats, g_w, g_b, rows, rpb,
                                                                                    C, T, F, T + 2 * pt, pitch, pf, pt, gamma_log);
  MPA_CHECK_LAUNCH("layernorm_cf_param_grad_cp8_stats");
  return MPA_OK;
}

int mpa_layernorm_cf_input_grad_cp8_stats(const float* x, const void* g_cp8, const float* stats, const float* ln_w, float* dx, float* g_w, float* g_b,
                                          int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, float gamma_log, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && g_cp8 && stats && ln_w && dx && g_w && g_b && B > 0 && C > 0 && C <= 8 && T > 0 && F > 0 && F <= kLnPixThreads &&
                  pitch >= pf + F && pt >= 0 && (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16) && (long long)B * T < (1ll << 31),
              "layernorm_cf_input_grad_cp8_stats: bad argument (C <= 8, F <= 256, 16-bit formats)");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(g_w, 0, sizeof(float) * (size_t)C * F, st);
  cudaMemsetAsync(g_b, 0, sizeof(float) * (size_t)C * F, st);
  const int rows = B * T, rpb = ln_rows_per_block(rows, 4), grid = ceil_div(rows, rpb);
  if (fmt == MPA_FMT_BF16)
    layernorm_pix_input_grad_kernel<MPA_FMT_BF16 + 1><<<grid, kLnPixThreads, 0, st>>>(x, nullptr, (const uint4*)g_cp8, (const float2*)stats, ln_w, dx,
                                                                                     g_w, g_b, rows, rpb, C, T, F, T + 2 * pt, pitch, pf, pt, 0.f,
                                                                                     gamma_log);
  else
    layernorm_pix_input_grad_kernel<MPA_FMT_F16 + 1><<<grid, kLnPixThreads, 0, st>>>(x, nullptr, (const uint4*)g_cp8, (const float2*)stats, ln_w, dx,
                                                                                    g_w, g_b, rows, rpb, C, T, F, T + 2 * pt, pitch, pf, pt, 0.f,
                                                                                    gamma_log);
  MPA_CHECK_LAUNCH("layernorm_cf_input_grad_cp8_stats");
  return MPA_OK;
}

int mpa_layernorm_cf_input_grad_f32(const float* x, const float* g_out, const float* ln_w, float* dx, float* g_w, float* g_b, int B, int C, int T,
                                    int F, float eps, float gamma_log, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && g_out && ln_w && dx && g_w && g_b && B > 0 && C > 0 && C <= 8 && T > 0 && F > 0 && F <= kLnPixThreads &&
                  (long long)B * T < (1ll << 31),
              "layernorm_cf_input_grad_f32: bad argument (C <= 8, F <= 256)");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(g_w, 0, sizeof(float) * (size_t)C * F, st);
  cudaMemsetAsync(g_b, 0, sizeof(float) * (size_t)C * F, st);
  const int rows = B * T, rpb = ln_rows_per_block(rows, 4), grid = ceil_div(rows, rpb);
  layernorm_pix_input_grad_kernel<0><<<grid, kLnPixThreads, 0, st>>>(x, g_out, nullptr, nullptr, ln_w, dx, g_w, g_b, rows, rpb, C, T, F, 0, 0, 0, 0,
                                                                     eps, gamma_log);
  MPA_CHECK_LAUNCH("layernorm_cf_input_grad_f32");
  return MPA_OK;
}

}  // extern "C"
