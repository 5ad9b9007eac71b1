// Backward / optimiser kernels of the CNN family (training configuration 2: CNN:XS fwd+bwd, SURVEY.md 8a N2/N11).
// fp32 NCHW, CUDA cores.  Reference semantics reproduced:
//   * MaxPool2d((k,1)) backward routes the gradient to the FIRST maximum of each window (ATen max_pool2d_with_indices),
//   * LeakyReLU backward uses the sign of the forward output,
//   * BCELoss backward = (p - t) / max(p (1-p), 1e-12) / n   (elementwise.cu), sigmoid backward = g * p * (1-p),
//   * AdamW exactly as torch.optim.AdamW (decoupled weight decay, bias correction, eps outside the sqrt).
// Convolution data-gradients of stride-1 layers reuse the forward direct kernel with transposed/flipped weights (host
// side packing); the strided head conv uses the generic gather kernel below.  Weight gradients are a blocked
// correlation with split-K over (batch, row) and one atomicAdd per output per CTA.
#include "common.cuh"
#include <cuda_fp16.h>

namespace mpa {

static inline int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  long long cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

// g_in = g_out * act'(out)   (act' expressed through the forward OUTPUT)
__global__ void act_bwd_kernel(const float* __restrict__ out, const float* __restrict__ g_out, float* __restrict__ g_in, long long n, int act,
                               float p) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float o = out[i], g = g_out[i];
    float d = 1.f;
    if (act == MPA_ACT_LRELU) d = o >= 0.f ? 1.f : p;
    else if (act == MPA_ACT_RELU) d = o > 0.f ? 1.f : 0.f;
    else if (act == MPA_ACT_SIGMOID) d = o * (1.f - o);
    g_in[i] = g * d;
  }
}

// a: forward input of the pool (post-activation), g_p: gradient wrt pool output.  g_a[t'] = act'(a[t']) * sum_t g_p[t]*[argmax_t == t']
// One CTA per (plane, 64 columns): the column tile of `a` is staged in shared memory, every thread owns one column and walks the T
// windows in order — the first arg-max of a window takes its gradient (ATen semantics) — accumulating into its own column of the tile.
constexpr int kPoolBwdCols = 64, kPoolBwdRowGroups = 4;
__global__ void __launch_bounds__(kPoolBwdCols * kPoolBwdRowGroups) maxpool_time_bwd_kernel(const float* __restrict__ a, const float* __restrict__ g_p,
                                                                                            float* __restrict__ g_a, int T, int F, int k, int act,
                                                                                            float act_param) {
  extern __shared__ float sm[];
  float* av = sm;                               // [T][64]
  float* acc = sm + (size_t)T * kPoolBwdCols;    // [T][64]
  const int h = k / 2;
  const long long plane = blockIdx.x;
  const int col = threadIdx.x % kPoolBwdCols, rg = threadIdx.x / kPoolBwdCols;
  const int f = blockIdx.y * kPoolBwdCols + col;
  const bool ok = f < F;
  const float* ap = a + plane * T * F + f;
  const float* gp = g_p + plane * T * F + f;
  for (int t = rg; t < T; t += kPoolBwdRowGroups) {
    av[t * kPoolBwdCols + col] = ok ? ap[(size_t)t * F] : 0.f;
    acc[t * kPoolBwdCols + col] = 0.f;
  }
  __syncthreads();
  if (ok) {
    for (int t = rg; t < T; t += kPoolBwdRowGroups) {
      const int lo = max(0, t - h), hi = min(T - 1, t + h);
      int am = lo;
      float best = av[lo * kPoolBwdCols + col];
      for (int s = lo + 1; s <= hi; ++s) {
        const float v = av[s * kPoolBwdCols + col];
        if (v > best) { best = v; am = s; }          // strict: the first maximum wins
      }
      atomicAdd(&acc[am * kPoolBwdCols + col], gp[(size_t)t * F]);   // <= k windows share an arg-max row
    }
  }
  __syncthreads();
  if (!ok) return;
  float* op = g_a + plane * T * F + f;
  for (int t = rg; t < T; t += kPoolBwdRowGroups) {
    const float mine = av[t * kPoolBwdCols + col];
    float d = 1.f;
    if (act == MPA_ACT_LRELU) d = mine >= 0.f ? 1.f : act_param;
    else if (act == MPA_ACT_RELU) d = mine > 0.f ? 1.f : 0.f;
    op[(size_t)t * F] = acc[t * kPoolBwdCols + col] * d;
  }
}

// Same result without shared memory or atomics for the two window lengths the models use (3 and 13): one thread owns one column and walks
// down the T rows with the window's k activations and the k pending gradient sums in registers; row t-h is final once window t is done.
// Loads / stores are coalesced across the threads of a row; HBM-bound (reads a and g_p once, writes g_a once).
template <int K>
// d.p > 0: g_p is the gradient BEHIND a dropout layer that followed the pool; its mask (same convention as dropout_kernel) is applied on the fly
__global__ void __launch_bounds__(128) maxpool_time_bwd_col_kernel(const float* __restrict__ a, const float* __restrict__ g_p, float* __restrict__ g_a,
                                                                   int T, int F, int act, float act_param, DropoutArgs d) {
  constexpr int H = K / 2;
  const int f = blockIdx.y * blockDim.x + threadIdx.x;
  if (f >= F) return;
  const size_t base = (size_t)blockIdx.x * T * F + f;
  const float* ap = a + base;
  const float* gp = g_p + base;
  float* op = g_a + base;
  const unsigned long long d_off = d.p > 0.f ? dropout_offset(d) : 0ull;
  const float d_scale = d.p > 0.f ? 1.f / (1.f - d.p) : 1.f;
  float win[K], acc[K];
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const int r = j - H;
    win[j] = (r >= 0 && r < T) ? ap[(size_t)r * F] : -INFINITY;
    acc[j] = 0.f;
  }
  for (int t = 0; t < T; ++t) {
    float g = gp[(size_t)t * F];
    if (d.p > 0.f) g = __fmul_rn(g, dropout_factor_at((long long)(base + (size_t)t * F), d.p, d_scale, d.seed, d_off));
    int am = 0;
    float best = win[0];
#pragma unroll
    for (int j = 1; j < K; ++j)
      if (win[j] > best) { best = win[j]; am = j; }        // strict: the first maximum of the window wins (ATen semantics)
#pragma unroll
    for (int j = 0; j < K; ++j) acc[j] += (j == am) ? g : 0.f;
    if (t - H >= 0) {
      float d = 1.f;
      if (act == MPA_ACT_LRELU) d = win[0] >= 0.f ? 1.f : act_param;
      else if (act == MPA_ACT_RELU) d = win[0] > 0.f ? 1.f : 0.f;
      op[(size_t)(t - H) * F] = acc[0] * d;
    }
#pragma unroll
    for (int j = 0; j < K - 1; ++j) {
      win[j] = win[j + 1];
      acc[j] = acc[j + 1];
    }
    const int r = t + H + 1;
    win[K - 1] = r < T ? ap[(size_t)r * F] : -INFINITY;
    acc[K - 1] = 0.f;
  }
  // rows T-H .. T-1 are now win[0..H-1]
#pragma unroll
  for (int j = 0; j < H; ++j) {
    const int r = T - H + j;
    if (r >= 0) {
      float d = 1.f;
      if (act == MPA_ACT_LRELU) d = win[j] >= 0.f ? 1.f : act_param;
      else if (act == MPA_ACT_RELU) d = win[j] > 0.f ? 1.f : 0.f;
      op[(size_t)r * F] = acc[j] * d;
    }
  }
}

// k = 13 (the head's MaxPool((13,1)), basic_cnns.py:180 / unet_cnns.py:379) for the training patch length T: same result as
// maxpool_time_bwd_col_kernel<13> bit for bit (the windows of a column are routed in the same order), with a fraction of its instructions.
// That kernel spent ~200 instructions per element: a 13-way compare / select scan per window, 13 predicated adds to route the gradient, 26
// register moves to slide the window and a whole Philox draw per element of which it used one lane of four.  Here
//  * the first arg-max of every window comes from a doubling table built on the fly (pairs -> fours -> eights -> two overlapping eights;
//    `>` keeps the left operand on ties, so the first maximum wins): 4 compare + select steps per row, the rows fully unrolled so that the
//    delay lines between the levels are register renaming,
//  * the gradient is routed with one read-modify-write of the thread's own shared-memory column,
//  * a Philox draw serves its 4 lanes = the 4 neighbouring bins of a thread quad: each thread draws for every fourth row and the quad
//    exchanges 16 keep bits with two shuffles,
//  * act'(a) needs one sign bit per row (3 registers).
constexpr int kPool13Threads = 128;

__device__ __forceinline__ void first_max(float& v, int& i, float bv, int bi) {
  const bool r = bv > v;
  v = r ? bv : v;
  i = r ? bi : i;
}

template <int T>
__global__ void __launch_bounds__(kPool13Threads) maxpool13_bwd_table_kernel(const float* __restrict__ a, const float* __restrict__ g_p,
                                                                            float* __restrict__ g_a, long long n_cols, int F, int act,
                                                                            float act_param, DropoutArgs d) {
  extern __shared__ float acc[];                        // [T][128]: column of thread x at acc[t * 128 + x]
  constexpr int H = 6, NW = (T + 31) / 32;
  const long long col_raw = blockIdx.x * (long long)kPool13Threads + threadIdx.x;
  const bool on = col_raw < n_cols;                     // n_cols % 4 == 0: a quad is on or off as a whole
  const long long col = on ? col_raw : n_cols - 1;
  const long long plane = col / F;
  const int f = (int)(col - plane * F);
  const size_t base = (size_t)plane * T * F + f;
  const float* ap = a + base;
  const float* gp = g_p + base;
  const int q = threadIdx.x & 3;                        // == f & 3 == lane of this bin in its Philox draw (F % 4 == 0)
  const bool drop = d.p > 0.f;
  const unsigned long long d_off = drop ? dropout_offset(d) : 0ull;
  const float d_scale = drop ? 1.f / (1.f - d.p) : 1.f;
  const uint32_t thr = drop ? (uint32_t)ceilf(d.p * 16777216.f) << 8 : 0u;
#pragma unroll
  for (int t = 0; t < T; ++t) acc[t * kPool13Threads + threadIdx.x] = 0.f;
  float a2v[3], a4v[5], a8v[6], gq[7], xs[8], gs[8];
  int a2i[3], a4i[5], a8i[6];
  uint32_t pos[NW], keep16 = 0u;
#pragma unroll
  for (int i = 0; i < 3; ++i) { a2v[i] = -INFINITY; a2i[i] = 0; }
#pragma unroll
  for (int i = 0; i < 5; ++i) { a4v[i] = -INFINITY; a4i[i] = 0; }
#pragma unroll
  for (int i = 0; i < 6; ++i) { a8v[i] = -INFINITY; a8i[i] = 0; }
#pragma unroll
  for (int i = 0; i < NW; ++i) pos[i] = 0u;
  float xprev = -INFINITY;
  // position p: sample a[p] arrives (p >= T: -inf); pairs [p-1,p], fours [p-3,p], eights [p-7,p] complete; window t = p - 6 = [p-12, p]
#pragma unroll
  for (int p = 0; p < T + H; ++p) {
    if ((p & 7) == 0) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        xs[j] = p + j < T ? ap[(size_t)(p + j) * F] : -INFINITY;
        gs[j] = p + j < T ? gp[(size_t)(p + j) * F] : 0.f;
      }
    }
    if (drop && (p & 3) == 0 && p < T) {
      // this thread draws for row p + q; afterwards bit 4 j + c of keep16 = keep flag of lane c of row p + j
      const uint4 r = dropout_bits((long long)((base - q + (size_t)(p + q) * F) >> 2), d.seed, d_off);
      uint32_t k4 = (r.x >= thr ? 1u : 0u) | (r.y >= thr ? 2u : 0u) | (r.z >= thr ? 4u : 0u) | (r.w >= thr ? 8u : 0u);
      k4 <<= 4 * q;
      k4 |= __shfl_xor_sync(0xffffffffu, k4, 1);
      k4 |= __shfl_xor_sync(0xffffffffu, k4, 2);
      keep16 = k4 >> q;
    }
    const float xp = xs[p & 7];
    float g = gs[p & 7];
    if (p < T) {
      if (drop) g = __fmul_rn(g, (keep16 >> (4 * (p & 3))) & 1u ? d_scale : 0.f);
      const bool ps = act == MPA_ACT_RELU ? xp > 0.f : xp >= 0.f;
      pos[p >> 5] |= ps ? 1u << (p & 31) : 0u;
    }
    gq[p % 7] = g;
    // pairs: A2[p-1] = first max of (a[p-1], a[p])
    {
      float v = xprev;
      int i = p - 1;
      first_max(v, i, xp, p);
      a2v[(p + 2) % 3] = v;      // slot of s = p - 1: (s + 3) % 3
      a2i[(p + 2) % 3] = i;
    }
    // fours: A4[p-3] = (A2[p-3], A2[p-1])
    {
      float v = a2v[p % 3];      // s = p - 3: (s + 3) % 3
      int i = a2i[p % 3];
      first_max(v, i, a2v[(p + 2) % 3], a2i[(p + 2) % 3]);
      a4v[(p + 2) % 5] = v;      // s = p - 3: (s + 5) % 5
      a4i[(p + 2) % 5] = i;
    }
    // eights: A8[p-7] = (A4[p-7], A4[p-3])
    {
      float v = a4v[(p + 3) % 5];   // s = p - 7: (s + 10) % 5
      int i = a4i[(p + 3) % 5];
      first_max(v, i, a4v[(p + 2) % 5], a4i[(p + 2) % 5]);
      a8v[(p + 5) % 6] = v;      // s = p - 7: (s + 12) % 6
      a8i[(p + 5) % 6] = i;
    }
    if (p >= H) {
      // window t = p - 6: (A8[p-12], A8[p-7])
      float v = a8v[p % 6];      // s = p - 12: (s + 12) % 6
      int i = a8i[p % 6];
      first_max(v, i, a8v[(p + 5) % 6], a8i[(p + 5) % 6]);
      acc[i * kPool13Threads + threadIdx.x] += gq[(p - H) % 7];
    }
    xprev = xp;
  }
  if (!on) return;
  const float dneg = act == MPA_ACT_LRELU ? act_param : (act == MPA_ACT_RELU ? 0.f : 1.f);
  float* op = g_a + base;
#pragma unroll
  for (int t = 0; t < T; ++t) op[(size_t)t * F] = acc[t * kPool13Threads + threadIdx.x] * ((pos[t >> 5] >> (t & 31)) & 1u ? 1.f : dneg);
}

constexpr int kPool13T = 75;       // the training patch length of every model (hcqt_datasets.py context 75)
static inline bool pool13_table_eligible(int k, int T, int F) { return k == 13 && T == kPool13T && F % 4 == 0; }
static int pool13_table_launch(const float* a, const float* g, float* g_a, int B, int C, int F, int act, float act_param, DropoutArgs d,
                               cudaStream_t st) {
  static unsigned char flags[64];
  constexpr size_t smem = (size_t)kPool13T * kPool13Threads * sizeof(float);
  if (opt_in_max_smem(maxpool13_bwd_table_kernel<kPool13T>, flags) != cudaSuccess) return MPA_ERR_CUDA;
  const long long n_cols = (long long)B * C * F;
  maxpool13_bwd_table_kernel<kPool13T><<<ceil_div(n_cols, kPool13Threads), kPool13Threads, smem, st>>>(a, g, g_a, n_cols, F, act, act_param, d);
  return MPA_OK;
}

// narrow tensors (the head's 72 bins): whole warps only, so that one wave of CTAs covers all (item, channel) planes
static inline int pool_col_threads(int F) { return F >= 128 ? 128 : (F + 31) / 32 * 32; }

// Philox-4x32-10 counter-based dropout (philox() in common.cuh): element i of call `offset` under `seed`
// step_dev != nullptr: offset = step_dev[0] * step_mul + offset (the step counter lives in device memory so that a captured CUDA graph of
// the training step draws fresh masks on every replay)
__global__ void dropout_kernel(const float* __restrict__ x, float* __restrict__ out, long long n, float p, unsigned long long seed,
                               unsigned long long offset, const long long* __restrict__ step_dev, unsigned long long step_mul) {
  if (step_dev) offset += (unsigned long long)step_dev[0] * step_mul;
  const float scale = 1.f / (1.f - p);
  for (long long i4 = blockIdx.x * (long long)blockDim.x + threadIdx.x; i4 * 4 < n; i4 += (long long)gridDim.x * blockDim.x) {
    const uint4 r = philox(make_uint4((uint32_t)i4, (uint32_t)(i4 >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)),
                           make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
    const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const long long i = i4 * 4 + e;
      if (i < n) {
        const float u = (float)(rr[e] >> 8) * (1.f / 16777216.f);
        out[i] = u >= p ? x[i] * scale : 0.f;
      }
    }
  }
}

// generic data gradient (gather form), any stride: gi[b,ci,h,w] = sum_{co,kh,kw} go[b,co,(h+ph-kh)/sh,(w+pw-kw)/sw] * w[co,ci,kh,kw]
__global__ void conv_dgrad_kernel(const float* __restrict__ go, const float* __restrict__ w, float* __restrict__ gi, long long total, int Cin,
                                  int H, int W, int Cout, int Ho, int Wo, int KH, int KW, int sh, int sw, int ph, int pw) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(i % W);
    long long r = i / W;
    const int y = (int)(r % H);
    r /= H;
    const int ci = (int)(r % Cin);
    const int b = (int)(r / Cin);
    float acc = 0.f;
    for (int kh = 0; kh < KH; ++kh) {
      const int yy = y + ph - kh;
      if (yy < 0 || yy % sh) continue;
      const int ho = yy / sh;
      if (ho >= Ho) continue;
      for (int kw = 0; kw < KW; ++kw) {
        const int xx = x + pw - kw;
        if (xx < 0 || xx % sw) continue;
        const int wo = xx / sw;
        if (wo >= Wo) continue;
        const float* gp = go + (((size_t)b * Cout) * Ho + ho) * Wo + wo;
        const float* wp = w + ((size_t)ci * KH + kh) * KW + kw;
        for (int co = 0; co < Cout; ++co) acc = fmaf(gp[(size_t)co * Ho * Wo], wp[(size_t)co * Cin * KH * KW], acc);
      }
    }
    gi[i] = acc;
  }
}

// weight gradient: gw[co,ci,kh,kw] += sum_{b,ho,wo} go[b,co,ho,wo] * x[b,ci,ho*sh+kh-ph,wo*sw+kw-pw]
// CTA: 32 output channels x 8 (ci,kh) combos x 16 kw; thread = 4 co x 4 kw for one combo; split-K over (b,ho) rows.
constexpr int WG_CO = 32, WG_COMBOS = 8, WG_KW = 16;
__global__ void __launch_bounds__(256) conv_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ go, float* __restrict__ gw, int B,
                                                         int Cin, int H, int W, int Cout, int Ho, int Wo, int KH, int KW, int sh, int sw, int ph,
                                                         int pw, int n_combos, int rows_per_cta) {
  extern __shared__ float sm[];
  const int XW = (Wo - 1) * sw + WG_KW;              // staged input row segment (zero padded)
  float* go_s = sm;                                   // [Wo][WG_CO]
  float* x_s = sm + (size_t)Wo * WG_CO;               // [WG_COMBOS][XW]
  const int co0 = blockIdx.x * WG_CO;
  const int combo0 = blockIdx.y * WG_COMBOS;
  const int tid = threadIdx.x;
  const int cl = tid >> 5;                            // local combo 0..7
  const int lane = tid & 31;
  const int co_t = (lane >> 2) * 4;                   // 0,4,..,28
  const int kw_t = (lane & 3) * 4;                    // 0,4,8,12
  const int combo = combo0 + cl;
  const bool combo_ok = combo < n_combos;
  const int ci = combo_ok ? combo / KH : 0, kh = combo_ok ? combo % KH : 0;
  float acc[4][4] = {};
  const long long n_rows = (long long)B * Ho;
  const long long r0 = (long long)blockIdx.z * rows_per_cta;
  for (long long rr = r0; rr < min(n_rows, r0 + rows_per_cta); ++rr) {
    const int b = (int)(rr / Ho), ho = (int)(rr % Ho);
    __syncthreads();
    for (int e = tid; e < Wo * WG_CO; e += 256) {
      const int c = e / Wo, f = e - c * Wo;           // coalesced along f in global
      const int co = co0 + c;
      go_s[f * WG_CO + c] = co < Cout ? go[(((size_t)b * Cout + co) * Ho + ho) * Wo + f] : 0.f;
    }
    for (int e = tid; e < WG_COMBOS * XW; e += 256) {
      const int c = e / XW, xx = e - c * XW;
      const int cb = combo0 + c;
      float v = 0.f;
      if (cb < n_combos) {
        const int cci = cb / KH, ckh = cb % KH;
        const int hy = ho * sh + ckh - ph, wx = xx - pw;
        if (hy >= 0 && hy < H && wx >= 0 && wx < W) v = x[(((size_t)b * Cin + cci) * H + hy) * W + wx];
      }
      x_s[e] = v;
    }
    __syncthreads();
    if (combo_ok) {
      const float* xr = x_s + cl * XW + kw_t;
      for (int f = 0; f < Wo; ++f) {
        const float4 g4 = *reinterpret_cast<const float4*>(go_s + f * WG_CO + co_t);
        const float* xp = xr + f * sw;
        const float x0 = xp[0], x1 = xp[1], x2 = xp[2], x3 = xp[3];
        acc[0][0] = fmaf(g4.x, x0, acc[0][0]); acc[0][1] = fmaf(g4.x, x1, acc[0][1]); acc[0][2] = fmaf(g4.x, x2, acc[0][2]); acc[0][3] = fmaf(g4.x, x3, acc[0][3]);
        acc[1][0] = fmaf(g4.y, x0, acc[1][0]); acc[1][1] = fmaf(g4.y, x1, acc[1][1]); acc[1][2] = fmaf(g4.y, x2, acc[1][2]); acc[1][3] = fmaf(g4.y, x3, acc[1][3]);
        acc[2][0] = fmaf(g4.z, x0, acc[2][0]); acc[2][1] = fmaf(g4.z, x1, acc[2][1]); acc[2][2] = fmaf(g4.z, x2, acc[2][2]); acc[2][3] = fmaf(g4.z, x3, acc[2][3]);
        acc[3][0] = fmaf(g4.w, x0, acc[3][0]); acc[3][1] = fmaf(g4.w, x1, acc[3][1]); acc[3][2] = fmaf(g4.w, x2, acc[3][2]); acc[3][3] = fmaf(g4.w, x3, acc[3][3]);
      }
    }
  }
  if (!combo_ok) return;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = co0 + co_t + i;
    if (co >= Cout) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int kw = kw_t + j;
      if (kw < KW) atomicAdd(&gw[(((size_t)co * Cin + ci) * KH + kh) * KW + kw], acc[i][j]);
    }
  }
}

// LayerNorm([C,F]) parameter gradients; one CTA per batch item, rows accumulated in registers, one atomicAdd per element per CTA
// G16 = MPA_FMT_* + 1: the gradient comes as 16-bit CP8 planes (one chunk, C <= 8) — what the first convolution's data gradient writes —
// instead of fp32 NCHW (no converter pass, 3.4 instead of 5.2 KB per row)
struct LnGradCp8 {
  const uint16_t* g;
  int TP, P, pf, pt;
};
template <int MAXV, int G16>
__global__ void __launch_bounds__(128) layernorm_cf_param_grad_kernel(const float* __restrict__ x, const float* __restrict__ g, LnGradCp8 gc,
                                                                      float* __restrict__ gw, float* __restrict__ gb, int C, int T, int F,
                                                                      float eps, float gamma_log) {
  __shared__ float sh[8];
  const int b = blockIdx.x;
  const int n = C * F;
  float aw[MAXV], ab[MAXV];
#pragma unroll
  for (int i = 0; i < MAXV; ++i) aw[i] = ab[i] = 0.f;
  // gridDim.y time slices per item (parallelism for small batches); the slices meet in the atomics below
  const int t_per = (T + (int)gridDim.y - 1) / (int)gridDim.y;
  const int t_begin = blockIdx.y * t_per, t_end = min(T, t_begin + t_per);
  for (int t = t_begin; t < t_end; ++t) {
    const float* xr = x + ((size_t)b * C * T + t) * F;
    const float* gr = G16 ? nullptr : g + ((size_t)b * C * T + t) * F;
    const uint16_t* gr16 = G16 ? gc.g + (((size_t)b * gc.TP + gc.pt + t) * gc.P + gc.pf) * 8 : nullptr;
    float v[MAXV];
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int e = threadIdx.x + i * 128;
      float val = 0.f;
      if (e < n) {
        const int c = e / F, f = e - c * F;
        val = xr[(size_t)c * T * F + f];
        if (gamma_log > 0.f) val = logf(__fadd_rn(1.f, __fmul_rn(gamma_log, val)));
        s += val;
      }
      v[i] = val;
    }
    s = warp_sum(s);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    const float mean = (sh[0] + sh[1] + sh[2] + sh[3]) / n;
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int e = threadIdx.x + i * 128;
      if (e < n) {
        const float d = v[i] - mean;
        q += d * d;
      }
    }
    q = warp_sum(q);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[4 + (threadIdx.x >> 5)] = q;
    __syncthreads();
    const float rstd = rsqrtf((sh[4] + sh[5] + sh[6] + sh[7]) / n + eps);
#pragma unroll
    for (int i = 0; i < MAXV; ++i) {
      const int e = threadIdx.x + i * 128;
      if (e < n) {
        const int c = e / F, f = e - c * F;
        float go;
        if (G16 == 0) {
          go = gr[(size_t)c * T * F + f];
        } else {
          const uint16_t h = gr16[(size_t)f * 8 + c];
          go = G16 == MPA_FMT_BF16 + 1 ? __uint_as_float((uint32_t)h << 16) : __half2float(__ushort_as_half(h));
        }
        aw[i] = fmaf(go, (v[i] - mean) * rstd, aw[i]);
        ab[i] += go;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int e = threadIdx.x + i * 128;
    if (e < n) {
      atomicAdd(&gw[e], aw[i]);
      atomicAdd(&gb[e], ab[i]);
    }
  }
}

__global__ void add_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out, long long n) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) out[i] = a[i] + b[i];
}

__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n, float lr,
                             float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt, float grad_scale) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * grad_scale;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

// AdamW of an fp16 training step with dynamic loss scaling (torch.amp.GradScaler + torch.optim.AdamW): skipped entirely when the overflow
// check set *found_inf; otherwise the update of adamw_kernel on g * grad_scale / *loss_scale, bias-corrected for the (*applied + 1)-th
// applied step.  Everything the decision needs is read from device memory: no host synchronisation, the same in eager and replayed steps.
__global__ void adamw_scaled_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                                    float lr, float b1, float b2, float eps, float wd, float grad_scale, const int* __restrict__ found_inf,
                                    const float* __restrict__ loss_scale, const int* __restrict__ applied) {
  if (*found_inf) return;
  const float step = (float)(*applied + 1);
  const float bc1 = 1.f - powf(b1, step), bc2_sqrt = sqrtf(1.f - powf(b2, step));
  const float gs = grad_scale * (1.f / *loss_scale);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * gs;
    float pi = p[i] * (1.f - lr * wd);
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}

// torch.amp.GradScaler.update after the step: on an overflow the scale backs off and the growth tracker restarts; otherwise the step
// counts as applied and, after growth_interval clean steps in a row, the scale grows (unless that would make it non-finite).
__global__ void loss_scale_update_kernel(const int* __restrict__ found_inf, float* __restrict__ loss_scale, int* __restrict__ growth_tracker,
                                         int* __restrict__ applied, float growth_factor, float backoff_factor, int growth_interval) {
  if (*found_inf) {
    *loss_scale *= backoff_factor;
    *growth_tracker = 0;
    return;
  }
  *applied += 1;
  const int clean = *growth_tracker + 1;
  if (clean >= growth_interval) {
    const float grown = *loss_scale * growth_factor;
    if (isfinite(grown)) *loss_scale = grown;
    *growth_tracker = 0;
  } else {
    *growth_tracker = clean;
  }
}

}  // namespace mpa

using namespace mpa;

extern "C" {

int mpa_add_f32(const float* a, const float* b, float* out, long long n, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(a && b && out && n > 0, "add: bad argument");
  add_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(a, b, out, n);
  MPA_CHECK_LAUNCH("add");
  return MPA_OK;
}

int mpa_act_bwd_f32(const float* out, const float* g_out, float* g_in, long long n, int act, float act_param, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(out && g_out && g_in && n > 0, "act_bwd: bad argument");
  act_bwd_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(out, g_out, g_in, n, act, act_param);
  MPA_CHECK_LAUNCH("act_bwd");
  return MPA_OK;
}

int mpa_maxpool_time_bwd_f32(const float* a, const float* g_pool, float* g_a, int B, int C, int T, int F, int k, int act, float act_param,
                             void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(a && g_pool && g_a && B > 0 && C > 0 && T > 0 && F > 0 && k >= 1 && (k & 1), "maxpool_time_bwd: bad argument");
  if ((k == 3 || k == 13) && T > k / 2) {
    const int threads = pool_col_threads(F);
    const dim3 grid(B * C, ceil_div(F, threads));
    const DropoutArgs nod{0.f, 0ull, 0ull, nullptr, 0ull};
    if (pool13_table_eligible(k, T, F)) {
      MPA_REQUIRE(pool13_table_launch(a, g_pool, g_a, B, C, F, act, act_param, nod, (cudaStream_t)stream) == MPA_OK, "maxpool_time_bwd: shared memory opt-in failed");
      MPA_CHECK_LAUNCH("maxpool_time_bwd_col");
      return MPA_OK;
    }
    if (k == 3) maxpool_time_bwd_col_kernel<3><<<grid, threads, 0, (cudaStream_t)stream>>>(a, g_pool, g_a, T, F, act, act_param, nod);
    else maxpool_time_bwd_col_kernel<13><<<grid, threads, 0, (cudaStream_t)stream>>>(a, g_pool, g_a, T, F, act, act_param, nod);
    MPA_CHECK_LAUNCH("maxpool_time_bwd_col");
    return MPA_OK;
  }
  const size_t smem = 2 * (size_t)T * kPoolBwdCols * sizeof(float);
  MPA_REQUIRE(smem <= 160 * 1024, "maxpool_time_bwd: T = %d too long for the column tile", T);
  if (smem > 48 * 1024) cudaFuncSetAttribute(maxpool_time_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  maxpool_time_bwd_kernel<<<dim3(B * C, ceil_div(F, kPoolBwdCols)), kPoolBwdCols * kPoolBwdRowGroups, smem, (cudaStream_t)stream>>>(a, g_pool, g_a, T, F, k, act, act_param);
  MPA_CHECK_LAUNCH("maxpool_time_bwd");
  return MPA_OK;
}

int mpa_dropout_f32(const float* x, float* out, long long n, float p, unsigned long long seed, unsigned long long offset, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && n > 0 && p >= 0.f && p < 1.f, "dropout: bad argument");
  dropout_kernel<<<grid_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(x, out, n, p, seed, offset, nullptr, 0);
  MPA_CHECK_LAUNCH("dropout");
  return MPA_OK;
}

int mpa_dropout_dev_f32(const float* x, float* out, long long n, float p, unsigned long long seed, unsigned long long site,
                        const long long* step_dev, unsigned long long step_mul, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out && step_dev && n > 0 && p >= 0.f && p < 1.f, "dropout_dev: bad argument");
  dropout_kernel<<<grid_for((n + 3) / 4, 256), 256, 0, (cudaStream_t)stream>>>(x, out, n, p, seed, site, step_dev, step_mul);
  MPA_CHECK_LAUNCH("dropout");
  return MPA_OK;
}

int mpa_conv2d_dgrad_f32(const float* g_out, const float* w, float* g_in, int B, int Cin, int H, int W, int Cout, int KH, int KW, int sh, int sw,
                         int ph, int pw, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(g_out && w && g_in && B > 0 && Cin > 0 && Cout > 0 && H > 0 && W > 0, "conv2d_dgrad: bad argument");
  const int Ho = (H + 2 * ph - KH) / sh + 1, Wo = (W + 2 * pw - KW) / sw + 1;
  const long long total = (long long)B * Cin * H * W;
  conv_dgrad_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(g_out, w, g_in, total, Cin, H, W, Cout, Ho, Wo, KH, KW, sh, sw, ph, pw);
  MPA_CHECK_LAUNCH("conv2d_dgrad");
  return MPA_OK;
}

int mpa_conv2d_wgrad_f32(const float* x, const float* g_out, float* g_w, float* g_b, int B, int Cin, int H, int W, int Cout, int KH, int KW, int sh,
                         int sw, int ph, int pw, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && g_out && g_w && B > 0 && Cin > 0 && Cout > 0 && H > 0 && W > 0 && KH > 0 && KW > 0, "conv2d_wgrad: bad argument");
  const int Ho = (H + 2 * ph - KH) / sh + 1, Wo = (W + 2 * pw - KW) / sw + 1;
  MPA_REQUIRE(Ho > 0 && Wo > 0, "conv2d_wgrad: empty output");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(g_w, 0, sizeof(float) * (size_t)Cout * Cin * KH * KW, st);
  const int n_combos = Cin * KH;
  const long long n_rows = (long long)B * Ho;
  // enough CTAs to fill the machine a few times; every CTA ends with <= 4096 atomics
  const int gx = ceil_div(Cout, WG_CO), gy = ceil_div(n_combos, WG_COMBOS);
  long long want = (148LL * 8) / ((long long)gx * gy);
  if (want < 1) want = 1;
  if (want > n_rows) want = n_rows;
  const int rows_per_cta = (int)((n_rows + want - 1) / want);
  const int gz = (int)((n_rows + rows_per_cta - 1) / rows_per_cta);
  const int XW = (Wo - 1) * sw + WG_KW;
  const size_t smem = ((size_t)Wo * WG_CO + (size_t)WG_COMBOS * XW) * sizeof(float);
  MPA_REQUIRE(smem <= 200 * 1024, "conv2d_wgrad: row of %d outputs needs %zu B of shared memory", Wo, smem);
  MPA_REQUIRE(KW <= WG_KW, "conv2d_wgrad: kernel width %d > %d not supported", KW, WG_KW);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("conv2d_wgrad: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return MPA_ERR_CUDA;
    }
  }
  conv_wgrad_kernel<<<dim3(gx, gy, gz), 256, smem, st>>>(x, g_out, g_w, B, Cin, H, W, Cout, Ho, Wo, KH, KW, sh, sw, ph, pw, n_combos, rows_per_cta);
  MPA_CHECK_LAUNCH("conv2d_wgrad");
  if (g_b) {
    int rc = channel_sum_launch(g_out, g_b, B, Cout, Ho * Wo, st);
    if (rc != MPA_OK) return rc;
    MPA_CHECK_LAUNCH("bias_grad");
  }
  return MPA_OK;
}

int mpa_maxpool_time_bwd_dropout_f32(const float* a, const float* g_out, float* g_a, int B, int C, int T, int F, int k, int act, float act_param,
                                     float p, unsigned long long seed, unsigned long long offset, const long long* step_dev,
                                     unsigned long long step_mul, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(a && g_out && g_a && B > 0 && C > 0 && F > 0 && (k == 3 || k == 13) && T > k / 2 && p >= 0.f && p < 1.f,
              "maxpool_time_bwd_dropout: bad argument (k must be 3 or 13)");
  const int threads = pool_col_threads(F);
  const dim3 grid(B * C, ceil_div(F, threads));
  const DropoutArgs d{p, seed, offset, step_dev, step_mul};
  if (pool13_table_eligible(k, T, F)) {
    MPA_REQUIRE(pool13_table_launch(a, g_out, g_a, B, C, F, act, act_param, d, (cudaStream_t)stream) == MPA_OK, "maxpool_time_bwd_dropout: shared memory opt-in failed");
    MPA_CHECK_LAUNCH("maxpool_time_bwd_dropout");
    return MPA_OK;
  }
  if (k == 3) maxpool_time_bwd_col_kernel<3><<<grid, threads, 0, (cudaStream_t)stream>>>(a, g_out, g_a, T, F, act, act_param, d);
  else maxpool_time_bwd_col_kernel<13><<<grid, threads, 0, (cudaStream_t)stream>>>(a, g_out, g_a, T, F, act, act_param, d);
  MPA_CHECK_LAUNCH("maxpool_time_bwd_dropout");
  return MPA_OK;
}

int mpa_layernorm_cf_param_grad_f32(const float* x, const float* g_out, float* g_w, float* g_b, int B, int C, int T, int F, float eps,
                                    float gamma_log, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && g_out && g_w && g_b && B > 0 && C > 0 && T > 0 && F > 0 && C * F <= 128 * 11, "layernorm_cf_param_grad: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(g_w, 0, sizeof(float) * (size_t)C * F, st);
  cudaMemsetAsync(g_b, 0, sizeof(float) * (size_t)C * F, st);
  int slices = ceil_div(148 * 8, B);
  slices = slices < 1 ? 1 : (slices > T ? T : slices);
  layernorm_cf_param_grad_kernel<11, 0><<<dim3(B, slices), 128, 0, st>>>(x, g_out, LnGradCp8{}, g_w, g_b, C, T, F, eps, gamma_log);
  MPA_CHECK_LAUNCH("layernorm_cf_param_grad");
  return MPA_OK;
}

int mpa_layernorm_cf_param_grad_cp8(const float* x, const void* g_cp8, float* g_w, float* g_b, int B, int C, int T, int F, int pitch, int pf, int pt,
                                    int fmt, float eps, float gamma_log, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && g_cp8 && g_w && g_b && B > 0 && C > 0 && C <= 8 && T > 0 && F > 0 && C * F <= 128 * 11 && pitch >= pf + F && pt >= 0 &&
                  (fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16),
              "layernorm_cf_param_grad_cp8: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  cudaMemsetAsync(g_w, 0, sizeof(float) * (size_t)C * F, st);
  cudaMemsetAsync(g_b, 0, sizeof(float) * (size_t)C * F, st);
  int slices = ceil_div(148 * 8, B);
  slices = slices < 1 ? 1 : (slices > T ? T : slices);
  const LnGradCp8 gc{(const uint16_t*)g_cp8, T + 2 * pt, pitch, pf, pt};
  if (fmt == MPA_FMT_BF16)
    layernorm_cf_param_grad_kernel<11, MPA_FMT_BF16 + 1><<<dim3(B, slices), 128, 0, st>>>(x, nullptr, gc, g_w, g_b, C, T, F, eps, gamma_log);
  else
    layernorm_cf_param_grad_kernel<11, MPA_FMT_F16 + 1><<<dim3(B, slices), 128, 0, st>>>(x, nullptr, gc, g_w, g_b, C, T, F, eps, gamma_log);
  MPA_CHECK_LAUNCH("layernorm_cf_param_grad_cp8");
  return MPA_OK;
}

int mpa_adamw_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1, float beta2, float eps,
                  float weight_decay, int step, float grad_scale, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(param && grad && exp_avg && exp_avg_sq && n > 0 && step >= 1, "adamw: bad argument");
  const float bc1 = 1.f - powf(beta1, (float)step);
  const float bc2s = sqrtf(1.f - powf(beta2, (float)step));
  adamw_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, bc1,
                                                                    bc2s, grad_scale);
  MPA_CHECK_LAUNCH("adamw");
  return MPA_OK;
}

int mpa_adamw_scaled_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1, float beta2,
                         float eps, float weight_decay, float grad_scale, const int* found_inf, float* loss_scale, int* growth_tracker,
                         int* applied_steps, float growth_factor, float backoff_factor, int growth_interval, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(param && grad && exp_avg && exp_avg_sq && found_inf && loss_scale && growth_tracker && applied_steps && n > 0 && growth_interval >= 1,
              "adamw_scaled: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  adamw_scaled_kernel<<<grid_for(n, 256), 256, 0, st>>>(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, grad_scale,
                                                        found_inf, loss_scale, applied_steps);
  MPA_CHECK_LAUNCH("adamw_scaled");
  loss_scale_update_kernel<<<1, 1, 0, st>>>(found_inf, loss_scale, growth_tracker, applied_steps, growth_factor, backoff_factor, growth_interval);
  MPA_CHECK_LAUNCH("loss_scale_update");
  return MPA_OK;
}

}  // extern "C"
