// HCQT feature extraction (reference: libdl/data_preprocessing/hcqt.py:89-164, which delegates to librosa.cqt /
// librosa.estimate_tuning).  B200 formulation: a batched multirate constant-Q filterbank.
//   * mpa_decimate(2)_f32   : the 2:1 kaiser_fast windowed-sinc decimator chain (one launch per octave level) and the one-shot
//                              2^c:1 decimator of librosa's early down-sampling (compute_hcqt's low harmonics)
//   * mpa_cqt_level_f32      : one CTA per frame: gather the reflect-padded frame, radix-2 FFT in shared memory,
//                              contract the spectrum with the banded (sparsified) filter rows of EVERY CQT that
//                              uses this rate, magnitude, per-row scale, scatter into the [H][frames][bins] patch
//                              layout the networks read.  No spectrum or complex CQT ever reaches HBM.
//   * mpa_estimate_tuning_f32: STFT-2048 (hann) + parabolic peak picking fused in one kernel, then an exact
//                              median (radix select) + 100-bin residual histogram in a single-CTA kernel; the result
//                              stays on the device as an index into the pre-built per-tuning filter banks.
// HBM-bound by design: per 30 s clip the algorithmic traffic is 2.65 MB in + 6.7 MB out.
#include "common.cuh"
#include <string.h>

namespace mpa {

// numpy.pad(mode='reflect') for any pad width: reflection without edge repeat has period 2(n-1)
__device__ __forceinline__ long long reflect_index(long long i, long long n) {
  if (i >= 0 && i < n) return i;
  const long long p = 2 * (n - 1);
  i %= p;
  if (i < 0) i += p;
  return i < n ? i : p - i;
}

// in-place radix-2 DIT FFT on shared memory; `a` holds the bit-reversed input; tw[k] = exp(-2*pi*i*k/n), k < n/2
__device__ __forceinline__ void fft_smem(float2* a, const float2* tw, int n, int log2n) {
  for (int s = 1; s <= log2n; ++s) {
    const int half = 1 << (s - 1);
    const int tstep = n >> s;
    for (int j = threadIdx.x; j < n / 2; j += blockDim.x) {
      const int pos = j & (half - 1);
      const int i0 = ((j - pos) << 1) + pos;
      const int i1 = i0 + half;
      const float2 w = tw[pos * tstep];
      const float2 u = a[i0], v = a[i1];
      const float2 t = make_float2(w.x * v.x - w.y * v.y, w.x * v.y + w.y * v.x);
      a[i0] = make_float2(u.x + t.x, u.y + t.y);
      a[i1] = make_float2(u.x - t.x, u.y - t.y);
    }
    __syncthreads();
  }
}

__device__ __forceinline__ void load_frame_bitrev(float2* a, float2* tw, const float* __restrict__ y, long long n, const float* __restrict__ window,
                                                  long long start, int n_fft, int log2n) {
  for (int k = threadIdx.x; k < n_fft; k += blockDim.x) {
    float v = y[reflect_index(start + k, n)];
    if (window) v *= window[k];
    a[__brev((unsigned)k) >> (32 - log2n)] = make_float2(v, 0.f);
  }
  for (int k = threadIdx.x; k < n_fft / 2; k += blockDim.x) {
    float s, c;
    sincospif(-2.0f * (float)k / (float)n_fft, &s, &c);
    tw[k] = make_float2(c, s);
  }
  __syncthreads();
}

// out[t] = gain * sum_{|j| < n_half} h[|j|] * yin[D*t + j]  (taps outside the signal are skipped, as resampy does); D = 2 for the
// octave chain, 2^c for librosa's one-shot early down-sampling (gain sqrt(D): librosa's scale=True) and for librosa.load's
// 44.1 -> 22.05 kHz kaiser_best resampling (gain 1).  float64 accumulation, one rounding to fp32.
__global__ void decimate_kernel(const float* __restrict__ yin, float* __restrict__ yout, const float* __restrict__ half, int n_half, int factor,
                                double gain, long long n_in, long long n_out_real, long long n_out) {
  extern __shared__ float h[];
  for (int i = threadIdx.x; i < n_half; i += blockDim.x) h[i] = half[i];
  __syncthreads();
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n_out; t += (long long)gridDim.x * blockDim.x) {
    double acc = 0.0;
    if (t < n_out_real) {
      const long long c = (long long)factor * t;
#pragma unroll 1
      for (int j = -(n_half - 1); j <= n_half - 1; ++j) {
        long long i = c + j;
        if (i >= 0 && i < n_in) acc += (double)h[j < 0 ? -j : j] * (double)yin[i];
      }
      acc *= gain;
    }
    yout[t] = (float)acc;
  }
}

// one CTA per output frame
__global__ void __launch_bounds__(256) cqt_level_kernel(const float* __restrict__ y, long long n, int n_fft, int log2n, int hop, const float2* __restrict__ basis,
                                                        const int* __restrict__ band_start, const float* __restrict__ row_scale, int n_rows, int band,
                                                        const int* __restrict__ tuning_idx, const int* __restrict__ dest, int n_dest,
                                                        float* __restrict__ out, int out_frames, int out_bins) {
  extern __shared__ float2 sm2[];
  float2* a = sm2;              // [n_fft]
  float2* tw = sm2 + n_fft;     // [n_fft/2]
  const int t = blockIdx.x;
  load_frame_bitrev(a, tw, y, n, nullptr, (long long)t * hop - n_fft / 2, n_fft, log2n);
  fft_smem(a, tw, n_fft, log2n);
  const int tune = tuning_idx ? tuning_idx[0] : 0;
  const float2* bs = basis + (size_t)tune * n_rows * band;
  const int* st = band_start + (size_t)tune * n_rows;
  const float* sc = row_scale + (size_t)tune * n_rows;
  const int nb = n_fft / 2 + 1;
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) {
    const int s0 = st[r];
    const float2* br = bs + (size_t)r * band;
    float re = 0.f, im = 0.f;
    for (int f = 0; f < band; ++f) {
      const int bin = s0 + f;
      if (bin < nb) {
        const float2 b = br[f], x = a[bin];
        re = fmaf(b.x, x.x, re);
        re = fmaf(-b.y, x.y, re);
        im = fmaf(b.x, x.y, im);
        im = fmaf(b.y, x.x, im);
      }
    }
    const float mag = sqrtf(re * re + im * im) * sc[r];
    for (int d = 0; d < n_dest; ++d) {
      const int code = dest[r * n_dest + d];
      if (code >= 0) out[((size_t)(code >> 16) * out_frames + t) * out_bins + (code & 0xffff)] = mag;
    }
  }
}

// Every (rate, FFT size) level of one HCQT in ONE launch: blockIdx.y selects the level, blockIdx.x the frame.  The levels are independent
// of each other (each reads its own decimated signal and scatters into its own rows of the output), and a single level (1,292 CTAs of
// one small FFT) does not fill the chip.  The per-level arguments travel in the kernel parameters.
constexpr int kMaxCqtLevels = 16;
struct CqtLevelsParams {
  mpa_cqt_level lv[kMaxCqtLevels];
  int log2n[kMaxCqtLevels];
  int n_frames, band, out_frames, out_bins;
  const int* tuning_idx;
  float* out;
};
__global__ void __launch_bounds__(256) cqt_levels_kernel(const __grid_constant__ CqtLevelsParams p) {
  extern __shared__ float2 sm2[];
  const mpa_cqt_level& L = p.lv[blockIdx.y];
  const int n_fft = L.n_fft, log2n = p.log2n[blockIdx.y];
  float2* a = sm2;              // [n_fft]
  float2* tw = sm2 + n_fft;     // [n_fft/2]
  const int t = blockIdx.x;
  load_frame_bitrev(a, tw, L.y, L.n, nullptr, (long long)t * L.hop - n_fft / 2, n_fft, log2n);
  fft_smem(a, tw, n_fft, log2n);
  const int tune = p.tuning_idx ? p.tuning_idx[0] : 0;
  const int n_rows = L.n_rows, band = p.band;
  const float2* bs = reinterpret_cast<const float2*>(L.basis) + (size_t)tune * n_rows * band;
  const int* st = L.band_start + (size_t)tune * n_rows;
  const float* sc = L.row_scale + (size_t)tune * n_rows;
  const int nb = n_fft / 2 + 1;
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) {
    const int s0 = st[r];
    const float2* br = bs + (size_t)r * band;
    float re = 0.f, im = 0.f;
    for (int f = 0; f < band; ++f) {
      const int bin = s0 + f;
      if (bin < nb) {
        const float2 b = br[f], x = a[bin];
        re = fmaf(b.x, x.x, re);
        re = fmaf(-b.y, x.y, re);
        im = fmaf(b.x, x.y, im);
        im = fmaf(b.y, x.x, im);
      }
    }
    const float mag = sqrtf(re * re + im * im) * sc[r];
    for (int d = 0; d < L.n_dest; ++d) {
      const int code = L.dest[r * L.n_dest + d];
      if (code >= 0) p.out[((size_t)(code >> 16) * p.out_frames + t) * p.out_bins + (code & 0xffff)] = mag;
    }
  }
}

// ---- backward: the adjoint of cqt_levels_kernel, of the reflect-padded framing and of decimate_kernel --------------------------------
// Every stage before the magnitude is linear, so with G_r = dL/d(re, im) of row r's complex response C_r,
//   dL/dx_k = Re( sum_bin V[bin] e^{-2 pi i bin k / n_fft} ),  V[bin] = sum_r w_r b_{r, bin - s0_r},  w_r = scale_r * g_r * conj(C_r) / |C_r|
// (g_r = sum of the upstream gradient over the row's destinations; w_r = 0 where |C_r| = 0, the convention of torch.abs): a transposed
// banded contraction followed by one forward FFT.  The spectrum is recomputed from the signal (the forward keeps nothing).  Each thread
// owns one output element and sums in a fixed order: two runs give the same bits, no atomics.
struct CqtLevelsBwdParams {
  mpa_cqt_level lv[kMaxCqtLevels];
  mpa_cqt_level_grad gr[kMaxCqtLevels];
  int log2n[kMaxCqtLevels];
  size_t ws_off[kMaxCqtLevels];      // floats: level l's [n_frames][n_fft] frame gradients
  int n_frames, band, out_frames, out_bins;
  const int* tuning_idx;
  const float* g_out;
  float* ws;
};
// one CTA per (frame, level): the frame's gradient wrt its n_fft (reflect-padded) samples -> ws
__global__ void __launch_bounds__(256) cqt_levels_bwd_kernel(const __grid_constant__ CqtLevelsBwdParams p) {
  extern __shared__ float2 sm2[];
  const mpa_cqt_level& L = p.lv[blockIdx.y];
  const int n_fft = L.n_fft, log2n = p.log2n[blockIdx.y];
  float2* a = sm2;              // [n_fft]
  float2* tw = sm2 + n_fft;     // [n_fft/2]
  float2* w = tw + n_fft / 2;   // [n_rows]
  const int t = blockIdx.x;
  load_frame_bitrev(a, tw, L.y, L.n, nullptr, (long long)t * L.hop - n_fft / 2, n_fft, log2n);
  fft_smem(a, tw, n_fft, log2n);
  const int tune = p.tuning_idx ? p.tuning_idx[0] : 0;
  const int n_rows = L.n_rows, band = p.band;
  const float2* bs = reinterpret_cast<const float2*>(L.basis) + (size_t)tune * n_rows * band;
  const int* st = L.band_start + (size_t)tune * n_rows;
  const float* sc = L.row_scale + (size_t)tune * n_rows;
  const int nb = n_fft / 2 + 1;
  for (int r = threadIdx.x; r < n_rows; r += blockDim.x) {
    const int s0 = st[r];
    const float2* br = bs + (size_t)r * band;
    float re = 0.f, im = 0.f;
    for (int f = 0; f < band; ++f) {            // the forward's contraction, same order
      const int bin = s0 + f;
      if (bin < nb) {
        const float2 b = br[f], x = a[bin];
        re = fmaf(b.x, x.x, re);
        re = fmaf(-b.y, x.y, re);
        im = fmaf(b.x, x.y, im);
        im = fmaf(b.y, x.x, im);
      }
    }
    float g = 0.f;
    for (int d = 0; d < L.n_dest; ++d) {
      const int code = L.dest[r * L.n_dest + d];
      if (code >= 0) g += p.g_out[((size_t)(code >> 16) * p.out_frames + t) * p.out_bins + (code & 0xffff)];
    }
    const float m = sqrtf(re * re + im * im);
    const float k = (m > 0.f) ? g * sc[r] / m : 0.f;
    w[r] = make_float2(k * re, -k * im);
  }
  __syncthreads();                              // the spectrum in `a` is dead from here on
  // transposed contraction over the bin -> rows table (rows whose band covers the bin), written bit-reversed for the FFT
  const int* off = p.gr[blockIdx.y].bin_off + (size_t)tune * (nb + 1);
  const int* rows = p.gr[blockIdx.y].bin_rows + (size_t)tune * n_rows * band;
  for (int k = threadIdx.x; k < n_fft; k += blockDim.x) {
    float vr = 0.f, vi = 0.f;
    if (k < nb) {
      for (int e = off[k]; e < off[k + 1]; ++e) {
        const int r = rows[e];
        const float2 b = bs[(size_t)r * band + (k - st[r])], wr = w[r];
        vr = fmaf(b.x, wr.x, vr);
        vr = fmaf(-b.y, wr.y, vr);
        vi = fmaf(b.x, wr.y, vi);
        vi = fmaf(b.y, wr.x, vi);
      }
    }
    a[__brev((unsigned)k) >> (32 - log2n)] = make_float2(vr, vi);
  }
  __syncthreads();
  fft_smem(a, tw, n_fft, log2n);
  float* out = p.ws + p.ws_off[blockIdx.y] + (size_t)t * n_fft;
  for (int k = threadIdx.x; k < n_fft; k += blockDim.x) out[k] = a[k].x;
}

__device__ __forceinline__ long long floor_div(long long a, long long b) {      // b > 0
  const long long q = a / b;
  return (a % b != 0 && a < 0) ? q - 1 : q;
}

// adjoint of the reflect-padded framing for one sample i of an n-sample signal: padded position q (frame t covers q = t*hop - n_fft/2 + k,
// k < n_fft) reads sample i exactly when q = +-i (mod 2(n-1)), so every preimage q of i is enumerated (a signal shorter than n_fft has
// several) and the frames covering it are summed, frame-major
__device__ double ola_sample(const float* __restrict__ ws, long long i, long long n, int n_fft, int hop, int n_frames) {
  const long long P = 2 * (n - 1);
  const long long lo = -(long long)(n_fft / 2), hi = (long long)(n_frames - 1) * hop + n_fft / 2;      // padded positions [lo, hi)
  double acc = 0.0;
  const int nsets = (i == 0 || i == n - 1) ? 1 : 2;     // at the two end samples +i and -i name the same residue class
  for (int s = 0; s < nsets; ++s) {
    const long long base = s == 0 ? i : -i;
    const long long m1 = floor_div(hi - 1 - base, P);
    for (long long m = floor_div(lo - base + P - 1, P); m <= m1; ++m) {
      const long long u = base + m * P + n_fft / 2;     // = t*hop + k
      const long long t1 = min((long long)n_frames - 1, u / hop);
      const long long t0 = max(0LL, floor_div(u - n_fft, hop) + 1);
      for (long long t = t0; t <= t1; ++t) acc += (double)ws[t * n_fft + (u - t * hop)];
    }
  }
  return acc;
}

// overlap-add of the frame gradients into the level signals' gradients; blockIdx.y = one signal, summing every level that reads it
struct CqtOlaParams {
  int grp_first[kMaxCqtLevels + 1];    // levels of signal g: order[grp_first[g] .. grp_first[g+1])
  int order[kMaxCqtLevels];
  int n_fft[kMaxCqtLevels], hop[kMaxCqtLevels];
  size_t ws_off[kMaxCqtLevels];
  float* g_y[kMaxCqtLevels];
  long long n[kMaxCqtLevels];          // per signal
  int n_frames, accumulate;
  const float* ws;
};
__global__ void __launch_bounds__(256) cqt_ola_bwd_kernel(const __grid_constant__ CqtOlaParams p) {
  const int g = blockIdx.y;
  const long long n = p.n[g];
  float* gy = p.g_y[g];
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double acc = p.accumulate ? (double)gy[i] : 0.0;
    for (int q = p.grp_first[g]; q < p.grp_first[g + 1]; ++q) {
      const int l = p.order[q];
      acc += ola_sample(p.ws + p.ws_off[l], i, n, p.n_fft[l], p.hop[l], p.n_frames);
    }
    gy[i] = (float)acc;
  }
}

// transpose of decimate_kernel: g_in[i] (+)= gain * sum_{t < n_out_real, |i - D*t| < n_half} h[|i - D*t|] * g_out[t]; float64 accumulation
__global__ void decimate_adjoint_kernel(const float* __restrict__ g_out, float* __restrict__ g_in, const float* __restrict__ half, int n_half,
                                        int factor, double gain, long long n_in, long long n_out_real, int accumulate) {
  extern __shared__ float h[];
  for (int i = threadIdx.x; i < n_half; i += blockDim.x) h[i] = half[i];
  __syncthreads();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_in; i += (long long)gridDim.x * blockDim.x) {
    const long long t0 = max(0LL, -floor_div(-(i - (n_half - 1)), factor));
    const long long t1 = min(n_out_real - 1, (i + n_half - 1) / factor);
    double acc = 0.0;
#pragma unroll 1
    for (long long t = t0; t <= t1; ++t) {
      const long long j = i - (long long)factor * t;
      acc += (double)h[j < 0 ? -j : j] * (double)g_out[t];
    }
    acc *= gain;
    g_in[i] = accumulate ? (float)((double)g_in[i] + acc) : (float)acc;
  }
}

// STFT-2048 (hann) + piptrack peak picking; peaks appended to ws: [0]=count, then pitch[max], mag[max]
__global__ void __launch_bounds__(256) tuning_peaks_kernel(const float* __restrict__ y, long long n, const float* __restrict__ window, float sr,
                                                           int* __restrict__ counter, float* __restrict__ pitch, float* __restrict__ mag, int max_peaks) {
  constexpr int NFFT = 2048, LOG2N = 11, NB = 1025;
  __shared__ float2 a[NFFT];
  __shared__ float2 tw[NFFT / 2];
  __shared__ float red[8];
  const int t = blockIdx.x;
  load_frame_bitrev(a, tw, y, n, window, (long long)t * 512 - NFFT / 2, NFFT, LOG2N);
  fft_smem(a, tw, NFFT, LOG2N);
  float* S = reinterpret_cast<float*>(tw);       // reuse: 1025 floats fit in the 8 KB twiddle table
  float mx = 0.f;
  for (int k = threadIdx.x; k < NB; k += blockDim.x) {
    const float2 v = a[k];
    const float m = sqrtf(v.x * v.x + v.y * v.y);
    mx = fmaxf(mx, m);
    S[k] = m;     // tw is dead after the FFT; every thread passed the trailing barrier of fft_smem
  }
  mx = warp_max(mx);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
  for (int i = 1; i < 8; ++i) mx = fmaxf(mx, red[i]);
  const float ref = 0.1f * mx;
  const float binhz = sr / (float)NFFT;
  for (int k = threadIdx.x + 1; k < NB - 1; k += blockDim.x) {
    const double fk = (double)k * (double)sr / 2.0 / (double)(NB - 1);       // fft_frequencies = linspace(0, sr/2, 1025)
    if (fk < 150.0 || fk >= 4000.0) continue;
    const float s0 = S[k - 1], s1 = S[k], s2 = S[k + 1];
    const float x0 = s0 > ref ? s0 : 0.f, x1 = s1 > ref ? s1 : 0.f, x2 = s2 > ref ? s2 : 0.f;
    if (!(x1 > x0 && x1 >= x2)) continue;
    const float avg = 0.5f * (s2 - s0);
    float shift = 2.f * s1 - s2 - s0;
    shift = avg / (shift + (fabsf(shift) < 1.17549435e-38f ? 1.f : 0.f));
    const float p = (float)(((double)k + (double)shift) * (double)sr / (double)NFFT);
    const float m = s1 + 0.5f * avg * shift;
    if (p > 0.f) {
      const int slot = atomicAdd(counter, 1);
      if (slot < max_peaks) {
        pitch[slot] = p;
        mag[slot] = m;
      }
    }
  }
  (void)binhz;
}

// single CTA: exact median of mag (two order statistics by 4-pass radix select), then residual histogram
__global__ void __launch_bounds__(1024) tuning_finalize_kernel(const int* __restrict__ counter, const float* __restrict__ pitch, const float* __restrict__ mag,
                                                               int max_peaks, int bins_per_octave, int* __restrict__ tuning_idx) {
  __shared__ unsigned hist[256];
  __shared__ unsigned sel_prefix, sel_rank;
  __shared__ float kth[2];
  __shared__ int counts[100];
  const int cnt = min(counter[0], max_peaks);
  if (cnt <= 0) {
    if (threadIdx.x == 0) tuning_idx[0] = 50;     // pitch_tuning() of an empty set returns 0.0
    return;
  }
  for (int which = 0; which < 2; ++which) {
    unsigned rank = which == 0 ? (unsigned)((cnt - 1) / 2) : (unsigned)(cnt / 2);     // 0-based order statistic
    unsigned prefix = 0, mask = 0;
    for (int pass = 3; pass >= 0; --pass) {
      for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
      __syncthreads();
      for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
        const unsigned u = __float_as_uint(mag[i]);
        if ((u & mask) == prefix) atomicAdd(&hist[(u >> (8 * pass)) & 255u], 1u);
      }
      __syncthreads();
      if (threadIdx.x == 0) {
        unsigned acc = 0, d = 0;
        for (; d < 256; ++d) {
          if (acc + hist[d] > rank) break;
          acc += hist[d];
        }
        sel_prefix = prefix | (d << (8 * pass));
        sel_rank = rank - acc;
      }
      __syncthreads();
      prefix = sel_prefix;
      rank = sel_rank;
      mask |= 255u << (8 * pass);
      __syncthreads();
    }
    if (threadIdx.x == 0) kth[which] = __uint_as_float(prefix);
    __syncthreads();
  }
  // np.median: mean of the two middle order statistics (float32 arithmetic on float32 data)
  const float threshold = (cnt & 1) ? kth[0] : 0.5f * (kth[0] + kth[1]);
  for (int i = threadIdx.x; i < 100; i += blockDim.x) counts[i] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
    if (mag[i] >= threshold) {
      // float32 chain as numpy evaluates it on a float32 array: log2(f / (440/16)) * bpo  mod 1
      const float octs = log2f(pitch[i] / 27.5f);
      float r = (float)bins_per_octave * octs;
      r = r - floorf(r);
      if (r >= 1.0f) r = 0.f;
      if (r >= 0.5f) r -= 1.0f;
      // np.histogram(residual, linspace(-0.5, 0.5, 101)): edges e_i = i*0.01 + (-0.5) in float64, last bin closed
      const double x = (double)r;
      int b = (int)floor((x + 0.5) * 100.0);
      b = max(0, min(99, b));
      while (b > 0 && x < __dadd_rn(__dmul_rn((double)b, 0.01), -0.5)) --b;
      while (b < 99 && x >= __dadd_rn(__dmul_rn((double)(b + 1), 0.01), -0.5)) ++b;
      atomicAdd(&counts[b], 1);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int best = 0;
    for (int i = 1; i < 100; ++i)
      if (counts[i] > counts[best]) best = i;
    tuning_idx[0] = best;
  }
}

// General-ratio band-limited resampling = resampy's table walk (resample_f) with one thread per output sample: output t sits at input
// time t / ratio; both filter wings walk the interpolation window `win` (float64, num_zeros * 2^precision + 1 entries, already multiplied
// by min(1, ratio)) in steps of index_step = int(min(1, ratio) * 2^precision) with linear interpolation between table entries
// (`delta` = forward differences).  float64 accumulation, one rounding to fp32.  Serves librosa.load(path, sr=22050) for files whose rate
// is not a power-of-two multiple of 22.05 kHz (48 kHz, 16 kHz, ...).
// `times` (optional): resampy's time register of every output sample, i.e. the SEQUENTIALLY accumulated sum of 1/ratio in float64 —
// resampy truncates index_step to an integer, so its output is discontinuous where the register crosses an integer and the accumulated
// rounding decides the side; without it the register is t * (1/ratio).
__global__ void resample_table_walk_kernel(const float* __restrict__ x, float* __restrict__ y, const double* __restrict__ win,
                                           const double* __restrict__ delta, const double* __restrict__ times, int nwin, int num_table,
                                           double ratio, long long n_in, long long n_out_real, long long n_out, double gain) {
  const double scale = ratio < 1.0 ? ratio : 1.0;
  const int index_step = (int)(scale * num_table);
  const double time_increment = 1.0 / ratio;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < n_out; t += (long long)gridDim.x * blockDim.x) {
    double acc = 0.0;
    if (t < n_out_real) {
      const double time_register = times ? times[t] : (double)t * time_increment;
      const long long n = (long long)time_register;
      double frac = scale * (time_register - (double)n);
      double index_frac = frac * num_table;
      int offset = (int)index_frac;
      double eta = index_frac - offset;
      long long i_max = (nwin - offset) / index_step;
      if (i_max > n + 1) i_max = n + 1;
      for (long long i = 0; i < i_max; ++i) {
        const int idx = offset + (int)i * index_step;
        acc += (win[idx] + eta * delta[idx]) * (double)x[n - i];
      }
      frac = scale - frac;
      index_frac = frac * num_table;
      offset = (int)index_frac;
      eta = index_frac - offset;
      long long k_max = (nwin - offset) / index_step;
      if (k_max > n_in - n - 1) k_max = n_in - n - 1;
      for (long long k = 0; k < k_max; ++k) {
        const int idx = offset + (int)k * index_step;
        acc += (win[idx] + eta * delta[idx]) * (double)x[n + k + 1];
      }
      acc *= gain;
    }
    y[t] = (float)acc;
  }
}

// on-disk HCQT [F][N][C] float64 (np.save of compute_efficient_hcqt's result) -> network layout [C][lead + N + trail][F] fp32 with zeroed
// pad frames (np.transpose(.., (2,1,0)) + np.pad + .float() of exp126a...py:413-420 in one pass); 32 bins x 32 frames per CTA
__global__ void __launch_bounds__(256) hcqt_npy_to_frames_kernel(const double* __restrict__ in, float* __restrict__ out, int F, int N, int C,
                                                                 int lead, int trail) {
  extern __shared__ float tile[];      // [32 f][32 n][C], +1 float of padding per f row
  const int f0 = blockIdx.x * 32, n0 = blockIdx.y * 32;
  const int row = 32 * C + 1;
  const int nn = min(32, N - n0), nf = min(32, F - f0);
  for (int i = threadIdx.x; i < nf * nn * C; i += blockDim.x) {
    const int fl = i / (nn * C), r = i % (nn * C);
    tile[fl * row + r] = (float)in[((size_t)(f0 + fl) * N + n0) * C + r];
  }
  __syncthreads();
  const int NT = lead + N + trail;
  for (int i = threadIdx.x; i < C * nn * nf; i += blockDim.x) {
    const int fl = i % nf, nl = (i / nf) % nn, c = i / (nf * nn);
    out[((size_t)c * NT + lead + n0 + nl) * F + f0 + fl] = tile[fl * row + nl * C + c];
  }
}

__global__ void zero_pad_frames_kernel(float* __restrict__ out, int F, int N, int C, int lead, int trail) {
  const int NT = lead + N + trail;
  const long long total = (long long)C * (lead + trail) * F;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F);
    const int r = (int)((i / F) % (lead + trail));
    const int c = (int)(i / ((long long)F * (lead + trail)));
    const int n = r < lead ? r : N + r;
    out[((size_t)c * NT + n) * F + f] = 0.f;
  }
}

static inline int ilog2(int n) {
  int l = 0;
  while ((1 << l) < n) ++l;
  return l;
}

}  // namespace mpa

using namespace mpa;

extern "C" {

int mpa_decimate_gain_f32(const float* y_in, float* y_out, const float* half_taps, int n_half, int factor, double gain, long long n_in,
                          void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(y_in && y_out && half_taps && factor >= 2 && (factor & (factor - 1)) == 0 && n_half >= 1 && n_half <= 4096 && n_in >= factor,
              "decimate: bad argument");
  const long long n_real = n_in / factor, n_out = (n_in + factor - 1) / factor;
  long long g = (n_out + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  decimate_kernel<<<(unsigned)g, 256, (size_t)n_half * sizeof(float), (cudaStream_t)stream>>>(y_in, y_out, half_taps, n_half, factor, gain, n_in, n_real, n_out);
  MPA_CHECK_LAUNCH("decimate");
  return MPA_OK;
}

int mpa_decimate_f32(const float* y_in, float* y_out, const float* half_taps, int n_half, int factor, long long n_in, void* stream) {
  return mpa_decimate_gain_f32(y_in, y_out, half_taps, n_half, factor, sqrt((double)factor), n_in, stream);
}

int mpa_decimate2_f32(const float* y_in, float* y_out, const float* half_taps, long long n_in, void* stream) {
  return mpa_decimate_f32(y_in, y_out, half_taps, 32, 2, n_in, stream);
}

int mpa_cqt_level_f32(const float* y_level, long long n_level, int n_fft, int hop, int n_frames, const float* basis, const int* band_start,
                      const float* row_scale, int n_rows, int band, const int* tuning_idx, const int* dest, int n_dest, float* out,
                      int out_frames, int out_bins, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(y_level && basis && band_start && row_scale && dest && out, "cqt_level: null argument");
  MPA_REQUIRE(n_fft >= 64 && n_fft <= 4096 && (n_fft & (n_fft - 1)) == 0, "cqt_level: n_fft must be a power of two in 64..4096");
  MPA_REQUIRE(n_level >= 2, "cqt_level: signal of %lld samples is too short", n_level);
  MPA_REQUIRE(hop >= 1 && n_frames >= 1 && n_frames <= out_frames && n_rows >= 1 && band >= 1 && n_dest >= 1 && out_bins < 65536,
              "cqt_level: bad shape");
  MPA_REQUIRE((long long)(n_frames - 1) * hop <= n_level, "cqt_level: %d frames at hop %d exceed the signal (%lld samples)", n_frames, hop, n_level);
  const size_t smem = (size_t)n_fft * 12;
  cqt_level_kernel<<<n_frames, 256, smem, (cudaStream_t)stream>>>(y_level, n_level, n_fft, ilog2(n_fft), hop, (const float2*)basis, band_start,
                                                                   row_scale, n_rows, band, tuning_idx, dest, n_dest, out, out_frames, out_bins);
  MPA_CHECK_LAUNCH("cqt_level");
  return MPA_OK;
}

int mpa_cqt_levels_f32(const mpa_cqt_level* levels, int n_levels, int n_frames, int band, const int* tuning_idx, float* out, int out_frames,
                       int out_bins, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(levels && out && n_levels >= 1 && n_levels <= kMaxCqtLevels, "cqt_levels: 1..%d levels", kMaxCqtLevels);
  MPA_REQUIRE(n_frames >= 1 && n_frames <= out_frames && band >= 1 && out_bins < 65536, "cqt_levels: bad shape");
  CqtLevelsParams p;
  memset(&p, 0, sizeof(p));
  int max_fft = 0;
  for (int i = 0; i < n_levels; ++i) {
    const mpa_cqt_level& L = levels[i];
    MPA_REQUIRE(L.y && L.basis && L.band_start && L.row_scale && L.dest, "cqt_levels: null argument in level %d", i);
    MPA_REQUIRE(L.n_fft >= 64 && L.n_fft <= 4096 && (L.n_fft & (L.n_fft - 1)) == 0, "cqt_levels: n_fft must be a power of two in 64..4096");
    MPA_REQUIRE(L.n >= 2 && L.hop >= 1 && L.n_rows >= 1 && L.n_dest >= 1, "cqt_levels: bad level %d", i);
    MPA_REQUIRE((long long)(n_frames - 1) * L.hop <= L.n, "cqt_levels: %d frames at hop %d exceed the signal (%lld samples)", n_frames, L.hop, L.n);
    p.lv[i] = L;
    p.log2n[i] = ilog2(L.n_fft);
    if (L.n_fft > max_fft) max_fft = L.n_fft;
  }
  p.n_frames = n_frames; p.band = band; p.out_frames = out_frames; p.out_bins = out_bins;
  p.tuning_idx = tuning_idx; p.out = out;
  cqt_levels_kernel<<<dim3(n_frames, n_levels), 256, (size_t)max_fft * 12, (cudaStream_t)stream>>>(p);
  MPA_CHECK_LAUNCH("cqt_levels");
  return MPA_OK;
}

size_t mpa_cqt_levels_bwd_workspace(const mpa_cqt_level* levels, int n_levels, int n_frames) {
  size_t floats = 0;
  for (int i = 0; levels && i < n_levels; ++i) floats += (size_t)(n_frames < 1 ? 1 : n_frames) * levels[i].n_fft;
  return floats * sizeof(float);
}

int mpa_cqt_levels_bwd_f32(const mpa_cqt_level* levels, const mpa_cqt_level_grad* grads, int n_levels, int n_frames, int band,
                           const int* tuning_idx, const float* g_out, int out_frames, int out_bins, int accumulate, void* workspace,
                           size_t ws_bytes, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(levels && grads && g_out && workspace && n_levels >= 1 && n_levels <= kMaxCqtLevels, "cqt_levels_bwd: 1..%d levels", kMaxCqtLevels);
  MPA_REQUIRE(n_frames >= 1 && n_frames <= out_frames && band >= 1 && out_bins < 65536, "cqt_levels_bwd: bad shape");
  if (ws_bytes < mpa_cqt_levels_bwd_workspace(levels, n_levels, n_frames)) {
    set_error("cqt_levels_bwd: workspace %zu < %zu bytes", ws_bytes, mpa_cqt_levels_bwd_workspace(levels, n_levels, n_frames));
    return MPA_ERR_WORKSPACE;
  }
  CqtLevelsBwdParams p;
  CqtOlaParams q;
  memset(&p, 0, sizeof(p));
  memset(&q, 0, sizeof(q));
  int max_fft = 0, max_rows = 0, n_groups = 0;
  size_t off = 0;
  for (int i = 0; i < n_levels; ++i) {
    const mpa_cqt_level& L = levels[i];
    const mpa_cqt_level_grad& G = grads[i];
    MPA_REQUIRE(L.y && L.basis && L.band_start && L.row_scale && L.dest && G.g_y && G.bin_off && G.bin_rows,
                "cqt_levels_bwd: null argument in level %d", i);
    MPA_REQUIRE(L.n_fft >= 64 && L.n_fft <= 4096 && (L.n_fft & (L.n_fft - 1)) == 0, "cqt_levels_bwd: n_fft must be a power of two in 64..4096");
    MPA_REQUIRE(L.n >= 2 && L.hop >= 1 && L.n_rows >= 1 && L.n_rows <= 2048 && L.n_dest >= 1, "cqt_levels_bwd: bad level %d", i);
    MPA_REQUIRE((long long)(n_frames - 1) * L.hop <= L.n, "cqt_levels_bwd: %d frames at hop %d exceed the signal (%lld samples)", n_frames, L.hop,
                L.n);
    p.lv[i] = L;
    p.gr[i] = G;
    p.log2n[i] = ilog2(L.n_fft);
    p.ws_off[i] = q.ws_off[i] = off;
    off += (size_t)n_frames * L.n_fft;
    q.n_fft[i] = L.n_fft;
    q.hop[i] = L.hop;
    if (L.n_fft > max_fft) max_fft = L.n_fft;
    if (L.n_rows > max_rows) max_rows = L.n_rows;
  }
  // group the levels by the signal gradient they write (first-occurrence order), so that one thread owns each signal sample
  for (int i = 0, k = 0; i < n_levels; ++i) {
    bool seen = false;
    for (int j = 0; j < i; ++j) seen |= grads[j].g_y == grads[i].g_y;
    if (seen) continue;
    q.grp_first[n_groups] = k;
    q.g_y[n_groups] = grads[i].g_y;
    q.n[n_groups] = levels[i].n;
    for (int j = i; j < n_levels; ++j) {
      if (grads[j].g_y != grads[i].g_y) continue;
      MPA_REQUIRE(levels[j].n == levels[i].n, "cqt_levels_bwd: levels %d and %d share a gradient buffer but not a length", i, j);
      q.order[k++] = j;
    }
    q.grp_first[++n_groups] = k;
  }
  p.n_frames = n_frames; p.band = band; p.out_frames = out_frames; p.out_bins = out_bins;
  p.tuning_idx = tuning_idx; p.g_out = g_out; p.ws = (float*)workspace;
  q.n_frames = n_frames; q.accumulate = accumulate ? 1 : 0; q.ws = (const float*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t smem = (size_t)max_fft * 12 + (size_t)max_rows * 8;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(cqt_levels_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      set_error("cqt_levels_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return MPA_ERR_CUDA;
    }
  }
  cqt_levels_bwd_kernel<<<dim3(n_frames, n_levels), 256, smem, st>>>(p);
  MPA_CHECK_LAUNCH("cqt_levels_bwd");
  long long n_max = 0;
  for (int g = 0; g < n_groups; ++g) n_max = q.n[g] > n_max ? q.n[g] : n_max;
  long long gx = (n_max + 255) / 256;
  if (gx > 148 * 8) gx = 148 * 8;
  cqt_ola_bwd_kernel<<<dim3((unsigned)gx, n_groups), 256, 0, st>>>(q);
  MPA_CHECK_LAUNCH("cqt_ola_bwd");
  return MPA_OK;
}

int mpa_decimate_adjoint_f32(const float* g_out, float* g_in, const float* half_taps, int n_half, int factor, double gain, long long n_in,
                             int accumulate, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(g_out && g_in && half_taps && factor >= 2 && (factor & (factor - 1)) == 0 && n_half >= 1 && n_half <= 4096 && n_in >= factor,
              "decimate_adjoint: bad argument");
  long long g = (n_in + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  decimate_adjoint_kernel<<<(unsigned)g, 256, (size_t)n_half * sizeof(float), (cudaStream_t)stream>>>(g_out, g_in, half_taps, n_half, factor, gain,
                                                                                                        n_in, n_in / factor, accumulate);
  MPA_CHECK_LAUNCH("decimate_adjoint");
  return MPA_OK;
}

int mpa_resample_f32(const float* y_in, float* y_out, const double* interp_win, const double* interp_delta, const double* time_register,
                     int n_win, int num_table, double ratio, double gain, long long n_in, long long n_out, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(y_in && y_out && interp_win && interp_delta && n_win > 1 && num_table > 0 && ratio > 0.0 && n_in > 0 && n_out > 0,
              "resample: bad argument");
  const double scale = ratio < 1.0 ? ratio : 1.0;
  MPA_REQUIRE((int)(scale * num_table) >= 1, "resample: ratio %g too small for a table of %d steps per zero crossing", ratio, num_table);
  long long n_real = (long long)((double)n_in * ratio);       // resampy's output length; librosa pads / trims to n_out
  if (n_real > n_out) n_real = n_out;
  long long g = (n_out + 127) / 128;
  if (g > 148 * 32) g = 148 * 32;
  resample_table_walk_kernel<<<(unsigned)g, 128, 0, (cudaStream_t)stream>>>(y_in, y_out, interp_win, interp_delta, time_register, n_win, num_table, ratio,
                                                                             n_in, n_real, n_out, gain);
  MPA_CHECK_LAUNCH("resample");
  return MPA_OK;
}

int mpa_hcqt_npy_to_frames_f64(const double* hcqt_fnc, float* out, int F, int N, int C, int lead, int trail, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(hcqt_fnc && out && F > 0 && N > 0 && C > 0 && C <= 32 && lead >= 0 && trail >= 0, "hcqt_npy_to_frames: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(ceil_div(F, 32), ceil_div(N, 32));
  hcqt_npy_to_frames_kernel<<<grid, 256, (size_t)(32 * (32 * C + 1)) * sizeof(float), st>>>(hcqt_fnc, out, F, N, C, lead, trail);
  MPA_CHECK_LAUNCH("hcqt_npy_to_frames");
  if (lead + trail > 0) {
    zero_pad_frames_kernel<<<ceil_div((long long)C * (lead + trail) * F, 256), 256, 0, st>>>(out, F, N, C, lead, trail);
    MPA_CHECK_LAUNCH("zero_pad_frames");
  }
  return MPA_OK;
}

size_t mpa_tuning_workspace(int n_frames) { return 256 + (size_t)(n_frames < 1 ? 1 : n_frames) * 180 * 2 * sizeof(float); }

int mpa_estimate_tuning_f32(const float* y, long long n, const float* hann2048, float sr, int bins_per_octave, int* tuning_idx, void* workspace,
                            size_t ws_bytes, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(y && hann2048 && tuning_idx && workspace && n > 1024, "estimate_tuning: bad argument (need > 1024 samples)");
  const int n_frames = (int)(n / 512) + 1;
  if (ws_bytes < mpa_tuning_workspace(n_frames)) {
    set_error("estimate_tuning: workspace %zu < %zu bytes", ws_bytes, mpa_tuning_workspace(n_frames));
    return MPA_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int max_peaks = n_frames * 180;
  int* counter = (int*)workspace;
  float* pitch = (float*)((char*)workspace + 256);
  float* mag = pitch + max_peaks;
  cudaMemsetAsync(counter, 0, sizeof(int), st);
  tuning_peaks_kernel<<<n_frames, 256, 0, st>>>(y, n, hann2048, sr, counter, pitch, mag, max_peaks);
  MPA_CHECK_LAUNCH("tuning_peaks");
  tuning_finalize_kernel<<<1, 1024, 0, st>>>(counter, pitch, mag, max_peaks, bins_per_octave, tuning_idx);
  MPA_CHECK_LAUNCH("tuning_finalize");
  return MPA_OK;
}

}  // extern "C"
