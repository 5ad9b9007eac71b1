/*
 * mpa.h — C ABI of libmpa.so, the B200 (sm_100a) replacement for the HCQT + patch-wise network hot path of
 * christofw/multipitch_architectures.
 *
 * The reference has no FFI of its own: its boundary is the Python API surface (SURVEY.md §8b).  The Python
 * host layer in multipitch_architectures_b200/libdl mirrors that surface and reaches the GPU only through
 * the entry points below (ctypes; see INTEGRATION.md for the binding a reference maintainer would add).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch tensors); the library never allocates
 *     or frees caller-visible memory and never synchronises the device or the stream;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it;
 *   - return value 0 = success, negative = error; mpa_last_error() returns a thread-local message;
 *   - no CPU fallback exists: on a non-sm_100 device every call returns MPA_ERR_ARCH.
 *   - layouts: "NCHW" = [B][C][T][F] fp32 contiguous (T = time frames, F = frequency bins), exactly the
 *     tensors the reference modules exchange (libdl/nn_models/basic_cnns.py:410-423).
 *     "CP8"  = bf16 channel-chunk planes [B][ceil(C/8)][TP][FP][8] with zero borders, TP = T + 2*PT,
 *     FP = row pitch (multiple of 16, >= F + PF); real pixel (t,f) sits at row PT+t, column PF+f.
 */
#ifndef MPA_H_
#define MPA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MPA_OK 0
#define MPA_ERR_ARG (-1)
#define MPA_ERR_ARCH (-2)
#define MPA_ERR_CUDA (-3)
#define MPA_ERR_WORKSPACE (-4)

/* activation codes for the fused epilogues */
#define MPA_ACT_NONE 0
#define MPA_ACT_LRELU 1   /* slope in `act_param` */
#define MPA_ACT_RELU 2
#define MPA_ACT_SIGMOID 3

/* 16-bit storage / tensor-core operand formats of the CP8 planes (fp32 accumulation in both cases) */
#define MPA_FMT_F16 0     /* IEEE half: 11-bit significand, the default (same operand precision as TF32) */
#define MPA_FMT_BF16 1    /* bfloat16: 8-bit significand */
#define MPA_FMT_F16X3 2   /* split precision: every value is a pair of fp16 planes (hi = fp16(x), lo = fp16(x - hi), ~22-bit significand);
                             a convolution is three tensor-core passes (W_hi x_hi + W_lo x_hi + W_hi x_lo) into one fp32 accumulator.
                             A buffer with `ncs` chunk planes per item holds its hi planes in chunks [0, ncs/2) and its lo planes in
                             [ncs/2, ncs); every CP8 entry point accepts this format with the same arguments (ncs even).  This is the
                             tensor-core mode that meets the reference's fp32 results to ~1e-5 (the north star's 1e-3 with margin). */

int mpa_version(void);
const char* mpa_last_error(void);
/* 0 when the current device is compute capability 10.x, MPA_ERR_ARCH otherwise. */
int mpa_device_check(void);
/* Number of kernels this library has launched since load (all streams); bench.py's `gpu_launches`. */
long long mpa_launch_count(void);

/* ---- N1: LayerNorm([C,F]) per (b,t) row with optional fused log compression ---------------------------
 * replaces nn.LayerNorm on the transposed view (basic_cnns.py:371,411) and, when gamma_log > 0, the dataset's
 * log(1 + gamma_log * x) (hcqt_datasets.py:105-106).  x,out NCHW [B,C,T,F]; ln_w, ln_b [C,F]. */
int mpa_layernorm_cf_f32(const float* x, const float* ln_w, const float* ln_b, float* out,
                         int B, int C, int T, int F, float eps, float gamma_log, void* stream);

/* The same LayerNorm written straight into 16-bit CP8 planes (one chunk, C <= 8; geometry as mpa_nchw_to_cp8) — the input of the first
 * tensor-core convolution of a training step, without the fp32 NCHW copy and its converter pass — and the matching parameter gradient
 * that reads the gradient wrt the LayerNorm output from the CP8 planes the first convolution's data gradient wrote
 * (nn.LayerNorm([C,F]).weight.grad / .bias.grad of basic_cnns.py:371 / unet_cnns.py:355 after loss.backward()). */
int mpa_layernorm_cf_cp8(const float* x, const float* ln_w, const float* ln_b, void* out_cp8, int B, int C, int T, int F, int pitch, int pf,
                         int pt, float eps, float gamma_log, int fmt, void* stream);
int mpa_layernorm_cf_param_grad_cp8(const float* x, const void* g_cp8, float* g_w, float* g_b, int B, int C, int T, int F, int pitch, int pf,
                                    int pt, int fmt, float eps, float gamma_log, void* stream);
/* Pixel-per-thread forms of the two calls above (F <= 256): the forward also leaves (mean, rstd) of every (b,t) row in stats [B*T][2]
 * (may be NULL), and the parameter gradient reads them instead of re-reducing every row (same reference lines). */
int mpa_layernorm_cf_cp8_stats(const float* x, const float* ln_w, const float* ln_b, void* out_cp8, float* stats, int B, int C, int T, int F,
                               int pitch, int pf, int pt, float eps, float gamma_log, int fmt, void* stream);
int mpa_layernorm_cf_param_grad_cp8_stats(const float* x, const void* g_cp8, const float* stats, float* g_w, float* g_b, int B, int C, int T,
                                          int F, int pitch, int pf, int pt, int fmt, float gamma_log, void* stream);
/* LayerNorm([C,F]) backward to the INPUT with the parameter gradients of the same pass (saliency maps, adversarial checks, eval-mode
 * backward): per (b,t) row dx = rstd * (gh - mean(gh) - xhat * mean(gh * xhat)), gh = g * ln_w, means over the C*F elements (times
 * gamma_log / (1 + gamma_log * x) when the log compression is fused); g_w / g_b overwritten as by the parameter-only calls above, dx fp32
 * NCHW [B,C,T,F] overwritten.  One thread per bin with all C <= 8 channels, F <= 256.
 *   _cp8_stats  g in the CP8 planes (one chunk) and (mean, rstd) from the rows mpa_layernorm_cf_cp8_stats saved
 *   _f32        g fp32 NCHW; the row statistics are re-reduced from x (the fp32 tape, or planes converted to NCHW) */
int mpa_layernorm_cf_input_grad_cp8_stats(const float* x, const void* g_cp8, const float* stats, const float* ln_w, float* dx, float* g_w,
                                          float* g_b, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, float gamma_log,
                                          void* stream);
int mpa_layernorm_cf_input_grad_f32(const float* x, const float* g_out, const float* ln_w, float* dx, float* g_w, float* g_b, int B, int C,
                                    int T, int F, float eps, float gamma_log, void* stream);

/* Frame-major variant used by the streaming inference engine: frames [C][N][F] (the HCQT layout) ->
 * normalised frames; rows s with s < lead or s >= lead+N are the patch zero padding and come out as ln_b
 * (LayerNorm of an all-zero row).  out_f32 [C][lead+N+trail][F] and/or out_cp8 CP8 plane (1 chunk). */
int mpa_layernorm_frames(const float* frames, const float* ln_w, const float* ln_b, float* out_f32,
                         void* out_cp8, int C, int N, int F, int lead, int trail, int cp8_pitch, int cp8_pf,
                         float eps, float gamma_log, int fmt, void* stream);

/* H4/H5: dataset_context patch extraction (hcqt_datasets.py:63-75,105-106): out[b] = log(1+gamma*in[:, (i0+b)*stride : +T, :]),
 * in [C][NT][F] (already zero-padded by the caller as exp126a:420 does), out [n][C][T][F]; gamma_log <= 0 -> no compression. */
int mpa_gather_patches_f32(const float* in, float* out, int C, int NT, int F, int i0, int n, int T, int stride,
                           float gamma_log, void* stream);
/* Its adjoint: g_in[c][r][f] = sum over the patches p covering frame r of g_out[p][c][r - (i0+p)*stride][f], times gamma_log / (1 +
 * gamma_log * in[c][r][f]) (1 when gamma_log <= 0; `in` is the forward input and may then be NULL).  g_in [C][NT][F] overwritten (rows no
 * patch covers are 0); one thread per element, deterministic. */
int mpa_gather_patches_bwd_f32(const float* g_out, const float* in, float* g_in, int C, int NT, int F, int i0, int n, int T, int stride,
                               float gamma_log, void* stream);

/* Training-time augmentation fused with the patch cut (hcqt_datasets.py:67-141; SURVEY.md 8f row 1): for each of n patches starting at
 * frame start[b] of in [C][NT][F]:  random EQ  w_c(f) = 1 - 2e-6*eq_alpha[b]*(f - (eq_beta[b] - eq_offset[c]))^2  (:80-97; eq_alpha NULL or 0 = off)
 * -> x = |x + noise_std*N(0,1)| (:99-102) -> log(1 + gamma_log*x) (:105-106) -> tuning shift by tune2[b]/2 bins, tune2 in -2..2 (:108-123)
 * -> transposition by transp[b] semitones of bins_per_semitone bins (:125-139); bins vacated by the two shifts hold |N(0, fill_std)|.
 * The integer decisions are drawn by the caller (host mirror, incl. the reference's rejection loop); Gaussian values are Philox-4x32-10
 * under (seed, offset).  out [n][C][T][F] fp32.  All index arrays are device pointers. */
int mpa_augment_patches_f32(const float* in, const long long* start, float* out, int C, int NT, int F, int n, int T, const int* eq_alpha,
                            const int* eq_beta, const int* eq_offset, float noise_std, float gamma_log, const int* tune2,
                            const int* transp, int bins_per_semitone, float fill_std, unsigned long long seed,
                            unsigned long long offset, void* stream);
/* Targets of those patches: y[b][q] = targets[frame[b]][q - transp[b]], wrapped entries zeroed (P = 12 pitch classes: plain roll)
 * (hcqt_datasets.py:75,127-137).  targets [N][P] fp32, frame [n] centre frames, y [n][P]. */
int mpa_augment_targets_f32(const float* targets, const long long* frame, const int* transp, float* y, int n, int P, void* stream);

/* ---- full-height VALID convolution = the head's 75x1 "time reduction" conv3 (basic_cnns.py:396-401) as GEMMs -----------------------
 * H == KH, KW == 1, one output row: Y[co][(b,w)] = sum_(ci,h) w[co][ci][h] * x[b][ci][h][w].  x [B][Cin][H][W], w [Cout][Cin][H][1]
 * (state_dict layout), out / g_out [B][Cout][1][W].  Forward fuses bias + activation (K is split across CTAs; the slices are kept apart in the workspace and added in order:
 * deterministic); the gradients overwrite their outputs (split-K, fp32 atomics). */
size_t mpa_conv_rows_fwd_workspace(int B, int Cin, int H, int W, int Cout);   /* split-K partial sums of the forward (may be 0) */
int mpa_conv_rows_fwd_f32(const float* x, const float* w, const float* bias, float* out, int B, int Cin, int H, int W, int Cout, int act,
                          float act_param, void* workspace, size_t ws_bytes, void* stream);
int mpa_conv_rows_dgrad_f32(const float* g_out, const float* w, float* g_in, int B, int Cin, int H, int W, int Cout, void* stream);
int mpa_conv_rows_wgrad_f32(const float* x, const float* g_out, float* g_w, int B, int Cin, int H, int W, int Cout, void* stream);

/* ---- BLUnet bottleneck: bidirectional LSTM over the time axis (unet_cnns.py:220-243, 1000-1101; SURVEY.md 8f row 2) -------------------
 * One nn.LSTM layer, batch_first: x [B][T][I] -> out [B][T][D*H] (forward direction in [0,H), reverse in [H,2H)), zero initial state.
 * w_ih [D][4H][I], w_hh [D][4H][H], b_ih, b_hh [D][4H] = weight_ih_l{k}(_reverse) ... stacked per direction; gate order i, f, g, o.
 * workspace >= mpa_lstm_layer_workspace() bytes. */
size_t mpa_lstm_layer_workspace(int B, int T, int H, int D);
int mpa_lstm_layer_f32(const float* x, const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, float* out, int B,
                       int T, int I, int H, int D, void* workspace, size_t ws_bytes, void* stream);
/* Training: the forward keeps the activated gates [D][B*T][4H] and all cell states [D][B][T][H]; the backward consumes them (gates holds
 * the pre-activation gradients afterwards) and overwrites g_x [B][T][I] (may be NULL), g_w_ih [D][4H][I], g_w_hh [D][4H][H] and
 * g_b [D][4H] (the gradient of bias_ih and of bias_hh).  Forward workspace >= D*B*H floats; backward >= mpa_lstm_layer_bwd_workspace(). */
int mpa_lstm_layer_train_f32(const float* x, const float* w_ih, const float* w_hh, const float* b_ih, const float* b_hh, float* out,
                             float* gates, float* c_all, int B, int T, int I, int H, int D, void* workspace, size_t ws_bytes,
                             void* stream);
size_t mpa_lstm_layer_bwd_workspace(int B, int T, int H, int D);
int mpa_lstm_layer_bwd_f32(const float* x, const float* w_ih, const float* w_hh, float* gates, const float* c_all, const float* out,
                           const float* g_out, float* g_x, float* g_w_ih, float* g_w_hh, float* g_b, int B, int T, int I, int H, int D,
                           void* workspace, size_t ws_bytes, void* stream);
/* blstm_temporal_enc_layer's layout changes: x NCHW [B,C,T,F] <-> seq [B][T][C*F] (feature = c*F + f). */
int mpa_lstm_seq_from_nchw_f32(const float* x, float* seq, int B, int C, int T, int F, void* stream);
int mpa_lstm_seq_to_nchw_f32(const float* seq, float* x, int B, int C, int T, int F, void* stream);

/* ---- evaluation measures (eval_metrics.py:8-110,158-189; SURVEY.md 8f row 4) --------------------------------------------------------
 * targ, pred [n_frames][n_bins] fp32 (device).  sums16 (device, 16 doubles) = sums over frames of the per-frame terms, float64 arithmetic:
 *  0 TP  1 #est (pred >= threshold)  2 #(targ > 0)  3 cosine of the L2-normalised frames (libfmp unit-vector fallback below 1e-10)
 *  4 sum_bins t*log2(p+eps)+(1-t)*log2(1-p+eps)  5 |t-p|_2  6 #((pred>=threshold) == targ)  7 sum_bins t*p+(1-t)*(1-p)
 *  8 sum(t*p)/(sum(t)+eps)  9 matched pitch classes (bin q is pitch min_pitch+q)  10 min(n_ref,n_est)  11 max(n_ref,n_est)
 *  12 max(0,n_ref-n_est)  13 max(0,n_est-n_ref)  14 n_ref = #(targ != 0)  15 zero.
 * workspace >= mpa_eval_workspace(n_frames) bytes; frames are added in a fixed order (bit-reproducible). */
size_t mpa_eval_workspace(int n_frames);
int mpa_eval_sums_f32(const float* targ, const float* pred, int n_frames, int n_bins, double threshold, int min_pitch, double* sums16,
                      void* workspace, size_t ws_bytes, void* stream);

/* ---- generic direct convolution, fp32 CUDA cores (all kernel sizes / strides of the model zoo) ---------
 * replaces nn.Conv2d (+ eval BatchNorm2d folded as per-channel scale/shift) + activation.
 * x NCHW [B,Cin,H,W]; if x2 != NULL the input is the channel concat [x (Cin1) | x2 (Cin-Cin1)] (U-Net skip).
 * w_packed [Cin][KH*KW][CoutPad] fp32 with CoutPad = ceil(Cout/16)*16; bias/scale/shift [Cout] or NULL.
 * out[b,co,ho,wo] = act( (conv + bias) * scale + shift ),  Ho = (H+2ph-KH)/sh+1, Wo likewise. */
int mpa_conv2d_f32(const float* x, const float* x2, int Cin1, const float* w_packed, const float* bias,
                   const float* scale, const float* shift, float* out, int B, int Cin, int H, int W,
                   int Cout, int KH, int KW, int sh, int sw, int ph, int pw, int act, float act_param,
                   void* stream);

/* time max-pool (k,1) stride 1 pad k/2 (-inf padding) with optional residual: out = pool(x) + res. */
int mpa_maxpool_time_f32(const float* x, const float* res, float* out, int B, int C, int T, int F, int k,
                         void* stream);
/* MaxPool2d((kh,kw), stride (sh,sw)), no padding, floor mode (unet_cnns.py:349-361, :2314). */
int mpa_maxpool2d_f32(const float* x, float* out, int B, int C, int H, int W, int kh, int kw, int sh, int sw,
                      void* stream);
/* unet_up_concat_padding (unet_cnns.py:85-104): out[B,Cs+Cl,Hs,Ws] = cat(skip, pad(bilinear_x2_ac(low))). */
int mpa_upsample2x_concat_f32(const float* low, const float* skip, float* out, int B, int Cl, int Hl, int Wl,
                              int Cs, int Hs, int Ws, void* stream);
/* train-mode BatchNorm2d statistics: mean/var (biased) per channel over (B,H,W) -> stats[2*C]. */
int mpa_bn_stats_f32(const float* x, float* stats, int B, int C, int HW, void* stream);
/* y = act((x - mean) * rsqrt(var+eps) * w + b) per channel, in place allowed. */
int mpa_bn_apply_f32(const float* x, const float* stats, const float* w, const float* b, float* out, int B,
                     int C, int HW, float eps, int act, float act_param, void* stream);

/* ---- N8: transformer_enc_layer (unet_cnns.py:107-159), attention over the BATCH axis -------------------
 * x, out NCHW [B,E,Th,Fw]; S = Th*Fw tokens per item.  Host-side folding (one-off, see nn_models/unet_cnns.py):
 *   w_qkv [3E,E] = in_proj_weight blocks times {q,k,v}_linear.weight, b_qkv = in_proj_bias,
 *   w_proj [E,E] = o_linear.weight @ out_proj.weight, b_proj = o_linear.weight @ out_proj.bias.
 * pe [S,E] sinusoidal table or NULL.  workspace >= mpa_encoder_layer_workspace() bytes. */
size_t mpa_encoder_layer_workspace(int B, int E, int S, int mlp_dim);
int mpa_encoder_layer_f32(const float* x, float* out, int B, int E, int Th, int Fw, int num_heads, int mlp_dim,
                          const float* pe, const float* w_qkv, const float* b_qkv, const float* w_proj,
                          const float* b_proj, const float* ln1_w, const float* ln1_b, const float* mlp0_w,
                          const float* mlp0_b, const float* mlp2_w, const float* mlp2_b, const float* ln2_w,
                          const float* ln2_b, float eps, void* workspace, size_t ws_bytes, void* stream);

/* Fused attention half of the encoder layer (unet_cnns.py:131-153), eval mode, ONE launch on the tensor cores: token gather (+ pe [S,E]
 * or NULL) -> folded q/k/v in-projection (tcgen05) -> batch-axis softmax attention (fp32) -> folded out-projection (tcgen05) -> + residual
 * -> LayerNorm1.  w_qkv_chunks / w_proj_chunks: the folded [3E,E] / [E,E] matrices of mpa_encoder_layer_f32 in the chunk layout of
 * mpa_gemm_tc_to_chunks (row tile 128).  h1 [B*S, E] fp32 tokens; h1_chunks (optional): the same tokens as the 16-bit X operand of
 * mpa_gemm_tc_f16 (row tile 256).  Needs B <= 64, E a multiple of 16 with 64 <= E <= 128; other shapes use the separate stages. */
int mpa_enc_attn_block_tc(const float* x, const float* pe, const void* w_qkv_chunks, const float* b_qkv, const void* w_proj_chunks,
                          const float* b_proj, const float* ln_w, const float* ln_b, float* h1, void* h1_chunks, int B, int E, int S,
                          int num_heads, float eps, int fmt, void* stream);

/* ---- tcgen05 implicit-GEMM convolution (the hot op: 96 % of DRCNN FLOPs) ------------------------------
 * KHxKW "same" convolution, stride 1, on CP8 bf16 planes.  Weights pre-packed by mpa_conv_tc_pack_weights
 * (host side, one-off).  out = act(conv + bias) in CP8 (pool / residual are applied by mpa_pool3_res_cp8).
 * in_patch_stride_rows: 0 for materialised patches [n][NC][T+2pt][pitch][8];
 * 1 for the streaming engine where patch i is rows [i, i+T) of one shared frame-major plane. */
size_t mpa_conv_tc_packed_bytes(int Cin, int Cout, int KH, int KW, int J);
/* the same for any fmt (MPA_FMT_F16X3: three tile passes + per-output-channel inverse scales) */
size_t mpa_conv_tc_packed_bytes_fmt(int Cin, int Cout, int KH, int KW, int J, int fmt);
/* HOST function: w [Cout][Cin][KH][KW] fp32 (host) -> packed 16-bit A-operand tiles (host buffer), fmt = MPA_FMT_*. */
int mpa_conv_tc_pack_weights(const float* w_host, void* packed_host, int Cin, int Cout, int KH, int KW, int fmt, int J);
/* out_mode 0: `out` is a CP8 plane set [n_patches][ceil(Cout/8)][T+2pt][pitch][8] (16-bit, same fmt);
 * out_mode 1: `out` is the compact plane set [n_patches][ceil(Cout/8)][T][F_out][8] holding only the columns
 *             f = sub_offset + k*sub_stride (a stride-(1,s) convolution evaluated as the stride-1 "same" convolution and
 *             sub-sampled in the epilogue), F_out = ceil((F - sub_offset)/sub_stride);
 * out_mode 2: phase-split planes for a following stride-(1,s) convolution (s = sub_stride, sub_offset = 0, Cout % 8 == 0):
 *             `out` is [n_patches][s][out_nc_stride/s][T+2pt][P2][8], column f of the result lands in phase set f % s at column
 *             8 + f/s, P2 = ceil((8 + F_out)/16)*16.  The strided KHxs convolution then is a stride-1 KHx1 convolution over s*Cin
 *             channels of width F_out: s times fewer MMA columns than the sub-sampled stride-1 form. */
int mpa_conv_tc_f16(const void* in_cp8, const void* w_packed, const float* bias, void* out, int out_mode,
                    int sub_stride, int sub_offset, int n_patches, int Cin, int Cout, int T, int F, int KH, int KW,
                    int pitch, int pf, int pt, long long in_patch_stride_rows, int in_nc_stride, int out_nc_stride,
                    int J, int row0, int n_rows, int act, float act_param, int fmt, void* stream);
/* Fused variant for the CNN / DCNN / DRCNN blocks (basic_cnns.py:373-378, 412-419): z = MaxPool((3,1), s1, p(1,0))(act(conv + bias))
 * [+ the layer input, residual] in ONE kernel, with "virtual" patch rows on both sides so that rows whose receptive field has
 * not reached the zero padding at the patch edges are computed ONCE PER FRAME instead of once per patch:
 *   row r of patch b = rows [0,e) and [T-e,T): per-patch edge planes [patch][chunk][2e rows][pitch][8] (row r at index r, resp. r-(T-2e));
 *                      every other row: the shared stream [chunk][rows][pitch][8] at row b*stream_patch_rows + r.
 * e == T means a fully materialised patch (index r), e == 0 a pure stream.  All pointers address (row 0, column 0) of patch 0, chunk 0;
 * the caller provides at least one readable row before and after every plane and zeroed gap columns, as for mpa_conv_tc_f16.
 * z rows [z_lo[s], z_hi[s]) of every patch are produced for each of the n_seg (1 or 2) segments; the conv rows one above / below
 * each segment are evaluated on the fly (the pool's halo).  workspace >= mpa_conv_tc_pool_workspace() bytes (L2-resident scratch). */
typedef struct mpa_conv_tc_desc {
  const void* in_edge;
  const void* in_stream;
  long long in_edge_patch_stride, in_edge_chunk_stride, in_stream_chunk_stride; /* bytes */
  long long in_stream_patch_rows;
  int in_e;
  const void* w_packed;
  const float* bias;
  void* out_edge;
  void* out_stream;
  long long out_edge_patch_stride, out_edge_chunk_stride, out_stream_chunk_stride; /* bytes */
  long long out_stream_patch_rows;
  int out_e;
  int n_patches, Cin, Cout, T, F, KH, KW, pitch, pf, J;
  int n_seg;
  int z_lo[2], z_hi[2];
  int residual, act;
  float act_param;
  int fmt;
  int weights_layout; /* 0: tiles of mpa_conv_tc_pack_weights; 1: ring pieces of mpa_conv_tc_ring_pack_weights (3x less L2->SM traffic at J = 3) */
  void* workspace;
  size_t ws_bytes;
  int out_split;      /* 0, or s >= 2 (needs out_e == T, n_seg == 1): z is written phase-split for a following stride-(1,s) convolution,
                         out_edge = [patch][s][Cout/8][T+2][P2][8] with column f at phase f % s, column 8 + f/s, P2 = ceil((8 + ceil(F/s))/16)*16;
                         out_edge_chunk_stride / out_edge_patch_stride describe THAT buffer (see mpa_conv_tc_f16 out_mode 2) */
} mpa_conv_tc_desc;
size_t mpa_conv_tc_pool_workspace(int Cout, int pitch, int J);
size_t mpa_conv_tc_pool_workspace_fmt(int Cout, int pitch, int J, int fmt);
/* DEVICE-side packing (training: the weights change every step): w_dev fp32 in state_dict layout.  Packs output channels
 * [co0, co0+Cout) of a convolution with Cout_total output channels (channels >= Cout_total are packed as zeros, so a block may be
 * padded to a multiple of 8).  transpose_flip = 1 packs the data-gradient convolution
 * w'[co'][ci'][kh][kw] = w[ci'][co'][KH-1-kh][KW-1-kw] of a forward weight w [Cin][Cout_total][KH][KW] (Cin = forward Cout). */
int mpa_conv_tc_pack_weights_dev(const float* w_dev, void* packed_dev, int Cin, int Cout, int KH, int KW, int fmt, int J,
                                 int transpose_flip, int Cout_total, int co0, void* stream);
/* All packed operands of a training step in one launch: a table of mpa_conv_tc_pack_weights_dev jobs (same argument meaning) is turned
 * into its device form on the host (mpa_conv_tc_pack_table_build writes mpa_conv_tc_pack_table_bytes(n) bytes into table_host and returns the
 * number of thread blocks of the flattened grid, negative on error; the caller copies the table to the device once), then mpa_conv_tc_pack_weights_multi re-packs every job from the current weights — the per-step
 * refresh of the A operands after the optimiser update (replaces 2 launches per nn.Conv2d and step). */
typedef struct mpa_pack_job {
  const float* w;
  void* packed;
  int Cin, Cout, KH, KW, fmt, J, transpose_flip, Cout_total, co0;
  int split, C0;          /* 0, 0 or the phase-split form (mpa_conv_tc_pack_weights_split_dev) */
} mpa_pack_job;
/* Phase-split form of a KH x s convolution with stride (1, s) (the head's conv2, s = 3; real weights w[Cout][C0][KH][s]): packed as the
 * stride-1 KH x 1 convolution over s * C0p logical input channels (channel ph * C0p + c = tap ph of real channel c; KW = 1, Cin = s * C0p),
 * whose input are phase-split planes (mpa_conv_tc_f16 out_mode 2).  transpose_flip: its data gradient, Cout_total = s * C0p logical output
 * channels (the gradient comes out phase-split), Cin = the real (padded) output channels.  Otherwise as mpa_conv_tc_pack_weights_dev. */
int mpa_conv_tc_pack_weights_split_dev(const float* w_dev, void* packed_dev, int Cin, int Cout, int KH, int KW, int fmt, int J,
                                       int transpose_flip, int Cout_total, int co0, int split, int C0, void* stream);
size_t mpa_conv_tc_pack_table_bytes(int n_jobs);
int mpa_conv_tc_pack_table_build(const mpa_pack_job* jobs, int n_jobs, void* table_host);
int mpa_conv_tc_pack_weights_multi(const void* table_dev, int n_jobs, int n_blocks, void* stream);
/* MPA_FMT_F16X3 jobs (split == 0; the same x3 layout as mpa_conv_tc_pack_weights, with the transposed / flipped weights for transpose_flip)
 * need their per-channel scales first: this launch writes them for every x3 job of the table and must precede mpa_conv_tc_pack_weights_multi
 * (a table without x3 jobs does not need it).  mpa_conv_tc_pack_weights_dev / _split_dev with MPA_FMT_F16X3 issue both launches. */
int mpa_conv_tc_pack_scales_multi(const void* table_dev, int n_jobs, void* stream);
/* HOST functions: un-duplicated weight pieces for weights_layout 1 (one filter row per piece; Cout a multiple of 8). */
size_t mpa_conv_tc_ring_packed_bytes(int Cin, int Cout, int KH, int KW, int J);
int mpa_conv_tc_ring_pack_weights(const float* w_host, void* packed_host, int Cin, int Cout, int KH, int KW, int fmt, int J);
int mpa_conv_tc_pool_f16(const mpa_conv_tc_desc* desc, void* stream);
/* J: output rows per work unit (0 = floor(128/Cout)); must match the J the weights were packed with.
 * row0 / n_rows: compute output rows [row0, row0+n_rows) only (n_rows 0 = to the end) and store them as rows 0.. of `out`;
 * a VALID (KH x 1) convolution such as conv3 (75 x 1, basic_cnns.py:398) is the "same" convolution restricted to
 * row0 = KH/2, n_rows = T-KH+1.  With KW == 1 the row pitch need not be a multiple of 16 and pt may be 0 (compact planes),
 * but the caller must leave >= 512 B of slack after the last input row. */
/* Chunk-strided views: every CP8 entry point takes the number of channel chunks per item of the UNDERLYING buffer
 * (`*_nc_stride` / `ncs_*`, 0 = the tensor's own chunk count) and a pointer already advanced to the view's first chunk.
 * This is how U-Net skip connections are concatenated without a copy: the producer of the skip writes chunks [0, Cs/8) and
 * the up-sampler writes chunks [Cs/8, (Cs+Cl)/8) of one buffer (unet_cnns.py:96-104). */
/* out = maxpool_time_k(y) + res (res may be NULL; k odd, -inf padding), CP8 in/out; with pitch=F, pf=pt=0 it serves
 * the compact out_mode-1 planes too. */
int mpa_pool_time_res_cp8(const void* y_cp8, const void* res_cp8, void* out_cp8, int n_patches, int C, int T, int F,
                          int pitch, int pf, int pt, int k, int fmt, int ncs_y, int ncs_res, int ncs_out, void* stream);
/* nn.MaxPool2d((2,2)) (floor) between two CP8 geometries (unet_cnns.py:349-361). */
int mpa_maxpool2x2_cp8(const void* in_cp8, void* out_cp8, int n, int C, int T, int F, int pitch_in, int pf_in,
                       int pt_in, int ncs_in, int pitch_out, int pf_out, int pt_out, int ncs_out, int fmt, void* stream);
/* nn.Upsample(x2, bilinear, align_corners=True) + F.pad to the skip's size, written at `out_cp8` (already advanced to the
 * first up-sampled chunk of the concat buffer). */
int mpa_upsample2x_cp8(const void* low_cp8, void* out_cp8, int n, int C, int Tl, int Fl, int pitch_l, int pf_l, int pt_l,
                       int ncs_l, int Ts, int Fs, int pitch_s, int pf_s, int pt_s, int ncs_out, int fmt, void* stream);
/* layout converters (tests, and the seams between the fp32 and the 16-bit paths). */
int mpa_nchw_to_cp8(const float* x, void* out_cp8, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt,
                    int ncs_out, void* stream);
/* x [B][C][T][Fs] fp32 -> CP8 planes of width F with source column f on column offset + f*stride; the other real columns are NOT
 * written (they must hold the zeros of the initial allocation): zero-inserted gradient of a stride-(1,stride) convolution.
 * MPA_FMT_F16X3 writes hi and lo planes (even ncs_out; 0 = 2 * ceil(C/8)); the columns not written stay zero in both halves. */
int mpa_nchw_to_cp8_strided(const float* x, void* out_cp8, int B, int C, int T, int Fs, int F, int stride, int offset, int pitch,
                            int pf, int pt, int fmt, int ncs_out, void* stream);
int mpa_cp8_to_nchw(const void* in_cp8, float* out, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt,
                    int ncs_in, void* stream);

/* Fused head tail for the patch-wise case (T == conv3 kernel height, conv4.3 kernel 1x1; basic_cnns.py:396-408):
 * x compact 16-bit planes [B][ceil(C1/8)][T][Fo][8] (max-pooled conv2 output) -> out [B,Fo] fp32 =
 * sigmoid(conv4.3(lrelu(conv4.0(lrelu(conv3(x)))))).  w3 [C2][C1][T], w40 [C3][C2], w43 [C3] in state_dict layout.
 * C2 <= 32, C3 <= 16, Fo <= 256. */
int mpa_head_tail_cp8(const void* x_cp8, const float* w3, const float* b3, const float* w40, const float* b40,
                      const float* w43, const float* b43, float* out, int B, int C1, int T, int Fo, int C2, int C3,
                      float a_lrelu, int fmt, void* stream);

/* The head behind conv2 for the CNN family in one launch (basic_cnns.py:180-195 / :396-408): y compact 16-bit planes
 * [B][ceil(C1/8)][75][Fo][8] = LeakyReLU(conv2) -> out [B,Fo] fp32 = sigmoid(conv4.3(lrelu(conv4.0(lrelu(conv3(maxpool13(y))))))).
 * w3_packed [ceil(C1/8)][75][8][C2P] fp32 (C2P = 12 for C2 <= 12, else 16; zero padded), w40 [C3][C2], w43 [C3].
 * T == 75, C1 <= 64, C2 <= 16, C3 <= 64, fp16 / bf16 planes. */
int mpa_head_pool_conv3_tail_cp8(const void* y_cp8, const float* w3_packed, const float* b3, const float* w40, const float* b40,
                                 const float* w43, const float* b43, float* out, int B, int C1, int T, int Fo, int C2, int C3,
                                 float a_lrelu, int fmt, void* stream);

/* conv4.0 (1x1) + LeakyReLU + conv4.3 (1x1) + sigmoid on the activated conv3 output h [B][ceil(C2/8)][R][Fo][8] (compact 16-bit
 * planes, any widths) -> out [B][R][Fo] fp32 (basic_cnns.py:403-408). */
int mpa_head_tail2_cp8(const void* h_cp8, const float* w40, const float* b40, const float* w43, const float* b43,
                       float* out, int B, int R, int Fo, int C2, int C3, float a_lrelu, int fmt, void* stream);

/* ---- HCQT (H1-H3): batched multirate constant-Q filterbank ---------------------------------------------
 * replaces librosa.cqt x3 + librosa.estimate_tuning as driven by libdl/data_preprocessing/hcqt.py:122,157-162;
 * host driver: multipitch_architectures_b200/libdl/data_preprocessing/hcqt.py. */
/* y_out[t] = sqrt(2) * sum_{|j|<=31} h[|j|] * y_in[2t+j] (resampy kaiser_fast at a 2:1 ratio, librosa scale=True);
 * n_out = ceil(n_in/2), the last sample is zero when n_in is odd.  half_taps: 32 floats (device). */
int mpa_decimate2_f32(const float* y_in, float* y_out, const float* half_taps, long long n_in, void* stream);
/* General power-of-two form (librosa's one-shot early down-sampling of a CQT whose top octave lies far below Nyquist, reached by
 * compute_hcqt, hcqt.py:66-81): y_out[t] = sqrt(factor) * sum_{|j|<n_half} h[|j|] * y_in[factor*t+j], n_out = ceil(n_in/factor),
 * samples t >= floor(n_in/factor) are zero.  half_taps: n_half = 16*factor floats (device). */
int mpa_decimate_f32(const float* y_in, float* y_out, const float* half_taps, int n_half, int factor, long long n_in, void* stream);
/* Same with an explicit gain instead of sqrt(factor): gain 1 = librosa.load's resampling of a 44.1 kHz file to 22.05 kHz (notebook 01
 * cell 3; res_type kaiser_best: n_half = 64*factor taps), which does not rescale. */
int mpa_decimate_gain_f32(const float* y_in, float* y_out, const float* half_taps, int n_half, int factor, double gain, long long n_in,
                          void* stream);
/* General-ratio resampling (resampy's table walk; librosa.load of a file whose rate is not a power-of-two multiple of the target):
 * interp_win = the resampy window (float64, n_win = num_zeros*num_table + 1 entries) pre-multiplied by min(1, ratio), interp_delta its
 * forward differences; output sample t sits at input time time_register[t] (resampy's sequentially accumulated float64 register, >=
 * floor(n_in*ratio) entries; NULL = t/ratio); samples t >= floor(n_in*ratio) are zero (librosa's length fix). */
int mpa_resample_f32(const float* y_in, float* y_out, const double* interp_win, const double* interp_delta, const double* time_register,
                     int n_win, int num_table, double ratio, double gain, long long n_in, long long n_out, void* stream);
/* On-disk feature format -> network layout (exp126a...py:413-420): hcqt_fnc [F][N][C] float64 (the .npy the reference's notebook 01
 * saves) -> out [C][lead+N+trail][F] fp32 with zero pad frames (lead = 37, trail = 38 for inference, 0/0 for training files). */
int mpa_hcqt_npy_to_frames_f64(const double* hcqt_fnc, float* out, int F, int N, int C, int lead, int trail, void* stream);
/* One octave level: frame t is centred on sample t*hop of y_level (reflect padding), rectangular window, FFT of
 * n_fft, then for each of the n_rows filter rows (every CQT that runs at this rate)
 *   out[ch][t][bin] = | sum_f basis[row][f] * X[start_row + f] | * row_scale[row]   for each destination of the row.
 * Tables are laid out [n_tunings][n_rows][...] and indexed by the device-resident tuning_idx[0] (NULL -> 0).
 * basis: complex64 interleaved [.][n_rows][band]; dest: int [n_rows][n_dest] = (channel<<16 | bin) or -1. */
int mpa_cqt_level_f32(const float* y_level, long long n_level, int n_fft, int hop, int n_frames, const float* basis,
                      const int* band_start, const float* row_scale, int n_rows, int band, const int* tuning_idx,
                      const int* dest, int n_dest, float* out, int out_frames, int out_bins, void* stream);
/* All levels of one HCQT in ONE launch (grid = frames x levels; same arithmetic per (level, frame) as mpa_cqt_level_f32, so the results
 * are bit-identical to the per-level calls).  `levels`: HOST array of n_levels <= 16 descriptors holding device pointers. */
typedef struct mpa_cqt_level {
  const float* y;            /* the level's (decimated) signal */
  long long n;               /* its length in samples */
  int n_fft, hop;            /* FFT size and hop at this rate */
  const float* basis;        /* complex64 interleaved [n_tunings][n_rows][band] */
  const int* band_start;     /* [n_tunings][n_rows] */
  const float* row_scale;    /* [n_tunings][n_rows] */
  int n_rows;
  const int* dest;           /* [n_rows][n_dest] = (channel << 16 | bin) or -1 */
  int n_dest;
} mpa_cqt_level;
int mpa_cqt_levels_f32(const mpa_cqt_level* levels, int n_levels, int n_frames, int band, const int* tuning_idx, float* out,
                       int out_frames, int out_bins, void* stream);
/* Backward of mpa_cqt_levels_f32 (autograd from the HCQT to the audio): given g_out = dL/d out [H][out_frames][out_bins], writes
 * dL/d y of every level's signal.  Per (frame, level) the spectrum is recomputed from y, w_r = row_scale * (sum of g_out over the row's
 * destinations) * conj(C_r) / |C_r| (0 where |C_r| = 0), V = the transposed banded contraction of w (over the bin -> rows table),
 * frame gradient = Re(FFT(V zero-extended to n_fft)) -> workspace; then the adjoint of the reflect-padded framing (overlap-add, with every
 * reflection of signals shorter than n_fft) sums the frame gradients into g_y.  Levels that read the same signal pass the same g_y and are
 * summed together; g_y is overwritten, or added to when `accumulate` is non-zero.  Deterministic (fixed summation order, no atomics).
 * Workspace: mpa_cqt_levels_bwd_workspace bytes = n_frames * sum(n_fft) floats. */
typedef struct mpa_cqt_level_grad {
  float* g_y;                /* [n] gradient of the level's signal */
  const int* bin_off;        /* [n_tunings][n_fft/2 + 2]: rows covering bin k are bin_rows[tuning][bin_off[tuning][k] .. bin_off[tuning][k+1]) */
  const int* bin_rows;       /* [n_tunings][n_rows * band]: row indices, grouped by bin (bins < n_fft/2 + 1 only), ascending within a bin */
} mpa_cqt_level_grad;
size_t mpa_cqt_levels_bwd_workspace(const mpa_cqt_level* levels, int n_levels, int n_frames);
int mpa_cqt_levels_bwd_f32(const mpa_cqt_level* levels, const mpa_cqt_level_grad* grads, int n_levels, int n_frames, int band,
                           const int* tuning_idx, const float* g_out, int out_frames, int out_bins, int accumulate, void* workspace,
                           size_t ws_bytes, void* stream);
/* Transpose of mpa_decimate_gain_f32 for the same (half_taps, factor, gain, n_in): g_in[i] (+)= gain * sum_{t < floor(n_in/factor)}
 * h[|i - factor*t|] * g_out[t] over the taps the forward reads (taps outside the signal are skipped there, so they carry nothing back).
 * g_out: ceil(n_in/factor) floats, g_in: n_in floats, overwritten or added to (`accumulate`).  float64 accumulation. */
int mpa_decimate_adjoint_f32(const float* g_out, float* g_in, const float* half_taps, int n_half, int factor, double gain, long long n_in,
                             int accumulate, void* stream);
/* librosa.estimate_tuning(y, sr, bins_per_octave) with n_fft=2048, hop=512, fmin=150, fmax=4000, threshold=0.1,
 * resolution=0.01: writes tuning_idx[0] in [0,100), tuning = -0.5 + 0.01*idx.  hann2048: periodic hann window. */
size_t mpa_tuning_workspace(int n_frames);
int mpa_estimate_tuning_f32(const float* y, long long n, const float* hann2048, float sr, int bins_per_octave,
                            int* tuning_idx, void* workspace, size_t ws_bytes, void* stream);

/* ---- training (configuration 2: CNN family forward + backward + AdamW), fp32 NCHW ------------------------------
 * Backward of the blocks of basic_cnns.py:373-408 as autograd would compute them for the reference modules. */
/* out = a + b (residual sums of activations / gradients; in place allowed). */
int mpa_add_f32(const float* a, const float* b, float* out, long long n, void* stream);
/* g_in = g_out * act'(.) with act' expressed through the forward OUTPUT `out` (LReLU / ReLU / sigmoid). */
int mpa_act_bwd_f32(const float* out, const float* g_out, float* g_in, long long n, int act, float act_param,
                    void* stream);
/* MaxPool2d((k,1), stride 1, pad k/2) backward fused with the preceding activation's derivative: `a` is the pool's
 * forward input (= activation output); the gradient goes to the FIRST maximum of each window (ATen semantics). */
int mpa_maxpool_time_bwd_f32(const float* a, const float* g_pool, float* g_a, int B, int C, int T, int F, int k,
                             int act, float act_param, void* stream);
/* nn.Dropout(p) in training mode with a Philox-4x32-10 stream: element i uses counter (i/4, offset), key seed. */
int mpa_dropout_f32(const float* x, float* out, long long n, float p, unsigned long long seed,
                    unsigned long long offset, void* stream);
/* MaxPool((k,1)) -> Dropout(p) (-> + res) of a CNN block in one pass, and its backward (g_out = the gradient behind the dropout layer; its
 * mask is re-drawn on the fly).  The masks are those of mpa_dropout_f32 / mpa_dropout_dev_f32 for the same (seed, offset[, step_dev]).
 * Forward: F % 4 == 0; backward: k = 3 or 13. */
int mpa_maxpool_time_dropout_f32(const float* x, const float* res, float* out, int B, int C, int T, int F, int k, float p,
                                 unsigned long long seed, unsigned long long offset, const long long* step_dev,
                                 unsigned long long step_mul, void* stream);
int mpa_maxpool_time_bwd_dropout_f32(const float* a, const float* g_out, float* g_a, int B, int C, int T, int F, int k, int act,
                                     float act_param, float p, unsigned long long seed, unsigned long long offset,
                                     const long long* step_dev, unsigned long long step_mul, void* stream);
/* The same two stages (k = 3) and the bias-gradient reduction directly on 16-bit CP8 planes [B][ceil(C/8)][T+2*pt][pitch][8]
 * (geometry as mpa_nchw_to_cp8): a training step of the CNN family then runs conv -> pool+dropout -> conv and
 * dgrad -> pool backward -> wgrad / dgrad without any nchw<->CP8 converter in between.  The dropout mask is the one the fp32
 * kernels above draw for the NCHW element index of the same (b, c, t, f); sums are formed in fp32 and rounded once on the store, so the
 * planes equal mpa_nchw_to_cp8 of the fp32 kernels' results bit for bit.  Replaces, for the bf16 training mode, the reference's
 * nn.MaxPool2d((3,1),(1,1),(1,0)) + nn.Dropout forward / backward (libdl/nn_models/basic_cnns.py:172-175, 376-377) and the bias
 * gradient of the following nn.Conv2d.  F % 4 == 0.  mpa_channel_sum_cp8: out[c] = sum over (b, t, f) of channel c, fixed order. */
int mpa_pool3_dropout_cp8(const void* a_cp8, void* out_cp8, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, float p,
                          unsigned long long seed, unsigned long long offset, const long long* step_dev, unsigned long long step_mul,
                          void* stream);
int mpa_pool3_bwd_dropout_cp8(const void* a_cp8, const void* g_out_cp8, void* g_a_cp8, int B, int C, int T, int F, int pitch, int pf,
                              int pt, int fmt, int act, float act_param, float p, unsigned long long seed, unsigned long long offset,
                              const long long* step_dev, unsigned long long step_mul, void* stream);
int mpa_channel_sum_cp8(const void* g_cp8, float* out, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, int ncs,
                        void* stream);
/* The same pair with a phase-split hand-over (CNN family, head conv2 = 3x3 / stride (1,3)): the forward writes the pooled activation into
 * phase-split planes (bin f -> phase set f % out_split, column f / out_split, pitch out_pitch; layout of mpa_conv_tc_f16 out_mode 2), the
 * backward reads the gradient wrt the pool output from such planes (what the stride-1 form of conv2's data gradient writes). */
int mpa_pool3_dropout_split_cp8(const void* a_cp8, void* out_cp8, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, float p,
                                unsigned long long seed, unsigned long long offset, const long long* step_dev,
                                unsigned long long step_mul, int out_split, int out_pitch, void* stream);
int mpa_pool3_bwd_dropout_split_cp8(const void* a_cp8, const void* g_out_cp8, void* g_a_cp8, int B, int C, int T, int F, int pitch, int pf,
                                    int pt, int fmt, int act, float act_param, float p, unsigned long long seed,
                                    unsigned long long offset, const long long* step_dev, unsigned long long step_mul, int g_split,
                                    int g_pitch, void* stream);
/* U-Net family, bf16 training mode, CP8-resident (train_unet_cp8.cu): the element-wise stages between two tensor-core convolutions of a
 * training step on the 16-bit planes themselves.  Geometry arguments as mpa_nchw_to_cp8; every `ncs_*` is the chunk-plane stride per item
 * of that buffer (0 = C/8; larger for a channel view of a concat buffer); C % 8 == 0; fmt = MPA_FMT_BF16 | MPA_FMT_F16.
 *   mpa_bn_stats_cp8       stats[0..C) = batch mean, stats[C..2C) = biased batch variance of y (one pass: per slice the sums of the deviations
 *                          from `pivot[c]` (optional; the producing convolution's bias) and of their squares, then Chan's merge in a fixed order); running_mean / running_var (optional) <- (1-m)*running + m*(mean | var*n/(n-1)), num_batches_tracked += 1:
 *                          nn.BatchNorm2d in training mode (libdl/nn_models/unet_cnns.py:39,44 — double_conv's BatchNorm2d layers)
 *   mpa_bn_relu_apply_cp8  out = max(0, (y - mean) * rsqrt(var + eps) * weight + bias)        (unet_cnns.py:39-41: BatchNorm2d -> ReLU)
 *   mpa_bn_relu_bwd_cp8    the backward of that pair: g' = g * [out > 0] (out recomputed from y), g_bias = sum g', g_weight = sum g' * xhat,
 *                          dy = weight * rstd * (g' - mean(g') - xhat * mean(g' * xhat)) written as CP8 (the operand of the preceding
 *                          convolution's weight / data gradient), g_conv_bias (optional) = sum dy — what loss.backward() leaves in
 *                          BatchNorm2d.weight.grad / .bias.grad and Conv2d.bias.grad
 *                          out_split / g_split = s > 0 (with the split planes' pitch): the activation is written to / the gradient is read from
 *                          PHASE-SPLIT planes (bin f -> phase set f % s, column f / s; mpa_conv_tc_f16 out_mode 2), the hand-over to the head's
 *                          stride-(1, s) convolution in its stride-1 form and back from its data gradient
 *   mpa_maxpool2x2_bwd_cp8 out = addend (optional) + MaxPool2d(2) backward of g_pool: the gradient goes to the first maximum of each 2x2 window
 *                          in row-major order (ATen); `a` is the un-pooled activation, pooled level = (T/2, F/2)   (unet_cnns.py:60-61 `down`)
 *   mpa_upsample2x_bwd_cp8 g_low = adjoint of mpa_upsample2x_cp8 (bilinear x2, align_corners=True, zero pad to (Ts, Fs)) applied to g_up
 *                          (unet_cnns.py:83-101 `unet_up_concat_padding`) */
int mpa_bn_stats_cp8(const void* y_cp8, float* stats, const float* pivot, int B, int C, int T, int F, int pitch, int pf, int pt, int ncs,
                     int fmt, float* running_mean, float* running_var, float momentum, long long* num_batches_tracked, void* stream);
int mpa_bn_relu_apply_cp8(const void* y_cp8, void* out_cp8, const float* stats, const float* weight, const float* bias, float eps, int B,
                          int C, int T, int F, int pitch, int pf, int pt, int ncs_y, int ncs_out, int out_split, int out_pitch, int fmt,
                          void* stream);
int mpa_bn_relu_bwd_cp8(const void* g_cp8, const void* y_cp8, void* dy_cp8, const float* stats, const float* weight, const float* bias,
                        float eps, float* g_weight, float* g_bias, float* g_conv_bias, int B, int C, int T, int F, int pitch, int pf, int pt,
                        int ncs_g, int ncs_y, int ncs_dy, int g_split, int g_pitch, int fmt, void* stream);
int mpa_maxpool2x2_bwd_cp8(const void* a_cp8, const void* g_pool_cp8, const void* addend_cp8, void* out_cp8, int B, int C, int T, int F,
                           int pitch, int pf, int pt, int ncs_a, int ncs_add, int ncs_out, int pitch_o, int pf_o, int pt_o, int ncs_gp,
                           int fmt, void* stream);
int mpa_upsample2x_bwd_cp8(const void* g_up_cp8, void* g_low_cp8, int B, int C, int Tl, int Fl, int pitch_l, int pf_l, int pt_l,
                           int ncs_low, int Ts, int Fs, int pitch_s, int pf_s, int pt_s, int ncs_up, int fmt, void* stream);
/* Eval-mode backward of BatchNorm2d -> ReLU on the planes (BatchNorm frozen: `stats` = [running_mean | running_var], the format
 * mpa_bn_relu_apply_cp8 reads; nothing is updated): g' = g * [out > 0] (out recomputed from y), dy = weight * rstd * g' written as CP8,
 * g_weight = sum g' * xhat, g_bias = sum g', g_conv_bias (optional) = sum dy — the convolution's bias gradient, NOT zero here.  One launch
 * on the (chunk, slice) grid of mpa_bn_relu_bwd_cp8 with the same ordered merge (bit-reproducible); g_split / g_pitch as there. */
int mpa_bn_relu_bwd_frozen_cp8(const void* g_cp8, const void* y_cp8, void* dy_cp8, const float* stats, const float* weight, const float* bias,
                               float eps, float* g_weight, float* g_bias, float* g_conv_bias, int B, int C, int T, int F, int pitch, int pf,
                               int pt, int ncs_g, int ncs_y, int ncs_dy, int g_split, int g_pitch, int fmt, void* stream);
/* Training path of the attention half of transformer_enc_layer (libdl/nn_models/unet_cnns.py:131-153: q/k/v Linear -> nn.MultiheadAttention over
 * the BATCH axis -> o Linear -> Dropout -> add -> LayerNorm1), fp32, one CTA per bottleneck position (enc_train.cu).
 *   mpa_enc_fold_f32        w_qkv [3E,E] (+ transpose w_qkvT [E,3E]) = in_proj_weight_z . {q,k,v}_linear.weight, w_proj [E,E] (+ w_projT) =
 *                           o_linear.weight . out_proj.weight, b_proj = o_linear.weight . out_proj.bias  — one launch
 *   mpa_enc_fold_bwd_f32    the chain rule through that fold: from d w_qkv / d w_proj / d b_proj to the gradients of the reference's seven
 *                           parameters (all overwritten) — one launch
 *   mpa_enc_attn_train_fwd_f32  x [B,E,S] (NCHW bottleneck) -> t = Dropout(tokens + PE) (only behind a positional encoding, as the reference),
 *                           qkv, att, u1 = t + Dropout(att W_proj^T + b_proj), h1 = LayerNorm1(u1); all [B*S, .] token-major, saved for the backward.
 *                           Dropout sites: element index of the [B*S,E] matrix, offset = site (+ step_dev[0] * step_mul), as mpa_dropout_f32.
 *   mpa_enc_attn_train_bwd_f32  g_h1 -> g_x [B,E,S] (overwritten), g_p (gradient wrt the projection output) and g_qkv for the weight-gradient
 *                           GEMMs, LayerNorm1 parameter gradients (overwritten)
 *   mpa_enc_train_supported 1 when the shape fits (E % 32 == 0, E <= 128, head dim <= 16, the B x E tiles of one position in shared memory) */
int mpa_enc_train_supported(int B, int E, int num_heads);
int mpa_enc_fold_f32(const float* in_proj_weight, const float* wq, const float* wk, const float* wv, const float* wo,
                     const float* out_proj_weight, const float* out_proj_bias, float* w_qkv, float* w_qkvT, float* w_proj, float* w_projT,
                     float* b_proj, int E, void* stream);
int mpa_enc_fold_bwd_f32(const float* d_w_qkv, const float* d_w_proj, const float* d_b_proj, const float* in_proj_weight, const float* wq,
                         const float* wk, const float* wv, const float* wo, const float* out_proj_weight, const float* out_proj_bias,
                         float* g_in_proj_weight, float* g_wq, float* g_wk, float* g_wv, float* g_wo, float* g_out_proj_weight,
                         float* g_out_proj_bias, int E, void* stream);
int mpa_enc_attn_train_fwd_f32(const float* x, const float* pe, const float* w_qkvT, const float* b_qkv, const float* w_projT,
                               const float* b_proj, const float* ln_w, const float* ln_b, float eps, float* t, float* qkv, float* att,
                               float* u1, float* h1, int B, int E, int S, int num_heads, float p_drop, unsigned long long seed,
                               unsigned long long site_tok, unsigned long long site_att, const long long* step_dev,
                               unsigned long long step_mul, void* stream);
int mpa_enc_attn_train_bwd_f32(const float* g_h1, const float* u1, const float* qkv, const float* w_qkv, const float* w_proj,
                               const float* ln_w, float eps, float* g_p, float* g_qkv, float* g_x, float* g_ln_w, float* g_ln_b, int B, int E,
                               int S, int num_heads, int has_pe, float p_drop, unsigned long long seed, unsigned long long site_tok,
                               unsigned long long site_att, const long long* step_dev, unsigned long long step_mul, void* stream);
/* Same with offset = step_dev[0] * step_mul + site, the step counter read from DEVICE memory: a training step captured in a CUDA graph
 * (UnetTrainStep(graph=True)) then draws fresh masks on every replay, identical to the eager step of the same number. */
int mpa_dropout_dev_f32(const float* x, float* out, long long n, float p, unsigned long long seed, unsigned long long site,
                        const long long* step_dev, unsigned long long step_mul, void* stream);
/* Conv2d data gradient, any stride (gather form); w in state_dict layout [Cout][Cin][KH][KW]. */
int mpa_conv2d_dgrad_f32(const float* g_out, const float* w, float* g_in, int B, int Cin, int H, int W, int Cout,
                         int KH, int KW, int sh, int sw, int ph, int pw, void* stream);
/* Conv2d weight (+ bias, g_b may be NULL) gradient; g_w [Cout][Cin][KH][KW] is overwritten.  KW <= 16. */
int mpa_conv2d_wgrad_f32(const float* x, const float* g_out, float* g_w, float* g_b, int B, int Cin, int H, int W,
                         int Cout, int KH, int KW, int sh, int sw, int ph, int pw, void* stream);
/* Gradients of the LayerNorm([C,F]) affine parameters (the network input needs no gradient); x is the layer INPUT. */
int mpa_layernorm_cf_param_grad_f32(const float* x, const float* g_out, float* g_w, float* g_b, int B, int C, int T,
                                    int F, float eps, float gamma_log, void* stream);
/* torch.optim.AdamW step on one flat tensor (exp126a…py:103-108,293); grad is multiplied by grad_scale first. */
int mpa_adamw_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                  float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale, void* stream);
/* Dynamic loss scaling of fp16 training (torch.amp.GradScaler defaults in the caller: 2^16, x2 after 2000 clean steps, x0.5 on an overflow).
 * The state lives in device memory, so a step needs no host synchronisation and a CUDA-graph replay behaves as the eager step.
 * *found_inf = 1 when any of x[0, n) is an inf or a NaN, else 0 (overwritten; any alignment, any n). */
int mpa_nonfinite_check_f32(const float* x, long long n, int* found_inf, void* stream);
/* mpa_adamw_f32 on grad * grad_scale / *loss_scale (grad_scale: the world-size factor of an all-reduced gradient), bias-corrected for step
 * *applied_steps + 1 — or, when *found_inf is set, nothing at all (param, exp_avg, exp_avg_sq untouched).  Then the scaler update:
 * overflow -> *loss_scale *= backoff_factor, *growth_tracker = 0; else ++*applied_steps, and after growth_interval clean steps in a row
 * *loss_scale *= growth_factor (kept if finite), *growth_tracker = 0. */
int mpa_adamw_scaled_f32(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr, float beta1, float beta2,
                         float eps, float weight_decay, float grad_scale, const int* found_inf, float* loss_scale, int* growth_tracker,
                         int* applied_steps, float growth_factor, float backoff_factor, int growth_interval, void* stream);

/* ---- tcgen05 GEMM for the token-wise Linear layers of transformer_enc_layer (unet_cnns.py:131-157) ------------------------
 * Y[M,N] fp32 row-major = act(X[M,K] * W[N,K]^T + bias[N]) with 16-bit operands in the chunk layout [ceil(K/64)*8][rows padded][8]
 * produced by mpa_gemm_tc_to_chunks (row_tile 256 for X = tokens, 128 for W = nn.Linear.weight); fp32 accumulate in TMEM.
 * Wide-K products with few output tiles are split over K and combined with atomicAdd (not with relu). */
size_t mpa_gemm_tc_chunked_bytes(int rows, int K, int row_tile);
/* transposed = 1: the source is stored [K][rows] (the operand is the transpose of a row-major matrix: weight / activation gradients). */
int mpa_gemm_tc_to_chunks(const float* x_rows, void* out_chunks, int rows, int K, int row_tile, int fmt, int transposed, void* stream);
int mpa_gemm_tc_f16(const void* x_chunks, const void* w_chunks, const float* bias, float* y, int M, int N, int K, int relu, int fmt,
                    void* stream);
/* out[b][c][.] = act(x[b][c][.] + bias[c]) on NCHW fp32 (in place allowed; bias may be NULL): bias + activation of a convolution whose
 * K slices met in atomics (the tensor-core form of the head's 75x1 convolution, nn.Conv2d + nn.LeakyReLU, unet_cnns.py:380-386). */
int mpa_bias_act_f32(const float* x, const float* bias, float* out, int B, int C, int HW, int act, float act_param, void* stream);
/* The same product described by a struct, with the options the training path needs:
 *  - operand-layout copies of the result written by the epilogue (no converter launch, no fp32 round trip of the [M, mlp_dim] tensors of
 *    the encoder MLP and its backward; only without K split):
 *      y_tok     16-bit token-chunked copy [y_tok_chunks][y_tok_rows][8] = the operand of a later product that reduces over the M tokens
 *                (weight gradients dW = g^T x): chunk = 8 consecutive tokens, row = output feature; chunks past ceil(M/8) must be
 *                pre-zeroed by the caller, they are never written
 *      y_feat    16-bit feature-chunked copy [ceil(N/128)*16][y_feat_rows][8] = the X operand of the next Linear layer (K = N)
 *      mask_tok  a tensor in y_tok's layout (same strides): the result is zeroed where it is <= 0 — ReLU backward against the saved
 *                activation;  colsum [N] += column sums of the (masked) result — the bias gradient (atomics; pre-zeroed)
 *  - x_rows / w_rows: row stride of the X / W operand buffers when they are padded further than this product needs (0 = default)
 *  - strided fp32 result: element (m, n) at y[moff(m) + noff(n)], moff(m) = (m / y_mn2) * y_ms1 + (m % y_mn2) * y_ms2 (y_mn2 == 0: m * y_ms2,
 *    y_ms2 == 0: N), noff alike (default 1): the product writes straight into an NCHW tensor whose (item, bin) pair is one GEMM
 *    dimension.  This is how the head's full-height 75x1 convolution (libdl/nn_models/unet_cnns.py:380-385, basic_cnns.py:396-401) and its
 *    two gradients run on the tensor cores: operands chunked by mpa_gemm_tc_strided_to_chunks, which reads element (r, k) of a tensor at
 *    (r / r_n2) * r_s1 + (r % r_n2) * r_s2 + (k / k_n2) * k_s1 + (k % k_n2) * k_s2.  With a strided result the K split (atomics) is used only
 *    when the caller has zeroed y (y_zeroed = 1).
 *  - residual add + LayerNorm epilogue (N <= 128, no K split, no other epilogue output): ln_out[b][n][s] (NCHW, s < ln_S) =
 *    LayerNorm_n(result + bias + ln_res[m][n]) * ln_w + ln_b for token m = b * ln_S + s — the second add & LayerNorm of transformer_enc_layer
 *    (unet_cnns.py:155-158) inside the MLP's second product, so that an encoder layer forward is 3 launches. */
typedef struct mpa_gemm_tc_desc {
  const void* x_chunks;
  const void* w_chunks;
  const float* bias;
  float* y;
  int M, N, K, relu, fmt, x_rows, w_rows;
  void* y_tok;
  int y_tok_rows, y_tok_chunks;
  void* y_feat;
  int y_feat_rows;
  const void* mask_tok;
  float* colsum;
  int y_mn2, y_nn2, y_zeroed;
  long long y_ms1, y_ms2, y_ns1, y_ns2;
  const float *ln_res, *ln_w, *ln_b;   /* residual + LayerNorm epilogue (see above); ln_out NULL = off */
  float* ln_out;
  float ln_eps;
  int ln_S;
} mpa_gemm_tc_desc;
int mpa_gemm_tc_run(const mpa_gemm_tc_desc* desc, void* stream);
int mpa_gemm_tc_strided_to_chunks(const float* x, void* out_chunks, int rows, int K, int row_tile, int fmt, int r_n2, long long r_s1,
                                  long long r_s2, int k_n2, long long k_s1, long long k_s2, void* stream);

/* ---- tensor-core training convolutions (bf16 / fp16 CP8 operands, fp32 accumulate) -------------------------------------
 * Weight gradient of a stride-1 "same" KHxKW convolution (nn.Conv2d backward): gw[co0+co][ci0+ci][kh][kw] +=
 * sum_{b,t,f} g[b,co,t,f] * x[b,ci,t+kh-KH/2,f+kw-KW/2]; x / g are CP8 planes of the same geometry (zero gap columns!), gw is the
 * fp32 gradient in state_dict layout [Cout_total][Cin_total][KH][KW] and must be ZEROED by the caller (results are accumulated with
 * atomicAdd).  zero_row: >= ceil(Cout/8)*pitch*16 bytes of zeros (rows outside the patch).  Cout <= 128 per call (use channel-block views). */
int mpa_conv_wgrad_tc(const void* x_cp8, const void* g_cp8, const void* zero_row, float* gw, int n_items, int Cin, int Cout, int T,
                      int F, int KH, int KW, int pitch, int pf, int pt, int x_nc_stride, int g_nc_stride, int Cin_total, int ci0,
                      int Cout_total, int co0, int fmt, void* stream);
/* The same weight gradient in split precision: x / g are MPA_FMT_F16X3 planes (hi planes in the first half of each item's chunk stride, lo
 * planes in the second; the strides must be even, 0 = 2 * ceil(C/8)); three MMA passes per K step, g_hi.x_hi + g_lo.x_hi + g_hi.x_lo, into
 * one fp32 accumulator.  KW >= 3 (there is no KW == 1 form).  Other arguments and conditions as mpa_conv_wgrad_tc. */
int mpa_conv_wgrad_tc_x3(const void* x_cp8, const void* g_cp8, const void* zero_row, float* gw, int n_items, int Cin, int Cout, int T,
                         int F, int KH, int KW, int pitch, int pf, int pt, int x_nc_stride, int g_nc_stride, int Cin_total, int ci0,
                         int Cout_total, int co0, void* stream);
/* out[c] = sum_{b,hw} x[b][c][hw] (bias gradient of a convolution). */
int mpa_channel_sum_f32(const float* x, float* out, int B, int C, int HW, void* stream);

/* ---- training of the U-Net / SAUnet family (configuration 5), fp32 NCHW ------------------------------------------------
 * BatchNorm2d(train) [+ ReLU] backward (unet_cnns.py:50-57): x = conv output (BN input), out = block output (ReLU mask),
 * stats = [mean | biased var] from mpa_bn_stats_f32; scratch2c: 2*C floats. */
int mpa_bn_relu_bwd_f32(const float* x, const float* out, const float* dy, const float* stats, const float* w, float* dx,
                        float* dw, float* db, float* scratch2c, int B, int C, int HW, float eps, int relu, void* stream);
/* The same with BatchNorm2d frozen (eval mode): stats = [running_mean | running_var]; dx = w * rstd * dy' (dy' = dy * [out > 0] when
 * relu), dw = sum dy' * xhat, db = sum dy'; d_conv_bias (optional) = sum dx, the preceding convolution's bias gradient. */
int mpa_bn_relu_bwd_frozen_f32(const float* x, const float* out, const float* dy, const float* stats, const float* w, float* dx, float* dw,
                               float* db, float* d_conv_bias, float* scratch2c, int B, int C, int HW, float eps, int relu, void* stream);
/* MaxPool2d((kh,kw), stride (sh,sw)) backward, floor mode, gradient to the first maximum of each window. */
int mpa_maxpool2d_bwd_f32(const float* x, const float* g_out, float* g_in, int B, int C, int H, int W, int kh, int kw,
                          int sh, int sw, void* stream);
/* unet_up_concat_padding backward: g_cat [B,Cs+Cl,Hs,Ws] -> g_skip (= or +=) and g_low [B,Cl,Hl,Wl]. */
int mpa_upsample2x_concat_bwd_f32(const float* g_cat, float* g_skip, int accumulate_skip, float* g_low, int B, int Cl,
                                  int Hl, int Wl, int Cs, int Hs, int Ws, void* stream);
/* encoder-layer stages as separate calls (transformer_enc_layer, unet_cnns.py:148-159) and their backward pieces. */
int mpa_enc_gather_f32(const float* x, const float* pe, float* tok, int B, int E, int S, void* stream);
int mpa_gemm_nt_f32(const float* A, const float* W, const float* bias, float* C, int M, int N, int K, int relu, void* stream);
int mpa_batch_axis_attention_f32(const float* qkv, float* out, int B, int S, int E, int num_heads, void* stream);
int mpa_add_layernorm_tok_f32(const float* a, const float* b, const float* w, const float* bias, float* out_tok,
                              float* out_nchw, long long n_tok, int E, int S, float eps, void* stream);
/* C[M,N] (=|+=) A*B with mode 0: A [M,K] B [K,N]; mode 1: A [K,M] (transposed) B [K,N]. */
int mpa_gemm_f32(const float* A, const float* B, float* C, int M, int N, int K, int mode, int accumulate, void* stream);
int mpa_colsum_f32(const float* A, float* out, int M, int N, void* stream);
/* y = LayerNorm_E(u)*w+b backward per token: g_u, and g_w / g_b (overwritten). */
int mpa_layernorm_tok_bwd_f32(const float* u, const float* g_y, const float* w, float* g_u, float* g_w, float* g_b,
                              long long n_tok, int E, float eps, void* stream);
int mpa_batch_axis_attention_bwd_f32(const float* qkv, const float* g_o, float* g_qkv, int B, int S, int E, int num_heads,
                                     void* stream);
/* tokens [(b*S+s)][E] <-> NCHW [B,E,S] */
int mpa_nchw_tokens_f32(const float* src, float* dst, int B, int E, int S, int to_tokens, void* stream);
/* PUnet degree-of-polyphony loss (RETRAIN4_exp195f...rerun1.py:343-345): scale * CrossEntropyLoss(mean)(logits [B,K],
 * class = (long) sum_p y_true[b,p]) forward (added to *loss_sum when accumulate_loss, else overwriting) + d/d logits. */
int mpa_ce_count_fwd_bwd_f32(const float* logits, const float* y_true, float* loss_sum, float* grad_logits, int B, int K,
                             int P, float scale, int accumulate_loss, void* stream);
/* The same with grad_logits multiplied by *loss_scale (device memory; the loss of fp16 training is scaled for its backward only). */
int mpa_ce_count_fwd_bwd_scaled_f32(const float* logits, const float* y_true, float* loss_sum, float* grad_logits, int B, int K, int P,
                                    float scale, int accumulate_loss, const float* loss_scale, void* stream);

/* ---- N11: BCELoss(mean) on sigmoid outputs with the -100 log clamp, forward + d(loss)/d(pred) ---------- */
int mpa_bce_fwd_bwd_f32(const float* y_pred, const float* y_true, float* loss_sum, float* grad_pred, long long n,
                        void* stream);
/* The same with grad_pred multiplied by *loss_scale (device memory); *loss_sum stays the unscaled loss. */
int mpa_bce_fwd_bwd_scaled_f32(const float* y_pred, const float* y_true, float* loss_sum, float* grad_pred, long long n,
                               const float* loss_scale, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MPA_H_ */
