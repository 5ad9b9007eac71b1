// tcgen05 / TMEM implicit-GEMM "same" convolution (stride 1) on 16-bit channel-chunk planes (CP8; fp16 or bf16).
//
// Formulation ("weights as A, one padded image row as N"):
//   D[(j,co), n] += sum_k  A[(j,co), k] * B[k, n]
//     M = 128 lanes  = J output rows x Cout channels  (J = floor(128/Cout); rows t0 .. t0+J-1 of one patch)
//     N = row pitch  = every column of ONE padded image row (224 for F=216), so a tap shift is a pure
//                      start-address shift of the shared-memory operand (no im2col is ever materialised)
//     K = input rows (KH+J-1) x taps KW x input channels, walked 16 channels-or-taps at a time.
//   A (weights) is pre-packed on the host in the exact order the MMA issuer walks K; the J row blocks hold the
//   same filter shifted down by j rows, so one pass over KH+J-1 input rows yields J output rows.
//   B (activations) lives in shared memory as [chunk][pixel][8 ch] (16 B per pixel per chunk), the K-major
//   SWIZZLE_NONE canonical layout with SBO = 128 B: operand row r sits at start + 16*r, so the tap (df) of a
//   15-wide filter is start + 16*df.  The second 16-byte K slice is reached through LBO: the next channel
//   chunk (LBO = plane stride) or, for an odd chunk count, the next tap (LBO = 16 B).
//   Zero padding in frequency is physical (zero gap columns between rows of the CP8 plane); zero padding in
//   time is realised by skipping the K steps of out-of-range input rows.
//
// Pipeline (one CTA per SM, persistent over work units = (patch, row group)):
//   warp 0  producer : cp.async.bulk (1-D TMA) of activation row slabs and packed weight stages -> mbarriers
//   warp 1  MMA      : one thread issues tcgen05.mma (kind::f16, fp16/bf16 in, fp32 accumulate in TMEM) from a
//                      pre-built shared-memory table of B descriptors
//   warps 2-9 epilogue: two warps per TMEM lane quadrant, alternating 32-column chunks: tcgen05.ld -> +bias ->
//                      activation -> 16-bit -> transposed through shared memory -> 16-byte coalesced CP8 stores
//   The accumulator is double buffered in TMEM (2 x 224 of 512 columns): the epilogue of unit k overlaps the
//   main loop of unit k+1.  Weights stream from L2 once per unit (36 B/clk/SM, ~30 % of L2 throughput).
#include "common.cuh"
#include <cuda.h>
#include <cuda_fp16.h>
#include <vector>
#include <string.h>
#include <math.h>

namespace mpa {

constexpr int kStageMMAs = 8;                 // MMAs (K=16 steps) per weight stage
constexpr int kATileBytes = 2 * 128 * 16;     // one MMA's A tile: [2 k-slices][128 rows][16 B]
constexpr int kAStageBytes = kStageMMAs * kATileBytes;
constexpr int kMaxAStages = 5;             // weight stages: as many as fit next to the activation slabs (>= 2)
constexpr int kNumBStages = 2;              // minimum number of activation stages (what the stage sizing guarantees)
constexpr int kMaxBStages = 8;              // thin inputs: as many as fit next to the weight stages (b_stages)
constexpr int kThreads = 320;                 // producer warp, MMA warp, 8 epilogue warps
constexpr int kMaxRingS = 24;                // ring positions (<= J + 4, J <= 16) and activation stages of the ring main loop
constexpr int kMaxRingB = 8;
constexpr int kMaxGrid = 160;                 // upper bound of the persistent grid (scratch-ring sizing)
constexpr int kEpiPitch = 40;                 // 80-byte rows: conflict-free 16-byte reads in the transposing epilogue
constexpr unsigned long long kWaitTimeoutNs = 4000000000ull;   // bounded waits: a protocol bug traps instead of hanging the GPU

struct ConvTcParams {
  // ---- input: virtual patch rows.  Rows [0,in_e) and [T-in_e,T) of patch b live in per-patch "edge" planes (in_e == T: the whole
  // patch is materialised), every other row r in ONE shared stream at row b*in_stream_patch_rows + r (patch-independent rows are
  // stored once per frame instead of once per patch).  All pointers address (row 0, column 0) of patch 0, chunk 0.
  const uint8_t* in_edge;
  const uint8_t* in_stream;
  long long in_edge_patch_stride, in_edge_chunk_stride, in_stream_chunk_stride;   // bytes
  long long in_stream_patch_rows;
  int in_e;
  const uint8_t* w;         // packed weights
  const float* bias;        // [Cout]
  // ---- output, legacy epilogue (pool == 0)
  uint16_t* out;            // out_mode 0: CP8 planes [n][NCo][T_out+2pt][P][8]; out_mode 1: compact [n][NCo][T_out][F_out][8] (sub-sampled columns)
  int out_mode, sub_stride, sub_offset, F_out, fmt;
  // out_mode 2 (phase split): column f goes to phase plane set f % sub_stride, column pf2 + f / sub_stride of CP8 planes of pitch P2;
  // the phase plane sets are `phase_planes` chunk planes apart: [n][sub_stride][phase_planes][T_out+2pt][P2][8]
  int P2, pf2, phase_planes;
  int out_split;            // fused epilogue (pool == 3, out_e == T): z written phase-split with sub_stride = out_split phases
  // ---- output, fused epilogue (pool == 3): z = maxpool_time3(act(conv + bias)) (+ input row) written with the same virtual row scheme
  uint8_t* out_edge;
  uint8_t* out_stream;
  long long out_edge_patch_stride, out_edge_chunk_stride, out_stream_chunk_stride, out_stream_patch_rows;
  int out_e, pool, residual;
  uint8_t* ring;            // per-CTA scratch of activated conv rows: [grid][2 banks][J][NCo][P][16 B]
  // ---- geometry
  int n_patches, NC, Cout, J, T, F, KH, KW, P, N, pf, pt_out, TP_out, T_out, row0, NCo;
  int n_seg, y_lo[2], y_hi[2], z_lo[2], z_hi[2], seg_groups[2], groups_per_patch;
  int mmas_per_row, n_units, slab_px, epi_off, a_stages, b_stages, btab_off;
  int resident;             // tile main loop: the whole weight set fits in the A stages -> loaded once per CTA, never re-streamed
  long long out_patch_stride;  // elements (16-bit) between patches in `out`
  int act;
  float act_param;
  uint32_t idesc;
  // ---- split-precision mode (MPA_FMT_F16X3): every tensor is a (hi, lo) pair of fp16 planes, x = hi + lo (hi = fp16(x), lo = fp16(x - hi));
  // the lo planes of a buffer sit `*_lo_off` chunk planes after its hi planes.  One input row is two B stages (hi planes, then lo planes) and
  // three passes of A tiles: W_hi x_hi, W_lo x_hi (same B stage), W_hi x_lo — 3 MMAs per product, ~2^-21 relative operand error.
  // The weights are pre-scaled per output channel by a power of two (so that W_lo stays clear of the fp16 subnormals); the epilogue
  // multiplies the accumulator by inv_scale[co].
  int x3, in_lo_off, out_lo_off, tiles_per_row;
  const float* inv_scale;
  // ---- wide-K / row-merged mode of the tile main loop (KW == 1 convolutions with many input chunks, e.g. the phase-split conv2 of the
  // U-Net heads, 384 -> 104 channels): (a) R consecutive image rows form ONE operand row of N = R * pitch columns (rows are contiguous in
  // memory and a KH x 1 filter has no horizontal taps), so every weight tile is used for R output rows instead of one; (b) an activation
  // stage holds G of the NC input chunks (the K loop of an input row walks ceil(NC / G) stages), which keeps the stages inside 227 KB.
  int R, G, n_groups;
  // Rs: image rows between two merged rows.  1: the R rows are consecutive (one bulk copy; needs J == 1).  J: merged row rr holds image
  // row (r + J*rr), so that row block j of the A tile and merged row rr together produce output row t0 + j + J*rr: R*J output rows
  // per unit with the J-fold weight reuse of the stacked filters kept (the head's 40-channel conv2: 9 rows per unit instead of 3; its
  // work units were so small that fixed per-unit costs, not the tensor pipe, set the pace).  The R rows arrive as R separate copies;
  // rows outside the plane (+ guard rows) are skipped, their columns only feed outputs that are never stored.
  int Rs, pt_in;
  // Row-merged modes (R > 1, consecutive or spaced rows): the R rows of ALL planes of a stage arrive as ONE tensor-map copy (cp.async.bulk.tensor, box = pitch x R rows at row
  // stride Rs x G planes; rows outside [0, T) are zero-filled by the copy unit) instead of R * G bulk copies of one 1.3 KB row each — the
  // copy unit retires ~1 bulk copy per 150 clocks whatever its size, which made these layers copy-issue bound (ncu, CNN:XS conv2: 127 copies
  // = 19 k clocks per work unit, the MMA warp waiting 57 % of its time for a stage).  tma = 0: the descriptor could not be built.
  int tma, tma_c0;   // 1: merged rows, 2: one row of all planes (narrow levels); tma_c0: inner start coordinate
  int bpad;          // zero bytes behind every activation stage (set with the tensor-map layouts; kept when the descriptor cannot be built)
  alignas(64) CUtensorMap tmap;
  uint32_t btab[256];       // tile main loop: B-descriptor low words of one K row, (offset >> 4) | (LBO >> 4) << 16 (x3: the row twice)
  // ---- ring main loop (conv_tc_ring_kernel): un-duplicated weight pieces, see below
  int ring_on, ring_S, ring_npos, ring_ps, ring_sbo, ring_nb, ring_b_off, ring_bar_off;
};

// ------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const unsigned long long t0 = global_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 255u) == 0 && global_ns() - t0 > kWaitTimeoutNs) __trap();
  }
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ uint16_t cvt16(float x, int fmt) {
  return fmt == MPA_FMT_BF16 ? __bfloat16_as_ushort(__float2bfloat16(x)) : __half_as_ushort(__float2half_rn(x));
}
__device__ __forceinline__ float cvt32(uint16_t v, int fmt) {
  return fmt == MPA_FMT_BF16 ? __bfloat162float(__ushort_as_bfloat16(v)) : __half2float(__ushort_as_half(v));
}

// split-precision halves of an fp32 value: part 0 = fp16(x), part 1 = fp16(x - fp16(x))
__device__ __forceinline__ uint16_t split16(float x, int part) {
  const __half h = __float2half_rn(x);
  return __half_as_ushort(part == 0 ? h : __float2half_rn(x - __half2float(h)));
}
__device__ __forceinline__ void join8(const uint4& hi, const uint4& lo, float* v) {
  const __half2* h = reinterpret_cast<const __half2*>(&hi);
  const __half2* l = reinterpret_cast<const __half2*>(&lo);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const float2 a = __half22float2(h[e]), b = __half22float2(l[e]);
    v[2 * e] = a.x + b.x;
    v[2 * e + 1] = a.y + b.y;
  }
}
__device__ __forceinline__ void split8(const float* v, uint4& hi, uint4& lo) {
  __half2* h = reinterpret_cast<__half2*>(&hi);
  __half2* l = reinterpret_cast<__half2*>(&lo);
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    h[e] = __floats2half2_rn(v[2 * e], v[2 * e + 1]);
    const float2 r = __half22float2(h[e]);
    l[e] = __floats2half2_rn(v[2 * e] - r.x, v[2 * e + 1] - r.y);
  }
}

// K-major, SWIZZLE_NONE shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}

// ------------------------------------------------------------------------------------------ unit decoding
struct UnitInfo {
  int b, seg, t0;        // patch, segment, first conv row of the unit
  bool first_in_seg;
};
__device__ __forceinline__ UnitInfo decode_unit(const ConvTcParams& p, int u) {
  UnitInfo ui;
  ui.b = u / p.groups_per_patch;
  int g = u - ui.b * p.groups_per_patch;
  ui.seg = 0;
  if (g >= p.seg_groups[0]) { g -= p.seg_groups[0]; ui.seg = 1; }
  ui.t0 = p.y_lo[ui.seg] + g * p.J * p.R;
  ui.first_in_seg = (g == 0);
  return ui;
}
// Work units are dealt to CTAs in CONTIGUOUS ranges (a CTA walks down the rows of a patch, so the fused pool finds the
// neighbouring conv rows in its own scratch ring).  In pool mode a range that starts in the middle of a segment is preceded
// by one warm-up unit (the previous row group) whose pooled output is suppressed.
__device__ __forceinline__ void unit_range(const ConvTcParams& p, int& u_begin, int& u_end, int& u_first_real) {
  const long long U = p.n_units;
  u_first_real = (int)(U * blockIdx.x / gridDim.x);
  u_end = (int)(U * (blockIdx.x + 1) / gridDim.x);
  u_begin = u_first_real;
  if (p.pool && u_first_real < u_end && !decode_unit(p, u_first_real).first_in_seg) u_begin = u_first_real - 1;
}
// byte address of (patch b, row, column 0, chunk 0) of the virtual input and the chunk stride that goes with it
__device__ __forceinline__ const uint8_t* in_row_ptr(const ConvTcParams& p, int b, int row, long long& chunk_stride) {
  if (row < p.in_e || row >= p.T - p.in_e) {
    const int idx = row < p.in_e ? row : row - (p.T - 2 * p.in_e);
    chunk_stride = p.in_edge_chunk_stride;
    return p.in_edge + (long long)b * p.in_edge_patch_stride + (long long)idx * p.P * 16;
  }
  chunk_stride = p.in_stream_chunk_stride;
  return p.in_stream + ((long long)b * p.in_stream_patch_rows + row) * p.P * 16;
}
__device__ __forceinline__ uint8_t* out_row_ptr(const ConvTcParams& p, int b, int row, long long& chunk_stride) {
  if (row < p.out_e || row >= p.T - p.out_e) {
    const int idx = row < p.out_e ? row : row - (p.T - 2 * p.out_e);
    chunk_stride = p.out_edge_chunk_stride;
    return p.out_edge + (long long)b * p.out_edge_patch_stride + (long long)idx * p.P * 16;
  }
  chunk_stride = p.out_stream_chunk_stride;
  return p.out_stream + ((long long)b * p.out_stream_patch_rows + row) * p.P * 16;
}
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

__device__ __forceinline__ uint4 max8_rt(uint4 c, const uint4 a, int fmt) {
  if (fmt == MPA_FMT_BF16) {
    __nv_bfloat162* cm = reinterpret_cast<__nv_bfloat162*>(&c);
    const __nv_bfloat162* am = reinterpret_cast<const __nv_bfloat162*>(&a);
#pragma unroll
    for (int e = 0; e < 4; ++e) cm[e] = __hmax2(cm[e], am[e]);
  } else {
    __half2* cm = reinterpret_cast<__half2*>(&c);
    const __half2* am = reinterpret_cast<const __half2*>(&a);
#pragma unroll
    for (int e = 0; e < 4; ++e) cm[e] = __hmax2(cm[e], am[e]);
  }
  return c;
}
__device__ __forceinline__ uint4 add8_rt(uint4 c, const uint4 r, int fmt) {
  if (fmt == MPA_FMT_BF16) {
    __nv_bfloat162* cm = reinterpret_cast<__nv_bfloat162*>(&c);
    const __nv_bfloat162* rm = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 a = __bfloat1622float2(cm[e]), b2 = __bfloat1622float2(rm[e]);
      cm[e] = __floats2bfloat162_rn(a.x + b2.x, a.y + b2.y);
    }
  } else {
    __half2* cm = reinterpret_cast<__half2*>(&c);
    const __half2* rm = reinterpret_cast<const __half2*>(&r);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 a = __half22float2(cm[e]), b2 = __half22float2(rm[e]);
      cm[e] = __floats2half2_rn(a.x + b2.x, a.y + b2.y);
    }
  }
  return c;
}

// ------------------------------------------------------------------------------------------ epilogue role (warps 2..9)
template <bool X3>
__device__ __forceinline__ void epilogue_role(const ConvTcParams& p, uint32_t tmem_base, uint16_t* epi_smem, uint64_t* acc_full, uint64_t* acc_empty,
                                              int u_begin, int u_end, int u_first_real) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  {
    // ===================================================== epilogue (warps 2..9: two warps per TMEM lane quadrant)
    const int quad = warp & 3;
    const int m = quad * 32 + lane;             // accumulator row = (j, co)
    const int j = m / p.Cout, co = m - j * p.Cout;
    const bool row_valid = (j < p.J);
    const float bias = row_valid ? p.bias[co] : 0.f;
    const float inv_scale = (X3 && row_valid) ? p.inv_scale[co] : 1.f;
    constexpr int n_parts = X3 ? 2 : 1;
    // activations of the form max(x, slope * x): none (slope 1), ReLU (0), LeakyReLU with 0 <= slope <= 1
    const float act_slope = p.act == MPA_ACT_NONE ? 1.f : p.act == MPA_ACT_RELU ? 0.f : p.act_param;
    const bool fast_act = p.act != MPA_ACT_SIGMOID && act_slope >= 0.f && act_slope <= 1.f;
    const int NCoP = n_parts * p.NCo;                                 // chunk planes of one activated conv row in the scratch ring
    // coalesced path: 8 consecutive lanes = the 8 channels of one chunk of one output row (needs Cout % 8 == 0)
    const bool staged = ((p.Cout & 7) == 0);
    const int ewarp = warp - 2;                                       // 0..7
    const int ehalf = ewarp >> 2;                                     // which half of the 32-column chunks this warp drains
    const int etid = threadIdx.x - 64;                                // 0..255 within the epilogue group
    uint16_t* stile = epi_smem + ewarp * (32 * kEpiPitch);            // [32 columns][kEpiPitch >= 32 lanes] 16-bit
    // per-thread constants of the transposed store phase: the 4 channel-chunk groups of this warp's 32 accumulator rows
    int grp_j[4], grp_plane[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int mg = quad * 32 + k * 8;
      grp_j[k] = mg / p.Cout;
      grp_plane[k] = (mg - grp_j[k] * p.Cout) >> 3;
    }
    const size_t plane_elems = (p.out_mode == 0) ? (size_t)p.TP_out * p.P * 8 : (p.out_mode == 2) ? (size_t)p.TP_out * p.P2 * 8 : (size_t)p.T_out * p.F_out * 8;
    const int row_pitch = (p.out_mode == 0) ? p.P : (p.out_mode == 2) ? p.P2 : p.F_out;
    const size_t ring_row_bytes = (size_t)NCoP * p.P * 16;
    uint8_t* ring_cta = p.pool ? p.ring + (size_t)blockIdx.x * 2 * p.J * ring_row_bytes : nullptr;
    uint32_t k_unit = 0;
    for (int u = u_begin; u < u_end; ++u, ++k_unit) {
      const UnitInfo ui = decode_unit(p, u);
      const int b = ui.b, t0 = ui.t0;
      const int y_hi = p.y_hi[ui.seg];
      const int t = t0 + j;
      const uint32_t buf = k_unit & 1u, acc_par = (k_unit >> 1) & 1u;
      uint8_t* ring_bank = p.pool ? ring_cta + (size_t)(k_unit & 1u) * p.J * ring_row_bytes : nullptr;
      mbar_wait(&acc_full[buf], acc_par);
      tc_fence_after();
      uint16_t* out_b = p.out + (size_t)b * p.out_patch_stride;
      for (int c0 = ehalf * 32; c0 < p.N; c0 += 64) {
        // which of the 32 columns of this chunk are stored at all (real, and selected by the sub-sampling)?
        const int n = c0 + lane;
        int rr = 0, nn = n;                      // row-merged operand rows: column n = row rr of the unit, column nn of that row
        if (p.R > 1) { rr = n / p.P; nn = n - rr * p.P; }
        int fo = nn - p.pf;
        bool col_ok = (fo >= 0 && fo < p.F && rr < p.R);
        int col_out = nn, ph_plane = 0;
        if (p.out_mode == 1) {
          fo -= p.sub_offset;
          col_ok = col_ok && fo >= 0 && (fo % p.sub_stride) == 0;
          col_out = fo / p.sub_stride;
        } else if (p.out_mode == 2 && col_ok) {
          const int q = fo / p.sub_stride;
          ph_plane = (fo - q * p.sub_stride) * p.phase_planes;
          col_out = p.pf2 + q;
        }
        const uint32_t keep = __ballot_sync(0xffffffffu, col_ok);
        if (keep == 0) continue;
        uint32_t v[32];
        tc_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * 256 + c0), v);
        tc_wait_ld();
        if (staged) {
          for (int part = 0; part < n_parts; ++part) {
            if (!X3 && fast_act) {
              // the common case, branch-free per element: none / ReLU / LeakyReLU(0 <= slope <= 1) are all max(x, slope * x); columns
              // that are not kept are converted too (finite accumulators; their staging slots are never read)
              if (p.fmt == MPA_FMT_BF16) {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                  const float x = fmaf(__uint_as_float(v[i]), inv_scale, bias);
                  stile[i * kEpiPitch + lane] = __bfloat16_as_ushort(__float2bfloat16(fmaxf(x, x * act_slope)));
                }
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                  const float x = fmaf(__uint_as_float(v[i]), inv_scale, bias);
                  stile[i * kEpiPitch + lane] = __half_as_ushort(__float2half_rn(fmaxf(x, x * act_slope)));
                }
              }
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                if ((keep >> i) & 1u) {
                  const float x = apply_act(fmaf(__uint_as_float(v[i]), inv_scale, bias), p.act, p.act_param);
                  stile[i * kEpiPitch + lane] = X3 ? split16(x, part) : cvt16(x, p.fmt);
                }
              }
            }
            __syncwarp();
            // lane -> column c0+lane; pass k -> the k-th 8-lane group (= one channel chunk of one output row) of this warp
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int tg = t0 + grp_j[k] + rr * p.Rs;
              if (col_ok && grp_j[k] < p.J && tg < y_hi) {
                const uint4 val = *reinterpret_cast<const uint4*>(stile + lane * kEpiPitch + k * 8);
                if (p.pool) {
                  *reinterpret_cast<uint4*>(ring_bank + ((size_t)grp_j[k] * NCoP + part * p.NCo + grp_plane[k]) * p.P * 16 + (size_t)n * 16) = val;
                } else {
                  const int orow = (p.out_mode != 1 ? p.pt_out : 0) + tg - p.row0;
                  *reinterpret_cast<uint4*>(out_b + (size_t)(part * p.out_lo_off + ph_plane + grp_plane[k]) * plane_elems +
                                            ((size_t)orow * row_pitch + col_out) * 8) = val;
                }
              }
            }
            __syncwarp();
          }
        } else if (row_valid && t < y_hi) {
          // scalar fallback (Cout not a multiple of 8; never used with the fused pool): one 16-bit store per value
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const int n2 = c0 + i;
            int fo2 = n2 - p.pf;
            bool ok = (fo2 >= 0 && fo2 < p.F);
            if (p.out_mode == 1) {
              fo2 -= p.sub_offset;
              ok = ok && fo2 >= 0 && (fo2 % p.sub_stride) == 0;
              fo2 /= p.sub_stride;
            }
            if (ok) {
              uint16_t* dst = (p.out_mode == 0)
                                  ? p.out + (size_t)b * p.out_patch_stride + ((((size_t)(co >> 3)) * p.TP_out + p.pt_out + t - p.row0) * p.P + n2) * 8 + (co & 7)
                                  : p.out + (size_t)b * p.out_patch_stride + ((((size_t)(co >> 3)) * p.T_out + t - p.row0) * p.F_out + fo2) * 8 + (co & 7);
              *dst = cvt16(apply_act(__uint_as_float(v[i]) + bias, p.act, p.act_param), p.fmt);
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&acc_empty[buf]);
      if (p.pool) {
        // ---- fused MaxPool((3,1), stride 1, pad (1,0)) + residual.  The activated conv rows of this unit are in the current
        // ring bank, the two rows above them in the other bank (written by this CTA one unit ago).
        epi_bar_sync();
        if (u >= u_first_real) {
          const int t_last = min(t0 + p.J, y_hi) - 1;
          int ze_lo = max(ui.first_in_seg ? p.z_lo[ui.seg] : t0 - 1, p.z_lo[ui.seg]);
          int ze_hi = min(t_last == p.T - 1 ? t_last : t_last - 1, p.z_hi[ui.seg] - 1);
          const uint8_t* ring_prev = ring_cta + (size_t)((k_unit & 1u) ^ 1u) * p.J * ring_row_bytes;
          const int n_items = (ze_hi - ze_lo + 1) * p.NCo * p.F;
          if (X3) {
            // split precision: max and residual add on the joined fp32 values (hi + lo is exact in fp32), re-split on the way out
            for (int it = etid; it < n_items; it += 256) {
              const int f = it % p.F;
              int r = it / p.F;
              const int ck = r % p.NCo;
              const int tz = ze_lo + r / p.NCo;
              const size_t col_off = (size_t)ck * p.P * 16 + (size_t)(p.pf + f) * 16;
              const size_t lo_off = (size_t)p.NCo * p.P * 16;
              auto yrow = [&](int ty, float* o) {
                const uint8_t* base = ty >= t0 ? ring_bank + (size_t)(ty - t0) * ring_row_bytes : ring_prev + (size_t)(p.J + ty - t0) * ring_row_bytes;
                join8(*reinterpret_cast<const uint4*>(base + col_off), *reinterpret_cast<const uint4*>(base + col_off + lo_off), o);
              };
              float c[8], o[8];
              yrow(tz, c);
              if (tz > 0) {
                yrow(tz - 1, o);
#pragma unroll
                for (int e = 0; e < 8; ++e) c[e] = fmaxf(c[e], o[e]);
              }
              if (tz < p.T - 1) {
                yrow(tz + 1, o);
#pragma unroll
                for (int e = 0; e < 8; ++e) c[e] = fmaxf(c[e], o[e]);
              }
              if (p.residual) {
                long long cs;
                const uint8_t* rp = in_row_ptr(p, b, tz, cs) + (size_t)(p.pf + f) * 16;
                join8(*reinterpret_cast<const uint4*>(rp + (long long)ck * cs), *reinterpret_cast<const uint4*>(rp + (long long)(p.in_lo_off + ck) * cs), o);
#pragma unroll
                for (int e = 0; e < 8; ++e) c[e] += o[e];
              }
              uint4 hi, lo;
              split8(c, hi, lo);
              if (p.out_split) {
                const int q = f / p.out_split, ph = f - q * p.out_split;
                uint8_t* op = p.out_edge + (long long)b * p.out_edge_patch_stride + ((long long)tz * p.P2 + p.pf2 + q) * 16;
                *reinterpret_cast<uint4*>(op + (long long)(ph * p.NCo + ck) * p.out_edge_chunk_stride) = hi;
                *reinterpret_cast<uint4*>(op + (long long)(p.out_lo_off + ph * p.NCo + ck) * p.out_edge_chunk_stride) = lo;
              } else {
                long long ocs;
                uint8_t* op = out_row_ptr(p, b, tz, ocs) + (size_t)(p.pf + f) * 16;
                *reinterpret_cast<uint4*>(op + (long long)ck * ocs) = hi;
                *reinterpret_cast<uint4*>(op + (long long)(p.out_lo_off + ck) * ocs) = lo;
              }
            }
          } else
          for (int it = etid; it < n_items; it += 256) {
            const int f = it % p.F;
            int r = it / p.F;
            const int ck = r % p.NCo;
            const int tz = ze_lo + r / p.NCo;
            const size_t col_off = (size_t)ck * p.P * 16 + (size_t)(p.pf + f) * 16;
            auto yrow = [&](int ty) -> uint4 {
              const uint8_t* base = ty >= t0 ? ring_bank + (size_t)(ty - t0) * ring_row_bytes : ring_prev + (size_t)(p.J + ty - t0) * ring_row_bytes;
              return *reinterpret_cast<const uint4*>(base + col_off);
            };
            uint4 c = yrow(tz);
            if (tz > 0) c = max8_rt(c, yrow(tz - 1), p.fmt);
            if (tz < p.T - 1) c = max8_rt(c, yrow(tz + 1), p.fmt);
            if (p.residual) {
              long long cs;
              const uint8_t* rp = in_row_ptr(p, b, tz, cs);
              c = add8_rt(c, *reinterpret_cast<const uint4*>(rp + (long long)ck * cs + (size_t)(p.pf + f) * 16), p.fmt);
            }
            if (p.out_split) {
              // materialised output in phase-split planes [patch][phase][chunk][T+2][P2][8] (the input of the head's stride-(1,s) conv2)
              const int q = f / p.out_split, ph = f - q * p.out_split;
              uint8_t* op = p.out_edge + (long long)b * p.out_edge_patch_stride + (long long)(ph * p.NCo + ck) * p.out_edge_chunk_stride +
                            ((long long)tz * p.P2 + p.pf2 + q) * 16;
              *reinterpret_cast<uint4*>(op) = c;
            } else {
              long long ocs;
              uint8_t* op = out_row_ptr(p, b, tz, ocs);
              *reinterpret_cast<uint4*>(op + (long long)ck * ocs + (size_t)(p.pf + f) * 16) = c;
            }
          }
        }
        epi_bar_sync();
      }
    }
  }
}

// ------------------------------------------------------------------------------------------ kernel
template <bool X3>
__global__ void __launch_bounds__(kThreads, 1) conv_tc_kernel(const __grid_constant__ ConvTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int slab_plane_bytes = p.slab_px * 16;
  const int bstage_bytes = min(p.G, p.NC) * slab_plane_bytes + p.bpad;   // one patch, one input row, one chunk group (+ zero pad: the odd chunk's dummy K slice over-reads one pixel)
  const int kNumAStages = p.a_stages;
  uint8_t* a_smem = smem;                                // [a_stages][kAStageBytes]
  uint8_t* b_smem = smem + kNumAStages * kAStageBytes;   // [kNumBStages][NC][slab_px][16B]
  const int nbs = p.b_stages;                            // 2 .. kMaxBStages activation stages
  uint64_t* bars = reinterpret_cast<uint64_t*>(b_smem + nbs * bstage_bytes);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + kMaxAStages;
  uint64_t* b_full = bars + 2 * kMaxAStages;
  uint64_t* b_empty = b_full + kMaxBStages;
  uint64_t* acc_full = b_empty + kMaxBStages;            // [2]
  uint64_t* acc_empty = acc_full + 2;                    // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  uint32_t* btab = reinterpret_cast<uint32_t*>(smem + p.btab_off);         // [mmas_per_row padded to 8] B-descriptor low words
  uint16_t* epi_smem = reinterpret_cast<uint16_t*>(smem + p.epi_off);      // 8 warps x [32][kEpiPitch] 16-bit staging

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kNumAStages; ++i) {
      mbar_init(&a_full[i], 1);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < nbs; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], kThreads - 64);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (p.Rs > 1 || p.bpad) {
    // skipped rows and the over-read tail of a stage are never written by a copy: they must hold finite values (their columns feed
    // outputs that are discarded, or meet zero weights)
    for (int i = threadIdx.x; i < nbs * bstage_bytes / 16; i += kThreads) reinterpret_cast<uint4*>(b_smem)[i] = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int ph = p.KH / 2, pw = p.KW / 2;
  const int rows_in = p.KH + p.J - 1;
  constexpr int n_parts = X3 ? 2 : 1;
  int u_begin, u_end, u_first_real;
  unit_range(p, u_begin, u_end, u_first_real);

  if (warp == 0) {
    // ===================================================== producer
    // The whole warp walks the (warp-uniform) loops; lane 0 waits on / arms the barriers and issues the weight copies, the activation
    // copies of a stage — one per chunk plane (x merged row) — are issued by 32 lanes at once.  (A single thread needs ~170 clocks per
    // bulk copy for the address arithmetic and the issue; wide-K stages of 16-45 copies per ~1,000 tensor-clocks were bound by that.)
    {
      int a_stage = 0, b_stage = 0;
      uint32_t a_phase = 0, b_phase = 0;
      if (lane == 0 && p.resident && u_begin < u_end) {
        // small filters (the head's 3x3): every weight stage has its own slot and is loaded exactly once
        const int spr = (p.mmas_per_row + kStageMMAs - 1) / kStageMMAs;
        for (int r = 0; r < rows_in; ++r)
          for (int m0 = 0; m0 < p.mmas_per_row; m0 += kStageMMAs) {
            const int nm = min(kStageMMAs, p.mmas_per_row - m0), idx = r * spr + m0 / kStageMMAs;
            mbar_expect_tx(&a_full[idx], (uint32_t)(nm * kATileBytes));
            bulk_g2s(a_smem + idx * kAStageBytes, p.w + ((size_t)r * p.mmas_per_row + m0) * kATileBytes, (uint32_t)(nm * kATileBytes), &a_full[idx]);
          }
      }
      __syncwarp();
      for (int u = u_begin; u < u_end; ++u) {
        const UnitInfo ui = decode_unit(p, u);
        for (int r = 0; r < rows_in; ++r) {
          const int row = ui.t0 - ph + r;
          if (p.R == 1 && (row < 0 || row >= p.T)) continue;      // row-merged mode: the zero guard rows stand in for the time padding
          for (int part = 0; part < n_parts; ++part) {
           for (int gi = 0; gi < p.n_groups; ++gi) {
            // activation slab of this input row: chunk group gi (split precision: the hi planes, then the lo planes)
            const int planes = min(p.G, p.NC - gi * p.G);
            uint8_t* dst = b_smem + b_stage * bstage_bytes;
            if (p.tma) {
              // spaced merged rows of all planes of the stage in one tensor-map copy
              if (lane == 0) {
                mbar_wait(&b_empty[b_stage], b_phase ^ 1);
                mbar_expect_tx(&b_full[b_stage], (uint32_t)(min(p.G, p.NC) * slab_plane_bytes));
                asm volatile(
                    "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
                        smem_u32(dst)),
                    "l"(reinterpret_cast<uint64_t>(&p.tmap)), "r"(p.tma_c0), "r"(row), "r"(gi * p.G), "r"(ui.b), "r"(smem_u32(&b_full[b_stage]))
                    : "memory");
              }
            } else if (p.Rs > 1) {
              // spaced merged rows: one copy of `pitch` pixels per (plane, merged row); rows beyond the guard rows are left out
              int n_ok = 0;
              for (int rr = 0; rr < p.R; ++rr) {
                const int rw = row + rr * p.Rs;
                n_ok += (rw >= -p.pt_in && rw < p.T + p.pt_in) ? 1 : 0;
              }
              if (lane == 0) {
                mbar_wait(&b_empty[b_stage], b_phase ^ 1);
                mbar_expect_tx(&b_full[b_stage], (uint32_t)(planes * n_ok * p.P * 16));
              }
              __syncwarp();
              long long cs;
              const uint8_t* src = in_row_ptr(p, ui.b, 0, cs) + (long long)(gi * p.G) * cs;       // materialised patches: row r at r * pitch
              for (int i = lane; i < planes * p.R; i += 32) {
                const int rr = i / planes, c = i - rr * planes;
                const int rw = row + rr * p.Rs;
                if (rw < -p.pt_in || rw >= p.T + p.pt_in) continue;
                bulk_g2s(dst + c * slab_plane_bytes + rr * p.P * 16, src + (long long)c * cs + (long long)rw * p.P * 16, (uint32_t)(p.P * 16),
                         &b_full[b_stage]);
              }
            } else {
              if (lane == 0) {
                mbar_wait(&b_empty[b_stage], b_phase ^ 1);
                mbar_expect_tx(&b_full[b_stage], (uint32_t)(planes * slab_plane_bytes));
              }
              __syncwarp();
              long long cs;
              const uint8_t* src = in_row_ptr(p, ui.b, row, cs) - pw * 16;
              src += (long long)((part ? p.in_lo_off : 0) + gi * p.G) * cs;
              for (int c = lane; c < planes; c += 32)
                bulk_g2s(dst + c * slab_plane_bytes, src + (long long)c * cs, (uint32_t)slab_plane_bytes, &b_full[b_stage]);
            }
            __syncwarp();
            if (++b_stage == nbs) { b_stage = 0; b_phase ^= 1; }
            // weight stages of this K row (split precision: W_hi and W_lo tiles against the hi planes, W_hi tiles against the lo planes)
            if (p.resident) continue;
            const int q0 = gi * (p.G / 2) * p.KW;
            const int n_tiles = (X3 && part == 0) ? 2 * p.mmas_per_row : (gi == p.n_groups - 1 ? p.mmas_per_row : (gi + 1) * (p.G / 2) * p.KW) - q0;
            const uint8_t* wrow = p.w + ((size_t)r * p.tiles_per_row + (part ? 2 * p.mmas_per_row : 0) + q0) * kATileBytes;
            for (int m0 = 0; m0 < n_tiles; m0 += kStageMMAs) {
              const int nm = min(kStageMMAs, n_tiles - m0);
              if (lane == 0) {
                mbar_wait(&a_empty[a_stage], a_phase ^ 1);
                mbar_expect_tx(&a_full[a_stage], (uint32_t)(nm * kATileBytes));
                bulk_g2s(a_smem + a_stage * kAStageBytes, wrow + (size_t)m0 * kATileBytes, (uint32_t)(nm * kATileBytes), &a_full[a_stage]);
              }
              if (++a_stage == kNumAStages) { a_stage = 0; a_phase ^= 1; }
            }
           }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    // The whole warp walks the loops and waits (warp-uniform control flow and operands); one elected lane issues.  The B-descriptor
    // words of one K row come from the kernel parameters (constant bank -> uniform registers), so an MMA costs a constant load
    // and two uniform adds in the issuing thread (the per-MMA cost of that thread bounds the kernel once L2 keeps up).
    {
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      int a_stage = 0, b_stage = 0;
      uint32_t a_phase = 0, b_phase = 0;
      constexpr uint32_t kDescHi = (128u >> 4) | (1u << 14);                 // SBO = 128 B, descriptor version 1
      constexpr uint32_t kALoFixed = ((128u * 16u) >> 4) << 16;              // A: LBO = 2048 B between the two k-slices
      const uint32_t asm16 = smem_u32(a_smem) >> 4, bsm16 = smem_u32(b_smem) >> 4, bst16 = (uint32_t)bstage_bytes >> 4;
      uint32_t k_unit = 0;
      const int spr = (p.mmas_per_row + kStageMMAs - 1) / kStageMMAs;
      if (p.resident && u_begin < u_end)
        for (int i = 0; i < rows_in * spr; ++i) mbar_wait(&a_full[i], 0);     // the resident weight set has landed
      for (int u = u_begin; u < u_end; ++u, ++k_unit) {
        const UnitInfo ui = decode_unit(p, u);
        const uint32_t buf = k_unit & 1u, acc_par = (k_unit >> 1) & 1u;
        mbar_wait(&acc_empty[buf], acc_par ^ 1);     // epilogue has drained this accumulator (two units ago)
        tc_fence_after();
        const uint32_t tmem_d = tmem_u + buf * 256;
        uint32_t accum = 0;
        for (int r = 0; r < rows_in; ++r) {
          const int row = ui.t0 - ph + r;
          if (p.R == 1 && (row < 0 || row >= p.T)) continue;
          for (int part = 0; part < n_parts; ++part) {
          for (int gi = 0; gi < p.n_groups; ++gi) {
          const int q0 = gi * (p.G / 2) * p.KW;
          const int n_tiles = (X3 && part == 0) ? 2 * p.mmas_per_row : (gi == p.n_groups - 1 ? p.mmas_per_row : (gi + 1) * (p.G / 2) * p.KW) - q0;
          mbar_wait(&b_full[b_stage], b_phase);
          const uint32_t bbase16 = bsm16 + (uint32_t)b_stage * bst16;
          for (int m0 = 0; m0 < n_tiles; m0 += kStageMMAs) {
            const int nm = min(kStageMMAs, n_tiles - m0);
            if (p.resident) a_stage = r * spr + m0 / kStageMMAs;
            else mbar_wait(&a_full[a_stage], a_phase);
            tc_fence_after();
            const uint32_t a_lo = (asm16 + (uint32_t)a_stage * (kAStageBytes >> 4)) | kALoFixed;
            if (elect_one_sync()) {
              const int qb = q0 + m0;
              if (nm == kStageMMAs) {
                tc_mma_f16(tmem_d, ((uint64_t)kDescHi << 32) | (uint64_t)a_lo, ((uint64_t)kDescHi << 32) | (uint64_t)(bbase16 + p.btab[qb]), p.idesc, accum);
#pragma unroll
                for (int i = 1; i < kStageMMAs; ++i)
                  tc_mma_f16(tmem_d, ((uint64_t)kDescHi << 32) | (uint64_t)(a_lo + (uint32_t)i * (kATileBytes >> 4)),
                             ((uint64_t)kDescHi << 32) | (uint64_t)(bbase16 + p.btab[qb + i]), p.idesc, 1u);
              } else {
                for (int i = 0; i < nm; ++i)
                  tc_mma_f16(tmem_d, ((uint64_t)kDescHi << 32) | (uint64_t)(a_lo + (uint32_t)i * (kATileBytes >> 4)),
                             ((uint64_t)kDescHi << 32) | (uint64_t)(bbase16 + p.btab[qb + i]), p.idesc, (i == 0) ? accum : 1u);
              }
              if (!p.resident) tc_commit(&a_empty[a_stage]);       // frees the weight stage when its MMAs have retired
            }
            __syncwarp();
            accum = 1;
            if (!p.resident && ++a_stage == kNumAStages) { a_stage = 0; a_phase ^= 1; }
          }
          if (elect_one_sync()) tc_commit(&b_empty[b_stage]);         // frees the activation slab of this row
          __syncwarp();
          if (++b_stage == nbs) { b_stage = 0; b_phase ^= 1; }
          }
          }
        }
        if (elect_one_sync()) tc_commit(&acc_full[buf]);              // accumulator complete -> epilogue
        __syncwarp();
      }
    }
    __syncwarp();
  } else {
    epilogue_role<X3>(p, tmem_base, epi_smem, acc_full, acc_empty, u_begin, u_end, u_first_real);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

// ------------------------------------------------------------------------------------------ ring main loop
// The J row blocks of the A operand hold the SAME filter rows shifted by one input row (block j of the tile of input row r =
// filter row r-j), so streaming ready-made 128-row tiles moves every weight J times through L2->SM (36 B/clk/SM at J = 3: the
// measured limiter of conv_tc_kernel).  Here the weights travel as "pieces" = one filter row, all Cout channels, for the K
// slices of one channel-chunk GROUP (two chunks x KW taps, or the odd last chunk with taps paired), laid out
//     ring[position][row group of 8 channels][q][k-slice][8 rows][16 B]        (SBO = Q*256 B between row groups, LBO = 128 B)
// in a shared-memory ring whose positions DESCEND as r grows: the tile of input row r is simply the J pieces starting at the
// position of filter row r (block j = the next position = filter row r-1 ...), i.e. a descriptor start address — nothing is
// copied twice except the J-1 pieces that wrap (mirrored behind the ring's end).  The K loop runs group-major (all input rows
// of a unit for chunk pair 0, then pair 1, ...), so only one group's pieces are resident: J+2..J+4 positions.
// Q MMAs of one tile: A descriptors step by 256 B (next q of the piece), B descriptors by BSTEP pixels (16 B each)
template <int Q, int BSTEP>
__device__ __forceinline__ void issue_tile(uint32_t tmem_d, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc, uint32_t first) {
  tc_mma_f16(tmem_d, ((uint64_t)a_hi << 32) | (uint64_t)a_lo, ((uint64_t)b_hi << 32) | (uint64_t)b_lo, idesc, first ? 0u : 1u);
#pragma unroll
  for (int q = 1; q < Q; ++q)
    tc_mma_f16(tmem_d, ((uint64_t)a_hi << 32) | (uint64_t)(a_lo + (uint32_t)q * 16u), ((uint64_t)b_hi << 32) | (uint64_t)(b_lo + (uint32_t)(q * BSTEP)), idesc, 1u);
}
__device__ __forceinline__ void ring_group(const ConvTcParams& p, int g, int& Q, int& planes, int& chunk0) {
  if (g < p.NC / 2) { Q = p.KW; planes = 2; chunk0 = 2 * g; }
  else { Q = (p.KW + 1) / 2; planes = 1; chunk0 = p.NC - 1; }
}

__global__ void __launch_bounds__(kThreads, 1) conv_tc_ring_kernel(const ConvTcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  const int slab_plane_bytes = p.slab_px * 16;
  const int bstage_bytes = 2 * slab_plane_bytes;
  const int S = p.ring_S, NB = p.ring_nb;
  uint8_t* ring = smem;                                   // [ring_npos][ring_ps]
  uint8_t* b_smem = smem + p.ring_b_off;                  // [NB][2 planes][slab_px][16 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.ring_bar_off);
  uint64_t* w_full = bars;                                // [S]
  uint64_t* w_empty = bars + kMaxRingS;                   // [S]
  uint64_t* b_full = bars + 2 * kMaxRingS;                // [NB]
  uint64_t* b_empty = b_full + kMaxRingB;
  uint64_t* acc_full = b_empty + kMaxRingB;               // [2]
  uint64_t* acc_empty = acc_full + 2;                     // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  uint32_t* btab = reinterpret_cast<uint32_t*>(smem + p.btab_off);         // [group][16] B-descriptor low words
  uint16_t* epi_smem = reinterpret_cast<uint16_t*>(smem + p.epi_off);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) { mbar_init(&w_full[i], 1); mbar_init(&w_empty[i], 1); }
    for (int i = 0; i < NB; ++i) { mbar_init(&b_full[i], 1); mbar_init(&b_empty[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], kThreads - 64); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int ph = p.KH / 2, pw = p.KW / 2;
  const int rows_in = p.KH + p.J - 1;
  const int NG = (p.NC + 1) / 2;
  const int G8 = p.Cout >> 3;
  const int n_kh = p.KH + 2 * (p.J - 1);                  // filter-row pieces per group in the packed array (zero pieces at both ends)
  int u_begin, u_end, u_first_real;
  unit_range(p, u_begin, u_end, u_first_real);

  if (warp == 0) {
    // ===================================================== producer: weight pieces + activation slabs, in consumption order
    if (lane == 0) {
      uint32_t n_piece = 0;                                 // running piece counter: position = S-1 - n % S
      int b_stage = 0;
      uint32_t b_phase = 0;
      for (int u = u_begin; u < u_end; ++u) {
        const UnitInfo ui = decode_unit(p, u);
        const int r_first = max(0, ph - ui.t0), r_last = min(rows_in - 1, p.T - 1 - ui.t0 + ph);
        size_t g_off = 0;
        for (int g = 0; g < NG; ++g) {
          int Q, planes, chunk0;
          ring_group(p, g, Q, planes, chunk0);
          const uint32_t row_bytes = (uint32_t)Q * 256u;                     // one row group of 8 channels, all q, both k-slices
          const uint8_t* wg = p.w + g_off;
          for (int kh = r_first - (p.J - 1); kh <= r_last; ++kh, ++n_piece) {
            const int pos = S - 1 - (int)(n_piece % (uint32_t)S);
            const uint32_t round = n_piece / (uint32_t)S;
            const bool mirror = pos <= p.J - 2;
            mbar_wait(&w_empty[pos], (round & 1u) ^ 1u);
            const bool mir = mirror;
            mbar_expect_tx(&w_full[pos], (uint32_t)G8 * row_bytes * (mir ? 2u : 1u));
            const uint8_t* src = wg + (size_t)(kh + p.J - 1) * G8 * row_bytes;
            uint8_t* dst = ring + (size_t)pos * p.ring_ps;
            if (row_bytes == (uint32_t)p.ring_sbo) {
              // the piece is contiguous in shared memory as well: one bulk copy (plus its mirror)
              bulk_g2s(dst, src, (uint32_t)G8 * row_bytes, &w_full[pos]);
              if (mir) bulk_g2s(dst + (size_t)S * p.ring_ps, src, (uint32_t)G8 * row_bytes, &w_full[pos]);
            } else {
              for (int g8 = 0; g8 < G8; ++g8) {
                bulk_g2s(dst + (size_t)g8 * p.ring_sbo, src + (size_t)g8 * row_bytes, row_bytes, &w_full[pos]);
                if (mir) bulk_g2s(dst + (size_t)S * p.ring_ps + (size_t)g8 * p.ring_sbo, src + (size_t)g8 * row_bytes, row_bytes, &w_full[pos]);
              }
            }
            if (kh >= r_first) {
              // activation slab (this group's planes) of input row kh
              const int row = ui.t0 - ph + kh;
              mbar_wait(&b_empty[b_stage], b_phase ^ 1);
              mbar_expect_tx(&b_full[b_stage], (uint32_t)(planes * slab_plane_bytes));
              long long cs;
              const uint8_t* bsrc = in_row_ptr(p, ui.b, row, cs) - pw * 16 + (long long)chunk0 * cs;
              uint8_t* bdst = b_smem + b_stage * bstage_bytes;
              for (int c = 0; c < planes; ++c)
                bulk_g2s(bdst + c * slab_plane_bytes, bsrc + (long long)c * cs, (uint32_t)slab_plane_bytes, &b_full[b_stage]);
              if (++b_stage == NB) { b_stage = 0; b_phase ^= 1; }
            }
          }
          g_off += (size_t)n_kh * G8 * row_bytes;
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================== MMA issuer
    // The whole warp walks the loops and waits on the barriers (warp-uniform control flow, every operand of the issue path
    // derived from kernel parameters / uniform values); one elected lane issues the MMAs and commits.  The issue sequence is
    // kept to two integer adds per MMA: the per-MMA cost of the single issuing thread is what bounds this kernel next to L2.
    {
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      uint32_t n_piece = 0;
      int b_stage = 0;
      uint32_t b_phase = 0;
      const uint32_t kDescHiB = (128u >> 4) | (1u << 14);                            // B: SBO = 128 B
      const uint32_t kDescHiA = ((uint32_t)p.ring_sbo >> 4) | (1u << 14);            // A: SBO = Q*256 B between 8-row groups
      constexpr uint32_t kALoFixed = (128u >> 4) << 16;                              // A: LBO = 128 B between the two k-slices
      const uint32_t ring16 = smem_u32(ring) >> 4, ps16 = (uint32_t)p.ring_ps >> 4;
      const uint32_t bsm16 = smem_u32(b_smem) >> 4, bst16 = (uint32_t)bstage_bytes >> 4;
      const uint32_t plane16 = (uint32_t)slab_plane_bytes >> 4;
      uint32_t k_unit = 0;
      for (int u = u_begin; u < u_end; ++u, ++k_unit) {
        const UnitInfo ui = decode_unit(p, u);
        const int r_first = max(0, ph - ui.t0), r_last = min(rows_in - 1, p.T - 1 - ui.t0 + ph);
        const uint32_t buf = k_unit & 1u, acc_par = (k_unit >> 1) & 1u;
        mbar_wait(&acc_empty[buf], acc_par ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_u + buf * 256;
        uint32_t first = 1;                                 // the unit's very first MMA overwrites the accumulator
        for (int g = 0; g < NG; ++g) {
          const bool pair = g < p.NC / 2;
          const int Q = pair ? p.KW : (p.KW + 1) / 2;
          const uint32_t b_lo_fixed = pair ? (plane16 << 16) : (1u << 16);           // LBO: the other chunk's plane / the next tap
          for (int kh = r_first - (p.J - 1); kh <= r_last; ++kh, ++n_piece) {
            const int pos = S - 1 - (int)(n_piece % (uint32_t)S);
            mbar_wait(&w_full[pos], (n_piece / (uint32_t)S) & 1u);
            if (kh < r_first) continue;                    // pre-loaded pieces of the first tile
            mbar_wait(&b_full[b_stage], b_phase);
            tc_fence_after();
            const uint32_t a_lo = (ring16 + (uint32_t)pos * ps16) | kALoFixed;
            const uint32_t b_lo = (bsm16 + (uint32_t)b_stage * bst16) | b_lo_fixed;
            const uint32_t n_old = n_piece - (uint32_t)(p.J - 1);
            if (elect_one_sync()) {
              if (pair && Q == 15) issue_tile<15, 1>(tmem_d, a_lo, kDescHiA, b_lo, kDescHiB, p.idesc, first);
              else if (!pair && Q == 8) issue_tile<8, 2>(tmem_d, a_lo, kDescHiA, b_lo, kDescHiB, p.idesc, first);
              else {
                const uint32_t bstep = pair ? 1u : 2u;
                for (int q = 0; q < Q; ++q)
                  tc_mma_f16(tmem_d, ((uint64_t)kDescHiA << 32) | (uint64_t)(a_lo + (uint32_t)q * 16u), ((uint64_t)kDescHiB << 32) | (uint64_t)(b_lo + (uint32_t)q * bstep),
                             p.idesc, (q == 0 && first) ? 0u : 1u);
              }
              tc_commit(&b_empty[b_stage]);
              // the oldest piece of this tile (filter row kh-(J-1)) is done; after the group's last row so are the J-1 others
              tc_commit(&w_empty[S - 1 - (int)(n_old % (uint32_t)S)]);
              if (kh == r_last)
                for (int jj = p.J - 2; jj >= 0; --jj) tc_commit(&w_empty[S - 1 - (int)((n_piece - (uint32_t)jj) % (uint32_t)S)]);
            }
            __syncwarp();
            first = 0;
            if (++b_stage == NB) { b_stage = 0; b_phase ^= 1; }
          }
        }
        if (elect_one_sync()) tc_commit(&acc_full[buf]);
        __syncwarp();
      }
    }
  } else {
    epilogue_role<false>(p, tmem_base, epi_smem, acc_full, acc_empty, u_begin, u_end, u_first_real);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

// ------------------------------------------------------------------------------------------ helpers
static inline int j_blocks(int Cout) { return Cout >= 128 ? 1 : 128 / Cout; }
static inline int mmas_per_row(int NC, int KW) { return (NC / 2) * KW + ((NC & 1) ? (KW + 1) / 2 : 0); }

static inline uint16_t f32_to_f16_rne(float f) {
  uint32_t x;
  memcpy(&x, &f, 4);
  const uint32_t sign = (x >> 16) & 0x8000u;
  const int32_t exp = (int32_t)((x >> 23) & 0xff) - 127 + 15;
  uint32_t man = x & 0x7fffffu;
  if (((x >> 23) & 0xff) == 0xff) return (uint16_t)(sign | 0x7c00u | (man ? 0x200u : 0));
  if (exp >= 31) return (uint16_t)(sign | 0x7c00u);
  if (exp <= 0) {
    if (exp < -10) return (uint16_t)sign;
    man |= 0x800000u;
    const int shift = 14 - exp;
    uint32_t h = man >> shift;
    const uint32_t rem = man & ((1u << shift) - 1), halfway = 1u << (shift - 1);
    if (rem > halfway || (rem == halfway && (h & 1))) ++h;
    return (uint16_t)(sign | h);
  }
  uint32_t h = ((uint32_t)exp << 10) | (man >> 13);
  const uint32_t rem = man & 0x1fffu;
  if (rem > 0x1000u || (rem == 0x1000u && (h & 1))) ++h;
  return (uint16_t)(sign | h);
}

static inline float f16_to_f32(uint16_t h) {
  const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
  const int exp = (h >> 10) & 0x1f;
  const uint32_t man = h & 0x3ffu;
  float f;
  if (exp == 0) {
    f = ldexpf((float)man, -24);
  } else if (exp == 31) {
    uint32_t u = 0x7f800000u | (man << 13);
    memcpy(&f, &u, 4);
  } else {
    uint32_t u = ((uint32_t)(exp - 15 + 127) << 23) | (man << 13);
    memcpy(&f, &u, 4);
  }
  uint32_t u;
  memcpy(&u, &f, 4);
  u |= sign;
  memcpy(&f, &u, 4);
  return f;
}

static inline uint16_t f32_to_bf16_rne(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}

// (f, t, ck, b) of a flat element index over [b][ck][t][f]: 32-bit divisions when the tensor has < 2^31 elements (always, in practice) —
// the three 64-bit divisions cost ~300 instructions per 16-byte pixel and bound the element-wise U-Net kernels
__device__ __forceinline__ void decode_ftcb(long long i, bool small, int Fd, int Td, int NCk, int& f, int& t, int& ck, long long& b) {
  if (small) {
    unsigned u = (unsigned)i;
    const unsigned q1 = u / (unsigned)Fd;
    f = (int)(u - q1 * (unsigned)Fd);
    const unsigned q2 = q1 / (unsigned)Td;
    t = (int)(q1 - q2 * (unsigned)Td);
    const unsigned q3 = q2 / (unsigned)NCk;
    ck = (int)(q2 - q3 * (unsigned)NCk);
    b = (long long)q3;
  } else {
    f = (int)(i % Fd);
    long long r = i / Fd;
    t = (int)(r % Td);
    r /= Td;
    ck = (int)(r % NCk);
    b = r / NCk;
  }
}

// CP8 <-> NCHW converters ------------------------------------------------------------------------------
__global__ void nchw_to_cp8_kernel(const float* __restrict__ x, uint16_t* __restrict__ out, long long total, int C, int T,
                                   int F, int NCk, int NCs, int TP, int P, int pf, int pt, int fmt) {
  // one thread per (b, chunk, t, f): gathers 8 channels -> one 16-byte store
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, F, T, NCk, f, t, ck, b);
    __align__(16) uint16_t v[8];
    if (fmt == MPA_FMT_F16X3) {
      __align__(16) uint16_t lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        int c = ck * 8 + e;
        const float xv = c < C ? x[(((size_t)b * C + c) * T + t) * F + f] : 0.f;
        v[e] = split16(xv, 0);
        lo[e] = split16(xv, 1);
      }
      *reinterpret_cast<uint4*>(out + ((((size_t)b * NCs + ck) * TP + pt + t) * P + pf + f) * 8) = *reinterpret_cast<uint4*>(v);
      *reinterpret_cast<uint4*>(out + ((((size_t)b * NCs + NCs / 2 + ck) * TP + pt + t) * P + pf + f) * 8) = *reinterpret_cast<uint4*>(lo);
      continue;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      int c = ck * 8 + e;
      v[e] = cvt16(c < C ? x[(((size_t)b * C + c) * T + t) * F + f] : 0.f, fmt);
    }
    *reinterpret_cast<uint4*>(out + ((((size_t)b * NCs + ck) * TP + pt + t) * P + pf + f) * 8) = *reinterpret_cast<uint4*>(v);
  }
}

// x [B][C][T][Fs] -> CP8 planes of width F: source column f lands on column offset + f*stride (every other real column keeps the
// zero it was initialised with): the zero-inserted gradient of a stride-(1,s) convolution evaluated as a sub-sampled stride-1 one.
// MPA_FMT_F16X3 writes the hi plane and, NCs/2 chunks further, the lo plane of each chunk.
__global__ void nchw_to_cp8_strided_kernel(const float* __restrict__ x, uint16_t* __restrict__ out, long long total, int C, int T, int Fs, int NCk,
                                           int NCs, int TP, int P, int pf, int pt, int fmt, int stride, int offset) {
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, Fs, T, NCk, f, t, ck, b);
    const long long col = pf + offset + (long long)f * stride;
    __align__(16) uint16_t v[8];
    if (fmt == MPA_FMT_F16X3) {
      __align__(16) uint16_t lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int c = ck * 8 + e;
        const float xv = c < C ? x[(((size_t)b * C + c) * T + t) * Fs + f] : 0.f;
        v[e] = split16(xv, 0);
        lo[e] = split16(xv, 1);
      }
      *reinterpret_cast<uint4*>(out + ((((size_t)b * NCs + ck) * TP + pt + t) * P + col) * 8) = *reinterpret_cast<uint4*>(v);
      *reinterpret_cast<uint4*>(out + ((((size_t)b * NCs + NCs / 2 + ck) * TP + pt + t) * P + col) * 8) = *reinterpret_cast<uint4*>(lo);
      continue;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      int c = ck * 8 + e;
      v[e] = cvt16(c < C ? x[(((size_t)b * C + c) * T + t) * Fs + f] : 0.f, fmt);
    }
    *reinterpret_cast<uint4*>(out + ((((size_t)b * NCs + ck) * TP + pt + t) * P + col) * 8) = *reinterpret_cast<uint4*>(v);
  }
}

// one thread per (b, chunk, t, f): one 16-byte load -> 8 channel planes (each store coalesced across the threads of a row)
__global__ void cp8_to_nchw_kernel(const uint16_t* __restrict__ in, float* __restrict__ out, long long total, int C, int T,
                                   int F, int NCk, int NCs, int TP, int P, int pf, int pt, int fmt) {
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, F, T, NCk, f, t, ck, b);
    __align__(16) uint16_t v[8];
    *reinterpret_cast<uint4*>(v) = *reinterpret_cast<const uint4*>(in + ((((size_t)b * NCs + ck) * TP + pt + t) * P + pf + f) * 8);
    if (fmt == MPA_FMT_F16X3) {
      float o[8];
      join8(*reinterpret_cast<const uint4*>(v), *reinterpret_cast<const uint4*>(in + ((((size_t)b * NCs + NCs / 2 + ck) * TP + pt + t) * P + pf + f) * 8), o);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int c = ck * 8 + e;
        if (c < C) out[(((size_t)b * C + c) * T + t) * F + f] = o[e];
      }
      continue;
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const int c = ck * 8 + e;
      if (c < C) out[(((size_t)b * C + c) * T + t) * F + f] = cvt32(v[e], fmt);
    }
  }
}

// out = maxpool_time3(y) + res on CP8 planes; one thread per 16-byte pixel-chunk (8 channels)
template <int FMT>
__device__ __forceinline__ void max8(uint4& c, const uint4& a) {
  if (FMT == MPA_FMT_BF16) {
    __nv_bfloat162* cm = reinterpret_cast<__nv_bfloat162*>(&c);
    const __nv_bfloat162* am = reinterpret_cast<const __nv_bfloat162*>(&a);
#pragma unroll
    for (int e = 0; e < 4; ++e) cm[e] = __hmax2(cm[e], am[e]);
  } else {
    __half2* cm = reinterpret_cast<__half2*>(&c);
    const __half2* am = reinterpret_cast<const __half2*>(&a);
#pragma unroll
    for (int e = 0; e < 4; ++e) cm[e] = __hmax2(cm[e], am[e]);
  }
}
template <int FMT>
__device__ __forceinline__ void add8(uint4& c, const uint4& r) {
  if (FMT == MPA_FMT_BF16) {
    __nv_bfloat162* cm = reinterpret_cast<__nv_bfloat162*>(&c);
    const __nv_bfloat162* rm = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 a = __bfloat1622float2(cm[e]), b2 = __bfloat1622float2(rm[e]);
      cm[e] = __floats2bfloat162_rn(a.x + b2.x, a.y + b2.y);
    }
  } else {
    __half2* cm = reinterpret_cast<__half2*>(&c);
    const __half2* rm = reinterpret_cast<const __half2*>(&r);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float2 a = __half22float2(cm[e]), b2 = __half22float2(rm[e]);
      cm[e] = __floats2half2_rn(a.x + b2.x, a.y + b2.y);
    }
  }
}
template <int FMT>
__global__ void pool_time_res_cp8_kernel(const uint4* __restrict__ y, const uint4* __restrict__ res, uint4* __restrict__ out,
                                         long long total, int NCk, int ncs_y, int ncs_res, int ncs_out, int T, int F, int TP, int P, int pf,
                                         int pt, int half) {
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, F, T, NCk, f, t, ck, b);
    const size_t in_plane = ((size_t)b * ncs_y + ck);
    const size_t base = (in_plane * TP + pt + t) * P + pf + f;
    uint4 c = y[base];
    if (half == 1) {
      if (t > 0) max8<FMT>(c, y[base - P]);
      if (t < T - 1) max8<FMT>(c, y[base + P]);
    } else {
      const int lo = max(-half, -t), hi = min(half, T - 1 - t);
      for (int d = lo; d <= hi; ++d)
        if (d != 0) max8<FMT>(c, y[base + (long long)d * P]);
    }
    if (res) add8<FMT>(c, res[((((size_t)b * ncs_res + ck) * TP + pt + t) * P) + pf + f]);
    out[((((size_t)b * ncs_out + ck) * TP + pt + t) * P) + pf + f] = c;
  }
}

// Wide time pools (k = 13 of the head): one thread per (item, chunk, column) walks down the T rows with the last k values in
// registers — one 16-byte load per output instead of k
template <int FMT, int K>
__global__ void pool_time_col_cp8_kernel(const uint4* __restrict__ y, const uint4* __restrict__ res, uint4* __restrict__ out, long long total,
                                         int NCk, int ncs_y, int ncs_res, int ncs_out, int T, int F, int TP, int P, int pf, int pt) {
  constexpr int H = K / 2;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F);
    long long r = i / F;
    const int ck = (int)(r % NCk);
    const long long b = r / NCk;
    const size_t yb = (((size_t)b * ncs_y + ck) * TP + pt) * P + pf + f;
    const size_t ob = (((size_t)b * ncs_out + ck) * TP + pt) * P + pf + f;
    const size_t rb = (((size_t)b * ncs_res + ck) * TP + pt) * P + pf + f;
    uint4 win[K];                                  // win[j] = row t - H + j (rows outside [0,T) hold a copy of a valid row: max-neutral)
    const uint4 first = y[yb];
#pragma unroll
    for (int j = 0; j < K; ++j) {
      const int t = j - H - 1;                     // window of the (virtual) output row -1
      win[j] = (t >= 0 && t < T) ? y[yb + (size_t)t * P] : first;
    }
    for (int t = 0; t < T; ++t) {
#pragma unroll
      for (int j = 0; j < K - 1; ++j) win[j] = win[j + 1];
      const int tn = t + H;
      win[K - 1] = tn < T ? y[yb + (size_t)tn * P] : win[K - 2];
      uint4 c = win[0];
#pragma unroll
      for (int j = 1; j < K; ++j) max8<FMT>(c, win[j]);
      if (res) add8<FMT>(c, res[rb + (size_t)t * P]);
      out[ob + (size_t)t * P] = c;
    }
  }
}

// k = 13, T = 75 (the head's MaxPool((13,1)) on a whole patch): the 13-frame maximum from a doubling table built on the fly — pairs -> fours ->
// eights -> two overlapping eights, 4 packed max operations per frame and chunk instead of 12 plus a 13-register window shift; the 81
// positions are fully unrolled so that the delay lines between the levels are register renaming.  (The column kernel above ran at
// 3.6 TB/s on the Unet:M head, bound by its ~110 instructions per 16-byte pixel.)
template <int FMT>
__global__ void __launch_bounds__(128) pool13_table_cp8_kernel(const uint4* __restrict__ y, const uint4* __restrict__ res, uint4* __restrict__ out,
                                                               long long total, int NCk, int ncs_y, int ncs_res, int ncs_out, int F, int TP, int P,
                                                               int pf, int pt) {
  constexpr int T = 75, H = 6;
  const uint32_t ninf = FMT == MPA_FMT_BF16 ? 0xFF80FF80u : 0xFC00FC00u;
  const uint4 NINF = make_uint4(ninf, ninf, ninf, ninf);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int f = (int)(i % F);
    long long r = i / F;
    const int ck = (int)(r % NCk);
    const long long b = r / NCk;
    const uint4* yp = y + (((size_t)b * ncs_y + ck) * TP + pt) * P + pf + f;
    uint4* op = out + (((size_t)b * ncs_out + ck) * TP + pt) * P + pf + f;
    const uint4* rp = res ? res + (((size_t)b * ncs_res + ck) * TP + pt) * P + pf + f : nullptr;
    uint4 xprev = NINF, a2[3], a4[5], a8[6], xs[6];
#pragma unroll
    for (int j = 0; j < 3; ++j) a2[j] = NINF;
#pragma unroll
    for (int j = 0; j < 5; ++j) a4[j] = NINF;
#pragma unroll
    for (int j = 0; j < 6; ++j) a8[j] = NINF;
#pragma unroll
    for (int p = 0; p < T + H; ++p) {
      if (p % 6 == 0) {
#pragma unroll
        for (int j = 0; j < 6; ++j) xs[j] = p + j < T ? yp[(size_t)(p + j) * P] : NINF;
      }
      const uint4 xp = xs[p % 6];
      // pairs [p-1,p] -> slot (p+2)%3; fours [p-3,p] -> slot (p+2)%5; eights [p-7,p] -> slot (p+5)%6
      a2[(p + 2) % 3] = xprev;
      max8<FMT>(a2[(p + 2) % 3], xp);
      a4[(p + 2) % 5] = a2[p % 3];
      max8<FMT>(a4[(p + 2) % 5], a2[(p + 2) % 3]);
      a8[(p + 5) % 6] = a4[(p + 3) % 5];
      max8<FMT>(a8[(p + 5) % 6], a4[(p + 2) % 5]);
      xprev = xp;
      if (p >= H) {
        uint4 c = a8[p % 6];                       // frames [p-12, p-5] and [p-7, p]: the window of frame p - 6
        max8<FMT>(c, a8[(p + 5) % 6]);
        if (rp) add8<FMT>(c, rp[(size_t)(p - H) * P]);
        op[(size_t)(p - H) * P] = c;
      }
    }
  }
}

// MaxPool2d((2,2)) floor mode between two CP8 geometries
template <int FMT>
__global__ void maxpool2x2_cp8_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, long long total, int NCk, int ncs_in, int ncs_out,
                                      int To, int Fo, int TPi, int Pi, int pfi, int pti, int TPo, int Po, int pfo, int pto) {
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, Fo, To, NCk, f, t, ck, b);
    const size_t ib = ((((size_t)b * ncs_in + ck) * TPi + pti + 2 * t) * Pi) + pfi + 2 * f;
    uint4 c = in[ib];
    max8<FMT>(c, in[ib + 1]);
    max8<FMT>(c, in[ib + Pi]);
    max8<FMT>(c, in[ib + Pi + 1]);
    out[((((size_t)b * ncs_out + ck) * TPo + pto + t) * Po) + pfo + f] = c;
  }
}

// nn.Upsample(x2, bilinear, align_corners=True) + zero pad to (Ts,Fs) (unet_up_concat_padding), written into the chunk range of the
// concat buffer that follows the skip channels
template <int FMT>
__global__ void upsample2x_cp8_kernel(const uint16_t* __restrict__ low, uint16_t* __restrict__ out, long long total, int NCk, int ncs_in,
                                      int ncs_out, int Tl, int Fl, int TPl, int Pl, int pfl, int ptl, int Ts, int Fs, int TPs, int Ps, int pfs,
                                      int pts) {
  const int Tu = 2 * Tl, Fu = 2 * Fl;
  const int top = (Ts - Tu) / 2, left = (Fs - Fu) / 2;
  const float ry = Tu > 1 ? (float)(Tl - 1) / (float)(Tu - 1) : 0.f;
  const float rx = Fu > 1 ? (float)(Fl - 1) / (float)(Fu - 1) : 0.f;
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, Fs, Ts, NCk, f, t, ck, b);
    __align__(16) uint16_t o[8];
    const int tu = t - top, fu = f - left;
    if (tu < 0 || tu >= Tu || fu < 0 || fu >= Fu) {
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = 0;
    } else {
      const float sy = ry * tu, sx = rx * fu;
      const int y0 = (int)sy, x0 = (int)sx;
      const int y1 = min(y0 + 1, Tl - 1), x1 = min(x0 + 1, Fl - 1);
      const float ly = sy - y0, lx = sx - x0;
      const size_t pb = (((size_t)b * ncs_in + ck) * TPl + ptl);
      const uint4 q00 = *reinterpret_cast<const uint4*>(low + ((pb + y0) * Pl + pfl + x0) * 8);
      const uint4 q01 = *reinterpret_cast<const uint4*>(low + ((pb + y0) * Pl + pfl + x1) * 8);
      const uint4 q10 = *reinterpret_cast<const uint4*>(low + ((pb + y1) * Pl + pfl + x0) * 8);
      const uint4 q11 = *reinterpret_cast<const uint4*>(low + ((pb + y1) * Pl + pfl + x1) * 8);
      const uint16_t* a00 = reinterpret_cast<const uint16_t*>(&q00);
      const uint16_t* a01 = reinterpret_cast<const uint16_t*>(&q01);
      const uint16_t* a10 = reinterpret_cast<const uint16_t*>(&q10);
      const uint16_t* a11 = reinterpret_cast<const uint16_t*>(&q11);
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float v = (1.f - ly) * ((1.f - lx) * cvt32(a00[e], FMT) + lx * cvt32(a01[e], FMT)) +
                        ly * ((1.f - lx) * cvt32(a10[e], FMT) + lx * cvt32(a11[e], FMT));
        o[e] = cvt16(v, FMT);
      }
    }
    *reinterpret_cast<uint4*>(out + (((((size_t)b * ncs_out + ck) * TPs + pts + t) * Ps) + pfs + f) * 8) = *reinterpret_cast<const uint4*>(o);
  }
}

// ---- split-precision (MPA_FMT_F16X3) forms of the element-wise CP8 kernels: values are joined to fp32 (exact), processed in fp32 and
// re-split; the lo planes of a buffer with `ncs` chunk planes per item start at chunk ncs/2
struct X3Plane {
  const uint4* p;
  size_t lo;     // distance (in 16-byte pixels) from a hi pixel to its lo pixel
  __device__ __forceinline__ void load(size_t i, float* v) const { join8(p[i], p[i + lo], v); }
};
__device__ __forceinline__ void x3_store(uint4* p, size_t lo, size_t i, const float* v) {
  uint4 h, l;
  split8(v, h, l);
  p[i] = h;
  p[i + lo] = l;
}
__global__ void pool_time_res_x3_kernel(const uint4* __restrict__ y, const uint4* __restrict__ res, uint4* __restrict__ out, long long total, int NCk,
                                        int ncs_y, int ncs_res, int ncs_out, int T, int F, int TP, int P, int pf, int pt, int half) {
  const size_t plane = (size_t)TP * P;
  const X3Plane Y{y, (size_t)(ncs_y / 2) * plane}, R{res, (size_t)(ncs_res / 2) * plane};
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, F, T, NCk, f, t, ck, b);
    const size_t base = (((size_t)b * ncs_y + ck) * TP + pt + t) * P + pf + f;
    float c[8], o[8];
    Y.load(base, c);
    const int lo = max(-half, -t), hi = min(half, T - 1 - t);
    for (int d = lo; d <= hi; ++d)
      if (d != 0) {
        Y.load(base + (long long)d * P, o);
#pragma unroll
        for (int e = 0; e < 8; ++e) c[e] = fmaxf(c[e], o[e]);
      }
    if (res) {
      R.load((((size_t)b * ncs_res + ck) * TP + pt + t) * P + pf + f, o);
#pragma unroll
      for (int e = 0; e < 8; ++e) c[e] += o[e];
    }
    x3_store(out, (size_t)(ncs_out / 2) * plane, (((size_t)b * ncs_out + ck) * TP + pt + t) * P + pf + f, c);
  }
}
__global__ void maxpool2x2_x3_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, long long total, int NCk, int ncs_in, int ncs_out, int To,
                                     int Fo, int TPi, int Pi, int pfi, int pti, int TPo, int Po, int pfo, int pto) {
  const X3Plane I{in, (size_t)(ncs_in / 2) * TPi * Pi};
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, Fo, To, NCk, f, t, ck, b);
    const size_t ib = ((((size_t)b * ncs_in + ck) * TPi + pti + 2 * t) * Pi) + pfi + 2 * f;
    float c[8], o[8];
    I.load(ib, c);
    const size_t nb[3] = {ib + 1, ib + (size_t)Pi, ib + (size_t)Pi + 1};
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      I.load(nb[k], o);
#pragma unroll
      for (int e = 0; e < 8; ++e) c[e] = fmaxf(c[e], o[e]);
    }
    x3_store(out, (size_t)(ncs_out / 2) * TPo * Po, ((((size_t)b * ncs_out + ck) * TPo + pto + t) * Po) + pfo + f, c);
  }
}
__global__ void upsample2x_x3_kernel(const uint4* __restrict__ low, uint4* __restrict__ out, long long total, int NCk, int ncs_in, int ncs_out, int Tl,
                                     int Fl, int TPl, int Pl, int pfl, int ptl, int Ts, int Fs, int TPs, int Ps, int pfs, int pts) {
  const int Tu = 2 * Tl, Fu = 2 * Fl;
  const int top = (Ts - Tu) / 2, left = (Fs - Fu) / 2;
  const float ry = Tu > 1 ? (float)(Tl - 1) / (float)(Tu - 1) : 0.f;
  const float rx = Fu > 1 ? (float)(Fl - 1) / (float)(Fu - 1) : 0.f;
  const X3Plane L{low, (size_t)(ncs_in / 2) * TPl * Pl};
  const bool small = total < (1ll << 31);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int f, t, ck;
    long long b;
    decode_ftcb(i, small, Fs, Ts, NCk, f, t, ck, b);
    float o[8];
    const int tu = t - top, fu = f - left;
    if (tu < 0 || tu >= Tu || fu < 0 || fu >= Fu) {
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = 0.f;
    } else {
      const float sy = ry * tu, sx = rx * fu;
      const int y0 = (int)sy, x0 = (int)sx;
      const int y1 = min(y0 + 1, Tl - 1), x1 = min(x0 + 1, Fl - 1);
      const float ly = sy - y0, lx = sx - x0;
      const size_t pb = (((size_t)b * ncs_in + ck) * TPl + ptl);
      float a00[8], a01[8], a10[8], a11[8];
      L.load((pb + y0) * Pl + pfl + x0, a00);
      L.load((pb + y0) * Pl + pfl + x1, a01);
      L.load((pb + y1) * Pl + pfl + x0, a10);
      L.load((pb + y1) * Pl + pfl + x1, a11);
#pragma unroll
      for (int e = 0; e < 8; ++e) o[e] = (1.f - ly) * ((1.f - lx) * a00[e] + lx * a01[e]) + ly * ((1.f - lx) * a10[e] + lx * a11[e]);
    }
    x3_store(out, (size_t)(ncs_out / 2) * TPs * Ps, ((((size_t)b * ncs_out + ck) * TPs + pts + t) * Ps) + pfs + f, o);
  }
}

// Device-side packing of the A-operand tiles (same layout as mpa_conv_tc_pack_weights) for the training path, where the weights
// change every step.  transpose_flip: pack the DATA-GRADIENT convolution w'[co'][ci'][kh][kw] = w[ci'][co'][KH-1-kh][KW-1-kw].
__device__ __forceinline__ void pack_weights_range(const float* __restrict__ w, uint16_t* __restrict__ out, long long total, int Cin, int Cout,
                                                   int KH, int KW, int J, int NC, int mpr, int fmt, int transpose_flip, int Cout_total, int co0,
                                                   long long first, long long step, int split = 0, int C0 = 0,
                                                   const float* __restrict__ inv = nullptr) {
  // MPA_FMT_F16X3 (inv = the 128 inverse channel scales already written by pack_scales_range): the layout of mpa_conv_tc_pack_weights, three
  // tile passes per filter row (W_hi, W_lo, W_hi) of the scaled weights
  // one thread per 16-byte group = the 8 input channels of one (tile row, K slice): the position is decoded once per group and the group
  // leaves as one 16-byte store; the all-zero groups of the shifted row blocks (j >= J, filter row outside [0, KH)) touch no weight.
  // (One thread per 16-bit element: 134 us per SAUnet:L training step for ~25 M elements, bound by the index arithmetic.)
  // first / step / total are in elements; groups never straddle a caller's range (all are multiples of 8).
  const int n_paired = (NC / 2) * KW;
  const long long total8 = total >> 3, step8 = step;       // thread i of the caller's step handles groups first/8 + i, + step, ...
  for (long long g = first; g < total8; g += step8) {
    const int mrow = (int)(g & 127);
    const int kc = (int)((g >> 7) & 1);
    const long long tile = g >> 8;
    const int q = (int)(tile % mpr), r = (int)(tile / mpr);
    int df, c;
    if (q < n_paired) {
      const int cp = q / KW;
      df = q - cp * KW;
      c = 2 * cp + kc;
    } else {
      df = 2 * (q - n_paired) + kc;
      c = NC - 1;
    }
    const int j = mrow / Cout, co = mrow - j * Cout;
    const int kh = r - j;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = 0.f;
    if (split) {
      // phase-split form of a KH x split / stride (1, split) convolution with real weights w[Cout][C0][KH][split]: logical input channel
      // ph * C0p + c = (tap ph, real channel c), one tap column.  Forward: Cin = split * C0p;  data gradient (transpose_flip): the logical
      // OUTPUT channels are the split ones (Cout_total = split * C0p), rows flipped, the column tap is the phase itself
      if (df < 1 && j < J && kh >= 0 && kh < KH) {
        if (!transpose_flip) {
          const int C0p = Cin / split;
          if (co0 + co < Cout_total) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int ci = c * 8 + e, ph = ci / C0p, c0r = ci - ph * C0p;
              if (ci < Cin && c0r < C0) v[e] = w[(((size_t)(co0 + co) * C0 + c0r) * KH + kh) * split + ph];
            }
          }
        } else {
          const int C0p = Cout_total / split, o = co0 + co, ph = o / C0p, c0r = o - ph * C0p;
          if (o < Cout_total && c0r < C0) {
#pragma unroll
            for (int e = 0; e < 8; ++e) {
              const int ci = c * 8 + e;
              if (ci < Cin) v[e] = w[(((size_t)ci * C0 + c0r) * KH + (KH - 1 - kh)) * split + ph];
            }
          }
        }
      }
    } else if (df < KW && j < J && kh >= 0 && kh < KH && co0 + co < Cout_total) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int ci = c * 8 + e;
        if (ci < Cin)
          v[e] = transpose_flip ? w[(((size_t)ci * Cout_total + co0 + co) * KH + (KH - 1 - kh)) * KW + (KW - 1 - df)]
                                : w[(((size_t)(co0 + co) * Cin + ci) * KH + kh) * KW + df];
      }
    }
    uint32_t h[4];
    if (fmt == MPA_FMT_F16X3) {
      const float sc = 1.f / inv[co];                   // a power of two: exact
      uint32_t l[4];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float ws = __fmul_rn(v[e], sc);
        const __half hi = __float2half_rn(ws);
        const uint32_t hb = __half_as_ushort(hi), lb = __half_as_ushort(__float2half_rn(__fsub_rn(ws, __half2float(hi))));
        if (e & 1) { h[e >> 1] |= hb << 16; l[e >> 1] |= lb << 16; }
        else { h[e >> 1] = hb; l[e >> 1] = lb; }
      }
      const long long g3 = (tile / mpr * 3 * mpr + q) * 256 + (g & 255), pass = (long long)mpr * 256;
      *reinterpret_cast<uint4*>(out + g3 * 8) = make_uint4(h[0], h[1], h[2], h[3]);
      *reinterpret_cast<uint4*>(out + (g3 + pass) * 8) = make_uint4(l[0], l[1], l[2], l[3]);
      *reinterpret_cast<uint4*>(out + (g3 + 2 * pass) * 8) = make_uint4(h[0], h[1], h[2], h[3]);
      continue;
    }
#pragma unroll
    for (int e = 0; e < 4; ++e) h[e] = (uint32_t)cvt16(v[2 * e], fmt) | ((uint32_t)cvt16(v[2 * e + 1], fmt) << 16);
    *reinterpret_cast<uint4*>(out + g * 8) = make_uint4(h[0], h[1], h[2], h[3]);
  }
}
// MPA_FMT_F16X3: the per-packed-channel inverse scales of mpa_conv_tc_pack_weights (max |w| of the channel's row scaled into [256, 512) by a
// power of two, exponent clamped to +-60; 1 for empty and padded channels), one warp per channel, written after the three tile passes.
// transpose_flip: the packed channel co0 + co is the forward weight's input channel; its row runs over the Cin forward output channels.
__device__ __forceinline__ void pack_scales_range(const float* __restrict__ w, float* __restrict__ inv, int Cin, int Cout, int KH, int KW,
                                                  int transpose_flip, int Cout_total, int co0, int warp, int n_warps) {
  const int lane = threadIdx.x & 31, K2 = KH * KW;
  for (int co = warp; co < 128; co += n_warps) {
    float m = 0.f;
    if (co < Cout && co0 + co < Cout_total)
      for (int i = lane; i < Cin * K2; i += 32) {
        const int ci = i / K2, k = i - ci * K2;
        m = fmaxf(m, fabsf(transpose_flip ? w[((size_t)ci * Cout_total + co0 + co) * K2 + k] : w[((size_t)(co0 + co) * Cin + ci) * K2 + k]));
      }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    int e = 0;
    if (m > 0.f && m < 3.0e38f) {
      frexpf(m, &e);
      e = 9 - e;
      e = e > 60 ? 60 : (e < -60 ? -60 : e);
    }
    if (lane == 0) inv[co] = ldexpf(1.f, -e);
  }
}
__global__ void pack_scales_kernel(const float* __restrict__ w, float* __restrict__ inv, int Cin, int Cout, int KH, int KW, int transpose_flip,
                                   int Cout_total, int co0) {
  pack_scales_range(w, inv, Cin, Cout, KH, KW, transpose_flip, Cout_total, co0, (blockIdx.x * blockDim.x + threadIdx.x) >> 5,
                    (gridDim.x * blockDim.x) >> 5);
}
__global__ void pack_weights_kernel(const float* __restrict__ w, uint16_t* __restrict__ out, long long total, int Cin, int Cout, int KH, int KW,
                                    int J, int NC, int mpr, int fmt, int transpose_flip, int Cout_total, int co0, int split, int C0) {
  pack_weights_range(w, out, total, Cin, Cout, KH, KW, J, NC, mpr, fmt, transpose_flip, Cout_total, co0,
                     blockIdx.x * (long long)blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x, split, C0,
                     fmt == MPA_FMT_F16X3 ? reinterpret_cast<const float*>(out + 3 * total) : nullptr);
}
// Every packed operand of a training step (forward and data-gradient tiles of all convolutions) in ONE launch: blockIdx.y = job of a
// device-resident table (the step's 39 separate 7-us launches were 3.6 % of the SAUnet:L step)
struct PackJobDev {
  const float* w;
  uint16_t* out;
  long long total;
  int Cin, Cout, KH, KW, J, NC, mpr, fmt, transpose_flip, Cout_total, co0;
  int block0;              // first block of this job in the flattened grid (2048 elements per block)
  int split, C0;
};
constexpr int kPackPerBlock = 2048;
__global__ void __launch_bounds__(256) pack_weights_multi_kernel(const PackJobDev* __restrict__ jobs, int n_jobs) {
  __shared__ int job;
  if (threadIdx.x == 0) {
    // last job whose first block is <= blockIdx.x (block0 ascending): bisection — the linear scan was a chain of up to n_jobs dependent loads
    // in front of every block's work
    int lo = 0, hi = n_jobs - 1;
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if ((int)blockIdx.x >= jobs[mid].block0) lo = mid;
      else hi = mid - 1;
    }
    job = lo;
  }
  __syncthreads();
  const PackJobDev j = jobs[job];
  const long long first = (long long)((int)blockIdx.x - j.block0) * kPackPerBlock;
  const long long last = first + kPackPerBlock < j.total ? first + kPackPerBlock : j.total;
  pack_weights_range(j.w, j.out, last, j.Cin, j.Cout, j.KH, j.KW, j.J, j.NC, j.mpr, j.fmt, j.transpose_flip, j.Cout_total, j.co0,
                     (first >> 3) + threadIdx.x, 256, j.split, j.C0,       // 2048 elements per block = one 16-byte group per thread
                     j.fmt == MPA_FMT_F16X3 ? reinterpret_cast<const float*>(j.out + 3 * j.total) : nullptr);
}
// the scales of every MPA_FMT_F16X3 job of a table (blockIdx.y = job; the other jobs return at once), launched before pack_weights_multi_kernel
__global__ void __launch_bounds__(256) pack_scales_multi_kernel(const PackJobDev* __restrict__ jobs) {
  const PackJobDev& j = jobs[blockIdx.y];
  if (j.fmt != MPA_FMT_F16X3) return;
  pack_scales_range(j.w, reinterpret_cast<float*>(j.out + 3 * j.total), j.Cin, j.Cout, j.KH, j.KW, j.transpose_flip, j.Cout_total, j.co0,
                    (blockIdx.x * blockDim.x + threadIdx.x) >> 5, (gridDim.x * blockDim.x) >> 5);
}

static inline int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  long long cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

}  // namespace mpa

using namespace mpa;

extern "C" {

size_t mpa_conv_tc_packed_bytes(int Cin, int Cout, int KH, int KW, int J) {
  if (Cin <= 0 || Cout <= 0 || Cout > 128 || KH <= 0 || KW <= 0 || J < 0 || J * Cout > 128) return 0;
  const int NC = (Cin + 7) / 8;
  if (J == 0) J = j_blocks(Cout);
  return (size_t)(KH + J - 1) * mmas_per_row(NC, KW) * kATileBytes;
}

/* MPA_FMT_F16X3: three tile passes per K row (W_hi, W_lo, W_hi) + 128 floats of per-output-channel inverse scales */
size_t mpa_conv_tc_packed_bytes_fmt(int Cin, int Cout, int KH, int KW, int J, int fmt) {
  const size_t n = mpa_conv_tc_packed_bytes(Cin, Cout, KH, KW, J);
  return (fmt == MPA_FMT_F16X3 && n) ? 3 * n + 128 * sizeof(float) : n;
}

int mpa_conv_tc_pack_weights(const float* w, void* packed, int Cin, int Cout, int KH, int KW, int fmt, int J) {
  MPA_REQUIRE(w && packed && Cin > 0 && Cout > 0 && Cout <= 128 && KH > 0 && KW > 0, "conv_tc_pack_weights: bad argument (Cout must be <= 128)");
  MPA_REQUIRE(J >= 0 && J * Cout <= 128, "conv_tc_pack_weights: J*Cout must be <= 128");
  if (J == 0) J = j_blocks(Cout);
  const int NC = (Cin + 7) / 8, mpr = mmas_per_row(NC, KW);
  const int n_paired = (NC / 2) * KW;
  uint16_t* o = (uint16_t*)packed;
  const bool x3 = fmt == MPA_FMT_F16X3;
  memset(o, 0, mpa_conv_tc_packed_bytes_fmt(Cin, Cout, KH, KW, J, fmt));
  std::vector<float> scale(Cout, 1.f);
  if (x3) {
    // per-output-channel power-of-two scale: max |w| lands in [256, 512), so that the low halves of all but the tiniest weights are
    // normal fp16 numbers; the epilogue multiplies by the (exact) inverse
    float* inv = (float*)((uint8_t*)packed + 3 * mpa_conv_tc_packed_bytes(Cin, Cout, KH, KW, J));
    for (int co = 0; co < Cout; ++co) {
      float m = 0.f;
      for (size_t i = 0; i < (size_t)Cin * KH * KW; ++i) m = fmaxf(m, fabsf(w[(size_t)co * Cin * KH * KW + i]));
      int e = 0;
      if (m > 0.f && m < 3.0e38f) {
        frexpf(m, &e);               // m = f * 2^e, f in [0.5, 1)
        e = 9 - e;                   // m * 2^e in [256, 512)
        if (e > 60) e = 60;
        if (e < -60) e = -60;
      }
      scale[co] = ldexpf(1.f, e);
      inv[co] = ldexpf(1.f, -e);
    }
    for (int co = Cout; co < 128; ++co) inv[co] = 1.f;
  }
  const int tpr = x3 ? 3 * mpr : mpr;
  for (int r = 0; r < KH + J - 1; ++r) {
    for (int q = 0; q < mpr; ++q) {
      uint16_t* tile = o + ((size_t)r * tpr + q) * (kATileBytes / 2);
      uint16_t* tile_lo = tile + (size_t)mpr * (kATileBytes / 2);          // x3: the W_lo pass, then the second W_hi pass
      uint16_t* tile_hi2 = tile + (size_t)2 * mpr * (kATileBytes / 2);
      for (int kc = 0; kc < 2; ++kc) {
        int df, c;
        if (q < n_paired) {
          int cp = q / KW;
          df = q - cp * KW;
          c = 2 * cp + kc;
        } else {
          df = 2 * (q - n_paired) + kc;
          c = NC - 1;
        }
        if (df >= KW) continue;     // dummy half of the last odd-chunk MMA
        for (int j = 0; j < J; ++j) {
          const int kh = r - j;
          if (kh < 0 || kh >= KH) continue;
          for (int co = 0; co < Cout; ++co) {
            const int mrow = j * Cout + co;
            for (int e = 0; e < 8; ++e) {
              const int ci = c * 8 + e;
              if (ci >= Cin) continue;
              const float wv = w[(((size_t)co * Cin + ci) * KH + kh) * KW + df];
              const size_t at = ((size_t)kc * 128 + mrow) * 8 + e;
              if (x3) {
                const float ws = wv * scale[co];
                const uint16_t hi = f32_to_f16_rne(ws);
                tile[at] = tile_hi2[at] = hi;
                tile_lo[at] = f32_to_f16_rne(ws - f16_to_f32(hi));
              } else {
                tile[at] = fmt == MPA_FMT_BF16 ? f32_to_bf16_rne(wv) : f32_to_f16_rne(wv);
              }
            }
          }
        }
      }
    }
  }
  return MPA_OK;
}

int mpa_conv_tc_pack_weights_split_dev(const float* w_dev, void* packed_dev, int Cin, int Cout, int KH, int KW, int fmt, int J, int transpose_flip,
                                       int Cout_total, int co0, int split, int C0, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(w_dev && packed_dev && Cin > 0 && Cout > 0 && Cout <= 128 && KH > 0 && KW > 0, "conv_tc_pack_weights_dev: bad argument (Cout <= 128 per block)");
  MPA_REQUIRE(J >= 0 && J * Cout <= 128 && co0 >= 0 && co0 < Cout_total, "conv_tc_pack_weights_dev: bad J / channel block");
  MPA_REQUIRE(split == 0 || (split > 1 && KW == 1 && C0 > 0 && (transpose_flip ? Cout_total : Cin) % split == 0),
              "conv_tc_pack_weights_dev: bad phase split (KW must be 1, the split channel count a multiple of split)");
  MPA_REQUIRE(fmt == MPA_FMT_F16 || fmt == MPA_FMT_BF16 || (fmt == MPA_FMT_F16X3 && split == 0),
              "conv_tc_pack_weights_dev: fmt must be MPA_FMT_F16, MPA_FMT_BF16 or MPA_FMT_F16X3 (no phase-split form)");
  if (J == 0) J = j_blocks(Cout);
  const int NC = (Cin + 7) / 8, mpr = mmas_per_row(NC, KW);
  const long long total = (long long)(KH + J - 1) * mpr * (kATileBytes / 2);
  if (fmt == MPA_FMT_F16X3) {
    pack_scales_kernel<<<16, 256, 0, (cudaStream_t)stream>>>(w_dev, reinterpret_cast<float*>((uint16_t*)packed_dev + 3 * total), Cin, Cout, KH, KW,
                                                             transpose_flip, Cout_total, co0);
    MPA_CHECK_LAUNCH("conv_tc_pack_weights_dev (scales)");
  }
  pack_weights_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(w_dev, (uint16_t*)packed_dev, total, Cin, Cout, KH, KW, J, NC, mpr, fmt,
                                                                              transpose_flip, Cout_total, co0, split, C0);
  MPA_CHECK_LAUNCH("conv_tc_pack_weights_dev");
  return MPA_OK;
}

int mpa_conv_tc_pack_weights_dev(const float* w_dev, void* packed_dev, int Cin, int Cout, int KH, int KW, int fmt, int J, int transpose_flip,
                                 int Cout_total, int co0, void* stream) {
  return mpa_conv_tc_pack_weights_split_dev(w_dev, packed_dev, Cin, Cout, KH, KW, fmt, J, transpose_flip, Cout_total, co0, 0, 0, stream);
}

size_t mpa_conv_tc_pack_table_bytes(int n_jobs) { return n_jobs > 0 ? (size_t)n_jobs * sizeof(PackJobDev) : 0; }

int mpa_conv_tc_pack_table_build(const mpa_pack_job* jobs, int n_jobs, void* table_host) {
  MPA_REQUIRE(jobs && table_host && n_jobs > 0, "conv_tc_pack_table_build: bad argument");
  PackJobDev* t = (PackJobDev*)table_host;
  int blocks = 0;
  for (int i = 0; i < n_jobs; ++i) {
    const mpa_pack_job& a = jobs[i];
    MPA_REQUIRE(a.w && a.packed && a.Cin > 0 && a.Cout > 0 && a.Cout <= 128 && a.KH > 0 && a.KW > 0 && a.J >= 0 && a.J * a.Cout <= 128 &&
                    a.co0 >= 0 && a.co0 < a.Cout_total &&
                    (a.fmt == MPA_FMT_F16 || a.fmt == MPA_FMT_BF16 || (a.fmt == MPA_FMT_F16X3 && a.split == 0)),
                "conv_tc_pack_table_build: bad job");
    const int J = a.J == 0 ? j_blocks(a.Cout) : a.J, NC = (a.Cin + 7) / 8, mpr = mmas_per_row(NC, a.KW);
    const long long total = (long long)(a.KH + J - 1) * mpr * (kATileBytes / 2);
    MPA_REQUIRE(a.split == 0 || (a.split > 1 && a.KW == 1 && a.C0 > 0 && (a.transpose_flip ? a.Cout_total : a.Cin) % a.split == 0),
                "conv_tc_pack_table_build: bad phase split");
    t[i] = PackJobDev{a.w, (uint16_t*)a.packed, total, a.Cin, a.Cout, a.KH, a.KW, J, NC, mpr, a.fmt, a.transpose_flip, a.Cout_total, a.co0, blocks,
                      a.split, a.C0};
    blocks += (int)((total + kPackPerBlock - 1) / kPackPerBlock);
  }
  return blocks;
}

int mpa_conv_tc_pack_weights_multi(const void* table_dev, int n_jobs, int n_blocks, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(table_dev && n_jobs > 0 && n_blocks > 0, "conv_tc_pack_weights_multi: bad argument");
  pack_weights_multi_kernel<<<n_blocks, 256, 0, (cudaStream_t)stream>>>((const PackJobDev*)table_dev, n_jobs);
  MPA_CHECK_LAUNCH("conv_tc_pack_weights_multi");
  return MPA_OK;
}

int mpa_conv_tc_pack_scales_multi(const void* table_dev, int n_jobs, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(table_dev && n_jobs > 0 && n_jobs <= 65535, "conv_tc_pack_scales_multi: bad argument");
  pack_scales_multi_kernel<<<dim3(16, n_jobs), 256, 0, (cudaStream_t)stream>>>((const PackJobDev*)table_dev);
  MPA_CHECK_LAUNCH("conv_tc_pack_scales_multi");
  return MPA_OK;
}

size_t mpa_conv_tc_ring_packed_bytes(int Cin, int Cout, int KH, int KW, int J) {
  if (Cin <= 0 || Cout <= 0 || Cout > 128 || (Cout & 7) || KH <= 0 || KW <= 0 || KW > 16 || J < 0 || J * Cout > 128) return 0;
  const int NC = (Cin + 7) / 8;
  if (J == 0) J = j_blocks(Cout);
  const size_t n_kh = (size_t)KH + 2 * (J - 1);
  const size_t q_total = (size_t)(NC / 2) * KW + ((NC & 1) ? (KW + 1) / 2 : 0);
  return n_kh * (Cout / 8) * q_total * 256;
}

/* Ring layout (conv_tc_ring_kernel): [group][filter row -(J-1) .. KH-1+(J-1)][row group of 8 channels][q][k-slice][8][8] 16-bit;
 * group g < NC/2: chunks (2g, 2g+1), q = tap; last group when NC is odd: chunk NC-1, q-th MMA = taps (2q, 2q+1).  Filter rows outside
 * [0, KH) are zero pieces (the shifted row blocks of the first / last tiles). */
int mpa_conv_tc_ring_pack_weights(const float* w, void* packed, int Cin, int Cout, int KH, int KW, int fmt, int J) {
  MPA_REQUIRE(w && packed && Cin > 0 && Cout > 0 && Cout <= 128 && (Cout & 7) == 0 && KH > 0 && KW > 0 && KW <= 16,
              "conv_tc_ring_pack_weights: bad argument (Cout multiple of 8, <= 128; KW <= 16)");
  MPA_REQUIRE(J >= 0 && J * Cout <= 128, "conv_tc_ring_pack_weights: J*Cout must be <= 128");
  if (J == 0) J = j_blocks(Cout);
  const int NC = (Cin + 7) / 8, NG = (NC + 1) / 2, G8 = Cout / 8, n_kh = KH + 2 * (J - 1);
  uint16_t* o = (uint16_t*)packed;
  memset(o, 0, mpa_conv_tc_ring_packed_bytes(Cin, Cout, KH, KW, J));
  size_t g_off = 0;   // in 16-bit elements
  for (int g = 0; g < NG; ++g) {
    const bool pair = g < NC / 2;
    const int Q = pair ? KW : (KW + 1) / 2;
    for (int khi = 0; khi < n_kh; ++khi) {
      const int kh = khi - (J - 1);
      if (kh < 0 || kh >= KH) continue;
      for (int g8 = 0; g8 < G8; ++g8)
        for (int q = 0; q < Q; ++q)
          for (int ks = 0; ks < 2; ++ks) {
            const int c = pair ? 2 * g + ks : NC - 1;
            const int df = pair ? q : 2 * q + ks;
            if (df >= KW) continue;
            for (int row = 0; row < 8; ++row) {
              const int co = g8 * 8 + row;
              for (int e = 0; e < 8; ++e) {
                const int ci = c * 8 + e;
                if (ci >= Cin) continue;
                const float wv = w[(((size_t)co * Cin + ci) * KH + kh) * KW + df];
                o[g_off + ((((size_t)khi * G8 + g8) * Q + q) * 2 + ks) * 64 + row * 8 + e] = fmt == MPA_FMT_BF16 ? f32_to_bf16_rne(wv) : f32_to_f16_rne(wv);
              }
            }
          }
    }
    g_off += (size_t)n_kh * G8 * Q * 128;
  }
  return MPA_OK;
}

// smem layout, grid and launch shared by both entry points (p: everything but the smem offsets filled in)
static int launch_conv_tc(ConvTcParams& p, int Cin, cudaStream_t stream, int* grid_out) {
  p.mmas_per_row = mmas_per_row(p.NC, p.KW);
  p.slab_px = (p.N + 2 * (p.KW / 2) + 1 + 7) / 8 * 8;
  if (p.R < 1) p.R = 1;
  if (p.Rs < 1) p.Rs = 1;
  p.tma = 0;
  p.tma_c0 = 0;
  const bool tma_ok = !p.x3 && !p.ring_on && p.in_e == p.T && tensor_map_encoder();      // decided before the stage sizing
  if (tma_ok && (p.Rs > 1 || p.R > 1) && p.KW == 1) {
    p.tma = 1;
    p.slab_px = p.N;                          // dense box: [plane][R rows][pitch] (the pad behind a stage takes the one-pixel over-read)
  } else if (tma_ok && p.R == 1 && p.Rs == 1 && p.NC >= 2 && p.slab_px <= 128) {
    // narrow planes (the deeper U-Net levels): one input row of ALL chunk planes of a stage in one copy.  A stage of a 3x3 / 5x5 / 9x9
    // filter on a <= 64-bin level feeds the tensor pipe for 100-300 clocks — less than two of the NC bulk copies it used to take.
    p.tma = 2;
    p.tma_c0 = -2 * (p.KW / 2);               // the slab starts KW/2 pixels left of column 0 (8-byte elements)
  }
  p.bpad = p.tma ? 128 : 0;
  size_t smem = 0;
  if (p.x3) {
    MPA_REQUIRE(!p.ring_on, "conv_tc: the ring main loop has no split-precision variant");
    MPA_REQUIRE((p.Cout & 7) == 0, "conv_tc(fp16x3): Cout must be a multiple of 8 (got %d)", p.Cout);
    p.inv_scale = (const float*)(p.w + (size_t)3 * (p.KH + p.J - 1) * p.mmas_per_row * kATileBytes);
  }
  if (p.ring_on) {
    const int qmax = p.NC >= 2 ? p.KW : (p.KW + 1) / 2;
    MPA_REQUIRE(p.KW <= 16 && (p.Cout & 7) == 0 && p.NC <= 16, "conv_tc(ring): KW <= 16, Cout %% 8 == 0, Cin <= 128 required");
    p.ring_sbo = qmax * 256;
    p.ring_ps = (p.Cout / 8) * p.ring_sbo;
    p.ring_nb = 4;
    const size_t bstage = 2 * (size_t)p.slab_px * 16;
    const size_t fixed = (size_t)p.ring_nb * bstage + 640 + 512 + 128 + 8 * 32 * kEpiPitch * 2;
    int S = p.J + 4;
    while (S > p.J + 1 && (size_t)(S + p.J - 1) * p.ring_ps + fixed > 227 * 1024) --S;
    MPA_REQUIRE(S >= p.J + 1 && S <= kMaxRingS, "conv_tc(ring): the weight ring does not fit (Cout=%d J=%d)", p.Cout, p.J);
    p.G = p.NC;
    p.n_groups = 1;
    p.ring_S = S;
    p.ring_npos = S + p.J - 1;
    p.ring_b_off = p.ring_npos * p.ring_ps;
    p.ring_bar_off = p.ring_b_off + (int)(p.ring_nb * bstage);
    p.btab_off = p.ring_bar_off + 640;
    size_t off = (size_t)p.btab_off + 512;
    off = (off + 127) / 128 * 128;
    p.epi_off = (int)off;
    smem = off + 8 * 32 * kEpiPitch * 2;
  } else {
    const size_t tail = 256 + (size_t)(p.mmas_per_row + 8) * 4 + 128 + 8 * 32 * kEpiPitch * 2 + (size_t)kMaxBStages * p.bpad;   // barriers, table, staging, stage pads
    // chunks per activation stage: all of them when two stages fit next to >= 2 weight stages, else the largest even group that does
    // (wide-K layers; one group = G/2 * KW consecutive MMAs of the row)
    p.G = p.NC;
    if (!p.x3)
      while (p.G > 2 && (size_t)kNumBStages * p.G * p.slab_px * 16 + 2 * (size_t)kAStageBytes + tail > 227 * 1024) p.G = (p.G - 1) / 2 * 2;
    if (p.G < p.NC && p.G >= 16) p.G = p.G / 16 * 16;      // whole weight stages (8 MMAs) per group when KW == 1
    p.n_groups = (p.NC + p.G - 1) / p.G;
    const size_t b_bytes = (size_t)kNumBStages * p.G * p.slab_px * 16;
    int a_stages = kMaxAStages;
    while (a_stages > 2 && (size_t)a_stages * kAStageBytes + b_bytes + tail > 227 * 1024) --a_stages;
    p.a_stages = a_stages;
    // thin inputs (one or two chunks: the first layer of every model, the 6 -> 20 / 8 -> 8 / 16 -> 16 convolutions): a stage feeds only
    // ~8 MMAs (~450 tensor clocks), so two stages cover less than the latency of a bulk copy that misses L2 (ncu: CNN:XS conv1 forward
    // 67 % tensor-active against 90 % for its 3-chunk data gradient); take as many stages as fit
    int b_stages = kNumBStages;
    const size_t bstage1 = (size_t)p.G * p.slab_px * 16 + p.bpad;
    while (b_stages < kMaxBStages && (size_t)a_stages * kAStageBytes + (size_t)(b_stages + 1) * bstage1 + tail <= 227 * 1024) ++b_stages;
    p.b_stages = b_stages;
    if (p.tma) {
      // global tensor [patch][plane][row 0 .. T-1][pitch * 2 x 8 bytes]; box = one stage
      const cuuint64_t gdim[4] = {(cuuint64_t)p.P * 2, (cuuint64_t)p.T, (cuuint64_t)p.NC, (cuuint64_t)p.n_patches};
      const cuuint64_t gstr[3] = {(cuuint64_t)p.P * 16, (cuuint64_t)p.in_edge_chunk_stride, (cuuint64_t)p.in_edge_patch_stride};
      const cuuint32_t box[4] = {(cuuint32_t)(p.tma == 2 ? p.slab_px * 2 : p.P * 2), (cuuint32_t)((p.R - 1) * p.Rs + 1), (cuuint32_t)p.G, 1u};
      const cuuint32_t estr[4] = {1u, (cuuint32_t)p.Rs, 1u, 1u};
      const CUresult r = tensor_map_encoder()(&p.tmap, CU_TENSOR_MAP_DATA_TYPE_UINT64, 4, const_cast<uint8_t*>(p.in_edge), gdim, gstr, box, estr,
                                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      // not encodable (an unusual geometry): the bulk-copy loops below handle the same stage layout
      if (!(r == CUDA_SUCCESS && box[0] <= 256 && box[1] <= 256 && p.G <= 256)) p.tma = 0;
    }
    p.resident = (!p.x3 && p.n_groups == 1 && (p.KH + p.J - 1) * ((p.mmas_per_row + kStageMMAs - 1) / kStageMMAs) <= a_stages) ? 1 : 0;
    MPA_REQUIRE(p.mmas_per_row <= 128, "conv_tc: too many K steps per row (%d)", p.mmas_per_row);
    p.tiles_per_row = p.x3 ? 3 * p.mmas_per_row : p.mmas_per_row;
    {
      const uint32_t plane = (uint32_t)p.slab_px * 16u;
      const int n_paired = (p.NC / 2) * p.KW;
      for (int q = 0; q < p.mmas_per_row; ++q) {
        uint32_t boff, lbo;
        if (q < n_paired) {
          const int cp = q / p.KW, df = q - cp * p.KW;
          boff = (uint32_t)((2 * cp) % p.G) * plane + (uint32_t)df * 16u;          // offset inside the chunk group's stage
          lbo = plane;
        } else {
          boff = (uint32_t)((p.NC - 1) % p.G) * plane + 2u * (uint32_t)(q - n_paired) * 16u;
          lbo = 16u;
        }
        p.btab[q] = (boff >> 4) | ((lbo >> 4) << 16);
        if (p.x3) p.btab[p.mmas_per_row + q] = p.btab[q];      // the W_lo pass walks the same (hi) slab again
      }
    }
    size_t off = (size_t)a_stages * kAStageBytes + (size_t)b_stages * bstage1;
    p.btab_off = (int)(off + 256);
    off += 256 + (size_t)(p.mmas_per_row + 8) * 4;      // barriers + tmem slot (256 B), descriptor table
    off = (off + 127) / 128 * 128;
    p.epi_off = (int)off;
    smem = off + 8 * 32 * kEpiPitch * 2;
  }
  MPA_REQUIRE(smem <= 227 * 1024, "conv_tc: needs %zu B of shared memory (Cin=%d pitch=%d)", smem, Cin, p.P);
  {
    static unsigned char flags_tile[64], flags_ring[64], flags_x3[64];
    cudaError_t e = p.ring_on ? opt_in_max_smem(conv_tc_ring_kernel, flags_ring)
                    : p.x3    ? opt_in_max_smem(conv_tc_kernel<true>, flags_x3)
                              : opt_in_max_smem(conv_tc_kernel<false>, flags_tile);
    if (e != cudaSuccess) {
      set_error("conv_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return MPA_ERR_CUDA;
    }
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (sms > kMaxGrid) sms = kMaxGrid;
  const int grid = p.n_units < sms ? p.n_units : sms;
  if (grid_out) *grid_out = grid;
  if (p.ring_on)
    conv_tc_ring_kernel<<<grid, kThreads, smem, stream>>>(p);
  else if (p.x3)
    conv_tc_kernel<true><<<grid, kThreads, smem, stream>>>(p);
  else
    conv_tc_kernel<false><<<grid, kThreads, smem, stream>>>(p);
  MPA_CHECK_LAUNCH("conv_tc");
  return MPA_OK;
}

int mpa_conv_tc_f16(const void* in_cp8, const void* w_packed, const float* bias, void* out, int out_mode, int sub_stride,
                    int sub_offset, int n_patches, int Cin, int Cout, int T, int F, int KH, int KW, int pitch, int pf, int pt,
                    long long in_patch_stride_rows, int in_nc_stride, int out_nc_stride, int J, int row0, int n_rows, int act,
                    float act_param, int fmt, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(in_cp8 && w_packed && bias && out && n_patches > 0, "conv_tc: null argument");
  MPA_REQUIRE(Cout > 0 && Cout <= 128 && Cin > 0, "conv_tc: Cout must be in 1..128 (got %d)", Cout);
  MPA_REQUIRE((KH & 1) && (KW & 1), "conv_tc: odd kernel sizes only");
  MPA_REQUIRE(fmt == MPA_FMT_F16 || fmt == MPA_FMT_BF16 || fmt == MPA_FMT_F16X3, "conv_tc: fmt must be MPA_FMT_F16, MPA_FMT_BF16 or MPA_FMT_F16X3");
  const bool x3 = fmt == MPA_FMT_F16X3;
  MPA_REQUIRE(!x3 || in_patch_stride_rows <= 0, "conv_tc(fp16x3): the streaming input goes through mpa_conv_tc_pool_f16");
  const int N = (pitch + 15) / 16 * 16;      // MMA N: one padded image row (columns >= pitch are never stored)
  MPA_REQUIRE(N >= 16 && N <= 256 && (pitch % 16 == 0 || KW == 1), "conv_tc: row pitch %d must be a multiple of 16 (<= 256) unless KW == 1", pitch);
  MPA_REQUIRE(pf >= KW / 2 && pitch - F >= KW / 2 && pitch >= pf + F, "conv_tc: pitch %d / left pad %d too small for F=%d KW=%d", pitch, pf, F, KW);
  MPA_REQUIRE(pt >= 1 || KW == 1, "conv_tc: at least one guard row above and below each plane is required (KW > 1)");
  MPA_REQUIRE(J >= 0 && J * Cout <= 128 && row0 >= 0 && n_rows >= 0 && row0 + n_rows <= T, "conv_tc: bad J / row window");
  MPA_REQUIRE(((uintptr_t)in_cp8 & 15) == 0 && ((uintptr_t)w_packed & 15) == 0 && ((uintptr_t)out & 15) == 0, "conv_tc: 16-byte alignment required");
  MPA_REQUIRE(out_mode == 0 || (out_mode == 1 && sub_stride >= 1 && sub_offset >= 0 && sub_offset < sub_stride) ||
                  (out_mode == 2 && sub_stride >= 2 && sub_offset == 0 && (Cout & 7) == 0 && out_nc_stride > 0 && out_nc_stride % sub_stride == 0),
              "conv_tc: bad output mode");
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  p.w = (const uint8_t*)w_packed;
  p.bias = bias;
  p.out = (uint16_t*)out;
  p.out_mode = out_mode;
  p.sub_stride = out_mode ? sub_stride : 1;
  p.sub_offset = out_mode ? sub_offset : 0;
  p.F_out = out_mode ? (F - p.sub_offset + p.sub_stride - 1) / p.sub_stride : F;
  p.pf2 = 8;
  p.P2 = (p.pf2 + p.F_out + 15) / 16 * 16;
  p.phase_planes = out_mode == 2 ? out_nc_stride / sub_stride / (x3 ? 2 : 1) : 0;
  p.fmt = fmt;
  p.x3 = x3 ? 1 : 0;
  p.n_patches = n_patches;
  p.NC = (Cin + 7) / 8;
  p.Cout = Cout;
  p.J = J > 0 ? J : j_blocks(Cout);
  p.T = T; p.F = F; p.KH = KH; p.KW = KW; p.P = pitch; p.N = N; p.pf = pf;
  p.row0 = row0;
  p.T_out = n_rows > 0 ? n_rows : T - row0;
  p.pt_out = pt;
  p.TP_out = p.T_out + 2 * pt;
  p.NCo = (Cout + 7) / 8;
  const long long TP = T + 2 * pt;
  const uint8_t* in0 = (const uint8_t*)in_cp8 + (long long)pt * pitch * 16;   // (row 0, column 0) of patch 0, chunk 0
  if (in_patch_stride_rows <= 0) {
    // materialised patches: [n_patches][NC][TP][P][8]
    p.in_e = T;
    p.in_edge = in0;
    p.in_edge_chunk_stride = TP * pitch * 16;
    p.in_edge_patch_stride = p.in_edge_chunk_stride * (in_nc_stride > 0 ? in_nc_stride : (x3 ? 2 : 1) * p.NC);
    p.in_lo_off = in_nc_stride > 0 ? in_nc_stride / 2 : p.NC;
  } else {
    // streaming: one shared frame-major plane [rows][P][8]; patch b starts at row b*stride (after pt guard rows)
    MPA_REQUIRE(p.NC == 1, "conv_tc: streaming input supports a single channel chunk");
    p.in_e = 0;
    p.in_stream = in0;
    p.in_stream_chunk_stride = 0;
    p.in_stream_patch_rows = in_patch_stride_rows;
  }
  MPA_REQUIRE(in_nc_stride == 0 || in_nc_stride >= p.NC, "conv_tc: in_nc_stride %d < %d input chunks", in_nc_stride, p.NC);
  MPA_REQUIRE(out_nc_stride == 0 || out_nc_stride >= p.NCo, "conv_tc: out_nc_stride %d < %d output chunks", out_nc_stride, p.NCo);
  MPA_REQUIRE(!x3 || ((in_nc_stride & 1) == 0 && (out_nc_stride & 1) == 0), "conv_tc(fp16x3): chunk strides must be even (hi planes, then lo planes)");
  p.out_lo_off = out_nc_stride > 0 ? out_nc_stride / 2 : p.NCo;
  p.out_patch_stride = (long long)(out_nc_stride > 0 ? out_nc_stride : (x3 ? 2 : 1) * p.NCo) *
                       (out_mode == 0 ? (long long)p.TP_out * pitch : out_mode == 2 ? (long long)p.TP_out * p.P2 : (long long)p.T_out * p.F_out) * 8;
  MPA_REQUIRE(out_mode != 2 || p.phase_planes >= p.NCo, "conv_tc: %d chunk planes per phase < %d output chunks", p.phase_planes, p.NCo);
  // row-merged operand rows (see ConvTcParams::R): KH x 1 filters on materialised patches whose zero guard rows cover the time padding
  p.R = 1;
  p.Rs = 1;
  p.pt_in = pt;
  if (KW == 1 && KH / 2 <= pt && pt >= 1 && in_patch_stride_rows <= 0 && p.J == 1 && !x3 && pitch % 16 == 0 && out_mode != 2) {
    int R = 256 / pitch;
    while (R > 1 && (p.T_out % R)) --R;
    p.R = R;
    p.N = R * pitch;
  } else if (KW == 1 && KH / 2 <= pt && pt >= 1 && in_patch_stride_rows <= 0 && p.J > 1 && !x3 && pitch % 16 == 0 && out_mode != 2 && 256 / pitch >= 2 &&
             p.T_out >= 2 * p.J) {
    p.R = 256 / pitch;
    p.Rs = p.J;
    p.N = p.R * pitch;
  }
  p.n_seg = 1;
  p.y_lo[0] = p.z_lo[0] = row0;
  p.y_hi[0] = p.z_hi[0] = row0 + p.T_out;
  p.seg_groups[0] = (p.T_out + p.J * p.R - 1) / (p.J * p.R);
  p.seg_groups[1] = 0;
  p.groups_per_patch = p.seg_groups[0];
  p.n_units = n_patches * p.groups_per_patch;
  p.act = act;
  p.act_param = act_param;
  const uint32_t f = (fmt == MPA_FMT_BF16) ? 1u : 0u;
  p.idesc = (1u << 4) | (f << 7) | (f << 10) | ((uint32_t)(p.N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  return launch_conv_tc(p, Cin, (cudaStream_t)stream, nullptr);
}

size_t mpa_conv_tc_pool_workspace(int Cout, int pitch, int J) {
  if (Cout <= 0 || Cout > 128 || pitch <= 0) return 0;
  if (J <= 0) J = j_blocks(Cout);
  return (size_t)kMaxGrid * 2 * J * ((Cout + 7) / 8) * pitch * 16;
}

size_t mpa_conv_tc_pool_workspace_fmt(int Cout, int pitch, int J, int fmt) {
  return mpa_conv_tc_pool_workspace(Cout, pitch, J) * (fmt == MPA_FMT_F16X3 ? 2 : 1);
}

int mpa_conv_tc_pool_f16(const mpa_conv_tc_desc* d, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(d && d->w_packed && d->bias && d->workspace && d->n_patches > 0, "conv_tc_pool: null argument");
  MPA_REQUIRE(d->Cout > 0 && d->Cout <= 64 && (d->Cout & 7) == 0 && d->Cin > 0, "conv_tc_pool: Cout must be a multiple of 8, <= 64 (got %d)", d->Cout);
  MPA_REQUIRE((d->KH & 1) && (d->KW & 1), "conv_tc_pool: odd kernel sizes only");
  MPA_REQUIRE(d->fmt == MPA_FMT_F16 || d->fmt == MPA_FMT_BF16 || d->fmt == MPA_FMT_F16X3, "conv_tc_pool: fmt must be MPA_FMT_F16, MPA_FMT_BF16 or MPA_FMT_F16X3");
  const int pitch = d->pitch, KW = d->KW, F = d->F, pf = d->pf, T = d->T;
  MPA_REQUIRE(pitch >= 16 && pitch <= 256 && pitch % 16 == 0, "conv_tc_pool: row pitch %d must be a multiple of 16 (<= 256)", pitch);
  MPA_REQUIRE(pf >= KW / 2 && pitch - F >= KW / 2 && pitch >= pf + F, "conv_tc_pool: pitch %d / left pad %d too small for F=%d KW=%d", pitch, pf, F, KW);
  const int J = d->J > 0 ? d->J : j_blocks(d->Cout);
  MPA_REQUIRE(J >= 2 && J * d->Cout <= 128, "conv_tc_pool: needs 2 <= J and J*Cout <= 128");
  MPA_REQUIRE(d->in_e == T || (d->in_e >= 0 && 2 * d->in_e <= T), "conv_tc_pool: in_e must be T or <= T/2");
  MPA_REQUIRE(d->out_e == T || (d->out_e >= 0 && 2 * d->out_e <= T), "conv_tc_pool: out_e must be T or <= T/2");
  MPA_REQUIRE((d->in_e == 0 || d->in_edge) && (d->in_e == T || d->in_stream), "conv_tc_pool: missing input plane");
  MPA_REQUIRE((d->out_e == 0 || d->out_edge) && (d->out_e == T || d->out_stream), "conv_tc_pool: missing output plane");
  MPA_REQUIRE(d->n_seg == 1 || d->n_seg == 2, "conv_tc_pool: 1 or 2 row segments");
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  p.in_edge = (const uint8_t*)d->in_edge;
  p.in_stream = (const uint8_t*)d->in_stream;
  p.in_edge_patch_stride = d->in_edge_patch_stride;
  p.in_edge_chunk_stride = d->in_edge_chunk_stride;
  p.in_stream_chunk_stride = d->in_stream_chunk_stride;
  p.in_stream_patch_rows = d->in_stream_patch_rows;
  p.in_e = d->in_e;
  p.out_edge = (uint8_t*)d->out_edge;
  p.out_stream = (uint8_t*)d->out_stream;
  p.out_edge_patch_stride = d->out_edge_patch_stride;
  p.out_edge_chunk_stride = d->out_edge_chunk_stride;
  p.out_stream_chunk_stride = d->out_stream_chunk_stride;
  p.out_stream_patch_rows = d->out_stream_patch_rows;
  p.out_e = d->out_e;
  p.out_split = d->out_split;
  MPA_REQUIRE(d->out_split == 0 || (d->out_split >= 2 && d->out_e == T && d->n_seg == 1), "conv_tc_pool: out_split needs a materialised single-segment output");
  p.pf2 = 8;
  p.P2 = d->out_split ? (8 + (F + d->out_split - 1) / d->out_split + 15) / 16 * 16 : 0;
  MPA_REQUIRE((((uintptr_t)p.in_edge | (uintptr_t)p.in_stream | (uintptr_t)p.out_edge | (uintptr_t)p.out_stream | (uintptr_t)d->w_packed |
                (uintptr_t)d->workspace) & 15) == 0, "conv_tc_pool: 16-byte alignment required");
  MPA_REQUIRE(((p.in_edge_patch_stride | p.in_edge_chunk_stride | p.in_stream_chunk_stride | p.out_edge_patch_stride | p.out_edge_chunk_stride |
                p.out_stream_chunk_stride) & 15) == 0, "conv_tc_pool: strides must be multiples of 16 bytes");
  p.pool = 3;
  p.ring_on = d->weights_layout == 1 ? 1 : 0;
  MPA_REQUIRE(d->weights_layout == 0 || d->weights_layout == 1, "conv_tc_pool: weights_layout must be 0 (tiles) or 1 (ring pieces)");
  p.residual = d->residual ? 1 : 0;
  p.w = (const uint8_t*)d->w_packed;
  p.bias = d->bias;
  p.fmt = d->fmt;
  p.x3 = d->fmt == MPA_FMT_F16X3 ? 1 : 0;
  // split precision: the lo planes follow the hi planes of every edge / stream buffer (2*NC chunk planes per row set); a phase-split
  // output holds [part][phase][chunk] planes
  p.in_lo_off = (d->Cin + 7) / 8;
  p.out_lo_off = (d->out_split ? d->out_split : 1) * (d->Cout / 8);
  p.n_patches = d->n_patches;
  p.NC = (d->Cin + 7) / 8;
  p.Cout = d->Cout;
  p.NCo = d->Cout / 8;
  MPA_REQUIRE(!p.residual || p.NC == p.NCo, "conv_tc_pool: the residual needs Cin == Cout");
  p.J = J;
  p.T = T; p.F = F; p.KH = d->KH; p.KW = KW; p.P = pitch; p.N = pitch; p.pf = pf;
  p.sub_stride = 1;
  p.F_out = F;
  p.n_seg = d->n_seg;
  p.groups_per_patch = 0;
  for (int s = 0; s < 2; ++s) {
    if (s >= d->n_seg) { p.seg_groups[s] = 0; continue; }
    MPA_REQUIRE(d->z_lo[s] >= 0 && d->z_lo[s] < d->z_hi[s] && d->z_hi[s] <= T, "conv_tc_pool: bad row segment %d: [%d,%d)", s, d->z_lo[s], d->z_hi[s]);
    p.z_lo[s] = d->z_lo[s];
    p.z_hi[s] = d->z_hi[s];
    p.y_lo[s] = d->z_lo[s] > 0 ? d->z_lo[s] - 1 : 0;
    p.y_hi[s] = d->z_hi[s] < T ? d->z_hi[s] + 1 : T;
    p.seg_groups[s] = (p.y_hi[s] - p.y_lo[s] + J - 1) / J;
    p.groups_per_patch += p.seg_groups[s];
  }
  MPA_REQUIRE(d->n_seg == 1 || p.y_hi[0] <= p.y_lo[1], "conv_tc_pool: row segments overlap");
  p.n_units = d->n_patches * p.groups_per_patch;
  p.ring = (uint8_t*)d->workspace;
  MPA_REQUIRE(d->ws_bytes >= mpa_conv_tc_pool_workspace_fmt(d->Cout, pitch, J, d->fmt), "conv_tc_pool: workspace too small (%zu B)", d->ws_bytes);
  p.act = d->act;
  p.act_param = d->act_param;
  const uint32_t f = (d->fmt == MPA_FMT_BF16) ? 1u : 0u;
  p.idesc = (1u << 4) | (f << 7) | (f << 10) | ((uint32_t)(p.N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  return launch_conv_tc(p, d->Cin, (cudaStream_t)stream, nullptr);
}

int mpa_pool_time_res_cp8(const void* y_cp8, const void* res_cp8, void* out_cp8, int n_patches, int C, int T, int F, int pitch, int pf,
                          int pt, int k, int fmt, int ncs_y, int ncs_res, int ncs_out, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(y_cp8 && out_cp8 && n_patches > 0 && C > 0 && k >= 1 && (k & 1) && pitch >= pf + F, "pool_time_res_cp8: bad argument");
  const int NCk = (C + 7) / 8;
  if (ncs_y <= 0) ncs_y = NCk;
  if (ncs_res <= 0) ncs_res = NCk;
  if (ncs_out <= 0) ncs_out = NCk;
  long long total = (long long)n_patches * NCk * T * F;
  if (fmt == MPA_FMT_F16X3) {
    if (ncs_y == NCk) ncs_y = 2 * NCk;
    if (ncs_res == NCk) ncs_res = 2 * NCk;
    if (ncs_out == NCk) ncs_out = 2 * NCk;
    MPA_REQUIRE(!((ncs_y | ncs_res | ncs_out) & 1), "pool_time_res_cp8(fp16x3): chunk strides must be even");
    pool_time_res_x3_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)y_cp8, (const uint4*)res_cp8, (uint4*)out_cp8, total, NCk,
                                                                                     ncs_y, ncs_res, ncs_out, T, F, T + 2 * pt, pitch, pf, pt, k / 2);
  } else if (k == 13 && T == 75) {
    const long long cols = (long long)n_patches * NCk * F;
    if (fmt == MPA_FMT_BF16)
      pool13_table_cp8_kernel<MPA_FMT_BF16><<<grid_for(cols, 128), 128, 0, (cudaStream_t)stream>>>(
          (const uint4*)y_cp8, (const uint4*)res_cp8, (uint4*)out_cp8, cols, NCk, ncs_y, ncs_res, ncs_out, F, T + 2 * pt, pitch, pf, pt);
    else
      pool13_table_cp8_kernel<MPA_FMT_F16><<<grid_for(cols, 128), 128, 0, (cudaStream_t)stream>>>(
          (const uint4*)y_cp8, (const uint4*)res_cp8, (uint4*)out_cp8, cols, NCk, ncs_y, ncs_res, ncs_out, F, T + 2 * pt, pitch, pf, pt);
  } else if (k == 13 && T >= 13) {
    const long long cols = (long long)n_patches * NCk * F;
    if (fmt == MPA_FMT_BF16)
      pool_time_col_cp8_kernel<MPA_FMT_BF16, 13><<<grid_for(cols, 128), 128, 0, (cudaStream_t)stream>>>(
          (const uint4*)y_cp8, (const uint4*)res_cp8, (uint4*)out_cp8, cols, NCk, ncs_y, ncs_res, ncs_out, T, F, T + 2 * pt, pitch, pf, pt);
    else
      pool_time_col_cp8_kernel<MPA_FMT_F16, 13><<<grid_for(cols, 128), 128, 0, (cudaStream_t)stream>>>(
          (const uint4*)y_cp8, (const uint4*)res_cp8, (uint4*)out_cp8, cols, NCk, ncs_y, ncs_res, ncs_out, T, F, T + 2 * pt, pitch, pf, pt);
  } else if (fmt == MPA_FMT_BF16)
    pool_time_res_cp8_kernel<MPA_FMT_BF16><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)y_cp8, (const uint4*)res_cp8, (uint4*)out_cp8, total, NCk, ncs_y, ncs_res, ncs_out, T, F, T + 2 * pt, pitch, pf, pt, k / 2);
  else
    pool_time_res_cp8_kernel<MPA_FMT_F16><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)y_cp8, (const uint4*)res_cp8, (uint4*)out_cp8, total, NCk, ncs_y, ncs_res, ncs_out, T, F, T + 2 * pt, pitch, pf, pt, k / 2);
  MPA_CHECK_LAUNCH("pool_time_res_cp8");
  return MPA_OK;
}

int mpa_maxpool2x2_cp8(const void* in_cp8, void* out_cp8, int n, int C, int T, int F, int pitch_in, int pf_in, int pt_in, int ncs_in,
                       int pitch_out, int pf_out, int pt_out, int ncs_out, int fmt, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(in_cp8 && out_cp8 && n > 0 && C > 0 && T >= 2 && F >= 2, "maxpool2x2_cp8: bad argument");
  const int NCk = (C + 7) / 8, To = T / 2, Fo = F / 2;
  MPA_REQUIRE(pitch_in >= pf_in + F && pitch_out >= pf_out + Fo, "maxpool2x2_cp8: pitch too small");
  if (ncs_in <= 0) ncs_in = NCk;
  if (ncs_out <= 0) ncs_out = NCk;
  long long total = (long long)n * NCk * To * Fo;
  if (fmt == MPA_FMT_F16X3) {
    if (ncs_in == NCk) ncs_in = 2 * NCk;
    if (ncs_out == NCk) ncs_out = 2 * NCk;
    MPA_REQUIRE(!((ncs_in | ncs_out) & 1), "maxpool2x2_cp8(fp16x3): chunk strides must be even");
    maxpool2x2_x3_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)in_cp8, (uint4*)out_cp8, total, NCk, ncs_in, ncs_out, To, Fo,
                                                                                  T + 2 * pt_in, pitch_in, pf_in, pt_in, To + 2 * pt_out, pitch_out, pf_out, pt_out);
  } else if (fmt == MPA_FMT_BF16)
    maxpool2x2_cp8_kernel<MPA_FMT_BF16><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)in_cp8, (uint4*)out_cp8, total, NCk, ncs_in, ncs_out, To, Fo, T + 2 * pt_in, pitch_in, pf_in, pt_in, To + 2 * pt_out, pitch_out,
        pf_out, pt_out);
  else
    maxpool2x2_cp8_kernel<MPA_FMT_F16><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint4*)in_cp8, (uint4*)out_cp8, total, NCk, ncs_in, ncs_out, To, Fo, T + 2 * pt_in, pitch_in, pf_in, pt_in, To + 2 * pt_out, pitch_out,
        pf_out, pt_out);
  MPA_CHECK_LAUNCH("maxpool2x2_cp8");
  return MPA_OK;
}

int mpa_upsample2x_cp8(const void* low_cp8, void* out_cp8, int n, int C, int Tl, int Fl, int pitch_l, int pf_l, int pt_l, int ncs_l, int Ts,
                       int Fs, int pitch_s, int pf_s, int pt_s, int ncs_out, int fmt, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(low_cp8 && out_cp8 && n > 0 && C > 0 && (C & 7) == 0 && Ts >= 2 * Tl && Fs >= 2 * Fl, "upsample2x_cp8: bad argument (C %% 8 == 0 required)");
  const int NCk = C / 8;
  if (ncs_l <= 0) ncs_l = NCk;
  MPA_REQUIRE(ncs_out >= NCk, "upsample2x_cp8: destination chunk stride too small");
  long long total = (long long)n * NCk * Ts * Fs;
  if (fmt == MPA_FMT_F16X3) {
    if (ncs_l == NCk) ncs_l = 2 * NCk;
    MPA_REQUIRE(!((ncs_l | ncs_out) & 1) && ncs_out >= 2 * NCk, "upsample2x_cp8(fp16x3): chunk strides must be even (hi planes, then lo planes)");
    upsample2x_x3_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const uint4*)low_cp8, (uint4*)out_cp8, total, NCk, ncs_l, ncs_out, Tl, Fl,
                                                                                  Tl + 2 * pt_l, pitch_l, pf_l, pt_l, Ts, Fs, Ts + 2 * pt_s, pitch_s, pf_s, pt_s);
  } else if (fmt == MPA_FMT_BF16)
    upsample2x_cp8_kernel<MPA_FMT_BF16><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint16_t*)low_cp8, (uint16_t*)out_cp8, total, NCk, ncs_l, ncs_out, Tl, Fl, Tl + 2 * pt_l, pitch_l, pf_l, pt_l, Ts, Fs, Ts + 2 * pt_s,
        pitch_s, pf_s, pt_s);
  else
    upsample2x_cp8_kernel<MPA_FMT_F16><<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(
        (const uint16_t*)low_cp8, (uint16_t*)out_cp8, total, NCk, ncs_l, ncs_out, Tl, Fl, Tl + 2 * pt_l, pitch_l, pf_l, pt_l, Ts, Fs, Ts + 2 * pt_s,
        pitch_s, pf_s, pt_s);
  MPA_CHECK_LAUNCH("upsample2x_cp8");
  return MPA_OK;
}

int mpa_nchw_to_cp8(const float* x, void* out_cp8, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, int ncs_out, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out_cp8 && B > 0 && C > 0 && pitch >= pf + F, "nchw_to_cp8: bad argument");
  const int NCk = (C + 7) / 8;
  if (ncs_out <= 0) ncs_out = (fmt == MPA_FMT_F16X3 ? 2 : 1) * NCk;
  MPA_REQUIRE(fmt != MPA_FMT_F16X3 || !(ncs_out & 1), "nchw_to_cp8(fp16x3): the chunk stride must be even");
  long long total = (long long)B * NCk * T * F;
  nchw_to_cp8_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, (uint16_t*)out_cp8, total, C, T, F, NCk, ncs_out, T + 2 * pt,
                                                                               pitch, pf, pt, fmt);
  MPA_CHECK_LAUNCH("nchw_to_cp8");
  return MPA_OK;
}

int mpa_nchw_to_cp8_strided(const float* x, void* out_cp8, int B, int C, int T, int Fs, int F, int stride, int offset, int pitch, int pf, int pt,
                            int fmt, int ncs_out, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x && out_cp8 && B > 0 && C > 0 && stride >= 1 && offset >= 0 && offset + (Fs - 1) * stride < F && pitch >= pf + F,
              "nchw_to_cp8_strided: bad argument");
  const int NCk = (C + 7) / 8;
  if (ncs_out <= 0) ncs_out = (fmt == MPA_FMT_F16X3 ? 2 : 1) * NCk;
  MPA_REQUIRE(fmt != MPA_FMT_F16X3 || !(ncs_out & 1), "nchw_to_cp8_strided(fp16x3): the chunk stride must be even");
  long long total = (long long)B * NCk * T * Fs;
  nchw_to_cp8_strided_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(x, (uint16_t*)out_cp8, total, C, T, Fs, NCk, ncs_out, T + 2 * pt,
                                                                                       pitch, pf, pt, fmt, stride, offset);
  MPA_CHECK_LAUNCH("nchw_to_cp8_strided");
  return MPA_OK;
}

int mpa_cp8_to_nchw(const void* in_cp8, float* out, int B, int C, int T, int F, int pitch, int pf, int pt, int fmt, int ncs_in, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(in_cp8 && out && B > 0 && C > 0 && pitch >= pf + F, "cp8_to_nchw: bad argument");
  const int NCk = (C + 7) / 8;
  if (ncs_in <= 0) ncs_in = (fmt == MPA_FMT_F16X3 ? 2 : 1) * NCk;
  MPA_REQUIRE(fmt != MPA_FMT_F16X3 || !(ncs_in & 1), "cp8_to_nchw(fp16x3): the chunk stride must be even");
  long long total = (long long)B * NCk * T * F;
  cp8_to_nchw_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>((const uint16_t*)in_cp8, out, total, C, T, F, NCk, ncs_in, T + 2 * pt,
                                                                               pitch, pf, pt, fmt);
  MPA_CHECK_LAUNCH("cp8_to_nchw");
  return MPA_OK;
}

}  // extern "C"
