// tcgen05 weight gradient of a stride-1 "same" convolution on CP8 planes (16-bit, fp32 accumulate in TMEM):
//     gw[co][ci][kh][kw] = sum_{b,t,f} g[b,co,t,f] * x[b,ci,t+kh-ph,f+kw-pw]          (nn.Conv2d backward, weight part)
//
// Formulation ("pixels as K"): both operands are read MN-major straight out of the CP8 layout [chunk][pixel][8 ch] — a core
// matrix of the SWIZZLE_NONE MN-major canonical layout is 8 pixels x 8 channels = 128 contiguous bytes:
//     D[(r, co), (kw, e)] += sum_{16 pixels}  A[(r, co), px] * B[px, (kw, e)]
//   A = RS consecutive g rows t_lo .. t_lo+RS-1 of one patch, stacked along M: row group (r, channel chunk ck) sits at
//       slot(t_lo) + (r*NCo + ck) * 3584 B  (uniform SBO), so M = 128 lanes hold RS = floor(16/NCo) filter rows kh = kh_hi - r;
//   B = ONE x row s = t + kh - ph of one input chunk: N-group kw is the same slab shifted by kw pixels (SBO = 16 B), so
//       N = KW*8 columns (rounded up to a multiple of 16) = every horizontal tap x 8 input channels of the chunk;
//   K walks the P pixels of the padded row (P/16 MMAs); zero gap columns of g make the frequency padding exact, rows outside the
//   patch are streamed from a zero row.
// Work items = (filter-row set, input-chunk group of <= 4 chunks, slice of the B*T x-rows); an item keeps its <= 4 accumulators
// (128 lanes x KW*8 columns each) in TMEM over its whole slice and flushes them with fp32 atomicAdd into gw.
// The g rows live in a shared-memory ring whose slots ascend with t (one new row per x row; the RS-1 wrapping slots are mirrored).
// KH x 1 filters (`wide`): with one tap an MMA per input chunk would have N = 16 columns; instead up to 16 input chunks of a group are the
// N groups of ONE MMA (their slabs sit at a uniform stride in the x stage: SBO = slab bytes), N = 8 * chunks <= 128, one accumulator.
// Because K walks every pixel of the padded row, the result is right only when the inputs keep these conditions:
//   - the gap columns of g's real channels are zero (its pad rows are never read);
//   - the x pixels within KW/2 of a real bin are zero where they are not real bins themselves, counted along the flattened rows: the band
//     right of a row may continue into the next row's first columns;
//   - every byte it reads is finite (NaN * 0 = NaN).
// Split precision (mpa_conv_wgrad_tc_x3, wgrad_tc_kernel<true>): x and g are (hi, lo) fp16 plane pairs. The ring holds the g rows' hi planes
// and, ring_lo bytes further, their lo planes; an x stage holds the CG hi slabs and then the CG lo slabs. Each K step issues three MMAs into
// the one accumulator, g_hi.x_hi + g_lo.x_hi + g_hi.x_lo (the lo.lo term is below 2^-22 of the product). Both halves double the shared
// memory of a row, so the output chunks are split into co-blocks of NCo chunks (n_coblk of them, a work-item dimension) where the planes
// are wide; only bulk copies are used.
#include "common.cuh"
#include <cuda.h>
#include <string.h>

namespace mpa {

constexpr int kWgThreads = 192;            // producer warp, MMA warp, 4 epilogue warps
constexpr int kWgMaxSlots = 40;
constexpr int kWgXStages = 3;
constexpr unsigned long long kWgTimeoutNs = 4000000000ull;

struct WgradParams {
  const uint8_t* x;            // (row 0, column 0) of item 0, chunk 0
  const uint8_t* g;
  const uint8_t* zero_row;     // >= NCo * P * 16 bytes of zeros
  float* gw;
  long long x_item_stride, x_chunk_stride, g_item_stride, g_chunk_stride;   // bytes
  int B, T, P, KH, KW, ph, pw, NC, NCo, Cin, Cout, Cin_total, co0, ci0;
  int RS, n_sets, CG, n_cgroups, n_splits, n_items;
  // split precision only: NCo output chunks per co-block, NCo_all = ceil(Cout/8); lo planes x_lo / g_lo bytes after the hi planes;
  // the lo half of the ring ring_lo bytes after the hi half
  int NCo_all, n_coblk, ring_lo;
  long long x_lo, g_lo;
  int slots, slot_bytes, gslab_bytes, xslab_bytes, xstage_bytes, x_off, bar_off;
  uint32_t idesc;
  int wide;                    // KW == 1: the CG input chunks of a group are the N groups of ONE accumulator (B descriptor SBO = slab stride)
  // one g row of ALL NCo output chunks as ONE tensor-map copy (rank 5: a 3.5 KB row is two halves of <= 256 8-byte elements; rows outside
  // [0, T) are zero-filled by the copy unit, which replaces the zero row).  The copy unit retires ~1 bulk copy per 150 clocks whatever
  // its size: NCo = 16 copies per x row against ~900 tensor clocks made the 16 -> 128 layer copy-issue bound.
  int tma;
  alignas(64) CUtensorMap tm_g;
  // narrow planes (slab <= 128 pixels): the x row of ALL chunks of the item's group in one copy (the wide-N mode of KH x 1 filters issued up
  // to 16 copies of 1.4 KB per x row for ~100 tensor clocks of MMAs)
  int tma_x;
  alignas(64) CUtensorMap tm_x;
};

__device__ __forceinline__ uint32_t wg_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void wg_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(wg_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void wg_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(wg_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void wg_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(wg_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool wg_mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(wg_smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void wg_mbar_wait(uint64_t* bar, uint32_t parity) {
  if (wg_mbar_try_wait(bar, parity)) return;
  unsigned long long t0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
  uint32_t spins = 0;
  while (!wg_mbar_try_wait(bar, parity)) {
    if ((++spins & 255u) == 0) {
      unsigned long long t1;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
      if (t1 - t0 > kWgTimeoutNs) __trap();
    }
  }
}
__device__ __forceinline__ void wg_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(wg_smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(wg_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ bool wg_elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void wg_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(wg_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void wg_mma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void wg_ld32(uint32_t taddr, uint32_t* r) {
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

struct WgItem {
  int set, cg, q0, q1, kh_hi, nset, c0, nchunks, cob;
};
template <bool X3>
__device__ __forceinline__ WgItem wg_decode(const WgradParams& p, int item) {
  WgItem it;
  int type = item / p.n_splits;
  const int sp = item - type * p.n_splits;
  it.cob = 0;
  if (X3) { it.cob = type % p.n_coblk; type /= p.n_coblk; }
  it.set = type / p.n_cgroups;
  it.cg = type - it.set * p.n_cgroups;
  const long long R = (long long)p.B * p.T;
  it.q0 = (int)(R * sp / p.n_splits);
  it.q1 = (int)(R * (sp + 1) / p.n_splits);
  const int kh_lo = it.set * p.RS;
  it.kh_hi = min(p.KH, kh_lo + p.RS) - 1;
  it.nset = it.kh_hi - kh_lo + 1;
  it.c0 = it.cg * p.CG;
  it.nchunks = min(p.CG, p.NC - it.c0);
  return it;
}

template <bool X3>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_tc_kernel(const __grid_constant__ WgradParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* ring = smem;                                   // [slots + RS - 1][NCo][P px][16 B] (X3: then the same for the lo planes)
  uint8_t* xs = smem + p.x_off;                           // [kWgXStages][CG (X3: hi, then lo: 2 * CG)][slab px][16 B]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.bar_off);
  uint64_t* g_full = bars;                                // [slots]
  uint64_t* g_empty = bars + kWgMaxSlots;                 // [slots]
  uint64_t* x_full = bars + 2 * kWgMaxSlots;              // [kWgXStages]
  uint64_t* x_empty = x_full + kWgXStages;
  uint64_t* acc_full = x_empty + kWgXStages;              // [1]
  uint64_t* acc_empty = acc_full + 1;                     // [1]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int S = p.slots;

  if (threadIdx.x == 0) {
    for (int i = 0; i < S; ++i) { wg_mbar_init(&g_full[i], 1); wg_mbar_init(&g_empty[i], 1); }
    for (int i = 0; i < kWgXStages; ++i) { wg_mbar_init(&x_full[i], 1); wg_mbar_init(&x_empty[i], 1); }
    wg_mbar_init(acc_full, 1);
    wg_mbar_init(acc_empty, 128);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(wg_smem_u32(tmem_slot)), "r"(512u));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *tmem_slot;
  const int ksteps = p.P >> 4;
  constexpr int halves = X3 ? 2 : 1;

  if (warp == 0) {
    // ===================================================== producer: g rows (ring, ascending t) and x row slabs
    // the whole warp walks the (warp-uniform) loops; lane 0 waits on / arms the barriers, the copies of a ring slot (one per output
    // chunk, plus its mirror) and of an x stage are issued by the lanes in parallel (one thread needs ~170 clocks per bulk copy)
    {
      uint32_t n_row = 0;
      int xst = 0;
      uint32_t xph = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const WgItem it = wg_decode<X3>(p, item);
        for (int q = it.q0; q < it.q1; ++q) {
          const int b = q / p.T, s = q - b * p.T;
          const int t_new = s + p.ph - it.kh_hi + it.nset - 1;            // newest g row of this x row's tile
          const int n_load = (s == 0 || q == it.q0) ? it.nset : 1;
          for (int k = n_load - 1; k >= 0; --k, ++n_row) {
            const int t = t_new - k;
            const int pos = (int)(n_row % (uint32_t)S);
            const bool mirror = pos < p.RS - 1;
            if (lane == 0) {
              wg_mbar_wait(&g_empty[pos], ((n_row / (uint32_t)S) & 1u) ^ 1u);
              wg_mbar_expect_tx(&g_full[pos], (uint32_t)(p.NCo * p.gslab_bytes * halves) * (mirror ? 2u : 1u));
            }
            __syncwarp();
            uint8_t* dst = ring + (size_t)pos * p.slot_bytes;
            const bool inside = (t >= 0 && t < p.T);
            const int n_copies = p.tma ? 0 : p.NCo * (mirror ? 2 : 1) * halves;
            if (p.tma && lane == 0) {
              for (int mir = 0; mir < (mirror ? 2 : 1); ++mir)
                asm volatile(
                    "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];" ::"r"(
                        wg_smem_u32(dst + (mir ? (size_t)S * p.slot_bytes : 0))),
                    "l"(reinterpret_cast<uint64_t>(&p.tm_g)), "r"(0), "r"(0), "r"(t), "r"(0), "r"(b), "r"(wg_smem_u32(&g_full[pos]))
                    : "memory");
            }
            for (int i = lane; i < n_copies; i += 32) {
              const int ck = i % p.NCo, rest = i / p.NCo;
              const int mir = X3 ? rest >> 1 : rest, h = X3 ? rest & 1 : 0;
              const int gck = it.cob * p.NCo + ck;                          // chunks past the last output chunk read zeros
              const uint8_t* src = (inside && (!X3 || gck < p.NCo_all))
                                       ? p.g + (long long)b * p.g_item_stride + (long long)gck * p.g_chunk_stride + (h ? p.g_lo : 0) +
                                             (long long)t * p.P * 16
                                       : p.zero_row + (size_t)ck * p.gslab_bytes;
              wg_bulk_g2s(dst + (h ? (size_t)p.ring_lo : 0) + (mir ? (size_t)S * p.slot_bytes : 0) + (size_t)ck * p.gslab_bytes, src,
                          (uint32_t)p.gslab_bytes, &g_full[pos]);
            }
            __syncwarp();
          }
          if (lane == 0) {
            wg_mbar_wait(&x_empty[xst], xph ^ 1);
            wg_mbar_expect_tx(&x_full[xst], (uint32_t)((p.tma_x ? p.CG : it.nchunks) * p.xslab_bytes * halves));
            if (p.tma_x)
              asm volatile(
                  "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
                      wg_smem_u32(xs + (size_t)xst * p.xstage_bytes)),
                  "l"(reinterpret_cast<uint64_t>(&p.tm_x)), "r"(-2 * p.pw), "r"(s), "r"(it.c0), "r"(b), "r"(wg_smem_u32(&x_full[xst]))
                  : "memory");
          }
          __syncwarp();
          const uint8_t* xsrc = p.x + (long long)b * p.x_item_stride + ((long long)s * p.P - p.pw) * 16;
          for (int i = lane; i < (p.tma_x ? 0 : it.nchunks * halves); i += 32) {
            const int h = X3 ? i / it.nchunks : 0, c = i - h * it.nchunks;
            wg_bulk_g2s(xs + (size_t)xst * p.xstage_bytes + (size_t)(h * p.CG + c) * p.xslab_bytes,
                        xsrc + (long long)(it.c0 + c) * p.x_chunk_stride + (h ? p.x_lo : 0), (uint32_t)p.xslab_bytes, &x_full[xst]);
          }
          __syncwarp();
          if (++xst == kWgXStages) { xst = 0; xph ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================== MMA issuer (whole warp walks, one elected lane issues)
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t ring16 = wg_smem_u32(ring) >> 4, slot16 = (uint32_t)p.slot_bytes >> 4;
    const uint32_t xs16 = wg_smem_u32(xs) >> 4, xst16 = (uint32_t)p.xstage_bytes >> 4, xsl16 = (uint32_t)p.xslab_bytes >> 4;
    // MN-major SWIZZLE_NONE descriptors: LBO = 128 B between 8-pixel K groups; SBO = stride between 8-element MN groups
    const uint32_t a_hi = ((uint32_t)p.gslab_bytes >> 4) | (1u << 14);       // A: next channel chunk / next g row
    const uint32_t b_hi = (16u >> 4) | (1u << 14);                           // B: next tap = next pixel
    const uint32_t lo_fixed = (128u >> 4) << 16;
    uint32_t n_row = 0;
    int xst = 0;
    uint32_t xph = 0, k_item = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++k_item) {
      const WgItem it = wg_decode<X3>(p, item);
      wg_mbar_wait(acc_empty, (k_item & 1u) ^ 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      uint32_t first = 1;
      for (int q = it.q0; q < it.q1; ++q) {
        const int b = q / p.T, s = q - b * p.T;
        const int n_load = (s == 0 || q == it.q0) ? it.nset : 1;
        for (int k = 0; k < n_load; ++k, ++n_row) wg_mbar_wait(&g_full[(int)(n_row % (uint32_t)S)], (n_row / (uint32_t)S) & 1u);
        wg_mbar_wait(&x_full[xst], xph);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const uint32_t n_old = n_row - (uint32_t)it.nset;                     // oldest row of the tile (rows n_old .. n_row-1)
        const uint32_t a_lo = (ring16 + (n_old % (uint32_t)S) * slot16) | lo_fixed;
        const uint32_t b_lo0 = (xs16 + (uint32_t)xst * xst16) | lo_fixed;
        const bool last_of_patch = (s == p.T - 1) || (q == it.q1 - 1);
        if (wg_elect_one()) {
          if (p.wide) {
            const uint32_t bw_hi = xsl16 | (1u << 14);                       // B: next N group = next input chunk's slab
            for (int ks = 0; ks < ksteps; ++ks)
              wg_mma(tmem_u, ((uint64_t)a_hi << 32) | (uint64_t)(a_lo + (uint32_t)ks * 16u), ((uint64_t)bw_hi << 32) | (uint64_t)(b_lo0 + (uint32_t)ks * 16u),
                     p.idesc, (first && ks == 0) ? 0u : 1u);
          } else {
            for (int c = 0; c < it.nchunks; ++c) {
              const uint32_t tmem_d = tmem_u + (uint32_t)c * 128u;
              const uint32_t b_lo = b_lo0 + (uint32_t)c * xsl16;
              for (int ks = 0; ks < ksteps; ++ks) {
                const uint64_t ad = ((uint64_t)a_hi << 32) | (uint64_t)(a_lo + (uint32_t)ks * 16u);
                const uint64_t bd = ((uint64_t)b_hi << 32) | (uint64_t)(b_lo + (uint32_t)ks * 16u);
                wg_mma(tmem_d, ad, bd, p.idesc, (first && ks == 0) ? 0u : 1u);
                if (X3) {
                  wg_mma(tmem_d, ad + ((uint32_t)p.ring_lo >> 4), bd, p.idesc, 1u);                     // g_lo . x_hi
                  wg_mma(tmem_d, ad, bd + (uint32_t)p.CG * xsl16, p.idesc, 1u);                          // g_hi . x_lo
                }
              }
            }
          }
          wg_commit(&x_empty[xst]);
          // the oldest g row is done; at the end of a patch (or of the slice) so are the others
          wg_commit(&g_empty[(int)(n_old % (uint32_t)S)]);
          if (last_of_patch)
            for (int k = 1; k < it.nset; ++k) wg_commit(&g_empty[(int)((n_old + (uint32_t)k) % (uint32_t)S)]);
        }
        __syncwarp();
        first = 0;
        if (++xst == kWgXStages) { xst = 0; xph ^= 1; }
      }
      if (wg_elect_one()) wg_commit(acc_full);
      __syncwarp();
    }
  } else {
    // ===================================================== epilogue: TMEM -> fp32 atomicAdd into gw
    const int quad = warp & 3;                            // TMEM lane quadrant of this warp
    const int m = quad * 32 + lane;
    const int r = m / (p.NCo * 8), co = m - r * (p.NCo * 8);
    const int ncols = p.KW * 8;
    uint32_t k_item = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x, ++k_item) {
      const WgItem it = wg_decode<X3>(p, item);
      wg_mbar_wait(acc_full, k_item & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const int co_g = it.cob * p.NCo * 8 + co;            // output channel of the call (co-blocks: X3 only)
      const bool row_ok = (r < it.nset) && (co_g < p.Cout);
      const int kh = it.kh_hi - r;
      if (p.wide) {
        // one accumulator: column n = (input chunk n / 8 of the group, channel n % 8), the single tap kw = 0
        for (int c0 = 0; c0 < it.nchunks * 8; c0 += 32) {
          uint32_t v[32];
          wg_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, v);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (row_ok) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int n = c0 + i;
              const int ci = (it.c0 + (n >> 3)) * 8 + (n & 7);
              if (n < it.nchunks * 8 && ci < p.Cin)
                atomicAdd(p.gw + ((size_t)(p.co0 + co_g) * p.Cin_total + p.ci0 + ci) * p.KH + kh, __uint_as_float(v[i]));
            }
          }
        }
      }
      for (int c = 0; c < (p.wide ? 0 : it.nchunks); ++c) {
        for (int c0 = 0; c0 < ncols; c0 += 32) {
          uint32_t v[32];
          wg_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(c * 128 + c0), v);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (row_ok) {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const int n = c0 + i;
              const int kw = n >> 3, ci = (it.c0 + c) * 8 + (n & 7);
              if (n < ncols && ci < p.Cin)
                atomicAdd(p.gw + (((size_t)(p.co0 + co_g) * p.Cin_total + p.ci0 + ci) * p.KH + kh) * p.KW + kw, __uint_as_float(v[i]));
            }
          }
        }
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      wg_mbar_arrive(acc_empty);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u));
  }
}

}  // namespace mpa

using namespace mpa;

extern "C" {

int mpa_conv_wgrad_tc(const void* x_cp8, const void* g_cp8, const void* zero_row, float* gw, int n_items, int Cin, int Cout, int T, int F,
                      int KH, int KW, int pitch, int pf, int pt, int x_nc_stride, int g_nc_stride, int Cin_total, int ci0, int Cout_total,
                      int co0, int fmt, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x_cp8 && g_cp8 && zero_row && gw && n_items > 0 && Cin > 0 && Cout > 0 && Cout <= 128, "conv_wgrad_tc: bad argument (Cout <= 128 per call)");
  MPA_REQUIRE((KH & 1) && (KW & 1) && KW <= 15, "conv_wgrad_tc: odd kernel sizes, KW <= 15");
  MPA_REQUIRE(fmt == MPA_FMT_F16 || fmt == MPA_FMT_BF16, "conv_wgrad_tc: fmt must be MPA_FMT_F16 or MPA_FMT_BF16");
  MPA_REQUIRE(pitch % 16 == 0 && pitch >= 16 && pitch <= 256 && pf >= KW / 2 && pitch - F >= KW / 2 && pitch >= pf + F && pt >= 1,
              "conv_wgrad_tc: CP8 geometry (pitch %d, pf %d, F %d, KW %d)", pitch, pf, F, KW);
  MPA_REQUIRE(ci0 >= 0 && co0 >= 0 && ci0 + Cin <= Cin_total && co0 + Cout <= Cout_total, "conv_wgrad_tc: channel block outside the weight tensor");
  MPA_REQUIRE((((uintptr_t)x_cp8 | (uintptr_t)g_cp8 | (uintptr_t)zero_row) & 15) == 0, "conv_wgrad_tc: 16-byte alignment required");
  WgradParams p;
  memset(&p, 0, sizeof(p));
  p.B = n_items; p.T = T; p.P = pitch; p.KH = KH; p.KW = KW; p.ph = KH / 2; p.pw = KW / 2;
  p.NC = (Cin + 7) / 8;
  p.NCo = (Cout + 7) / 8;
  p.Cin = Cin; p.Cout = Cout; p.Cin_total = Cin_total; p.co0 = co0; p.ci0 = ci0;
  const long long plane = (long long)(T + 2 * pt) * pitch * 16;
  p.x_chunk_stride = plane;
  p.g_chunk_stride = plane;
  p.x_item_stride = plane * (x_nc_stride > 0 ? x_nc_stride : p.NC);
  p.g_item_stride = plane * (g_nc_stride > 0 ? g_nc_stride : p.NCo);
  p.x = (const uint8_t*)x_cp8 + (long long)pt * pitch * 16;
  p.g = (const uint8_t*)g_cp8 + (long long)pt * pitch * 16;
  p.zero_row = (const uint8_t*)zero_row;
  p.gw = gw;
  p.RS = 16 / p.NCo;
  if (p.RS > KH) p.RS = KH;
  p.n_sets = (KH + p.RS - 1) / p.RS;
  p.wide = KW == 1 && p.NC >= 2;
  p.CG = p.wide ? (p.NC < 16 ? (p.NC + 1) / 2 * 2 : 16) : (p.NC < 4 ? p.NC : 4);
  p.n_cgroups = (p.NC + p.CG - 1) / p.CG;
  p.gslab_bytes = pitch * 16;
  p.slot_bytes = p.NCo * p.gslab_bytes;
  p.xslab_bytes = ((pitch + 2 * (KW / 2) + 1 + 7) / 8 * 8) * 16;
  // wide mode: as many chunks per group as leave room for a minimal row ring
  while (p.wide && p.CG > 2 && (size_t)kWgXStages * p.CG * p.xslab_bytes + 1024 + (size_t)(2 * p.RS) * p.NCo * p.gslab_bytes > 227 * 1024) p.CG -= 2;
  p.n_cgroups = (p.NC + p.CG - 1) / p.CG;
  p.xstage_bytes = p.CG * p.xslab_bytes;
  const size_t fixed = (size_t)kWgXStages * p.xstage_bytes + 1024;
  int slots = p.RS + 3;
  while (slots > p.RS + 1 && (size_t)(slots + p.RS - 1) * p.slot_bytes + fixed > 227 * 1024) --slots;
  MPA_REQUIRE(slots >= p.RS + 1 && slots <= kWgMaxSlots && (size_t)(slots + p.RS - 1) * p.slot_bytes + fixed <= 227 * 1024,
              "conv_wgrad_tc: the row ring does not fit in shared memory (Cout=%d pitch=%d)", Cout, pitch);
  p.slots = slots;
  p.x_off = (slots + p.RS - 1) * p.slot_bytes;
  p.bar_off = p.x_off + kWgXStages * p.xstage_bytes;
  // M = 128 always reads 16 row groups from the tile start; when RS*NCo < 16 the surplus groups (ignored lanes) reach past the ring
  size_t smem = (size_t)p.bar_off + 1024;
  const size_t reach = (size_t)(slots - 1) * p.slot_bytes + 16 * (size_t)p.gslab_bytes;
  if (smem < reach) smem = reach;
  MPA_REQUIRE(smem <= 227 * 1024, "conv_wgrad_tc: needs %zu B of shared memory", smem);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int n_types = p.n_sets * p.n_cgroups;
  const long long R = (long long)n_items * T;
  int splits = sms / n_types;                              // one wave of items
  if (splits > R) splits = (int)R;
  if (splits < 1) splits = 1;
  p.n_splits = splits;
  p.n_items = n_types * splits;
  const uint32_t f = (fmt == MPA_FMT_BF16) ? 1u : 0u;
  const int N = p.wide ? p.CG * 8 : (KW * 8 + 15) / 16 * 16;   // M = 128 needs N % 16 == 0: the extra taps / chunks land in ignored columns
  p.idesc = (1u << 4) | (f << 7) | (f << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  {
    static unsigned char flags[64];
    cudaError_t e = opt_in_max_smem(wgrad_tc_kernel<false>, flags);
    if (e != cudaSuccess) {
      set_error("conv_wgrad_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return MPA_ERR_CUDA;
    }
  }
  p.tma = 0;
  if (TensorMapEncodeFn enc = tensor_map_encoder()) {
    if (p.NCo >= 2) {
      const cuuint64_t gd[5] = {(cuuint64_t)pitch, 2, (cuuint64_t)T, (cuuint64_t)p.NCo, (cuuint64_t)n_items};
      const cuuint64_t gs[4] = {(cuuint64_t)pitch * 8, (cuuint64_t)pitch * 16, (cuuint64_t)p.g_chunk_stride, (cuuint64_t)p.g_item_stride};
      const cuuint32_t bx[5] = {(cuuint32_t)pitch, 2, 1, (cuuint32_t)p.NCo, 1}, es[5] = {1, 1, 1, 1, 1};
      const CUresult r = enc(&p.tm_g, CU_TENSOR_MAP_DATA_TYPE_UINT64, 5, const_cast<uint8_t*>(p.g), gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      p.tma = r == CUDA_SUCCESS ? 1 : 0;                                 // else: one bulk copy per output chunk
    }
  }
  p.tma_x = 0;
  if (TensorMapEncodeFn enc = tensor_map_encoder()) {
    const int xslab_px = p.xslab_bytes / 16;
    if (p.NC >= 2 && xslab_px <= 128 && (p.xstage_bytes % 128) == 0) {
      const cuuint64_t xd[4] = {(cuuint64_t)pitch * 2, (cuuint64_t)T, (cuuint64_t)p.NC, (cuuint64_t)n_items};
      const cuuint64_t xs_[3] = {(cuuint64_t)pitch * 16, (cuuint64_t)p.x_chunk_stride, (cuuint64_t)p.x_item_stride};
      const cuuint32_t bx[4] = {(cuuint32_t)xslab_px * 2, 1, (cuuint32_t)p.CG, 1}, es[4] = {1, 1, 1, 1};
      const CUresult r = enc(&p.tm_x, CU_TENSOR_MAP_DATA_TYPE_UINT64, 4, const_cast<uint8_t*>(p.x), xd, xs_, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      p.tma_x = r == CUDA_SUCCESS ? 1 : 0;
    }
  }
  const int grid = p.n_items < sms ? p.n_items : sms;
  wgrad_tc_kernel<false><<<grid, kWgThreads, smem, (cudaStream_t)stream>>>(p);
  MPA_CHECK_LAUNCH("conv_wgrad_tc");
  return MPA_OK;
}

int mpa_conv_wgrad_tc_x3(const void* x_cp8, const void* g_cp8, const void* zero_row, float* gw, int n_items, int Cin, int Cout, int T, int F,
                         int KH, int KW, int pitch, int pf, int pt, int x_nc_stride, int g_nc_stride, int Cin_total, int ci0, int Cout_total,
                         int co0, void* stream) {
  MPA_CHECK_ARCH();
  MPA_REQUIRE(x_cp8 && g_cp8 && zero_row && gw && n_items > 0 && Cin > 0 && Cout > 0 && Cout <= 128,
              "conv_wgrad_tc_x3: bad argument (Cout <= 128 per call)");
  MPA_REQUIRE((KH & 1) && (KW & 1) && KW >= 3 && KW <= 15, "conv_wgrad_tc_x3: odd kernel sizes, 3 <= KW <= 15 (no KW == 1 form)");
  MPA_REQUIRE(pitch % 16 == 0 && pitch >= 16 && pitch <= 256 && pf >= KW / 2 && pitch - F >= KW / 2 && pitch >= pf + F && pt >= 1,
              "conv_wgrad_tc_x3: CP8 geometry (pitch %d, pf %d, F %d, KW %d)", pitch, pf, F, KW);
  MPA_REQUIRE(ci0 >= 0 && co0 >= 0 && ci0 + Cin <= Cin_total && co0 + Cout <= Cout_total, "conv_wgrad_tc_x3: channel block outside the weight tensor");
  MPA_REQUIRE((((uintptr_t)x_cp8 | (uintptr_t)g_cp8 | (uintptr_t)zero_row) & 15) == 0, "conv_wgrad_tc_x3: 16-byte alignment required");
  const int NC = (Cin + 7) / 8, NCo_all = (Cout + 7) / 8;
  const int xs_ = x_nc_stride > 0 ? x_nc_stride : 2 * NC, gs_ = g_nc_stride > 0 ? g_nc_stride : 2 * NCo_all;
  MPA_REQUIRE(xs_ % 2 == 0 && gs_ % 2 == 0 && xs_ >= 2 * NC && gs_ >= 2 * NCo_all,
              "conv_wgrad_tc_x3: the chunk strides (%d, %d) must be even and hold hi and lo planes of every chunk", xs_, gs_);
  WgradParams p;
  memset(&p, 0, sizeof(p));
  p.B = n_items; p.T = T; p.P = pitch; p.KH = KH; p.KW = KW; p.ph = KH / 2; p.pw = KW / 2;
  p.NC = NC; p.NCo_all = NCo_all;
  p.Cin = Cin; p.Cout = Cout; p.Cin_total = Cin_total; p.co0 = co0; p.ci0 = ci0;
  const long long plane = (long long)(T + 2 * pt) * pitch * 16;
  p.x_chunk_stride = plane;
  p.g_chunk_stride = plane;
  p.x_item_stride = plane * xs_;
  p.g_item_stride = plane * gs_;
  p.x_lo = plane * (xs_ / 2);
  p.g_lo = plane * (gs_ / 2);
  p.x = (const uint8_t*)x_cp8 + (long long)pt * pitch * 16;
  p.g = (const uint8_t*)g_cp8 + (long long)pt * pitch * 16;
  p.zero_row = (const uint8_t*)zero_row;
  p.gw = gw;
  p.gslab_bytes = pitch * 16;
  p.xslab_bytes = ((pitch + 2 * (KW / 2) + 1 + 7) / 8 * 8) * 16;
  // Shared memory: both halves of the ring (slots + RS - 1 rows of NCo chunks each) and of kWgXStages x stages of CG chunks, 1 KB of
  // barriers, and the reach of the last tile's M = 128 rows past the lo ring. Shrink RS, then CG, then halve the co-block until it fits;
  // NCo = RS = CG = 1 at pitch 256 needs max(16 KB + 6 * 4.25 KB + 1 KB, 3 * 4 KB + 64 KB of reach) = 76 KB, so every admissible call fits.
  auto need = [&](int NCo, int RS, int CG, int slots) {
    const size_t slot = (size_t)NCo * p.gslab_bytes;
    const size_t top = 2 * (size_t)(slots + RS - 1) * slot + (size_t)kWgXStages * 2 * CG * p.xslab_bytes + 1024;
    const size_t reach = (size_t)(2 * slots + RS - 2) * slot + 16 * (size_t)p.gslab_bytes;
    return top > reach ? top : reach;
  };
  const size_t kMax = 227 * 1024;
  int NCo = NCo_all, RS, CG;
  for (;;) {
    RS = 16 / NCo < KH ? 16 / NCo : KH;
    CG = NC < 4 ? NC : 4;
    while (RS > 1 && need(NCo, RS, CG, RS + 1) > kMax) --RS;
    while (CG > 1 && need(NCo, RS, CG, RS + 1) > kMax) --CG;
    if (need(NCo, RS, CG, RS + 1) <= kMax || NCo == 1) break;
    NCo = (NCo + 1) / 2;
  }
  p.NCo = NCo; p.RS = RS; p.CG = CG;
  p.n_coblk = (NCo_all + NCo - 1) / NCo;
  p.n_sets = (KH + RS - 1) / RS;
  p.n_cgroups = (NC + CG - 1) / CG;
  p.slot_bytes = NCo * p.gslab_bytes;
  p.xstage_bytes = 2 * CG * p.xslab_bytes;
  int slots = RS + 3;
  while (slots > RS + 1 && need(NCo, RS, CG, slots) > kMax) --slots;
  MPA_REQUIRE(need(NCo, RS, CG, slots) <= kMax, "conv_wgrad_tc_x3: the row ring does not fit in shared memory (Cout=%d pitch=%d)", Cout, pitch);
  p.slots = slots;
  p.ring_lo = (slots + RS - 1) * p.slot_bytes;
  p.x_off = 2 * p.ring_lo;
  p.bar_off = p.x_off + kWgXStages * p.xstage_bytes;
  const size_t smem = need(NCo, RS, CG, slots);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int n_types = p.n_sets * p.n_cgroups * p.n_coblk;
  const long long R = (long long)n_items * T;
  int splits = sms / n_types;
  if (splits > R) splits = (int)R;
  if (splits < 1) splits = 1;
  p.n_splits = splits;
  p.n_items = n_types * splits;
  const int N = (KW * 8 + 15) / 16 * 16;
  p.idesc = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);   // fp16 x fp16 -> fp32
  {
    static unsigned char flags[64];
    cudaError_t e = opt_in_max_smem(wgrad_tc_kernel<true>, flags);
    if (e != cudaSuccess) {
      set_error("conv_wgrad_tc_x3: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
      return MPA_ERR_CUDA;
    }
  }
  const int grid = p.n_items < sms ? p.n_items : sms;
  wgrad_tc_kernel<true><<<grid, kWgThreads, smem, (cudaStream_t)stream>>>(p);
  MPA_CHECK_LAUNCH("conv_wgrad_tc_x3");
  return MPA_OK;
}

}  // extern "C"
