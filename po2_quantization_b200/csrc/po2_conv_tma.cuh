// K3T: the TMA-fed form of the tcgen05 implicit-GEMM conv (included by po2_conv.cu, same namespace).
//
// models/quantized_conv.py:36 -> F.conv2d(x, Q(w)) for the dense stride-1 layers (3x3 pad 1, 1x1 pad 0),
// operands tf32 -- the arithmetic of the reference's own cuDNN default on a GPU.
//
// The activation tensor never passes through registers.  fp32 NCHW has the PIXEL index contiguous, i.e.
// it already is an "MN-major" A operand of the implicit GEMM (M = pixels, K = channels), and kind::tf32
// reads fp32 containers as they are.  tcgen05 accepts MN-major tf32 operands in exactly one shared-memory
// layout, SWIZZLE_128B_BASE32B: runs of 32 pixels (128 bytes) per channel, 32-byte chunks XOR-swizzled
// over 4 channel rows; its TMA counterpart is CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B.  One elected thread
// issues tensor-map loads (cp.async.bulk.tensor.5d) over the tensor viewed as
//     ( w | image | c % 8 | h | c / 8 )
// with box { 32, 1, 8, rows, channel groups }: in shared memory that is [c/8][row][c%8][32 pixels] --
// one 1 KB "atom" of 8 channel rows x 32 pixels per (channel group, image row), which is the canonical
// layout (LBO = 1 KB between atoms along M, SBO = 512 B between the two 4-channel halves of a K = 8 MMA).
//   * filter row r is a shift of the A descriptor's start address by r atoms (the box carries one halo
//     row above and below; rows outside the image are zero-filled by the TMA unit: padding costs nothing);
//   * filter column s cannot be an address shift in this layout (4 bytes; descriptors and TMA box starts
//     have 16-byte granularity -- a box at w0-1 is an illegal instruction), so the shift is moved to the
//     OUTPUT side: the three filter columns accumulate into three TMEM accumulators
//         Y_s[h][w] = sum over r, c of x[h+r-1][w][c] * W[k][c][r][s]
//     and the epilogue forms out[h][w] = Y_0[h][w-1] + Y_1[h][w] + Y_2[h][w+1] with two warp shuffles
//     (TMEM lane = pixel; a 32-pixel run is one image row, or 32/W whole rows of different images, so
//     the neighbour of an edge pixel is the zero padding).  x is staged ONCE per tile.
//   * image rows shorter than 32 pixels (W = 16, 8, 4; measured: a swizzled TMA box always pitches its
//     inner rows at 128 bytes, so two images cannot share a run): the image plane is viewed FLAT, a run =
//     32 consecutive pixels = 32/W whole rows.  A filter row is then half a run or less, not an atom
//     shift, so x is staged as three row-shifted copies (run j of copy r starts at pixel (r-1)*W + 32*j;
//     one TMA per run, pixels before/after the plane are zero fill) and tap (r, s) reads copy r.
// 1x1 convs view the image as H*W/32 runs.  Weights: the
// packed exact +-2^q tf32 operand of the register-fed kernel, unchanged (K-major, no swizzle, whole-K slab
// per CTA by bulk copy).  Accumulators: two TMEM stages; the epilogue warps read them with tcgen05.ld,
// apply the per-tensor scale and store NCHW fp32.
//
// Roles (6 warps, persistent, one CTA per SM): warps 0-3 epilogue, warp 4 MMA issuer + TMEM owner +
// weight slab, warp 5 TMA producer (one elected lane).
#pragma once
#include <cuda.h>      // CUtensorMap and the encoder's enums (types only: the entry point is looked up at run time)

namespace po2 {

constexpr int KT_ATOM = 1024;     // 8 channel rows x 32 pixels x 4 bytes

struct TmaPlan {
  int mode;                  // 0: 3x3 pad 1 stride 1, 16 < W <= 32 (a run = one image row, halo rows in the box);
                             // 4: 3x3 pad 1 stride 1, W = 16/8/4 (flat runs, three row-shifted copies);
                             // 1x1 pad 0 stride 1: 1 = runs of one image per tile, 2 = whole images per tile
  int ntaps;                 // 9 or 1
  int WB, lgWB, IPR;         // pixels of one image row inside a 32-pixel run: 32/16/8/4 (IPR: unused, 1)
  int MT, APT;               // MMA M (128 or 64) and atoms (32-pixel runs) per tile = MT / 32
  int rows_st;               // atoms per channel group of a stage: APT + 2 halo rows (3x3) or APT
  int nacc;                  // TMEM accumulator stages (2, or 1 when 2 do not fit 512 columns)
  int ncol, nrb, ngrp;       // mode 0: column chunks per row (1), row blocks per image, images
  int AH, lgAH;              // modes 1, 2, 4: runs per image
  int IPT;                   // mode 2: images per tile
  int tiles_per_img;         // mode 1
  int nitems_m, m_step;
  int NCGS, nchunk;          // 8-channel groups per pipeline stage, stages per tile
  int nst;
  int cps;                   // CTAs per SM the plan was sized for (2 when two CTAs' shared memory and TMEM fit)
  int pdl;                   // launched with programmatic stream serialization: 1 = behind the weight-pack kernel (the
                             // slab copy waits for it, x is older), 2 = behind any kernel, e.g. the norm that produced x
                             // (the slab copy, the TMA producer and the epilogue all wait)
  int debug;                 // PO2_TMA_DEBUG bit mask (1: no TMA loads, 2: no MMAs, 4: no descriptor prefetch)
  int HW, Himg, Wimg;        // image geometry (ConvGeom's H/W are flattened for 1x1 layers)
  uint32_t stage_bytes, cg_bytes;                 // per stage / per channel group (modes 0-2)
  uint32_t a_lbo16, a_ks16, a_r16;                // A descriptor strides in 16-byte units: next run along M, next
                                                  // 8 channels, next filter row
  FastDiv div_ncol, div_nrb, div_tpi;
};

constexpr int KT_MAX_ACC = 8;         // accumulator barrier slots in shared memory (nacc <= 2 used); sizes the stage count
constexpr int KT_EPI_WARPS = 4;
constexpr int KT_THREADS = 32 * (KT_EPI_WARPS + 2);
constexpr uint32_t KT_SMEM_BUDGET = 222 * 1024;
constexpr uint32_t KT_SMEM_BUDGET_2 = 110 * 1024;     // per CTA when two share an SM (228 KB - 1 KB reserved each)
constexpr uint32_t KT_STAGE_TARGET = 32 * 1024;

__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, int c4,
                                            uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
      ::"r"(smem_u32(dst)), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(tm) : "memory");
}

__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// instruction descriptor: D = f32, A = B = tf32, A MN-major (pixels contiguous), B K-major, M, N
__device__ __forceinline__ uint32_t make_idesc_tma(uint32_t m, uint32_t n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

template <int NTAPS>
__global__ void __launch_bounds__(KT_THREADS, 2) conv_tma_kernel(const __grid_constant__ CUtensorMap tmx,
                                                                 const uint8_t* __restrict__ Bp,
                                                                 const float* __restrict__ scale,
                                                                 float* __restrict__ out, ConvGeom g, TmaPlan tp,
                                                                 ConvEpilogue ep) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  uint8_t* sB = smem;
  const uint32_t a_off = ((smem_base + g.b_slab_bytes + 1023u) & ~1023u) - smem_base;   // swizzle atoms: 1 KB aligned
  uint8_t* sA = smem + a_off;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA + (size_t)tp.nst * tp.stage_bytes);
  uint64_t* full = bars;                        // [nst]  TMA -> MMA
  uint64_t* empty = bars + K3_MAX_STAGES;       // [nst]  MMA (commit) -> TMA
  uint64_t* tfull = bars + 2 * K3_MAX_STAGES;   // [nacc] MMA (commit) -> epilogue
  uint64_t* tempty = tfull + KT_MAX_ACC;        // [nacc] epilogue -> MMA
  uint64_t* bfull = tempty + KT_MAX_ACC;        // weight slab landed
  uint64_t* tready = bfull + 1;                 // TMEM allocated, address published
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tready + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#ifdef PO2_K3_TRACE
  for (int i = tid; i < 8 * 64; i += KT_THREADS) k3_trace_smem[i] = 0;
  __syncthreads();
#endif
  if (tid == 0) K3_TRACE(6, 0);
  const int nt = blockIdx.x % g.ntiles_n;
  const int m_first = blockIdx.x / g.ntiles_n;
  const int nitems = tp.nitems_m, m_step = tp.m_step, nst = tp.nst, nchunk = tp.nchunk;
  constexpr int NACCW = NTAPS == 9 ? 3 : 1;       // accumulators per tile: one per filter column
  const uint32_t acc_cols = (uint32_t)(NACCW * g.NT);
  uint32_t ncols = 32;
  while (ncols < (uint32_t)tp.nacc * acc_cols) ncols <<= 1;

  // Barrier initialisation is spread over the producer warp's lanes (one mbarrier.init each instead of ~18 in
  // a row on one thread); the producer does not wait for the rest of the CTA: it arrives on named barrier 1
  // and starts issuing TMA loads, the other warps sync on it.
  if (warp == KT_EPI_WARPS + 1) {
    if (lane == 0 && !(tp.debug & 4)) tma_prefetch_desc(&tmx);
    if (lane < nst) mbar_init(full + lane, 1);
    else if (lane < 2 * nst) mbar_init(empty + (lane - nst), 1);
    else if (lane < 2 * nst + tp.nacc) mbar_init(tfull + (lane - 2 * nst), 1);
    else if (lane < 2 * nst + 2 * tp.nacc) mbar_init(tempty + (lane - 2 * nst - tp.nacc), KT_EPI_WARPS);
    else if (lane == 2 * nst + 2 * tp.nacc) mbar_init(bfull, 1);
    else if (lane == 2 * nst + 2 * tp.nacc + 1) mbar_init(tready, 1);      // 2 * 6 + 2 * 8 + 2 <= 32 lanes
    fence_mbar_init();
    __syncwarp();
    asm volatile("bar.arrive 1, %0;" ::"n"(KT_THREADS) : "memory");
  } else {
    asm volatile("bar.sync 1, %0;" ::"n"(KT_THREADS) : "memory");
  }
  uint32_t tmem_base = 0;
  if (warp == KT_EPI_WARPS) {
    // The weight slab is the longest single transfer of a CTA: it goes out before the TMEM allocation --
    // unless this grid was launched programmatically behind the kernel that packs the slab, in which case
    // the allocation overlaps that kernel and the copy waits for its completion.
    if (!tp.pdl && lane == 0) {
      mbar_expect_tx(bfull, g.b_slab_bytes);
      bulk_g2s(sB, Bp + (size_t)nt * g.b_slab_bytes, g.b_slab_bytes, bfull);
    }
    __syncwarp();
    tmem_alloc(tmem_slot, ncols);
    if (tp.pdl && lane == 0) {
      asm volatile("griddepcontrol.wait;" ::: "memory");       // the weight-pack kernel has completed and flushed
      mbar_expect_tx(bfull, g.b_slab_bytes);
      bulk_g2s(sB, Bp + (size_t)nt * g.b_slab_bytes, g.b_slab_bytes, bfull);
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(tready);
    tc_fence_after();
    tmem_base = *tmem_slot;
  } else if (warp < KT_EPI_WARPS) {
    mbar_wait(tready, 0);
    tc_fence_after();
    tmem_base = *tmem_slot;
  }

  if (tid == 0) K3_TRACE(6, 1);
  if (warp == KT_EPI_WARPS + 1) {
    // =========================== TMA producer (one lane) ===========================
    // x was complete before the kernel in front of this one started (see launch_conv: programmatic
    // launch only behind our own pack / quantize kernels), so no griddepcontrol.wait here.
    // (mode 4 issues 3 * APT boxes per stage: they are spread over the lanes of the warp -- a TMA issue costs a
    // thread ~150 cycles -- lane i owns box i; the other modes have one box per stage, issued by lane 0)
    // pdl == 2 (the layer chain): the kernel in front -- a norm kernel that triggered its dependents early -- is the
    // producer of x; everything up to here (launch, barriers, TMEM, tensor-map fetch) overlapped its tail
    if (tp.pdl == 2) asm volatile("griddepcontrol.wait;" ::: "memory");
    {
      uint32_t s = 0, sphase = 0;
      int tr_it = 0;
      (void)tr_it;
      const int nbox = tp.mode == 4 ? 3 * tp.APT : 1;
      for (int m = m_first; m < nitems; m += m_step) {
        int c0 = 0, c1 = 0, c3 = 0;                          // box coordinates of the tile
        if (tp.mode == 0) {                                  // (w, image, c % 8, h, c / 8)
          const int t = fdiv(m, tp.div_ncol);
          const int j = m - t * tp.ncol;
          const int ng = fdiv(t, tp.div_nrb);
          const int rb = t - ng * tp.nrb;
          c0 = j * tp.WB; c1 = ng * tp.IPR; c3 = rb * tp.APT - 1;
        } else if (tp.tiles_per_img > 0) {                   // modes 1, 4: c0 = first run of the tile, c3 = image
          const int n = fdiv(m, tp.div_tpi);
          c3 = n;
          c0 = (m - n * tp.tiles_per_img) * tp.APT;
        } else {                                             // modes 2, 4: whole images per tile
          c3 = m * tp.IPT;
        }
        for (int chunk = 0; chunk < nchunk; ++chunk) {
          if (lane == 0) {
            mbar_wait(empty + s, sphase ^ 1);
            K3_TRACE(2, 2 * tr_it);
            if (tp.debug & 1) mbar_arrive(full + s);
            else mbar_expect_tx(full + s, tp.stage_bytes);
          }
          __syncwarp();
          uint8_t* stage = sA + (size_t)s * tp.stage_bytes;
          const int cg0 = chunk * tp.NCGS;
          if (lane < nbox && !(tp.debug & 1)) {
            if (tp.mode == 0) {
              tma_load_5d(stage, &tmx, c0, c1, 0, c3, cg0, full + s);
            } else if (tp.mode == 4) {                       // (flat pixel, c % 8, c / 8, image, -): one box per run
              const uint32_t run_bytes = (uint32_t)tp.NCGS * KT_ATOM;
              const int r = lane / tp.APT, j = lane - r * tp.APT;
              const int n = tp.tiles_per_img > 0 ? c3 : c3 + (j >> tp.lgAH);
              const int run = tp.tiles_per_img > 0 ? c0 + j : (j & (tp.AH - 1));
              tma_load_5d(stage + (size_t)lane * run_bytes, &tmx, (r - 1) * tp.Wimg + 32 * run, 0, cg0, n, 0, full + s);
            } else {                                         // (pixel % 32, c % 8, run, image, c / 8)
              tma_load_5d(stage, &tmx, 0, 0, c0, c3, cg0, full + s);
            }
          }
          if (lane == 0) K3_TRACE(2, 2 * tr_it + 1);
          ++tr_it;
          if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
        }
      }
    }
  } else if (warp == KT_EPI_WARPS) {
    // =========================== MMA issuer ===========================
    const bool leader = elect_one();
    mbar_wait(bfull, 0);
    if (leader) K3_TRACE(3, 0);
    const uint32_t idesc = make_idesc_tma((uint32_t)tp.MT, acc_cols);        // N = NT, or 3 * NT (3x3: [s][n])
    constexpr uint32_t atom16 = KT_ATOM >> 4;
    // A: MN-major, SWIZZLE_128B_BASE32B (layout type 1).  lo = start >> 4 | LBO >> 4 << 16 (LBO: next 32-pixel
    //    run along M = next atom);  hi = SBO >> 4 (next 4 channels along K = half an atom) | version 1 | layout
    const uint32_t a_hi = (uint32_t)(512 >> 4) | (1u << 14) | (1u << 29);
    const uint32_t a_lo_fixed = tp.a_lbo16 << 16;
    const uint32_t a_ks16 = tp.a_ks16, a_r16 = tp.a_r16;
    (void)atom16; (void)a_r16;
    // B: K-major, no swizzle (planes of 4 channels x N rows x 16 bytes): LBO = plane, SBO = 8 rows
    const uint32_t b_plane16 = acc_cols;
    const uint32_t b_hi = 8u | (1u << 14);
    const uint32_t b_lo_fixed = b_plane16 << 16;
    const uint32_t b0_16 = smem_u32(sB) >> 4, a0_16 = smem_u32(sA) >> 4;
    const uint32_t stage16 = tp.stage_bytes >> 4;
    const int ncg4 = g.Cpad >> 2, NCGS = tp.NCGS, ncg8_total = g.Cpad >> 3;
    const uint32_t accmask = (uint32_t)tp.nacc - 1u;
    uint32_t s = 0, sphase = 0, aph = 0, tile = 0;            // aph: phase bit per accumulator
    for (int m = m_first; m < nitems; m += m_step, ++tile) {
      const uint32_t acc = tile & accmask;
      const uint32_t d = tmem_base + acc * acc_cols;
      if (leader) K3_TRACE(4, 3 * (int)tile);
      mbar_wait(tempty + acc, ((aph >> acc) & 1u) ^ 1u);       // the epilogue has drained this accumulator
      if (leader) K3_TRACE(4, 3 * (int)tile + 1);
      for (int chunk = 0; chunk < nchunk; ++chunk) {
        mbar_wait(full + s, sphase);
        if (leader && chunk == 0) K3_TRACE(4, 3 * (int)tile + 2);
        tc_fence_after();
        if (leader) {
          K3_TRACE(0, 2 * (int)(tile * nchunk + chunk));
          const uint32_t a_s16 = a0_16 + s * stage16;
          const int ksteps = min(NCGS, ncg8_total - chunk * NCGS);
          for (int ks = 0; ks < ksteps; ++ks) {
            const uint32_t cg4 = (uint32_t)((chunk * NCGS + ks) * 2);     // first of the two 4-channel planes of this k-step
            if (NTAPS == 9) {
              // one MMA per filter row: its three filter columns are N rows [s][n] of the operand and land in
              // the three accumulators Y_s = TMEM columns [s * NT, s * NT + NT)
#pragma unroll
              for (int r = 0; r < 3; ++r) {
                const uint32_t a16 = a_s16 + (uint32_t)ks * a_ks16 + (uint32_t)r * a_r16;
                const uint32_t b16 = b0_16 + ((uint32_t)r * (uint32_t)ncg4 + cg4) * b_plane16;
                const uint64_t ad = ((uint64_t)a_hi << 32) | (a_lo_fixed | (a16 & 0x3FFFu));
                const uint64_t bd = ((uint64_t)b_hi << 32) | (b_lo_fixed | (b16 & 0x3FFFu));
                umma<true>(d, ad, bd, idesc, (uint32_t)((chunk | ks | r) != 0));
              }
            } else {
              const uint32_t a16 = a_s16 + (uint32_t)ks * a_ks16;
              const uint32_t b16 = b0_16 + cg4 * b_plane16;
              const uint64_t ad = ((uint64_t)a_hi << 32) | (a_lo_fixed | (a16 & 0x3FFFu));
              const uint64_t bd = ((uint64_t)b_hi << 32) | (b_lo_fixed | (b16 & 0x3FFFu));
              umma<true>(d, ad, bd, idesc, (uint32_t)((chunk | ks) != 0));
            }
          }
          umma_commit(empty + s);                              // stage reusable once these MMAs retire
          if (chunk == nchunk - 1) umma_commit(tfull + acc);   // accumulator complete
          K3_TRACE(0, 2 * (int)(tile * nchunk + chunk) + 1);
        }
        __syncwarp();
        if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
      }
      aph ^= 1u << acc;
    }
  } else {
    // =========================== epilogue: TMEM -> scale -> NCHW fp32 ===========================
    asm volatile("griddepcontrol.wait;" ::: "memory");         // `scale` may come from the kernel in front
    const float sc = scale ? *reinterpret_cast<const volatile float*>(scale) : 1.0f;
    const int K = g.K, NT = g.NT, HW = tp.HW;
    const int kbase = nt * NT;
    // tile pixel of this thread: M = 128 -> TMEM lane = pixel; M = 64 -> lanes 0..15 of each warp's partition
    const int pix = tp.MT == 128 ? warp * 32 + lane : warp * 16 + lane;
    const bool lane_ok = tp.MT == 128 || lane < 16;
    const int atom = pix >> 5, q = pix & 31;                  // 32-pixel run inside the tile, position in the run
    const int qw = q & (tp.WB - 1);                            // pixel inside its image row
    const bool edge_l = qw == 0, edge_r = qw == tp.WB - 1;     // image-row borders inside the run (3x3 only)
    // folded BatchNorm: this CTA's NT scale / shift values are staged in shared memory once (the epilogue is on
    // the critical path: 2 x 16 broadcast global loads per thread and tile were measured to double the kernel)
    __shared__ float s_ep[2][256];                             // scale, shift
    if (ep.a) {
      for (int i = tid; i < NT; i += 32 * KT_EPI_WARPS) {
        const bool ok = kbase + i < K;
        s_ep[0][i] = ok ? __ldg(ep.a + kbase + i) : 0.f;
        s_ep[1][i] = ok ? __ldg(ep.b + kbase + i) : 0.f;
      }
      asm volatile("bar.sync 2, %0;" ::"n"(32 * KT_EPI_WARPS) : "memory");
    }
    const uint32_t accmask = (uint32_t)tp.nacc - 1u;
    uint32_t acc = 0, aphase = 0;
    int tr_item = 0;
    (void)tr_item;
    for (int m = m_first; m < nitems; m += m_step) {
      bool valid = lane_ok;
      int obase = 0;
      if (tp.mode == 0) {
        const int t = fdiv(m, tp.div_ncol);
        const int j = m - t * tp.ncol;
        const int ng = fdiv(t, tp.div_nrb);
        const int rb = t - ng * tp.nrb;
        const int n = ng, h = rb * tp.APT + atom, w = j * tp.WB + qw;
        valid = valid && h < tp.Himg && w < tp.Wimg;
        obase = (n * K + kbase) * HW + h * tp.Wimg + w;
      } else if (tp.tiles_per_img > 0) {                     // modes 1, 4: runs of one image
        const int n = fdiv(m, tp.div_tpi);
        const int pimg = ((m - n * tp.tiles_per_img) * tp.APT + atom) * 32 + q;
        valid = valid && pimg < HW;
        obase = (n * K + kbase) * HW + pimg;
      } else {                                               // modes 2, 4: whole images per tile
        const int n = m * tp.IPT + (atom >> tp.lgAH);
        const int pimg = (atom & (tp.AH - 1)) * 32 + q;
        valid = valid && n < g.B && pimg < HW;
        obase = (n * K + kbase) * HW + pimg;
      }
      // a kernel launched programmatically behind this conv may be scheduled once every CTA is at its last tile (not
      // earlier: a resident dependent that only waits takes registers and CTA slots from this grid's tail); it waits
      // for this grid's completion (griddepcontrol.wait) before it reads the output
      if (m + m_step >= nitems) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
      mbar_wait(tfull + acc, aphase);
      tc_fence_after();
      if (warp == 0 && lane == 0) K3_TRACE(1, 2 * tr_item);
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + acc * acc_cols;
      for (int cb = 0; cb < NT / 16; ++cb) {
        float v[16];
        if (NTAPS == 9) {
          // out[h][w] = Y0[h][w-1] + Y1[h][w] + Y2[h][w+1]: the pixel's neighbours sit in the adjacent TMEM
          // lanes = adjacent threads; at the first / last pixel of an image row the neighbour is padding
          uint32_t y0[16], y1[16], y2[16];
          tmem_ld16_issue(trow + (uint32_t)cb * 16, y0);
          tmem_ld16_issue(trow + (uint32_t)(NT + cb * 16), y1);
          tmem_ld16_issue(trow + (uint32_t)(2 * NT + cb * 16), y2);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            const float l = __shfl_up_sync(0xFFFFFFFFu, __uint_as_float(y0[j]), 1);
            const float r = __shfl_down_sync(0xFFFFFFFFu, __uint_as_float(y2[j]), 1);
            v[j] = ((edge_l ? 0.f : l) + __uint_as_float(y1[j]) + (edge_r ? 0.f : r)) * sc;
          }
        } else {
          uint32_t r[16];
          tmem_ld16(trow + (uint32_t)cb * 16, r);
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]) * sc;
        }
        if (valid) {
          float* po = out + obase + cb * 16 * HW;
          const int kleft = K - (kbase + cb * 16);
          if (ep.a) {                                          // BatchNorm (+ residual) (+ activation)
            float rs[16];
            if (ep.res) {
              const float* pr = ep.res + obase + cb * 16 * HW;
#pragma unroll
              for (int j = 0; j < 16; ++j) rs[j] = j < kleft ? __ldg(pr + j * HW) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              float t = fmaf(v[j], s_ep[0][cb * 16 + j], s_ep[1][cb * 16 + j]);   // folded eval-mode norm
              if (ep.res) t += rs[j];
              v[j] = conv_act(t, ep.act);
            }
          }
          if (kleft >= 16) {
#pragma unroll
            for (int j = 0; j < 16; ++j) po[j * HW] = v[j];
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j < kleft) po[j * HW] = v[j];
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty + acc);
      if (warp == 0 && lane == 0) K3_TRACE(1, 2 * tr_item + 1);
      ++tr_item;
      acc = (acc + 1) & accmask;
      aphase ^= (acc == 0);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) K3_TRACE(6, 2);
#ifdef PO2_K3_TRACE
  __syncthreads();
  if (g_k3_trace && blockIdx.x < 4)
    for (int i = tid; i < 8 * 64; i += KT_THREADS) g_k3_trace[blockIdx.x * 8 * 64 + i] = k3_trace_smem[i];
#endif
  if (warp == KT_EPI_WARPS) tmem_dealloc(tmem_base, ncols);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tma_encoder() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return (EncodeTiledFn)p;
  }();
  return fn;
}

static size_t tma_smem_bytes(const ConvGeom& g, const TmaPlan& tp) {
  return (size_t)g.b_slab_bytes + 1024 + (size_t)tp.nst * tp.stage_bytes + (2 * K3_MAX_STAGES + 2 * KT_MAX_ACC + 4) * 8 + 64;
}

// g: through plan_umma(g, tf32 = true) (supplies the weight-operand plan NT / ntiles_n / Cpad / slab bytes,
// so that every existing pack path feeds this kernel unchanged).  False: shape stays on the register-fed kernel.
static bool plan_tma(const ConvGeom& g, TmaPlan& tp) {
  if (!g.tf32 || g.groups != 1 || g.stride != 1 || !tc_window(g.R, g.S, g.pad)) return false;
  if (g.C % 8 || g.Cpad != g.C) return false;
  tp = TmaPlan{};
  tp.ntaps = g.R * g.S;
  tp.HW = g.H * g.W;
  const int sms = sm_count();
  tp.WB = 32; tp.IPR = 1;
  if (tp.ntaps == 9) {
    tp.Himg = g.H; tp.Wimg = g.W;
    if (g.W % 4 || g.W > 32) return false;                   // tensor-map strides are multiples of 16 bytes; one run per row
    if (g.W > 16) tp.mode = 0;
    else if (g.W == 16 || g.W == 8 || g.W == 4) { tp.mode = 4; tp.WB = g.W; tp.AH = (tp.HW + 31) / 32; }
    else return false;
  } else {
    tp.Himg = 1; tp.Wimg = tp.HW;
    if (tp.HW % 32) return false;
    tp.mode = 1; tp.AH = tp.HW / 32;
  }
  tp.lgWB = tp.WB == 32 ? 5 : (tp.WB == 16 ? 4 : (tp.WB == 8 ? 3 : 2));
  // tile height: 128 pixels unless that leaves SMs without a tile
  auto count_items = [&](int MT) -> int {
    const int APT = MT / 32;
    if (tp.mode == 0) return g.B * ((g.H + APT - 1) / APT);
    if (tp.AH >= APT) return g.B * ((tp.AH + APT - 1) / APT);
    return (g.B + APT / tp.AH - 1) / (APT / tp.AH);
  };
  // (a 64-pixel tile puts half a run in each epilogue warp: for 3x3 only when an image row is <= 16 pixels,
  // so that no pixel's horizontal neighbour lives in another warp)
  tp.MT = 128;
  if (count_items(128) * g.ntiles_n < sms && count_items(64) > count_items(128) && (tp.ntaps == 1 || tp.WB <= 16)) tp.MT = 64;
  const int accw = (tp.ntaps == 9 ? 3 : 1) * g.NT;
  if (accw > 256) return false;                              // one MMA spans the accumulator row (N <= 256)
  tp.nacc = 2 * accw <= 512 ? 2 : 1;
  tp.APT = tp.MT / 32;
  tp.rows_st = tp.APT + (tp.mode == 0 ? 2 : 0);
  tp.nitems_m = count_items(tp.MT);
  if (tp.mode == 0) {
    tp.ncol = 1;
    tp.nrb = (g.H + tp.APT - 1) / tp.APT;
    tp.ngrp = g.B;
  } else if (tp.AH >= tp.APT) {
    tp.tiles_per_img = (tp.AH + tp.APT - 1) / tp.APT;
  } else {
    if (tp.AH > 2) return false;                            // AH is 1 or 2 here (APT <= 4)
    if (tp.mode == 1) tp.mode = 2;
    tp.lgAH = tp.AH == 1 ? 0 : 1;
    tp.IPT = tp.APT / tp.AH;
  }
  const int ncg = g.C / 8;
  const size_t per_group = (size_t)(tp.mode == 4 ? 3 * tp.APT : tp.rows_st) * KT_ATOM;   // stage bytes per 8 channels
  int NCGS = ncg;
  while (NCGS > 1 && NCGS * per_group > KT_STAGE_TARGET) --NCGS;
  // balance the chunks (a box always carries NCGS groups; channel groups past C are TMA zero fill)
  tp.nchunk = (ncg + NCGS - 1) / NCGS;
  NCGS = (ncg + tp.nchunk - 1) / tp.nchunk;
  if (NCGS > 256) return false;
  tp.NCGS = NCGS;
  tp.cg_bytes = (uint32_t)tp.rows_st * KT_ATOM;
  tp.stage_bytes = (uint32_t)(NCGS * per_group);
  if (tp.mode == 4) {        // [row copy][run][channel group][8][32]
    tp.a_lbo16 = (uint32_t)NCGS * (KT_ATOM >> 4); tp.a_ks16 = KT_ATOM >> 4; tp.a_r16 = (uint32_t)(tp.APT * NCGS) * (KT_ATOM >> 4);
  } else {                   // [channel group][run (+ halo)][8][32]
    tp.a_lbo16 = KT_ATOM >> 4; tp.a_ks16 = tp.cg_bytes >> 4; tp.a_r16 = tp.mode == 0 ? (KT_ATOM >> 4) : 0;
  }
  const size_t fixed = (size_t)g.b_slab_bytes + 1024 + (2 * K3_MAX_STAGES + 2 * KT_MAX_ACC + 4) * 8 + 64;
  if (fixed + 2 * (size_t)tp.stage_bytes > KT_SMEM_BUDGET) return false;
  // Two CTAs per SM when both fit (shared memory, 2 x TMEM columns <= 512) and there are tiles for them: the
  // kernel is bound by the serial latency of its single-thread roles (mbarrier waits, MMA issue), which a
  // second resident CTA hides.
  uint32_t ncols = 32;
  while (ncols < (uint32_t)(tp.nacc * accw)) ncols <<= 1;
  size_t budget = KT_SMEM_BUDGET;
  tp.cps = 1;
  if (fixed + 3 * (size_t)tp.stage_bytes <= KT_SMEM_BUDGET_2 && 2 * ncols <= 512 && tp.nitems_m * g.ntiles_n > sms &&
      !(getenv("PO2_TMA_CPS") && getenv("PO2_TMA_CPS")[0] == '1')) {
    tp.cps = 2;
    budget = KT_SMEM_BUDGET_2;
  }
  int nst = (int)((budget - fixed) / tp.stage_bytes);
  if (nst > K3_MAX_STAGES) nst = K3_MAX_STAGES;
  tp.nst = nst;
  int per_n = tp.cps * sms / g.ntiles_n;
  if (per_n < 1) per_n = 1;
  tp.m_step = tp.nitems_m < per_n ? tp.nitems_m : per_n;
  tp.div_ncol = make_fastdiv((uint32_t)(tp.ncol > 0 ? tp.ncol : 1));
  tp.div_nrb = make_fastdiv((uint32_t)(tp.nrb > 0 ? tp.nrb : 1));
  tp.div_tpi = make_fastdiv((uint32_t)(tp.tiles_per_img > 0 ? tp.tiles_per_img : 1));
  { const char* e = getenv("PO2_TMA_DEBUG"); tp.debug = e ? atoi(e) : 0; }
  return tma_encoder() != nullptr;
}

static bool encode_x_map(CUtensorMap* tm, const void* x, const ConvGeom& g, const TmaPlan& tp) {
  EncodeTiledFn enc = tma_encoder();
  if (!enc || (reinterpret_cast<uintptr_t>(x) & 15)) return false;
  const cuuint64_t HW = (cuuint64_t)tp.HW, C = (cuuint64_t)g.C, B = (cuuint64_t)g.B;
  cuuint64_t dims[5], strides[4];
  cuuint32_t box[5], estr[5] = {1, 1, 1, 1, 1};
  if (tp.mode == 0) {
    // (w, image, c % 8, h, c / 8)
    dims[0] = (cuuint64_t)tp.Wimg; dims[1] = B; dims[2] = 8; dims[3] = (cuuint64_t)tp.Himg; dims[4] = C / 8;
    strides[0] = C * HW * 4; strides[1] = HW * 4; strides[2] = (cuuint64_t)tp.Wimg * 4; strides[3] = 8 * HW * 4;
    box[0] = 32; box[1] = 1; box[2] = 8; box[3] = (cuuint32_t)tp.rows_st; box[4] = (cuuint32_t)tp.NCGS;
  } else if (tp.mode == 4) {
    // (flat pixel, c % 8, c / 8, image, 1): one run of 32 pixels x all channel groups of the stage per box
    dims[0] = HW; dims[1] = 8; dims[2] = C / 8; dims[3] = B; dims[4] = 1;
    strides[0] = HW * 4; strides[1] = 8 * HW * 4; strides[2] = C * HW * 4; strides[3] = B * C * HW * 4;
    box[0] = 32; box[1] = 8; box[2] = (cuuint32_t)tp.NCGS; box[3] = 1; box[4] = 1;
  } else {
    // (pixel % 32, c % 8, pixel / 32, image, c / 8)
    dims[0] = 32; dims[1] = 8; dims[2] = (cuuint64_t)tp.AH; dims[3] = B; dims[4] = C / 8;
    strides[0] = HW * 4; strides[1] = 128; strides[2] = C * HW * 4; strides[3] = 8 * HW * 4;
    box[0] = 32; box[1] = 8;
    box[2] = (cuuint32_t)(tp.mode == 1 ? tp.APT : tp.AH);
    box[3] = (cuuint32_t)(tp.mode == 1 ? 1 : tp.IPT);
    box[4] = (cuuint32_t)tp.NCGS;
  }
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<void*>(x), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// the conv launch behind the packed operand (same contract as the register-fed launch in launch_conv)
static int launch_tma(const void* x, const uint8_t* Bp, const float* scale, void* out, const ConvGeom& g, const TmaPlan& tp_in,
                      cudaStream_t st, int pdl, const ConvEpilogue& ep) {
  TmaPlan tp = tp_in;
  tp.pdl = pdl;
  CUtensorMap tm;
  if (!encode_x_map(&tm, x, g, tp)) return PO2_E_UNSUPPORTED;
  static PerDeviceOnce attr_once;
  cudaError_t e = attr_once.run([]() -> cudaError_t {
    const int smax = (int)KT_SMEM_BUDGET + 1024;
    cudaError_t a = cudaSuccess;
    const void* kerns[2] = {(const void*)conv_tma_kernel<1>, (const void*)conv_tma_kernel<9>};
    for (int i = 0; i < 2 && a == cudaSuccess; ++i) {
      // dynamic + static shared memory <= 227 KB per CTA
      cudaFuncAttributes fa;
      a = cudaFuncGetAttributes(&fa, kerns[i]);
      if (a != cudaSuccess) break;
      const int room = 227 * 1024 - (int)fa.sharedSizeBytes;
      a = cudaFuncSetAttribute(kerns[i], cudaFuncAttributeMaxDynamicSharedMemorySize, smax < room ? smax : room);
      if (a == cudaSuccess) a = cudaFuncSetAttribute(kerns[i], cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    }
    return a;
  });
  if (e != cudaSuccess) return (int)e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(g.ntiles_n * tp.m_step));
  cfg.blockDim = dim3(KT_THREADS);
  cfg.dynamicSmemBytes = tma_smem_bytes(g, tp);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  float* of = (float*)out;
  if (tp.ntaps == 1) e = cudaLaunchKernelEx(&cfg, conv_tma_kernel<1>, tm, Bp, scale, of, g, tp, ep);
  else e = cudaLaunchKernelEx(&cfg, conv_tma_kernel<9>, tm, Bp, scale, of, g, tp, ep);
  return (int)e;
}

}  // namespace po2
