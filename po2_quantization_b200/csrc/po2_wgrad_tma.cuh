// K5T: the TMA-fed tf32 weight gradient (included by po2_conv.cu, same namespace).
//
//   gw[k][c][r][s] = sum over (n, h, w) of  go[n][k][h][w] * x[n][c][h + r - 1][w + s - 1]
//
// the autograd of models/quantized_conv.py:36 with respect to the weight; through the straight-through
// estimator (utils/quantizers.py:34-36) it is the gradient of the fp32 master weight.  A GEMM whose
// reduction index is the pixel: D[k][(r, s, c)] += go^T x_(r,s).  In fp32 NCHW the pixel index is the
// contiguous one for BOTH operands, i.e. both are "K-major" as they lie in memory, and kind::tf32 reads fp32
// containers as they are -- so nothing is converted or transposed:
//   * go: tensor-map TMA (SWIZZLE_128B) drops runs of 32 consecutive pixels x 8 channels as the canonical
//     K-major 128-byte-swizzle atoms (8 rows of 128 bytes); a k-step (K = 8 pixels) is a 32-byte advance of
//     the descriptor start inside the atom.  (A 32-byte-swizzle layout with one 256-byte atom per k-step was
//     measured too: the MMAs are compute-bound either way -- M = 64 tf32 runs at ~950 MAC/cycle -- but the
//     TMA unit moves 32-byte rows at 16 B/cycle/SM against 31 B/cycle/SM for 128-byte rows,
//     tools/probes/tma_rate.cu.)
//   * x: the same, once per filter ROW (the run of row copy r starts (r-1)*W pixels earlier/later; pixels
//     outside the image plane are TMA zero fill);
//   * a filter COLUMN is a shift by one pixel = 4 bytes, which neither TMA (16-byte box starts) nor an MMA
//     descriptor can express: four warps derive the two shifted copies from the TMA-written one inside
//     shared memory (LDS.128, two lane shuffles, two STS.128 per 16 bytes, zeroing the image-row borders).
// The nine (row, column) variants of a run sit 1 KB apart in the order (r, s, channel group), so ONE MMA per
// 8-pixel k-step covers all taps (N = 9*C <= 256, else one per filter row).  A CTA accumulates all its tiles in
// TMEM and writes one partial [tap][k][c]; conv_wgrad_reduce_kernel adds the partials in a fixed order
// (deterministic).  When 9*C accumulator columns exceed TMEM's 512 the filter rows are split over blockIdx.y.
//
// Roles (6 warps): warps 0-3 column shifters, then the epilogue; warp 4 MMA issuer + TMEM owner; warp 5 TMA.
#pragma once

namespace po2 {

struct WgTmaPlan {
  int ntaps;                 // 9 (3x3 pad 1) or 1 (1x1 pad 0); stride 1
  int K, C, KG, NCG;         // out / in channels and their 8-channel groups
  int W, HW, B;
  int RPI, lgRPI;            // 32-pixel runs per image
  int APT;                   // runs per tile (pipeline stage)
  int tiles_per_img, IPT;    // tiles per image (a tile never spans images; IPT unused)
  int nitems, m_ctas;
  int M;                     // MMA M: 64 (K <= 64) or 128
  int rsplit;                // 3: the filter rows are split over blockIdx.y (TMEM columns), else 1
  int nrv;                   // filter rows per CTA: 3, or 1 (rsplit == 3 or 1x1)
  int nsplit;                // MMAs per k-step: 1 (N = nrv*3*C) or nrv (N = 3*C each)
  int nst;
  int merged;                // W == 32 / 1x1: a filter row is a whole run, so ONE box per operand variant spans the
                             // tile's runs ([c/8][run][8][128 B]); else one box per run ([run][variant][c/8][8][128 B])
  uint32_t g_run_bytes, x_run_bytes;                // distance between the runs of go / of an x variant
  uint32_t sbo_bytes;                               // distance between 8-channel groups (descriptor SBO)
  int shift_units, shift_lines;                     // shifter: blocks of consecutive 128-byte lines per filter row variant
  uint32_t copy_bytes, x_rv_bytes;                  // one (filter row, column) variant of a run; the 3 variants of a filter row
  uint32_t g_bytes, stage_bytes, tx_bytes;
  uint32_t ncols;
  int nacc;                  // independent accumulators (k-steps alternate between them; summed in the epilogue)
  int debug;                 // PO2_WT_DEBUG bit mask (1: shifters idle, 2: no MMAs, 4: shifters load only, 8: no fence)
  FastDiv div_tpi;
};

constexpr int WT_THREADS = 32 * 6;
constexpr uint32_t WT_SMEM_BUDGET = 220 * 1024;
constexpr uint32_t WT_STAGE_TARGET = 104 * 1024;   // default; PO2_WT_STAGE_KB overrides (tuning)

__device__ __forceinline__ unsigned long long global_ns_wt() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// instruction descriptor: D = f32, A = B = tf32, both K-major, M, N
__device__ __forceinline__ uint32_t make_idesc_wt(uint32_t m, uint32_t n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

__global__ void __launch_bounds__(WT_THREADS, 1) conv_wgrad_tma_kernel(const __grid_constant__ CUtensorMap tmg,
                                                                       const __grid_constant__ CUtensorMap tmx,
                                                                       float* __restrict__ partial, WgTmaPlan wp,
                                                                       float* __restrict__ gw, unsigned int* tickets) {
  extern __shared__ __align__(128) uint8_t smem[];
  const uint32_t smem_base = smem_u32(smem);
  uint8_t* sS = smem + (((smem_base + 1023u) & ~1023u) - smem_base);          // stages: 1 KB aligned swizzle atoms
  uint64_t* bars = reinterpret_cast<uint64_t*>(sS + (size_t)wp.nst * wp.stage_bytes + 8192);   // 8 KB slack: see A rows >= K
  uint64_t* tfull_tma = bars;                   // [nst] TMA -> shifters (or MMA when there is nothing to shift)
  uint64_t* full = bars + K3_MAX_STAGES;        // [nst] shifters -> MMA
  uint64_t* empty = bars + 2 * K3_MAX_STAGES;   // [nst] MMA (commit) -> TMA
  uint64_t* dfull = bars + 3 * K3_MAX_STAGES;   // accumulators complete
  uint64_t* tready = dfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tready + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#ifdef PO2_K3_TRACE
  for (int i = tid; i < 8 * 64; i += WT_THREADS) k3_trace_smem[i] = 0;
  __syncthreads();
#endif
  if (tid == 0) K3_TRACE(6, 0);
  const int nst = wp.nst, nitems = wp.nitems, m_first = blockIdx.x, m_step = wp.m_ctas;
  const bool shift = wp.ntaps == 9;
  // conv_wgrad_reduce_kernel (programmatic launch) may be scheduled early; it waits for this grid's completion
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp == 5) {
    if (lane == 0) { tma_prefetch_desc(&tmg); tma_prefetch_desc(&tmx); }
    if (lane < nst) mbar_init(tfull_tma + lane, 1);
    else if (lane < 2 * nst) mbar_init(full + (lane - nst), 4);
    else if (lane < 3 * nst) mbar_init(empty + (lane - 2 * nst), 1);
    else if (lane == 3 * nst) mbar_init(dfull, 1);
    else if (lane == 3 * nst + 1) mbar_init(tready, 1);
    fence_mbar_init();
    __syncwarp();
    asm volatile("bar.arrive 1, %0;" ::"n"(WT_THREADS) : "memory");
  } else {
    asm volatile("bar.sync 1, %0;" ::"n"(WT_THREADS) : "memory");
  }
  uint32_t tmem_base = 0;
  if (warp == 4) {
    tmem_alloc(tmem_slot, wp.ncols);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(tready);
    tc_fence_after();
    tmem_base = *tmem_slot;
  }
  if (tid == 0) K3_TRACE(6, 1);

  if (warp == 5) {
    // =========================== TMA producer ===========================
    // One box per (run, operand variant): APT * (1 + nrv) <= 16 per stage.  An issue costs a thread ~150 cycles,
    // so the boxes are spread over the lanes of the warp (lane i issues box i of every stage).
    {
      const int nbox = (wp.merged ? 1 : wp.APT) * (1 + wp.nrv);
      const int j = lane / (1 + wp.nrv), which = lane - j * (1 + wp.nrv);       // which == 0: go, else x row copy which-1
      uint32_t s = 0, sphase = 0;
      int tr = 0;
      (void)tr;
      for (int m = m_first; m < nitems; m += m_step, ++tr) {
        if (lane == 0) {
          mbar_wait(empty + s, sphase ^ 1);
          K3_TRACE(2, 2 * tr);
          mbar_expect_tx(tfull_tma + s, wp.tx_bytes);
        }
        __syncwarp();
        if (lane < nbox) {
          uint8_t* stage = sS + (size_t)s * wp.stage_bytes;
          const int n = fdiv(m, wp.div_tpi);
          const int p0 = ((m - n * wp.tiles_per_img) * wp.APT + j) * 32;            // first pixel of the run
          const int rv = which - 1;
          const int r = shift ? (wp.rsplit == 3 ? (int)blockIdx.y : rv) : 1;
          // the TMA-written x copy is the centre column (s = 1) of filter row r
          uint8_t* xdst = stage + wp.g_bytes + (size_t)rv * wp.x_rv_bytes + (shift ? (size_t)wp.copy_bytes : 0);
          if (wp.merged) {
            // (pixel % 32, c % 8, run, c / 8, image): runs outside the image plane are zero fill
            const int run0 = p0 >> 5;
            if (which == 0) tma_load_5d(stage, &tmg, 0, 0, run0, 0, n, tfull_tma + s);
            else tma_load_5d(xdst, &tmx, 0, 0, run0 + (r - 1), 0, n, tfull_tma + s);
          } else {
            // (flat pixel, c % 8, c / 8, image, -): pixels outside the image plane are zero fill
            if (which == 0) tma_load_5d(stage + (size_t)j * wp.g_run_bytes, &tmg, p0, 0, 0, n, 0, tfull_tma + s);
            else tma_load_5d(xdst + (size_t)j * wp.x_run_bytes, &tmx, p0 + (r - 1) * wp.W, 0, 0, n, 0, tfull_tma + s);
          }
        }
        if (lane == 0) K3_TRACE(2, 2 * tr + 1);
        if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
      }
    }
  } else if (warp == 4) {
    // =========================== MMA issuer ===========================
    const bool leader = elect_one();
    const uint32_t nwidth = (uint32_t)((wp.nsplit == 1 ? wp.nrv : 1) * (shift ? 3 : 1) * wp.C);   // N of one MMA
    const uint32_t idesc = make_idesc_wt((uint32_t)wp.M, nwidth);
    const uint32_t acc_stride = (uint32_t)(wp.nrv * (shift ? 3 : 1) * wp.C);
    // K-major, 128-byte swizzle (layout type 2): SBO = distance between 8-row (channel) groups; LBO unused
    const uint32_t d_hi = (wp.sbo_bytes >> 4) | (1u << 14) | (2u << 29);
    const uint32_t lo_fixed = 1u << 16;
    const uint32_t s0_16 = smem_u32(sS) >> 4, stage16 = wp.stage_bytes >> 4, g_run16 = wp.g_run_bytes >> 4;
    const uint32_t x0_16 = wp.g_bytes >> 4, x_run16 = wp.x_run_bytes >> 4, x_rv16 = wp.x_rv_bytes >> 4;
    uint64_t* fullbar = shift ? full : tfull_tma;
    uint32_t s = 0, sphase = 0, tile = 0;
    for (int m = m_first; m < nitems; m += m_step, ++tile) {
      mbar_wait(fullbar + s, sphase);
      tc_fence_after();
      if (leader) {
        K3_TRACE(0, 2 * (int)tile);
        const uint32_t st16 = s0_16 + s * stage16;
        for (int j = 0; j < wp.APT; ++j) {
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {                       // 8 pixels (32 bytes) per MMA
            const uint32_t a16 = st16 + (uint32_t)j * g_run16 + (uint32_t)ks * 2u;          // k-step: 32 bytes into the atom rows
            const uint64_t ad = ((uint64_t)d_hi << 32) | (lo_fixed | (a16 & 0x3FFFu));
            for (int q = 0; q < wp.nsplit; ++q) {
              const uint32_t b16 = st16 + x0_16 + (uint32_t)j * x_run16 + (uint32_t)q * x_rv16 + (uint32_t)ks * 2u;
              const uint64_t bd = ((uint64_t)d_hi << 32) | (lo_fixed | (b16 & 0x3FFFu));
              // consecutive k-steps go to different accumulators: an MMA that accumulates into the tile its
              // predecessor wrote waits for it (measured ~100-150 cycles per dependent N = 144 MMA)
              const uint32_t acc = (uint32_t)ks & (uint32_t)(wp.nacc - 1);
              if (!(wp.debug & 2))
                umma<true>(tmem_base + acc * acc_stride + (uint32_t)q * nwidth, ad, bd, idesc,
                           (uint32_t)((tile | (uint32_t)j) != 0 || ks >= wp.nacc));
            }
          }
        }
        umma_commit(empty + s);
        K3_TRACE(0, 2 * (int)tile + 1);
      }
      __syncwarp();
      if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
    }
    if (leader) umma_commit(dfull);
    __syncwarp();
  } else {
    // =========================== column shifters (warps 0-3), then the epilogue ===========================
    if (shift) {
      // A channel row of a run = one 128-byte line = 8 lanes x float4 (so every quarter-warp reads / writes one
      // whole line: no bank conflicts); 16 lane groups take the 8 * NCG lines of a (run, filter row) variant.
      const int grp = warp * 4 + (lane >> 3);                    // 0..15
      const int sub = lane & 7;                                  // 4 pixels of the run
      const int Wm = wp.W - 1;
      // the first pixel of the chunk starts an image row / its last pixel ends one: the neighbour is padding
      const bool zl = ((4 * sub) & Wm) == 0, zr = ((4 * sub + 4) & Wm) == 0;
      const uint32_t copy = wp.copy_bytes;
      const int nlines = wp.shift_lines, nrv = wp.nrv;
      uint32_t s = 0, sphase = 0;
      int tr = 0;
      (void)tr;
      for (int m = m_first; m < nitems; m += m_step, ++tr) {
        mbar_wait(tfull_tma + s, sphase);
        if (tid == 0) K3_TRACE(1, 2 * tr);
        uint8_t* xs = sS + (size_t)s * wp.stage_bytes + wp.g_bytes + copy;       // centre copy of run 0, filter row variant 0
        for (int ln = grp; ln < nlines && !(wp.debug & 1); ln += 16) {
          const uint32_t off = (uint32_t)ln * 128u + (uint32_t)((sub ^ (ln & 7)) << 4);   // SWIZZLE_128B: chunk ^ (line & 7)
          for (int u = 0; u < wp.shift_units; ++u) {
            uint8_t* base = xs + (size_t)u * wp.x_run_bytes + off;
            float4 v[3];
#pragma unroll
            for (int rv = 0; rv < 3; ++rv)
              if (rv < nrv) v[rv] = *reinterpret_cast<const float4*>(base + (size_t)rv * wp.x_rv_bytes);
#pragma unroll
            for (int rv = 0; rv < 3; ++rv)
              if (rv < nrv) {
                float left = __shfl_up_sync(0xFFFFFFFFu, v[rv].w, 1, 8);
                float right = __shfl_down_sync(0xFFFFFFFFu, v[rv].x, 1, 8);
                if (zl) left = 0.f;
                if (zr) right = 0.f;
                uint8_t* c = base + (size_t)rv * wp.x_rv_bytes;
                // column s = 0 reads x[w - 1], column s = 2 reads x[w + 1]
                if (!(wp.debug & 4) || left == 12345.f) {
                  *reinterpret_cast<float4*>(c - copy) = make_float4(left, v[rv].x, v[rv].y, v[rv].z);
                  *reinterpret_cast<float4*>(c + copy) = make_float4(v[rv].y, v[rv].z, v[rv].w, right);
                }
              }
          }
        }
        if (!(wp.debug & 8)) fence_proxy_async();                // generic-proxy smem writes -> tensor-core reads
        __syncwarp();
        if (lane == 0) mbar_arrive(full + s);
        if (tid == 0) K3_TRACE(1, 2 * tr + 1);
        if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
      }
    }
    // ---- epilogue: TMEM -> partial[cta][tap][k][c]
    mbar_wait(tready, 0);
    tc_fence_after();
    tmem_base = *tmem_slot;
    mbar_wait(dfull, 0);
    tc_fence_after();
    if (tid == 0) K3_TRACE(3, 0);
    const int K = wp.K, C = wp.C;
    const int rows_per_warp = wp.M == 64 ? 16 : 32;
    if (warp * rows_per_warp < K) {
      const int k = lane < rows_per_warp ? warp * rows_per_warp + lane : K;
      const int ntap_cta = wp.nrv * (shift ? 3 : 1);
      const int tap0 = wp.rsplit == 3 ? 3 * (int)blockIdx.y : 0;
      // partial[cta][tap][k][c]; 32-bit index arithmetic, loads batched three column blocks deep (often a single
      // warp runs this epilogue alone, so every instruction's latency is exposed)
      float* prow0 = partial + ((size_t)blockIdx.x * wp.ntaps + tap0) * C * K + (k < K ? k : 0) * C;
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16);
      if ((C & 15) == 0) {
        const int cbt = C >> 4, nblk = ntap_cta * cbt;           // 16-column blocks; a block never straddles a tap
        for (int b0 = 0; b0 < nblk; b0 += 3) {
          uint32_t r[3][16];
#pragma unroll
          for (int u = 0; u < 3; ++u)
            if (b0 + u < nblk) tmem_ld16_issue(trow + (uint32_t)((b0 + u) * 16), r[u]);
          tmem_ld_wait();
          for (int a2 = 1; a2 < wp.nacc; ++a2) {                 // the other accumulators of the same columns
            uint32_t r2[3][16];
#pragma unroll
            for (int u = 0; u < 3; ++u)
              if (b0 + u < nblk) tmem_ld16_issue(trow + (uint32_t)(a2 * ntap_cta * C + (b0 + u) * 16), r2[u]);
            tmem_ld_wait();
#pragma unroll
            for (int u = 0; u < 3; ++u)
#pragma unroll
              for (int e = 0; e < 16; ++e) r[u][e] = __float_as_uint(__uint_as_float(r[u][e]) + __uint_as_float(r2[u][e]));
          }
          if (k < K) {
#pragma unroll
            for (int u = 0; u < 3; ++u)
              if (b0 + u < nblk) {
                const int t = (b0 + u) / cbt, cb = (b0 + u) - t * cbt;
                float* prow = prow0 + t * (K * C) + cb * 16;
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4)
                  *reinterpret_cast<uint4*>(prow + 4 * q4) = make_uint4(r[u][4 * q4], r[u][4 * q4 + 1], r[u][4 * q4 + 2], r[u][4 * q4 + 3]);
              }
          }
        }
      } else {
        const int ncol = ntap_cta * C;
        for (int cb = 0; cb < (ncol + 15) / 16; ++cb) {
          uint32_t r[16];
          tmem_ld16(trow + (uint32_t)(cb * 16), r);
          if (k < K) {
#pragma unroll
            for (int q4 = 0; q4 < 4; ++q4) {                      // C % 8 == 0: a group of 4 columns never straddles a tap
              const int col = cb * 16 + q4 * 4;
              if (col < ncol) {
                const int t = col / C, c = col - t * C;
                *reinterpret_cast<uint4*>(prow0 + t * (K * C) + c) = make_uint4(r[4 * q4], r[4 * q4 + 1], r[4 * q4 + 2], r[4 * q4 + 3]);
              }
            }
          }
        }
      }
    }
    tc_fence_before();
  }
  tc_fence_before();
  if (gw) {
    // ---- fused fixed-order reduction of the partials (instead of a second launch): a grid barrier (the grid
    // is launched cooperatively: every CTA is resident), then CTA i adds the m_ctas partials of its slice of
    // the [tap][k][c] outputs in partial order -- the same sums in the same order as conv_wgrad_reduce_kernel.
    __threadfence();
    __syncthreads();
    const unsigned int nctas = gridDim.x * gridDim.y;
    if (tid == 0) {
      atomicAdd(tickets, 1u);
      const unsigned long long t0 = global_ns_wt();
      while (*reinterpret_cast<volatile unsigned int*>(tickets) < nctas) {
        if (global_ns_wt() - t0 > 2000000000ull) break;          // never hang the GPU (the result is then incomplete)
        __nanosleep(32);
      }
      __threadfence();
    }
    __syncthreads();
    const int n = wp.ntaps * wp.C * wp.K, P = wp.m_ctas;
    const int cta = (int)(blockIdx.y * gridDim.x + blockIdx.x);
    const int per = (n + (int)nctas - 1) / (int)nctas;
    const int o0 = cta * per;
    const int cnt = max(0, min(per, n - o0));
    int L = 1;
    while (L < 32 && 2 * L * cnt <= WT_THREADS) L <<= 1;           // lanes per output (cnt * L <= threads), or 1
    float* scratch = reinterpret_cast<float*>(sS);                 // the stages are idle now
    for (int base = 0; base < cnt * L; base += WT_THREADS) {
      const int idx = base + tid;
      const bool live = idx < cnt * L;
      const int o = o0 + (live ? idx / L : 0), l = live ? idx % L : 0;
      float acc = 0.f;
      if (live) {
        const float* src = partial + o;
        int p = l;
        for (; p + 3 * L < P; p += 4 * L) {                        // four independent loads per round, fixed order
          const float v0 = __ldcg(src + (size_t)p * n), v1 = __ldcg(src + (size_t)(p + L) * n);
          const float v2 = __ldcg(src + (size_t)(p + 2 * L) * n), v3 = __ldcg(src + (size_t)(p + 3 * L) * n);
          acc += v0; acc += v1; acc += v2; acc += v3;
        }
        for (; p < P; p += L) acc += __ldcg(src + (size_t)p * n);
      }
      if (L > 1) {
        scratch[tid] = acc;
        __syncthreads();
        if (live && l == 0) {
          float t = 0.f;
          for (int q = 0; q < L; ++q) t += scratch[tid + q];
          acc = t;
        }
        __syncthreads();
      }
      if (live && l == 0) {
        const int c = o % wp.C, tk = o / wp.C, k = tk % wp.K, tap = tk / wp.K;
        gw[((size_t)k * wp.C + c) * wp.ntaps + tap] = acc;
      }
    }
    __syncthreads();
    if (tid == 0) {                                                // self-resetting: the last CTA to leave clears both counters
      const unsigned int d = atomicAdd(tickets + 1, 1u);
      if (d == nctas - 1) { tickets[0] = 0u; tickets[1] = 0u; __threadfence(); }
    }
  }
  __syncthreads();
  if (tid == 0) K3_TRACE(6, 2);
#ifdef PO2_K3_TRACE
  __syncthreads();
  if (g_k3_trace && blockIdx.x < 4 && blockIdx.y == 0)
    for (int i = tid; i < 8 * 64; i += WT_THREADS) g_k3_trace[blockIdx.x * 8 * 64 + i] = k3_trace_smem[i];
#endif
  if (warp == 4) tmem_dealloc(tmem_base, wp.ncols);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static bool plan_wgrad_tma(WgTmaPlan& wp, int B, int C, int H, int W, int K, int R, int S, int pad) {
  if (!tc_window(R, S, pad)) return false;
  if (C % 8 || K % 8 || K > 128 || C > 256) return false;
  wp = WgTmaPlan{};
  wp.ntaps = R * S;
  wp.K = K; wp.C = C; wp.KG = K / 8; wp.NCG = C / 8;
  wp.W = W; wp.HW = H * W; wp.B = B;
  if (wp.HW % 4) return false;                                 // tensor-map strides are multiples of 16 bytes
  if (wp.ntaps == 9 && !(W == 32 || W == 16 || W == 8 || W == 4)) return false;   // a run holds whole image rows
  if (wp.ntaps == 1) wp.W = 32;
  wp.RPI = (wp.HW + 31) / 32;
  if (!index_fits(B, C, wp.HW, K, wp.HW)) return false;
  const int sms = sm_count();
  // accumulator columns: all nine taps in one CTA, else the filter rows over blockIdx.y
  const int taps_w = wp.ntaps == 9 ? 3 : 1;
  wp.rsplit = (wp.ntaps == 9 && 9 * C > 512) ? 3 : 1;
  wp.nrv = (wp.ntaps == 9 && wp.rsplit == 1) ? 3 : 1;
  if (wp.nrv * taps_w * C > 512) return false;
  wp.nsplit = (wp.nrv * taps_w * C <= 256) ? 1 : wp.nrv;
  if ((wp.nsplit == 1 ? wp.nrv : 1) * taps_w * C > 256) return false;
  wp.nacc = 1;
  { const char* e = getenv("PO2_WT_NACC");
    const int want = e ? atoi(e) : 1;          // measured: no gain from splitting the accumulation (profiles/r02 notes)
    while (wp.nacc * 2 <= want && wp.nacc * 2 * wp.nrv * taps_w * C <= 512 && (C & 15) == 0) wp.nacc *= 2; }
  uint32_t ncols = 32;
  while (ncols < (uint32_t)(wp.nacc * wp.nrv * taps_w * C)) ncols <<= 1;
  wp.ncols = ncols;
  wp.M = K <= 64 ? 64 : 128;
  // a tile = APT runs of ONE image, a power of two, shrunk until a stage fits its budget
  const size_t per_run = (size_t)(wp.KG + wp.nrv * taps_w * wp.NCG) * 1024u;
  size_t target = WT_STAGE_TARGET;
  { const char* e = getenv("PO2_WT_STAGE_KB"); if (e && atoi(e) > 0) target = (size_t)atoi(e) * 1024; }
  int APT = 4;
  while (APT > 1 && (APT > wp.RPI || (size_t)APT * per_run > target)) APT >>= 1;
  wp.tiles_per_img = (wp.RPI + APT - 1) / APT;
  wp.nitems = B * wp.tiles_per_img;
  wp.APT = APT;
  wp.merged = (wp.W == 32 && wp.HW % 32 == 0) ? 1 : 0;
  if (wp.merged) {           // go [kg][run][8][128 B]; x [rv][s][cg][run][8][128 B]
    wp.g_run_bytes = 1024u; wp.x_run_bytes = 1024u; wp.sbo_bytes = (uint32_t)APT * 1024u;
    wp.copy_bytes = (uint32_t)(wp.NCG * APT) * 1024u;
    wp.x_rv_bytes = (uint32_t)taps_w * wp.copy_bytes;
    wp.g_bytes = (uint32_t)(wp.KG * APT) * 1024u;
    wp.stage_bytes = wp.g_bytes + (uint32_t)wp.nrv * wp.x_rv_bytes;
    wp.shift_units = 1; wp.shift_lines = wp.NCG * APT * 8;
  } else {                   // go [run][kg][8][128 B]; x [run][rv][s][cg][8][128 B]
    wp.g_run_bytes = (uint32_t)wp.KG * 1024u; wp.sbo_bytes = 1024u;
    wp.copy_bytes = (uint32_t)wp.NCG * 1024u;
    wp.x_rv_bytes = (uint32_t)taps_w * wp.copy_bytes;
    wp.x_run_bytes = (uint32_t)wp.nrv * wp.x_rv_bytes;
    wp.g_bytes = (uint32_t)APT * wp.g_run_bytes;
    wp.stage_bytes = (uint32_t)APT * (wp.g_run_bytes + wp.x_run_bytes);
    wp.shift_units = APT; wp.shift_lines = wp.NCG * 8;
  }
  wp.tx_bytes = (uint32_t)APT * (uint32_t)(wp.KG + wp.nrv * wp.NCG) * 1024u;
  // rows >= K of the A operand read the shared memory behind the go block (never used): keep them in bounds
  if ((size_t)(wp.M / 8) * wp.sbo_bytes > (size_t)wp.stage_bytes + 8192) return false;
  if (APT * (1 + wp.nrv) > 32) return false;
  const size_t fixed = 1024 + 8192 + (3 * K3_MAX_STAGES + 8) * 8 + 64;
  int nst = (int)((WT_SMEM_BUDGET - fixed) / wp.stage_bytes);
  if (nst > K3_MAX_STAGES) nst = K3_MAX_STAGES;
  { const char* e = getenv("PO2_WT_NST"); if (e && atoi(e) >= 2 && atoi(e) < nst) nst = atoi(e); }   // tuning: shared-memory footprint
  if (nst < 2) return false;
  wp.nst = nst;
  int m_ctas = sms / wp.rsplit;
  if (m_ctas < 1) m_ctas = 1;
  if (m_ctas > wp.nitems) m_ctas = wp.nitems;
  wp.m_ctas = m_ctas;
  wp.div_tpi = make_fastdiv((uint32_t)(wp.tiles_per_img > 0 ? wp.tiles_per_img : 1));
  { const char* e = getenv("PO2_WT_DEBUG"); wp.debug = e ? atoi(e) : 0; }
  return tma_encoder() != nullptr;
}

// (flat pixel, c % 8, c / 8, image, 1) over a (B, Cn, HW) fp32 tensor; box = one 32-pixel run x `groups` channel
// groups, landing as [c / 8][c % 8][32 pixels]: K-major 128-byte-swizzle atoms
// (runs > 0: the merged form (pixel % 32, c % 8, run, c / 8, image) with `runs` runs per box: [c / 8][run][c % 8][32])
static bool encode_flat_map(CUtensorMap* tm, const void* p, int B, int Cn, int HW, int groups, int runs) {
  EncodeTiledFn enc = tma_encoder();
  if (!enc || (reinterpret_cast<uintptr_t>(p) & 15)) return false;
  const cuuint64_t hw = (cuuint64_t)HW, c = (cuuint64_t)Cn, b = (cuuint64_t)B;
  cuuint64_t dims[5] = {hw, 8, c / 8, b, 1};
  cuuint64_t strides[4] = {hw * 4, 8 * hw * 4, c * hw * 4, b * c * hw * 4};
  cuuint32_t box[5] = {32, 8, (cuuint32_t)groups, 1, 1}, estr[5] = {1, 1, 1, 1, 1};
  if (runs > 0) {
    dims[0] = 32; dims[1] = 8; dims[2] = hw / 32; dims[3] = c / 8; dims[4] = b;
    strides[0] = hw * 4; strides[1] = 128; strides[2] = 8 * hw * 4; strides[3] = c * hw * 4;
    box[2] = (cuuint32_t)runs; box[3] = (cuuint32_t)groups;
  }
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<void*>(p), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static size_t wgrad_tma_partial_bytes(const WgTmaPlan& wp) {
  return (size_t)wp.m_ctas * wp.ntaps * wp.C * wp.K * sizeof(float);
}

// tickets != nullptr: 8 zero bytes (left zero) -> the partials are reduced inside the main kernel, launched
// cooperatively; nullptr: conv_wgrad_reduce_kernel as a second (programmatic dependent) launch
static int launch_wgrad_tma(const void* g_out, const void* x, void* gw, void* workspace, const WgTmaPlan& wp,
                            cudaStream_t st, unsigned int* tickets = nullptr) {
  CUtensorMap tmg, tmx;
  const int runs = wp.merged ? wp.APT : 0;
  if (!encode_flat_map(&tmg, g_out, wp.B, wp.K, wp.HW, wp.KG, runs) ||
      !encode_flat_map(&tmx, x, wp.B, wp.C, wp.HW, wp.NCG, runs))
    return PO2_E_UNSUPPORTED;
  static PerDeviceOnce once;
  if (cudaError_t e0 = once.run([]() -> cudaError_t {
        return cudaFuncSetAttribute(conv_wgrad_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)WT_SMEM_BUDGET + 1024);
      })) return (int)e0;
  const size_t smem = 1024 + (size_t)wp.nst * wp.stage_bytes + 8192 + (3 * K3_MAX_STAGES + 8) * 8 + 64;
  float* partial = (float*)workspace;
  float* gwf = (float*)gw;
  if (tickets) {
    WgTmaPlan wpv = wp;
    void* args[] = {&tmg, &tmx, &partial, &wpv, &gwf, &tickets};
    const cudaError_t e = cudaLaunchCooperativeKernel((const void*)conv_wgrad_tma_kernel, dim3(wp.m_ctas, wp.rsplit),
                                                      dim3(WT_THREADS), args, smem, st);
    if (e != cudaErrorCooperativeLaunchTooLarge) return (int)e;
    (void)cudaGetLastError();                                     // not co-resident on this device: two launches
  }
  float* nogw = nullptr;
  unsigned int* notk = nullptr;
  conv_wgrad_tma_kernel<<<dim3(wp.m_ctas, wp.rsplit), WT_THREADS, smem, st>>>(tmg, tmx, partial, wp, nogw, notk);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  return launch_wgrad_reduce(partial, gwf, wp.m_ctas, wp.K, wp.C, wp.ntaps, st);
}

}  // namespace po2
