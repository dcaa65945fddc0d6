// Quantized-conv forward for B200 (sm_100a): out = conv2d(x, W_q), x/out fp32 NCHW, bias=None, dilation=1
// (reference models/quantized_conv.py:36,38 -> nn.Conv2d._conv_forward -> F.conv2d).
//
// Three kernels behind po2_conv2d_fwd:
//   K3  conv_umma_kernel     dense convs on the 5th-gen tensor cores: an implicit GEMM whose A operand is
//                            the activation strip converted fp32 NCHW -> bf16 *in shared memory* in a
//                            "flat padded" K-major layout, so every filter tap is the SAME smem tile
//                            read through a UMMA descriptor whose start address is shifted by
//                            (r*pitch + s) pixels (no im2col copy); B is the PO2 weight tensor decoded
//                            to exact bf16 (+-2^q) and pre-packed per tap; accumulators live in TMEM
//                            (tcgen05.mma, one issuing thread) and are read back with tcgen05.ld for
//                            the epilogue, which applies the per-tensor scale and stores NCHW fp32.
//   K4  conv_depthwise_kernel groups == C == K, 3x3: CUDA-core, HBM/L2-bound.
//   --  conv_direct_kernel    any dense/grouped shape in fp32 FMA (the "fp32-accumulate" parity path and
//                            the fallback for shapes K3 does not take).
#include <limits.h>
#include <stdlib.h>

#include <type_traits>

#include "po2_common.cuh"

namespace po2 {

// ------------------------------------------------------------------------------------------------
// small PTX wrappers (tcgen05 / mbarrier / bulk copy)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE_%=;\n\t"
      "bra WAIT_%=;\n\t"
      "DONE_%=:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// contiguous global -> shared bulk copy (TMA engine, no tensor map), completion on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc] -> fp32; operands bf16 (kind::f16, K = 16 per instruction)
// or fp32 read as tf32 (kind::tf32, K = 8 per instruction)
template <bool TF32>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if (TF32)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
template <bool TF32>
__device__ __forceinline__ void umma_acc(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  if (TF32)
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.b32 p, 0, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
  else
    asm volatile("{\n\t.reg .pred p;\n\tsetp.eq.b32 p, 0, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr) : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major, no-swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
//   [0,14) start>>4 | [16,30) LBO>>4 (stride between the two 8-element K halves) |
//   [32,46) SBO>>4 (stride between 8-row groups) | [46,48) version=1 | [61,64) layout=0 (none)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46);
}
// instruction descriptor: D=f32, A=B=bf16 (format 1) or tf32 (format 2), both K-major, M=128, N
__device__ __forceinline__ uint32_t make_idesc(uint32_t n, bool tf32) {
  const uint32_t fmt = tf32 ? 2u : 1u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((n >> 3) << 17) | ((128u >> 4) << 24);
}

// 16 bytes of one strip position: G channels, as 8 x bf16 or 4 x fp32(tf32)
template <bool TF32>
__device__ __forceinline__ uint4 pack_channels(const float* v) {
  if (TF32) return make_uint4(__float_as_uint(v[0]), __float_as_uint(v[1]), __float_as_uint(v[2]), __float_as_uint(v[3]));
  __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
  return make_uint4(*reinterpret_cast<uint32_t*>(&p0), *reinterpret_cast<uint32_t*>(&p1),
                    *reinterpret_cast<uint32_t*>(&p2), *reinterpret_cast<uint32_t*>(&p3));
}

// ------------------------------------------------------------------------------------------------
// geometry shared by host and device
// ------------------------------------------------------------------------------------------------
struct ConvGeom {
  int B, C, H, W, K, R, S, stride, pad, groups;
  int P, Q;              // output height / width
  // ---- K3 "flat padded" output-position space: position L = row * pitch + col, rows of all images
  // stacked; one zero column per row / one zero row per image are shared by neighbouring windows
  int pitch, rows_img, top;   // Q + (S==3), P + (R==3), number of pad rows before image 0
  int Ltot;              // number of flat positions
  int halo_before;       // flat positions of context in front of a 128-position tile
  int strip;             // positions per A stage = 128 + halo_before + halo_after
  int nphase;            // 1, or 4 input parity phases for 3x3 stride 2
  int ntaps;
  int tap_phase[9];      // which phase plane set a tap reads
  int tap_off[9];        // strip index of the tap's row for tile row 0 (>= 0)
  int tf32, G;           // operand kind: bf16 (G = 8 channels per 16-byte plane entry) or tf32 (G = 4)
  int Cpad, CC, nchunk;  // channels padded to 2G (one MMA k-step); channels per pipeline stage; stages per item
  int NT, ntiles_n;      // out-channel tile (multiple of 16, <= 256) and their count
  int nitems_m, m_step;  // 128-position items; items advance by m_step per CTA iteration (nitems_m < 2^24 and
                         // m_step <= 148: the 32-bit item loops stay far below 2^31)
  int nst;               // A pipeline stages
  uint32_t a_stage_bytes, b_slab_bytes;
  FastDiv div_pitch, div_rows, div_strip, div_ipr, div_NT, div_ncg, div_taps;
  int vec4, items_per_row;   // producer fast path: float4 loads along W
  int prod_groups;           // independent producer groups (stages in flight per CTA)
  int dual_issue;            // two MMA issuers alternate tiles (only when a tile is one stage)
  int tapminor;              // weight operand layout Bp[nt][r][c/G][s][n][G] (the TMA-fed kernel, 3x3): see PackArgs
};

// ------------------------------------------------------------------------------------------------
// weight pack: fp32 PO2-grid weights (or codes) -> exact bf16 +-2^q in the B-operand layout
//   Bp[nt][tap][cg][n][8]   (cg: group of 8 input channels, n: out channel inside the N tile)
// ------------------------------------------------------------------------------------------------
__global__ void pack_weights_kernel(const float* __restrict__ w, const uint8_t* __restrict__ codes,
                                    const float* __restrict__ scale, void* __restrict__ Bp,
                                    ConvGeom g, int bits, int fsr, int transpose) {
  // programmatic dependent launch: the conv kernel behind us may start now; its MMA warp executes
  // griddepcontrol.wait before it touches Bp, everything else (TMEM alloc, barrier init, the
  // activation producers) overlaps with this kernel.  THIS kernel is launched with a normal
  // (full) dependency on its predecessor, so everything earlier in the stream -- in particular the
  // kernel that produced the conv's input x -- has completed and is visible before either starts.
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int G = g.G, lgG = (G == 8) ? 3 : 2;
  const int taps = g.ntaps, ncg = g.Cpad / G;
  const int total = g.ntiles_n * taps * ncg * g.NT * G;           // < 2^30 (plan_tc): i + stride cannot wrap
  const float s = scale ? *scale : 1.0f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    // i = (((nt * taps + tap) * ncg + cg) * NT + n) * G + j, decoded with mul-hi divisions
    // (tapminor: i = ((((nt * 3 + r) * ncg + cg) * 3 + s) * NT + n) * G + j, tap = 3 r + s)
    const int j = i & (G - 1);
    int t = i >> lgG;
    int q = fdiv(t, g.div_NT);  const int n = t - q * g.NT;  t = q;
    int cg, tap, nt;
    if (g.tapminor) {
      const int s3 = t % 3; t /= 3;
      q = fdiv(t, g.div_ncg); cg = t - q * ncg; t = q;
      tap = (t % 3) * 3 + s3; nt = t / 3;
    } else {
      q = fdiv(t, g.div_ncg);     cg = t - q * ncg;   t = q;
      q = fdiv(t, g.div_taps);    tap = t - q * taps; nt = q;
    }
    const int c = cg * G + j;
    const int k = nt * g.NT + n;
    float v = 0.0f;
    if (c < g.C && k < g.K) {
      // transpose (data-gradient conv): this conv's (k, c, tap) reads W_src[c][k][taps-1-tap], i.e. the
      // forward weight with in/out channels swapped and the 3x3 window rotated by 180 degrees
      const int64_t wi = transpose ? ((int64_t)c * g.K + k) * taps + (taps - 1 - tap)
                                   : ((int64_t)k * g.C + c) * taps + tap;
      if (codes) {
        const uint32_t code = (bits <= 4) ? ((codes[wi >> 1] >> ((wi & 1) * 4)) & 0xFu) : codes[wi];
        const int mag = code & ((1u << (bits - 1)) - 1u);
        v = exp2_int((fsr - 1) - mag);
        if ((code >> (bits - 1)) & 1u) v = -v;
      } else {
        // w = +-s*2^q exactly, so w/s is exactly +-2^q and the bf16 conversion is lossless; a weight
        // that is not on the grid (unquantized layer) is rounded to bf16 like any bf16 GEMM would
        v = (s == 1.0f) ? w[wi] : __fdiv_rn(w[wi], s);
      }
    }
    if (g.tf32) reinterpret_cast<float*>(Bp)[i] = v;       // +-2^q is exact in tf32 as well
    else reinterpret_cast<__nv_bfloat16*>(Bp)[i] = __float2bfloat16_rn(v);
  }
}

// ------------------------------------------------------------------------------------------------
// K3: persistent, warp-specialised tcgen05 implicit-GEMM conv (groups == 1; 3x3 pad 1 or 1x1 pad 0;
// stride 1 or 2).  Per CTA: warps 0-3 epilogue (TMEM lane quarter = warp id), warp 4 = TMEM
// allocator + weight-slab bulk copy + the single MMA-issuing thread, warps 5-12 activation producers.
//   producers --full[s]--> MMA --tcgen05.commit: empty[s]--> producers      (A stages, ring of nst)
//   MMA --tcgen05.commit: tmem_full[a]--> epilogue --tmem_empty[a]--> MMA   (2 accumulator stages)
// ------------------------------------------------------------------------------------------------
#ifdef PO2_K3_TRACE
// debug-only event trace (tools/trace_conv.py builds a separate library with -DPO2_K3_TRACE):
// SM-clock timestamps into shared memory (cheap), dumped to global memory at kernel end
__device__ long long* g_k3_trace = nullptr;              // [cta < 4][role 0..7][event 0..63] = clock64
__shared__ long long k3_trace_smem[8 * 64];
__device__ __forceinline__ void k3_trace(int role, int ev) {
  if (ev < 64) k3_trace_smem[role * 64 + ev] = clock64();
}
#define K3_TRACE(role, ev) k3_trace(role, ev)
#else
#define K3_TRACE(role, ev)
#endif

constexpr int K3_EPI_WARPS = 4;
constexpr int K3_PROD_WARPS = 8;
constexpr int PU = 4;               // producer items in flight per thread (x8 loads each)
constexpr int K3_MMA_WARPS = 2;         // two issuing warps alternate tiles so one's barrier/fence latency hides behind the other's MMAs
constexpr int K3_THREADS = 32 * (K3_EPI_WARPS + K3_MMA_WARPS + K3_PROD_WARPS);
constexpr int K3_MAX_STAGES = 6;
constexpr uint32_t K3_SMEM_BUDGET = 220 * 1024;
constexpr uint32_t K3_B_BUDGET = 112 * 1024;

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// flat position -> (image, out row, out col); false for the shared zero pads / out of range
__device__ __forceinline__ bool decode_pos(const ConvGeom& g, int L, int& img, int& a, int& b) {
  if (L < 0 || L >= g.Ltot) return false;
  const int row = fdiv(L, g.div_pitch);
  b = L - row * g.pitch;
  const int r0 = row - g.top;
  if (r0 < 0) return false;
  img = fdiv(r0, g.div_rows);
  a = r0 - img * g.rows_img;
  return (b < g.Q) && (a < g.P) && (img < g.B);
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xFFFFFFFF;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// XT: the activation storage of x, out and the residual -- float, or __nv_bfloat16 (a bf16 model at inference: its
// values are exact bf16 operands, copied into the strips without conversion; the MMA is kind::f16, accumulation fp32)
template <int NTAPS, bool TF32, typename XT>
__global__ void __launch_bounds__(K3_THREADS, 1) conv_umma_kernel(const XT* __restrict__ x,
                                                                  const uint8_t* __restrict__ Bp,
                                                                  const float* __restrict__ scale,
                                                                  XT* __restrict__ out, ConvGeom g, ConvEpilogue ep) {
  constexpr bool BF16X = sizeof(XT) == 2;
  static_assert(!(BF16X && TF32), "bf16 activations are kind::f16 operands");
  extern __shared__ __align__(128) uint8_t smem[];
  uint8_t* sB = smem;
  uint8_t* sA = smem + g.b_slab_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA + (size_t)g.nst * g.a_stage_bytes);
  uint64_t* full = bars;                        // [nst]   producers -> MMA
  uint64_t* empty = bars + K3_MAX_STAGES;       // [nst]   MMA (commit) -> producers
  uint64_t* tfull = bars + 2 * K3_MAX_STAGES;   // [2]     MMA (commit) -> epilogue
  uint64_t* tempty = tfull + 2;                 // [2]     epilogue -> MMA
  uint64_t* bfull = tempty + 2;                 // weight slab landed
  uint64_t* tready = bfull + 1;                 // TMEM allocated, address published
  uint64_t* turn = tready + 1;                  // [2]     issuer hand-over (dual-issuer mode)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(turn + 2);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
#ifdef PO2_K3_TRACE
  for (int i = tid; i < 8 * 64; i += K3_THREADS) k3_trace_smem[i] = 0;
  __syncthreads();
#endif
  if (tid == 0) K3_TRACE(6, 0);
  const int nt = blockIdx.x % g.ntiles_n;
  const int m_first = blockIdx.x / g.ntiles_n;
  uint32_t ncols = 32;
  while ((int)ncols < 2 * g.NT) ncols <<= 1;

  // Only the barrier initialisation sits in front of the CTA-wide sync; TMEM allocation is taken
  // off the producers' critical path: the first issuer warp allocates after the sync and publishes
  // the address through `tready`, which its consumers (second issuer, epilogue warps) wait on.
  if (warp == K3_EPI_WARPS + 1 && lane == 0) {
    for (int i = 0; i < g.nst; ++i) { mbar_init(full + i, K3_PROD_WARPS / g.prod_groups); mbar_init(empty + i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(tfull + i, 1); mbar_init(tempty + i, K3_EPI_WARPS); }
    mbar_init(bfull, 1);
    mbar_init(tready, 1);
    mbar_init(turn, 1);
    mbar_init(turn + 1, 1);
    fence_mbar_init();
  }
  __syncthreads();
  uint32_t tmem_base = 0;
  if (warp == K3_EPI_WARPS) {
    tmem_alloc(tmem_slot, ncols);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(tready);
    tc_fence_after();
    tmem_base = *tmem_slot;
  } else if (warp < K3_EPI_WARPS + K3_MMA_WARPS) {
    mbar_wait(tready, 0);
    tc_fence_after();
    tmem_base = *tmem_slot;
  }
  if (tid == 0) K3_TRACE(6, 1);
  const int HW = g.H * g.W, PQ = g.P * g.Q;
  constexpr int G = TF32 ? 4 : 8;                 // channels per 16-byte plane entry
  constexpr int KCH = 2 * G;                      // channels per MMA k-step (two planes)
  const int ngrpCC = g.CC / G;

  if (warp >= K3_EPI_WARPS && warp < K3_EPI_WARPS + K3_MMA_WARPS) {
    // =========================== MMA issuers ===========================
    // Issuer q takes the tiles whose index has parity q and always accumulates into TMEM stage q.
    // The whole warp runs this loop with warp-uniform values (so descriptors stay on the uniform
    // datapath); one elected lane issues tcgen05.mma / tcgen05.commit.
    const bool leader = elect_one();
    const uint32_t me = (uint32_t)(warp - K3_EPI_WARPS);
    if (leader && me == 0) {
      asm volatile("griddepcontrol.wait;" ::: "memory");       // the weight-pack kernel has completed and flushed
      mbar_expect_tx(bfull, g.b_slab_bytes);
      bulk_g2s(sB, Bp + (size_t)nt * g.b_slab_bytes, g.b_slab_bytes, bfull);
    }
    mbar_wait(bfull, 0);
    const uint32_t idesc = make_idesc((uint32_t)g.NT, TF32);
    const uint32_t a_plane16 = (uint32_t)g.strip, b_plane16 = (uint32_t)g.NT;     // plane strides in 16-byte units
    // descriptor words: lo = start>>4 | LBO>>4 << 16 ; hi = SBO>>4 (=8) | version 1 << 14
    const uint32_t desc_hi = 8u | (1u << 14);
    const uint32_t a_lo_fixed = a_plane16 << 16, b_lo_fixed = b_plane16 << 16;
    const uint32_t b0_16 = smem_u32(sB) >> 4, a0_16 = smem_u32(sA) >> 4;
    const uint32_t a_stage16 = g.a_stage_bytes >> 4;
    const int ncg = g.Cpad / G, nchunk = g.nchunk, nst = g.nst, CC = g.CC, Cpad = g.Cpad, NT = g.NT;
    uint32_t a_tap16[NTAPS], b_tap16[NTAPS];
#pragma unroll
    for (int tap = 0; tap < NTAPS; ++tap) {
      a_tap16[tap] = (uint32_t)(g.tap_phase[tap] * ngrpCC) * a_plane16 + (uint32_t)g.tap_off[tap];
      b_tap16[tap] = (uint32_t)(tap * ncg) * b_plane16;
    }
    const int nitems = g.nitems_m, m_step = g.m_step;
    // mbarrier phases are one bit: a waiter must never target a phase more than one ahead of the
    // barrier's current one.  Hence (1) two issuers alternate tiles only when a tile is a single
    // stage (g.dual_issue), and then hand a token to each other so that the `full` waits of the whole
    // CTA happen in stage order; (2) otherwise issuer 0 does everything.
    const bool dual = g.dual_issue != 0;
    uint32_t s = 0, sphase = 0, tkphase = 0;                       // A-stage ring position, token phase
    uint32_t aph0 = 0, aph1 = 0;                                   // phase of each accumulator's `tempty`
    uint32_t tile = 0;
    for (int m = m_first; m < nitems && (dual || me == 0); m += m_step, ++tile) {
      if (dual && (tile & 1u) != me) {                           // the other issuer's tile: just advance the ring
        if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
        continue;
      }
      const uint32_t acc = tile & 1u;
      const uint32_t d = tmem_base + acc * (uint32_t)NT;
      if (dual && tile > 0) { mbar_wait(turn + me, tkphase); tkphase ^= 1; }   // stages < mine have been waited for
      mbar_wait(tempty + acc, (acc ? aph1 : aph0) ^ 1);          // epilogue has drained this accumulator
      for (int chunk = 0; chunk < nchunk; ++chunk) {
        mbar_wait(full + s, sphase);
        tc_fence_after();                                        // orders the MMAs after both waits above
        if (dual && leader) mbar_arrive(turn + (me ^ 1u));       // hand over: the other issuer may wait for the next stage
        if (leader) K3_TRACE((int)me * 7, 2 * (int)((tile >> 1) * nchunk + chunk));
        const uint32_t a_s16 = a0_16 + s * a_stage16;
        const uint32_t b_c16 = b0_16 + (uint32_t)(chunk * ngrpCC) * b_plane16;
        const int ksteps = min(CC, Cpad - chunk * CC) / KCH;
        if (leader) {
          // k-step outer (1-4 iterations), taps inner and fully unrolled: straight-line MMA issue with
          // per-tap descriptor words that only need the stage / k-step offset added
          uint32_t a_off = a_s16 | a_lo_fixed, b_off = b_c16 | b_lo_fixed;
          for (int ks = 0; ks < ksteps; ++ks) {
#pragma unroll
            for (int tap = 0; tap < NTAPS; ++tap) {
              const uint64_t ad = ((uint64_t)desc_hi << 32) | (a_off + a_tap16[tap]);
              const uint64_t bd = ((uint64_t)desc_hi << 32) | (b_off + b_tap16[tap]);
              if (tap == 0) umma<TF32>(d, ad, bd, idesc, (uint32_t)((chunk | ks) != 0));
              else umma_acc<TF32>(d, ad, bd, idesc);
            }
            a_off += 2 * a_plane16;                              // next k-step: two planes on
            b_off += 2 * b_plane16;
          }
          umma_commit(empty + s);                                // stage reusable once these MMAs retire
          if (chunk == nchunk - 1) umma_commit(tfull + acc);     // accumulator complete
          K3_TRACE((int)me * 7, 2 * (int)((tile >> 1) * nchunk + chunk) + 1);
        }
        __syncwarp();
        if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
      }
      if (acc) aph1 ^= 1; else aph0 ^= 1;
    }
  } else if (warp < K3_EPI_WARPS) {
    // =========================== epilogue: TMEM -> scale -> NCHW fp32 / bf16 ===========================
    // `scale` may be written by the kernel this one was launched behind with programmatic dependent
    // launch (the fused quantize+pack kernel of po2_qconv2d_fwd): like the weight slab it must not be
    // read before that grid has completed.  The wait costs nothing here -- the first accumulator
    // cannot be ready before the slab, which sits behind the same wait in the issuer.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    const float sc = scale ? *reinterpret_cast<const volatile float*>(scale) : 1.0f;
    const int K = g.K, NT = g.NT, m_step = g.m_step, nitems = g.nitems_m;
    const int kbase = nt * NT;
    // folded BatchNorm: this CTA's NT scale / shift values staged in shared memory once
    __shared__ float s_ep[2][256];
    if (ep.a) {
      for (int i = tid; i < NT; i += 32 * K3_EPI_WARPS) {
        const bool ok = kbase + i < K;
        s_ep[0][i] = ok ? __ldg(ep.a + kbase + i) : 0.f;
        s_ep[1][i] = ok ? __ldg(ep.b + kbase + i) : 0.f;
      }
      asm volatile("bar.sync 2, %0;" ::"n"(32 * K3_EPI_WARPS) : "memory");
    }
    uint32_t item = 0, acc = 0, aphase = 0;
    for (int m = m_first; m < nitems; m += m_step, ++item) {
      int img = 0, a = 0, b = 0;
      const bool valid = decode_pos(g, m * 128 + warp * 32 + lane, img, a, b);
      const int obase = (img * K + kbase) * PQ + a * g.Q + b;          // < 2^31 (checked on the host)
      mbar_wait(tfull + acc, aphase);
      tc_fence_after();
      if (warp == 0 && lane == 0) K3_TRACE(1, 2 * (int)item);
      const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + acc * (uint32_t)NT;
      for (int cb = 0; cb < NT / 16; ++cb) {
        uint32_t r[16];
        tmem_ld16(trow + (uint32_t)cb * 16, r);
        if (valid) {
          XT* po = out + obase + cb * 16 * PQ;
          const int kleft = K - (kbase + cb * 16);
          if (ep.a) {                                            // folded BatchNorm (+ residual) (+ activation)
            float rs[16];
            if (ep.res) {
              const XT* pr = reinterpret_cast<const XT*>(ep.res) + obase + cb * 16 * PQ;
#pragma unroll
              for (int j = 0; j < 16; ++j) rs[j] = j < kleft ? act_ld(pr + j * PQ) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j < kleft) {
                float t = fmaf(__uint_as_float(r[j]) * sc, s_ep[0][cb * 16 + j], s_ep[1][cb * 16 + j]);
                if (ep.res) t += rs[j];
                act_st(po, j * PQ, conv_act(t, ep.act));
              }
          } else if (kleft >= 16) {
#pragma unroll
            for (int j = 0; j < 16; ++j) act_st(po, j * PQ, __uint_as_float(r[j]) * sc);
          } else {
#pragma unroll
            for (int j = 0; j < 16; ++j)
              if (j < kleft) act_st(po, j * PQ, __uint_as_float(r[j]) * sc);
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty + acc);
      if (warp == 0 && lane == 0) K3_TRACE(1, 2 * (int)item + 1);
      acc ^= 1;
      aphase ^= (acc == 0);
    }
  } else {
    // =========================== producers: fp32 / bf16 NCHW -> bf16 (tf32) flat K-major strips ===========================
    // The producer warps form K3_PROD_GROUPS independent groups; group q fills every stage `it` with
    // it % groups == q on its own, so that many stages are in flight against global-memory latency
    // at once (a thread cannot start its next stage before the loads of the current one return).
    const int ngroups = g.prod_groups;                    // 1, 2 or 4 (few tiles per CTA -> fewer, wider groups)
    const int WPG = K3_PROD_WARPS / ngroups;              // warps per group
    const int NPG = 32 * WPG;                             // threads per group
    const int pw = warp - (K3_EPI_WARPS + K3_MMA_WARPS);
    const int grp_id = pw / WPG;
    const int gt = tid - 32 * (K3_EPI_WARPS + K3_MMA_WARPS) - grp_id * NPG;
    const int strip = g.strip, C = g.C, H = g.H, W = g.W, stride = g.stride, CC = g.CC, Cpad = g.Cpad;
    const int nphase = g.nphase, nchunk = g.nchunk, nst = g.nst, m_step = g.m_step, nitems = g.nitems_m;
    const int halo = g.halo_before;
    const uint32_t a_stage_bytes = g.a_stage_bytes;
    const bool hw1 = (HW == 1) && (C % (BF16X ? 8 : 4) == 0);
    uint32_t it = 0, s = 0, sphase = 0;
    int turn = 0;                                         // which group owns stage `it`
    for (int m = m_first; m < nitems; m += m_step) {
      const int Ls = m * 128 - halo;
      for (int chunk = 0; chunk < nchunk; ++chunk, ++it) {
        const uint32_t s_cur = s, ph_cur = sphase;
        const bool mine = (turn == grp_id);
        if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
        if (++turn == ngroups) turn = 0;
        if (!mine) continue;
        mbar_wait(empty + s_cur, ph_cur ^ 1);
        if (gt == 0) K3_TRACE(2 + grp_id, 2 * (int)(it / ngroups));
        uint8_t* stage = sA + (size_t)s_cur * a_stage_bytes;
        const int cbase = chunk * CC;
        const int ngrp = min(CC, Cpad - cbase) / G;
        const int nitem = ngrp * strip;                    // (channel group, position) items per phase
        if (g.vec4) {
          // ---- fast path (stride 1, W % PX == 0): one item = PX consecutive pixels of one image row x
          // 8 channels = 8 x LDG.128 -> PX x STS.128 (PX = 4 fp32 / 8 bf16 pixels per 16 bytes); the shared zero
          // column is one extra item per row
          constexpr int PX = BF16X ? 8 : 4, LPX = BF16X ? 3 : 2;
          using VT = typename std::conditional<BF16X, uint4, float4>::type;
          const int pitch = g.pitch, W4 = W >> LPX, ipr = g.items_per_row;     // W4 (+1 with a pad column)
          const int rowA = Ls >= 0 ? fdiv(Ls, g.div_pitch) : -((-Ls + pitch - 1) / pitch);
          const int rowB = fdiv(Ls + strip - 1, g.div_pitch);
          // only the row items that overlap the strip: [jA, jB] in the linearised (row, item) space
          const int jA = min((Ls - rowA * pitch) >> LPX, ipr - 1);
          const int jB = (rowB - rowA) * ipr + min((Ls + strip - 1 - rowB * pitch) >> LPX, ipr - 1);
          const int nrow_items = jB - jA + 1;
          const int nall = ngrp * nrow_items;                 // (channel group, row item) pairs of this stage
          const float inv_items = 1.0f / (float)nrow_items;
          for (int i0 = gt; i0 < nall; i0 += 2 * NPG) {
            VT v[2][G];
            int lbase[2], npos[2], gsel[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {                // 16 x 128-bit loads in flight per thread
              const int i = i0 + u * NPG;
              lbase[u] = 0; npos[u] = 0; gsel[u] = 0;
              bool ok = false;
              int idx = 0, cvalid = 0;
              if (i < nall) {
                int grp = (int)(((float)i + 0.5f) * inv_items);         // i / nrow_items (exact for these sizes)
                int j = i - grp * nrow_items;
                if (j < 0) { --grp; j += nrow_items; } else if (j >= nrow_items) { ++grp; j -= nrow_items; }
                j += jA;
                const int rr = fdiv(j, g.div_ipr);
                const int q4 = j - rr * ipr;
                const int row = rowA + rr;
                const int c0 = cbase + grp * G;
                gsel[u] = grp;
                cvalid = C - c0;
                lbase[u] = row * pitch + q4 * PX - Ls;                      // strip index of pixel 0 of the item
                npos[u] = q4 < W4 ? PX : pitch - W;                         // the pad item covers only the pad column
                const int r0 = row - g.top;
                if (q4 < W4 && r0 >= 0) {
                  const int img = fdiv(r0, g.div_rows);
                  const int a = r0 - img * g.rows_img;
                  if (a < H && img < g.B) { ok = true; idx = ((img * C + c0) * H + a) * W + q4 * PX; }
                }
              }
              const VT* px = reinterpret_cast<const VT*>(x + idx);
#pragma unroll
              for (int c = 0; c < G; ++c)
                v[u][c] = (ok && c < cvalid) ? __ldg(px + (size_t)c * (HW >> LPX)) : VT{};
            }
#pragma unroll
            for (int u = 0; u < 2; ++u) {
              uint8_t* sgrp = stage + (size_t)gsel[u] * strip * 16;
#pragma unroll
              for (int e = 0; e < PX; ++e) {
                const int lloc = lbase[u] + e;
                if (e < npos[u] && lloc >= 0 && lloc < strip) {
#define PO2_C4(q, e_) ((e_) == 0 ? (q).x : (e_) == 1 ? (q).y : (e_) == 2 ? (q).z : (q).w)
                  uint4 val;
                  if constexpr (BF16X) {
                    // pixel e of channels 2j, 2j+1: the low or high halves of word e / 2 of both loads
                    const uint32_t sel = (e & 1) ? 0x7632u : 0x5410u;
                    val = make_uint4(__byte_perm(PO2_C4(v[u][0], e >> 1), PO2_C4(v[u][1], e >> 1), sel),
                                     __byte_perm(PO2_C4(v[u][2], e >> 1), PO2_C4(v[u][3], e >> 1), sel),
                                     __byte_perm(PO2_C4(v[u][4], e >> 1), PO2_C4(v[u][5], e >> 1), sel),
                                     __byte_perm(PO2_C4(v[u][6], e >> 1), PO2_C4(v[u][7], e >> 1), sel));
                  } else {
                    float ch[G];                                  // pixel e of every channel of the item
#pragma unroll
                    for (int c = 0; c < G; ++c) ch[c] = PO2_C4(v[u][c], e);
                    val = pack_channels<TF32>(ch);
                  }
#undef PO2_C4
                  *reinterpret_cast<uint4*>(sgrp + (size_t)lloc * 16) = val;
                }
              }
            }
          }
        } else
        for (int ph = 0; ph < nphase; ++ph) {
          const int pr = ph >> 1, pc = ph & 1;
          uint8_t* sph = stage + (size_t)ph * ngrpCC * strip * 16;
          for (int i0 = gt; i0 < nitem; i0 += PU * NPG) {
            // PU items (PU*G independent loads) in flight per thread before the first conversion
            // (bf16: the raw 16-bit patterns, stored without conversion)
            typename std::conditional<BF16X, uint32_t, float>::type v[PU][G];
#pragma unroll
            for (int u = 0; u < PU; ++u) {
              const int i = i0 + u * NPG;
              int cvalid = 0, idx = 0;
              if (i < nitem) {
                const int grp = fdiv(i, g.div_strip);
                const int lloc = i - grp * strip;
                int img, a, b;
                if (decode_pos(g, Ls + lloc, img, a, b)) {
                  const int ih = a * stride + pr, iw = b * stride + pc;
                  if (ih < H && iw < W) {
                    const int c0 = cbase + grp * G;
                    cvalid = C - c0;
                    idx = ((img * C + c0) * H + ih) * W + iw;
                  }
                }
              }
              const XT* px = x + idx;
              if constexpr (BF16X) {
                if (hw1) {                                 // 1x1 feature map: the 8 channels are 16 contiguous bytes
                  const uint4 q = cvalid > 0 ? __ldg(reinterpret_cast<const uint4*>(px)) : make_uint4(0u, 0u, 0u, 0u);
                  const uint32_t w4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                  for (int j = 0; j < G; ++j) v[u][j] = (w4[j >> 1] >> (16 * (j & 1))) & 0xFFFFu;
                } else {
#pragma unroll
                  for (int j = 0; j < G; ++j) v[u][j] = (j < cvalid) ? __bfloat16_as_ushort(__ldg(px + j * HW)) : 0u;
                }
              } else if (hw1) {                            // 1x1 feature map: the G channels are contiguous bytes
                const float4 lo = cvalid > 0 ? __ldg(reinterpret_cast<const float4*>(px)) : make_float4(0.f, 0.f, 0.f, 0.f);
                v[u][0] = lo.x; v[u][1] = lo.y; v[u][2] = lo.z; v[u][3] = lo.w;
                if (G == 8) {
                  const float4 hi = cvalid > 4 ? __ldg(reinterpret_cast<const float4*>(px) + 1) : make_float4(0.f, 0.f, 0.f, 0.f);
                  v[u][G - 4] = hi.x; v[u][G - 3] = hi.y; v[u][G - 2] = hi.z; v[u][G - 1] = hi.w;
                }
              } else {
#pragma unroll
                for (int j = 0; j < G; ++j) v[u][j] = (j < cvalid) ? __ldg(px + j * HW) : 0.0f;
              }
            }
#pragma unroll
            for (int u = 0; u < PU; ++u) {
              const int i = i0 + u * NPG;
              if (i < nitem) {
                uint4 val;
                if constexpr (BF16X)
                  val = make_uint4(v[u][0] | (v[u][1] << 16), v[u][2] | (v[u][3] << 16), v[u][4] | (v[u][5] << 16),
                                   v[u][6] | (v[u][7] << 16));
                else
                  val = pack_channels<TF32>(v[u]);
                *reinterpret_cast<uint4*>(sph + (size_t)i * 16) = val;   // i == grp*strip + lloc
              }
            }
          }
        }
        fence_proxy_async();                          // generic-proxy smem writes -> tensor-core reads
        __syncwarp();
        if (lane == 0) mbar_arrive(full + s_cur);
        if (gt == 0) K3_TRACE(2 + grp_id, 2 * (int)(it / ngroups) + 1);
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) K3_TRACE(6, 2);
#ifdef PO2_K3_TRACE
  __syncthreads();
  if (g_k3_trace && blockIdx.x < 4)
    for (int i = tid; i < 8 * 64; i += K3_THREADS) g_k3_trace[blockIdx.x * 8 * 64 + i] = k3_trace_smem[i];
#endif
  if (warp == K3_EPI_WARPS) tmem_dealloc(tmem_base, ncols);
}

// ------------------------------------------------------------------------------------------------
// K4: depthwise 3x3 (groups == C == K), stride 1 or 2, pad 1: CUDA cores, HBM/L2-bound.
// One thread = 4 consecutive outputs of one row (128-bit store); per input row it issues one or two
// 128-bit loads plus the halo scalars instead of 3 (or 9) scalar loads per output.  32-bit index
// arithmetic with mul-hi divisions.  Other depthwise shapes take the scalar kernel below.
// ------------------------------------------------------------------------------------------------
struct DwGeom {
  int C, H, W, P, Q, Q4, stride;
  int total;                 // B*C*P*Q4 threads' worth of work: < 2^29, so the 32-bit loop never nears 2^31
  FastDiv div_q4, div_p, div_c;
};

// XT: float, or __nv_bfloat16 (x, out and the residual of a bf16 model; fp32 arithmetic, 64-bit loads and stores)
template <int STRIDE, typename XT>
__global__ void __launch_bounds__(256) conv_depthwise_vec_kernel(const XT* __restrict__ x,
                                                                 const float* __restrict__ w,
                                                                 XT* __restrict__ out, DwGeom g, ConvEpilogue ep) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < g.total; i += gridDim.x * blockDim.x) {
    int t = fdiv(i, g.div_q4);
    const int q0 = (i - t * g.Q4) * 4;
    int u = fdiv(t, g.div_p);
    const int p = t - u * g.P;
    const int plane = u;                                   // n * C + c
    const int c = plane - fdiv(plane, g.div_c) * g.C;
    const XT* px = x + (size_t)plane * g.H * g.W;
    const float* pw = w + c * 9;
    float wk[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) wk[k] = __ldg(pw + k);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    constexpr int NIN = STRIDE == 1 ? 6 : 9;               // input columns feeding 4 outputs
    const int iw0 = q0 * STRIDE - 1;                       // leftmost input column (may be -1)
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int ih = p * STRIDE - 1 + r;
      if (ih < 0 || ih >= g.H) continue;
      const XT* row = px + ih * g.W;
      float in[NIN];
      // columns iw0+1 .. iw0+4 (and +5..+8 for stride 2) are 16-byte (bf16: 8-byte) aligned groups inside the row
      if constexpr (sizeof(XT) == 2) {
        const uint2 a = __ldg(reinterpret_cast<const uint2*>(row + iw0 + 1));
        in[0] = iw0 >= 0 ? act_ld(row + iw0) : 0.f;
        in[1] = __uint_as_float(a.x << 16); in[2] = __uint_as_float(a.x & 0xFFFF0000u);
        in[3] = __uint_as_float(a.y << 16); in[4] = __uint_as_float(a.y & 0xFFFF0000u);
        if (STRIDE == 1) {
          in[5] = (iw0 + 5 < g.W) ? act_ld(row + iw0 + 5) : 0.f;
        } else {
          const uint2 b = __ldg(reinterpret_cast<const uint2*>(row + iw0 + 5));
          in[5] = __uint_as_float(b.x << 16); in[6] = __uint_as_float(b.x & 0xFFFF0000u);
          in[7] = __uint_as_float(b.y << 16); in[8] = __uint_as_float(b.y & 0xFFFF0000u);
        }
      } else {
        const float4 a = __ldg(reinterpret_cast<const float4*>(row + iw0 + 1));
        in[0] = iw0 >= 0 ? __ldg(row + iw0) : 0.f;
        in[1] = a.x; in[2] = a.y; in[3] = a.z; in[4] = a.w;
        if (STRIDE == 1) {
          in[5] = (iw0 + 5 < g.W) ? __ldg(row + iw0 + 5) : 0.f;
        } else {
          const float4 b = __ldg(reinterpret_cast<const float4*>(row + iw0 + 5));
          in[5] = b.x; in[6] = b.y; in[7] = b.z; in[8] = b.w;
        }
      }
#pragma unroll
      for (int o = 0; o < 4; ++o)
#pragma unroll
        for (int s2 = 0; s2 < 3; ++s2) acc[o] = fmaf(in[o * STRIDE + s2], wk[r * 3 + s2], acc[o]);
    }
    const size_t o = ((size_t)plane * g.P + p) * g.Q + q0;
    if (ep.a) {
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[e] = conv_epilogue<XT>(acc[e], ep, c, o + e);
    }
    if constexpr (sizeof(XT) == 2) {
      const __nv_bfloat162 lo = __floats2bfloat162_rn(acc[0], acc[1]), hi = __floats2bfloat162_rn(acc[2], acc[3]);
      *reinterpret_cast<uint2*>(out + o) = make_uint2(*reinterpret_cast<const uint32_t*>(&lo), *reinterpret_cast<const uint32_t*>(&hi));
    } else {
      *reinterpret_cast<float4*>(out + o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
    }
  }
}

// any other depthwise shape: one thread per output element
template <typename XT>
__global__ void __launch_bounds__(256) conv_depthwise_kernel(const XT* __restrict__ x,
                                                             const float* __restrict__ w,
                                                             XT* __restrict__ out, ConvGeom g,
                                                             FastDiv div_q, FastDiv div_p, FastDiv div_c, ConvEpilogue ep) {
  const int total = g.B * g.C * g.P * g.Q;                 // < 2^31 (checked on the host)
  // total may lie within one grid stride of 2^31: a 32-bit i would wrap on its last step
  for (int64_t i64 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i64 < total; i64 += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)i64;
    int t = fdiv(i, div_q);
    const int q = i - t * g.Q;
    const int plane = fdiv(t, div_p);
    const int p = t - plane * g.P;
    const int c = plane - fdiv(plane, div_c) * g.C;
    const XT* px = x + (size_t)plane * g.H * g.W;
    const float* pw = w + (size_t)c * g.R * g.S;
    float acc = 0.0f;
    for (int r = 0; r < g.R; ++r) {
      const int ih = p * g.stride - g.pad + r;
      if (ih < 0 || ih >= g.H) continue;
      for (int s = 0; s < g.S; ++s) {
        const int iw = q * g.stride - g.pad + s;
        if (iw < 0 || iw >= g.W) continue;
        acc = fmaf(act_ld(px + ih * g.W + iw), __ldg(pw + r * g.S + s), acc);
      }
    }
    act_st(out, i, ep.a ? conv_epilogue<XT>(acc, ep, c, (size_t)i) : acc);
  }
}

// ------------------------------------------------------------------------------------------------
// direct fp32 conv: any groups/stride/pad/kernel.  One thread: one output pixel x DK out channels.
// ------------------------------------------------------------------------------------------------
constexpr int DK = 8;
__global__ void __launch_bounds__(128) conv_direct_kernel(const float* __restrict__ x,
                                                          const float* __restrict__ w,
                                                          float* __restrict__ out, ConvGeom g, ConvEpilogue ep) {
  extern __shared__ float sw[];                             // [DK][Cg*R*S] weights of this k block
  const int Cg = g.C / g.groups, Kg = g.K / g.groups;
  const int kblocks_g = (Kg + DK - 1) / DK;
  const int kb = blockIdx.y;                                // (group, k block)
  const int grp = kb / kblocks_g;
  const int k0 = grp * Kg + (kb - grp * kblocks_g) * DK;
  const int kend = min(k0 + DK, (grp + 1) * Kg);
  const int wsz = Cg * g.R * g.S;
  for (int i = threadIdx.x; i < DK * wsz; i += blockDim.x) {
    const int kk = i / wsz;
    sw[i] = (k0 + kk < kend) ? w[(int64_t)(k0 + kk) * wsz + (i - kk * wsz)] : 0.0f;
  }
  __syncthreads();
  const int64_t npix = (int64_t)g.B * g.P * g.Q;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < npix; i += (int64_t)gridDim.x * blockDim.x) {
    const int q = (int)(i % g.Q);
    const int64_t t = i / g.Q;
    const int p = (int)(t % g.P);
    const int n = (int)(t / g.P);
    float acc[DK];
#pragma unroll
    for (int kk = 0; kk < DK; ++kk) acc[kk] = 0.0f;
    for (int c = 0; c < Cg; ++c) {
      const float* px = x + ((int64_t)n * g.C + grp * Cg + c) * g.H * g.W;
      for (int r = 0; r < g.R; ++r) {
        const int ih = p * g.stride - g.pad + r;
        if (ih < 0 || ih >= g.H) continue;
        for (int s = 0; s < g.S; ++s) {
          const int iw = q * g.stride - g.pad + s;
          if (iw < 0 || iw >= g.W) continue;
          const float v = __ldg(px + ih * g.W + iw);
          const float* pw = sw + (c * g.R + r) * g.S + s;
#pragma unroll
          for (int kk = 0; kk < DK; ++kk) acc[kk] = fmaf(v, pw[kk * wsz], acc[kk]);
        }
      }
    }
    for (int kk = 0; kk < DK && k0 + kk < kend; ++kk) {
      const size_t o = (size_t)((((int64_t)n * g.K + k0 + kk) * g.P + p) * g.Q + q);
      out[o] = ep.a ? conv_epilogue(acc[kk], ep, k0 + kk, o) : acc[kk];
    }
  }
}

// codes -> fp32 weights for the CUDA-core kernels
__global__ void decode_weights_kernel(const uint8_t* __restrict__ codes, const float* __restrict__ scale,
                                      float* __restrict__ w, int64_t n, int bits, int fsr) {
  const float s = *scale;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const uint32_t code = (bits <= 4) ? ((codes[i >> 1] >> ((i & 1) * 4)) & 0xFu) : codes[i];
    const int mag = code & ((1u << (bits - 1)) - 1u);
    float v = __fmul_rn(exp2_int((fsr - 1) - mag), s);
    w[i] = ((code >> (bits - 1)) & 1u) ? -v : v;
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static int sm_count() { return device_sm_count(); }     // per device (po2_common.cuh)

static bool fill_geom(ConvGeom& g, int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups) {
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || K <= 0 || R <= 0 || S <= 0 || stride <= 0 || pad < 0 || groups <= 0) return false;
  if (C % groups || K % groups) return false;
  g = ConvGeom{};
  g.B = B; g.C = C; g.H = H; g.W = W; g.K = K; g.R = R; g.S = S; g.stride = stride; g.pad = pad; g.groups = groups;
  g.P = (H + 2 * pad - R) / stride + 1;
  g.Q = (W + 2 * pad - S) / stride + 1;
  return g.P > 0 && g.Q > 0;
}

// the tensor-core kernels index activations with 32-bit offsets: x (B, Cin, HWin) and out (B, Cout, HWout) must each
// stay below 2^31 elements
static bool index_fits(int64_t B, int64_t Cin, int64_t HWin, int64_t Cout, int64_t HWout) {
  return B * Cin * HWin < (1ll << 31) && B * Cout * HWout < (1ll << 31);
}
static bool index_fits(const ConvGeom& g) { return index_fits(g.B, g.C, (int64_t)g.H * g.W, g.K, (int64_t)g.P * g.Q); }

// the filter windows of the tensor-core kernels: square 3x3 pad 1 or 1x1 pad 0
static bool tc_window(int R, int S, int pad) { return (R == 3 && S == 3 && pad == 1) || (R == 1 && S == 1 && pad == 0); }

// K3 takes: dense, tc_window, stride 1 or 2
static bool umma_shape_ok(const ConvGeom& g) {
  return g.groups == 1 && (g.stride == 1 || g.stride == 2) && tc_window(g.R, g.S, g.pad);
}

static size_t umma_smem_bytes(const ConvGeom& g) {
  return (size_t)g.b_slab_bytes + (size_t)g.nst * g.a_stage_bytes + (3 * K3_MAX_STAGES + 8) * 8 + 64;
}

// returns false if the shape does not fit the kernel's shared-memory plan.  bf16x: x is bf16 (16 bytes = 8 pixels on
// the producers' fast path)
static bool plan_umma(ConvGeom& g, bool tf32, bool bf16x = false) {
  const bool k3 = (g.R == 3);
  g.tf32 = tf32 ? 1 : 0;
  g.G = tf32 ? 4 : 8;
  const int G = g.G, KCH = 2 * G;                   // channels per plane entry / per MMA k-step
  if (!k3 && g.stride == 1) {
    // a 1x1 stride-1 conv has no spatial structure: view each image as ONE row of H*W pixels, which
    // makes 2x2 / 4x4 feature maps eligible for the 128-bit producer path (W % 4 == 0)
    g.W = g.H * g.W; g.H = 1; g.Q = g.P * g.Q; g.P = 1;
  }
  g.ntaps = g.R * g.S;
  g.pitch = g.Q + (k3 ? 1 : 0);
  g.rows_img = g.P + (k3 ? 1 : 0);
  g.top = k3 ? 1 : 0;
  g.Ltot = (g.B * g.rows_img + g.top) * g.pitch;
  int halo_after = 0;
  if (!k3) {
    g.nphase = 1; g.halo_before = 0;
    g.tap_phase[0] = 0; g.tap_off[0] = 0;
  } else if (g.stride == 1) {
    g.nphase = 1; g.halo_before = g.pitch + 1; halo_after = g.pitch + 1;
    for (int r = 0; r < 3; ++r) for (int s = 0; s < 3; ++s) {
      g.tap_phase[r * 3 + s] = 0;
      g.tap_off[r * 3 + s] = g.halo_before + (r - 1) * g.pitch + (s - 1);
    }
  } else {
    // stride 2: input row 2p+r-1 is parity phase (r != 1) at half-res row p - (r == 0); same for columns
    g.nphase = 4; g.halo_before = g.pitch + 1;
    for (int r = 0; r < 3; ++r) for (int s = 0; s < 3; ++s) {
      g.tap_phase[r * 3 + s] = ((r != 1) ? 2 : 0) | ((s != 1) ? 1 : 0);
      g.tap_off[r * 3 + s] = g.halo_before - (r == 0 ? g.pitch : 0) - (s == 0 ? 1 : 0);
    }
  }
  g.strip = 128 + g.halo_before + halo_after;
  g.Cpad = (g.C + KCH - 1) / KCH * KCH;
  // N tile: the whole-K weight slab of one tile must fit its smem budget
  const int Kp = (g.K + 15) / 16 * 16;
  int NT = Kp < 256 ? Kp : 256;
  const size_t eb = tf32 ? 4 : 2;                   // operand element bytes
  while (NT > 16 && (size_t)g.ntaps * g.Cpad * NT * eb > K3_B_BUDGET) NT -= 16;
  if ((size_t)g.ntaps * g.Cpad * NT * eb > K3_B_BUDGET) return false;
  g.ntiles_n = (Kp + NT - 1) / NT;
  g.nitems_m = (g.Ltot + 127) / 128;
  // too few (M item, N tile) pairs to occupy the SMs: narrow the N tile (each CTA then moves a
  // smaller weight slab; the activation strip is produced redundantly by CTAs that would otherwise idle)
  while (NT > 16 && g.nitems_m * ((Kp + (NT - 16) - 1) / (NT - 16)) <= sm_count()) NT -= 16;
  g.ntiles_n = (Kp + NT - 1) / NT;
  g.NT = ((Kp + g.ntiles_n - 1) / g.ntiles_n + 15) / 16 * 16;
  g.b_slab_bytes = (uint32_t)((size_t)g.ntaps * g.Cpad * g.NT * eb);
  // channels per A stage: keep a stage <= 32 KB so that >= 3 stages fit beside the slab
  int CC = g.Cpad;
  while (CC > KCH && (size_t)g.nphase * CC * g.strip * eb > 32 * 1024) CC -= KCH;
  g.CC = CC;
  g.nchunk = (g.Cpad + CC - 1) / CC;
  g.a_stage_bytes = (uint32_t)((size_t)g.nphase * CC * g.strip * eb);
  int nst = (int)((K3_SMEM_BUDGET - g.b_slab_bytes - 512) / g.a_stage_bytes);
  if (nst > K3_MAX_STAGES) nst = K3_MAX_STAGES;
  if (nst < 2) return false;
  g.nst = nst;
  int per_n = sm_count() / g.ntiles_n;
  if (per_n < 1) per_n = 1;
  g.m_step = g.nitems_m < per_n ? g.nitems_m : per_n;
  const int stages_per_cta = ((g.nitems_m + g.m_step - 1) / g.m_step) * g.nchunk;
  g.dual_issue = (g.nchunk == 1) ? 1 : 0;
  // a producer group skips the other groups' stages, so it can run ahead of the consumer; with one-bit
  // mbarrier phases it must stay within one wrap of the ring: groups (+ the one-tile reordering two
  // issuers can introduce) <= stages
  const int max_groups = g.nst - g.dual_issue;
  g.prod_groups = (stages_per_cta >= 4 && max_groups >= 4) ? 4 : ((stages_per_cta >= 2 && max_groups >= 2) ? 2 : 1);
  g.div_pitch = make_fastdiv((uint32_t)g.pitch);
  g.div_rows = make_fastdiv((uint32_t)g.rows_img);
  g.div_strip = make_fastdiv((uint32_t)g.strip);
  g.div_NT = make_fastdiv((uint32_t)g.NT);
  g.div_ncg = make_fastdiv((uint32_t)(g.Cpad / G));
  g.div_taps = make_fastdiv((uint32_t)g.ntaps);
  const int px = bf16x ? 8 : 4;
  g.vec4 = (g.stride == 1 && g.W % px == 0) ? 1 : 0;
  g.items_per_row = g.W / px + (g.pitch > g.W ? 1 : 0);
  g.div_ipr = make_fastdiv((uint32_t)(g.items_per_row > 0 ? g.items_per_row : 1));
  return true;
}

// PO2_CONV_TMA=0 keeps every shape on the register-fed kernel (A/B measurements)
static bool tma_enabled() {
  static const bool on = [] { const char* e = getenv("PO2_CONV_TMA"); return !(e && e[0] == '0'); }();
  return on;
}

}  // namespace po2
#include "po2_conv_tma.cuh"   // K3T: the TMA-fed tf32 form (plan_tma / launch_tma)
namespace po2 {

// Which kernel runs a conv, and how.  The forward plans with plan_fwd and the data gradient with plan_dgrad; every
// query and launch of a shape goes through one of them, so all of them make the same decision.
struct ConvPlan {
  int kind;              // po2_conv2d_kernel_kind: 0 direct fp32, 1 depthwise, 2 K3, 3 K3T, 4 small-pointwise GEMM
  ConvGeom g;            // through fill_geom, and for kinds 2 / 3 through plan_umma
  TmaPlan tp;            // kind 3
  size_t pack_bytes;     // the packed weight operand of kinds 2 / 3; 0 for the other kinds
  size_t workspace;      // what the launching entry point needs
  bool unpadded;         // kinds 2 / 3: the operand has no channel padding, so the fused quantizers can emit it
  int dtype;             // storage of x / out / residual: PO2_F32, or PO2_BF16 (kinds 1, 2 and 4 only)
};

static size_t round256(size_t n) { return (n + 255) / 256 * 256; }

// K3, or K3T where the TMA-fed kernel takes the planned geometry (it reads the 3x3 operand tap-minor); false: the
// shape does not fit K3's shared-memory plan.  A bf16 x runs on K3 with bf16 operands (exact, whatever the mode).
static bool plan_tc(ConvPlan& p, bool tf32) {
  const bool bf16x = p.dtype == PO2_BF16;
  if (!plan_umma(p.g, tf32 && !bf16x, bf16x)) return false;
  // pack_weights_kernel's 32-bit grid-stride loop runs over the operand's elements: keep it a stride below 2^31
  // (checked before the plan is filled in: a refused shape keeps kind, tapminor and pack_bytes of a CUDA-core plan)
  if ((int64_t)p.g.ntiles_n * p.g.NT * p.g.ntaps * p.g.Cpad >= (1ll << 30)) return false;
  p.kind = (tf32 && !bf16x && tma_enabled() && plan_tma(p.g, p.tp)) ? 3 : 2;
  p.g.tapminor = (p.kind == 3 && p.g.ntaps == 9) ? 1 : 0;
  p.pack_bytes = (size_t)p.g.ntiles_n * p.g.b_slab_bytes;
  p.unpadded = p.g.Cpad == p.g.C && p.g.ntiles_n * p.g.NT == p.g.K;
  return true;
}

// 0, PO2_E_SHAPE (not a conv shape), PO2_E_DTYPE, or PO2_E_UNSUPPORTED: a bf16 x on the fp32 CUDA cores (compute 1)
// or on the direct kernel.  dtype: the storage of x / out / residual, PO2_F32 or PO2_BF16 (weights are fp32 either way)
static int plan_fwd(ConvPlan& p, int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                    int compute, int dtype = PO2_F32) {
  p = ConvPlan{};
  if (dtype != PO2_F32 && dtype != PO2_BF16) return PO2_E_DTYPE;
  p.dtype = dtype;
  if (!fill_geom(p.g, B, C, H, W, K, R, S, stride, pad, groups)) return PO2_E_SHAPE;
  if (!index_fits(p.g)) return PO2_E_SIZE;
  // the pointwise layers on tiny feature maps go to the fp32 cluster GEMM of csrc/po2_conv_bwd.cu, not to K3 / K3T
  const bool pw_small = pw_small_takes(B, C, H, W, K, R, S, stride, pad, groups);
  if (compute == 1 || !umma_shape_ok(p.g) || pw_small || !plan_tc(p, compute == 2))
    p.kind = pw_small ? 4 : (groups == C && groups == K) ? 1 : 0;
  if (dtype == PO2_BF16 && (compute == 1 || p.kind == 0)) return PO2_E_UNSUPPORTED;
  // the decoded fp32 weights (codes input), then the packed operand
  const size_t wbytes = (size_t)K * (C / groups) * R * S * sizeof(float);
  p.workspace = round256(wbytes + (p.pack_bytes ? p.pack_bytes + 256 : 0));
  return 0;
}

// The data gradient of a stride-1 dense layer (x: B, C, H, W; w: K, C, R, S) is the forward conv of the output
// gradient (K channels) into C channels with the channel-transposed, 180-degree-rotated weight, on K3 / K3T.
// Returns 0, or the code po2_conv2d_dgrad refuses the shape with.
static int plan_dgrad(ConvPlan& p, int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                      int compute) {
  p = ConvPlan{};
  if (compute == 1 || stride != 1 || groups != 1 || !tc_window(R, S, pad)) return PO2_E_UNSUPPORTED;
  if (!fill_geom(p.g, B, K, H, W, C, R, S, 1, pad, 1)) return PO2_E_SHAPE;
  if (!index_fits(p.g)) return PO2_E_SIZE;
  if (!plan_tc(p, compute == 2)) return PO2_E_UNSUPPORTED;
  p.workspace = round256(p.pack_bytes + 256);
  return 0;
}

// the fused quantizers' description of the planned operand (layout: pack_weights_kernel / pack_store)
static PackArgs pack_args(const ConvGeom& g, void* Bp) {
  PackArgs pk = {};
  pk.Bp = Bp;
  pk.G = g.G; pk.C = g.C; pk.K = g.K; pk.taps = g.ntaps; pk.NT = g.NT; pk.ncg = g.C / g.G; pk.tapminor = g.tapminor;
  pk.div_ct = make_fastdiv((uint32_t)(g.C * g.ntaps));
  pk.div_t = make_fastdiv((uint32_t)g.ntaps);
  pk.div_nt = make_fastdiv((uint32_t)g.NT);
  return pk;
}
// ... and the data-gradient operand of the same weight; gd: the plan_dgrad geometry
static void add_dgrad_operand(PackArgs& pk, const ConvGeom& gd, void* Bp2) {
  pk.Bp2 = Bp2;
  pk.NT2 = gd.NT; pk.ncg2 = gd.C / gd.G; pk.tapminor2 = gd.tapminor;
  pk.div_nt2 = make_fastdiv((uint32_t)gd.NT);
}

// PO2_CONV_PDL_CHAIN=0: the entry points that take a packed operand launch the conv with a full dependency
static bool pdl_chain_enabled() {
  static const bool on = []() { const char* e = getenv("PO2_CONV_PDL_CHAIN"); return !(e && e[0] == '0'); }();
  return on;
}
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// K3's activation producers read x with 128-bit loads on the vec4 path (stride 1, W % 4 == 0; bf16: W % 8 == 0) and on
// the hw1 path (1x1 feature map, C % 4 == 0; bf16: C % 8 == 0); K3T's tensor map needs a 16-byte-aligned base too, and
// every geometry plan_tma takes is stride 1 with W % 4 == 0, i.e. has vec4 set.  PO2_E_ALIGN before any launch when x
// does not allow that.
static int umma_check_x(const void* x, const ConvPlan& p) {
  const ConvGeom& g = p.g;
  const bool wide_loads = g.vec4 || (g.H * g.W == 1 && g.C % (p.dtype == PO2_BF16 ? 8 : 4) == 0);
  return (wide_loads && !aligned16(x)) ? PO2_E_ALIGN : 0;
}

// w (fp32 PO2-grid weights, or codes) -> the planned operand at Bp.  transpose: the data-gradient conv's operand
// from the forward weight
static int launch_pack(const ConvPlan& p, const void* w, int w_format, const float* scale, int bits, int fsr,
                       int transpose, void* Bp, cudaStream_t st) {
  const int64_t total = (int64_t)p.pack_bytes / (p.g.tf32 ? 4 : 2);
  const int pblocks = (int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
  const bool codes = w_format == PO2_W_CODES;
  pack_weights_kernel<<<pblocks, 256, 0, st>>>(codes ? nullptr : (const float*)w, codes ? (const uint8_t*)w : nullptr,
                                               codes ? nullptr : scale, Bp, p.g, bits, fsr, transpose);
  return (int)cudaGetLastError();
}

// The K3 / K3T conv on the packed operand Bp.  pdl 1: launched with programmatic stream serialization -- ONLY legal
// when the kernel directly in front of it in the stream is one of ours that was launched with a full dependency
// (pack_weights_kernel, fused_kernel): the conv's producers read x without a griddepcontrol.wait, which is safe only if
// x's producer finished before that kernel started.  pdl 2 (chain): the operand was packed earlier and the kernel
// directly in front produced x (a norm kernel): K3T is launched programmatically with the waits of TmaPlan::pdl == 2,
// K3 with a full dependency.  pdl 0: a full dependency.
static int launch_conv(const ConvPlan& p, const void* x, const void* Bp, const float* scale, void* out, int pdl,
                       const ConvEpilogue& ep, cudaStream_t st) {
  const ConvGeom& g = p.g;
  // (the operand may already be packed in K3T's layout: an x that cannot be described by a tensor map is an error
  // here, not a fallback; a misaligned one is refused with PO2_E_ALIGN before any launch)
  if (p.kind == 3) return launch_tma(x, (const uint8_t*)Bp, scale, out, g, p.tp, st, pdl, ep);
  static PerDeviceOnce attr_once;                       // the opt-in shared-memory size is a per-device attribute
  cudaError_t e = attr_once.run([]() -> cudaError_t {
    const int smax = (int)K3_SMEM_BUDGET + 1024;
    cudaError_t a = cudaFuncSetAttribute(conv_umma_kernel<1, false, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (a == cudaSuccess) a = cudaFuncSetAttribute(conv_umma_kernel<9, false, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (a == cudaSuccess) a = cudaFuncSetAttribute(conv_umma_kernel<1, true, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (a == cudaSuccess) a = cudaFuncSetAttribute(conv_umma_kernel<9, true, float>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (a == cudaSuccess)
      a = cudaFuncSetAttribute(conv_umma_kernel<1, false, __nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    if (a == cudaSuccess)
      a = cudaFuncSetAttribute(conv_umma_kernel<9, false, __nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
    return a;
  });
  if (e != cudaSuccess) return (int)e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(g.ntiles_n * g.m_step));
  cfg.blockDim = dim3(K3_THREADS);
  cfg.dynamicSmemBytes = umma_smem_bytes(g);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // overlap our prologue with the pack kernel
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl == 1 ? 1 : 0;
  const float* xf = (const float*)x;
  const uint8_t* bpc = (const uint8_t*)Bp;
  float* of = (float*)out;
  if (p.dtype == PO2_BF16) {
    const __nv_bfloat16* xb = (const __nv_bfloat16*)x;
    __nv_bfloat16* ob = (__nv_bfloat16*)out;
    if (g.ntaps == 1) e = cudaLaunchKernelEx(&cfg, conv_umma_kernel<1, false, __nv_bfloat16>, xb, bpc, scale, ob, g, ep);
    else e = cudaLaunchKernelEx(&cfg, conv_umma_kernel<9, false, __nv_bfloat16>, xb, bpc, scale, ob, g, ep);
  } else if (g.tf32) {
    if (g.ntaps == 1) e = cudaLaunchKernelEx(&cfg, conv_umma_kernel<1, true, float>, xf, bpc, scale, of, g, ep);
    else e = cudaLaunchKernelEx(&cfg, conv_umma_kernel<9, true, float>, xf, bpc, scale, of, g, ep);
  } else {
    if (g.ntaps == 1) e = cudaLaunchKernelEx(&cfg, conv_umma_kernel<1, false, float>, xf, bpc, scale, of, g, ep);
    else e = cudaLaunchKernelEx(&cfg, conv_umma_kernel<9, false, float>, xf, bpc, scale, of, g, ep);
  }
  return (int)e;
}


// ------------------------------------------------------------------------------------------------
// K5: weight gradient of the dense stride-1 convs on the tensor cores (SURVEY.md section 8f "next" #2:
// the gradient lands in the fp32 master weight through the straight-through estimator, so this IS the
// STE backward of QuantizedConv2d).
//
//   gw[k][c][r][s] = sum over (n, p, q) of  go[n][k][p][q] * x[n][c][p + r - pad][q + s - pad]
//
// A GEMM whose reduction dimension is the pixel index: D[k][(tap, c)] += go^T x_tap.  Both operands
// are staged exactly like the forward kernel's activation strips -- planes [channel / 8][flat padded
// position][8 channels] of bf16, 16 bytes per position -- which is UMMA's MN-major no-swizzle
// canonical layout with the reduction (position) index running along K: 8 consecutive positions
// form a core matrix (LBO = 128 B between K blocks, SBO = plane stride between 8-channel blocks).  A
// filter tap is again nothing but a shift of the x descriptor's start address by (r*pitch + s)
// positions; go's pad positions are zero, so the shared zero column / row contribute nothing.
//   * one CTA accumulates ALL its 128-position tiles into TMEM (M = 128 rows = out channels, of which
//     K are real; one N = Cpad column block per tap) and runs the epilogue once;
//   * per-CTA partial results go to a workspace, conv_wgrad_reduce_kernel adds them in a fixed order
//     (deterministic, unlike atomics) and writes gw[K][C][R][S];
//   * taps are split over blockIdx.y when 9 * Cpad columns exceed TMEM's 512.
// ------------------------------------------------------------------------------------------------
struct WgGeom {
  int K, Kplanes;            // out channels (<= 128), ceil(K / 8)
  int M;                     // MMA M: 64 (K <= 64) or 128 -- rows >= K are garbage and never read
  int Cplanes;               // Cpad / 8
  int ntaps, taps_per_cta, tap_splits;
  int copies;                // 3: x is staged as three column-shifted copies, one MMA covers the taps (r, 0..2)
  int groups_per_cta;        // MMA groups (taps, or filter rows when copies == 3) per CTA = taps_per_cta / copies
  int m_ctas;                // CTAs along the position dimension
  int nst, prod_groups;
  uint32_t go_bytes, x_bytes, stage_bytes;
  uint32_t ncols;            // TMEM columns
};
constexpr uint32_t WG_A_SPAN = 16 * 128 * 16;      // the A descriptor spans M/8 <= 16 planes of 128 positions

// idesc: D=f32, A=B=bf16, both MN-major ("transposed"), M=128, N
__device__ __forceinline__ uint32_t make_idesc_mn(uint32_t m, uint32_t n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((n >> 3) << 17) | ((m >> 4) << 24);
}

// fill planes [ngrp][strip][8 x bf16] of `stage` with channels [0, 8*ngrp) of src (fp32 NCHW, nC
// channels, zero beyond) at flat positions [Ls, Ls + strip); stride-1 geometry of g
// copies == 3: the planes are written three times, copy s shifted by (s - 1) positions
// (copy_s[i] = strip[i + s - 1]; copy stride = ngrp * strip * 16 bytes), so that the three taps of a
// filter row become ONE MMA with N = 3 * channels.
__device__ __forceinline__ void store_copies(uint8_t* plane, int lloc, int strip, const uint4& val, int copies,
                                             size_t copy_bytes) {
  if (copies == 1) { *reinterpret_cast<uint4*>(plane + (size_t)lloc * 16) = val; return; }
  if (lloc + 1 < strip) *reinterpret_cast<uint4*>(plane + (size_t)(lloc + 1) * 16) = val;                // s = 0
  *reinterpret_cast<uint4*>(plane + copy_bytes + (size_t)lloc * 16) = val;                               // s = 1
  if (lloc >= 1) *reinterpret_cast<uint4*>(plane + 2 * copy_bytes + (size_t)(lloc - 1) * 16) = val;      // s = 2
}

__device__ __forceinline__ void produce_planes_bf16(const ConvGeom& g, const float* __restrict__ src, int nC, int ngrp,
                                                    int strip, int Ls, uint8_t* stage, int gt, int NPG,
                                                    int copies = 1) {
  const size_t copy_bytes = (size_t)ngrp * strip * 16;
  const int H = g.H, W = g.W, HW = H * W;
  if (g.vec4) {
    const int pitch = g.pitch, W4 = W >> 2, ipr = g.items_per_row;
    const int rowA = Ls >= 0 ? fdiv(Ls, g.div_pitch) : -((-Ls + pitch - 1) / pitch);
    const int rowB = fdiv(Ls + strip - 1, g.div_pitch);
    const int jA = min((Ls - rowA * pitch) >> 2, ipr - 1);
    const int jB = (rowB - rowA) * ipr + min((Ls + strip - 1 - rowB * pitch) >> 2, ipr - 1);
    const int nrow_items = jB - jA + 1;
    const int nall = ngrp * nrow_items;
    const float inv_items = 1.0f / (float)nrow_items;
    for (int i0 = gt; i0 < nall; i0 += 2 * NPG) {
      float4 v[2][8];
      int lbase[2], npos[2], gsel[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {                    // 16 x 128-bit loads in flight per thread
        const int i = i0 + u * NPG;
        lbase[u] = 0; npos[u] = 0; gsel[u] = 0;
        bool ok = false;
        int idx = 0, cvalid = 0;
        if (i < nall) {
          int grp = (int)(((float)i + 0.5f) * inv_items);
          int j = i - grp * nrow_items;
          if (j < 0) { --grp; j += nrow_items; } else if (j >= nrow_items) { ++grp; j -= nrow_items; }
          j += jA;
          const int rr = fdiv(j, g.div_ipr);
          const int q4 = j - rr * ipr;
          const int row = rowA + rr;
          const int c0 = grp * 8;
          gsel[u] = grp;
          cvalid = nC - c0;
          lbase[u] = row * pitch + q4 * 4 - Ls;
          npos[u] = q4 < W4 ? 4 : pitch - W;
          const int r0 = row - g.top;
          if (q4 < W4 && r0 >= 0) {
            const int img = fdiv(r0, g.div_rows);
            const int a = r0 - img * g.rows_img;
            if (a < H && img < g.B) { ok = true; idx = ((img * nC + c0) * H + a) * W + q4 * 4; }
          }
        }
        const float4* px = reinterpret_cast<const float4*>(src + idx);
#pragma unroll
        for (int c = 0; c < 8; ++c)
          v[u][c] = (ok && c < cvalid) ? __ldg(px + (size_t)c * (HW >> 2)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        uint8_t* sgrp = stage + (size_t)gsel[u] * strip * 16;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int lloc = lbase[u] + e;
          if (e < npos[u] && lloc >= 0 && lloc < strip) {
            float ch[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) ch[c] = e == 0 ? v[u][c].x : e == 1 ? v[u][c].y : e == 2 ? v[u][c].z : v[u][c].w;
            store_copies(sgrp, lloc, strip, pack_channels<false>(ch), copies, copy_bytes);
          }
        }
      }
    }
  } else {
    const int nitem = ngrp * strip;
    for (int i = gt; i < nitem; i += NPG) {
      const int grp = i / strip;
      const int lloc = i - grp * strip;
      float v[8];
      int img, a, b, cvalid = 0, idx = 0;
      if (decode_pos(g, Ls + lloc, img, a, b) && a < H && b < W) {
        cvalid = nC - grp * 8;
        idx = ((img * nC + grp * 8) * H + a) * W + b;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = (j < cvalid) ? __ldg(src + idx + j * HW) : 0.0f;
      store_copies(stage + (size_t)grp * strip * 16, lloc, strip, pack_channels<false>(v), copies, copy_bytes);
    }
  }
}

__global__ void __launch_bounds__(K3_THREADS, 1) conv_wgrad_umma_kernel(const float* __restrict__ x,
                                                                        const float* __restrict__ go,
                                                                        float* __restrict__ partial, ConvGeom g,
                                                                        WgGeom wg) {
  extern __shared__ __align__(128) uint8_t smem[];
  // stage = [go planes | x planes]; WG_A_SPAN bytes of slack behind the ring keep the 16-plane A
  // descriptor of the last stage inside the allocation (rows >= K of D are garbage and never read)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)wg.nst * wg.stage_bytes + WG_A_SPAN);
  uint64_t* full = bars;
  uint64_t* empty = bars + K3_MAX_STAGES;
  uint64_t* tfull = bars + 2 * K3_MAX_STAGES;
  uint64_t* tready = tfull + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tready + 1);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m_first = blockIdx.x, m_step = wg.m_ctas, nitems = g.nitems_m, nst = wg.nst;
  const int tap0 = blockIdx.y * wg.taps_per_cta;
  const int ntap = min(wg.taps_per_cta, wg.ntaps - tap0);
  const int Cpad = wg.Cplanes * 8;
  // conv_wgrad_reduce_kernel (launched with programmatic stream serialization) may be scheduled early;
  // it waits for this grid's completion before reading the partials
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
#ifdef PO2_K3_TRACE
  for (int i = tid; i < 8 * 64; i += K3_THREADS) k3_trace_smem[i] = 0;
  __syncthreads();
#endif
  if (tid == 0) K3_TRACE(6, 0);

  if (warp == K3_EPI_WARPS + 1 && lane == 0) {
    for (int i = 0; i < nst; ++i) { mbar_init(full + i, K3_PROD_WARPS / wg.prod_groups); mbar_init(empty + i, 1); }
    mbar_init(tfull, 1);
    mbar_init(tready, 1);
    fence_mbar_init();
  }
  __syncthreads();
  uint32_t tmem_base = 0;
  if (warp == K3_EPI_WARPS) {
    tmem_alloc(tmem_slot, wg.ncols);
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(tready);
    tc_fence_after();
    tmem_base = *tmem_slot;
  } else if (warp < K3_EPI_WARPS) {
    mbar_wait(tready, 0);
    tc_fence_after();
    tmem_base = *tmem_slot;
  }
  if (tid == 0) K3_TRACE(6, 1);

  if (warp == K3_EPI_WARPS) {
    // =========================== MMA issuer ===========================
    const bool leader = elect_one();
    const uint32_t idesc = make_idesc_mn((uint32_t)wg.M, (uint32_t)(wg.copies * Cpad));
    // descriptor words: lo = start>>4 | LBO>>4 << 16 (K-block stride: 8 positions = 128 B);
    //                   hi = SBO>>4 (MN-block stride: one plane) | version 1 << 14
    const uint32_t a_hi = (uint32_t)(128 * 16 >> 4) | (1u << 14);
    const uint32_t b_hi = (uint32_t)g.strip | (1u << 14);
    const uint32_t lo_fixed = 8u << 16;
    const uint32_t s0_16 = smem_u32(smem) >> 4, stage16 = wg.stage_bytes >> 4, go16 = wg.go_bytes >> 4;
    uint32_t s = 0, sphase = 0, tile = 0;
    for (int m = m_first; m < nitems; m += m_step, ++tile) {
      mbar_wait(full + s, sphase);
      tc_fence_after();
      if (leader) K3_TRACE(0, 2 * (int)tile);
      if (leader) {
        const uint32_t a16 = s0_16 + s * stage16, b16 = a16 + go16;
        // one MMA group = one tap, or (copies == 3) one filter row: N = 3*Cpad columns (s, c) read from
        // the three shifted copies at the CENTRE tap's offset -- the same column order tap*Cpad + c
        for (int t = 0; t < ntap; t += wg.copies) {
          const uint32_t d = tmem_base + (uint32_t)(t * Cpad);
          const uint32_t boff = b16 + (uint32_t)g.tap_off[tap0 + t + (wg.copies == 3 ? 1 : 0)];
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {                       // 16 positions per MMA
            const uint64_t ad = ((uint64_t)a_hi << 32) | (lo_fixed | ((a16 + ks * 16) & 0x3FFFu));
            const uint64_t bd = ((uint64_t)b_hi << 32) | (lo_fixed | ((boff + ks * 16) & 0x3FFFu));
            umma<false>(d, ad, bd, idesc, (uint32_t)((tile | ks) != 0));
          }
        }
        umma_commit(empty + s);
        K3_TRACE(0, 2 * (int)tile + 1);
      }
      __syncwarp();
      if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
    }
    if (leader) umma_commit(tfull);
    __syncwarp();
  } else if (warp < K3_EPI_WARPS) {
    // =========================== epilogue: TMEM -> partial[cta][tap][k][c] ===========================
    const int K = wg.K, C = g.C;
    mbar_wait(tfull, 0);
    tc_fence_after();
    if (warp == 0 && lane == 0) K3_TRACE(1, 0);
    // M = 128: D row i sits in TMEM lane i.  M = 64: each warp's 32-lane partition holds 16 rows in its
    // lanes 0..15 (row = 16 * warp + lane)
    const int rows_per_warp = wg.M == 64 ? 16 : 32;
    if (warp * rows_per_warp < K) {                              // this warp's TMEM lanes hold real out channels
      const int k = lane < rows_per_warp ? warp * rows_per_warp + lane : K;
      // partial[cta][tap][k][c]: a lane owns row k and writes its 16 channels of a column block as four
      // 128-bit stores (one warp runs this epilogue alone, so every instruction's latency is exposed:
      // few, wide stores and 32-bit index arithmetic)
      float* pbase = partial + (size_t)blockIdx.x * wg.ntaps * C * K;
      const bool vec = (C & 3) == 0;
      for (int t = 0; t < ntap; ++t) {
        float* prow = pbase + ((tap0 + t) * K + k) * C;            // k == K for idle lanes: never dereferenced
        for (int cb = 0; cb < Cpad / 16; ++cb) {
          uint32_t r[16];
          tmem_ld16(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(t * Cpad + cb * 16), r);
          if (k < K) {
            const int c0 = cb * 16;
            if (vec && c0 + 16 <= C) {
#pragma unroll
              for (int q = 0; q < 4; ++q)
                *reinterpret_cast<uint4*>(prow + c0 + 4 * q) = make_uint4(r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]);
            } else {
#pragma unroll
              for (int j = 0; j < 16; ++j)
                if (c0 + j < C) prow[c0 + j] = __uint_as_float(r[j]);
            }
          }
        }
      }
    }
    tc_fence_before();
    if (warp == 0 && lane == 0) K3_TRACE(1, 1);
  } else if (warp >= K3_EPI_WARPS + K3_MMA_WARPS) {
    // =========================== producers: go tile + x strip of every stage ===========================
    const int ngroups = wg.prod_groups;
    const int WPG = K3_PROD_WARPS / ngroups, NPG = 32 * WPG;
    const int pw = warp - (K3_EPI_WARPS + K3_MMA_WARPS);
    const int grp_id = pw / WPG;
    const int gt = tid - 32 * (K3_EPI_WARPS + K3_MMA_WARPS) - grp_id * NPG;
    uint32_t s = 0, sphase = 0, it = 0;
    int turn = 0;
    for (int m = m_first; m < nitems; m += m_step, ++it) {
      const uint32_t s_cur = s, ph_cur = sphase;
      const bool mine = (turn == grp_id);
      if (++s == (uint32_t)nst) { s = 0; sphase ^= 1; }
      if (++turn == ngroups) turn = 0;
      if (!mine) continue;
      mbar_wait(empty + s_cur, ph_cur ^ 1);
      if (gt == 0) K3_TRACE(2 + grp_id, 2 * (int)(it / ngroups));
      uint8_t* stage = smem + (size_t)s_cur * wg.stage_bytes;
      produce_planes_bf16(g, go, wg.K, wg.Kplanes, 128, m * 128, stage, gt, NPG);
      produce_planes_bf16(g, x, g.C, wg.Cplanes, g.strip, m * 128 - g.halo_before, stage + wg.go_bytes, gt, NPG,
                          wg.copies);
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(full + s_cur);
      if (gt == 0) K3_TRACE(2 + grp_id, 2 * (int)(it / ngroups) + 1);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (tid == 0) K3_TRACE(6, 2);
#ifdef PO2_K3_TRACE
  __syncthreads();
  if (g_k3_trace && blockIdx.x < 4 && blockIdx.y == 0)
    for (int i = tid; i < 8 * 64; i += K3_THREADS) g_k3_trace[blockIdx.x * 8 * 64 + i] = k3_trace_smem[i];
#endif
  if (warp == K3_EPI_WARPS) tmem_dealloc(tmem_base, wg.ncols);
}

// gw[(k*C + c)*ntaps + tap] = sum over CTAs of partial[cta][tap][k][c], in CTA order
__global__ void __launch_bounds__(256) conv_wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ gw,
                                                                int nparts, int K, int C, int ntaps) {
  __shared__ float sm[8][32];
  asm volatile("griddepcontrol.wait;" ::: "memory");            // the partials are the main kernel's output
  const int n = ntaps * C * K;
  const int o = blockIdx.x * 32 + (threadIdx.x & 31);           // index in the partial layout [tap][k][c]
  const int j = threadIdx.x >> 5;
  float acc = 0.f;
  if (o < n) {
    // four independent loads per round (an in-order warp would otherwise pay one L2 latency per partial);
    // the summation order stays fixed: p = j, j+8, j+16, ...
    const float* src = partial + o;
    int p = j;
    for (; p + 24 < nparts; p += 32) {
      const float v0 = __ldcg(src + (size_t)p * n), v1 = __ldcg(src + (size_t)(p + 8) * n);
      const float v2 = __ldcg(src + (size_t)(p + 16) * n), v3 = __ldcg(src + (size_t)(p + 24) * n);
      acc += v0; acc += v1; acc += v2; acc += v3;
    }
    for (; p < nparts; p += 8) acc += __ldcg(src + (size_t)p * n);
  }
  sm[j][threadIdx.x & 31] = acc;
  __syncthreads();
  if (j == 0 && o < n) {
    float t = 0.f;
#pragma unroll
    for (int q = 0; q < 8; ++q) t += sm[q][threadIdx.x];
    const int c = o % C, tk = o / C, k = tk % K, tap = tk / K;
    gw[((size_t)k * C + c) * ntaps + tap] = t;
  }
}

int launch_wgrad_reduce(const float* partial, float* gw, int nparts, int K, int C, int ntaps, cudaStream_t st) {
  const int n = ntaps * C * K;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)((n + 31) / 32));
  cfg.blockDim = dim3(256);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return (int)cudaLaunchKernelEx(&cfg, conv_wgrad_reduce_kernel, partial, gw, nparts, K, C, ntaps);
}

static bool plan_wgrad(ConvGeom& g, WgGeom& wg) {
  // g: forward geometry already through plan_umma(g, false) (flat padded space, tap offsets, producer fast path)
  if (g.K > 128 || g.Cpad > 256) return false;
  wg.K = g.K;
  wg.M = g.K <= 64 ? 64 : 128;
  wg.Kplanes = (g.K + 7) / 8;
  wg.Cplanes = g.Cpad / 8;
  wg.ntaps = g.ntaps;
  // three shifted copies triple the producers' shared-memory stores: a win while the MMAs are tiny
  // (N = 16 / 32 per tap), a loss from 64 channels on (measured, profiles/r01_wgrad_layers_*.json)
  wg.copies = (g.ntaps == 9 && g.Cpad <= 32) ? 3 : 1;
  const int ngroups = wg.ntaps / wg.copies;                                // MMA groups: taps or filter rows
  int gpc = 512 / (wg.copies * g.Cpad);                                    // groups whose columns fit TMEM
  if (gpc > ngroups) gpc = ngroups;
  if (gpc < 1) return false;
  wg.tap_splits = (ngroups + gpc - 1) / gpc;
  gpc = (ngroups + wg.tap_splits - 1) / wg.tap_splits;                     // balance the splits
  wg.groups_per_cta = gpc;
  wg.taps_per_cta = gpc * wg.copies;
  uint32_t ncols = 32;
  while ((int)ncols < wg.taps_per_cta * g.Cpad) ncols <<= 1;
  wg.ncols = ncols;
  wg.go_bytes = (uint32_t)wg.Kplanes * 128 * 16;
  wg.x_bytes = (uint32_t)wg.copies * wg.Cplanes * g.strip * 16;
  wg.stage_bytes = wg.go_bytes + wg.x_bytes;
  int nst = (int)((K3_SMEM_BUDGET - WG_A_SPAN - 512) / wg.stage_bytes);
  if (nst > K3_MAX_STAGES) nst = K3_MAX_STAGES;
  if (nst < 2) return false;
  wg.nst = nst;
  int m_ctas = sm_count() / wg.tap_splits;
  if (m_ctas < 1) m_ctas = 1;
  if (m_ctas > g.nitems_m) m_ctas = g.nitems_m;
  wg.m_ctas = m_ctas;
  // producer groups fill different stages concurrently; a CTA with a single tile wants all eight
  // warps on that one stage, so size the groups for the typical (floor) number of tiles per CTA
  const int stages_per_cta = g.nitems_m / m_ctas;
  wg.prod_groups = (stages_per_cta >= 4 && nst >= 4) ? 4 : ((stages_per_cta >= 2 && nst >= 2) ? 2 : 1);
  // the 14-bit descriptor start field (>> 4) covers 256 KB: every stage address fits
  return true;
}

static size_t wgrad_partial_bytes(const ConvGeom& g, const WgGeom& wg) {
  return (size_t)wg.m_ctas * wg.ntaps * g.C * g.K * sizeof(float);
}

}  // namespace po2
#include "po2_wgrad_tma.cuh"   // K5T: the TMA-fed tf32 weight gradient

using namespace po2;

extern "C" {

#ifdef PO2_K3_TRACE
int po2_debug_set_trace(void* buf) {
  long long* p = (long long*)buf;
  return (int)cudaMemcpyToSymbol(g_k3_trace, &p, sizeof(p));
}
#endif

size_t po2_conv2d_workspace(int B, int C, int H, int W, int K, int R, int S, int stride, int pad,
                            int groups, int compute) {
  return po2_conv2d_workspace_dt(B, C, H, W, K, R, S, stride, pad, groups, compute, PO2_F32);
}

size_t po2_conv2d_workspace_dt(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                               int compute, int dtype) {
  ConvPlan p;
  return plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute, dtype) ? 0 : p.workspace;
}

// which kernel po2_conv2d_fwd runs for this geometry: 0 direct fp32, 1 depthwise, 2 tcgen05 with the
// register-fed activation producer, 3 tcgen05 with the tensor-map TMA producer (K3T), 4 fp32 cluster GEMM for
// pointwise layers on <= 16-pixel feature maps; < 0: PO2_E_*
int po2_conv2d_kernel_kind(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                           int compute) {
  return po2_conv2d_kernel_kind_dt(B, C, H, W, K, R, S, stride, pad, groups, compute, PO2_F32);
}

int po2_conv2d_kernel_kind_dt(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                              int compute, int dtype) {
  ConvPlan p;
  const int e = plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute, dtype);
  return e ? e : p.kind;
}

static int check_epilogue(const float* ep_a, const float* ep_b, int act) {
  if (act < 0 || act > 3) return PO2_E_MODE;
  if (!ep_a != !ep_b) return PO2_E_NULL;
  return 0;
}

int po2_conv2d_fwd(const void* x, const void* w, const float* scale, void* out, int B, int C, int H,
                   int W, int K, int R, int S, int stride, int pad, int groups, int w_format,
                   int bits, int fsr, int compute, void* workspace, size_t workspace_bytes,
                   void* stream) {
  return po2_conv2d_fwd_ep(x, w, scale, out, B, C, H, W, K, R, S, stride, pad, groups, w_format, bits, fsr, compute, workspace,
                           workspace_bytes, nullptr, nullptr, nullptr, 0, stream);
}

// the same conv with a per-out-channel affine (eval-mode BatchNorm folded in), residual add and activation in
// its epilogue: out = act(conv(x, W) * ep_a[k] + ep_b[k] + residual)
int po2_conv2d_fwd_ep(const void* x, const void* w, const float* scale, void* out, int B, int C, int H,
                      int W, int K, int R, int S, int stride, int pad, int groups, int w_format,
                      int bits, int fsr, int compute, void* workspace, size_t workspace_bytes,
                      const float* ep_a, const float* ep_b, const void* residual, int act, void* stream) {
  return po2_conv2d_fwd_ep_dt(x, w, scale, out, B, C, H, W, K, R, S, stride, pad, groups, w_format, bits, fsr, compute,
                              workspace, workspace_bytes, ep_a, ep_b, residual, act, PO2_F32, stream);
}

int po2_conv2d_fwd_ep_dt(const void* x, const void* w, const float* scale, void* out, int B, int C, int H,
                         int W, int K, int R, int S, int stride, int pad, int groups, int w_format,
                         int bits, int fsr, int compute, void* workspace, size_t workspace_bytes,
                         const float* ep_a, const float* ep_b, const void* residual, int act, int dtype, void* stream) {
  if (!x || !w || !out) return PO2_E_NULL;
  if (int e = check_epilogue(ep_a, ep_b, act)) return e;
  if (!ep_a && (residual || act)) return PO2_E_NULL;
  const ConvEpilogue ep{ep_a, ep_b, (const float*)residual, act};
  ConvPlan p;
  if (int e = plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute, dtype)) return e;
  const ConvGeom& g = p.g;
  if (w_format != PO2_W_F32_PO2 && w_format != PO2_W_CODES) return PO2_E_UNSUPPORTED;
  if (w_format == PO2_W_CODES && (!scale || bits < 2 || bits > 8)) return PO2_E_BITS;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t wn = (int64_t)K * (C / groups) * R * S;
  const size_t wbytes = round256((size_t)wn * sizeof(float));

  if (p.pack_bytes) {
    if (!workspace || workspace_bytes < p.workspace) return PO2_E_WORKSPACE;
    if (int a = umma_check_x(x, p)) return a;
    void* Bp = reinterpret_cast<char*>(workspace) + wbytes;
    if (int e = launch_pack(p, w, w_format, scale, bits, fsr, 0, Bp, st)) return e;
    return launch_conv(p, x, Bp, scale, out, 1, ep, st);
  }
  // the small-pointwise GEMM reads rows of the fp32 weight with 128-bit loads when C % 4 == 0
  if (p.kind == 4 && C % 4 == 0 && !aligned16(w_format == PO2_W_CODES ? workspace : w)) return PO2_E_ALIGN;
  // CUDA-core paths work on fp32 weights
  const float* wf = (const float*)w;
  if (w_format == PO2_W_CODES) {
    if (!workspace || workspace_bytes < wbytes) return PO2_E_WORKSPACE;
    decode_weights_kernel<<<(int)((wn + 255) / 256 < 1184 ? (wn + 255) / 256 : 1184), 256, 0, st>>>(
        (const uint8_t*)w, scale, (float*)workspace, wn, bits, fsr);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    wf = (const float*)workspace;
  }
  if (p.kind == 4) return launch_pw_small(x, wf, out, B, C, H * W, K, ep, dtype, st);
  if (p.kind == 1) {
    const int64_t total = (int64_t)B * C * g.P * g.Q;
    // vector kernel: 3x3 pad 1, stride 1 or 2, rows and outputs in whole 16-byte groups
    if (R == 3 && S == 3 && pad == 1 && (stride == 1 || stride == 2) && W % 4 == 0 && g.Q % 4 == 0 &&
        (stride == 1 || W == 2 * g.Q) && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
      DwGeom d;
      d.C = C; d.H = H; d.W = W; d.P = g.P; d.Q = g.Q; d.Q4 = g.Q / 4; d.stride = stride;
      d.total = (int)(total / 4);
      d.div_q4 = make_fastdiv((uint32_t)d.Q4); d.div_p = make_fastdiv((uint32_t)g.P); d.div_c = make_fastdiv((uint32_t)C);
      const int blocks = (int)((d.total + 255) / 256 < sm_count() * 16 ? (d.total + 255) / 256 : sm_count() * 16);
      const bool bf = dtype == PO2_BF16;
      using BF = __nv_bfloat16;
      if (stride == 1 && bf) conv_depthwise_vec_kernel<1, BF><<<blocks, 256, 0, st>>>((const BF*)x, wf, (BF*)out, d, ep);
      else if (stride == 1) conv_depthwise_vec_kernel<1, float><<<blocks, 256, 0, st>>>((const float*)x, wf, (float*)out, d, ep);
      else if (bf) conv_depthwise_vec_kernel<2, BF><<<blocks, 256, 0, st>>>((const BF*)x, wf, (BF*)out, d, ep);
      else conv_depthwise_vec_kernel<2, float><<<blocks, 256, 0, st>>>((const float*)x, wf, (float*)out, d, ep);
      return (int)cudaGetLastError();
    }
    const int blocks = (int)((total + 255) / 256 < (int64_t)sm_count() * 16 ? (total + 255) / 256 : (int64_t)sm_count() * 16);
    const FastDiv dq = make_fastdiv((uint32_t)g.Q), dp = make_fastdiv((uint32_t)g.P), dc = make_fastdiv((uint32_t)C);
    if (dtype == PO2_BF16)
      conv_depthwise_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>((const __nv_bfloat16*)x, wf, (__nv_bfloat16*)out, g,
                                                                   dq, dp, dc, ep);
    else
      conv_depthwise_kernel<float><<<blocks, 256, 0, st>>>((const float*)x, wf, (float*)out, g, dq, dp, dc, ep);
    return (int)cudaGetLastError();
  }
  const int Cg = C / groups, Kg = K / groups;
  const size_t smem = (size_t)DK * Cg * R * S * sizeof(float);
  if (smem > 200 * 1024) return PO2_E_SHAPE;
  static PerDeviceOnce direct_once;
  if (cudaError_t e = direct_once.run([]() -> cudaError_t {
        return cudaFuncSetAttribute(conv_direct_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      })) return (int)e;
  const int64_t npix = (int64_t)B * g.P * g.Q;
  const int kblocks = groups * ((Kg + DK - 1) / DK);
  int bx = (int)((npix + 127) / 128);
  const int cap = sm_count() * 16 / (kblocks < 16 ? kblocks : 16) + 1;
  if (bx > cap) bx = cap;
  conv_direct_kernel<<<dim3(bx, kblocks), 128, smem, st>>>((const float*)x, wf, (float*)out, g, ep);
  return (int)cudaGetLastError();
}

// Data gradient of the quantized conv: gx = conv_transpose(g, W), computed as a forward conv of g with
// the channel-transposed, 180-degree-rotated weights on the same tensor-core kernel (stride 1 only).
// g: (B, K, P, Q) fp32, gx: (B, C, H, W) fp32, w: the FORWARD weight (K, C, R, S).
int po2_conv2d_dgrad(const void* g_out, const void* w, const float* scale, void* gx, int B, int C, int H,
                     int W, int K, int R, int S, int stride, int pad, int groups, int w_format, int bits,
                     int fsr, int compute, void* workspace, size_t workspace_bytes, void* stream) {
  if (!g_out || !w || !gx) return PO2_E_NULL;
  if (w_format != PO2_W_F32_PO2 && w_format != PO2_W_CODES) return PO2_E_UNSUPPORTED;
  ConvPlan p;
  if (int e = plan_dgrad(p, B, C, H, W, K, R, S, stride, pad, groups, compute)) return e;
  if (!workspace || workspace_bytes < p.workspace) return PO2_E_WORKSPACE;
  if (int a = umma_check_x(g_out, p)) return a;
  cudaStream_t st = (cudaStream_t)stream;
  if (int e = launch_pack(p, w, w_format, scale, bits, fsr, 1, workspace, st)) return e;
  return launch_conv(p, g_out, workspace, scale, gx, 1, ConvEpilogue{}, st);
}

// Static weights (PTQ / eval): build the packed tensor-core operand once, reuse it every forward.
// po2_conv2d_pack_bytes == 0 means the shape does not run on the tensor-core kernel.
size_t po2_conv2d_pack_bytes(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                             int compute) {
  return po2_conv2d_pack_bytes_dt(B, C, H, W, K, R, S, stride, pad, groups, compute, PO2_F32);
}

size_t po2_conv2d_pack_bytes_dt(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                                int compute, int dtype) {
  ConvPlan p;
  return plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute, dtype) ? 0 : round256(p.pack_bytes);
}

int po2_conv2d_pack(const void* w, const float* scale, void* packed, size_t packed_bytes, int B, int C, int H,
                    int W, int K, int R, int S, int stride, int pad, int groups, int w_format, int bits,
                    int fsr, int compute, void* stream) {
  return po2_conv2d_pack_dt(w, scale, packed, packed_bytes, B, C, H, W, K, R, S, stride, pad, groups, w_format, bits, fsr,
                            compute, PO2_F32, stream);
}

int po2_conv2d_pack_dt(const void* w, const float* scale, void* packed, size_t packed_bytes, int B, int C, int H,
                       int W, int K, int R, int S, int stride, int pad, int groups, int w_format, int bits,
                       int fsr, int compute, int dtype, void* stream) {
  if (!w || !packed) return PO2_E_NULL;
  if (w_format != PO2_W_F32_PO2 && w_format != PO2_W_CODES) return PO2_E_UNSUPPORTED;
  if (w_format == PO2_W_CODES && (!scale || bits < 2 || bits > 8)) return PO2_E_BITS;
  ConvPlan p;
  if (int e = plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute, dtype)) return e;
  if (!p.pack_bytes) return PO2_E_UNSUPPORTED;
  if (packed_bytes < p.pack_bytes) return PO2_E_WORKSPACE;
  return launch_pack(p, w, w_format, scale, bits, fsr, 0, packed, (cudaStream_t)stream);
}

int po2_conv2d_fwd_packed(const void* x, const void* packed, const float* scale, void* out, int B, int C, int H,
                          int W, int K, int R, int S, int stride, int pad, int groups, int compute, void* stream) {
  return po2_conv2d_fwd_packed_ep(x, packed, scale, out, B, C, H, W, K, R, S, stride, pad, groups, compute, nullptr, nullptr,
                                  nullptr, 0, stream);
}

int po2_conv2d_fwd_packed_ep(const void* x, const void* packed, const float* scale, void* out, int B, int C, int H,
                             int W, int K, int R, int S, int stride, int pad, int groups, int compute,
                             const float* ep_a, const float* ep_b, const void* residual, int act, void* stream) {
  return po2_conv2d_fwd_packed_ep_dt(x, packed, scale, out, B, C, H, W, K, R, S, stride, pad, groups, compute, ep_a, ep_b,
                                     residual, act, PO2_F32, stream);
}

int po2_conv2d_fwd_packed_ep_dt(const void* x, const void* packed, const float* scale, void* out, int B, int C, int H,
                                int W, int K, int R, int S, int stride, int pad, int groups, int compute,
                                const float* ep_a, const float* ep_b, const void* residual, int act, int dtype,
                                void* stream) {
  if (!x || !packed || !out) return PO2_E_NULL;
  if (int e = check_epilogue(ep_a, ep_b, act)) return e;
  if (!ep_a && (residual || act)) return PO2_E_NULL;
  const ConvEpilogue ep{ep_a, ep_b, (const float*)residual, act};
  ConvPlan p;
  if (int e = plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute, dtype)) return e;
  if (!p.pack_bytes) return PO2_E_UNSUPPORTED;
  if (int a = umma_check_x(x, p)) return a;
  return launch_conv(p, x, packed, scale, out, pdl_chain_enabled() ? 2 : 0, ep, (cudaStream_t)stream);
}

// QuantizedConv2d.forward in QAT mode as ONE call (models/quantized_conv.py:34-36): quantize the fp32
// master weight (utils/quantizers.py:21-32 / 41-52) and convolve.  When the shape runs on the
// tensor-core kernel and needs no channel padding, the quantizer kernel itself emits the packed
// bf16 operand (no separate pack launch) and the conv kernel starts behind it with programmatic
// dependent launch.  qw_out / scale_out receive the quantized weight and its scale (backward needs them).
int po2_qconv2d_fwd(const void* x, const void* w_master, void* qw_out, float* scale_out, void* out, int B,
                    int C, int H, int W, int K, int R, int S, int stride, int pad, int groups, int bits,
                    int fsr, int mode, int flavor, int compute, void* workspace, size_t workspace_bytes,
                    void* quant_workspace, void* stream) {
  if (!x || !w_master || !qw_out || !scale_out || !out) return PO2_E_NULL;
  if (!quant_workspace) return PO2_E_WORKSPACE;
  ConvPlan p;
  if (int e = plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t wn = (int64_t)K * (C / groups) * R * S;
  if (p.pack_bytes)
    if (int a = umma_check_x(x, p)) return a;                 // before the quantizer runs
  if (p.unpadded) {
    if (!workspace || workspace_bytes < p.workspace) return PO2_E_WORKSPACE;
    const PackArgs pk = pack_args(p.g, reinterpret_cast<char*>(workspace) + round256((size_t)wn * sizeof(float)));
    const int rc = fused_quantize_pack(w_master, qw_out, scale_out, wn, bits, fsr, mode, flavor, quant_workspace, pk, st);
    if (rc == 0) return launch_conv(p, x, pk.Bp, scale_out, out, 1, ConvEpilogue{}, st);
    if (rc != PO2_E_UNSUPPORTED) return rc;
  }
  if (int e = po2_quantize_fused(w_master, qw_out, nullptr, nullptr, nullptr, scale_out, wn, PO2_F32, bits, fsr,
                                 mode, flavor, quant_workspace, stream)) return e;
  return po2_conv2d_fwd(x, qw_out, scale_out, out, B, C, H, W, K, R, S, stride, pad, groups, PO2_W_F32_PO2, bits,
                        fsr, compute, workspace, workspace_bytes, stream);
}

// The first half of po2_qconv2d_fwd on its own: quantize the master weight and emit the packed
// tensor-core operand of conv2d(x of shape (B, C, H, W), Q(w)).  Lets a caller quantize all layers of a
// model ahead of the activations (on another stream), then run each conv with po2_conv2d_fwd_packed.
int po2_quantize_pack(const void* w_master, void* qw_out, float* scale_out, void* packed, size_t packed_bytes, int B,
                      int C, int H, int W, int K, int R, int S, int stride, int pad, int groups, int bits, int fsr,
                      int mode, int flavor, int compute, void* quant_workspace, void* stream) {
  if (!w_master || !qw_out || !scale_out || !packed) return PO2_E_NULL;
  if (!quant_workspace) return PO2_E_WORKSPACE;
  ConvPlan p;
  if (int e = plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute)) return e;
  if (!p.pack_bytes) return PO2_E_UNSUPPORTED;
  if (packed_bytes < p.pack_bytes) return PO2_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t wn = (int64_t)K * (C / groups) * R * S;
  if (p.unpadded) {
    const int rc = fused_quantize_pack(w_master, qw_out, scale_out, wn, bits, fsr, mode, flavor, quant_workspace,
                                       pack_args(p.g, packed), st);
    if (rc != PO2_E_UNSUPPORTED) return rc;
  }
  if (int e = po2_quantize_fused(w_master, qw_out, nullptr, nullptr, nullptr, scale_out, wn, PO2_F32, bits, fsr, mode,
                                 flavor, quant_workspace, stream)) return e;
  return po2_conv2d_pack(qw_out, scale_out, packed, packed_bytes, B, C, H, W, K, R, S, stride, pad, groups,
                         PO2_W_F32_PO2, bits, fsr, compute, stream);
}

// ---- multi-tensor quantize + pack: one launch for all QAT weights of a model --------------------------
size_t po2_multi_desc_bytes(void) { return sizeof(MultiDesc); }

int po2_multi_desc_fill(void* host_table, int index, const void* w_master, void* qw_out, float* scale_out, void* packed,
                        size_t packed_bytes, int B, int C, int H, int W, int K, int R, int S, int stride, int pad,
                        int groups, int bits, int fsr, int mode, int flavor, int compute, double* sse_out) {
  if (!host_table || index < 0 || !w_master || !qw_out || !scale_out || !packed) return PO2_E_NULL;
  if (int e = check_quant_args(bits, fsr, mode, flavor)) return e;
  ConvPlan p;
  if (int e = plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute)) return e;
  if (!p.unpadded) return PO2_E_UNSUPPORTED;             // no tensor-core operand, or one with channel padding
  if (packed_bytes < p.pack_bytes) return PO2_E_WORKSPACE;
  const int64_t wn = (int64_t)K * (C / groups) * R * S;
  if (wn % 4 || (reinterpret_cast<uintptr_t>(w_master) & 15) || (reinterpret_cast<uintptr_t>(qw_out) & 15))
    return PO2_E_UNSUPPORTED;
  const int cap = multi_fused_capacity();
  int csize = 1;
  while (csize < 8 && (int64_t)csize * cap < wn) csize <<= 1;
  if ((int64_t)csize * cap < wn) return PO2_E_UNSUPPORTED;                        // does not fit one cluster
  MultiDesc d = {};
  d.x = (const uint4*)w_master; d.y = (uint4*)qw_out; d.scale_out = scale_out; d.sse_out = sse_out; d.n = wn;
  d.bits = bits; d.fsr = fsr; d.mode = mode; d.flavor = flavor;
  d.pk = pack_args(p.g, packed);
  reinterpret_cast<MultiDesc*>(host_table)[index] = d;
  return csize;
}

int po2_quantize_pack_multi(const void* device_table, int ntensors, int cluster_size, void* stream) {
  return multi_fused_launch((const MultiDesc*)device_table, ntensors, cluster_size, (cudaStream_t)stream);
}

// ---- the data-gradient operand packed ahead of time (by the multi-tensor quantizer of the forward pass) ----
size_t po2_conv2d_dgrad_pack_bytes(int B, int C, int H, int W, int K, int R, int S, int pad, int compute) {
  ConvPlan p;
  if (plan_dgrad(p, B, C, H, W, K, R, S, 1, pad, 1, compute) || !p.unpadded) return 0;   // the fused emitter writes no padding
  return round256(p.pack_bytes);
}

// amend entry `index` of a MultiDesc table (after po2_multi_desc_fill): also emit the data-gradient operand
int po2_multi_desc_fill_dgrad(void* host_table, int index, void* packed_dgrad, size_t packed_bytes, int B, int C, int H,
                              int W, int K, int R, int S, int stride, int pad, int groups, int compute) {
  if (!host_table || index < 0 || !packed_dgrad) return PO2_E_NULL;
  ConvPlan p;
  if (plan_dgrad(p, B, C, H, W, K, R, S, stride, pad, groups, compute) || !p.unpadded) return PO2_E_UNSUPPORTED;
  if (packed_bytes < p.pack_bytes) return PO2_E_WORKSPACE;
  MultiDesc& d = reinterpret_cast<MultiDesc*>(host_table)[index];
  if (d.pk.G != p.g.G || d.pk.taps != p.g.ntaps) return PO2_E_SHAPE;
  add_dgrad_operand(d.pk, p.g, packed_dgrad);
  return 0;
}

// ---- lin / lin+ weights on the tensor-core kernels ----------------------------------------------------------------
// A lin weight is n * 2^k per input channel, |n| <= 2^(bits-1) - 1: exact as a bf16 operand for bits <= 9 and as a
// tf32 operand for bits <= 12, so the packed operand holds y itself and the conv runs with scale = 1.0.  The
// quantizer kernel writes it (and the stride-1 data-gradient operand) from the CTA that owns the input channel.
// Fills pk for conv2d(x of shape (B, C, H, W), w (K, C/groups, R, S)); PO2_E_UNSUPPORTED when the geometry has no
// tensor-core operand, needs channel padding (the per-channel emitter writes no padding) or bits is not exact.
static int lin_pack_args(PackArgs& pk, ConvPlan& p, void* packed, size_t packed_bytes, void* packed_dgrad,
                         size_t dgrad_bytes, int B, int C, int H, int W, int K, int R, int S, int stride, int pad,
                         int groups, int bits, int num_iters, int compute) {
  if (int e = plan_fwd(p, B, C, H, W, K, R, S, stride, pad, groups, compute)) return e;
  if (!p.pack_bytes) return PO2_E_UNSUPPORTED;
  if (num_iters < 1 || bits > (p.g.tf32 ? 12 : 9)) return PO2_E_UNSUPPORTED;    // step not a power of two / not exact
  if (packed_bytes < p.pack_bytes) return PO2_E_WORKSPACE;
  pk = pack_args(p.g, packed);
  if (packed_dgrad) {
    ConvPlan d;
    if (plan_dgrad(d, B, C, H, W, K, R, S, stride, pad, groups, compute) || !d.unpadded || d.g.G != p.g.G ||
        d.g.ntaps != p.g.ntaps) return PO2_E_UNSUPPORTED;
    if (dgrad_bytes < d.pack_bytes) return PO2_E_WORKSPACE;
    add_dgrad_operand(pk, d.g, packed_dgrad);
  }
  return 0;
}

// y = lin(w) and the packed operand(s) of conv2d(x of shape (B, C, H, W), y): one launch, or two (quantizer + pack)
// when the operand needs channel padding.
int po2_lin_quantize_pack(const void* w, void* y_out, void* packed, size_t packed_bytes, void* packed_dgrad,
                          size_t packed_dgrad_bytes, int B, int C, int H, int W, int K, int R, int S, int stride, int pad,
                          int groups, int bits, int num_iters, int plus, int flavor, int compute, void* stream) {
  if (!w || !y_out || !packed) return PO2_E_NULL;
  const int Cg = groups > 0 ? C / groups : 0;
  if (int e = lin_check_args(K, Cg, R * S, bits, num_iters, flavor)) return e;
  PackArgs pk;
  ConvPlan p;
  if (int e = lin_pack_args(pk, p, packed, packed_bytes, packed_dgrad, packed_dgrad_bytes, B, C, H, W, K, R, S, stride,
                            pad, groups, bits, num_iters, compute)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  if (p.unpadded) return lin_launch((const float*)w, (float*)y_out, K, C, R * S, bits, num_iters, plus, flavor, pk, st);
  if (packed_dgrad) return PO2_E_UNSUPPORTED;
  if (int e = lin_launch((const float*)w, (float*)y_out, K, Cg, R * S, bits, num_iters, plus, flavor, PackArgs{}, st))
    return e;
  return po2_conv2d_pack(y_out, nullptr, packed, packed_bytes, B, C, H, W, K, R, S, stride, pad, groups, PO2_W_F32_PO2,
                         bits, 1, compute, stream);
}

// entry `index` of a LinDesc table (host memory, filled in index order 0, 1, ...: the entry starts its CTAs behind
// those of entry index - 1).  Returns this tensor's CTA count (C) or a PO2_E_* code.
int po2_lin_multi_desc_fill(void* host_table, int index, const void* w, void* y_out, void* packed, size_t packed_bytes,
                            void* packed_dgrad, size_t packed_dgrad_bytes, int B, int C, int H, int W, int K, int R,
                            int S, int stride, int pad, int groups, int bits, int num_iters, int plus, int flavor,
                            int compute) {
  if (!host_table || index < 0 || !w || !y_out || !packed) return PO2_E_NULL;
  const int Cg = groups > 0 ? C / groups : 0;
  if (int e = lin_check_args(K, Cg, R * S, bits, num_iters, flavor)) return e;
  PackArgs pk;
  ConvPlan p;
  if (int e = lin_pack_args(pk, p, packed, packed_bytes, packed_dgrad, packed_dgrad_bytes, B, C, H, W, K, R, S, stride,
                            pad, groups, bits, num_iters, compute)) return e;
  if (!p.unpadded) return PO2_E_UNSUPPORTED;
  LinDesc* t = reinterpret_cast<LinDesc*>(host_table);
  LinDesc d = {};
  d.w = (const float*)w; d.y = (float*)y_out;
  d.K = K; d.C = C; d.RS = R * S; d.bits = bits; d.iters = num_iters; d.plus = plus; d.flavor = flavor;
  d.cta0 = index == 0 ? 0 : t[index - 1].cta0 + t[index - 1].C;
  d.pk = pk;
  t[index] = d;
  return C;
}

// gx = dL/dx from g = dL/dout and the pre-packed data-gradient operand: one launch
int po2_conv2d_dgrad_packed(const void* g_out, const void* packed, const float* scale, void* gx, int B, int C, int H,
                            int W, int K, int R, int S, int pad, int compute, void* stream) {
  if (!g_out || !packed || !gx) return PO2_E_NULL;
  ConvPlan p;
  if (plan_dgrad(p, B, C, H, W, K, R, S, 1, pad, 1, compute)) return PO2_E_UNSUPPORTED;
  if (int a = umma_check_x(g_out, p)) return a;
  return launch_conv(p, g_out, packed, scale, gx, pdl_chain_enabled() ? 2 : 0, ConvEpilogue{}, (cudaStream_t)stream);
}

size_t po2_conv2d_dgrad_workspace(int B, int C, int H, int W, int K, int R, int S, int pad, int compute) {
  ConvPlan p;
  return plan_dgrad(p, B, C, H, W, K, R, S, 1, pad, 1, compute) ? 0 : p.workspace;
}


// Weight gradient of the same conv (SURVEY.md section 8f "next" #2, second half): gw = dL/dW given
// g = dL/dout and the forward input x -- through the straight-through estimator this is the gradient
// of the fp32 master weight.  Which kernel runs a shape, and its plan:
struct WgradPlan {
  int kind;              // po2_conv2d_wgrad_kernel_kind: 0 not taken, 1 K5, 2 K5T, 3 pointwise GEMM
  WgTmaPlan wp;          // kind 2
  ConvGeom g;            // kind 1: the forward geometry through plan_umma(g, false)
  WgGeom wg;             // kind 1
  size_t partial_bytes;  // the workspace: per-CTA partial sums
};

// K5 / K5T take the dense stride-1 shapes (3x3 pad 1, 1x1 pad 0) with K <= 128.  compute == 2 (tf32 operands): K5T
// where the shape allows, else the bf16-operand K5 (the weight gradient is a leaf of the backward pass: its rounding
// does not propagate into other gradients).  The small 1x1 layers neither takes go to the pointwise GEMM.
static void plan_wgrad_conv(WgradPlan& p, int B, int C, int H, int W, int K, int R, int S, int stride, int pad,
                            int groups, int compute) {
  static const bool k5t_off = [] { const char* e = getenv("PO2_WGRAD_TMA"); return e && e[0] == '0'; }();
  p = WgradPlan{};
  const bool dense1 = stride == 1 && groups == 1;
  if (compute == 2 && dense1 && tma_enabled() && !k5t_off && plan_wgrad_tma(p.wp, B, C, H, W, K, R, S, pad)) {
    p.kind = 2;
    p.partial_bytes = wgrad_tma_partial_bytes(p.wp);
  } else if ((compute == 0 || compute == 2) && dense1 && tc_window(R, S, pad) &&
             fill_geom(p.g, B, C, H, W, K, R, S, 1, pad, 1) && index_fits(p.g) && plan_umma(p.g, false) &&
             plan_wgrad(p.g, p.wg)) {
    p.kind = 1;
    p.partial_bytes = wgrad_partial_bytes(p.g, p.wg);
  } else if (pw_wgrad_takes(B, C, H, W, K, R, S, stride, pad, groups, compute)) {
    p.kind = 3;
    p.partial_bytes = pw_wgrad_partial_bytes(B, C, H, W, K);
  }
}

size_t po2_conv2d_wgrad_workspace(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                                  int compute) {
  WgradPlan p;
  plan_wgrad_conv(p, B, C, H, W, K, R, S, stride, pad, groups, compute);
  return round256(p.partial_bytes);
}

// 0: not taken (aten), 1: bf16-operand tcgen05 kernel (K5), 2: TMA-fed tf32 kernel (K5T), 3: fp32 CUDA-core GEMM of
// the small 1x1 layers that neither K5T nor K5 takes (csrc/po2_conv_bwd.cu, conv_wgrad_pw_kernel)
int po2_conv2d_wgrad_kernel_kind(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                                 int compute) {
  WgradPlan p;
  plan_wgrad_conv(p, B, C, H, W, K, R, S, stride, pad, groups, compute);
  return p.kind;
}

int po2_conv2d_wgrad(const void* g_out, const void* x, void* gw, int B, int C, int H, int W, int K, int R, int S,
                     int stride, int pad, int groups, int compute, void* workspace, size_t workspace_bytes,
                     void* stream) {
  return po2_conv2d_wgrad_z(g_out, x, gw, B, C, H, W, K, R, S, stride, pad, groups, compute, workspace, workspace_bytes,
                            nullptr, stream);
}

// the same with `zeroed_tickets`: 8 bytes of device memory that are zero before the first call (the kernels leave
// them zero) and are not shared by calls that may run concurrently.  With them the TMA-fed kernel reduces its
// partial sums itself (one launch instead of two); NULL: two launches.
int po2_conv2d_wgrad_z(const void* g_out, const void* x, void* gw, int B, int C, int H, int W, int K, int R, int S,
                       int stride, int pad, int groups, int compute, void* workspace, size_t workspace_bytes,
                       void* zeroed_tickets, void* stream) {
  if (!g_out || !x || !gw) return PO2_E_NULL;
  WgradPlan p;
  plan_wgrad_conv(p, B, C, H, W, K, R, S, stride, pad, groups, compute);
  if (p.kind == 0) return PO2_E_UNSUPPORTED;
  if (!workspace || workspace_bytes < p.partial_bytes) return PO2_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  if (p.kind == 2) {
    // measured (profiles/README.md, r02): the in-kernel reduction is SLOWER than the second launch -- 21.5 / 22.3 /
    // 22.5 us against 20.0 / 15.4 / 13.2 us per ResNet-56 layer class, 3.33 against 3.00 ms per step: the grid
    // barrier costs more than the launch it saves, and 148 CTAs have far less load parallelism for the partials
    // than the 1152-CTA reduce kernel (the cooperative launch itself is free: the fused BatchNorm kernels run the
    // same with a plain launch).  Opt-in only (PO2_WGRAD_FUSED_REDUCE=1).
    static const bool fuse = [] { const char* e = getenv("PO2_WGRAD_FUSED_REDUCE"); return e && e[0] == '1'; }();
    if (!aligned16(g_out) || !aligned16(x)) return PO2_E_ALIGN;          // the bases of both tensor maps
    return launch_wgrad_tma(g_out, x, gw, workspace, p.wp, st, fuse ? (unsigned int*)zeroed_tickets : nullptr);
  }
  if (p.kind == 3)
    return launch_pw_wgrad((const float*)g_out, (const float*)x, (float*)gw, workspace, B, C, H * W, K, st);
  if (p.g.vec4 && (!aligned16(g_out) || !aligned16(x))) return PO2_E_ALIGN;   // produce_planes_bf16: 128-bit loads
  static PerDeviceOnce wgrad_once;
  if (cudaError_t e0 = wgrad_once.run([]() -> cudaError_t {
        return cudaFuncSetAttribute(conv_wgrad_umma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)K3_SMEM_BUDGET + 1024);
      })) return (int)e0;
  const size_t smem = (size_t)p.wg.nst * p.wg.stage_bytes + WG_A_SPAN + 512;
  conv_wgrad_umma_kernel<<<dim3(p.wg.m_ctas, p.wg.tap_splits), K3_THREADS, smem, st>>>((const float*)x, (const float*)g_out,
                                                                                       (float*)workspace, p.g, p.wg);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  return launch_wgrad_reduce((const float*)workspace, (float*)gw, p.wg.m_ctas, K, C, p.wg.ntaps, st);
}

}  // extern "C"
