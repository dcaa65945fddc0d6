// Backward of the quantized conv for the layer kinds the tensor-core kernels do not take directly
// (autograd of models/quantized_conv.py:36 for models/resnet.py's stride-2 layers and
// models/mobilenet.py:64-74,106-116's depthwise layers):
//
//   * stride 2, dense: both gradients of conv(x, W, stride 2) equal the gradients of the STRIDE-1 conv whose
//     output gradient is the zero-inserted one, g_up[2p][2q] = g[p][q]:
//         gx = conv_transpose(g, W, 2) = dgrad_stride1(g_up, W),   gw = wgrad_stride1(g_up, x)
//     so one small kernel (dilate2_kernel; dilate2_into_kernel for odd sizes) puts these layers on the stride-1
//     kernels (K3T / K5T where they take the shape).  For 3x3 pad 1 and 1x1 pad 0 this holds for any H x W: output
//     row p reads input rows 2p - 1 .. 2p + 1, as row 2p of the stride-1 conv does, and 2(P - 1) <= H - 1.
//   * depthwise 3x3 pad 1 (groups == C == K): data gradient = the depthwise forward kernel's arithmetic with
//     the filter rotated by 180 degrees (on g, or on g_up for stride 2); weight gradient = nine per-channel
//     inner products over the batch, a two-stage fixed-order reduction (deterministic).
#include <stdlib.h>

#include "po2_common.cuh"

namespace po2 {

// g (planes, P, Q) -> g_up (planes, 2P, 2Q): g_up[2p][2q] = g[p][q], zero elsewhere.  One thread = 4 output
// columns of an even row pair: reads two inputs, writes two 128-bit vectors.
__global__ void __launch_bounds__(256) dilate2_kernel(const float* __restrict__ g, float* __restrict__ up, int Q2,
                                                      int rows, int Q) {
  // rows = planes * P input rows; Q2 = Q / 2 (pairs of input columns per row)
  const int total = rows * Q2;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int row = i / Q2, c2 = i - row * Q2;
    const float2 v = __ldg(reinterpret_cast<const float2*>(g + (size_t)row * Q) + c2);
    float4* o = reinterpret_cast<float4*>(up + (size_t)row * 4 * Q) + c2;        // output row 2*row has 2Q floats
    o[0] = make_float4(v.x, 0.f, v.y, 0.f);
    o[Q2] = make_float4(0.f, 0.f, 0.f, 0.f);                                      // output row 2*row + 1
  }
}

// The same zero-insertion for any H x W with P = (H - 1) / 2 + 1, Q = (W - 1) / 2 + 1 (odd H or W, odd Q), at any
// 4-byte alignment: g (planes, P, Q) -> g_up (planes, H, W).  One thread = one output element, scalar accesses.
__global__ void __launch_bounds__(256) dilate2_into_kernel(const float* __restrict__ g, float* __restrict__ up, int P,
                                                           int Q, int H, int W, int total) {
  // total < 2^31 may lie within one grid stride of 2^31: a 32-bit i would wrap on its last step
  for (int64_t i64 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i64 < total; i64 += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)i64;
    const int row = i / W, w = i - row * W;                                       // row = plane * H + h
    const int plane = row / H, h = row - plane * H;
    up[i] = ((h | w) & 1) ? 0.f : __ldg(g + ((size_t)plane * P + (h >> 1)) * Q + (w >> 1));
  }
}

// depthwise 3x3 pad 1 stride 1 data gradient on g (already zero-inserted for stride 2):
//   gx[h][w] = sum_{r,s} g[h + 1 - r][w + 1 - s] * w[c][r][s]
__global__ void __launch_bounds__(256) dw_dgrad_kernel(const float* __restrict__ g, const float* __restrict__ w,
                                                       float* __restrict__ gx, int C, int H, int W, int total) {
  for (int64_t i64 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i64 < total; i64 += (int64_t)gridDim.x * blockDim.x) {
    const int i = (int)i64;                                     // 64-bit step: total may lie within a stride of 2^31
    const int x = i % W;
    const int t = i / W;
    const int y = t % H;
    const int plane = t / H;
    const int c = plane % C;
    const float* pg = g + (size_t)plane * H * W;
    const float* pw = w + c * 9;
    float acc = 0.f;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const int gy = y + 1 - r;
      if (gy < 0 || gy >= H) continue;
#pragma unroll
      for (int s = 0; s < 3; ++s) {
        const int gxx = x + 1 - s;
        if (gxx < 0 || gxx >= W) continue;
        acc = fmaf(__ldg(pg + gy * W + gxx), __ldg(pw + r * 3 + s), acc);
      }
    }
    gx[i] = acc;
  }
}

// depthwise 3x3 pad 1 weight gradient (stride-1 form; g zero-inserted for stride 2):
//   gw[c][r][s] = sum_{n,h,w} g[n][c][h][w] * x[n][c][h + r - 1][w + s - 1]
// CTA (split, c) sums the images n = split, split + S, ...; partials [c][split][9]; the last CTA of a channel
// (ticket) adds them in split order.
constexpr int DWG_THREADS = 256;
__global__ void __launch_bounds__(DWG_THREADS) dw_wgrad_kernel(const float* __restrict__ g, const float* __restrict__ x,
                                                               float* __restrict__ gw, float* __restrict__ partial,
                                                               unsigned int* __restrict__ ticket, int B, int C, int H,
                                                               int W, int S) {
  __shared__ float sm[DWG_THREADS / 32][9];
  __shared__ int last;
  const int split = blockIdx.x, c = blockIdx.y, HW = H * W;
  float acc[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) acc[k] = 0.f;
  // 64-bit steps: B and HW may each lie within one step of 2^31 (B * C * H * W < 2^31 is all the host checks)
  for (int64_t n = split; n < B; n += S) {
    const float* pg = g + ((size_t)n * C + c) * HW;
    const float* px = x + ((size_t)n * C + c) * HW;
    for (int64_t i64 = threadIdx.x; i64 < HW; i64 += DWG_THREADS) {
      const int i = (int)i64;
      const float gv = __ldg(pg + i);
      if (gv == 0.f) continue;                                  // zero-inserted gradients: 3 of 4 positions
      const int y = i / W, xx = i - y * W;
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int iy = y + r - 1;
        if (iy < 0 || iy >= H) continue;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const int ix = xx + s - 1;
          if (ix < 0 || ix >= W) continue;
          acc[r * 3 + s] = fmaf(gv, __ldg(px + iy * W + ix), acc[r * 3 + s]);
        }
      }
    }
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    float v = acc[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if (lane == 0) sm[warp][k] = v;
  }
  __syncthreads();
  if (threadIdx.x < 9) {
    float v = 0.f;
#pragma unroll
    for (int q = 0; q < DWG_THREADS / 32; ++q) v += sm[q][threadIdx.x];
    partial[((size_t)c * S + split) * 9 + threadIdx.x] = v;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ticket + c, 1u);
    last = (t == (unsigned int)(S - 1));
    if (last) ticket[c] = 0u;                                   // self-resetting
  }
  __syncthreads();
  if (last && threadIdx.x < 9) {
    __threadfence();
    float v = 0.f;
    for (int q = 0; q < S; ++q) v += __ldcg(partial + ((size_t)c * S + q) * 9 + threadIdx.x);
    gw[c * 9 + threadIdx.x] = v;
  }
}

// ------------------------------------------------------------------------------------------------
// Weight gradient of a plain 3x3 pad-1 stride-1 conv with very few input channels -- the full-precision stem of the
// reference's models (models/resnet.py:99-102: nn.Conv2d(3, 16, 3, 1, 1)); the input needs no gradient, so this is
// the layer's whole backward.  cuDNN's wgrad takes 40 us on the 128 x 3 x 32 x 32 batch (the last cuDNN kernel of the
// ResNet-56 step besides the stem's forward).  CUDA cores, exact fp32 FMA:
//   gw[k][c][r][s] = sum_{n,h,w} g[n][k][h][w] * x[n][c][h + r - 1][w + s - 1]
// One CTA per image (grid-stride): g[n] (K rows, padded by one float against bank conflicts) and the zero-haloed
// x[n] are staged in shared memory; thread (row group, k, c) walks its rows with a sliding 3x3 window -- one g load
// and three x loads per nine FMAs --, the row groups are added through shared memory in a fixed order, and the CTA's
// partial [tap][k][c] goes to conv_wgrad_reduce_kernel (fixed order over CTAs: deterministic).
// ------------------------------------------------------------------------------------------------
constexpr int SW_THREADS = 256;
__global__ void __launch_bounds__(SW_THREADS) stem_wgrad_kernel(const float* __restrict__ g, const float* __restrict__ x,
                                                                float* __restrict__ partial, int B, int C, int H, int W,
                                                                int K) {
  extern __shared__ float sw_smem[];
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the reduce kernel waits for this grid's completion
  const int HW = H * W, GS = HW + 1, XW = W + 2, XS = (H + 2) * XW;
  float* sg = sw_smem;                          // [K][HW + 1]
  float* sx = sg + K * GS;                      // [C][H + 2][W + 2]
  float* red = sx + C * XS;                     // [RG][K * C][9]
  const int KC = K * C, RG = SW_THREADS / KC;   // row groups
  const int tid = threadIdx.x, pair = tid % KC, rg = tid / KC;
  const bool active = rg < RG;
  const int k = pair / C, c = pair - k * C;
  float tot[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) tot[i] = 0.f;
  for (int i = tid; i < C * XS; i += SW_THREADS) sx[i] = 0.f;       // the halo stays zero for every image
  for (int n = blockIdx.x; n < B; n += gridDim.x) {
    __syncthreads();
    const float* pg = g + (size_t)n * K * HW;
    const float* px = x + (size_t)n * C * HW;
    for (int i = tid; i < K * HW; i += SW_THREADS) {
      const int kk = i / HW;
      sg[kk * GS + (i - kk * HW)] = __ldg(pg + i);
    }
    for (int i = tid; i < C * HW; i += SW_THREADS) {
      const int cc = i / HW, p = i - cc * HW, h = p / W, w = p - h * W;
      sx[cc * XS + (h + 1) * XW + (w + 1)] = __ldg(px + i);
    }
    __syncthreads();
    float acc[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) acc[i] = 0.f;
    if (active) {
      const float* gk = sg + k * GS;
      const float* xc = sx + c * XS;
      for (int h = rg; h < H; h += RG) {
        const float* x0 = xc + h * XW;          // rows h-1, h, h+1 of the image = rows h, h+1, h+2 of the padded plane
        float a0 = x0[0], a1 = x0[1], b0 = x0[XW], b1 = x0[XW + 1], c0 = x0[2 * XW], c1 = x0[2 * XW + 1];
        for (int w = 0; w < W; ++w) {
          const float gv = gk[h * W + w];
          const float a2 = x0[w + 2], b2 = x0[XW + w + 2], c2 = x0[2 * XW + w + 2];
          acc[0] = fmaf(gv, a0, acc[0]); acc[1] = fmaf(gv, a1, acc[1]); acc[2] = fmaf(gv, a2, acc[2]);
          acc[3] = fmaf(gv, b0, acc[3]); acc[4] = fmaf(gv, b1, acc[4]); acc[5] = fmaf(gv, b2, acc[5]);
          acc[6] = fmaf(gv, c0, acc[6]); acc[7] = fmaf(gv, c1, acc[7]); acc[8] = fmaf(gv, c2, acc[8]);
          a0 = a1; a1 = a2; b0 = b1; b1 = b2; c0 = c1; c1 = c2;
        }
      }
#pragma unroll
      for (int i = 0; i < 9; ++i) red[(rg * KC + pair) * 9 + i] = acc[i];
    }
    __syncthreads();
    if (tid < KC) {
#pragma unroll
      for (int i = 0; i < 9; ++i) {
        float v = 0.f;
        for (int q = 0; q < RG; ++q) v += red[(q * KC + tid) * 9 + i];
        tot[i] += v;
      }
    }
  }
  if (tid < KC) {
#pragma unroll
    for (int i = 0; i < 9; ++i) partial[((size_t)blockIdx.x * 9 + i) * KC + k * C + c] = tot[i];   // [cta][tap][k][c]
  }
}
static size_t stem_wgrad_smem(int C, int H, int W, int K) {
  const int KC = K * C, RG = SW_THREADS / (KC > 0 ? KC : 1);
  return ((size_t)K * (H * W + 1) + (size_t)C * (H + 2) * (W + 2) + (size_t)RG * KC * 9) * sizeof(float);
}
static bool stem_wgrad_takes(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups) {
  if (R != 3 || S != 3 || stride != 1 || pad != 1 || groups != 1 || B < 1) return false;
  if (C < 1 || C > 4 || K < 1 || K * C > SW_THREADS || H < 1 || W < 1) return false;
  // B < 2^30 keeps the image loop's 32-bit n += gridDim.x (<= 148) from wrapping; the other loops stay in shared memory
  return stem_wgrad_smem(C, H, W, K) <= 200 * 1024 && (int64_t)B * K * H * W < (1ll << 31) && B < (1 << 30);
}
static int stem_wgrad_ctas(int B) {
  const int sms = device_sm_count();
  return B < sms ? B : sms;
}

// blocks of 256 threads for a grid-stride loop over total < 2^31 elements, at most 16 per SM (64-bit: total + 255
// must not wrap)
static int grid_blocks(int total) {
  const int64_t need = ((int64_t)total + 255) / 256, cap = (int64_t)device_sm_count() * 16;
  return (int)(need < cap ? need : cap);
}

constexpr int DWG_MAX_C = 4096;
constexpr int DWG_MAX_SPLIT = 32;

}  // namespace po2

using namespace po2;

extern "C" {

size_t po2_conv2d_stem_wgrad_workspace(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups) {
  if (!stem_wgrad_takes(B, C, H, W, K, R, S, stride, pad, groups)) return 0;
  return (size_t)stem_wgrad_ctas(B) * 9 * K * C * sizeof(float);
}

int po2_conv2d_stem_wgrad(const void* g, const void* x, void* gw, int B, int C, int H, int W, int K, int R, int S, int stride,
                          int pad, int groups, void* workspace, size_t workspace_bytes, void* stream) {
  if (!g || !x || !gw || !workspace) return PO2_E_NULL;
  if (!stem_wgrad_takes(B, C, H, W, K, R, S, stride, pad, groups)) return PO2_E_UNSUPPORTED;
  const int ctas = stem_wgrad_ctas(B);
  if (workspace_bytes < (size_t)ctas * 9 * K * C * sizeof(float)) return PO2_E_WORKSPACE;
  const size_t smem = stem_wgrad_smem(C, H, W, K);
  static PerDeviceOnce once;
  if (cudaError_t e0 = once.run([]() -> cudaError_t {
        return cudaFuncSetAttribute(stem_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      })) return (int)e0;
  cudaStream_t st = (cudaStream_t)stream;
  stem_wgrad_kernel<<<ctas, SW_THREADS, smem, st>>>((const float*)g, (const float*)x, (float*)workspace, B, C, H, W, K);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  return launch_wgrad_reduce((const float*)workspace, (float*)gw, ctas, K, C, 9, st);
}

int po2_dilate2(const void* g, void* g_up, int planes, int P, int Q, void* stream) {
  if (!g || !g_up) return PO2_E_NULL;
  if (planes <= 0 || P <= 0 || Q <= 0) return PO2_E_SHAPE;
  if (Q % 2 || (reinterpret_cast<uintptr_t>(g) & 7) || (reinterpret_cast<uintptr_t>(g_up) & 15)) return PO2_E_UNSUPPORTED;
  if ((int64_t)planes * P * Q * 4 >= (1ll << 31)) return PO2_E_SIZE;
  const int rows = planes * P, total = rows * (Q / 2);          // < 2^28: dilate2_kernel's 32-bit i never nears 2^31
  const int blocks = grid_blocks(total);
  dilate2_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)g, (float*)g_up, Q / 2, rows, Q);
  return (int)cudaGetLastError();
}

int po2_dilate2_into(const void* g, void* g_up, int planes, int P, int Q, int H, int W, void* stream) {
  if (!g || !g_up) return PO2_E_NULL;
  if (planes <= 0 || H <= 0 || W <= 0 || P != (H - 1) / 2 + 1 || Q != (W - 1) / 2 + 1) return PO2_E_SHAPE;
  if ((int64_t)planes * H * W >= (1ll << 31)) return PO2_E_SIZE;
  const int total = planes * H * W;
  const int blocks = grid_blocks(total);
  dilate2_into_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)g, (float*)g_up, P, Q, H, W, total);
  return (int)cudaGetLastError();
}

// g: (B, C, H, W) -- the output gradient at the INPUT resolution (stride 2: zero-inserted with po2_dilate2 / _into)
int po2_conv2d_depthwise_dgrad(const void* g, const void* w, void* gx, int B, int C, int H, int W, void* stream) {
  if (!g || !w || !gx) return PO2_E_NULL;
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return PO2_E_SHAPE;
  if ((int64_t)B * C * H * W >= (1ll << 31)) return PO2_E_SIZE;
  const int total = B * C * H * W;
  const int blocks = grid_blocks(total);
  dw_dgrad_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>((const float*)g, (const float*)w, (float*)gx, C, H, W, total);
  return (int)cudaGetLastError();
}

size_t po2_conv2d_depthwise_wgrad_workspace(int C) {
  return (size_t)DWG_MAX_C * sizeof(unsigned int) + (size_t)C * DWG_MAX_SPLIT * 9 * sizeof(float);
}

// workspace: po2_conv2d_depthwise_wgrad_workspace(C) bytes whose first DWG_MAX_C * 4 bytes (the tickets) are zero
// before the first call (the kernel leaves them zero)
int po2_conv2d_depthwise_wgrad(const void* g, const void* x, void* gw, int B, int C, int H, int W, void* workspace,
                               size_t workspace_bytes, void* stream) {
  if (!g || !x || !gw || !workspace) return PO2_E_NULL;
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return PO2_E_SHAPE;
  if (C > DWG_MAX_C) return PO2_E_UNSUPPORTED;
  if (workspace_bytes < po2_conv2d_depthwise_wgrad_workspace(C)) return PO2_E_WORKSPACE;
  if ((int64_t)B * C * H * W >= (1ll << 31)) return PO2_E_SIZE;
  int S = (4 * device_sm_count() + C - 1) / C;
  if (S > B) S = B;
  if (S > DWG_MAX_SPLIT) S = DWG_MAX_SPLIT;
  if (S < 1) S = 1;
  unsigned int* ticket = reinterpret_cast<unsigned int*>(workspace);
  float* partial = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(workspace) + (size_t)DWG_MAX_C * sizeof(unsigned int));
  dw_wgrad_kernel<<<dim3(S, C), DWG_THREADS, 0, (cudaStream_t)stream>>>((const float*)g, (const float*)x, (float*)gw, partial,
                                                                         ticket, B, C, H, W, S);
  return (int)cudaGetLastError();
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Pointwise (1x1, stride 1) convs on tiny feature maps -- MobileNetV2's 4x4 / 2x2 / 1x1 stages
// (models/mobilenet.py:106-116: 576->160, 160->960, 960->160, 960->320 at 1x1 ...): out[m][k] = sum_c x[m][c] w[k][c]
// with m = (image, pixel), a GEMM with M = B*HW <= a few thousand rows and up to 960 channels on either side.
// The tcgen05 kernels have nothing to pipeline there (one 128-pixel tile, all the time in weight traffic and
// fixed costs: 41 us for 960->320 against cuDNN's 6).  This is a plain fp32 CUDA-core GEMM (exact fp32 FMA,
// i.e. the precision of the fp32-accumulate mode): 32 x 64 output tiles, the channel dimension split over
// a thread-block CLUSTER of up to 8 CTAs whose partial tiles are added through distributed shared memory
// in rank order (deterministic, no global scratch).
// ------------------------------------------------------------------------------------------------
namespace po2 {

constexpr int PW_TM = 32, PW_TN = 64, PW_TK = 16, PW_THREADS = 128;

struct PwGeom {
  int M, C, K, HW, KS;      // KS: cluster size along the channel split
  FastDiv div_hw;
};

__device__ __forceinline__ uint32_t pw_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void pw_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float pw_ld_remote(const float* local, uint32_t rank) {
  uint32_t a = (uint32_t)__cvta_generic_to_shared(local), ra;
  float v;
  asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(rank));
  asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(ra));
  return v;
}

// XT: the activation storage (float, or __nv_bfloat16 for a bf16 conv; the arithmetic is fp32 either way)
template <typename XT>
__global__ void __launch_bounds__(PW_THREADS) conv_pw_small_kernel(const XT* __restrict__ x, const float* __restrict__ w,
                                                                   XT* __restrict__ out, PwGeom g, ConvEpilogue ep) {
  __shared__ __align__(16) float As[PW_TK][PW_TM + 4];
  __shared__ __align__(16) float Bs[PW_TK][PW_TN + 4];
  __shared__ float red[PW_TM][PW_TN + 1];                  // this CTA's partial tile, read by cluster rank 0
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int m0 = blockIdx.x * PW_TM, k0 = blockIdx.y * PW_TN;
  const int rank = g.KS > 1 ? (int)pw_cluster_rank() : 0;
  const int M = g.M, C = g.C, K = g.K, HW = g.HW;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  // loader roles: A element (c = tid / 8, m = (tid % 8) * 4 .. +3); B rows k = tid / 2, channels (tid % 2) * 8 .. +7
  const int ac = tid >> 3, am = (tid & 7) * 4;
  const int bk = tid >> 1, bc = (tid & 1) * 8;
  const bool cvec = (C & 3) == 0;
  float av[4], bv[8];
  auto load_chunk = [&](int c0) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int m = m0 + am + e, c = c0 + ac;
      float v = 0.f;
      if (m < M && c < C) {
        const int n = fdiv(m, g.div_hw);
        v = act_ld(x + ((size_t)n * C + c) * HW + (m - n * HW));
      }
      av[e] = v;
    }
    const int k = k0 + bk, cb = c0 + bc;
    if (cvec && k < K && cb + 8 <= C) {
      const float4 lo = __ldg(reinterpret_cast<const float4*>(w + (size_t)k * C + cb));
      const float4 hi = __ldg(reinterpret_cast<const float4*>(w + (size_t)k * C + cb) + 1);
      bv[0] = lo.x; bv[1] = lo.y; bv[2] = lo.z; bv[3] = lo.w; bv[4] = hi.x; bv[5] = hi.y; bv[6] = hi.z; bv[7] = hi.w;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) bv[e] = (k < K && cb + e < C) ? __ldg(w + (size_t)k * C + cb + e) : 0.f;
    }
  };
  const int cstep = g.KS * PW_TK;
  int c0 = rank * PW_TK;
  if (c0 < C) load_chunk(c0);
  for (; c0 < C; c0 += cstep) {
    __syncthreads();                                        // the previous chunk has been consumed
    *reinterpret_cast<float4*>(&As[ac][am]) = make_float4(av[0], av[1], av[2], av[3]);
#pragma unroll
    for (int e = 0; e < 8; ++e) Bs[bc + e][bk] = bv[e];
    __syncthreads();
    if (c0 + cstep < C) load_chunk(c0 + cstep);             // the next chunk's loads fly during this chunk's FMAs
#pragma unroll
    for (int c = 0; c < PW_TK; ++c) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[c][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[c][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
  }
  if (g.KS > 1) {
    // Partial tiles of the cluster: every rank publishes its tile in its own shared memory; rank r then owns the
    // tile rows r, r + KS, ... and adds the KS partials of each of its outputs in rank order through distributed
    // shared memory (deterministic; the reduction is spread over the whole cluster instead of queued on one CTA).
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) red[ty * 4 + i][tx * 4 + j] = acc[i][j];
    pw_cluster_sync();
    for (int row = rank; row < PW_TM; row += g.KS) {
      const int m = m0 + row;
      if (m >= M) break;
      const int n = fdiv(m, g.div_hw), hw = m - n * HW;
      if (tid < PW_TN) {
        const int k = k0 + tid;
        float t[8];
#pragma unroll
        for (int r = 0; r < 8; ++r) t[r] = r < g.KS ? pw_ld_remote(&red[row][tid], (uint32_t)r) : 0.f;
        float v = t[0];
#pragma unroll
        for (int r = 1; r < 8; ++r) v += t[r];
        if (k < K) {
          const size_t o = ((size_t)n * K + k) * HW + hw;
          act_st(out, o, ep.a ? conv_epilogue<XT>(v, ep, k, o) : v);
        }
      }
    }
    pw_cluster_sync();                                      // nobody leaves while its shared memory is still being read
    return;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
    const int n = fdiv(m, g.div_hw), hw = m - n * HW;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k >= K) continue;
      const size_t o = ((size_t)n * K + k) * HW + hw;
      act_st(out, o, ep.a ? conv_epilogue<XT>(acc[i][j], ep, k, o) : acc[i][j]);
    }
  }
}

// 1x1 stride-1 dense layers whose feature map is too small for the TMA-fed kernel's 32-pixel runs
bool pw_small_takes(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups) {
  static const bool off = [] { const char* e = getenv("PO2_PW_SMALL"); return e && e[0] == '0'; }();
  if (off || R != 1 || S != 1 || stride != 1 || pad != 0 || groups != 1) return false;
  const int64_t HW = (int64_t)H * W;
  return HW <= 16 && (int64_t)B * HW <= 16384;
}

int launch_pw_small(const void* x, const float* w, void* out, int B, int C, int HW, int K, const ConvEpilogue& ep,
                    int dtype, cudaStream_t st) {
  PwGeom g;
  g.M = B * HW; g.C = C; g.K = K; g.HW = HW;
  g.div_hw = make_fastdiv((uint32_t)HW);
  const int tiles = ((g.M + PW_TM - 1) / PW_TM) * ((K + PW_TN - 1) / PW_TN);
  int KS = (device_sm_count() + tiles - 1) / tiles;         // fill the SMs; every CTA keeps at least two channel chunks
  const int max_ks = C / (2 * PW_TK);
  if (KS > max_ks) KS = max_ks;
  if (KS > 8) KS = 8;
  { const char* e = getenv("PO2_PW_KS"); if (e && atoi(e) > 0 && KS > atoi(e)) KS = atoi(e); }
  if (KS < 1) KS = 1;
  g.KS = KS;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)((g.M + PW_TM - 1) / PW_TM), (unsigned)((K + PW_TN - 1) / PW_TN), (unsigned)KS);
  cfg.blockDim = dim3(PW_THREADS);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 1; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = (unsigned)KS;
  cfg.attrs = attr;
  cfg.numAttrs = KS > 1 ? 1 : 0;
  if (dtype == PO2_BF16)
    return (int)cudaLaunchKernelEx(&cfg, conv_pw_small_kernel<__nv_bfloat16>, (const __nv_bfloat16*)x, w,
                                   (__nv_bfloat16*)out, g, ep);
  return (int)cudaLaunchKernelEx(&cfg, conv_pw_small_kernel<float>, (const float*)x, w, (float*)out, g, ep);
}

// ------------------------------------------------------------------------------------------------
// Weight gradient of the same small pointwise layers, and of every 1x1 stride-1 layer with a short reduction that is
// wider than the tcgen05 weight-gradient kernels take (K > 128 output or C > 256 input channels: MobileNetV2's
// expansion / projection layers, MobileViT's 1x1 layers at 32x32):
//   gw[k][c] = sum_{m = (image, pixel)} g[n][k][p] * x[n][c][p],   m < B*HW <= PWW_MAX_M
// a GEMM with up to 960 x 960 outputs, a reduction of at most 8192 and at most 2^26 multiply-adds (MobileNetV2's
// largest: 39 M).  Beyond that cuDNN's tensor-core kernels win (measured on a B200: 24->144 at B*H*W = 16384
// 20.2 against 16.4 us, 160->960 at 8192 170 against 45 us).  fp32 CUDA cores, exact fmaf (no operand
// rounding).  CTA (k tile, c tile, split) = 64 x 64 outputs, 256 threads with 4 x 4 accumulators each, summing
// the contiguous range of 16-pixel chunks of its split; the reduction is split over blockIdx.z so that a small K x C
// still fills the SMs.  Every CTA writes its partial tile [split][k][c]; conv_wgrad_reduce_kernel (ntaps = 1,
// launched programmatically behind this grid) adds the splits in a fixed order: deterministic, no atomics.
// ------------------------------------------------------------------------------------------------
constexpr int PWW_TK = 64, PWW_TC = 64, PWW_TM = 16, PWW_THREADS = 256;
constexpr int PWW_MAX_M = 8192;            // B*HW: MobileNetV2's largest reduction (24->144 @8x8, batch 128)
constexpr int64_t PWW_MAX_FMA = 1ll << 26;  // B*HW*C*K

struct PwWgGeom {
  int M, C, K, HW;
  int chunks_per_split;                    // 16-pixel chunks summed by one CTA
  int vec;                                 // HW % 4 == 0 and 16-byte aligned operands: 128-bit loads
  int vst;                                 // C % 4 == 0 and a 16-byte aligned workspace: 128-bit partial stores
  FastDiv div_hw;
};

__global__ void __launch_bounds__(PWW_THREADS) conv_wgrad_pw_kernel(const float* __restrict__ g,
                                                                    const float* __restrict__ x,
                                                                    float* __restrict__ partial, PwWgGeom q) {
  __shared__ __align__(16) float Gs[PWW_TM][PWW_TK + 4];   // [m][k]
  __shared__ __align__(16) float Xs[PWW_TM][PWW_TC + 4];   // [m][c]
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the reduce kernel waits for this grid's completion
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const int k0 = blockIdx.x * PWW_TK, c0 = blockIdx.y * PWW_TC;
  const int M = q.M, C = q.C, K = q.K, HW = q.HW;
  const int m_begin = blockIdx.z * q.chunks_per_split * PWW_TM;
  const int m_end = min(M, m_begin + q.chunks_per_split * PWW_TM);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  // loader role: channel lane = tid % 64 of both tiles, pixels (tid / 64) * 4 .. +3 of the chunk.  Consecutive lanes
  // read consecutive channels: one 128-byte line per warp when HW == 1, 128-bit vectors along the pixels otherwise.
  const int lch = tid & 63, lm = (tid >> 6) * 4;
  const int lk = k0 + lch, lc = c0 + lch;
  float gv[4], xv[4];
  auto load_chunk = [&](int m0) {
    const int m = m0 + lm;
    if (q.vec) {                            // the quad m .. m + 3 lies in one image (HW % 4 == 0, m % 4 == 0)
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
      if (m < m_end) {
        const int n = fdiv(m, q.div_hw), p = m - n * HW;
        if (lk < K) a = __ldg(reinterpret_cast<const float4*>(g + ((size_t)n * K + lk) * HW + p));
        if (lc < C) b = __ldg(reinterpret_cast<const float4*>(x + ((size_t)n * C + lc) * HW + p));
      }
      gv[0] = a.x; gv[1] = a.y; gv[2] = a.z; gv[3] = a.w;
      xv[0] = b.x; xv[1] = b.y; xv[2] = b.z; xv[3] = b.w;
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float a = 0.f, b = 0.f;
        if (m + e < m_end) {
          const int n = fdiv(m + e, q.div_hw), p = m + e - n * HW;
          if (lk < K) a = __ldg(g + ((size_t)n * K + lk) * HW + p);
          if (lc < C) b = __ldg(x + ((size_t)n * C + lc) * HW + p);
        }
        gv[e] = a; xv[e] = b;
      }
    }
  };
  int m0 = m_begin;
  if (m0 < m_end) load_chunk(m0);
  for (; m0 < m_end; m0 += PWW_TM) {
    __syncthreads();                                        // the previous chunk has been consumed
#pragma unroll
    for (int e = 0; e < 4; ++e) { Gs[lm + e][lch] = gv[e]; Xs[lm + e][lch] = xv[e]; }
    __syncthreads();
    if (m0 + PWW_TM < m_end) load_chunk(m0 + PWW_TM);       // the next chunk's loads fly during this chunk's FMAs
#pragma unroll
    for (int mm = 0; mm < PWW_TM; ++mm) {
      const float4 a4 = *reinterpret_cast<const float4*>(&Gs[mm][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Xs[mm][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
  }
  const int c = c0 + tx * 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = k0 + ty * 4 + i;
    if (k >= K || c >= C) continue;
    float* dst = partial + ((size_t)blockIdx.z * K + k) * C + c;
    if (q.vst) {
      *reinterpret_cast<float4*>(dst) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (c + j < C) dst[j] = acc[i][j];
    }
  }
}

// 1x1 stride-1 dense layers small enough for one CUDA-core GEMM (compute 0 / 2: the fp32 mode's backward is
// aten.convolution_backward by design)
bool pw_wgrad_takes(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups, int compute) {
  if (R != 1 || S != 1 || stride != 1 || pad != 0 || groups != 1 || !(compute == 0 || compute == 2)) return false;
  if (B < 1 || C < 1 || H < 1 || W < 1 || K < 1) return false;
  const int64_t M = (int64_t)B * H * W;
  return M <= PWW_MAX_M && M * C * K <= PWW_MAX_FMA;
}

// splits of the reduction: about two CTAs per SM, every CTA at least four 16-pixel chunks, and every split non-empty
// (a pure function of the shape and the SM count, so the summation order -- the bits -- is too)
static void pw_wgrad_split(int M, int C, int K, int& splits, int& chunks_per_split) {
  const int tiles = ((K + PWW_TK - 1) / PWW_TK) * ((C + PWW_TC - 1) / PWW_TC);
  const int chunks = (M + PWW_TM - 1) / PWW_TM;
  int want = (2 * device_sm_count() + tiles - 1) / tiles;
  if (want > chunks / 4) want = chunks / 4;
  if (want < 1) want = 1;
  chunks_per_split = (chunks + want - 1) / want;
  splits = (chunks + chunks_per_split - 1) / chunks_per_split;
}

size_t pw_wgrad_partial_bytes(int B, int C, int H, int W, int K) {
  int splits, cps;
  pw_wgrad_split(B * H * W, C, K, splits, cps);
  return (size_t)splits * K * C * sizeof(float);
}

int launch_pw_wgrad(const float* g, const float* x, float* gw, void* workspace, int B, int C, int HW, int K,
                    cudaStream_t st) {
  PwWgGeom q;
  q.M = B * HW; q.C = C; q.K = K; q.HW = HW;
  q.div_hw = make_fastdiv((uint32_t)HW);
  q.vec = HW % 4 == 0 && (reinterpret_cast<uintptr_t>(g) & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0;
  q.vst = C % 4 == 0 && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0;
  int splits;
  pw_wgrad_split(q.M, C, K, splits, q.chunks_per_split);
  const dim3 grid((unsigned)((K + PWW_TK - 1) / PWW_TK), (unsigned)((C + PWW_TC - 1) / PWW_TC), (unsigned)splits);
  conv_wgrad_pw_kernel<<<grid, PWW_THREADS, 0, st>>>(g, x, (float*)workspace, q);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  return launch_wgrad_reduce((const float*)workspace, gw, splits, K, C, 1, st);
}

}  // namespace po2
