// Shared device helpers for the PO2 kernels (sm_100a).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "../../include/po2_b200.h"

#define PO2_NEVER 0xFFFFFFFFu

namespace po2 {

// ---- storage-dtype traits: the kernels work on raw bit patterns of the storage type ----------
template <int DT> struct Tr;

template <> struct Tr<PO2_F32> {
  using T = float;                  // the storage type
  static constexpr int EB = 4;      // bytes per element
  static constexpr int MB = 23;     // mantissa bits (binade index = magnitude >> MB)
  static constexpr int EPV = 4;     // elements per 16-byte vector
  static constexpr int NBIN = 256;  // number of binades
  static constexpr uint32_t MAG = 0x7FFFFFFFu, SGN = 0x80000000u, QNAN = 0x7FC00000u, INF = 0x7F800000u;
  static __device__ __forceinline__ float val(uint32_t p) { return __uint_as_float(p); }
  static __device__ __forceinline__ uint32_t pat(float f) { return __float_as_uint(f); }
};
template <> struct Tr<PO2_BF16> {
  using T = __nv_bfloat16;
  static constexpr int EB = 2, MB = 7, EPV = 8, NBIN = 256;
  static constexpr uint32_t MAG = 0x7FFFu, SGN = 0x8000u, QNAN = 0x7FC0u, INF = 0x7F80u;
  static __device__ __forceinline__ float val(uint32_t p) { return __uint_as_float(p << 16); }
  static __device__ __forceinline__ uint32_t pat(float f) {
    return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(f));
  }
};
template <> struct Tr<PO2_F16> {
  using T = __half;
  static constexpr int EB = 2, MB = 10, EPV = 8, NBIN = 32;
  static constexpr uint32_t MAG = 0x7FFFu, SGN = 0x8000u, QNAN = 0x7E00u, INF = 0x7C00u;
  static __device__ __forceinline__ float val(uint32_t p) {
    return __half2float(__ushort_as_half((unsigned short)p));
  }
  static __device__ __forceinline__ uint32_t pat(float f) {
    return (uint32_t)__half_as_ushort(__float2half_rn(f));
  }
};

// round an fp32 intermediate to the storage grid (torch rounds half types after every op)
template <int DT> __device__ __forceinline__ float round_storage(float f) {
  if (DT == PO2_F32) return f;
  return Tr<DT>::val(Tr<DT>::pat(f));
}

// exact 2^k as fp32 for any integer k (0 below 2^-149, +inf above 2^127) == torch's 2**q
__device__ __forceinline__ float exp2_int(int k) {
  if (k > 127) return __uint_as_float(0x7F800000u);
  if (k >= -126) return __uint_as_float((uint32_t)(k + 127) << 23);
  if (k >= -149) return __uint_as_float(1u << (k + 149));
  return 0.0f;
}

// ---- streaming 128-bit global access ----------------------------------------------------------
__device__ __forceinline__ uint4 ldg_stream(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ uint4 ldg_keep(const uint4* p) {   // normal policy: leave it in L2
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream(uint4* p, const uint4& v) {
  asm volatile("st.global.L1::no_allocate.v4.u32 [%0], {%1,%2,%3,%4};"
               :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

__device__ __forceinline__ uint32_t warp_max_u32(uint32_t v) {
  return __reduce_max_sync(0xFFFFFFFFu, v);
}

// ---- n / d for 0 <= n < 2^31 via one mul-hi (d >= 1) -----------------------------------------------
struct FastDiv {
  uint32_t mul, shr, d;
};
__host__ __device__ __forceinline__ int fdiv(int n, const FastDiv& f) {
  if (f.d <= 1) return n;
#ifdef __CUDA_ARCH__
  return (int)(__umulhi((uint32_t)n, f.mul) >> f.shr);
#else
  return (int)(((uint64_t)(uint32_t)n * f.mul) >> 32 >> f.shr);
#endif
}
inline FastDiv make_fastdiv(uint32_t d) {
  // s = ceil(log2 d), mul = ceil(2^(31+s) / d) in [2^31, 2^32): floor(n/d) == umulhi(n, mul) >> (s-1)
  // for every 0 <= n < 2^31 (error term e = mul*d - 2^(31+s) < d <= 2^s, so n*e < 2^(31+s)).
  FastDiv f; f.d = d; f.mul = 0; f.shr = 0;
  if (d <= 1) return f;
  uint32_t sh = 0;
  while ((1u << sh) < d) ++sh;
  f.mul = (uint32_t)(((1ull << (31 + sh)) + d - 1) / d);
  f.shr = sh - 1;
  return f;
}

// Optional epilogue of the fused quantizer: besides y it emits the conv's tensor-core B operand
// Bp[nt][tap][c/G][n][G] = y / scale = exact +-2^q as bf16 or tf32 (layout: csrc/po2_conv.cu).  Only for
// weights whose C and K need no padding, so that every Bp entry is written.
struct PackArgs {
  void* Bp;                  // nullptr: off
  int G;                     // 8: bf16 operand, 4: tf32 (fp32) operand -- channels per 16-byte plane entry
  int C, K, taps, NT, ncg;   // ncg = C / G
  int tapminor;              // 1 (3x3, TMA-fed conv): Bp[nt][r][c/G][s][n][G] -- the three filter columns of a row are
                             // consecutive N rows, so one MMA covers them (N = 3 * NT)
  FastDiv div_ct, div_t, div_nt;   // by C*taps, taps, NT
  // second operand of the same weight: the DATA-GRADIENT conv's (in = K, out = C channels, taps rotated by 180
  // degrees), so that backward needs no pack launch.  Bp2 == nullptr: off.
  void* Bp2;
  int NT2, ncg2, tapminor2;        // ncg2 = K / G
  FastDiv div_nt2;
};

// The packed layout in one place: store r, the operand value of weight element (k, c, tap) of a (K, C, taps) tensor,
// into Bp (and, when on, its data-gradient twin Bp2).  r must be exact in the operand type (bf16 / tf32).
__device__ __forceinline__ void pack_store(const PackArgs& pk, int k, int c, int tap, float r) {
  const int nt = fdiv(k, pk.div_nt);
  const int n = k - nt * pk.NT;
  const int cg = pk.G == 8 ? (c >> 3) : (c >> 2), cj = c & (pk.G - 1);
  const size_t idx = pk.tapminor
      ? (((((size_t)nt * 3 + tap / 3) * pk.ncg + cg) * 3 + tap % 3) * pk.NT + n) * pk.G + cj
      : ((((size_t)nt * pk.taps + tap) * pk.ncg + cg) * pk.NT + n) * pk.G + cj;
  if (pk.G == 8) reinterpret_cast<__nv_bfloat16*>(pk.Bp)[idx] = __float2bfloat16_rn(r);
  else reinterpret_cast<float*>(pk.Bp)[idx] = r;
  if (pk.Bp2) {
    // data-gradient operand: out channel = c, in channel = k, tap rotated (csrc/po2_conv.cu, transpose)
    const int tap2 = pk.taps - 1 - tap;
    const int nt2 = fdiv(c, pk.div_nt2);
    const int n2 = c - nt2 * pk.NT2;
    const int cg2 = pk.G == 8 ? (k >> 3) : (k >> 2), cj2 = k & (pk.G - 1);
    const size_t idx2 = pk.tapminor2
        ? (((((size_t)nt2 * 3 + tap2 / 3) * pk.ncg2 + cg2) * 3 + tap2 % 3) * pk.NT2 + n2) * pk.G + cj2
        : ((((size_t)nt2 * pk.taps + tap2) * pk.ncg2 + cg2) * pk.NT2 + n2) * pk.G + cj2;
    if (pk.G == 8) reinterpret_cast<__nv_bfloat16*>(pk.Bp2)[idx2] = __float2bfloat16_rn(r);
    else reinterpret_cast<float*>(pk.Bp2)[idx2] = r;
  }
}

// quantize w (fp32, n = K*C*taps elements) into y + scale AND the packed operand, one launch
int fused_quantize_pack(const void* w, void* y, float* scale_out, int64_t n, int bits, int fsr, int mode,
                        int flavor, void* workspace, const PackArgs& pk, cudaStream_t st);

// one tensor of the multi-tensor quantize+pack kernel (fp32 weights)
struct MultiDesc {
  const uint4* x; uint4* y; float* scale_out;
  double* sse_out;           // sum((y - x)^2) of this tensor (models/quantized_conv.py:43), or nullptr
  int64_t n;
  int bits, fsr, mode, flavor;
  PackArgs pk;
};
int multi_fused_capacity();
int multi_fused_launch(const MultiDesc* descs_dev, int ntensors, int csize, cudaStream_t st);
int check_quant_args(int bits, int fsr, int mode, int flavor);

// csrc/po2_lin.cu: lin / lin+ quantizer with optional operand emission.  A lin weight is n * 2^k (|n| <= 2^(bits-1) - 1,
// one power-of-two step per input channel), so the packed operand holds y itself (the conv's scale is 1.0).
struct LinDesc {             // one tensor of the multi-tensor launch
  const float* w; float* y;
  int K, C, RS, bits, iters, plus, flavor;
  int cta0;                  // first CTA of this tensor: the tensors' CTAs are consecutive, one per input channel
  PackArgs pk;
};
int lin_check_args(int K, int C, int RS, int bits, int num_iters, int flavor);
int lin_launch(const float* w, float* y, int K, int C, int RS, int bits, int iters, int plus, int flavor,
               const PackArgs& pk, cudaStream_t st);

// ---- optional conv epilogue: eval-mode BatchNorm folded into the conv (per-out-channel affine), the residual add
// and the activation of the block -- y = act(conv * a[k] + b[k] + res) -- models/resnet.py:55-71 at inference.
// a == nullptr: plain conv.  act: 0 none, 1 ReLU, 2 ReLU6, 3 SiLU (the codes of the BatchNorm kernels).
struct ConvEpilogue {
  const float* a;
  const float* b;
  const float* res;      // same shape as the output, or nullptr; stored in the output's type (bf16 for a bf16 conv)
  int act;
};
__device__ __forceinline__ float conv_act(float v, int act) {
  if (act == 1) return fmaxf(v, 0.f);
  if (act == 2) return fminf(fmaxf(v, 0.f), 6.f);
  if (act == 3) return v / (1.f + __expf(-v));
  return v;
}

// ---- activation storage of the conv forward: fp32, or bf16 (inference of bf16 models).  Arithmetic stays fp32; a
// bf16 value widens exactly and a result is rounded to bf16 once, when it is stored.
__device__ __forceinline__ float act_ld(const float* p) { return __ldg(p); }
__device__ __forceinline__ float act_ld(const __nv_bfloat16* p) { return __bfloat162float(__ldg(p)); }
template <typename I> __device__ __forceinline__ void act_st(float* p, I i, float v) { p[i] = v; }
template <typename I> __device__ __forceinline__ void act_st(__nv_bfloat16* p, I i, float v) { p[i] = __float2bfloat16_rn(v); }

// v: conv result of out channel k; idx: its offset in the output tensor (and the residual, stored as T)
template <typename T = float>
__device__ __forceinline__ float conv_epilogue(float v, const ConvEpilogue& ep, int k, size_t idx) {
  v = fmaf(v, __ldg(ep.a + k), __ldg(ep.b + k));
  if (ep.res) v += act_ld(reinterpret_cast<const T*>(ep.res) + idx);
  return conv_act(v, ep.act);
}

// csrc/po2_conv.cu: gw[(k*C + c)*ntaps + tap] = sum over parts of partial[part][tap][k][c], in part order (launched
// programmatically behind the kernel that wrote the partials)
int launch_wgrad_reduce(const float* partial, float* gw, int nparts, int K, int C, int ntaps, cudaStream_t st);
// csrc/po2_conv_bwd.cu: fp32 cluster split-K GEMM for 1x1 convs on feature maps of <= 16 pixels
bool pw_small_takes(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups);
// x / out: fp32 (dtype PO2_F32) or bf16 (PO2_BF16) NCHW; w: fp32
int launch_pw_small(const void* x, const float* w, void* out, int B, int C, int HW, int K, const ConvEpilogue& ep,
                    int dtype, cudaStream_t st);
// csrc/po2_conv_bwd.cu: the weight gradient of 1x1 stride-1 layers with B*H*W <= 8192 and B*H*W*C*K <= 2^26 -- fp32
// split-reduction GEMM
// + the fixed-order reduce kernel (two launches); the workspace holds the partials
bool pw_wgrad_takes(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups, int compute);
size_t pw_wgrad_partial_bytes(int B, int C, int H, int W, int K);
int launch_pw_wgrad(const float* g, const float* x, float* gw, void* workspace, int B, int C, int HW, int K,
                    cudaStream_t st);

// ---- per-device one-time host state ---------------------------------------------------------------
// Kernel attributes (cudaFuncSetAttribute) and the SM count belong to a DEVICE, not to the process:
// a process that drives several GPUs must set them once per device, and two host threads may race
// to be first.  One std::once_flag per device ordinal; a failed initialisation stays failed (the
// error is returned by every later call on that device).
constexpr int PO2_MAX_DEVICES = 64;
inline int current_device() {
  int d = 0;
  return (cudaGetDevice(&d) == cudaSuccess && d >= 0 && d < PO2_MAX_DEVICES) ? d : -1;
}
struct PerDeviceOnce {
  std::once_flag flag[PO2_MAX_DEVICES];
  cudaError_t err[PO2_MAX_DEVICES];
  template <class F> cudaError_t run(F&& f) {
    const int d = current_device();
    if (d < 0) return cudaErrorInvalidDevice;
    std::call_once(flag[d], [&] { err[d] = f(); });
    return err[d];
  }
};
int device_sm_count();          // SMs of the CURRENT device (cached per device; 148 if the query fails)

}  // namespace po2
