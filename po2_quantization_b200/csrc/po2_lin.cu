// lin / lin+ quantizers (SURVEY.md section 8f "next" #1, reference utils/quantizers.py:8-16, 59-136):
// a per-input-channel uniform quantizer whose step is constrained to a power of two and refined by
// num_iters rounds of  step = 2^round(log2(<q, w> / <q, q>))  (lin+: the ratio times sqrt(8/9) first).
//
// One CTA per input channel: the channel's K*R*S weights are staged in shared memory once and every
// round (two reductions + a re-quantisation) runs out of it, so the whole quantizer is ONE launch
// instead of ~16 ATen launches per round.  The arithmetic follows the reference op by op in fp32
// (IEEE division, round-half-even, the multiply-then-divide of uniform_quantize); the two inner
// products are accumulated in double from fp32 products, i.e. they are the correctly rounded sums,
// where torch's own fp32 summation order may be a few ulp off -- the power-of-two rounding absorbs
// that except at an exact tie.  round(log2(.)) uses the same scanned boundary table as the PO2
// quantizer (csrc/po2_boundaries.inc) for steps <= 1, libdevice log2f above.
#include "po2_common.cuh"

namespace po2 {
namespace {                                    // this translation unit's own copy of the boundary table
#include "po2_boundaries.inc"
}

constexpr int LIN_THREADS = 256;
constexpr int LIN_MAX_ELEMS = 12000;          // per input channel (< 48 KB of shared memory with the statics)

__device__ __forceinline__ double lin_warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}

__device__ __forceinline__ float lin_clamp(float t, float lim) { return t != t ? t : fminf(fmaxf(t, -lim), lim); }

// 2 ** round(log2(step)) as torch evaluates it in the storage type DT (fp32 or bf16)
template <int DT>
__device__ __forceinline__ float lin_pow2_round_log2(float step, int flavor) {
  const uint32_t pat = __float_as_uint(step);
  if (step > 0.0f && step <= 1.0f) {
    // exponent of the binade, then one table lookup decides between k and k + 1
    int e = (int)(pat >> 23) - 127;
    if ((pat >> 23) == 0) e = -127 - (__clz(pat) - 9);           // subnormal: position of the leading bit
    int k = e;
    if (e + 1 <= PO2_KMAX && e + 1 >= PO2_KMIN && pat >= PO2_BOUNDS[flavor][DT][0][e + 1 - PO2_KMIN]) k = e + 1;
    if (k < PO2_KMIN) k = PO2_KMIN;                               // round(log2) of the smallest subnormals
    return exp2_int(k);
  }
  // step > 1, zero, negative, inf, NaN: the float ops themselves (NaN / inf propagate as in torch)
  return exp2f(rintf(round_storage<DT>(log2f(step))));
}

// input channel c of w (K, C, RS) -> y; with pk.Bp set, also the channel's entries of the conv's packed operand(s)
// (the operand value is y itself: n * 2^k with |n| <= 2^(bits-1) - 1 -- exact in bf16 for bits <= 9, in tf32 for
// bits <= 12 -- once at least one refinement round has made the step a power of two).  w, y: float (PO2_F32) or
// __nv_bfloat16 (PO2_BF16)
template <int DT>
__device__ __forceinline__ void lin_channel(const typename Tr<DT>::T* __restrict__ w,
                                            typename Tr<DT>::T* __restrict__ y, int K, int C, int RS, int bits,
                                            int iters, int plus, int flavor, int c, const PackArgs& pk) {
  extern __shared__ float sw[];
  __shared__ double red[LIN_THREADS / 32][2];
  __shared__ float bc[2];
  const int n = K * RS;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  // ---- stage the channel, min / max (torch.amax / amin propagate NaN)
  float hi = -INFINITY, lo = INFINITY;
  bool nan = false;
  for (int i = tid; i < n; i += LIN_THREADS) {
    const int k = i / RS, j = i - k * RS;
    float v;
    if constexpr (DT == PO2_F32) v = __ldg(w + ((size_t)k * C + c) * RS + j);
    else v = __bfloat162float(__ldg(w + ((size_t)k * C + c) * RS + j));     // exact widening
    sw[i] = v;
    nan |= (v != v);
    hi = fmaxf(hi, v);
    lo = fminf(lo, v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    hi = fmaxf(hi, __shfl_xor_sync(0xFFFFFFFFu, hi, o));
    lo = fminf(lo, __shfl_xor_sync(0xFFFFFFFFu, lo, o));
  }
  nan = __any_sync(0xFFFFFFFFu, nan);
  if (lane == 0) { red[warp][0] = (double)hi; red[warp][1] = nan ? (double)NAN : (double)lo; }
  __syncthreads();
  if (tid == 0) {
    float H = -INFINITY, L = INFINITY;
    bool anynan = false;
    for (int q = 0; q < LIN_THREADS / 32; ++q) {
      H = fmaxf(H, (float)red[q][0]);
      const double l = red[q][1];
      if (l != l) anynan = true; else L = fminf(L, (float)l);
    }
    const float levels = (float)((1 << bits) - 1);
    bc[0] = anynan ? NAN : round_storage<DT>(__fdiv_rn(round_storage<DT>(H - L), levels));  // (max - min) / (2**bits - 1)
  }
  __syncthreads();
  float step = bc[0];
  const float lim = (float)((1 << (bits - 1)) - 1);
  const float c89 = __fsqrt_rn(8.0f / 9.0f);                       // torch.sqrt(torch.tensor(8/9))
  // q = uniform_quantize(w, step) / step = (step * clamp(round(w / step), -lim, lim)) / step
  // (torch.clamp propagates NaN, fminf / fmaxf would swallow it); in bf16 each op's result is rounded to bf16
#define LIN_R(t) round_storage<DT>(t)
#define LIN_Q(v, s) LIN_R(__fdiv_rn(LIN_R(__fmul_rn((s), LIN_R(lin_clamp(rintf(LIN_R(__fdiv_rn((v), (s)))), lim)))), (s)))
  for (int it = 0; it < iters; ++it) {
    double num = 0.0, den = 0.0;
    for (int i = tid; i < n; i += LIN_THREADS) {
      const float v = sw[i];
      const float q = LIN_Q(v, step);
      num += (double)LIN_R(__fmul_rn(q, v));
      den += (double)LIN_R(__fmul_rn(q, q));
    }
    num = lin_warp_sum(num);
    den = lin_warp_sum(den);
    __syncthreads();                                              // red / bc reuse
    if (lane == 0) { red[warp][0] = num; red[warp][1] = den; }
    __syncthreads();
    if (tid == 0) {
      double a = 0.0, b = 0.0;
      for (int q = 0; q < LIN_THREADS / 32; ++q) { a += red[q][0]; b += red[q][1]; }
      float s = LIN_R(__fdiv_rn(LIN_R((float)a), LIN_R((float)b)));
      if (plus) s = LIN_R(__fmul_rn(c89, s));                     // the fp32 constant, as torch uses it for bf16 too
      bc[0] = lin_pow2_round_log2<DT>(s, flavor);
    }
    __syncthreads();
    step = bc[0];
  }
  for (int i = tid; i < n; i += LIN_THREADS) {
    const int k = i / RS, j = i - k * RS;
    const float q = LIN_Q(sw[i], step);
    const float yv = LIN_R(__fmul_rn(q, step));
    if constexpr (DT == PO2_F32) y[((size_t)k * C + c) * RS + j] = yv;
    else y[((size_t)k * C + c) * RS + j] = __float2bfloat16_rn(yv);     // exact: yv is on the bf16 grid
    if (pk.Bp) pack_store(pk, k, c, j, yv);
  }
#undef LIN_Q
#undef LIN_R
}

template <int DT>
__global__ void __launch_bounds__(LIN_THREADS) lin_quantize_kernel(const typename Tr<DT>::T* __restrict__ w,
                                                                   typename Tr<DT>::T* __restrict__ y, int K, int C,
                                                                   int RS, int bits, int iters, int plus, int flavor,
                                                                   PackArgs pk) {
  lin_channel<DT>(w, y, K, C, RS, bits, iters, plus, flavor, blockIdx.x, pk);
}

// Multi-tensor form: ONE launch for the lin layers of a model, one CTA per (tensor, input channel).  The tensor of a
// CTA is found by binary search over the descriptors' first CTAs (ascending by construction).
__global__ void __launch_bounds__(LIN_THREADS) lin_multi_kernel(const LinDesc* __restrict__ descs, int ntensors) {
  const int b = blockIdx.x;
  int lo = 0, hi = ntensors - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (descs[mid].cta0 <= b) lo = mid; else hi = mid - 1;
  }
  const LinDesc& d = descs[lo];
  lin_channel<PO2_F32>(d.w, d.y, d.K, d.C, d.RS, d.bits, d.iters, d.plus, d.flavor, b - d.cta0, d.pk);
}

int lin_check_args(int K, int C, int RS, int bits, int num_iters, int flavor) {
  if (K <= 0 || C <= 0 || RS <= 0 || (int64_t)K * C * RS >= (1ll << 31)) return PO2_E_SIZE;
  if (bits < 2 || bits > 16 || num_iters < 0) return PO2_E_BITS;
  if (flavor < 0 || flavor >= PO2_NUM_FLAVORS) return PO2_E_FLAVOR;
  if (flavor == PO2_FLAVOR_TORCH_CUDA && !PO2_HAVE_TORCH_CUDA_TABLE) return PO2_E_FLAVOR;
  if ((int64_t)K * RS > LIN_MAX_ELEMS) return PO2_E_UNSUPPORTED;
  return 0;
}

int lin_launch(const float* w, float* y, int K, int C, int RS, int bits, int iters, int plus, int flavor,
               const PackArgs& pk, cudaStream_t st) {
  const size_t smem = (size_t)K * RS * sizeof(float);
  lin_quantize_kernel<PO2_F32><<<C, LIN_THREADS, smem, st>>>(w, y, K, C, RS, bits, iters, plus, flavor, pk);
  return (int)cudaGetLastError();
}

}  // namespace po2

using namespace po2;

extern "C" {

int po2_lin_max_channel_elems(void) { return LIN_MAX_ELEMS; }

int po2_lin_quantize_dt(const void* w, void* y, int K, int C, int RS, int bits, int num_iters, int plus, int flavor,
                        int dtype, void* stream) {
  if (!w || !y) return PO2_E_NULL;
  if (dtype != PO2_F32 && dtype != PO2_BF16) return PO2_E_DTYPE;
  if (int e = lin_check_args(K, C, RS, bits, num_iters, flavor)) return e;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == PO2_F32)
    return lin_launch((const float*)w, (float*)y, K, C, RS, bits, num_iters, plus, flavor, PackArgs{}, st);
  const size_t smem = (size_t)K * RS * sizeof(float);           // the channel's fp32 widening
  lin_quantize_kernel<PO2_BF16><<<C, LIN_THREADS, smem, st>>>((const __nv_bfloat16*)w, (__nv_bfloat16*)y, K, C, RS, bits,
                                                              num_iters, plus, flavor, PackArgs{});
  return (int)cudaGetLastError();
}

int po2_lin_quantize(const void* w, void* y, int K, int C, int RS, int bits, int num_iters, int plus, int flavor,
                     void* stream) {
  return po2_lin_quantize_dt(w, y, K, C, RS, bits, num_iters, plus, flavor, PO2_F32, stream);
}

size_t po2_lin_multi_desc_bytes(void) { return sizeof(LinDesc); }

int po2_lin_quantize_pack_multi(const void* device_table, int ntensors, int total_ctas, int max_channel_elems,
                                void* stream) {
  if (!device_table) return PO2_E_NULL;
  if (ntensors < 0 || total_ctas < 0) return PO2_E_SIZE;
  if (ntensors == 0 || total_ctas == 0) return 0;
  if (max_channel_elems <= 0 || max_channel_elems > LIN_MAX_ELEMS) return PO2_E_UNSUPPORTED;
  const size_t smem = (size_t)max_channel_elems * sizeof(float);
  lin_multi_kernel<<<total_ctas, LIN_THREADS, smem, (cudaStream_t)stream>>>((const LinDesc*)device_table, ntensors);
  return (int)cudaGetLastError();
}

}  // extern "C"
