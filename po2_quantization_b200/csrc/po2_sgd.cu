// The QAT step's parameter update (train.py:54-56, :92: torch.optim.SGD with momentum and weight decay) for ALL
// parameters in one launch per <= 96 tensors.  torch's foreach implementation needs 14 launches for the 171
// parameters of ResNet-56 (~ 88 us of a 2.8 ms step); this is the same arithmetic, rounding by rounding:
//     g   = fma(weight_decay, p, grad)            torch._foreach_add(grads, params, alpha=weight_decay)
//     buf = rn(rn(buf * momentum) + g)            _foreach_mul_(bufs, momentum); _foreach_add_(bufs, grads)
//           (first step: buf = g)                 torch.clone(grad)
//     p   = fma(-lr, buf, p)                      _foreach_add_(params, bufs, alpha=-lr)
// (ATen's add functor computes a + alpha * b, which nvcc contracts into one fma; alpha == 1 is a plain add.)
#include "po2_common.cuh"

namespace po2 {

constexpr int SGD_MAX_TENSORS = 96;
constexpr int SGD_THREADS = 256;
constexpr int SGD_CHUNK = SGD_THREADS * 4 * 4;      // elements per CTA: 4 x float4 per thread

struct SgdTable {                                   // 96 * 28 + 4 * 97 = 3076 bytes of kernel parameters
  float* p[SGD_MAX_TENSORS];
  const float* g[SGD_MAX_TENSORS];
  float* buf[SGD_MAX_TENSORS];
  int n[SGD_MAX_TENSORS];
  int first_chunk[SGD_MAX_TENSORS + 1];             // CTA index of a tensor's first chunk
  int ntensors;
};

__device__ __forceinline__ float sgd_one(float p, float g, float* buf, float lr, float mom, float wd, int first) {
  if (wd != 0.f) g = fmaf(wd, p, g);
  float b = g;
  if (mom != 0.f) {
    if (!first) b = __fadd_rn(__fmul_rn(*buf, mom), g);
    *buf = b;
  }
  return fmaf(-lr, b, p);
}

__global__ void __launch_bounds__(SGD_THREADS) sgd_multi_kernel(const __grid_constant__ SgdTable t, float lr, float mom,
                                                                 float wd, int first) {
  // which tensor does this CTA belong to: binary search over <= 97 prefix entries
  int lo = 0, hi = t.ntensors;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (t.first_chunk[mid] <= (int)blockIdx.x) lo = mid; else hi = mid;
  }
  const int n = t.n[lo];
  const int e0 = ((int)blockIdx.x - t.first_chunk[lo]) * SGD_CHUNK;
  float* __restrict__ p = t.p[lo];
  const float* __restrict__ g = t.g[lo];
  float* __restrict__ buf = t.buf[lo];
  const bool vec = ((reinterpret_cast<uintptr_t>(p) | reinterpret_cast<uintptr_t>(g) | reinterpret_cast<uintptr_t>(buf)) & 15) == 0;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int e = e0 + (u * SGD_THREADS + (int)threadIdx.x) * 4;
    if (e >= n) break;
    if (vec && e <= n - 4) {                        // n < 2^31 may be within 4 of 2^31: e + 4 would wrap
      float4 pv = *reinterpret_cast<const float4*>(p + e);
      const float4 gv = __ldg(reinterpret_cast<const float4*>(g + e));
      float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
      if (mom != 0.f && !first) bv = *reinterpret_cast<const float4*>(buf + e);
      pv.x = sgd_one(pv.x, gv.x, &bv.x, lr, mom, wd, first);
      pv.y = sgd_one(pv.y, gv.y, &bv.y, lr, mom, wd, first);
      pv.z = sgd_one(pv.z, gv.z, &bv.z, lr, mom, wd, first);
      pv.w = sgd_one(pv.w, gv.w, &bv.w, lr, mom, wd, first);
      *reinterpret_cast<float4*>(p + e) = pv;
      if (mom != 0.f) *reinterpret_cast<float4*>(buf + e) = bv;
    } else {
      for (int i = e; i < e + min(4, n - e); ++i) {
        float b = (mom != 0.f && !first) ? buf[i] : 0.f;
        const float pn = sgd_one(p[i], g[i], &b, lr, mom, wd, first);
        p[i] = pn;
        if (mom != 0.f) buf[i] = b;
      }
    }
  }
}

}  // namespace po2

extern "C" {

int po2_sgd_step(void* const* params, const void* const* grads, void* const* bufs, const long long* numels, int ntensors,
                 float lr, float momentum, float weight_decay, int first_step, void* stream) {
  using namespace po2;
  if (ntensors < 0) return PO2_E_SIZE;
  if (ntensors == 0) return 0;
  if (!params || !grads || !numels || (momentum != 0.f && !bufs)) return PO2_E_NULL;
  for (int i = 0; i < ntensors; ++i) {
    if (!params[i] || !grads[i] || (momentum != 0.f && !bufs[i])) return PO2_E_NULL;
    if (numels[i] <= 0 || numels[i] >= (1ll << 31)) return PO2_E_SIZE;
    if ((reinterpret_cast<uintptr_t>(params[i]) | reinterpret_cast<uintptr_t>(grads[i]) |
         (momentum != 0.f ? reinterpret_cast<uintptr_t>(bufs[i]) : 0)) & 3) return PO2_E_ALIGN;
  }
  for (int t0 = 0; t0 < ntensors; t0 += SGD_MAX_TENSORS) {
    SgdTable t;
    const int nt = ntensors - t0 < SGD_MAX_TENSORS ? ntensors - t0 : SGD_MAX_TENSORS;
    long long chunks = 0;
    for (int i = 0; i < nt; ++i) {
      t.p[i] = (float*)params[t0 + i];
      t.g[i] = (const float*)grads[t0 + i];
      t.buf[i] = momentum != 0.f ? (float*)bufs[t0 + i] : nullptr;
      t.n[i] = (int)numels[t0 + i];
      t.first_chunk[i] = (int)chunks;
      chunks += (numels[t0 + i] + SGD_CHUNK - 1) / SGD_CHUNK;
      if (chunks >= (1ll << 31)) return PO2_E_SIZE;
    }
    for (int i = nt; i < SGD_MAX_TENSORS; ++i) { t.p[i] = nullptr; t.g[i] = nullptr; t.buf[i] = nullptr; t.n[i] = 0; }
    for (int i = nt; i <= SGD_MAX_TENSORS; ++i) t.first_chunk[i] = (int)chunks;
    t.ntensors = nt;
    sgd_multi_kernel<<<(unsigned)chunks, SGD_THREADS, 0, (cudaStream_t)stream>>>(t, lr, momentum, weight_decay, first_step);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
  }
  return 0;
}

int po2_sgd_max_tensors_per_launch(void) { return po2::SGD_MAX_TENSORS; }

}  // extern "C"
