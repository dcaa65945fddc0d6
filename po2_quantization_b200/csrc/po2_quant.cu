// PO2 / PO2+ quantizer kernels for B200 (sm_100a) and their C ABI (include/po2_b200.h).
//
// What is computed (bit-exact to the reference, utils/quantizers.py:21-32 and :41-52):
//     s = max|x|;  v = |x / s|;  q = clamp(round(log2 v) [or round(log2(v/1.5)+0.5)], qmin, qmax)
//     y = 2^q * sign(x) * s
// How: no libm.  q is a monotone step function of |x|, so for a given s there is, per level
// j = q - qmin, one smallest bit pattern X[j] of |x| that reaches it, and one output pattern Y[j].
// Every CTA derives X[] from the scanned rounding-boundary table (po2_boundaries.inc, in v-space)
// with a few IEEE divisions (build_levels), buckets the thresholds by binade, and then each
// element costs: mask, shift, one 64-bit shared load, one compare, one 32-bit shared load, sign
// merge.  Loads/stores are 128-bit and coalesced; the max-abs reduction compares magnitude bit
// patterns as integers (NaN patterns sort above Inf, which reproduces torch.max's NaN
// propagation) with redux.sync + one atomicMax per CTA.
#include <stdio.h>

#include "po2_common.cuh"
#include "po2_boundaries.inc"

namespace po2 {

struct Workspace {            // zero-initialised by the caller once; kernels leave it zeroed
  unsigned int absmax;        // running max of magnitude bit patterns
  unsigned int arrive;        // CTA arrival counter
  unsigned int depart;        // CTA departure counter (fused kernel)
  unsigned int pad;
};

struct LevelTab {
  uint2 bt[256];              // per binade of |x| (fast path): .x = first threshold above the
                              //   binade's base level, .y = output pattern of the base level,
                              //   bit 31 = "irregular binade, take the exact slow path"
  uint8_t cb[256];            // per binade: base level (number of thresholds below the binade)
  uint32_t X[132];            // X[j]: smallest magnitude pattern with level >= j; X[nlev] = never
  uint32_t Y[128];            // Y[j]: output magnitude pattern of level j
  int special;                // 0: finite scale > 0; 1: scale NaN or 0 (all NaN); 2: scale +Inf
  uint32_t yinf;              // special == 2: pattern of 2^qmin * Inf in the storage dtype
};

#define PO2_IRR 0x80000000u

// Smallest magnitude pattern x (storage grid) with round_storage(x / s) >= b.  The predicate is
// monotone in x; start from fl(b*s) and walk (<= 2 steps in practice), bisect if that fails.
template <int DT>
__device__ uint32_t search_threshold(float b, float s, uint32_t s_pat) {
  auto pred = [&](uint32_t p) -> bool {
    return round_storage<DT>(__fdiv_rn(Tr<DT>::val(p), s)) >= b;
  };
  if (!pred(s_pat)) return PO2_NEVER;             // not even |x| == s reaches this level
  uint32_t g = Tr<DT>::pat(__fmul_rn(b, s));
  if (g > s_pat) g = s_pat;
  int guard = 0;
  while (!pred(g) && guard < 16) { ++g; ++guard; }
  while (g > 0 && pred(g - 1) && guard < 32) { --g; ++guard; }
  if (guard >= 16 && !(pred(g) && (g == 0 || !pred(g - 1)))) {
    uint32_t lo = 0, hi = s_pat;                  // pred(lo) false (v = 0 < b), pred(hi) true
    while (hi - lo > 1) {
      uint32_t mid = lo + ((hi - lo) >> 1);
      if (pred(mid)) hi = mid; else lo = mid;
    }
    g = hi;
  }
  return g;
}

// Builds the level table for scale s in shared memory.  All threads of the CTA must call it.
// The boundary of level `threadIdx.x` can be fetched before the scale is known (it does not depend on
// it); kernels whose critical path runs through the scale pass it in to take the table's global load
// off that path.
__device__ __forceinline__ uint32_t prefetch_bound(int dt, int bits, int fsr, int mode, int flavor) {
  const int k = fsr - (1 << (bits - 1)) + (int)threadIdx.x;
  if ((int)threadIdx.x >= (1 << (bits - 1)) || k < PO2_KMIN || k > PO2_KMAX) return PO2_NEVER;
  return PO2_BOUNDS[flavor][dt][mode][k - PO2_KMIN];
}

template <int DT>
__device__ void build_levels(LevelTab& T, float s, int bits, int fsr, int mode, int flavor,
                             bool have_pre = false, uint32_t pre_b = PO2_NEVER) {
  const int nlev = 1 << (bits - 1);
  const int qmin = fsr - nlev;
  const int tid = threadIdx.x, nthr = blockDim.x;
  const uint32_t s_bits = __float_as_uint(s);
  const bool s_nan = (s_bits & 0x7FFFFFFFu) > 0x7F800000u;
  const bool s_inf = (s_bits & 0x7FFFFFFFu) == 0x7F800000u;
  if (tid == 0) {
    T.special = (s_nan || s == 0.0f) ? 1 : (s_inf ? 2 : 0);
    const float pmin = round_storage<DT>(exp2_int(qmin));
    T.yinf = (pmin == 0.0f) ? Tr<DT>::QNAN : Tr<DT>::INF;
    T.X[nlev] = PO2_NEVER;
  }
  const bool special = s_nan || s_inf || s == 0.0f;
  const uint32_t s_pat = Tr<DT>::pat(s);
  for (int j = tid; j < nlev; j += nthr) {
    const int k = qmin + j;
    uint32_t X;
    if (j == 0 || special || k < PO2_KMIN) X = 0;
    else if (k > PO2_KMAX) X = PO2_NEVER;
    else {
      const uint32_t b = (have_pre && j == tid) ? pre_b : PO2_BOUNDS[flavor][DT][mode][k - PO2_KMIN];
      X = (b == PO2_NEVER) ? PO2_NEVER : search_threshold<DT>(__uint_as_float(b), s, s_pat);
    }
    T.X[j] = X;
    // utils/quantizers.py:31-32: (2**q * sign) * scale, each product rounded to the storage type
    const float p = round_storage<DT>(exp2_int(k));
    T.Y[j] = special ? 0u : (Tr<DT>::pat(__fmul_rn(p, s)) & Tr<DT>::MAG);
  }
  __syncthreads();
  for (int ex = tid; ex < Tr<DT>::NBIN; ex += nthr) {
    const uint32_t lo = (uint32_t)ex << Tr<DT>::MB;
    const uint32_t hi = lo + (1u << Tr<DT>::MB);
    int cnt = 0, inside = 0;
    for (int j = 1; j < nlev; ++j) {
      const uint32_t X = T.X[j];
      cnt += (X < lo);
      inside += (X >= lo && X < hi);
    }
    // Fast path in this binade: y = Y[cnt] + ((a >= X[cnt+1]) << MB).  That is exact when there is
    // at most one threshold inside and stepping one level up doubles the output pattern exactly.
    // Binade 0 (zeros and subnormal inputs) always takes the slow path, which also owns the
    // sign(0) == 0 rule, so the fast path never tests for zero.
    const uint32_t ylo = T.Y[cnt];
    bool regular = (ex != 0) && inside <= 1;
    if (inside == 1) regular = regular && (cnt + 1 < nlev) && (T.Y[cnt + 1] == ylo + (1u << Tr<DT>::MB));
    T.bt[ex] = make_uint2(T.X[cnt + 1], ylo | (regular ? 0u : PO2_IRR));
    T.cb[ex] = (uint8_t)cnt;
  }
  __syncthreads();
}

struct Acc {                  // per-thread side outputs
  uint32_t zeros;
  float sse;
};

// One element, exact general path: storage pattern in, storage pattern out; `code` gets
// sign<<(bits-1) | magnitude.
template <int DT>
__device__ __forceinline__ uint32_t quant_one(uint32_t u, const LevelTab& T, int nlev_m1,
                                           int sign_shift, uint32_t& code, Acc& acc,
                                           bool want_sse) {
  const uint32_t a = u & Tr<DT>::MAG;
  uint32_t j = T.cb[a >> Tr<DT>::MB];
  while (a >= T.X[j + 1]) ++j;
  const uint32_t yb = T.Y[j];
  const bool nz = (a != 0);
  const uint32_t sg = nz ? (u & Tr<DT>::SGN) : 0u;      // torch.sign(+-0) == 0 -> y = +0
  const uint32_t out = nz ? (yb | sg) : 0u;
  code = (uint32_t)(nlev_m1 - (int)j) | ((sg ? 1u : 0u) << sign_shift);
  acc.zeros += nz ? 0u : 1u;
  if (want_sse) {
    const float d = Tr<DT>::val(out) - Tr<DT>::val(u);
    acc.sse = fmaf(d, d, acc.sse);
  }
  return out;
}

// One element, fast path (regular binades): mask, shift, one 64-bit shared load, compare, add,
// sign merge.  `irr` collects the irregular flag; the caller redoes the vector if it is set.
template <int DT, bool CODES>
__device__ __forceinline__ uint32_t quant_fast(uint32_t u, const LevelTab& T, uint32_t& irr,
                                               int nlev_m1, int sign_shift, uint32_t& code) {
  const uint32_t a = u & Tr<DT>::MAG;
  const uint32_t ex = a >> Tr<DT>::MB;
  const uint2 e = T.bt[ex];
  const uint32_t up = (a >= e.x) ? 1u : 0u;
  const uint32_t t = e.y + (up << Tr<DT>::MB);
  irr |= e.y;
  if (CODES) code = (uint32_t)(nlev_m1 - (int)T.cb[ex] - (int)up) | (((u & Tr<DT>::SGN) ? 1u : 0u) << sign_shift);
  return (t & Tr<DT>::MAG) | (u & Tr<DT>::SGN);
}

// Non-finite / zero scale: the reference's float pipeline evaluated literally.
template <int DT>
__device__ __forceinline__ uint32_t quant_special(uint32_t u, const LevelTab& T, int nlev_m1,
                                                  int sign_shift, uint32_t& code) {
  const uint32_t a = u & Tr<DT>::MAG;
  const uint32_t sg = u & Tr<DT>::SGN;
  code = (uint32_t)nlev_m1 | ((sg && a) ? (1u << sign_shift) : 0u);
  if (T.special == 1) return Tr<DT>::QNAN;               // x/NaN, 0/0
  if (a == 0 || a >= Tr<DT>::INF) return Tr<DT>::QNAN;   // 0*Inf, Inf/Inf
  return T.yinf == Tr<DT>::QNAN ? Tr<DT>::QNAN : (T.yinf | sg);
}

template <int DT>
__device__ __forceinline__ uint32_t load_pat(const void* x, int64_t i) {
  if (DT == PO2_F32) return reinterpret_cast<const uint32_t*>(x)[i];
  return reinterpret_cast<const unsigned short*>(x)[i];
}
template <int DT>
__device__ __forceinline__ void store_pat(void* y, int64_t i, uint32_t p) {
  if (DT == PO2_F32) reinterpret_cast<uint32_t*>(y)[i] = p;
  else reinterpret_cast<unsigned short*>(y)[i] = (unsigned short)p;
}

// Elements 2*ip and 2*ip+1 (one code byte at bits<=4), scalar accesses: tails, unaligned
// tensors and the special-scale path.
template <int DT>
__device__ void quant_pair(const void* x, void* y, uint8_t* codes, int64_t ip, int64_t n,
                           const LevelTab& T, int bits, Acc& acc, bool want_sse) {
  const int nlev_m1 = (1 << (bits - 1)) - 1, sshift = bits - 1;
  uint32_t c[2] = {0, 0};
  for (int h = 0; h < 2; ++h) {
    const int64_t i = 2 * ip + h;
    if (i >= n) break;
    const uint32_t u = load_pat<DT>(x, i);
    const uint32_t o = T.special ? quant_special<DT>(u, T, nlev_m1, sshift, c[h])
                                 : quant_one<DT>(u, T, nlev_m1, sshift, c[h], acc, want_sse);
    store_pat<DT>(y, i, o);
  }
  if (codes) {
    if (bits <= 4) codes[ip] = (uint8_t)(c[0] | (c[1] << 4));
    else {
      codes[2 * ip] = (uint8_t)c[0];
      if (2 * ip + 1 < n) codes[2 * ip + 1] = (uint8_t)c[1];
    }
  }
}

// codes travel as one byte per element in a register pair (element i in byte i)
template <int DT>
__device__ __forceinline__ void store_codes(uint8_t* codes, int64_t iv, bool codes4, uint2 cb) {
  if (codes4) {                                          // squeeze bytes to nibbles
    uint32_t a = cb.x | (cb.x >> 4);                     // bytes 0,2 now hold nibble pairs (0,1),(2,3)
    a = (a & 0xFFu) | ((a >> 8) & 0xFF00u);
    if (DT == PO2_F32) { reinterpret_cast<unsigned short*>(codes)[iv] = (unsigned short)a; return; }
    uint32_t b = cb.y | (cb.y >> 4);
    b = (b & 0xFFu) | ((b >> 8) & 0xFF00u);
    reinterpret_cast<uint32_t*>(codes)[iv] = a | (b << 16);
  } else if (DT == PO2_F32) {
    reinterpret_cast<uint32_t*>(codes)[iv] = cb.x;
  } else {
    reinterpret_cast<uint2*>(codes)[iv] = cb;
  }
}

struct SlowOut { uint4 o; uint2 cb; uint32_t zeros; float sse; };

// exact general path for a whole vector (rare: zeros, subnormals, irregular binades); everything
// is passed and returned by value so the hot loop keeps its vectors in registers
template <int DT>
__device__ __noinline__ SlowOut quant_vec_slow(uint4 v, const LevelTab* Tp, int nlev_m1, int sshift,
                                               bool want_sse) {
  const LevelTab& T = *Tp;
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint32_t ow[4], c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  Acc acc{0u, 0.0f};
  if (DT == PO2_F32) {
#pragma unroll
    for (int i = 0; i < 4; ++i) ow[i] = quant_one<DT>(w[i], T, nlev_m1, sshift, c[i], acc, want_sse);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t lo = quant_one<DT>(w[i] & 0xFFFFu, T, nlev_m1, sshift, c[2 * i], acc, want_sse);
      const uint32_t hi = quant_one<DT>(w[i] >> 16, T, nlev_m1, sshift, c[2 * i + 1], acc, want_sse);
      ow[i] = lo | (hi << 16);
    }
  }
  SlowOut r;
  r.o = make_uint4(ow[0], ow[1], ow[2], ow[3]);
  r.cb = make_uint2(c[0] | (c[1] << 8) | (c[2] << 16) | (c[3] << 24), c[4] | (c[5] << 8) | (c[6] << 16) | (c[7] << 24));
  r.zeros = acc.zeros;
  r.sse = acc.sse;
  return r;
}

// One 16-byte vector (EPV elements) in registers -> quantized vector (+ packed codes, + SSE).
template <int DT, bool CODES, bool SSE>
__device__ __forceinline__ uint4 quant_vec_t(const uint4& v, const LevelTab& T, int nlev_m1, int sshift,
                                             bool codes4, uint8_t* codes, int64_t iv, Acc& acc) {
  constexpr bool want_sse = SSE;
  const uint32_t w[4] = {v.x, v.y, v.z, v.w};
  uint32_t ow[4], irr = 0;
  uint2 cb = make_uint2(0u, 0u);
  if (DT == PO2_F32) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint32_t c = 0;
      ow[i] = quant_fast<DT, CODES>(w[i], T, irr, nlev_m1, sshift, c);
      if (CODES) cb.x |= c << (8 * i);
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint32_t c0 = 0, c1 = 0;
      const uint32_t lo = quant_fast<DT, CODES>(w[i] & 0xFFFFu, T, irr, nlev_m1, sshift, c0);
      const uint32_t hi = quant_fast<DT, CODES>(w[i] >> 16, T, irr, nlev_m1, sshift, c1);
      ow[i] = lo | (hi << 16);
      if (CODES) {
        const uint32_t cc = (c0 | (c1 << 8)) << (16 * (i & 1));
        if (i < 2) cb.x |= cc; else cb.y |= cc;
      }
    }
  }
  uint4 o = make_uint4(ow[0], ow[1], ow[2], ow[3]);
  if (irr & PO2_IRR) {
    const SlowOut r = quant_vec_slow<DT>(v, &T, nlev_m1, sshift, want_sse);
    o = r.o; cb = r.cb;
    acc.zeros += r.zeros; acc.sse += r.sse;
  } else if (want_sse) {
    if (DT == PO2_F32) {
#pragma unroll
      for (int i = 0; i < 4; ++i) { const float d = __uint_as_float(ow[i]) - __uint_as_float(w[i]); acc.sse = fmaf(d, d, acc.sse); }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float d0 = Tr<DT>::val(ow[i] & 0xFFFFu) - Tr<DT>::val(w[i] & 0xFFFFu);
        const float d1 = Tr<DT>::val(ow[i] >> 16) - Tr<DT>::val(w[i] >> 16);
        acc.sse = fmaf(d0, d0, acc.sse); acc.sse = fmaf(d1, d1, acc.sse);
      }
    }
  }
  if (CODES) store_codes<DT>(codes, iv, codes4, cb);
  return o;
}

template <int DT> __device__ __forceinline__ uint32_t vec_absmax(const uint4& v, uint32_t m) {
  if (DT == PO2_F32) {
    m = max(m, v.x & 0x7FFFFFFFu); m = max(m, v.y & 0x7FFFFFFFu);
    m = max(m, v.z & 0x7FFFFFFFu); m = max(m, v.w & 0x7FFFFFFFu);
    return m;
  }
  // two 15-bit magnitudes per word, kept as a packed pair
  m = __vmaxu2(m, v.x & 0x7FFF7FFFu); m = __vmaxu2(m, v.y & 0x7FFF7FFFu);
  m = __vmaxu2(m, v.z & 0x7FFF7FFFu); m = __vmaxu2(m, v.w & 0x7FFF7FFFu);
  return m;
}
template <int DT> __device__ __forceinline__ uint32_t absmax_finish(uint32_t m) {
  return (DT == PO2_F32) ? m : max(m & 0xFFFFu, m >> 16);
}

__device__ __forceinline__ uint32_t block_max_u32(uint32_t m, uint32_t* sm /*32 words*/) {
  m = warp_max_u32(m);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  if (lane == 0) sm[wid] = m;
  __syncthreads();
  if (wid == 0) {
    uint32_t t = (lane < nw) ? sm[lane] : 0u;
    t = warp_max_u32(t);
    if (lane == 0) sm[0] = t;
  }
  __syncthreads();
  const uint32_t r = sm[0];
  __syncthreads();
  return r;
}

__device__ void flush_acc(const Acc& acc, unsigned int* zero_count, double* sse, float* sm) {
  // zero counter: almost always 0 -> one ballot per warp, no atomics
  uint32_t z = acc.zeros;
  for (int o = 16; o; o >>= 1) z += __shfl_xor_sync(0xFFFFFFFFu, z, o);
  if (zero_count && z && (threadIdx.x & 31) == 0) atomicAdd(zero_count, z);
  if (sse) {
    float v = acc.sse;
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    __syncthreads();
    if (lane == 0) sm[wid] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int i = 0; i < nw; ++i) t += (double)sm[i];
      atomicAdd(sse, t);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// pass 1: scale = max|x|
// ------------------------------------------------------------------------------------------------
template <int DT>
__global__ void __launch_bounds__(256) absmax_kernel(const void* __restrict__ x, int64_t n,
                                                     float* __restrict__ scale_out,
                                                     Workspace* __restrict__ ws) {
  __shared__ uint32_t sm[32];
  constexpr int EB = Tr<DT>::EB, EPV = Tr<DT>::EPV;
  const uintptr_t addr = reinterpret_cast<uintptr_t>(x);
  int64_t head = (int64_t)(((16 - (addr & 15)) & 15) / EB);
  if (head > n) head = n;
  const uint4* xv = reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(x) + head * EB);
  const int64_t n_vec = (n - head) / EPV;
  const int64_t tail0 = head + n_vec * EPV;
  uint32_t m = 0;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  for (; i + 3 * stride < n_vec; i += 4 * stride) {      // 4 independent 128-bit loads in flight
    const uint4 a = ldg_keep(xv + i), b = ldg_keep(xv + i + stride);
    const uint4 c = ldg_keep(xv + i + 2 * stride), d = ldg_keep(xv + i + 3 * stride);
    m = vec_absmax<DT>(a, m); m = vec_absmax<DT>(b, m);
    m = vec_absmax<DT>(c, m); m = vec_absmax<DT>(d, m);
  }
  for (; i < n_vec; i += stride) m = vec_absmax<DT>(ldg_keep(xv + i), m);
  m = absmax_finish<DT>(m);
  if (blockIdx.x == 0) {
    for (int64_t k = threadIdx.x; k < head; k += blockDim.x) m = max(m, load_pat<DT>(x, k) & Tr<DT>::MAG);
    for (int64_t k = tail0 + threadIdx.x; k < n; k += blockDim.x) m = max(m, load_pat<DT>(x, k) & Tr<DT>::MAG);
  }
  m = block_max_u32(m, sm);
  if (threadIdx.x == 0) {
    atomicMax(&ws->absmax, m);
    __threadfence();
    const unsigned int t = atomicAdd(&ws->arrive, 1u);
    if (t == gridDim.x - 1) {                            // last CTA: publish and re-zero
      __threadfence();
      const uint32_t v = atomicExch(&ws->absmax, 0u);
      ws->arrive = 0u;
      *scale_out = Tr<DT>::val(v);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// pass 2: quantize / dequantize / code emit
// ------------------------------------------------------------------------------------------------
#ifndef PO2_Q_UNROLL
#define PO2_Q_UNROLL 4
#endif
#ifndef PO2_Q_MINBLOCKS
#define PO2_Q_MINBLOCKS 1
#endif
#ifndef PO2_Q_CTAS_PER_SM
#define PO2_Q_CTAS_PER_SM 16
#endif

template <int DT, bool CODES, bool SSE>
__global__ void __launch_bounds__(256, PO2_Q_MINBLOCKS) quantize_kernel(const uint4* __restrict__ x,
                                                       uint4* __restrict__ y, uint8_t* codes,
                                                       unsigned int* zero_count, double* sse,
                                                       const float* __restrict__ scale, int64_t n,
                                                       int bits, int fsr, int mode, int flavor,
                                                       int reverse) {
  __shared__ LevelTab T;
  __shared__ float smf[32];
  constexpr int EPV = Tr<DT>::EPV;
  build_levels<DT>(T, *scale, bits, fsr, mode, flavor);
  const int nlev_m1 = (1 << (bits - 1)) - 1, sshift = bits - 1;
  const bool codes4 = bits <= 4;
  constexpr bool want_sse = SSE;
  const int64_t n_vec = n / EPV;
  Acc acc{0u, 0.0f};
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
#define QV(v, iv) quant_vec_t<DT, CODES, SSE>(v, T, nlev_m1, sshift, codes4, codes, iv, acc)
  if (!T.special) {
    // the absmax pass left the END of x in L2 last; walking backwards re-reads it from there
    const int64_t last = n_vec - 1;
    constexpr int U = PO2_Q_UNROLL;                       // independent 128-bit loads in flight per thread
    for (; i + (U - 1) * stride < n_vec; i += U * stride) {
      uint4 v[U];
      int64_t idx[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        idx[u] = reverse ? last - (i + u * stride) : i + u * stride;
        v[u] = ldg_stream(x + idx[u]);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) stg_stream(y + idx[u], QV(v[u], idx[u]));
    }
    for (; i < n_vec; i += stride) {
      const int64_t i0 = reverse ? last - i : i;
      stg_stream(y + i0, QV(ldg_stream(x + i0), i0));
    }
    if (blockIdx.x == 0 && threadIdx.x < EPV / 2) {
      const int64_t ip = n_vec * (EPV / 2) + threadIdx.x;
      if (2 * ip < n) quant_pair<DT>(x, y, codes, ip, n, T, bits, acc, want_sse);
    }
  } else {
    const int64_t n_pair = (n + 1) / 2;
    for (; i < n_pair; i += stride) quant_pair<DT>(x, y, codes, i, n, T, bits, acc, false);
  }
#undef QV
  flush_acc(acc, zero_count, sse, smf);
}

// any alignment: scalar accesses, two elements per thread
template <int DT>
__global__ void __launch_bounds__(256) quantize_scalar_kernel(const void* __restrict__ x,
                                                              void* __restrict__ y, uint8_t* codes,
                                                              unsigned int* zero_count, double* sse,
                                                              const float* __restrict__ scale,
                                                              int64_t n, int bits, int fsr, int mode,
                                                              int flavor) {
  __shared__ LevelTab T;
  __shared__ float smf[32];
  build_levels<DT>(T, *scale, bits, fsr, mode, flavor);
  Acc acc{0u, 0.0f};
  const int64_t n_pair = (n + 1) / 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_pair; i += stride)
    quant_pair<DT>(x, y, codes, i, n, T, bits, acc, sse != nullptr && !T.special);
  flush_acc(acc, zero_count, sse, smf);
}

// ------------------------------------------------------------------------------------------------
// fused: absmax + quantize with x held in registers across the (grid-wide) max reduction.
// Launched cooperatively when gridDim.x > 1 (all CTAs co-resident), plainly when it is 1.
// ------------------------------------------------------------------------------------------------
// Emit 4 consecutive quantized fp32 weights (element indices e0..e0+3 of a (K, C, R, S) tensor) into
// the conv's B-operand layout as exact bf16 +-2^q (= y / scale).
__device__ __forceinline__ void pack_vec(const PackArgs& pk, const uint4& o, int e0, float s) {
  const uint32_t ob[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int e = e0 + j;
    const int k = fdiv(e, pk.div_ct);
    const int rem = e - k * pk.C * pk.taps;
    const int c = fdiv(rem, pk.div_t);
    const int tap = rem - c * pk.taps;
    const float yv = __uint_as_float(ob[j]);
    pack_store(pk, k, c, tap, (s == 1.0f) ? yv : __fdiv_rn(yv, s));
  }
}

constexpr int FUSED_THREADS = 512;
constexpr int FUSED_R = 8;    // 16-byte vectors held per thread

template <int DT, bool CODES, bool SSE>
__device__ __forceinline__ void fused_body(const uint4* __restrict__ x,
                                                              uint4* __restrict__ y, uint8_t* codes,
                                                              unsigned int* zero_count, double* sse,
                                                              float* __restrict__ scale_out,
                                                              int64_t n, int bits, int fsr, int mode,
                                                              int flavor, Workspace* ws, int cluster,
                                                              const PackArgs& pk, const uint32_t lgrid,
                                                              const uint32_t lblock) {
  // lgrid / lblock: number and index of the CTAs working on THIS tensor (the whole grid for the
  // single-tensor kernel, one cluster for the multi-tensor kernel)
  __shared__ LevelTab T;
  __shared__ uint32_t sm[32];
  __shared__ float smf[32];
  __shared__ uint32_t cl_max;                            // this CTA's max, read by its cluster peers
  constexpr int EPV = Tr<DT>::EPV;
  const int64_t n_vec = n / EPV;
  const int64_t total = (int64_t)lgrid * blockDim.x;
  const int64_t gtid = (int64_t)lblock * blockDim.x + threadIdx.x;
  const uint32_t pre_b = prefetch_bound(DT, bits, fsr, mode, flavor);   // in flight together with the data
  uint4 v[FUSED_R];
  uint32_t m = 0;
#pragma unroll
  for (int r = 0; r < FUSED_R; ++r) {
    const int64_t i = gtid + r * total;
    v[r] = (i < n_vec) ? ldg_stream(x + i) : make_uint4(0, 0, 0, 0);
  }
#pragma unroll
  for (int r = 0; r < FUSED_R; ++r) m = vec_absmax<DT>(v[r], m);
  m = absmax_finish<DT>(m);
  if (lblock == 0)
    for (int64_t k = n_vec * EPV + threadIdx.x; k < n; k += blockDim.x)
      m = max(m, load_pat<DT>(x, k) & Tr<DT>::MAG);
  m = block_max_u32(m, sm);
  if (lgrid > 1 && cluster) {
    // the whole grid is one thread-block cluster: exchange the per-CTA maxima through distributed
    // shared memory (two cluster barriers) instead of global atomics and a spin
    if (threadIdx.x == 0) cl_max = m;
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    uint32_t mm = 0;
    const uint32_t laddr = (uint32_t)__cvta_generic_to_shared(&cl_max);
    for (uint32_t r = 0; r < lgrid; ++r) {
      uint32_t raddr, val;
      asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(raddr) : "r"(laddr), "r"(r));
      asm volatile("ld.shared::cluster.u32 %0, [%1];" : "=r"(val) : "r"(raddr) : "memory");
      mm = max(mm, val);
    }
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
    m = mm;
  } else if (lgrid > 1) {
    if (threadIdx.x == 0) {
      atomicMax(&ws->absmax, m);
      __threadfence();
      atomicAdd(&ws->arrive, 1u);
      while (*reinterpret_cast<volatile unsigned int*>(&ws->arrive) < lgrid) __nanosleep(20);
      __threadfence();
      sm[0] = *reinterpret_cast<volatile unsigned int*>(&ws->absmax);
      const unsigned int d = atomicAdd(&ws->depart, 1u);
      if (d == lgrid - 1) {                          // everyone has read it: re-zero
        ws->absmax = 0u; ws->arrive = 0u; ws->depart = 0u;
      }
    }
    __syncthreads();
    m = sm[0];
  }
  const float s = Tr<DT>::val(m);
  if (gtid == 0) *scale_out = s;
  build_levels<DT>(T, s, bits, fsr, mode, flavor, true, pre_b);
  const int nlev_m1 = (1 << (bits - 1)) - 1, sshift = bits - 1;
  const bool codes4 = bits <= 4;
  constexpr bool want_sse = SSE;
  Acc acc{0u, 0.0f};
  if (!T.special) {
#pragma unroll
    for (int r = 0; r < FUSED_R; ++r) {
      const int64_t i = gtid + r * total;
      if (i < n_vec) {
        const uint4 o = quant_vec_t<DT, CODES, SSE>(v[r], T, nlev_m1, sshift, codes4, codes, i, acc);
        stg_stream(y + i, o);
        if (DT == PO2_F32 && pk.Bp) pack_vec(pk, o, (int)i * 4, s);
      }
    }
    if (lblock == 0 && threadIdx.x < EPV / 2) {
      const int64_t ip = n_vec * (EPV / 2) + threadIdx.x;
      if (2 * ip < n) quant_pair<DT>(x, y, codes, ip, n, T, bits, acc, want_sse);
    }
  } else {
    const int64_t n_pair = (n + 1) / 2;
    for (int64_t i = gtid; i < n_pair; i += total) quant_pair<DT>(x, y, codes, i, n, T, bits, acc, false);
    if (DT == PO2_F32 && pk.Bp)                             // NaN / Inf weights: the operand is NaN, like y
      for (int64_t i = gtid; i < n_vec; i += total)
        pack_vec(pk, make_uint4(0x7FC00000u, 0x7FC00000u, 0x7FC00000u, 0x7FC00000u), (int)i * 4, 1.0f);
  }
  flush_acc(acc, zero_count, sse, smf);
}

template <int DT, bool CODES, bool SSE>
__global__ void __launch_bounds__(FUSED_THREADS) fused_kernel(const uint4* __restrict__ x,
                                                              uint4* __restrict__ y, uint8_t* codes,
                                                              unsigned int* zero_count, double* sse,
                                                              float* __restrict__ scale_out,
                                                              int64_t n, int bits, int fsr, int mode,
                                                              int flavor, Workspace* ws, int cluster,
                                                              PackArgs pk) {
  // a kernel launched behind us with programmatic stream serialization (the conv that consumes the
  // packed operand) may start its prologue now; it executes griddepcontrol.wait before reading Bp
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  fused_body<DT, CODES, SSE>(x, y, codes, zero_count, sse, scale_out, n, bits, fsr, mode, flavor, ws, cluster, pk,
                             gridDim.x, blockIdx.x);
}

// Multi-tensor form (SURVEY.md section 8f "next" #4): ONE launch quantizes (and packs) many weight
// tensors, one thread-block cluster per tensor.  Per-tensor arguments come from a device table.
__global__ void __launch_bounds__(FUSED_THREADS) multi_fused_kernel(const MultiDesc* __restrict__ descs, int csize) {
  const uint32_t t = blockIdx.x / (uint32_t)csize, lblock = blockIdx.x % (uint32_t)csize;
  const MultiDesc d = descs[t];
  // The squared quantization error of every tensor comes out of the same pass (x and y are both in
  // registers): this is what QuantizedConv2d.get_quantization_error / the models' error walkers
  // (train.py:106) read, so they cost no launch of their own.  The CTAs of the cluster add their shares
  // atomically; CTA 0 clears the slot first, ordered before the adds by the cluster barriers of the max
  // exchange (csize > 1) or by program order (csize == 1: the same thread clears and adds).
  if (d.sse_out && lblock == 0 && threadIdx.x == 0) { *d.sse_out = 0.0; __threadfence(); }
  if (d.sse_out)
    fused_body<PO2_F32, false, true>(d.x, d.y, nullptr, nullptr, d.sse_out, d.scale_out, d.n, d.bits, d.fsr, d.mode,
                                     d.flavor, nullptr, 1, d.pk, (uint32_t)csize, lblock);
  else
    fused_body<PO2_F32, false, false>(d.x, d.y, nullptr, nullptr, nullptr, d.scale_out, d.n, d.bits, d.fsr, d.mode,
                                      d.flavor, nullptr, 1, d.pk, (uint32_t)csize, lblock);
}


// ------------------------------------------------------------------------------------------------
// codes -> values
// ------------------------------------------------------------------------------------------------
template <int DT>
__global__ void __launch_bounds__(256) dequantize_kernel(const uint8_t* __restrict__ codes,
                                                         const float* __restrict__ scale,
                                                         void* __restrict__ y, int64_t n, int bits,
                                                         int fsr) {
  __shared__ uint32_t Y[128];
  const int nlev = 1 << (bits - 1), qmin = fsr - nlev;
  const float s = *scale;
  for (int j = threadIdx.x; j < nlev; j += blockDim.x) {
    const float p = round_storage<DT>(exp2_int(qmin + j));
    Y[j] = Tr<DT>::pat(__fmul_rn(p, s));                 // NaN/Inf scales propagate as in torch
  }
  __syncthreads();
  const int64_t n_pair = (n + 1) / 2;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t ip = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; ip < n_pair; ip += stride) {
    uint32_t c0, c1;
    if (bits <= 4) { const uint32_t b = codes[ip]; c0 = b & 0xF; c1 = b >> 4; }
    else { c0 = codes[2 * ip]; c1 = (2 * ip + 1 < n) ? codes[2 * ip + 1] : 0; }
    const uint32_t c[2] = {c0, c1};
    for (int h = 0; h < 2; ++h) {
      const int64_t i = 2 * ip + h;
      if (i >= n) break;
      const uint32_t mag = c[h] & (uint32_t)(nlev - 1);
      const uint32_t neg = (c[h] >> (bits - 1)) & 1u;
      store_pat<DT>(y, i, Y[nlev - 1 - mag] ^ (neg ? Tr<DT>::SGN : 0u));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// straight-through estimator backward (utils/quantizers.py:34-36): gx = g, or gx += g
// ------------------------------------------------------------------------------------------------
template <int DT> __device__ __forceinline__ uint32_t add_pat(uint32_t a, uint32_t b) {
  return Tr<DT>::pat(Tr<DT>::val(a) + Tr<DT>::val(b));
}
template <int DT>
__global__ void __launch_bounds__(256) ste_backward_kernel(const void* __restrict__ g, void* gx,
                                                           int64_t n, int accumulate, int vec_ok) {
  constexpr int EPV = Tr<DT>::EPV;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t n_vec = vec_ok ? n / EPV : 0;
  const uint4* gv = reinterpret_cast<const uint4*>(g);
  uint4* xv = reinterpret_cast<uint4*>(gx);
  for (int64_t i = t0; i < n_vec; i += stride) {
    uint4 a = ldg_stream(gv + i);
    if (accumulate) {
      const uint4 b = xv[i];
      if (DT == PO2_F32) {
        a.x = add_pat<DT>(a.x, b.x); a.y = add_pat<DT>(a.y, b.y);
        a.z = add_pat<DT>(a.z, b.z); a.w = add_pat<DT>(a.w, b.w);
      } else {
        uint32_t aw[4] = {a.x, a.y, a.z, a.w};
        const uint32_t bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int k = 0; k < 4; ++k)
          aw[k] = add_pat<DT>(aw[k] & 0xFFFFu, bw[k] & 0xFFFFu) | (add_pat<DT>(aw[k] >> 16, bw[k] >> 16) << 16);
        a = make_uint4(aw[0], aw[1], aw[2], aw[3]);
      }
    }
    xv[i] = a;
  }
  for (int64_t i = n_vec * EPV + t0; i < n; i += stride) {
    uint32_t a = load_pat<DT>(g, i);
    if (accumulate) a = add_pat<DT>(a, load_pat<DT>(gx, i));
    store_pat<DT>(gx, i, a);
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct DevInfo { int sms; int fused_blocks_per_sm[3]; };
static DevInfo g_dev[PO2_MAX_DEVICES];
static PerDeviceOnce g_dev_once;

template <int DT> static int fused_occupancy() {
  int nb = 0;
  int a = 0, b = 0;
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, fused_kernel<DT, false, false>, FUSED_THREADS, 0);
  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, fused_kernel<DT, true, true>, FUSED_THREADS, 0);
  nb = a < b ? a : b;
  return nb;
}

static const DevInfo* dev_info() {
  const int d = current_device();
  if (d < 0) return nullptr;
  const cudaError_t e = g_dev_once.run([&]() -> cudaError_t {
    DevInfo& I = g_dev[d];
    int sms = 0;
    const cudaError_t q = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, d);
    if (q != cudaSuccess) return q;
    I.sms = sms;
    I.fused_blocks_per_sm[0] = fused_occupancy<PO2_F32>();
    I.fused_blocks_per_sm[1] = fused_occupancy<PO2_BF16>();
    I.fused_blocks_per_sm[2] = fused_occupancy<PO2_F16>();
    return cudaSuccess;
  });
  return e == cudaSuccess ? &g_dev[d] : nullptr;
}

int device_sm_count() {
  const DevInfo* I = dev_info();
  return (I && I->sms > 0) ? I->sms : 148;
}

static inline int elem_bytes(int dtype) { return dtype == PO2_F32 ? 4 : 2; }
static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

static int check_common(int64_t n, int dtype) {
  if (dtype != PO2_F32 && dtype != PO2_BF16 && dtype != PO2_F16) return PO2_E_DTYPE;
  if (n <= 0) return PO2_E_SIZE;
  return 0;
}
static int check_quant(int bits, int fsr, int mode, int flavor) {
  if (bits < 2 || bits > 8) return PO2_E_BITS;
  if (fsr < -64 || fsr > 64) return PO2_E_BITS;
  if (mode != PO2_MODE_PO2 && mode != PO2_MODE_PO2_PLUS) return PO2_E_MODE;
  if (flavor < 0 || flavor >= PO2_NUM_FLAVORS) return PO2_E_FLAVOR;
  return 0;
}

int check_quant_args(int bits, int fsr, int mode, int flavor) {
  if (flavor == PO2_FLAVOR_TORCH_CUDA && !po2_have_torch_cuda_table()) return PO2_E_FLAVOR;
  return check_quant(bits, fsr, mode, flavor);
}

static int grid_for(int64_t work_items, int threads, int per_thread, int max_blocks) {
  int64_t b = (work_items + (int64_t)threads * per_thread - 1) / ((int64_t)threads * per_thread);
  if (b < 1) b = 1;
  if (b > max_blocks) b = max_blocks;
  return (int)b;
}

// compile-time (CODES, SSE) variants selected from the optional pointers
#define PO2_VARIANT(codes, sse, ...)                                                   \
  if (codes) { if (sse) { constexpr bool CODES = true, SSE = true; __VA_ARGS__; }      \
               else { constexpr bool CODES = true, SSE = false; __VA_ARGS__; } }       \
  else { if (sse) { constexpr bool CODES = false, SSE = true; __VA_ARGS__; }           \
         else { constexpr bool CODES = false, SSE = false; __VA_ARGS__; } }

#define PO2_DISPATCH(dtype, ...)                                        \
  switch (dtype) {                                                      \
    case PO2_F32: { constexpr int DT = PO2_F32; __VA_ARGS__; } break;   \
    case PO2_BF16: { constexpr int DT = PO2_BF16; __VA_ARGS__; } break; \
    default: { constexpr int DT = PO2_F16; __VA_ARGS__; } break;        \
  }

static int launch_absmax(const void* x, int64_t n, int dtype, float* scale_out, void* workspace,
                         cudaStream_t st) {
  const DevInfo* I = dev_info();
  if (!I) return (int)cudaErrorInvalidDevice;
  const int epv = 16 / elem_bytes(dtype);
  const int blocks = grid_for(n / epv + 1, 256, 4, I->sms * 8);
  PO2_DISPATCH(dtype, absmax_kernel<DT><<<blocks, 256, 0, st>>>(x, n, scale_out, (Workspace*)workspace));
  return (int)cudaGetLastError();
}

static int launch_quantize(const void* x, void* y, void* codes, unsigned int* zc, double* sse,
                           const float* scale, int64_t n, int dtype, int bits, int fsr, int mode,
                           int flavor, int reverse, cudaStream_t st) {
  const DevInfo* I = dev_info();
  if (!I) return (int)cudaErrorInvalidDevice;
  const int epv = 16 / elem_bytes(dtype);
  const bool codes_ok = !codes || aligned16(codes);
  if (aligned16(x) && aligned16(y) && codes_ok) {
    const int blocks = grid_for(n / epv + 1, 256, PO2_Q_UNROLL, I->sms * PO2_Q_CTAS_PER_SM);
    PO2_DISPATCH(dtype, PO2_VARIANT(codes, sse, quantize_kernel<DT, CODES, SSE><<<blocks, 256, 0, st>>>(
        (const uint4*)x, (uint4*)y, (uint8_t*)codes, zc, sse, scale, n, bits, fsr, mode, flavor, reverse)));
  } else {
    const int blocks = grid_for((n + 1) / 2, 256, 4, I->sms * 8);
    PO2_DISPATCH(dtype, quantize_scalar_kernel<DT><<<blocks, 256, 0, st>>>(
        x, y, (uint8_t*)codes, zc, sse, scale, n, bits, fsr, mode, flavor));
  }
  return (int)cudaGetLastError();
}

// fp32 weights -> y, scale and the conv's packed operand in one launch (see PackArgs)
int fused_quantize_pack(const void* w, void* y, float* scale_out, int64_t n, int bits, int fsr, int mode,
                        int flavor, void* workspace, const PackArgs& pk_in, cudaStream_t st) {
  if (int e = check_common(n, PO2_F32)) return e;
  if (int e = check_quant(bits, fsr, mode, flavor)) return e;
  if (!w || !y || !scale_out || !pk_in.Bp) return PO2_E_NULL;
  if (!workspace) return PO2_E_WORKSPACE;
  if (n % 4 || !aligned16(w) || !aligned16(y) || n >= (1ll << 31)) return PO2_E_UNSUPPORTED;
  const DevInfo* I = dev_info();
  if (!I) return (int)cudaErrorInvalidDevice;
  const int64_t n_vec = n / 4;
  const int64_t per_block = (int64_t)FUSED_THREADS * FUSED_R;
  const int64_t max_blocks = (int64_t)I->sms * I->fused_blocks_per_sm[PO2_F32];
  if (max_blocks <= 0 || n_vec > max_blocks * per_block) return PO2_E_UNSUPPORTED;
  int64_t blocks = (n_vec + FUSED_THREADS - 1) / FUSED_THREADS;
  int cluster = 0;
  if (n_vec <= per_block) blocks = 1;
  else if (n_vec <= 8 * per_block) { if (blocks > 8) blocks = 8; cluster = 1; }
  else if (blocks > max_blocks) blocks = max_blocks;
  Workspace* ws = (Workspace*)workspace;
  const uint4* xv = (const uint4*)w; uint4* yv = (uint4*)y; uint8_t* cp = nullptr;
  unsigned int* zc = nullptr; double* sse = nullptr;
  PackArgs pk = pk_in;
  void* args[] = {&xv, &yv, &cp, &zc, &sse, &scale_out, &n, &bits, &fsr, &mode, &flavor, &ws, &cluster, &pk};
  cudaError_t err;
  if (blocks == 1) {
    fused_kernel<PO2_F32, false, false><<<1, FUSED_THREADS, 0, st>>>(xv, yv, cp, zc, sse, scale_out, n, bits, fsr, mode, flavor, ws, 0, pk);
    err = cudaGetLastError();
  } else if (cluster) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks);
    cfg.blockDim = dim3(FUSED_THREADS);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)blocks; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    err = cudaLaunchKernelEx(&cfg, fused_kernel<PO2_F32, false, false>, xv, yv, cp, zc, sse, scale_out, n, bits, fsr, mode, flavor, ws, 1, pk);
  } else {
    err = cudaLaunchCooperativeKernel((const void*)fused_kernel<PO2_F32, false, false>, dim3((unsigned)blocks),
                                      dim3(FUSED_THREADS), args, 0, st);
  }
  return (int)err;
}

int multi_fused_capacity() { return FUSED_THREADS * FUSED_R * 4; }      // elements one CTA holds in registers

int multi_fused_launch(const MultiDesc* descs_dev, int ntensors, int csize, cudaStream_t st) {
  if (!descs_dev) return PO2_E_NULL;
  if (ntensors <= 0) return 0;
  if (csize != 1 && csize != 2 && csize != 4 && csize != 8) return PO2_E_SIZE;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(ntensors * csize));
  cfg.blockDim = dim3(FUSED_THREADS);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)csize; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return (int)cudaLaunchKernelEx(&cfg, multi_fused_kernel, descs_dev, csize);
}

}  // namespace po2

using namespace po2;

extern "C" {

int po2_abi_version(void) { return 2; }

int po2_have_torch_cuda_table(void) { return PO2_HAVE_TORCH_CUDA_TABLE; }

const char* po2_error_string(int code) {
  switch (code) {
    case 0: return "success";
    case PO2_E_DTYPE: return "po2: unsupported dtype (fp32, bf16, fp16 only)";
    case PO2_E_BITS: return "po2: bits must be in [2, 8] and |fsr| <= 64";
    case PO2_E_NULL: return "po2: null pointer argument";
    case PO2_E_SIZE: return "po2: empty tensor (torch.max of an empty tensor raises in the reference)";
    case PO2_E_ALIGN: return "po2: pointer alignment";
    case PO2_E_SHAPE: return "po2: unsupported convolution shape";
    case PO2_E_FLAVOR: return "po2: unknown log2 flavor";
    case PO2_E_WORKSPACE: return "po2: workspace missing or too small";
    case PO2_E_MODE: return "po2: unknown quantizer mode";
    case PO2_E_UNSUPPORTED: return "po2: unsupported argument combination";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "po2: unknown error";
  }
}

size_t po2_workspace_bytes(void) { return 256; }

int po2_absmax(const void* x, int64_t n, int dtype, float* scale_out, void* workspace, void* stream) {
  if (int e = check_common(n, dtype)) return e;
  if (!x || !scale_out) return PO2_E_NULL;
  if (!workspace) return PO2_E_WORKSPACE;
  return launch_absmax(x, n, dtype, scale_out, workspace, (cudaStream_t)stream);
}

int po2_quantize(const void* x, void* y, void* codes, unsigned int* zero_count, double* sse,
                 const float* scale, int64_t n, int dtype, int bits, int fsr, int mode, int flavor,
                 void* stream) {
  if (int e = check_common(n, dtype)) return e;
  if (int e = check_quant(bits, fsr, mode, flavor)) return e;
  if (!x || !y || !scale) return PO2_E_NULL;
  return launch_quantize(x, y, codes, zero_count, sse, scale, n, dtype, bits, fsr, mode, flavor, 0,
                         (cudaStream_t)stream);
}

// 1 if a tensor of n elements takes the single register-resident launch, 2 for the two passes
int po2_quantize_fused_launches(int64_t n, int dtype) {
  if (check_common(n, dtype)) return 0;
  const DevInfo* I = dev_info();
  if (!I) return 0;
  const int64_t n_vec = n / (16 / elem_bytes(dtype));
  const int64_t max_blocks = (int64_t)I->sms * I->fused_blocks_per_sm[dtype];
  return (max_blocks > 0 && n_vec <= max_blocks * (int64_t)FUSED_THREADS * FUSED_R) ? 1 : 2;
}

int po2_quantize_fused(const void* x, void* y, void* codes, unsigned int* zero_count, double* sse,
                       float* scale_out, int64_t n, int dtype, int bits, int fsr, int mode,
                       int flavor, void* workspace, void* stream) {
  if (int e = check_common(n, dtype)) return e;
  if (int e = check_quant(bits, fsr, mode, flavor)) return e;
  if (!x || !y || !scale_out) return PO2_E_NULL;
  if (!workspace) return PO2_E_WORKSPACE;
  const DevInfo* I = dev_info();
  if (!I) return (int)cudaErrorInvalidDevice;
  cudaStream_t st = (cudaStream_t)stream;
  const int epv = 16 / elem_bytes(dtype);
  const int64_t n_vec = n / epv;
  const int64_t max_blocks = (int64_t)I->sms * I->fused_blocks_per_sm[dtype];
  const int64_t per_block = (int64_t)FUSED_THREADS * FUSED_R;
  const bool vec_ok = aligned16(x) && aligned16(y) && (!codes || aligned16(codes));
  if (vec_ok && max_blocks > 0 && n_vec <= max_blocks * per_block) {
    // one launch, x read from HBM once.  Up to 8 CTAs form one thread-block cluster (max exchanged
    // through DSMEM); larger tensors use a cooperative grid with a global-memory barrier.
    int64_t blocks = (n_vec + FUSED_THREADS - 1) / FUSED_THREADS;
    if (blocks < 1) blocks = 1;
    int cluster = 0;
    if (n_vec <= per_block) blocks = 1;                  // fits one CTA: no exchange at all
    else if (n_vec <= 8 * per_block) { if (blocks > 8) blocks = 8; cluster = 1; }
    else if (blocks > max_blocks) blocks = max_blocks;
    Workspace* ws = (Workspace*)workspace;
    const uint4* xv = (const uint4*)x; uint4* yv = (uint4*)y; uint8_t* cp = (uint8_t*)codes;
    PackArgs pk = {};
    void* args[] = {&xv, &yv, &cp, &zero_count, &sse, &scale_out, &n, &bits, &fsr, &mode, &flavor, &ws, &cluster, &pk};
    cudaError_t err;
    if (blocks == 1) {
      PO2_DISPATCH(dtype, PO2_VARIANT(codes, sse, fused_kernel<DT, CODES, SSE><<<1, FUSED_THREADS, 0, st>>>(
          xv, yv, cp, zero_count, sse, scale_out, n, bits, fsr, mode, flavor, ws, 0, pk)));
      err = cudaGetLastError();
    } else if (cluster) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3((unsigned)blocks);
      cfg.blockDim = dim3(FUSED_THREADS);
      cfg.stream = st;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = (unsigned)blocks; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      PO2_DISPATCH(dtype, PO2_VARIANT(codes, sse, err = cudaLaunchKernelEx(
          &cfg, fused_kernel<DT, CODES, SSE>, xv, yv, cp, zero_count, sse, scale_out, n, bits, fsr, mode, flavor, ws, 1, pk)));
    } else {
      PO2_DISPATCH(dtype, PO2_VARIANT(codes, sse, err = cudaLaunchCooperativeKernel(
          (const void*)fused_kernel<DT, CODES, SSE>, dim3((unsigned)blocks), dim3(FUSED_THREADS), args, 0, st)));
    }
    return (int)err;
  }
  if (int e = launch_absmax(x, n, dtype, scale_out, workspace, st)) return e;
  // small enough that the first pass left a useful part of x in L2 -> second pass runs backwards
  const int reverse = ((double)n * elem_bytes(dtype) <= 512.0 * 1024 * 1024) ? 1 : 0;
  return launch_quantize(x, y, codes, zero_count, sse, scale_out, n, dtype, bits, fsr, mode, flavor,
                         reverse, st);
}

int po2_dequantize(const void* codes, const float* scale, void* y, int64_t n, int dtype, int bits,
                   int fsr, void* stream) {
  if (int e = check_common(n, dtype)) return e;
  if (int e = check_quant(bits, fsr, 0, 0)) return e;
  if (!codes || !scale || !y) return PO2_E_NULL;
  const DevInfo* I = dev_info();
  if (!I) return (int)cudaErrorInvalidDevice;
  const int blocks = grid_for((n + 1) / 2, 256, 4, I->sms * 8);
  PO2_DISPATCH(dtype, dequantize_kernel<DT><<<blocks, 256, 0, (cudaStream_t)stream>>>(
      (const uint8_t*)codes, scale, y, n, bits, fsr));
  return (int)cudaGetLastError();
}

int po2_ste_backward(const void* g, void* gx, int64_t n, int dtype, int accumulate, void* stream) {
  if (int e = check_common(n, dtype)) return e;
  if (!g || !gx) return PO2_E_NULL;
  const DevInfo* I = dev_info();
  if (!I) return (int)cudaErrorInvalidDevice;
  const int epv = 16 / elem_bytes(dtype);
  const int vec_ok = aligned16(g) && aligned16(gx);
  const int blocks = grid_for(n / epv + 1, 256, 4, I->sms * 8);
  PO2_DISPATCH(dtype, ste_backward_kernel<DT><<<blocks, 256, 0, (cudaStream_t)stream>>>(g, gx, n, accumulate, vec_ok));
  return (int)cudaGetLastError();
}

}  // extern "C"
