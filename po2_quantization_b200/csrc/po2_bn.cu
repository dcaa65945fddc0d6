// Batch normalisation around the quantized convs (SURVEY.md section 8(f) row 3): train-mode batch
// statistics, normalise (+ residual add) (+ ReLU) and the matching backward, for fp32 NCHW tensors.
//
// The reference models put an nn.SyncBatchNorm (+ ReLU, + the residual add) behind every
// QuantizedConv2d (models/resnet.py:38-61, :100-141).  On one GPU torch sends that to cuDNN's
// bn_fw_tr / bn_bw kernels, which take 44 / 84 us for an 8.4 MB tensor -- 49 % of a ResNet-56 QAT
// step (profiles/r01_launches_resnet56_qat_step_po2_conv.csv).  These kernels are HBM/L2-bound
// streaming passes with 128-bit accesses:
//
//   bn_reduce_kernel<0>    x -> per-channel (mean, M2, count)          reads x once
//   bn_apply_kernel        y = act((x-mean)*invstd*gamma+beta [+res])  reads x (L2), [res], writes y
//   bn_reduce_kernel<1|2>  per-channel sum(g), sum(g*(x-mean)), g = dy masked by the activation
//   bn_bwd_apply_kernel    dx (and the masked gradient for the residual branch)
//   bn_fwd_fused_kernel    the first two in ONE launch for tensors that fit in registers (one rank)
//   act: none / ReLU / ReLU6 / SiLU (forward + backward; SiLU's backward only without a residual branch)
//
// The split between the two halves of each direction is where SyncBatchNorm's collective goes
// (all_gather of the 2C+1 statistics forward, all_reduce of the 2C sums backward) -- done by the
// kernels themselves over NVLink peer stores (BnMailbox below), or by NCCL between the launches; with
// one rank the second kernel consumes the first one's output directly.
//
// Layout: x[B][C][HW].  A reduce CTA (s, c) owns the slabs b = s, s+S, ... of channel c; its partial
// sums go to a workspace and the last CTA of a channel to finish (ticket counter, self-resetting)
// combines them in double precision.  Sums are shifted by the channel's first element so that
// E[x^2]-E[x]^2 cancellation stays harmless when |mean| >> std.
#include <type_traits>

#include "po2_common.cuh"

namespace po2 {

constexpr int BN_THREADS = 256;
constexpr int BN_MAX_SPLIT = 64;
constexpr int BN_UNROLL = 4;
constexpr int BN_MAX_C = 4096;           // per-channel parameters live in shared memory (16 B each)

struct BnGeom {
  int B, C, HW;
  int L;          // vector lanes per slab: HW/4 (vec) or HW (scalar)
  int S;          // reduce splits per channel
  int cluster;    // one-launch kernels: the S CTAs of a channel are one thread-block cluster (barrier + partial sums
                  // through distributed shared memory instead of global counters)
  int total;      // B*C*L
  FastDiv div_l, div_c;
};

struct BnWorkspace {              // caller-provided, zero-initialised once; kernels leave counters zero
  unsigned int* ticket;           // [BN_MAX_C + 1] (per channel + one for the whole grid), first in the buffer
  unsigned int* depart;           // [BN_MAX_C]     second counter of the fused kernel's per-channel barrier
  double2* partial;               // [C][BN_MAX_SPLIT]
};

// ---- peer exchange: SyncBatchNorm's collectives inside the kernels ---------------------------------
// Every rank owns one BnMailbox in memory that all ranks of the NVLink domain have mapped (symmetric
// allocation; box[r] is rank r's mailbox in THIS rank's address space).  An exchange moves one small
// vector per rank (2C+1 statistics forward, 2C sums backward) with a flag-less low-latency protocol:
// every value travels as ONE 8-byte store {value bits, epoch tag} (8-byte stores are single
// transactions on the GPU and over NVLink), so there is no separate flag, no system-scope fence and
// no round trip on the producer -- the CTA that finishes channel c stores that channel's values
// straight into slot [epoch % BN_SLOTS].ll[rank] of EVERY rank's mailbox and is done.  The
// consuming kernel (apply / backward apply), next in the stream, polls the R tagged copies of each
// value it needs in its own mailbox until the tag equals the current epoch.  No collective launch,
// no host involvement, CUDA-graph replayable (the epoch lives in device memory; the last CTA of the
// producing grid advances it).  All ranks perform the same sequence of exchanges, so their epochs
// agree; a rank can be at most one exchange ahead of a peer (it needs the peer's values to get
// past the consumer), so with BN_SLOTS >= 2 a slot is never overwritten while it is being read, and
// a stale tag (epoch - BN_SLOTS) can never be mistaken for the current one.
constexpr int BN_MAX_RANKS = 8;
constexpr int BN_SLOTS = 4;
constexpr int BN_PAYLOAD = 2 * BN_MAX_C + 32;      // values per rank per slot (>= 2C+1)
struct BnMailSlot {
  uint2 ll[BN_MAX_RANKS][BN_PAYLOAD];              // {value bits, epoch tag}
};
struct BnMailbox {
  uint32_t epoch;                                  // exchanges this rank has completed producing
  uint32_t error;                                  // set when a poll timed out (a peer died); sticky
  uint32_t timeout_s;                              // poll timeout in seconds, written by the host (0: 20 s)
  uint32_t pad[13];
  BnMailSlot slot[BN_SLOTS];
};
struct BnPeers {
  BnMailbox* box[BN_MAX_RANKS];
  int rank, world;                                 // world <= 1: no exchange
};

__device__ __forceinline__ void st_ll(uint2* p, float v, uint32_t tag) {
  asm volatile("st.volatile.global.v2.u32 [%0], {%1, %2};" :: "l"(p), "r"(__float_as_uint(v)), "r"(tag) : "memory");
}
__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
// poll one tagged value of this rank's own mailbox.  A poll that times out (a peer stopped publishing:
// stalled in its data loader, crashed, ...) must not pass for a result: it raises the sticky error flag
// and returns NaN, so the statistics, the output and the loss of this step are NaN, the consumers skip
// the running-statistics update, and the host-side check (PeerExchange.check) raises.
__device__ __forceinline__ bool mailbox_failed(const BnMailbox* me) {
  return me && *reinterpret_cast<const volatile uint32_t*>(&me->error) != 0u;
}
__device__ __forceinline__ float ld_ll(const uint2* p, uint32_t tag, BnMailbox* me) {
  uint32_t v, t;
  asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v), "=r"(t) : "l"(p) : "memory");
  if (t != tag) {
    const uint32_t ts = *reinterpret_cast<const volatile uint32_t*>(&me->timeout_s);
    const unsigned long long limit = (unsigned long long)(ts ? ts : 20u) * 1000000000ull;
    const unsigned long long t0 = global_ns();
    do {
      // once any poll of this mailbox has failed, later polls give up quickly instead of each
      // waiting the full timeout (2C+1 values per exchange)
      if (global_ns() - t0 > (mailbox_failed(me) ? 1000000ull : limit)) {
        me->error = 1;
        __threadfence();
        return __uint_as_float(0x7FC00000u);
      }
      __nanosleep(64);
      asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v), "=r"(t) : "l"(p) : "memory");
    } while (t != tag);
  }
  return __uint_as_float(v);
}

// R vectors of the current exchange: dense rows (stats != nullptr) or this rank's mailbox.
// fetch<N>: values idx[0..N) of every rank at once -- all loads are issued before the first tag is
// looked at (N*R independent L2 reads instead of a chain of dependent polls); a value whose tag is
// not there yet falls to the polling loop.
struct BnGather {
  const float* dense; int stride;
  const uint2* ll; uint32_t tag; BnMailbox* me;
  template <int N>
  __device__ __forceinline__ void fetch(int R, const int (&idx)[N], float (&out)[N][BN_MAX_RANKS]) const {
    if (ll) {
      uint2 raw[N][BN_MAX_RANKS];
#pragma unroll
      for (int r = 0; r < BN_MAX_RANKS; ++r)
#pragma unroll
        for (int k = 0; k < N; ++k)
          if (r < R) raw[k][r] = __ldcv(ll + (size_t)r * BN_PAYLOAD + idx[k]);
#pragma unroll
      for (int r = 0; r < BN_MAX_RANKS; ++r)
#pragma unroll
        for (int k = 0; k < N; ++k)
          if (r < R)
            out[k][r] = raw[k][r].y == tag ? __uint_as_float(raw[k][r].x)
                                           : ld_ll(ll + (size_t)r * BN_PAYLOAD + idx[k], tag, me);
    } else {
#pragma unroll
      for (int r = 0; r < BN_MAX_RANKS; ++r)
#pragma unroll
        for (int k = 0; k < N; ++k)
          if (r < R) out[k][r] = __ldcg(dense + (size_t)r * stride + idx[k]);
    }
  }
};
__device__ __forceinline__ BnGather gather_from(const float* dense, int stride, BnMailbox* mailbox) {
  BnGather g;
  g.dense = dense; g.stride = stride; g.ll = nullptr; g.tag = 0; g.me = mailbox;
  if (mailbox) {
    g.tag = *reinterpret_cast<volatile uint32_t*>(&mailbox->epoch);       // advanced by the producing grid
    g.ll = &mailbox->slot[g.tag % BN_SLOTS].ll[0][0];
  }
  return g;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}

// sum (a, b) over the CTA; valid in every thread of warp 0
__device__ __forceinline__ void block_sum2(double& a, double& b, double (*sm)[2]) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  a = warp_sum(a);
  b = warp_sum(b);
  __syncthreads();                                   // sm may still be read from a previous call
  if (lane == 0) { sm[warp][0] = a; sm[warp][1] = b; }
  __syncthreads();
  if (warp == 0) {
    a = lane < BN_THREADS / 32 ? sm[lane][0] : 0.0;
    b = lane < BN_THREADS / 32 ? sm[lane][1] : 0.0;
    a = warp_sum(a);
    b = warp_sum(b);
  }
}

// publish this CTA's partial, and tell whether it is the last CTA of channel c to do so
__device__ __forceinline__ bool publish_partial(double a, double b, const BnWorkspace& ws, int c, int s, int S,
                                                int* flag) {
  if (threadIdx.x == 0) {
    ws.partial[c * BN_MAX_SPLIT + s] = make_double2(a, b);
    __threadfence();
    const unsigned int t = atomicAdd(ws.ticket + c, 1u);
    *flag = (t == (unsigned int)(S - 1));
    if (*flag) { ws.ticket[c] = 0; __threadfence(); }
  }
  __syncthreads();
  return *flag != 0;
}

// activations behind the norm: 0 none, 1 ReLU, 2 ReLU6 (hardtanh(0, 6): gradient passes for 0 < y < 6),
// 3 SiLU (backward: bn_silu_slope, z recomputed from x)
__device__ __forceinline__ float bn_act(float v, int act) {
  if (act == 1) return fmaxf(v, 0.f);
  if (act == 2) return fminf(fmaxf(v, 0.f), 6.f);
  if (act == 3) return v / (1.f + __expf(-v));
  return v;
}
__device__ __forceinline__ bool bn_act_open(float y, int act) { return y > 0.f && (act != 2 || y < 6.f); }
// SiLU behind the norm (no residual branch): d silu(z) / dz at z = (x - mean) * a + b, a = gamma * invstd, b = beta --
// the forward's own expression for z (bn_apply_kernel), sigmoid from the same __expf
__device__ __forceinline__ float bn_silu_slope(float x, float mu, float a, float b) {
  const float z = fmaf(x - mu, a, b);
  const float sg = 1.f / (1.f + __expf(-z));
  return sg * fmaf(z, 1.f - sg, 1.f);
}

#ifdef PO2_BN_TRACE
// debug-only phase stamps of the one-launch kernels (tools/trace_bn.py builds a separate library with -DPO2_BN_TRACE)
__device__ unsigned long long* g_bn_trace = nullptr;
#define BN_STAMP(i)                                                                                   \
  do {                                                                                                \
    if (g_bn_trace && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {                       \
      unsigned long long t_;                                                                          \
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                          \
      g_bn_trace[i] = t_;                                                                             \
    }                                                                                                 \
  } while (0)
#else
#define BN_STAMP(i) do {} while (0)
#endif

// Index of the element loops.  The VEC forms count float4s, so their counts stay below 2^29 and a 32-bit index never
// nears 2^31.  The scalar forms count floats: a count below 2^31 may lie within one step of 2^31, so they step in
// 64 bits.
template <bool VEC> using BnIdx = typename std::conditional<VEC, int, int64_t>::type;

// MODE 0: forward statistics (p = x - shift, q = p);  1: backward sums (p = dy, q = x - mean);
// MODE 2: backward sums behind a ReLU (p = y > 0 ? dy : 0).
template <bool VEC, int MODE>
__global__ void __launch_bounds__(BN_THREADS) bn_reduce_kernel(const float* __restrict__ x,
                                                               const float* __restrict__ dy,
                                                               const float* __restrict__ y,
                                                               const float* __restrict__ mean,
                                                               const float* __restrict__ invstd,
                                                               float* __restrict__ out,      // MODE 0: stat[2C+1]; else sums[2C]
                                                               float* __restrict__ dgamma,
                                                               float* __restrict__ dbeta, BnGeom g,
                                                               BnWorkspace ws, BnPeers peers, int act,
                                                               const float* __restrict__ gamma = nullptr,
                                                               const float* __restrict__ beta = nullptr,
                                                               const float* __restrict__ dy2 = nullptr) {
  // dy2 (backward): a second gradient of the same tensor -- the skip connection's -- added on the fly (dy + dy2),
  // instead of an accumulation kernel in front of this one
  // (PO2_BN_REDUCE_PDL=1: this grid is itself a programmatic dependent of the kernel that produced its input)
  asm volatile("griddepcontrol.wait;" ::: "memory");
  // the consuming kernel (apply / backward apply, launched with programmatic stream serialization) may
  // be scheduled as soon as every CTA of this grid is running; it waits for this grid's completion
  // (griddepcontrol.wait) before it reads anything this grid writes
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  __shared__ double sm[BN_THREADS / 32][2];
  __shared__ int flag;
  __shared__ uint32_t s_epoch;
  __shared__ float s_val[2];
  const int s = blockIdx.x, c = blockIdx.y;
  const int L = g.L, C = g.C;
  const int nslab = (g.B - s + g.S - 1) / g.S;                 // slabs b = s, s+S, ...
  const int n = nslab * L;
  const float shift = MODE == 0 ? __ldg(x + (size_t)c * g.HW) : __ldg(mean + c);
  const bool silu = MODE == 2 && act == 3;
  const float za = silu ? (gamma ? __ldg(gamma + c) : 1.f) * __ldg(invstd + c) : 0.f, zb = silu && beta ? __ldg(beta + c) : 0.f;
  // tag of the exchange this grid produces; read before any CTA can have advanced it (the advance
  // needs every CTA's ticket, taken below), visible to the CTA after the first barrier in block_sum2
  if (threadIdx.x == 0 && peers.world > 1)
    s_epoch = *reinterpret_cast<volatile uint32_t*>(&peers.box[peers.rank]->epoch) + 1;
  float s1 = 0.f, s2 = 0.f;
  for (BnIdx<VEC> i0 = threadIdx.x; i0 < n; i0 += BN_UNROLL * BN_THREADS) {
    if (VEC) {
      float4 vx[BN_UNROLL], vd[BN_UNROLL], vy[BN_UNROLL];
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        const int i = i0 + u * BN_THREADS;
        vx[u] = vd[u] = vy[u] = make_float4(shift, shift, shift, shift);
        if (MODE != 0) vd[u] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n) {
          const int k = fdiv(i, g.div_l);
          const size_t off = ((size_t)(s + k * g.S) * C + c) * L + (i - k * L);
          vx[u] = __ldg(reinterpret_cast<const float4*>(x) + off);
          if (MODE != 0) vd[u] = __ldg(reinterpret_cast<const float4*>(dy) + off);
          if (MODE != 0 && dy2) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(dy2) + off);
            vd[u].x += t.x; vd[u].y += t.y; vd[u].z += t.z; vd[u].w += t.w;
          }
          if (MODE == 2 && !silu) vy[u] = __ldg(reinterpret_cast<const float4*>(y) + off);
        }
      }
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        const float xs[4] = {vx[u].x, vx[u].y, vx[u].z, vx[u].w};
        const float ds[4] = {vd[u].x, vd[u].y, vd[u].z, vd[u].w};
        const float ys[4] = {vy[u].x, vy[u].y, vy[u].z, vy[u].w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float q = xs[e] - shift;
          if (MODE == 0) { s1 += q; s2 = fmaf(q, q, s2); }
          else {
            float p = ds[e];
            if (MODE == 2) p = silu ? p * bn_silu_slope(xs[e], shift, za, zb) : (bn_act_open(ys[e], act) ? p : 0.f);
            s1 += p; s2 = fmaf(p, q, s2);
          }
        }
      }
    } else {
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        if (i0 + u * BN_THREADS < n) {
          const int i = (int)(i0 + u * BN_THREADS);
          const int k = fdiv(i, g.div_l);
          const size_t off = ((size_t)(s + k * g.S) * C + c) * L + (i - k * L);
          const float xv = __ldg(x + off);
          const float q = xv - shift;
          if (MODE == 0) { s1 += q; s2 = fmaf(q, q, s2); }
          else {
            float p = __ldg(dy + off);
            if (dy2) p += __ldg(dy2 + off);
            if (MODE == 2) p = silu ? p * bn_silu_slope(xv, shift, za, zb) : (bn_act_open(__ldg(y + off), act) ? p : 0.f);
            s1 += p; s2 = fmaf(p, q, s2);
          }
        }
      }
    }
  }
  double a = (double)s1, b = (double)s2;
  block_sum2(a, b, sm);
  if (!publish_partial(a, b, ws, c, s, g.S, &flag)) return;
  // last CTA of this channel: combine the S partials
  double pa = 0.0, pb = 0.0;
  if ((int)threadIdx.x < g.S) {
    const double2 p = __ldcg(ws.partial + c * BN_MAX_SPLIT + threadIdx.x);
    pa = p.x; pb = p.y;
  }
  block_sum2(pa, pb, sm);
  if (threadIdx.x == 0) {
    float v0, v1;
    if (MODE == 0) {
      const double cnt = (double)g.B * (double)g.HW;
      const double m = pa / cnt;
      v0 = (float)((double)shift + m);
      v1 = (float)fmax(pb - pa * m, 0.0);                        // M2 = sum (x-mean)^2
      if (c == 0) out[2 * C] = (float)cnt;
    } else {
      v0 = (float)pa;                                            // sum g
      v1 = (float)pb;                                            // sum g*(x-mean)
      if (dbeta) dbeta[c] = v0;
      if (dgamma) dgamma[c] = (float)(pb * (double)__ldg(invstd + c));
    }
    out[c] = v0;
    out[C + c] = v1;
    s_val[0] = v0; s_val[1] = v1;
  }
  if (peers.world <= 1) return;
  __syncthreads();
  // this channel's values go straight to every rank's mailbox (one thread per destination)
  if ((int)threadIdx.x < peers.world) {
    const uint32_t tag = s_epoch;
    uint2* dst = peers.box[threadIdx.x]->slot[tag % BN_SLOTS].ll[peers.rank];
    st_ll(dst + c, s_val[0], tag);
    st_ll(dst + C + c, s_val[1], tag);
    if (MODE == 0 && c == 0) st_ll(dst + 2 * C, (float)((double)g.B * (double)g.HW), tag);
  }
  // the CTA that finishes the last channel advances this rank's epoch for the consuming kernel
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int t = atomicAdd(ws.ticket + BN_MAX_C, 1u);
    if (t == (unsigned int)(C - 1)) {
      ws.ticket[BN_MAX_C] = 0;
      peers.box[peers.rank]->epoch = s_epoch;
    }
  }
}

// ---- per-channel parameters in shared memory ----------------------------------------------------
// forward: {mean, gamma*invstd, beta, -};  statistics = R entries of [mean[C] | M2[C] | count] (train)
// or the running statistics (eval).
__device__ __forceinline__ void combine_stats(const BnGather& src, int R, int C, int c, double& mean,
                                              double& var_biased, double& count) {
  const int idx[3] = {c, C + c, 2 * C};
  float v[3][BN_MAX_RANKS];                          // mean, M2, count of every rank
  src.fetch<3>(R, idx, v);
  double n = 0.0, m = 0.0;
  for (int r = 0; r < R; ++r) {
    n += (double)v[2][r];
    m += (double)v[2][r] * (double)v[0][r];
  }
  m /= n;
  double m2 = 0.0;
  for (int r = 0; r < R; ++r) {
    const double d = (double)v[0][r] - m;
    m2 += (double)v[1][r] + (double)v[2][r] * d * d;
  }
  mean = m; var_biased = m2 / n; count = n;
}

template <bool VEC>
__global__ void __launch_bounds__(BN_THREADS, 4) bn_apply_kernel(const float* __restrict__ x,
                                                              const float* __restrict__ res,
                                                              float* __restrict__ y,
                                                              const float* stats, int R, BnMailbox* mailbox,
                                                              float* __restrict__ stats_dense,
                                                              const float* __restrict__ gamma,
                                                              const float* __restrict__ beta,
                                                              float* running_mean, float* running_var,
                                                              long long* num_batches_tracked, float momentum,
                                                              float eps, int act, int use_running,
                                                              float* __restrict__ save_mean,
                                                              float* __restrict__ save_invstd, BnGeom g) {
  extern __shared__ float4 prm[];
  const int C = g.C;
  // x / residual were complete before the statistics kernel started; the statistics (and the mailbox
  // epoch) are that kernel's output
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the conv behind may set up under this kernel
  const BnGather src = gather_from(stats, 2 * C + 1, use_running ? nullptr : mailbox);
  if (src.ll && blockIdx.x == 0 && stats_dense)          // dense copy of the gathered statistics for backward
    for (int i = threadIdx.x; i < 2 * C + 1; i += BN_THREADS) {
      const int idx[1] = {i};
      float v[1][BN_MAX_RANKS];
      src.fetch<1>(R, idx, v);
      for (int r = 0; r < R; ++r) stats_dense[(size_t)r * (2 * C + 1) + i] = v[0][r];
    }
  for (int c = threadIdx.x; c < C; c += BN_THREADS) {
    double mean, var, cnt = 0.0;
    if (use_running) { mean = (double)running_mean[c]; var = (double)running_var[c]; }
    else combine_stats(src, R, C, c, mean, var, cnt);
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    const float ga = gamma ? gamma[c] : 1.0f, be = beta ? beta[c] : 0.0f;
    prm[c] = make_float4((float)mean, ga * invstd, be, 0.f);
    if (blockIdx.x == 0 && !use_running) {
      if (save_mean) save_mean[c] = (float)mean;
      if (save_invstd) save_invstd[c] = invstd;
      if (running_mean && !mailbox_failed(src.ll ? mailbox : nullptr)) {   // a timed-out exchange must not reach the running statistics
        const double unbiased = var * cnt / fmax(cnt - 1.0, 1.0);
        running_mean[c] = (float)((1.0 - (double)momentum) * (double)running_mean[c] + (double)momentum * mean);
        running_var[c] = (float)((1.0 - (double)momentum) * (double)running_var[c] + (double)momentum * unbiased);
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && !use_running && num_batches_tracked) *num_batches_tracked += 1;
  __syncthreads();
  const int L = g.L;
  for (BnIdx<VEC> i0 = blockIdx.x * (BN_UNROLL * BN_THREADS) + threadIdx.x; i0 < g.total;
       i0 += gridDim.x * (BN_UNROLL * BN_THREADS)) {
    if (VEC) {
      float4 vx[BN_UNROLL], vr[BN_UNROLL];
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        const int i = i0 + u * BN_THREADS;
        if (i < g.total) {
          vx[u] = __ldg(reinterpret_cast<const float4*>(x) + i);
          if (res) vr[u] = __ldg(reinterpret_cast<const float4*>(res) + i);
        }
      }
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        const int i = i0 + u * BN_THREADS;
        if (i < g.total) {
          const int slab = fdiv(i, g.div_l);
          const int c = slab - fdiv(slab, g.div_c) * C;
          const float4 p = prm[c];
          float4 o;
          o.x = fmaf(vx[u].x - p.x, p.y, p.z); o.y = fmaf(vx[u].y - p.x, p.y, p.z);
          o.z = fmaf(vx[u].z - p.x, p.y, p.z); o.w = fmaf(vx[u].w - p.x, p.y, p.z);
          if (res) { o.x += vr[u].x; o.y += vr[u].y; o.z += vr[u].z; o.w += vr[u].w; }
          if (act) { o.x = bn_act(o.x, act); o.y = bn_act(o.y, act); o.z = bn_act(o.z, act); o.w = bn_act(o.w, act); }
          reinterpret_cast<float4*>(y)[i] = o;
        }
      }
    } else {
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        if (i0 + u * BN_THREADS < g.total) {
          const int i = (int)(i0 + u * BN_THREADS);
          const int slab = fdiv(i, g.div_l);
          const int c = slab - fdiv(slab, g.div_c) * C;
          const float4 p = prm[c];
          float o = fmaf(__ldg(x + i) - p.x, p.y, p.z);
          if (res) o += __ldg(res + i);
          o = bn_act(o, act);
          y[i] = o;
        }
      }
    }
  }
}

// backward: dx = (g - sum_g/M - (x-mean) * invstd^2 * sum_gx/M) * gamma*invstd;  dres = g (masked dy)
template <bool VEC>
__global__ void __launch_bounds__(BN_THREADS, 4) bn_bwd_apply_kernel(const float* __restrict__ dy,
                                                                  const float* __restrict__ x,
                                                                  const float* __restrict__ y,
                                                                  const float* __restrict__ mean,
                                                                  const float* __restrict__ invstd,
                                                                  const float* __restrict__ gamma,
                                                                  const float* sums,
                                                                  const float* __restrict__ stats, int R,
                                                                  BnMailbox* mailbox,
                                                                  float* __restrict__ dx,
                                                                  float* __restrict__ dres, int act, BnGeom g,
                                                                  const float* __restrict__ beta,
                                                                  const float* __restrict__ dy2) {
  extern __shared__ float4 prm[];
  const int C = g.C;
  float* prb = reinterpret_cast<float*>(prm + C);                 // beta per channel (SiLU: z is recomputed from x)
  asm volatile("griddepcontrol.wait;" ::: "memory");            // sums / mailbox epoch come from the reduce kernel
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the conv behind may set up under this kernel
  double M = 0.0;
  for (int r = 0; r < R; ++r) M += (double)stats[(size_t)r * (2 * C + 1) + 2 * C];
  const BnGather src = gather_from(nullptr, 0, mailbox);          // R ranks' sums: add them here, in rank order
  for (int c = threadIdx.x; c < C; c += BN_THREADS) {
    const double is = (double)invstd[c];
    const float ga = gamma ? gamma[c] : 1.0f;
    double sg, sgx;
    if (src.ll) {
      const int idx[2] = {c, C + c};
      float v[2][BN_MAX_RANKS];
      src.fetch<2>(R, idx, v);
      float a = 0.f, b = 0.f;                                      // fp32 adds in rank order == all_reduce(SUM) semantics
      for (int r = 0; r < R; ++r) { a += v[0][r]; b += v[1][r]; }
      sg = (double)a; sgx = (double)b;
    } else { sg = (double)sums[c]; sgx = (double)sums[C + c]; }
    prm[c] = make_float4(mean[c], (float)(sg / M), (float)(is * is * sgx / M), (float)((double)ga * is));
    prb[c] = beta ? beta[c] : 0.f;
  }
  __syncthreads();
  const bool silu = act == 3;
  const bool relu = act != 0 && !silu;                         // masked by the activation's open interval
  for (BnIdx<VEC> i0 = blockIdx.x * (BN_UNROLL * BN_THREADS) + threadIdx.x; i0 < g.total;
       i0 += gridDim.x * (BN_UNROLL * BN_THREADS)) {
    if (VEC) {
      float4 vd[BN_UNROLL], vx[BN_UNROLL], vy[BN_UNROLL];
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        const int i = i0 + u * BN_THREADS;
        if (i < g.total) {
          vd[u] = __ldg(reinterpret_cast<const float4*>(dy) + i);
          if (dy2) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(dy2) + i);
            vd[u].x += t.x; vd[u].y += t.y; vd[u].z += t.z; vd[u].w += t.w;
          }
          vx[u] = __ldg(reinterpret_cast<const float4*>(x) + i);
          if (relu) vy[u] = __ldg(reinterpret_cast<const float4*>(y) + i);
        }
      }
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        const int i = i0 + u * BN_THREADS;
        if (i < g.total) {
          const int slab = fdiv(i, g.div_l);
          const int c = slab - fdiv(slab, g.div_c) * C;
          const float4 p = prm[c];
          float4 gr = vd[u];
          if (relu) {
            gr.x = bn_act_open(vy[u].x, act) ? gr.x : 0.f; gr.y = bn_act_open(vy[u].y, act) ? gr.y : 0.f;
            gr.z = bn_act_open(vy[u].z, act) ? gr.z : 0.f; gr.w = bn_act_open(vy[u].w, act) ? gr.w : 0.f;
          } else if (silu) {
            const float zb = prb[c];                               // p.w = gamma * invstd
            gr.x *= bn_silu_slope(vx[u].x, p.x, p.w, zb); gr.y *= bn_silu_slope(vx[u].y, p.x, p.w, zb);
            gr.z *= bn_silu_slope(vx[u].z, p.x, p.w, zb); gr.w *= bn_silu_slope(vx[u].w, p.x, p.w, zb);
          }
          float4 o;
          o.x = (gr.x - p.y - (vx[u].x - p.x) * p.z) * p.w; o.y = (gr.y - p.y - (vx[u].y - p.x) * p.z) * p.w;
          o.z = (gr.z - p.y - (vx[u].z - p.x) * p.z) * p.w; o.w = (gr.w - p.y - (vx[u].w - p.x) * p.z) * p.w;
          reinterpret_cast<float4*>(dx)[i] = o;
          if (dres) reinterpret_cast<float4*>(dres)[i] = gr;
        }
      }
    } else {
#pragma unroll
      for (int u = 0; u < BN_UNROLL; ++u) {
        if (i0 + u * BN_THREADS < g.total) {
          const int i = (int)(i0 + u * BN_THREADS);
          const int slab = fdiv(i, g.div_l);
          const int c = slab - fdiv(slab, g.div_c) * C;
          const float4 p = prm[c];
          float gr = __ldg(dy + i);
          if (dy2) gr += __ldg(dy2 + i);
          if (relu && !bn_act_open(__ldg(y + i), act)) gr = 0.f;
          if (silu) gr *= bn_silu_slope(__ldg(x + i), p.x, p.w, prb[c]);
          dx[i] = (gr - p.y - (__ldg(x + i) - p.x) * p.z) * p.w;
          if (dres) dres[i] = gr;
        }
      }
    }
  }
}

// ---- fused forward for tensors that fit in registers ---------------------------------------------------
// Statistics and apply in ONE launch: CTA (s, c) loads its slabs of channel c once (<= BN_FUSED_R
// 128-bit vectors per thread, kept in registers), the S CTAs of a channel meet at a per-channel
// barrier (two counters in the workspace, self-resetting; all CTAs are co-resident: the host caps the
// grid at two CTAs per SM), the channel's statistics are combined -- through the peer mailboxes when
// there are several ranks: CTA (0, c) publishes, every CTA of the channel polls -- and the CTA
// normalises its registers and writes y.  Saves a launch and the second read of x per layer.
constexpr int BN_FUSED_R = 8;

// ---- the S CTAs of a channel as one thread-block cluster (S <= 16): each CTA leaves its partial sums in its own
// shared memory, the hardware cluster barrier replaces the global ticket / poll / depart sequence (measured ~2 us per
// kernel on the 16-channel layers), every CTA reads the S partials over DSMEM in rank order
__device__ __forceinline__ void bn_cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void bn_cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ double2 bn_ld_cluster(const double2* p, uint32_t rank) {
  const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
  uint32_t ra;
  double2 v;
  asm("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(a), "r"(rank));
  asm volatile("ld.shared::cluster.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(ra));
  return v;
}

// returns false if the barrier timed out (the CTAs of the channel were not co-resident for 10 s --
// e.g. another stream held the SMs); the caller then poisons its output with NaN so the failure is loud
__device__ __forceinline__ bool channel_barrier(const BnWorkspace& ws, int c, int S, BnMailbox* errbox, int* s_ok) {
  if (threadIdx.x == 0) *s_ok = 1;
  __syncthreads();
  if (threadIdx.x == 0 && S > 1) {
    __threadfence();
    atomicAdd(ws.ticket + c, 1u);
    const unsigned long long t0 = global_ns();
    while (*reinterpret_cast<volatile unsigned int*>(ws.ticket + c) < (unsigned int)S) {
      if (global_ns() - t0 > 10000000000ull) { *s_ok = 0; if (errbox) errbox->error = 2; break; }   // never hang the GPU
      __nanosleep(32);
    }
    __threadfence();
    const unsigned int d = atomicAdd(ws.depart + c, 1u);
    if (d == (unsigned int)(S - 1)) { ws.ticket[c] = 0u; ws.depart[c] = 0u; __threadfence(); }   // everyone has passed
  }
  __syncthreads();
  return *s_ok != 0;
}

// thread 0 of a CTA: turn the channel's shifted sums into (mean, gamma*invstd, beta), with the peer
// exchange when there are several ranks; CTA s == 0 of the channel also writes the per-channel outputs
// what thread 0 of a CTA keeps of the channel's statistics for the bookkeeping stores behind the apply phase
struct BnChannelStats { double mean, var, n_tot, m2; float invstd; };

__device__ __noinline__ float4 fused_channel_finish(double pa, double pb, float shift, int s, int c, const BnGeom& g,
                                                    const BnPeers& peers, BnMailbox* me, uint32_t tag, int R,
                                                    float ga, float be, float eps, float* __restrict__ stats_dense,
                                                    BnChannelStats& cs) {
  const int C = g.C;
  float4 prm_out;
    const double cnt = (double)g.B * (double)g.HW;
    const double m = pa / cnt;
    double mean = (double)shift + m, m2 = fmax(pb - pa * m, 0.0), n_tot = cnt;
    if (me) {
      // all_gather inside the kernel: CTA (0, c) stores this rank's values into every mailbox, every CTA polls
      const float lmean = (float)mean, lm2 = (float)m2, lcnt = (float)cnt;
      if (s == 0)
        for (int p = 0; p < peers.world; ++p) {
          uint2* dst = peers.box[p]->slot[tag % BN_SLOTS].ll[peers.rank];
          st_ll(dst + c, lmean, tag);
          st_ll(dst + C + c, lm2, tag);
          if (c == 0) st_ll(dst + 2 * C, lcnt, tag);
        }
      BnGather src;
      src.dense = nullptr; src.stride = 0; src.tag = tag; src.me = me;
      src.ll = &me->slot[tag % BN_SLOTS].ll[0][0];
      double var;
      combine_stats(src, R, C, c, mean, var, n_tot);
      m2 = var * n_tot;
      if (s == 0 && stats_dense) {
        const int idx[3] = {c, C + c, 2 * C};
        float g3[3][BN_MAX_RANKS];
        src.fetch<3>(R, idx, g3);
        for (int r = 0; r < R; ++r) {
          stats_dense[(size_t)r * (2 * C + 1) + c] = g3[0][r];
          stats_dense[(size_t)r * (2 * C + 1) + C + c] = g3[1][r];
          if (c == 0) stats_dense[(size_t)r * (2 * C + 1) + 2 * C] = g3[2][r];
        }
      }
    }
    const double var = m2 / n_tot;
    const float invstd = (float)(1.0 / sqrt(var + (double)eps));
    prm_out = make_float4((float)mean, ga * invstd, be, 0.f);
    cs.mean = mean; cs.var = var; cs.n_tot = n_tot; cs.m2 = m2; cs.invstd = invstd;
  return prm_out;
}

// the stores nobody inside the kernel waits for (CTA (0, c), thread 0, behind the apply phase): saved statistics for
// the backward pass, the running statistics (their old values were loaded at the start of the kernel)
__device__ __forceinline__ void fused_channel_book(const BnChannelStats& cs, int c, int C, bool single_rank, BnMailbox* me,
                                                   float* running_mean, float* running_var, float rm_old, float rv_old,
                                                   long long* num_batches_tracked, long long nbt_old, float momentum,
                                                   float* __restrict__ save_mean, float* __restrict__ save_invstd,
                                                   float* __restrict__ stats_dense, double cnt_local) {
  if (single_rank && stats_dense) {
    stats_dense[c] = (float)cs.mean;
    stats_dense[C + c] = (float)cs.m2;
    if (c == 0) stats_dense[2 * C] = (float)cnt_local;
  }
  if (save_mean) save_mean[c] = (float)cs.mean;
  if (save_invstd) save_invstd[c] = cs.invstd;
  if (running_mean && !mailbox_failed(me)) {               // a timed-out exchange must not reach the running statistics
    const double unbiased = cs.var * cs.n_tot / fmax(cs.n_tot - 1.0, 1.0);
    running_mean[c] = (float)((1.0 - (double)momentum) * (double)rm_old + (double)momentum * cs.mean);
    running_var[c] = (float)((1.0 - (double)momentum) * (double)rv_old + (double)momentum * unbiased);
  }
  if (c == 0 && num_batches_tracked) *num_batches_tracked = nbt_old + 1;
}

__global__ void __launch_bounds__(BN_THREADS, 2) bn_fwd_fused_kernel(const float* __restrict__ x,
                                                                     const float* __restrict__ res,
                                                                     float* __restrict__ y,
                                                                     const float* __restrict__ gamma,
                                                                     const float* __restrict__ beta,
                                                                     float* running_mean, float* running_var,
                                                                     long long* num_batches_tracked, float momentum,
                                                                     float eps, int act, float* __restrict__ save_mean,
                                                                     float* __restrict__ save_invstd,
                                                                     float* __restrict__ stats_dense, BnGeom g,
                                                                     BnWorkspace ws, BnPeers peers) {
  __shared__ double sm[BN_THREADS / 32][2];
  __shared__ float4 s_prm;
  __shared__ int s_ok;
  const int s = blockIdx.x, c = blockIdx.y, C = g.C, L = g.L;
  const int nslab = (g.B - s + g.S - 1) / g.S;
  const int n = nslab * L;
  const int R = peers.world > 1 ? peers.world : 1;
  BnMailbox* me = peers.world > 1 ? peers.box[peers.rank] : nullptr;
  const uint32_t tag = me ? *reinterpret_cast<volatile uint32_t*>(&me->epoch) + 1 : 0;   // read before anyone advances it
  BN_STAMP(0);
  // thread 0 needs these after the channel barrier: their loads go out now, under phase 1 (behind the barrier
  // they were three serialised round trips of the whole CTA's critical path: measured 2.7 us of 8.9)
  float ga = 1.0f, be = 0.0f, rm_old = 0.f, rv_old = 0.f;
  long long nbt_old = 0;
  if (threadIdx.x == 0) {
    // (volatile asm: the compiler must not sink these loads to their uses behind the barrier)
    if (gamma) asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(ga) : "l"(gamma + c));
    if (beta) asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(be) : "l"(beta + c));
    if (s == 0 && running_mean) {
      asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(rm_old) : "l"(running_mean + c));
      asm volatile("ld.global.cg.f32 %0, [%1];" : "=f"(rv_old) : "l"(running_var + c));
    }
    if (s == 0 && c == 0 && num_batches_tracked)
      asm volatile("ld.global.cg.s64 %0, [%1];" : "=l"(nbt_old) : "l"(num_batches_tracked));
  }
  // launched programmatically behind the conv that produces x: everything above ran under its tail.  Then: a conv
  // launched programmatically behind THIS kernel may set up (barriers, TMEM, tensor map) under it; it waits for this
  // grid's completion before it touches y
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const float shift = __ldg(x + (size_t)c * g.HW);
  // ---- phase 1: load into registers, shifted sums
  float4 v[BN_FUSED_R];
  int off[BN_FUSED_R];                                   // in 128-bit units (< 2^29, checked on the host)
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int u = 0; u < BN_FUSED_R; ++u) {
    const int i = threadIdx.x + u * BN_THREADS;
    v[u] = make_float4(shift, shift, shift, shift);
    off[u] = 0;
    if (i < n) {
      const int k = fdiv(i, g.div_l);
      off[u] = ((s + k * g.S) * C + c) * L + (i - k * L);
      v[u] = __ldg(reinterpret_cast<const float4*>(x) + off[u]);
    }
  }
#pragma unroll
  for (int u = 0; u < BN_FUSED_R; ++u) {
    const float q0 = v[u].x - shift, q1 = v[u].y - shift, q2 = v[u].z - shift, q3 = v[u].w - shift;
    s1 += (q0 + q1) + (q2 + q3);
    s2 = fmaf(q0, q0, s2); s2 = fmaf(q1, q1, s2); s2 = fmaf(q2, q2, s2); s2 = fmaf(q3, q3, s2);
  }
  BN_STAMP(1);
  double a = (double)s1, b = (double)s2;
  block_sum2(a, b, sm);
  __shared__ double2 s_part;
  bool barrier_ok = true;
  if (g.cluster) {
    if (threadIdx.x == 0) s_part = make_double2(a, b);
    BN_STAMP(2);
    bn_cluster_arrive();
    bn_cluster_wait();
  } else {
    if (threadIdx.x == 0) ws.partial[c * BN_MAX_SPLIT + s] = make_double2(a, b);
    BN_STAMP(2);
    barrier_ok = channel_barrier(ws, c, g.S, me, &s_ok);
  }
  BN_STAMP(3);
  // ---- phase 2: this channel's statistics (every CTA of the channel computes the same numbers)
  double pa = 0.0, pb = 0.0;
  if ((int)threadIdx.x < g.S) {
    const double2 p = g.cluster ? bn_ld_cluster(&s_part, threadIdx.x) : __ldcg(ws.partial + c * BN_MAX_SPLIT + threadIdx.x);
    pa = p.x; pb = p.y;
  }
  block_sum2(pa, pb, sm);
  if (g.cluster) bn_cluster_arrive();                     // this CTA has read its peers' partials (wait: at the end)
  __shared__ BnChannelStats cs;                           // thread 0 only
  if (threadIdx.x == 0) s_prm = fused_channel_finish(pa, pb, shift, s, c, g, peers, me, tag, R, ga, be, eps, stats_dense, cs);
  __syncthreads();
  BN_STAMP(4);
  // ---- phase 3: normalise the registers
  float4 p = s_prm;
  if (!barrier_ok) p.z = __uint_as_float(0x7FC00000u);     // incomplete statistics must not pass for a result
  // the residual branch: all loads in flight before the first use (one round trip instead of eight)
  float4 rr[BN_FUSED_R];
#pragma unroll
  for (int u = 0; u < BN_FUSED_R; ++u) {
    rr[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (res && threadIdx.x + u * BN_THREADS < n) rr[u] = __ldg(reinterpret_cast<const float4*>(res) + off[u]);
  }
#pragma unroll
  for (int u = 0; u < BN_FUSED_R; ++u) {
    const int i = threadIdx.x + u * BN_THREADS;
    if (i < n) {
      float4 o;
      o.x = fmaf(v[u].x - p.x, p.y, p.z); o.y = fmaf(v[u].y - p.x, p.y, p.z);
      o.z = fmaf(v[u].z - p.x, p.y, p.z); o.w = fmaf(v[u].w - p.x, p.y, p.z);
      if (res) { o.x += rr[u].x; o.y += rr[u].y; o.z += rr[u].z; o.w += rr[u].w; }
      if (act) { o.x = bn_act(o.x, act); o.y = bn_act(o.y, act); o.z = bn_act(o.z, act); o.w = bn_act(o.w, act); }
      reinterpret_cast<float4*>(y)[off[u]] = o;
    }
  }
  if (s == 0 && threadIdx.x == 0)
    fused_channel_book(cs, c, C, me == nullptr, me, running_mean, running_var, rm_old, rv_old, num_batches_tracked, nbt_old,
                       momentum, save_mean, save_invstd, stats_dense, (double)g.B * (double)g.HW);
  BN_STAMP(5);
  if (g.cluster) bn_cluster_wait();                       // nobody leaves while its shared memory may still be read
  // the CTA that finishes the grid last advances this rank's epoch for the next exchange
  if (me && threadIdx.x == 0) {
    __threadfence();
    const unsigned int t = atomicAdd(ws.ticket + BN_MAX_C, 1u);
    if (t == gridDim.x * gridDim.y - 1) {
      ws.ticket[BN_MAX_C] = 0;
      me->epoch = tag;
    }
  }
}


// ---- fused backward for tensors that fit in registers (one rank) -------------------------------------------
// Sums and apply in ONE launch, the mirror image of bn_fwd_fused_kernel: CTA (s, c) loads its slabs of
// dy (masked by the activation's open interval on y), and x once into registers, the S CTAs of a channel
// meet at the per-channel barrier, every CTA combines the channel's sums and writes dx (and the masked
// gradient of the residual branch) from its registers.  dy / x / y are read once instead of twice.
__global__ void __launch_bounds__(BN_THREADS, 2) bn_bwd_fused_kernel(const float* __restrict__ dy,
                                                                     const float* __restrict__ x,
                                                                     const float* __restrict__ y,
                                                                     const float* __restrict__ mean,
                                                                     const float* __restrict__ invstd,
                                                                     const float* __restrict__ gamma,
                                                                     float* __restrict__ dgamma,
                                                                     float* __restrict__ dbeta,
                                                                     float* __restrict__ dx,
                                                                     float* __restrict__ dres, int act, BnGeom g,
                                                                     BnWorkspace ws, const float* __restrict__ beta,
                                                                     const float* __restrict__ dy2) {
  __shared__ double sm[BN_THREADS / 32][2];
  __shared__ int s_ok;
  const int s = blockIdx.x, c = blockIdx.y, C = g.C, L = g.L;
  const int nslab = (g.B - s + g.S - 1) / g.S;
  const int n = nslab * L;
  BN_STAMP(8);
  const float mu = __ldg(mean + c);                         // (the forward's: older than the kernel in front)
  asm volatile("griddepcontrol.wait;" ::: "memory");        // launched programmatically behind the producer of dy
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // the data-gradient conv behind may set up under this kernel
  // ---- phase 1: masked gradient and x into registers, local sums.  All loads (dy, x and the
  // activation's y: 24 128-bit loads per thread, 124 registers) are issued before the first is used -- masking right behind
  // each load serialised eight round trips (measured 4.4 us of this kernel's 10)
  float4 vg[BN_FUSED_R], vx[BN_FUSED_R];
  int off[BN_FUSED_R];
  float s1 = 0.f, s2 = 0.f;
  const float za = act == 3 ? (gamma ? __ldg(gamma + c) : 1.f) * __ldg(invstd + c) : 0.f;
  const float zb = (act == 3 && beta) ? __ldg(beta + c) : 0.f;
#pragma unroll
  for (int u = 0; u < BN_FUSED_R; ++u) {
    const int i = threadIdx.x + u * BN_THREADS;
    off[u] = -1;
    if (i < n) {
      const int k = fdiv(i, g.div_l);
      off[u] = ((s + k * g.S) * C + c) * L + (i - k * L);
    }
  }
  if (dy2) {
    // two gradients of this tensor (conv branch + skip connection): summed here, one round trip ahead of the rest
    float4 t2[BN_FUSED_R];
#pragma unroll
    for (int u = 0; u < BN_FUSED_R; ++u) {
      vg[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      t2[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (off[u] >= 0) {
        vg[u] = __ldg(reinterpret_cast<const float4*>(dy) + off[u]);
        t2[u] = __ldg(reinterpret_cast<const float4*>(dy2) + off[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < BN_FUSED_R; ++u) { vg[u].x += t2[u].x; vg[u].y += t2[u].y; vg[u].z += t2[u].z; vg[u].w += t2[u].w; }
  }
#pragma unroll
  for (int h = 0; h < BN_FUSED_R; h += 8) {
    float4 vy[8];
#pragma unroll
    for (int u = h; u < h + 8; ++u) {
      if (!dy2) vg[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      vx[u] = make_float4(mu, mu, mu, mu);
      vy[u - h] = make_float4(1.f, 1.f, 1.f, 1.f);
      if (off[u] >= 0) {
        if (!dy2) vg[u] = __ldg(reinterpret_cast<const float4*>(dy) + off[u]);
        vx[u] = __ldg(reinterpret_cast<const float4*>(x) + off[u]);
        if (act == 1 || act == 2) vy[u - h] = __ldg(reinterpret_cast<const float4*>(y) + off[u]);
      }
    }
#pragma unroll
    for (int u = h; u < h + 8; ++u) {
      if (act == 3) {
        vg[u].x *= bn_silu_slope(vx[u].x, mu, za, zb); vg[u].y *= bn_silu_slope(vx[u].y, mu, za, zb);
        vg[u].z *= bn_silu_slope(vx[u].z, mu, za, zb); vg[u].w *= bn_silu_slope(vx[u].w, mu, za, zb);
      } else if (act) {
        const float4 m4 = vy[u - h];
        vg[u].x = bn_act_open(m4.x, act) ? vg[u].x : 0.f; vg[u].y = bn_act_open(m4.y, act) ? vg[u].y : 0.f;
        vg[u].z = bn_act_open(m4.z, act) ? vg[u].z : 0.f; vg[u].w = bn_act_open(m4.w, act) ? vg[u].w : 0.f;
      }
    }
  }
#pragma unroll
  for (int u = 0; u < BN_FUSED_R; ++u) {
    s1 += (vg[u].x + vg[u].y) + (vg[u].z + vg[u].w);
    s2 = fmaf(vg[u].x, vx[u].x - mu, s2); s2 = fmaf(vg[u].y, vx[u].y - mu, s2);
    s2 = fmaf(vg[u].z, vx[u].z - mu, s2); s2 = fmaf(vg[u].w, vx[u].w - mu, s2);
  }
  BN_STAMP(9);
  double a = (double)s1, b = (double)s2;
  block_sum2(a, b, sm);
  __shared__ double2 s_part;
  bool barrier_ok = true;
  if (g.cluster) {
    if (threadIdx.x == 0) s_part = make_double2(a, b);
    BN_STAMP(10);
    bn_cluster_arrive();
    bn_cluster_wait();
  } else {
    if (threadIdx.x == 0) ws.partial[c * BN_MAX_SPLIT + s] = make_double2(a, b);
    BN_STAMP(10);
    barrier_ok = channel_barrier(ws, c, g.S, nullptr, &s_ok);
  }
  BN_STAMP(11);
  // ---- phase 2: the channel's sums (every CTA of the channel computes the same numbers)
  double pa = 0.0, pb = 0.0;
  if ((int)threadIdx.x < g.S) {
    const double2 p = g.cluster ? bn_ld_cluster(&s_part, threadIdx.x) : __ldcg(ws.partial + c * BN_MAX_SPLIT + threadIdx.x);
    pa = p.x; pb = p.y;
  }
  block_sum2(pa, pb, sm);                                   // valid in warp 0: broadcast through shared memory
  if (g.cluster) bn_cluster_arrive();                       // this CTA has read its peers' partials (wait: at the end)
  __shared__ double s_tot[2];
  if (threadIdx.x == 0) { s_tot[0] = pa; s_tot[1] = pb; }
  __syncthreads();
  pa = s_tot[0]; pb = s_tot[1];
  const double is = (double)__ldg(invstd + c), M = (double)g.B * (double)g.HW;
  const float sg = (float)pa, sgx = (float)pb;              // the values the two-kernel form passes through `sums`
  if (s == 0 && threadIdx.x == 0) {
    if (dbeta) dbeta[c] = sg;
    if (dgamma) dgamma[c] = (float)(pb * is);
  }
  const float ga = gamma ? __ldg(gamma + c) : 1.0f;
  float p_y = (float)((double)sg / M), p_z = (float)(is * is * (double)sgx / M);
  const float p_w = (float)((double)ga * is);
  if (!barrier_ok) p_y = __uint_as_float(0x7FC00000u);      // incomplete sums must not pass for a result
  BN_STAMP(12);
  // ---- phase 3: dx from the registers
#pragma unroll
  for (int u = 0; u < BN_FUSED_R; ++u) {
    const int i = threadIdx.x + u * BN_THREADS;
    if (i < n) {
      float4 o;
      o.x = (vg[u].x - p_y - (vx[u].x - mu) * p_z) * p_w; o.y = (vg[u].y - p_y - (vx[u].y - mu) * p_z) * p_w;
      o.z = (vg[u].z - p_y - (vx[u].z - mu) * p_z) * p_w; o.w = (vg[u].w - p_y - (vx[u].w - mu) * p_z) * p_w;
      reinterpret_cast<float4*>(dx)[off[u]] = o;
      if (dres) reinterpret_cast<float4*>(dres)[off[u]] = vg[u];
    }
  }
  BN_STAMP(13);
  if (g.cluster) bn_cluster_wait();                         // nobody leaves while its shared memory may still be read
}

// ---- host side ---------------------------------------------------------------------------------------
static int bn_sms() { return device_sm_count(); }        // per device (po2_common.cuh)

static bool aligned16(const void* p) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

static int bn_geom(BnGeom& g, int B, int C, int HW, bool vec_ok) {
  if (B <= 0 || C <= 0 || HW <= 0) return PO2_E_SIZE;
  if ((int64_t)B * C * HW >= (int64_t)1 << 31) return PO2_E_SIZE;
  if (C > BN_MAX_C) return PO2_E_UNSUPPORTED;
  g.B = B; g.C = C; g.HW = HW; g.cluster = 0;
  const bool vec = vec_ok && (HW % 4 == 0);
  g.L = vec ? HW / 4 : HW;
  g.total = B * C * g.L;
  int S = (4 * bn_sms() + C - 1) / C;                         // ~4 reduce CTAs per SM over all channels
  const int per_cta = BN_UNROLL * BN_THREADS;                 // do not split below one full pass per CTA
  const int max_useful = (int)(((int64_t)B * g.L + per_cta - 1) / per_cta);
  if (S > max_useful) S = max_useful;
  if (S > B) S = B;
  if (S > BN_MAX_SPLIT) S = BN_MAX_SPLIT;
  if (S < 1) S = 1;
  g.S = S;
  g.div_l = make_fastdiv((uint32_t)g.L);
  g.div_c = make_fastdiv((uint32_t)C);
  return vec ? 1 : 0;
}

static BnWorkspace bn_ws(void* workspace, int C) {
  // the ticket counters sit at a FIXED place (they must stay zero between calls of any C); the
  // partial sums behind them are scratch
  BnWorkspace ws;
  (void)C;
  ws.ticket = reinterpret_cast<unsigned int*>(workspace);
  ws.depart = ws.ticket + (BN_MAX_C + 4);
  ws.partial = reinterpret_cast<double2*>(reinterpret_cast<uint8_t*>(workspace) + 2 * (BN_MAX_C + 4) * sizeof(unsigned int));
  return ws;
}

// peers: host array of `world` device pointers (every rank's mailbox as mapped in this process)
static int make_peers(BnPeers& p, void* const* peers, int rank, int world) {
  p.rank = 0; p.world = 0;
  for (int i = 0; i < BN_MAX_RANKS; ++i) p.box[i] = nullptr;
  if (!peers || world <= 1) return 0;
  if (world > BN_MAX_RANKS || rank < 0 || rank >= world) return PO2_E_SIZE;
  for (int i = 0; i < world; ++i) {
    if (!peers[i]) return PO2_E_NULL;
    p.box[i] = reinterpret_cast<BnMailbox*>(peers[i]);
  }
  p.rank = rank; p.world = world;
  return 0;
}

static int elementwise_grid(const BnGeom& g) {
  const int per_cta = BN_UNROLL * BN_THREADS;
  int64_t ctas = ((int64_t)g.total + per_cta - 1) / per_cta;
  const int64_t cap = (int64_t)bn_sms() * 16;
  if (ctas > cap) ctas = cap;
  return (int)(ctas < 1 ? 1 : ctas);
}

// bn_reduce_kernel launches (optionally as a programmatic dependent of the kernel in front: PO2_BN_REDUCE_PDL=1)
template <typename... KArgs, typename... Args>
static cudaError_t launch_reduce(void (*kern)(KArgs...), dim3 grid, cudaStream_t st, Args... args) {
  static const bool pdl = []() { const char* e = getenv("PO2_BN_REDUCE_PDL"); return e && e[0] == '1'; }();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(BN_THREADS);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

}  // namespace po2

using namespace po2;

#ifdef PO2_BN_TRACE
extern "C" int po2_debug_set_bn_trace(void* p) {
  unsigned long long* q = (unsigned long long*)p;
  return (int)cudaMemcpyToSymbol(po2::g_bn_trace, &q, sizeof(q));
}
#endif

extern "C" {

size_t po2_bn_workspace_bytes(int C) {
  if (C <= 0) return 0;
  return (size_t)2 * (BN_MAX_C + 4) * sizeof(unsigned int) + (size_t)C * BN_MAX_SPLIT * sizeof(double2);
}

size_t po2_bn_mailbox_bytes(void) { return sizeof(BnMailbox); }

int po2_bn_stats(const void* x, int B, int C, int HW, float* stat, void* workspace, size_t workspace_bytes,
                 void* const* peers, int rank, int world, void* stream) {
  if (!x || !stat || !workspace) return PO2_E_NULL;
  if (workspace_bytes < po2_bn_workspace_bytes(C)) return PO2_E_WORKSPACE;
  if (!aligned16(workspace)) return PO2_E_ALIGN;
  BnGeom g;
  const int v = bn_geom(g, B, C, HW, aligned16(x));
  if (v < 0) return v;
  BnPeers pr;
  const int pe = make_peers(pr, peers, rank, world);
  if (pe) return pe;
  const BnWorkspace ws = bn_ws(workspace, C);
  const dim3 grid(g.S, C);
  cudaStream_t st = (cudaStream_t)stream;
  const float* xf = (const float*)x;
  cudaError_t e_launch;
  if (v) e_launch = launch_reduce(bn_reduce_kernel<true, 0>, grid, st, xf, nullptr, nullptr, nullptr, nullptr, stat, nullptr, nullptr, g, ws, pr, 0, nullptr, nullptr, nullptr);
  else e_launch = launch_reduce(bn_reduce_kernel<false, 0>, grid, st, xf, nullptr, nullptr, nullptr, nullptr, stat, nullptr, nullptr, g, ws, pr, 0, nullptr, nullptr, nullptr);
  return (int)e_launch;
}

int po2_bn_apply(const void* x, const void* residual, void* y, const float* stats, int R, void* mailbox,
                 float* stats_dense, const float* gamma, const float* beta, float* running_mean,
                 float* running_var, long long* num_batches_tracked, float momentum, float eps, int act,
                 int use_running, float* save_mean, float* save_invstd, int B, int C, int HW, void* stream) {
  if (!x || !y) return PO2_E_NULL;
  if (use_running ? (!running_mean || !running_var) : ((!stats && !mailbox) || R < 1)) return PO2_E_NULL;
  if (R > BN_MAX_RANKS && mailbox) return PO2_E_SIZE;
  if (act < 0 || act > 3) return PO2_E_MODE;
  BnGeom g;
  const int v = bn_geom(g, B, C, HW, aligned16(x) && aligned16(y) && aligned16(residual));
  if (v < 0) return v;
  const size_t smem = (size_t)C * sizeof(float4);
  cudaStream_t st = (cudaStream_t)stream;
  auto kern = v ? bn_apply_kernel<true> : bn_apply_kernel<false>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)elementwise_grid(g));
  cfg.blockDim = dim3(BN_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = use_running ? 0 : 1;                       // train mode: directly behind po2_bn_stats
  return (int)cudaLaunchKernelEx(&cfg, kern, (const float*)x, (const float*)residual, (float*)y, stats, R,
                                 (BnMailbox*)mailbox, stats_dense, gamma, beta, running_mean, running_var,
                                 num_batches_tracked, momentum, eps, act, use_running, save_mean, save_invstd, g);
}

// One-launch kernels: the S CTAs of a channel as one thread-block cluster when 2 <= S <= 16 (hardware co-scheduling
// and barrier; an ordinary launch), else -- or when the cluster launch is refused -- a cooperative launch with the
// global per-channel barrier.  g (inside args) gets its `cluster` flag here.
// The one-launch norm kernels as programmatic dependents of the conv in front (they wait before their first tensor
// load): measured 2.49 vs 2.32 ms per ResNet-56 step -- their CTAs need every register of an SM, scheduled early they
// only stand in the way of the conv's tail -- so it is off unless PO2_BN_PDL=1.  (The other direction, the conv as a
// dependent of the norm, is what pays: po2_conv.cu, pdl_chain_enabled.)
static bool bn_pdl() {
  static const bool on = []() { const char* e = getenv("PO2_BN_PDL"); return e && e[0] == '1'; }();
  return on;
}
static cudaError_t launch_bn_one(const void* kern, BnGeom& g, int C, void** args, cudaStream_t st) {
  // Measured on the ResNet-56 step: clusters of 4 (the 32-channel layers) take ~1.2 us off each kernel (2.53 -> 2.47 ms
  // per step); clusters of 16 (the 16-channel layers) halve the barrier inside the kernel too, but gang-scheduling 16
  // CTAs = 8 whole SMs of one GPC behind another kernel costs ~5 us per launch (2.60 ms): portable sizes only.
  static const int smax = []() { const char* e = getenv("PO2_BN_CLUSTER"); return e ? atoi(e) : 8; }();   // 0: off
  if (g.S >= 2 && g.S <= smax && g.S <= 16) {
    static PerDeviceOnce once_f, once_b;
    PerDeviceOnce& once = kern == (const void*)bn_fwd_fused_kernel ? once_f : once_b;
    cudaError_t e = once.run([kern]() -> cudaError_t {
      return cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    });
    if (e == cudaSuccess) {
      g.cluster = 1;
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(g.S, C);
      cfg.blockDim = dim3(BN_THREADS);
      cfg.stream = st;
      cudaLaunchAttribute attr[2];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = (unsigned)g.S; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // both kernels wait before they read tensors
      attr[1].val.programmaticStreamSerializationAllowed = 1;
      cfg.attrs = attr;
      cfg.numAttrs = bn_pdl() ? 2 : 1;
      e = cudaLaunchKernelExC(&cfg, kern, args);
      if (e == cudaSuccess) return e;
    }
    (void)cudaGetLastError();                            // cluster shape not schedulable here: the global barrier form
  }
  g.cluster = 0;
  if (g.S == 1) {
    // one CTA per channel: no barrier between CTAs, an ordinary launch (optionally programmatic)
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(1, C);
    cfg.blockDim = dim3(BN_THREADS);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = bn_pdl() ? 1 : 0;
    return cudaLaunchKernelExC(&cfg, kern, args);
  }
  return cudaLaunchCooperativeKernel(kern, dim3(g.S, C), dim3(BN_THREADS), args, 0, st);
}

int po2_bn_fwd_fused(const void* x, const void* residual, void* y, const float* gamma, const float* beta,
                     float* running_mean, float* running_var, long long* num_batches_tracked, float momentum,
                     float eps, int act, float* save_mean, float* save_invstd, float* stats_dense, int B, int C,
                     int HW, void* workspace, size_t workspace_bytes, void* const* peers, int rank, int world,
                     void* stream) {
  if (!x || !y || !workspace) return PO2_E_NULL;
  if (act < 0 || act > 3) return PO2_E_MODE;
  if (workspace_bytes < po2_bn_workspace_bytes(C)) return PO2_E_WORKSPACE;
  if (!aligned16(workspace)) return PO2_E_ALIGN;
  BnGeom g;
  const int v = bn_geom(g, B, C, HW, aligned16(x) && aligned16(y) && aligned16(residual));
  if (v < 0) return v;
  if (v == 0) return PO2_E_UNSUPPORTED;                                   // 128-bit path only
  // one CTA holds at most BN_FUSED_R vectors per thread; all CTAs must be co-resident (2 per SM)
  const int64_t per_cta = (int64_t)BN_FUSED_R * BN_THREADS;
  const int64_t need_s = ((int64_t)B * g.L + per_cta - 1) / per_cta;
  if (need_s > BN_MAX_SPLIT || need_s > B || need_s * C > 2 * (int64_t)bn_sms()) return PO2_E_UNSUPPORTED;
  g.S = (int)need_s;
  // slabs are dealt round-robin: the largest share must fit too
  if ((int64_t)((B + g.S - 1) / g.S) * g.L > per_cta) {
    if (g.S + 1 > BN_MAX_SPLIT || g.S + 1 > B || (int64_t)(g.S + 1) * C > 2 * (int64_t)bn_sms()) return PO2_E_UNSUPPORTED;
    g.S += 1;
    if ((int64_t)((B + g.S - 1) / g.S) * g.L > per_cta) return PO2_E_UNSUPPORTED;
  }
  BnPeers pr;
  const int pe = make_peers(pr, peers, rank, world);
  if (pe) return pe;
  const BnWorkspace ws = bn_ws(workspace, C);
  // The CTAs of a channel wait for each other (channel_barrier): launch COOPERATIVELY, so the runtime
  // guarantees that the whole grid is co-resident -- also when another stream (a NCCL kernel, another
  // process under MPS) holds SMs -- or refuses the launch, in which case the caller takes the
  // statistics + apply pair.
  const float *xf = (const float*)x, *rf = (const float*)residual;
  float* yf = (float*)y;
  BnWorkspace wsv = ws;
  void* args[] = {&xf, &rf, &yf, &gamma, &beta, &running_mean, &running_var, &num_batches_tracked, &momentum, &eps, &act,
                  &save_mean, &save_invstd, &stats_dense, &g, &wsv, &pr};
  const cudaError_t e = launch_bn_one((const void*)bn_fwd_fused_kernel, g, C, args, (cudaStream_t)stream);
  if (e == cudaErrorCooperativeLaunchTooLarge) {
    (void)cudaGetLastError();
    return PO2_E_UNSUPPORTED;
  }
  return (int)e;
}

// Backward of the same layer as ONE launch (one rank, tensors that fit the CTAs' registers): sums + apply.
// PO2_E_UNSUPPORTED: take po2_bn_bwd_reduce + po2_bn_bwd_apply.
int po2_bn_bwd_fused(const void* dy, const void* dy2, const void* x, const void* y, const float* save_mean,
                     const float* save_invstd, const float* gamma, const float* beta, float* dgamma, float* dbeta, void* dx,
                     void* dres, int act, int B, int C, int HW, void* workspace, size_t workspace_bytes, void* stream) {
  if (!dy || !x || !save_mean || !save_invstd || !dx || !workspace) return PO2_E_NULL;
  if (act < 0 || act > 3 || (act == 3 && dres)) return PO2_E_MODE;      // SiLU: only without a residual branch
  if ((act == 1 || act == 2) && !y) return PO2_E_NULL;
  if (workspace_bytes < po2_bn_workspace_bytes(C)) return PO2_E_WORKSPACE;
  if (!aligned16(workspace)) return PO2_E_ALIGN;
  BnGeom g;
  const int v = bn_geom(g, B, C, HW, aligned16(dy) && aligned16(dy2) && aligned16(x) && aligned16(y) && aligned16(dx) && aligned16(dres));
  if (v < 0) return v;
  if (v == 0) return PO2_E_UNSUPPORTED;                                   // 128-bit path only
  const int64_t per_cta = (int64_t)BN_FUSED_R * BN_THREADS;
  int64_t need_s = ((int64_t)B * g.L + per_cta - 1) / per_cta;
  for (int attempt = 0; attempt < 2; ++attempt, ++need_s) {
    if (need_s > BN_MAX_SPLIT || need_s > B || need_s * C > 2 * (int64_t)bn_sms()) return PO2_E_UNSUPPORTED;
    if ((int64_t)((B + need_s - 1) / need_s) * g.L <= per_cta) break;     // slabs are dealt round-robin: largest share fits
    if (attempt == 1) return PO2_E_UNSUPPORTED;
  }
  g.S = (int)need_s;
  BnWorkspace wsv = bn_ws(workspace, C);
  const float *df = (const float*)dy, *xf = (const float*)x, *yf = (const float*)y, *d2f = (const float*)dy2;
  float *dxf = (float*)dx, *drf = (float*)dres;
  void* args[] = {&df, &xf, &yf, &save_mean, &save_invstd, &gamma, &dgamma, &dbeta, &dxf, &drf, &act, &g, &wsv, &beta, &d2f};
  const cudaError_t e = launch_bn_one((const void*)bn_bwd_fused_kernel, g, C, args, (cudaStream_t)stream);
  if (e == cudaErrorCooperativeLaunchTooLarge) {
    (void)cudaGetLastError();
    return PO2_E_UNSUPPORTED;
  }
  return (int)e;
}

int po2_bn_bwd_reduce(const void* dy, const void* dy2, const void* x, const void* y, const float* save_mean,
                      const float* save_invstd, const float* gamma, const float* beta, float* sums, float* dgamma,
                      float* dbeta, int act, int B, int C, int HW, void* workspace, size_t workspace_bytes,
                      void* const* peers, int rank, int world, void* stream) {
  if (!dy || !x || !save_mean || !save_invstd || !sums || !workspace) return PO2_E_NULL;
  if (act < 0 || act > 3) return PO2_E_MODE;
  if ((act == 1 || act == 2) && !y) return PO2_E_NULL;
  if (workspace_bytes < po2_bn_workspace_bytes(C)) return PO2_E_WORKSPACE;
  if (!aligned16(workspace)) return PO2_E_ALIGN;
  BnGeom g;
  const int v = bn_geom(g, B, C, HW, aligned16(dy) && aligned16(dy2) && aligned16(x) && aligned16(y));
  if (v < 0) return v;
  BnPeers pr;
  const int pe = make_peers(pr, peers, rank, world);
  if (pe) return pe;
  const BnWorkspace ws = bn_ws(workspace, C);
  const dim3 grid(g.S, C);
  cudaStream_t st = (cudaStream_t)stream;
  const float *xf = (const float*)x, *df = (const float*)dy, *yf = (const float*)y, *d2f = (const float*)dy2;
  cudaError_t e_launch;
  if (act != 0) {
    if (v) e_launch = launch_reduce(bn_reduce_kernel<true, 2>, grid, st, xf, df, yf, save_mean, save_invstd, sums, dgamma, dbeta, g, ws, pr, act, gamma, beta, d2f);
    else e_launch = launch_reduce(bn_reduce_kernel<false, 2>, grid, st, xf, df, yf, save_mean, save_invstd, sums, dgamma, dbeta, g, ws, pr, act, gamma, beta, d2f);
  } else {
    if (v) e_launch = launch_reduce(bn_reduce_kernel<true, 1>, grid, st, xf, df, yf, save_mean, save_invstd, sums, dgamma, dbeta, g, ws, pr, act, nullptr, nullptr, d2f);
    else e_launch = launch_reduce(bn_reduce_kernel<false, 1>, grid, st, xf, df, yf, save_mean, save_invstd, sums, dgamma, dbeta, g, ws, pr, act, nullptr, nullptr, d2f);
  }
  return (int)e_launch;
}

int po2_bn_bwd_apply(const void* dy, const void* dy2, const void* x, const void* y, const float* save_mean,
                     const float* save_invstd, const float* gamma, const float* beta, const float* sums, const float* stats,
                     int R, void* mailbox, void* dx, void* dres, int act, int B, int C, int HW, void* stream) {
  if (!dy || !x || !save_mean || !save_invstd || (!sums && !mailbox) || !stats || !dx || R < 1) return PO2_E_NULL;
  if (R > BN_MAX_RANKS && mailbox) return PO2_E_SIZE;
  if (act < 0 || act > 3 || (act == 3 && dres)) return PO2_E_MODE;      // SiLU: only without a residual branch
  if ((act == 1 || act == 2) && !y) return PO2_E_NULL;
  BnGeom g;
  const int v = bn_geom(g, B, C, HW, aligned16(dy) && aligned16(dy2) && aligned16(x) && aligned16(y) && aligned16(dx) && aligned16(dres));
  if (v < 0) return v;
  const size_t smem = (size_t)C * (sizeof(float4) + sizeof(float));
  cudaStream_t st = (cudaStream_t)stream;
  auto kern = v ? bn_bwd_apply_kernel<true> : bn_bwd_apply_kernel<false>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)elementwise_grid(g));
  cfg.blockDim = dim3(BN_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;   // directly behind po2_bn_bwd_reduce
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return (int)cudaLaunchKernelEx(&cfg, kern, (const float*)dy, (const float*)x, (const float*)y, save_mean, save_invstd,
                                 gamma, sums, stats, R, (BnMailbox*)mailbox, (float*)dx, (float*)dres, act, g, beta,
                                 (const float*)dy2);
}

}  // extern "C"
