/*
 * po2_b200.h -- C ABI of libpo2b200.so: the B200 (sm_100a) implementation of the
 * mschoenb97/po2_quantization hot path (PO2 / PO2+ quantizers + quantized-conv forward).
 *
 * The reference has no native interface for this path: it is ~13 ATen calls per tensor in
 * utils/quantizers.py and one F.conv2d in models/quantized_conv.py.  Each entry point below
 * names the reference lines whose *body* it replaces; INTEGRATION.md shows the ctypes binding a
 * maintainer of the reference would add.
 *
 * Conventions (all entry points)
 *   - every pointer is a DEVICE pointer owned by the caller; the library allocates nothing and
 *     keeps no reference after the call returns;
 *   - work is enqueued on `stream` (a CUstream / cudaStream_t passed as void*), never
 *     synchronised, and is CUDA-graph capturable;
 *   - return value: 0 = success, > 0 = a cudaError_t from the launch, < 0 = PO2_E_* argument
 *     error.  Nothing throws or exits;
 *   - alignment: any 4-byte-aligned fp32 tensor is accepted, except where the kernel a conv entry point
 *     picks reads it with 128-bit loads or a tensor map.  Then po2_conv2d_fwd(_ep), po2_conv2d_fwd_packed(_ep),
 *     po2_qconv2d_fwd, po2_conv2d_dgrad(_packed) and po2_conv2d_wgrad(_z) return PO2_E_ALIGN, before any
 *     launch, unless x (the output gradient for the data gradient; both x and the output gradient for the
 *     weight gradient) starts on a 16-byte boundary.  That is the tcgen05 forward / data gradient at
 *     stride 1 with W % 4 == 0 (W = H*W for 1x1), or on a 1x1 feature map with C % 4 == 0, and the
 *     tcgen05 weight gradients (po2_conv2d_wgrad_kernel_kind 1 or 2) at W % 4 == 0.  The direct,
 *     depthwise and small-pointwise kernels take x at any alignment; the small-pointwise one
 *     (po2_conv2d_kernel_kind 4) needs a 16-byte-aligned fp32 weight when C % 4 == 0.  A bf16 x (the _dt forward
 *     entry points) carries 8 pixels per 16 bytes, so the same rule reads W % 8 == 0 (W = H*W for 1x1) and, on a
 *     1x1 feature map, C % 8 == 0; any 2-byte-aligned bf16 x is accepted otherwise;
 *   - re-entrant; the only process-global state is lazily cached device attributes;
 *   - element counts are 64-bit (the quantizer sweep reaches 2^32 elements).
 */
#ifndef PO2_B200_H_
#define PO2_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* storage dtypes of x / y (the arithmetic is integer exponent/mantissa work on these bits) */
enum { PO2_F32 = 0, PO2_BF16 = 1, PO2_F16 = 2 };

/* quantizer: utils/quantizers.py:19-36 (PowerOfTwoQuantizer), :39-56 (PowerOfTwoPlusQuantizer) */
enum { PO2_MODE_PO2 = 0, PO2_MODE_PO2_PLUS = 1 };

/* which float log2 the rounding boundaries reproduce (tools/scan_boundaries.py):
 *   IEEE       = correctly rounded log2 == torch's CPU kernels (the reference on a CPU);
 *   TORCH_CUDA = torch's CUDA log2f / scalar-division kernels (the reference on a GPU).     */
enum { PO2_FLAVOR_IEEE = 0, PO2_FLAVOR_TORCH_CUDA = 1 };

/* weight formats accepted by po2_conv2d_fwd */
enum {
  PO2_W_F32_PO2 = 0,  /* fp32 values already on the grid +-scale*2^q (what quantize writes)   */
  PO2_W_CODES = 1     /* packed sign+exponent codes (po2_quantize's `codes`) + scale           */
};

enum {
  PO2_E_DTYPE = -1, PO2_E_BITS = -2, PO2_E_NULL = -3, PO2_E_SIZE = -4, PO2_E_ALIGN = -5,
  PO2_E_SHAPE = -6, PO2_E_FLAVOR = -7, PO2_E_WORKSPACE = -8, PO2_E_MODE = -9,
  PO2_E_UNSUPPORTED = -10
};

int po2_abi_version(void);
/* static string for any return code of this library (also maps cudaError_t values) */
const char* po2_error_string(int code);
/* 1 if the torch_cuda boundary table was scanned on hardware and compiled in */
int po2_have_torch_cuda_table(void);

/* Bytes of zero-initialised device scratch that po2_absmax / po2_quantize_fused need.  The
 * kernels leave it zeroed again, so one cudaMemset at allocation time is enough; it must not be
 * shared by calls that can run concurrently (one per stream). */
size_t po2_workspace_bytes(void);

/* scale = max(abs(x))        -- utils/quantizers.py:23, :43 (torch.max(torch.abs(input))).
 * NaN propagates (any NaN -> scale NaN), as torch.max does.  n == 0 -> PO2_E_SIZE (torch raises). */
int po2_absmax(const void* x, int64_t n, int dtype, float* scale_out, void* workspace,
               void* stream);

/* y = 2^clamp(round(log2|x/scale|), fsr-2^(bits-1), fsr-1) * sign(x) * scale
 *                            -- utils/quantizers.py:22-32 (mode 0) / :42-52 (mode 1), bit-exact.
 * codes (optional): packed sign+exponent codes, bits<=4 two per byte (element 2i in the low
 *   nibble), else one per byte; code = signbit<<(bits-1) | ((fsr-1)-q).
 * zero_count (optional, caller-zeroed u32): number of inputs equal to +-0; those produce y = +0
 *   (the reference's sign() is 0) but have no code of their own and are emitted as (+, min level).
 *   A u32: an input with 2^32 or more zeros wraps it (the count is modulo 2^32).
 * sse (optional, caller-zeroed double): accumulates sum((y-x)^2) -- models/quantized_conv.py:43,
 *   utils/quantizers.py:149.
 * bits in [2, 8].  x, y 16-byte aligned for the vector path (any alignment is accepted). */
int po2_quantize(const void* x, void* y, void* codes, unsigned int* zero_count, double* sse,
                 const float* scale, int64_t n, int dtype, int bits, int fsr, int mode,
                 int flavor, void* stream);

/* absmax + quantize in one call (what Quantizer.forward does): one register-resident
 * cooperative launch when the tensor fits on chip, otherwise two streaming passes. */
int po2_quantize_fused(const void* x, void* y, void* codes, unsigned int* zero_count,
                       double* sse, float* scale_out, int64_t n, int dtype, int bits, int fsr,
                       int mode, int flavor, void* workspace, void* stream);

/* how many kernels po2_quantize_fused launches for an aligned tensor of n elements (1 or 2) */
int po2_quantize_fused_launches(int64_t n, int dtype);

/* y = +-2^q * scale from packed codes (inverse of the `codes` output above) */
int po2_dequantize(const void* codes, const float* scale, void* y, int64_t n, int dtype,
                   int bits, int fsr, void* stream);

/* Straight-through estimator -- utils/quantizers.py:34-36, :54-56: grad_input = grad_output.
 * accumulate = 0: gx = g;  accumulate = 1: gx += g (fused .grad accumulation). */
int po2_ste_backward(const void* g, void* gx, int64_t n, int dtype, int accumulate,
                     void* stream);

/* out = conv2d(x, W)  -- models/quantized_conv.py:36,38 (nn.Conv2d._conv_forward, bias=None,
 * dilation=1, zero padding).  x: fp32 NCHW (B,C,H,W); out: fp32 NCHW (B,K,P,Q); W: (K,C/groups,R,S)
 * in `w_format`.  compute = 0: tensor cores with bf16 operands where the shape allows (weights exact,
 * activations rounded to bf16), 2: tensor cores with tf32 operands (activations keep 10 mantissa bits --
 * the precision of the reference's own cuDNN default), 1: fp32 CUDA cores everywhere. */
size_t po2_conv2d_workspace(int B, int C, int H, int W, int K, int R, int S, int stride, int pad,
                            int groups, int compute);
/* Which kernel po2_conv2d_fwd runs for a geometry (planning query, no launch): 0 direct fp32 CUDA cores,
 * 1 depthwise, 2 tcgen05 implicit GEMM with the register-fed activation producer, 3 tcgen05 implicit
 * GEMM fed by tensor-map TMA (tf32 operands straight from fp32 NCHW), 4 fp32 CUDA-core GEMM split over a
 * thread-block cluster (1x1 stride-1 layers on feature maps of <= 16 pixels); negative: PO2_E_*. */
int po2_conv2d_kernel_kind(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                           int compute);
int po2_conv2d_fwd(const void* x, const void* w, const float* scale, void* out, int B, int C,
                   int H, int W, int K, int R, int S, int stride, int pad, int groups,
                   int w_format, int bits, int fsr, int compute, void* workspace,
                   size_t workspace_bytes, void* stream);

/* Static weights (post-training-quantized models, test.py:118-130): build the packed bf16 operand of the
 * tensor-core kernel once (po2_conv2d_pack) and run every forward from it (po2_conv2d_fwd_packed: one
 * launch).  The packed layout depends on the full conv geometry including the batch size; pack_bytes
 * returns 0 when the shape is not taken by the tensor-core kernel. */
size_t po2_conv2d_pack_bytes(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                             int compute);
int po2_conv2d_pack(const void* w, const float* scale, void* packed, size_t packed_bytes, int B, int C, int H,
                    int W, int K, int R, int S, int stride, int pad, int groups, int w_format, int bits,
                    int fsr, int compute, void* stream);
int po2_conv2d_fwd_packed(const void* x, const void* packed, const float* scale, void* out, int B, int C,
                          int H, int W, int K, int R, int S, int stride, int pad, int groups, int compute,
                          void* stream);

/* Inference with eval-mode BatchNorm folded into the conv (models/resnet.py:55-71, models/mobilenet.py:29-31 in
 * eval()): out = act(conv(x, W) * ep_a[k] + ep_b[k] + residual), ep_a[k] = gamma / sqrt(running_var + eps),
 * ep_b[k] = beta - running_mean * ep_a[k]; residual (same shape as out) may be NULL; act: 0 none, 1 ReLU, 2 ReLU6,
 * 3 SiLU.  Same arguments as po2_conv2d_fwd / po2_conv2d_fwd_packed otherwise. */
int po2_conv2d_fwd_ep(const void* x, const void* w, const float* scale, void* out, int B, int C, int H, int W, int K,
                      int R, int S, int stride, int pad, int groups, int w_format, int bits, int fsr, int compute,
                      void* workspace, size_t workspace_bytes, const float* ep_a, const float* ep_b,
                      const void* residual, int act, void* stream);
int po2_conv2d_fwd_packed_ep(const void* x, const void* packed, const float* scale, void* out, int B, int C, int H,
                             int W, int K, int R, int S, int stride, int pad, int groups, int compute,
                             const float* ep_a, const float* ep_b, const void* residual, int act, void* stream);

/* The forward of a bf16 model at inference: the same entry points with the storage type of x, out and the residual as
 * `dtype` (PO2_F32: exactly the forms above; PO2_BF16).  Weights, scale, ep_a / ep_b and the packed operand keep their
 * formats: a bf16 weight is handed in as its exact fp32 widening.  A bf16 value is exact as a bf16 tensor-core operand,
 * so a bf16 x runs on the register-fed tcgen05 kernel (kind 2) with bf16 operands in compute 0 and 2 alike (same result;
 * compute 2 never gives the TMA-fed kind 3 here), on the depthwise kernel (kind 1) or the small-pointwise GEMM (kind 4);
 * accumulation and the epilogue are fp32, and out is rounded to bf16 (round to nearest even) once.  Training (the
 * gradients) is fp32 only.  PO2_E_UNSUPPORTED for a bf16 x with compute 1 or a shape that only the direct kernel
 * takes (kind 0); PO2_E_DTYPE for any other dtype.  NULL ep_a / ep_b / residual with act 0 give the plain forms.
 * Alignment of a bf16 x: 16 bytes (8 pixels) where the tcgen05 kernel reads it with 128-bit loads -- stride 1 with
 * W % 8 == 0 (W = H*W for 1x1), or a 1x1 feature map with C % 8 == 0 -- else PO2_E_ALIGN before any launch; the
 * depthwise kernel takes x at any 2-byte alignment. */
size_t po2_conv2d_workspace_dt(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                               int compute, int dtype);
int po2_conv2d_kernel_kind_dt(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                              int compute, int dtype);
size_t po2_conv2d_pack_bytes_dt(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                                int compute, int dtype);
int po2_conv2d_pack_dt(const void* w, const float* scale, void* packed, size_t packed_bytes, int B, int C, int H,
                       int W, int K, int R, int S, int stride, int pad, int groups, int w_format, int bits,
                       int fsr, int compute, int dtype, void* stream);
int po2_conv2d_fwd_ep_dt(const void* x, const void* w, const float* scale, void* out, int B, int C, int H, int W, int K,
                         int R, int S, int stride, int pad, int groups, int w_format, int bits, int fsr, int compute,
                         void* workspace, size_t workspace_bytes, const float* ep_a, const float* ep_b,
                         const void* residual, int act, int dtype, void* stream);
int po2_conv2d_fwd_packed_ep_dt(const void* x, const void* packed, const float* scale, void* out, int B, int C, int H,
                                int W, int K, int R, int S, int stride, int pad, int groups, int compute,
                                const float* ep_a, const float* ep_b, const void* residual, int act, int dtype,
                                void* stream);

/* QuantizedConv2d.forward in QAT mode as one call -- models/quantized_conv.py:34-36: quantize the fp32
 * master weight w (K, C/groups, R, S) with PO2 (mode 0) / PO2+ (mode 1), then convolve.  qw_out receives
 * the quantized weight (what quantize_fn.apply returns), scale_out its scale.  Where the shape allows,
 * the quantizer kernel writes the conv's packed tensor-core operand itself (two launches in total).
 * workspace: po2_conv2d_workspace(...) bytes; quant_workspace: po2_workspace_bytes() zeroed bytes. */
int po2_qconv2d_fwd(const void* x, const void* w, void* qw_out, float* scale_out, void* out, int B, int C,
                    int H, int W, int K, int R, int S, int stride, int pad, int groups, int bits, int fsr,
                    int mode, int flavor, int compute, void* workspace, size_t workspace_bytes,
                    void* quant_workspace, void* stream);

/* The first half of po2_qconv2d_fwd on its own: quantize the master weight (qw_out, scale_out) and emit
 * the packed tensor-core operand (`packed`, po2_conv2d_pack_bytes(...) bytes) for inputs of shape
 * (B, C, H, W).  Weight quantization does not depend on the activations, so a caller can run it for
 * every layer of a model ahead of time on another stream and feed po2_conv2d_fwd_packed.
 * PO2_E_UNSUPPORTED when the shape does not run on the tensor-core kernel. */
int po2_quantize_pack(const void* w, void* qw_out, float* scale_out, void* packed, size_t packed_bytes, int B, int C,
                      int H, int W, int K, int R, int S, int stride, int pad, int groups, int bits, int fsr, int mode,
                      int flavor, int compute, void* quant_workspace, void* stream);

/* Multi-tensor form (SURVEY.md section 8f "next" #4): ONE launch quantizes and packs many weight tensors
 * (one thread-block cluster per tensor).  The caller builds a table of po2_multi_desc_bytes()-sized
 * descriptors in HOST memory with po2_multi_desc_fill (same arguments as po2_quantize_pack; returns the
 * cluster size 1/2/4/8 this tensor needs, or PO2_E_UNSUPPORTED when the layer must take
 * po2_quantize_pack), copies it to the device once, and calls po2_quantize_pack_multi every step with
 * cluster_size = the largest value po2_multi_desc_fill returned.
 * sse_out (device, fp64, may be NULL): receives sum((Q(w) - w)^2) of this tensor on every launch -- the
 * value QuantizedConv2d.get_quantization_error returns (models/quantized_conv.py:40-45) and the models'
 * error walkers sum (train.py:106), produced by the pass that quantizes instead of by 12 more launches. */
size_t po2_multi_desc_bytes(void);
int po2_multi_desc_fill(void* host_table, int index, const void* w, void* qw_out, float* scale_out, void* packed,
                        size_t packed_bytes, int B, int C, int H, int W, int K, int R, int S, int stride, int pad,
                        int groups, int bits, int fsr, int mode, int flavor, int compute, double* sse_out);
int po2_quantize_pack_multi(const void* device_table, int ntensors, int cluster_size, void* stream);

/* The data-gradient operand packed ahead of time: po2_multi_desc_fill_dgrad amends entry `index` of a
 * MultiDesc table so that the multi-tensor quantizer launch of the FORWARD pass also emits the operand of
 * the layer's data-gradient conv (in/out channels swapped, taps rotated; po2_conv2d_dgrad_pack_bytes bytes,
 * 0 = shape not taken); po2_conv2d_dgrad_packed then computes gx = dL/dx in one launch (autograd of
 * models/quantized_conv.py:36 for the stride-1 dense layers). */
size_t po2_conv2d_dgrad_pack_bytes(int B, int C, int H, int W, int K, int R, int S, int pad, int compute);
int po2_multi_desc_fill_dgrad(void* host_table, int index, void* packed_dgrad, size_t packed_bytes, int B, int C, int H,
                              int W, int K, int R, int S, int stride, int pad, int groups, int compute);
int po2_conv2d_dgrad_packed(const void* g, const void* packed, const float* scale, void* gx, int B, int C, int H,
                            int W, int K, int R, int S, int pad, int compute, void* stream);

/* Data gradient of the same conv (SURVEY.md section 8f "next" #2, first half): gx = dL/dx given g = dL/dout,
 * for the stride-1 dense shapes (3x3 pad 1, 1x1 pad 0), on the tensor-core kernel with the
 * channel-transposed, 180-degree-rotated PO2 weights (exact in bf16; g is rounded to bf16).
 * po2_conv2d_dgrad returns PO2_E_UNSUPPORTED for other shapes (the caller keeps aten.convolution_backward), and
 * po2_conv2d_dgrad_workspace returns 0 for exactly the shapes po2_conv2d_dgrad refuses. */
size_t po2_conv2d_dgrad_workspace(int B, int C, int H, int W, int K, int R, int S, int pad, int compute);
int po2_conv2d_dgrad(const void* g, const void* w, const float* scale, void* gx, int B, int C, int H,
                     int W, int K, int R, int S, int stride, int pad, int groups, int w_format,
                     int bits, int fsr, int compute, void* workspace, size_t workspace_bytes, void* stream);

/* Backward of the layer kinds the tensor-core kernels do not take directly (csrc/po2_conv_bwd.cu):
 * po2_dilate2: g (planes, P, Q) -> g_up (planes, 2P, 2Q) with g_up[2p][2q] = g[p][q], zero elsewhere -- both
 * gradients of a STRIDE-2 dense conv are the stride-1 gradients (po2_conv2d_dgrad / po2_conv2d_wgrad) taken with
 * g_up (models/resnet.py:25-50, the four stride-2 layers of ResNet-20/56).  Q must be even, g 8-byte and g_up
 * 16-byte aligned (PO2_E_UNSUPPORTED otherwise).
 * po2_dilate2_into: the same for any size, g (planes, P, Q) -> g_up (planes, H, W) with P == (H - 1) / 2 + 1 and
 * Q == (W - 1) / 2 + 1 (the output of a 3x3 pad 1 or 1x1 pad 0 stride-2 conv on H x W, odd H, W or Q included),
 * any 4-byte alignment; writes every element of g_up.  PO2_E_SHAPE for non-positive or mismatched sizes,
 * PO2_E_SIZE from 2^31 elements of g_up.
 * Depthwise 3x3 pad 1 (models/mobilenet.py:64-74): the data gradient and the deterministic weight gradient;
 * `g` is the output gradient at the INPUT resolution (stride 2: zero-inserted with po2_dilate2 / _into); the
 * workspace's first 16 KB (tickets) must be zero before the first call and are left zero. */
int po2_dilate2(const void* g, void* g_up, int planes, int P, int Q, void* stream);
int po2_dilate2_into(const void* g, void* g_up, int planes, int P, int Q, int H, int W, void* stream);
int po2_conv2d_depthwise_dgrad(const void* g, const void* w, void* gx, int B, int C, int H, int W, void* stream);
size_t po2_conv2d_depthwise_wgrad_workspace(int C);
int po2_conv2d_depthwise_wgrad(const void* g, const void* x, void* gw, int B, int C, int H, int W, void* workspace,
                               size_t workspace_bytes, void* stream);

/* Weight gradient of the same conv (SURVEY.md section 8f "next" #2, second half): gw (K, C, R, S) = dL/dW
 * given g = dL/dout (B, K, P, Q) and the forward input x (B, C, H, W).  QuantizedConv2d's quantizer is
 * a straight-through estimator (utils/quantizers.py:34-36), so this is the gradient of the fp32
 * master weight.  Dense stride-1 shapes (3x3 pad 1, 1x1 pad 0), K <= 128, compute 0 (bf16 operands:
 * x and g rounded to bf16, fp32 accumulation in TMEM, per-CTA partials summed in a fixed order ->
 * deterministic).  PO2_E_UNSUPPORTED for anything else (the caller keeps aten.convolution_backward). */
size_t po2_conv2d_wgrad_workspace(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                                  int compute);
/* planning query: 0 = shape not taken (the caller keeps aten.convolution_backward), 1 = tcgen05 kernel with
 * bf16 operands, 2 = the TMA-fed tf32 kernel (compute == 2, dense stride-1 3x3 with W in {4,8,16,32} / 1x1),
 * 3 = fp32 CUDA-core GEMM for the 1x1 stride-1 layers neither tensor-core kernel takes (K > 128 or C > 256) that
 * are small: B*H*W <= 8192 and B*H*W*C*K <= 2^26, compute 0 or 2, exact fp32 FMA, per-CTA partials summed in a fixed order
 * (deterministic); its workspace (never 0) holds the partials.  Answers without a device. */
int po2_conv2d_wgrad_kernel_kind(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups,
                                 int compute);
/* po2_conv2d_wgrad_z: the same as po2_conv2d_wgrad with `zeroed_tickets` = 8 bytes of device memory that are zero
 * before the first call (left zero by the kernels; not to be shared by calls that may run concurrently): the TMA-fed
 * kernel then adds its per-CTA partial sums itself, in the same fixed order, after a grid barrier (cooperative
 * launch) -- one launch instead of two.  Measured slower than the two launches on the ResNet shapes; the library
 * takes this path only with PO2_WGRAD_FUSED_REDUCE=1 in the environment. */
int po2_conv2d_wgrad_z(const void* g, const void* x, void* gw, int B, int C, int H, int W, int K, int R, int S,
                       int stride, int pad, int groups, int compute, void* workspace, size_t workspace_bytes,
                       void* zeroed_tickets, void* stream);
int po2_conv2d_wgrad(const void* g, const void* x, void* gw, int B, int C, int H, int W, int K, int R, int S,
                     int stride, int pad, int groups, int compute, void* workspace, size_t workspace_bytes,
                     void* stream);

/* lin / lin+ quantizers (SURVEY.md section 8f "next" #1) -- utils/quantizers.py:59-96 (plus = 0), :99-136
 * (plus = 1): per-input-channel uniform quantizer with a power-of-two step refined by num_iters rounds.
 * w, y: fp32 (K, C, R*S) contiguous; one launch.  PO2_E_UNSUPPORTED when K*R*S exceeds
 * po2_lin_max_channel_elems() (the caller keeps the op-by-op form).
 * po2_lin_quantize_dt: the same for w, y of storage `dtype`.  PO2_F32 is exactly po2_lin_quantize; PO2_BF16 (a bf16
 * model's weights) evaluates every op of the reference in fp32 and rounds its result to bf16, as torch does for bf16
 * tensors, and writes a bf16 y.  PO2_E_DTYPE for any other dtype; otherwise the errors of po2_lin_quantize, all
 * before any launch. */
int po2_lin_max_channel_elems(void);
int po2_lin_quantize(const void* w, void* y, int K, int C, int RS, int bits, int num_iters, int plus, int flavor,
                     void* stream);
int po2_lin_quantize_dt(const void* w, void* y, int K, int C, int RS, int bits, int num_iters, int plus, int flavor,
                        int dtype, void* stream);

/* lin / lin+ weights on the tensor-core conv: after num_iters >= 1 rounds every weight is n * 2^k (one power-of-two
 * step per input channel, |n| <= 2^(bits-1) - 1), which is exact as a bf16 operand for bits <= 9 (compute 0) and as
 * a tf32 operand for bits <= 12 (compute 2).  So the packed operand holds y itself and every consumer of
 * (packed, scale) -- po2_conv2d_fwd_packed(_ep / _stats), po2_conv2d_dgrad_packed, po2_conv2d_dgrad -- takes it with a
 * scale of 1.0f.
 * po2_lin_quantize_pack: po2_lin_quantize (y_out bit-identical) that also writes the operand of conv2d(x of shape
 * (B, C, H, W), y) into `packed` (po2_conv2d_pack_bytes bytes) and, if packed_dgrad != NULL, the data-gradient operand
 * (po2_conv2d_dgrad_pack_bytes bytes; stride-1 dense layers).  One launch; two (quantizer + po2_conv2d_pack) when the
 * operand needs channel padding.  PO2_E_UNSUPPORTED: no tensor-core operand for this geometry / compute, bits not
 * exact in it, num_iters < 1, or a channel above po2_lin_max_channel_elems().
 * Multi-tensor form: ONE launch for many lin weights, one CTA per (tensor, input channel).  po2_lin_multi_desc_fill
 * writes entry `index` of a HOST table of po2_lin_multi_desc_bytes()-sized entries (same arguments as
 * po2_lin_quantize_pack; fill in index order 0, 1, ...) and returns the tensor's CTA count C (> 0), or
 * PO2_E_UNSUPPORTED when the layer must take po2_lin_quantize_pack (channel padding).  The caller copies the table
 * to the device once and calls po2_lin_quantize_pack_multi with total_ctas = the sum of the returned counts and
 * max_channel_elems = the largest K*R*S of the table. */
int po2_lin_quantize_pack(const void* w, void* y_out, void* packed, size_t packed_bytes, void* packed_dgrad,
                          size_t packed_dgrad_bytes, int B, int C, int H, int W, int K, int R, int S, int stride, int pad,
                          int groups, int bits, int num_iters, int plus, int flavor, int compute, void* stream);
size_t po2_lin_multi_desc_bytes(void);
int po2_lin_multi_desc_fill(void* host_table, int index, const void* w, void* y_out, void* packed, size_t packed_bytes,
                            void* packed_dgrad, size_t packed_dgrad_bytes, int B, int C, int H, int W, int K, int R,
                            int S, int stride, int pad, int groups, int bits, int num_iters, int plus, int flavor,
                            int compute);
int po2_lin_quantize_pack_multi(const void* device_table, int ntensors, int total_ctas, int max_channel_elems,
                                void* stream);

/* ---- batch normalisation around the quantized convs (SURVEY.md section 8f "next" #3) -----------------
 * The reference models follow every QuantizedConv2d with nn.SyncBatchNorm (+ ReLU, + the residual add):
 * models/resnet.py:38-61, models/mobilenet.py:29-33.  x, y, dy, dx are fp32 [B][C][HW] (NCHW), parameters
 * and statistics fp32 [C].  act: 0 none, 1 ReLU.
 *
 * po2_bn_stats: this rank's batch statistics, stat[0..C) = mean, stat[C..2C) = sum (x-mean)^2,
 *   stat[2C] = B*HW.  workspace: po2_bn_workspace_bytes(C) bytes, zero-initialised once (left zeroed).
 * po2_bn_apply: y = act((x - mean) * invstd * gamma + beta [+ residual]).  stats = R entries of 2C+1
 *   floats (R ranks' po2_bn_stats results, combined with the parallel-variance formula as
 *   torch.batch_norm_gather_stats_with_counts does), or use_running != 0: the running statistics
 *   (eval mode).  In train mode also updates running_mean / running_var (unbiased variance,
 *   `momentum`) and num_batches_tracked when given, and writes save_mean / save_invstd for backward.
 * po2_bn_bwd_reduce: sums[0..C) = sum g, sums[C..2C) = sum g*(x-mean) with g = dy (act 0),
 *   dy*(y>0) (act 1), dy*(0<y<6) (act 2) or dy*silu'(z), z = (x-mean)*gamma*invstd + beta (act 3: SiLU behind the
 *   norm, models/mobile_vit.py:16-22; z is recomputed from x, so gamma / beta are needed and y is not);
 *   dgamma = sums[C+c]*invstd, dbeta = sums[c] (local sums, as SyncBatchNorm).
 *   dy2 (all three backward entries, may be NULL): a second gradient of the same tensor, added on the fly (g is
 *   formed from dy + dy2) -- the gradient that reaches a block's input over its skip connection
 *   (models/resnet.py:69 `out += self.shortcut(x)`), instead of an accumulation kernel in front of the norm's backward.
 * po2_bn_bwd_apply: dx = (g - sum_g/M - (x-mean)*invstd^2*sum_gx/M) * gamma*invstd, M = total count
 *   over the R stats entries; `sums` all-reduced over ranks by the caller.  dres (optional): g, the
 *   gradient of the residual branch behind the ReLU. */
size_t po2_bn_workspace_bytes(int C);
int po2_bn_stats(const void* x, int B, int C, int HW, float* stat, void* workspace, size_t workspace_bytes,
                 void* const* peers, int rank, int world, void* stream);
int po2_bn_apply(const void* x, const void* residual, void* y, const float* stats, int R, void* mailbox,
                 float* stats_dense, const float* gamma, const float* beta, float* running_mean,
                 float* running_var, long long* num_batches_tracked, float momentum, float eps, int act,
                 int use_running, float* save_mean, float* save_invstd, int B, int C, int HW, void* stream);
/* The backward of FusedSyncBatchNorm as ONE launch (one rank; tensors that fit the CTAs' registers, the same
 * condition as po2_bn_fwd_fused): per-channel sums of the activation-masked gradient, dgamma / dbeta, dx and
 * the masked gradient of the residual branch (dres, may be NULL) -- models/resnet.py:55-71 under autograd.
 * Returns PO2_E_UNSUPPORTED when the pair po2_bn_bwd_reduce + po2_bn_bwd_apply has to be used. */
int po2_bn_bwd_fused(const void* dy, const void* dy2, const void* x, const void* y, const float* save_mean,
                     const float* save_invstd, const float* gamma, const float* beta, float* dgamma, float* dbeta, void* dx,
                     void* dres, int act, int B, int C, int HW, void* workspace, size_t workspace_bytes, void* stream);

/* po2_bn_stats + po2_bn_apply in ONE launch for tensors whose per-channel slice fits the registers of
 * the CTAs working on it (the CIFAR-scale layers): x is read once, the CTAs of a channel meet at a
 * barrier in the workspace, statistics are combined (through the mailboxes when world > 1) and y is
 * written from registers.  stats_dense (optional, [world][2C+1]) receives what po2_bn_bwd_apply needs.
 * PO2_E_UNSUPPORTED when the tensor is too large / not 16-byte friendly: use the two-kernel form. */
int po2_bn_fwd_fused(const void* x, const void* residual, void* y, const float* gamma, const float* beta,
                     float* running_mean, float* running_var, long long* num_batches_tracked, float momentum,
                     float eps, int act, float* save_mean, float* save_invstd, float* stats_dense, int B, int C,
                     int HW, void* workspace, size_t workspace_bytes, void* const* peers, int rank, int world,
                     void* stream);
int po2_bn_bwd_reduce(const void* dy, const void* dy2, const void* x, const void* y, const float* save_mean,
                      const float* save_invstd, const float* gamma, const float* beta, float* sums, float* dgamma,
                      float* dbeta, int act, int B, int C, int HW, void* workspace, size_t workspace_bytes,
                      void* const* peers, int rank, int world, void* stream);
int po2_bn_bwd_apply(const void* dy, const void* dy2, const void* x, const void* y, const float* save_mean,
                     const float* save_invstd, const float* gamma, const float* beta, const float* sums, const float* stats,
                     int R, void* mailbox, void* dx, void* dres, int act, int B, int C, int HW, void* stream);

/* Peer exchange (one NVLink domain, <= 8 ranks): SyncBatchNorm's two collectives done by the kernels
 * themselves.  Every rank allocates one zero-initialised mailbox of po2_bn_mailbox_bytes() in memory
 * that its peers have mapped (torch.distributed._symmetric_memory); `peers` is a HOST array of
 * `world` device pointers -- rank r's mailbox as mapped in this process.  With peers != NULL and
 * world > 1, po2_bn_stats / po2_bn_bwd_reduce additionally store this rank's vector into every
 * rank's mailbox (the all_gather / all_reduce over NVLink stores, flagged with an epoch number);
 * po2_bn_apply / po2_bn_bwd_apply given mailbox = this rank's own mailbox (and R = world) wait for
 * the R vectors of the current epoch instead of reading `stats` / `sums` (which may then be NULL;
 * po2_bn_apply copies the gathered statistics to stats_dense[R][2C+1] for the backward call).
 * All ranks must issue the same sequence of exchanges (the rule of any collective). */
size_t po2_bn_mailbox_bytes(void);

/* ---- weight gradient of the full-precision stem (models/resnet.py:99-102 nn.Conv2d(3, 16, 3, 1, 1); autograd of F.conv2d
 * w.r.t. the weight -- the stem's input needs no gradient, so this is its whole backward): 3x3, pad 1, stride 1,
 * C <= 4 input channels, K*C <= 256.  CUDA cores, exact fp32 FMA, one CTA per image + the fixed-order reduce kernel
 * (deterministic).  Workspace: po2_conv2d_stem_wgrad_workspace(...) bytes (0: shape not taken). */
size_t po2_conv2d_stem_wgrad_workspace(int B, int C, int H, int W, int K, int R, int S, int stride, int pad, int groups);
int po2_conv2d_stem_wgrad(const void* g, const void* x, void* gw, int B, int C, int H, int W, int K, int R, int S, int stride,
                          int pad, int groups, void* workspace, size_t workspace_bytes, void* stream);

/* ---- the QAT step's parameter update (train.py:54-56 optim.SGD(lr, momentum, weight_decay), :92 optimizer.step()) ----
 * All parameters in one launch per po2_sgd_max_tensors_per_launch() tensors, torch.optim.SGD's arithmetic rounding by
 * rounding (dampening 0, no Nesterov): g = fma(wd, p, grad); buf = rn(rn(buf*momentum) + g) (first_step: buf = g);
 * p = fma(-lr, buf, p).  params / grads / bufs / numels: HOST arrays of `ntensors` device pointers (fp32,
 * contiguous) and element counts; bufs may be NULL when momentum == 0. */
int po2_sgd_step(void* const* params, const void* const* grads, void* const* bufs, const long long* numels, int ntensors,
                 float lr, float momentum, float weight_decay, int first_step, void* stream);
int po2_sgd_max_tensors_per_launch(void);

#ifdef __cplusplus
}
#endif
#endif /* PO2_B200_H_ */
