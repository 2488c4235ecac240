/* fi_b200.h — C ABI of the B200-native UNet frame-synthesis path (libfi_b200.so).
 *
 * The reference (daultanigaurav/AI-BASED-FRAME-INTERPOLATION) has no FFI: its boundary for this path is the Python
 * module surface of model/unet.py, model/inference.py and model/evaluation.py. Each entry point below names the
 * reference interface it replaces (file:line, relative to the reference root). The Python drop-ins in
 * ai-based-frame-interpolation_b200/model/ bind these symbols with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success or a negative fiStatus; fiLastError() gives the thread-local message;
 *   - nothing aborts or throws across the boundary;
 *   - all pointers are DEVICE pointers unless the parameter name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; calls are stream-ordered and never synchronise, except the
 *     *_host convenience calls (documented below) and fiNetCreate/fiNetLoadWeights/fiNetDestroy;
 *   - a fiNet must not be used from two threads at once (one handle per worker);
 *   - there is no CPU fallback: without a CUDA device every compute call fails with FI_ERR_CUDA.
 */
#ifndef FI_B200_H
#define FI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum fiStatus {
    FI_OK = 0,
    FI_ERR_INVALID = -1, /* bad argument / unsupported shape */
    FI_ERR_CUDA = -2,    /* CUDA runtime or driver error */
    FI_ERR_STATE = -3,   /* e.g. forward before weights are loaded */
    FI_ERR_WEIGHTS = -4, /* missing / mis-sized state-dict entry */
    FI_ERR_NOMEM = -5
} fiStatus;

int fiVersion(void);
const char* fiLastError(void);

/* ------------------------------------------------------------------------------------------------------------------
 * Whole-network handle: replaces UNet / FrameInterpolationUNet (model/unet.py:65-112) in eval mode.
 * ---------------------------------------------------------------------------------------------------------------- */
typedef struct fiNet fiNet;

/* UNet(n_channels, n_classes, bilinear) — model/unet.py:66. n_channels in 1..8, n_classes in 1..4. */
int fiNetCreate(fiNet** out, int device, int n_channels, int n_classes, int bilinear);
int fiNetDestroy(fiNet* net);

/* Arithmetic of the tensor-core convolutions. Call before fiNetLoadWeights (it invalidates loaded weights).
 *   FI_PRECISION_BF16   (default) bf16 operands, fp32 accumulate: max |err| <= 2e-2 in [0,1] pixel units.
 *   FI_PRECISION_FP32X3 the "fp32 path": every activation and weight is a bf16 hi + bf16 lo pair and each MAC is
 *                       x_hi*w_hi + x_hi*w_lo + x_lo*w_hi in fp32 (~16 mantissa bits per operand): <= 1e-3.
 *                       3x the tensor work and 2x the activation bytes of the bf16 path. */
#define FI_PRECISION_BF16 0
#define FI_PRECISION_FP32X3 1
int fiNetSetPrecision(fiNet* net, int precision);

/* load_state_dict (model/inference.py:83-94, schema SURVEY.md A.5). names[i] are state-dict keys with or without the
 * "unet." prefix; data_host[i] is the fp32 host tensor, numel[i] its element count. Eval-mode BatchNorm
 * (model/unet.py:13,16) is folded here: W' = W*gamma/sqrt(var+eps) (rounded once to bf16), b' = beta - mean*scale. */
int fiNetLoadWeights(fiNet* net, const char* const* names, const float* const* data_host, const int64_t* numel,
                     int count);

/* One group of input channel planes: element (n,c,y,x) at ptr[n*batch_stride + c*chan_stride + y*row_stride +
 * x*px_stride] (strides in ELEMENTS). Covers NCHW fp32 tensors, planar u8 frames and interleaved HWC u8 frames. */
typedef struct fiPlanes {
    const void* ptr;
    int64_t batch_stride, chan_stride, row_stride, px_stride;
    int channels;
} fiPlanes;

#define FI_IN_F32 0 /* already-normalised fp32 (what preprocess_image returns, model/inference.py:11-41) */
#define FI_IN_U8 1  /* raw uint8 pixels; u8/255*2-1 is applied in the stem kernel (model/inference.py:32-35) */

/* FrameInterpolationUNet.forward(frame1, frame2) (model/unet.py:105-112) / UNet.forward(x) (model/unet.py:84-95):
 * channels of in0 followed by channels of in1 (in1 may be NULL) form the n_channels input (the torch.cat of
 * unet.py:109 is fused into the stem loader). Outputs, either may be NULL but not both:
 *   out_f32: fp32 NCHW [N, n_classes, H, W] logits (what forward() returns);
 *   out_u8 : uint8 NCHW [N, n_classes, H, W] = postprocess_image(logits) (model/inference.py:43-63). */
int fiNetForward(fiNet* net, const fiPlanes* in0, const fiPlanes* in1, int in_dtype, float* out_f32, uint8_t* out_u8,
                 int N, int H, int W, void* stream);

/* interpolate_frames + postprocess_image with HOST buffers (model/inference.py:101-122, 43-63): planar u8 frames
 * [N, C, H, W] on the host in, u8 [N, n_classes, H, W] on the host out. Copies through internal pinned staging buffers
 * on `stream` and synchronises it before returning. */
int fiNetInterpolateHostU8(fiNet* net, const uint8_t* frame1_host, const uint8_t* frame2_host, int channels_per_frame,
                           uint8_t* out_host, int N, int H, int W, void* stream);

/* Host clips (main.py video; the reference never wrote its video loop, SURVEY.md D3, and has no --fps): frames at
 * dyadic times between the frames of a clip, by recursive bisection on the device. The network has no time input, so
 * node (i, a/2^d) with a odd is the network midpoint of (i, (a-1)/2^d) and (i, (a+1)/2^d), each in lowest terms; (i, 0)
 * is frame i and (i, 1) frame i+1. That is exactly the frame host-side recursive bisection produces (the forward gives
 * the same bits at any batch size). depth = 1 with req_pair = i, req_num = 1 for every pair i (the nodes (i, 1/2)) is
 * the midpoint clip that FrameInterpolator.interpolate_clip and the video loop run.
 *   frames_host: n_frames planar u8 frames [C, H, W], frame_stride bytes apart (each frame contiguous; strides let
 *                interpolate_sequence read every other frame of an interleaved sequence and write the new midpoints
 *                straight between them); C = channels_per_frame, and n_classes must equal C when depth > 1, because
 *                nodes below level 1 are computed from nodes fed back into the network;
 *   request j:   node (req_pair_host[j], req_num_host[j] / 2^depth), depth in 1..6, 0 <= pair < n_frames-1,
 *                0 < num < 2^depth, requests sorted by pair (any order of num, repeats allowed); it is written to
 *                out_host + j*out_stride as u8 [n_classes, H, W].
 * Pairs go in groups of pairs_per_batch; each group's frames are uploaded once, the closure of its requests is evaluated
 * level by level in batches of <= pairs_per_batch images with every node kept in a device pool, and only the requested
 * nodes are copied back. A level-1 batch of consecutive pairs reads its parents where they were uploaded; any other
 * batch gathers them with device-to-device copies. Upload of group g+1 (copy stream), the levels of group g (`stream`)
 * and the download of group g-1 (a second copy stream) overlap through double-buffered pinned staging.
 * pair_sad_host (optional; the reference has no scene detection) receives n_frames-1 uint64 values, pair_sad_host[i] =
 * sum |f[i+1] - f[i]| over all C*H*W bytes (exact), computed by fiPairSadU8 on `stream` from each group's uploaded
 * frames, so the host frames are not read again; with NULL, groups without requests are never uploaded.
 * n_forwards_host (optional) receives the number of images forwarded. Any invalid argument returns FI_ERR_INVALID,
 * naming it, before anything is launched or written. Synchronous: returns when out_host is complete. */
int fiNetInterpolateDyadicHostU8(fiNet* net, const uint8_t* frames_host, int64_t frame_stride, int n_frames,
                                 int channels_per_frame, int H, int W, int depth, const int32_t* req_pair_host,
                                 const int32_t* req_num_host, int n_req, uint8_t* out_host, int64_t out_stride,
                                 int pairs_per_batch, void* stream, uint64_t* pair_sad_host, int64_t* n_forwards_host);

/* Algorithmic FLOPs (2*MACs, no padding) of one forward at this shape, and the number of kernel launches it makes. */
int fiNetForwardCost(fiNet* net, int N, int H, int W, double* flops, int* launches);
/* Measurement hook for bench.py: when enabled, every launch of the following forwards is bracketed by a CUDA event
 * pair on the caller's stream; fiNetGetProfile synchronises the device and returns, per launch of the schedule, the
 * accumulated device time, its algorithmic FLOPs and bytes. kind: 0 = stem conv (CUDA cores), 1 = tcgen05 conv GEMM,
 * 2 = bilinear upsample. Call with out == NULL to query the launch count. */
typedef struct fiLaunchProfile {
    char name[48];
    int kind;
    int calls;
    double flops;
    double bytes;
    double ms_total;
} fiLaunchProfile;
int fiNetSetProfiling(fiNet* net, int enable);
int fiNetGetProfile(fiNet* net, fiLaunchProfile* out, int capacity, int* count);
/* Plan cache: a plan (activation arena + tensor maps + prepared launches) is kept per frame size, most recently used
 * first, at most $FI_PLAN_CACHE (default 4) of them, so alternating shapes — one 256x256 pair per POST /interpolate
 * (reference api/app.py:121-205) between 1080p video batches — neither re-allocate nor re-encode. Outputs (any may be
 * NULL): plans currently cached, plans built since fiNetCreate, bytes of device memory held by their arenas. */
int fiNetPlanStats(fiNet* net, int* cached, long long* builds, size_t* arena_bytes);
/* Debug tap: copy an intermediate activation (bf16 NHWC) of the last forward to the host as fp32 NCHW.
 * name in {inc, down1..down4, up1..up4 (block outputs), up1.up..up4.up (upsampled tensors)}. */
int fiNetReadActivation(fiNet* net, const char* name, float* out_host, int64_t capacity, int* C, int* H, int* W);
/* Device tap: the same activation as fiNetReadActivation (any tensor of the current plan: also pool1..pool4, the
 * .mid tensors, and inc.mid where the stem is its own launch), copied device to device in its own layout, bf16 NHWC [n_last_forward, H, W, C], with cudaMemcpyAsync on
 * `stream` (ordered after the forward enqueued on it). In the fp32-grade mode the lo half goes to dst_lo (required
 * there, ignored otherwise); value = hi + lo. capacity_elems: bf16 elements each of dst and dst_lo can hold. dst NULL:
 * only C, H, W are reported. Refuses a plan with arena reuse (the tensor may be overwritten) and a too-small buffer,
 * like the host tap. */
int fiNetCopyActivation(fiNet* net, const char* name, void* dst, void* dst_lo, int64_t capacity_elems, int* C, int* H,
                        int* W, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Single layers (the same kernels the handle launches), for layer-level parity tests and reuse.
 * ---------------------------------------------------------------------------------------------------------------- */
#define FI_EPI_STORE 0      /* conv3x3+BN+ReLU -> bf16 NHWC                         (DoubleConv, model/unet.py:5-21)  */
#define FI_EPI_STORE_POOL 1 /* ... plus MaxPool2d(2) of the result                  (Down, model/unet.py:23-33)       */
#define FI_EPI_CONVT 2      /* ConvTranspose2d(k=2,s=2)+bias as a 1-tap GEMM        (Up, model/unet.py:43)            */
#define FI_EPI_HEAD 3       /* ... plus Conv2d(64,n_classes,1)+bias (+postprocess)  (OutConv, model/unet.py:57-63)    */

typedef struct fiConvDesc {
    const void* src0;   /* bf16 NHWC [N,H,W,c0] */
    int c0;
    const void* src1;   /* optional: bf16 NHWC [N,h1,w1,c1], placed at (off_y,off_x) of the HxW frame; zero elsewhere.
                           K-range [c0, c0+c1) — the fused F.pad + torch.cat([skip, up]) of model/unet.py:49-54 */
    int c1, h1, w1, off_y, off_x;
    const void* wpack;  /* bf16 [n_total][taps*(c0+c1)], K index = tap*(c0+c1)+channel, tap = 3*ky+kx */
    const float* bias;  /* fp32 [n_total] */
    int n_total;        /* Cout, or 4*Cout ordered (ky,kx,co) for FI_EPI_CONVT */
    int taps;           /* 9 or 1 */
    int mode;           /* FI_EPI_* */
    int relu;
    void* dst;          /* STORE*: bf16 [N,H,W,n_total]; CONVT: bf16 [N,2H,2W,n_total/4] */
    void* dst_pool;     /* STORE_POOL: bf16 [N,H/2,W/2,n_total] */
    const float* head_w; /* HEAD: fp32 [n_classes][64] */
    const float* head_b; /* HEAD: fp32 [n_classes] */
    int n_classes;
    float* out_f32;     /* HEAD: fp32 NCHW [N,n_classes,H,W] or NULL */
    uint8_t* out_u8;    /* HEAD: u8 NCHW or NULL */
    int N, H, W;
    /* precise ("fp32x3") mode: activations are bf16 hi + bf16 lo pairs (value = hi + lo) and the GEMM accumulates
     * x_hi*w_hi + x_hi*w_lo + x_lo*w_hi in fp32. wpack is then bf16 [n_total][taps*3*(c0+c1)], per tap
     * [w0_hi | w0_lo | w0_hi | w1_hi | w1_lo | w1_hi] (w0 / w1 = the weight columns of src0 / src1 channels). */
    int precise;
    const void* src0_lo; /* lo halves, same shapes as src0 / src1 */
    const void* src1_lo;
    void* dst_lo;        /* lo halves of dst / dst_pool (not used by HEAD) */
    void* dst_pool_lo;
} fiConvDesc;

int fiConvGemm(const fiConvDesc* desc, void* stream);

/* inc.double_conv.0..2 (model/unet.py:12-14) on raw planes, computed on the tensor cores with bf16 hi/lo operand
 * splitting (fp32-grade result). wpack: DEVICE bf16 [64][fiStemPackedK(cin)] produced on the host by
 * fiStemPackWeights from the BN-folded fp32 weight [64][cin][3][3]; bias fp32 [64]; dst bf16 NHWC [N,H,W,64]. */
int fiStemPackedK(int cin);
int fiStemPackWeights(const float* w_host, int cin, uint16_t* out_host);
int fiStemConv(const fiPlanes* in0, const fiPlanes* in1, int in_dtype, const void* wpack, const float* bias, void* dst,
               int N, int H, int W, void* stream);
/* Same without the ReLU: the training forward keeps the pre-BatchNorm conv output. */
int fiStemConvLinear(const fiPlanes* in0, const fiPlanes* in1, int in_dtype, const void* wpack, const float* bias,
                     void* dst, int N, int H, int W, void* stream);
/* nn.MaxPool2d(2) (model/unet.py:28) on bf16 NHWC [N,H,W,C] -> [N,H/2,W/2,C]; inside fiNetForward the pool is fused into
 * the producing convolution, this entry point serves the stand-alone Down module. */
int fiMaxPool2x2(const void* src, void* dst, int N, int H, int W, int C, void* stream);
/* nn.Upsample(scale_factor=2, bilinear, align_corners=True) (model/unet.py:40): bf16 NHWC [N,h,w,C] -> [N,2h,2w,C]. */
int fiUpsample2x(const void* src, void* dst, int N, int h, int w, int C, void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Memory-bound kernels of the path.
 * ---------------------------------------------------------------------------------------------------------------- */
/* preprocess_image normalisation (model/inference.py:32-35) + the frame-pair torch.cat (model/unet.py:109):
 * two u8 planar batches [N,C,H,W] -> fp32 NCHW [N,2C,H,W]. */
int fiPackPairU8(const uint8_t* frame1, const uint8_t* frame2, float* out, int N, int C, int H, int W, void* stream);
/* postprocess_image (model/inference.py:43-63) on n fp32 values: trunc(clamp((t+1)/2,0,1)*255). */
int fiHeadPostU8(const float* logits, uint8_t* out, size_t n, void* stream);
/* compute_psnr / compute_ssim (model/evaluation.py:194-218 = evaluation_simple.py:103-109; scikit-image semantics,
 * data_range=255) for N u8 image pairs [N,H,W]: out[2n] = PSNR (dB, +inf when identical), out[2n+1] = SSIM. */
size_t fiSsimPsnrWorkspaceBytes(int N, int H, int W);
int fiSsimPsnrU8(const uint8_t* pred, const uint8_t* target, int N, int H, int W, double* out, void* workspace,
                 void* stream);
/* Scene-cut statistic (what ffmpeg's scdet and RIFE's video script compute on the host; the reference has none):
 * sad[i] = sum over k < frame_bytes of |frames[(i+1)*frame_stride + k] - frames[i*frame_stride + k]| for the n_frames-1
 * consecutive pairs of u8 frames, exact in 64 bit. sad is zeroed on `stream` first. Any alignment and stride work;
 * 16-byte aligned frames take the vector path. FI_ERR_INVALID on NULL pointers, n_frames < 2, frame_bytes < 1 or
 * frame_stride < frame_bytes. */
int fiPairSadU8(const uint8_t* frames, int64_t frame_stride, int64_t frame_bytes, int n_frames, uint64_t* sad,
                void* stream);
/* FrameTripletDataset.__getitem__ + the DataLoader collate (model/train.py:89-151) for frames already on the device:
 * frames u8 [n_frames][H][W], triplets int32 [n_triplets][3] = frame indices of (t0, t1, ground truth), samples int64
 * [n] = triplet indices, all device pointers. frame1[b] = frames[triplets[samples[b]][0]] / 255, frame2 from column 1,
 * target from column 2, each fp32 [n][1][H][W] and bit-identical to img.astype(float32) / 255.0. A sample index outside
 * [0, n_triplets) or a triplet entry outside [0, n_frames) is never dereferenced: that sample's three outputs are NaN.
 * FI_ERR_INVALID on NULL pointers, n < 1, H < 1, W < 1 or negative counts. */
int fiGatherTripletsU8(const uint8_t* frames, int64_t n_frames, const int32_t* triplets, int64_t n_triplets,
                       const int64_t* samples, int n, int H, int W, float* frame1, float* frame2, float* target,
                       void* stream);

/* ------------------------------------------------------------------------------------------------------------------
 * Training step (model/train.py:153-249; SURVEY.md §8f row 2): the kernels around the tensor-core convolutions.
 * Activations / activation gradients: bf16 NHWC [P = N*H*W][C]; statistics, weight gradients, optimizer state: fp32.
 * Conv forward and the data gradient reuse fiConvGemm (the latter with the flipped/transposed weights that
 * fiPackConvWeights writes); the host side of one step is model/train.py:TrainStep.
 * ---------------------------------------------------------------------------------------------------------------- */
/* nn.BatchNorm2d in training mode (model/unet.py:13,16): per-channel sum / sum of squares (accumulated into sum, sumsq).
 * fiBnStats: plain sums (also the bias gradient of ConvTranspose2d). fiBnStatsShifted: pivot[c] = z[0][c] is written and
 * the sums are taken about it, sum += sum (z - pivot), sumsq += sum (z - pivot)^2, for fiBnFinalizeShifted: the variance
 * then does not cancel on channels whose mean is large against their spread. */
int fiBnStats(const void* z, int64_t P, int C, float* sum, float* sumsq, void* stream);
int fiBnStatsShifted(const void* z, int64_t P, int C, float* pivot, float* sum, float* sumsq, void* stream);
/* a = relu(z*scale[c] + shift[c]) with scale = gamma*rstd, shift = beta - mean*scale. */
int fiBnApplyRelu(const void* z, int64_t P, int C, const float* scale, const float* shift, void* a, void* stream);
/* OutConv (model/unet.py:57-63) on bf16 [N*HW][64] -> fp32 NCHW [N,n_classes,H,W]. */
int fiHeadForward(const void* a, int N, int64_t HW, const float* w, const float* b, int n_classes, float* y, void* stream);
/* CombinedLoss (model/train.py:75-87): loss += mse_weight * mean((y-t)^2) + ssim_weight * (1 - mean SSIM(y, t)) with
 * the 11x11 Gaussian-window SSIM of SSIMLoss (model/train.py:18-73), and dy = d loss / d y. y, target, dy: fp32
 * [planes][H][W] (planes = N * n_classes; each plane is filtered on its own, like the grouped conv2d). */
int fiCombinedLossGrad(const float* y, const float* target, int planes, int H, int W, float mse_weight, float ssim_weight,
                       float* loss, float* dy, void* stream);
/* nn.MSELoss (model/train.py:81): loss += mean((y-t)^2); dy = 2(y-t)/n. */
int fiMseLossGrad(const float* y, const float* target, int64_t n, float* loss, float* dy, void* stream);
int fiHeadBackward(const void* a, const float* dy, int N, int64_t HW, const float* w, int n_classes, void* da, float* dw,
                   float* db, void* stream);
/* Backward of relu(bn(z)) with batch statistics. The ReLU mask is recomputed from z (scale * z + shift > 0, the
 * forward's expression; scale = gamma * rstd, shift = beta - mean * scale), so the stored activation is not read.
 * Reduce: dbeta[c] += sum dy, dgamma[c] += sum dy * zhat (dy = dA * mask, zhat = (z - mean) * rstd).
 * Apply: dz = gamma * rstd * (dy - dbeta / P - zhat * dgamma / P), bf16. */
int fiBnReluBackwardReduce(const void* dA, const void* z, int64_t P, int C, const float* mean, const float* rstd,
                           const float* scale, const float* shift, float* dbeta, float* dgamma, void* stream);
int fiBnReluBackwardApply(const void* dA, const void* z, int64_t P, int C, const float* mean, const float* rstd,
                          const float* gamma, const float* beta, const float* dbeta, const float* dgamma, void* dz,
                          void* stream);
/* MaxPool2d(2) backward (gradient to the first maximum of each window) plus the skip-connection gradient. */
int fiMaxPoolBackwardAdd(const void* a_full, const void* a_pool, const void* d_pool, const void* d_skip, void* d_full,
                         int N, int H, int W, int C, void* stream);
/* Backward of nn.Upsample(scale_factor=2, bilinear, align_corners=True): [N,2h,2w,C] -> [N,h,w,C]. */
int fiUpsample2xBackward(const void* d_up, void* d_lo, int N, int h, int w, int C, void* stream);
/* Weight gradient of conv3x3 (padding 1): dW[tap][cout][cin] (fp32, ACCUMULATED into) from dz [N,H,W,cout] and the
 * layer input x = channel concat of x0 [N,H,W,c0] | x1 [N,H,W,c1] (x1 NULL / c1 0 for single-source layers), all bf16
 * NHWC, channel counts multiples of 64. tcgen05 GEMM over the pixel dimension reading both operands as they lie
 * (MN-major), split-K with fp32 atomics. fiStemWgrad: the <= 8 input-channel first conv (x fp32 NCHW), dW[64][cin][9]. */
int fiWgrad(const void* dz, const void* x0, int c0, const void* x1, int c1, int N, int H, int W, int cout, float* dW,
            void* stream);
int fiStemWgrad(const void* dz, const float* x, int N, int H, int W, int cin, float* dW, void* stream);
/* The same GEMM over the pixel dimension without taps: dW[cout][cin] (fp32, ACCUMULATED into) = sum over the N*H*W
 * pixels q of dz[q][cout] * x[q][cin]. This is the weight gradient of nn.ConvTranspose2d(k=2, s=2) (Up, model/unet.py:43)
 * once its output gradient is viewed per low-resolution pixel as [N,h,w,(ky,kx,co)] (cout = 4*Cout); cin/64 even. */
int fiWgradPointwise(const void* dz, const void* x, int cin, int N, int H, int W, int cout, float* dW, void* stream);
/* Batch sums -> mean, rstd = 1/sqrt(var + eps), scale = gamma * rstd, shift = beta - mean * scale (C floats each), and
 * the nn.BatchNorm2d running estimates updated in place (momentum, unbiased variance; either may be NULL).
 * fiBnFinalize: from fiBnStats' plain sums. fiBnFinalizeShifted: from the sums and the pivot fiBnStatsShifted wrote
 * (what the training step uses). */
int fiBnFinalize(const float* sum, const float* sumsq, int C, int64_t P, float eps, float momentum, const float* gamma,
                 const float* beta, float* mean, float* rstd, float* scale, float* shift, float* running_mean,
                 float* running_var, void* stream);
int fiBnFinalizeShifted(const float* sum, const float* sumsq, const float* pivot, int C, int64_t P, float eps,
                        float momentum, const float* gamma, const float* beta, float* mean, float* rstd, float* scale,
                        float* shift, float* running_mean, float* running_var, void* stream);
/* fiWgrad's dW[tap][cout][cin] added into the parameter-gradient layout grad[cout][cin][3][3]. */
int fiUnpackConvGrad(const float* dW, int cout, int cin, float* grad, void* stream);
/* torch.optim.Adam (model/train.py:160) on one flat fp32 parameter vector; step counts from 1. hyper_dev (optional,
 * device float[2] = {lr, step}) overrides lr / step at run time so that a captured CUDA graph of the step can be
 * replayed while the schedule advances. */
int fiAdamStep(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
               int step, const float* hyper_dev, void* stream);
/* fiStemPackWeights on the device: w_dev fp32 [64][cin][3][3] -> packed_dev bf16 [64][fiStemPackedK(cin)]. */
int fiStemPackWeightsDevice(const float* w_dev, int cin, void* packed_dev, void* stream);
/* fp32 [cout][cin][3][3] -> bf16 forward rows [cout][tap*cin+ci] and data-gradient rows [cin][(8-tap)*cout+co]
 * (either may be NULL). */
int fiPackConvWeights(const float* w, int cout, int cin, void* fwd, void* bwd, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FI_B200_H */
