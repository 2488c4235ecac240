// Bandwidth-/ALU-bound kernels around the tensor-core convolutions (aux_kernels.cu).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace fi {

// One logical input channel plane set of the stem convolution: element (n, c, y, x) lives at
// ptr[n*batch_stride + c*chan_stride + y*row_stride + x*px_stride] (strides in elements).
struct PlaneSrc {
    const void* ptr;
    long long batch_stride, chan_stride, row_stride, px_stride;
    int channels;
};

struct StemDesc {
    PlaneSrc src[2];     // channels [0, src[0].channels) come from src[0], the rest from src[1] (fused torch.cat)
    int is_u8;           // 1: uint8 pixels, normalised in-kernel as u8/255*2-1 (reference inference.py:32-35); 0: fp32
    int cin;             // total input channels (<= 8)
    int N, H, W;
    const void* wpack;   // bf16 [64][stem_packed_k(cin)], hi/lo split rows (stem_pack_weights), BN folded
    const float* bias;   // fp32 [64]
    void* dst;           // bf16 NHWC [N,H,W,64]
    void* dst_lo;        // precise mode: lo halves (value = dst + dst_lo), else null
    int linear;          // 1: no ReLU (training forward keeps the pre-BatchNorm conv output)
};
const char* stem_conv_launch(const StemDesc& d, cudaStream_t stream);  // stem_mma.cu
int stem_packed_k(int cin);                                               // packed K length (multiple of 64)
void stem_pack_weights(const float* w /*[64][cin][3][3]*/, int cin, uint16_t* out /*[64][stem_packed_k]*/);

// nn.Upsample(scale_factor=2, mode='bilinear', align_corners=True) on bf16 NHWC (reference unet.py:40).
const char* upsample2x_launch(const void* src, void* dst, int N, int h, int w, int C, cudaStream_t stream,
                              const void* src_lo = nullptr, void* dst_lo = nullptr);  // lo halves: precise mode

// nn.MaxPool2d(2) on bf16 NHWC [N,H,W,C] -> [N,H/2,W/2,C] (stand-alone Down module; fused elsewhere).
const char* maxpool2x2_launch(const void* src, void* dst, int N, int H, int W, int C, cudaStream_t stream);

// Frame-pair packing + normalisation: two u8 planar frame batches [N,C,H,W] -> fp32 NCHW [N,2C,H,W] = cat(2*f/255-1).
const char* pack_pair_launch(const uint8_t* f0, const uint8_t* f1, float* out, int N, int C, int H, int W,
                             cudaStream_t stream);
// postprocess_image (reference inference.py:54-61) on n fp32 values.
const char* head_post_launch(const float* y, uint8_t* out, size_t n, cudaStream_t stream);

// skimage-equivalent SSIM (7x7 uniform window, sample covariance, data_range 255, channel_axis=-1: mean of the channel
// SSIMs) and PSNR (over all C*H*W samples) of N u8 image pairs of C = 1 or 3 channels. Each operand is planar
// (px_stride 1) or interleaved BGR (px_stride 3, chan_stride 1); N*C <= 65535. Returns a message naming the bad argument.
size_t ssim_psnr_workspace_bytes(int N, int C, int H, int W);
const char* ssim_psnr_launch(const PlaneSrc& pred, const PlaneSrc& target, int N, int H, int W, double* out /*[N][2]*/,
                             void* workspace, cudaStream_t stream);

// Scene-cut statistic: sad[p] = sum |f[p+1] - f[p]| over the frame_bytes bytes of each of the n_frames-1 consecutive
// pairs of u8 frames frame_stride bytes apart (exact; zeroes sad on `stream` first).
const char* pair_sad_launch(const uint8_t* frames, int64_t frame_stride, int64_t frame_bytes, int n_frames,
                            uint64_t* sad, cudaStream_t stream);

// Training batch from the device frame cache: frame1/frame2/target[b] = frames[triplets[samples[b]][0|1|2]] / 255 as
// fp32 [n][H*W]; out-of-range samples or frame indices give NaN rows (fiGatherTripletsU8).
// S x S windows (rows[b] = f1, f2, gt, y0, x0, mirror) of C-plane u8 frames of any size in one flat buffer ->
// three fp32 [n][C][S][S]; bad indices or windows give NaN rows (fiGatherCropsU8).
const char* gather_crops_u8_launch(const uint8_t* frames, int64_t frames_bytes, const int64_t* offsets,
                                   const int32_t* sizes, int64_t n_frames, int C, const int32_t* rows, int n, int S,
                                   float* frame1, float* frame2, float* target, cudaStream_t stream);
const char* gather_triplets_u8_launch(const uint8_t* frames, int64_t n_frames, const int32_t* triplets,
                                      int64_t n_triplets, const int64_t* samples, int n, int H, int W, float* frame1,
                                      float* frame2, float* target, cudaStream_t stream);

}  // namespace fi
