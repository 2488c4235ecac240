// Launchers of the training-step kernels (train_kernels.cu, wgrad_gemm.cu). Device pointers; nullptr return = ok.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

namespace fi {

// pivot: NULL = plain sums; else pivot[c] = z[0][c] is written and the sums are taken about it
const char* bn_stats_launch(const void* z, long long P, int C, float* sum, float* sumsq, float* pivot, cudaStream_t st);
const char* bn_finalize_launch(const float* sum, const float* sumsq, const float* pivot, int C, long long P, float eps,
                               float momentum, const float* gamma, const float* beta, float* mean, float* rstd,
                               float* scale, float* shift, float* running_mean, float* running_var, cudaStream_t st);
const char* bn_apply_relu_launch(const void* z, long long P, int C, const float* scale, const float* shift, void* a,
                                 cudaStream_t st);
const char* head_forward_launch(const void* a, int N, long long HW, const float* w, const float* b, int ncls, float* y,
                                cudaStream_t st);
const char* mse_launch(const float* y, const float* t, long long n, float* loss, float* dy, cudaStream_t st);
const char* combined_loss_launch(const float* y, const float* t, int planes, int H, int W, float mse_w, float ssim_w,
                                 float* loss, float* dy, cudaStream_t st);
const char* head_backward_launch(const void* a, const float* dy, int N, long long HW, const float* w, int ncls, void* da,
                                 float* dw, float* db, cudaStream_t st);
const char* bn_relu_bwd_reduce_launch(const void* dA, const void* z, long long P, int C, const float* mean,
                                      const float* rstd, const float* scale, const float* shift, float* dbeta,
                                      float* dgamma, cudaStream_t st);
const char* bn_relu_bwd_apply_launch(const void* dA, const void* z, long long P, int C, const float* mean,
                                     const float* rstd, const float* gamma, const float* beta, const float* dbeta,
                                     const float* dgamma, void* dz, cudaStream_t st);
const char* maxpool_bwd_add_launch(const void* a_full, const void* a_pool, const void* d_pool, const void* d_skip,
                                   void* d_full, int N, int H, int W, int C, cudaStream_t st);
const char* upsample2x_bwd_launch(const void* d_up, void* d_lo, int N, int h, int w, int C, cudaStream_t st);
const char* stem_wgrad_launch(const void* dz, const float* x, int N, int H, int W, int cin, float* dW, cudaStream_t st);
const char* unpack_conv_grad_launch(const float* dW, int cout, int cin, float* grad, cudaStream_t st);
const char* adam_launch(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps,
                        int step, const float* hyper_dev, cudaStream_t st);
const char* stem_pack_device_launch(const float* w_dev, int cin, void* out_dev, cudaStream_t st);
const char* pack_conv_launch(const float* w, int co, int ci, void* fwd, void* bwd, cudaStream_t st);

// wgrad_gemm.cu: dW[tap][co][ci] += sum_q dz[q][co] * x[q + tap][ci], x = channel concat of x0 | x1, all bf16 NHWC
// (tcgen05 GEMM over the pixel dimension with MN-major operands straight from NHWC, split-K, fp32 atomics)
const char* wgrad_launch(const void* dz, const void* x0, int c0, const void* x1, int c1, int N, int H, int W, int cout,
                         float* dW, int num_sms, cudaStream_t st, int taps = 9);

}  // namespace fi
