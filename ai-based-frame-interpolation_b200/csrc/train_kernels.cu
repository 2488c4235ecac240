// Training-step kernels around the tensor-core convolutions (reference model/train.py:153-249: forward with
// batch-statistics BatchNorm, MSE loss, backward, Adam). Activations and activation gradients are bf16 NHWC,
// statistics / weight gradients / optimizer state are fp32. The conv forward and the data gradient (a conv with the
// flipped, transposed weights) reuse conv_gemm*.cu / conv_halo*.cu; the weight gradient is wgrad_gemm.cu.
#include "ptx.cuh"
#include "aux_kernels.cuh"
#include "train_kernels.cuh"

namespace fi {

namespace {

__device__ __forceinline__ float2 unpack2(uint32_t v) { return make_float2(bf16lo_f(v), bf16hi_f(v)); }

const char* last_error() {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}
int blocks_for(long long items, int threads, int cap = 148 * 8) {
    long long b = (items + threads - 1) / threads;
    return static_cast<int>(b < 1 ? 1 : (b > cap ? cap : b));
}

// ------------------------------------------------------------------------------------------------ BN statistics
// Per-channel reductions over z: bf16 [P][C]. A thread owns one 8-channel group (16-byte loads) and walks pixels with a
// block-wide stride, four independent loads in flight; when C/8 divides 256 the 256/(C/8) pixel lanes of a block are
// combined with shared-memory atomics so that a block issues one global atomic per channel and quantity.
// With a pivot the sums are shifted, S = sum (z - k) and Q = sum (z - k)^2 with k = z[0][c] (every thread can load it),
// so that var = Q/P - (S/P)^2 does not cancel when a channel's mean is large against its spread: a constant channel is
// exact, and a flat one (dark frame, letterbox bar, the bias-free stem output) keeps its variance.
constexpr int RED_MAX_C = 2048;

template <typename Acc>
__device__ __forceinline__ void channel_reduce_walk(long long P, int c8, Acc&& per_group) {
    const bool packed = c8 <= 256 && 256 % c8 == 0;
    const int rows_par = packed ? 256 / c8 : 1;
    const int r0 = packed ? threadIdx.x / c8 : 0;
    for (int g = packed ? threadIdx.x % c8 : threadIdx.x; g < c8; g += 256)
        per_group(g, static_cast<long long>(blockIdx.x) * rows_par + r0, static_cast<long long>(gridDim.x) * rows_par,
                  packed && rows_par > 1);
}

// adds v[0..7] of channel group g to out[8g..8g+7]: through shared memory first when several pixel lanes share g
__device__ __forceinline__ void flush_group(float* sh, float* out, int g, const float (&v)[8], bool via_smem) {
    if (via_smem) {
#pragma unroll
        for (int j = 0; j < 8; ++j) atomicAdd(sh + 8 * g + j, v[j]);
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) atomicAdd(out + 8 * g + j, v[j]);
    }
}

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        f[2 * k] = bf16lo_f(w[k]);
        f[2 * k + 1] = bf16hi_f(w[k]);
    }
}

__global__ void __launch_bounds__(256, 4)
bn_stats_kernel(const uint4* __restrict__ z, long long P, int c8, float* __restrict__ sum, float* __restrict__ sumsq,
                float* __restrict__ pivot) {
    __shared__ float sh[2][RED_MAX_C];
    const int C = 8 * c8;
    for (int i = threadIdx.x; i < C; i += 256) sh[0][i] = sh[1][i] = 0.f;
    __syncthreads();
    bool any_smem = false;
    channel_reduce_walk(P, c8, [&](int g, long long p, long long step, bool via_smem) {
        float s[8], q[8], k[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) s[j] = q[j] = k[j] = 0.f;
        if (pivot) {
            unpack8(__ldg(z + g), k);   // pixel 0 of the group's channels
            if (p == 0) {               // the one lane that starts at pixel 0 publishes the pivot for bn_finalize
#pragma unroll
                for (int j = 0; j < 8; ++j) pivot[8 * g + j] = k[j];
            }
        }
        auto add = [&](const uint4& v) {
            float f[8];
            unpack8(v, f);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float d = f[j] - k[j];   // exact for bf16 values within a factor 2^16 of each other
                s[j] += d;
                q[j] = fmaf(d, d, q[j]);
            }
        };
        for (; p + 3 * step < P; p += 4 * step) {
            const uint4 v0 = __ldg(z + p * c8 + g), v1 = __ldg(z + (p + step) * c8 + g);
            const uint4 v2 = __ldg(z + (p + 2 * step) * c8 + g), v3 = __ldg(z + (p + 3 * step) * c8 + g);
            add(v0); add(v1); add(v2); add(v3);
        }
        for (; p < P; p += step) add(__ldg(z + p * c8 + g));
        flush_group(sh[0], sum, g, s, via_smem);
        flush_group(sh[1], sumsq, g, q, via_smem);
        any_smem = via_smem;
    });
    if (any_smem) {   // uniform across the block
        __syncthreads();
        for (int i = threadIdx.x; i < C; i += 256) { atomicAdd(sum + i, sh[0][i]); atomicAdd(sumsq + i, sh[1][i]); }
    }
}

// Batch statistics -> per-channel affine + the nn.BatchNorm2d running estimates (momentum update, unbiased variance).
// sum / sumsq are taken about pivot[c] (NULL: about 0).
__global__ void __launch_bounds__(256)
bn_finalize_kernel(const float* __restrict__ sum, const float* __restrict__ sumsq, const float* __restrict__ pivot,
                   int C, float inv_p, float unbias,
                   float eps, float momentum, const float* __restrict__ gamma, const float* __restrict__ beta,
                   float* __restrict__ mean_out, float* __restrict__ rstd_out, float* __restrict__ scale,
                   float* __restrict__ shift, float* __restrict__ running_mean, float* __restrict__ running_var) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float ms = sum[c] * inv_p;   // mean - pivot
    const float mean = (pivot ? pivot[c] : 0.f) + ms;
    const float var = fmaxf(sumsq[c] * inv_p - ms * ms, 0.f);
    const float rstd = rsqrtf(var + eps);
    const float sc = gamma[c] * rstd;
    mean_out[c] = mean;
    rstd_out[c] = rstd;
    scale[c] = sc;
    shift[c] = beta[c] - mean * sc;
    if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
    if (running_var) running_var[c] = (1.f - momentum) * running_var[c] + momentum * var * unbias;
}

// a = relu(z * scale[c] + shift[c]) (scale = gamma * rstd, shift = beta - mean * scale); 8 channels per thread.
__global__ void __launch_bounds__(256)
bn_apply_relu_kernel(const uint4* __restrict__ z, long long n8, int c8, const float* __restrict__ scale,
                     const float* __restrict__ shift, uint4* __restrict__ a) {
    // the launcher makes gridDim.x * 256 a multiple of c8, so a thread keeps its channel group: parameters in registers
    const long long i0 = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long step = static_cast<long long>(gridDim.x) * blockDim.x;
    const int c = static_cast<int>(i0 % c8) * 8;
    float sc[8], sf[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j] = scale[c + j]; sf[j] = shift[c + j]; }
    auto one = [&](long long i, const uint4& v) {
        float f[8];
        unpack8(v, f);
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k)
            o[k] = pack_bf16x2(fmaxf(fmaf(f[2 * k], sc[2 * k], sf[2 * k]), 0.f),
                               fmaxf(fmaf(f[2 * k + 1], sc[2 * k + 1], sf[2 * k + 1]), 0.f));
        a[i] = make_uint4(o[0], o[1], o[2], o[3]);
    };
    long long i = i0;
    for (; i + step < n8; i += 2 * step) {
        const uint4 v0 = __ldg(z + i), v1 = __ldg(z + i + step);
        one(i, v0);
        one(i + step, v1);
    }
    if (i < n8) one(i, __ldg(z + i));
}

// ------------------------------------------------------------------------------------------------ head + loss
// y[n][k][pix] = b[k] + sum_c a[n][pix][c] * w[k][c]   (a: bf16 [N*HW][64])
template <int NCLS>
__global__ void __launch_bounds__(256)
head_forward_kernel(const uint4* __restrict__ a, long long P, long long HW, const float* __restrict__ w,
                    const float* __restrict__ b, float* __restrict__ y) {
    constexpr int ncls = NCLS;
    __shared__ float ws[4 * 64];
    for (int i = threadIdx.x; i < ncls * 64; i += blockDim.x) ws[i] = w[i];
    __syncthreads();
    // 8 consecutive lanes share a pixel (one 16-byte load each: a warp reads 512 contiguous bytes), partial dot
    // products are combined with three xor-shuffles; the trip count is uniform across the warp
    const int cg = threadIdx.x & 7;
    float wr[NCLS][8];
#pragma unroll
    for (int cls = 0; cls < ncls; ++cls)
#pragma unroll
        for (int j = 0; j < 8; ++j) wr[cls][j] = ws[cls * 64 + cg * 8 + j];
    const long long total = (P * 8 + 31) / 32 * 32;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long p = i >> 3;
        float f[8];
        unpack8(p < P ? __ldg(a + i) : make_uint4(0, 0, 0, 0), f);
        float acc[NCLS];
#pragma unroll
        for (int cls = 0; cls < ncls; ++cls) {
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) s = fmaf(f[j], wr[cls][j], s);
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            acc[cls] = s;
        }
        if (cg == 0 && p < P) {
            const long long n = p / HW, pix = p - n * HW;
#pragma unroll
            for (int cls = 0; cls < ncls; ++cls) y[(n * ncls + cls) * HW + pix] = acc[cls] + b[cls];
        }
    }
}

// loss += sum (y-t)^2 / n ; dy = 2 (y - t) / n
__global__ void __launch_bounds__(256)
mse_kernel(const float* __restrict__ y, const float* __restrict__ t, long long n, float inv_n, float* __restrict__ loss,
           float* __restrict__ dy) {
    float part = 0.f;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const float d = y[i] - t[i];
        part += d * d;
        dy[i] = 2.f * d * inv_n;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(loss, part * inv_n);
}

__global__ void ssim_offset_kernel(float* loss, float v) { atomicAdd(loss, v); }

// ------------------------------------------------------------------------------------------------ combined loss
// loss = mse_w * mean((y-t)^2) + ssim_w * (1 - mean(SSIM(y, t)))  and its gradient w.r.t. y  (reference model/train.py:18-87:
// 11x11 Gaussian window, sigma 1.5, zero-padded 'same' filtering per plane, C1 = 0.01^2, C2 = 0.03^2).
// With mu1 = G*y, mu2 = G*t, E11 = G*y^2, E22 = G*t^2, E12 = G*(y t):
//   S = A1 A2 / (B1 B2),  A1 = 2 mu1 mu2 + C1, A2 = 2 (E12 - mu1 mu2) + C2, B1 = mu1^2 + mu2^2 + C1,
//                          B2 = (E11 - mu1^2) + (E22 - mu2^2) + C2
//   dSum/dy = G*(dS/dmu1) + 2 y G*(dS/dE11) + t G*(dS/dE12)       (G symmetric, derivative maps zero outside the image)
// One block owns a 32x32 tile of one plane: inputs with a 10-pixel halo, the five filtered maps and the three derivative
// maps on the 5-pixel halo, all in shared memory, every filter separable (11 + 11 taps).
constexpr int SL_TILE = 32, SL_R = 5;
constexpr int SL_IN = SL_TILE + 4 * SL_R;    // 52: input region
constexpr int SL_MID = SL_TILE + 2 * SL_R;   // 42: region of the SSIM map / derivative maps
constexpr int SL_SMEM_FLOATS = 2 * SL_IN * SL_IN + 5 * SL_IN * SL_MID + 3 * SL_MID * SL_MID;
struct GaussWindow { float g[2 * SL_R + 1]; };

__global__ void __launch_bounds__(256)
combined_loss_kernel(const float* __restrict__ y, const float* __restrict__ t, int H, int W, const GaussWindow gw,
                     float mse_scale, float ssim_scale, float* __restrict__ loss, float* __restrict__ dy) {
    extern __shared__ float sl[];
    float* sx = sl;                             // [SL_IN][SL_IN]  prediction
    float* sy = sx + SL_IN * SL_IN;             // [SL_IN][SL_IN]  target
    float* hb = sy + SL_IN * SL_IN;             // [5][SL_IN][SL_MID] horizontally filtered x, y, xx, yy, xy
    float* dm = hb + 5 * SL_IN * SL_MID;        // [3][SL_MID][SL_MID] dS/dmu1, dS/dE11, dS/dE12
    float* hb2 = hb;                            // [3][SL_MID][SL_TILE] (reuses hb)
    const int tiles_x = (W + SL_TILE - 1) / SL_TILE;
    const int tx0 = (blockIdx.x % tiles_x) * SL_TILE, ty0 = (blockIdx.x / tiles_x) * SL_TILE;
    const long long plane = static_cast<long long>(blockIdx.y) * H * W;
    const float* yp = y + plane;
    const float* tp = t + plane;
    for (int i = threadIdx.x; i < SL_IN * SL_IN; i += 256) {
        const int r = i / SL_IN, c = i - r * SL_IN;
        const int gy = ty0 - 2 * SL_R + r, gx = tx0 - 2 * SL_R + c;
        const bool in = gy >= 0 && gy < H && gx >= 0 && gx < W;
        sx[i] = in ? __ldg(yp + static_cast<long long>(gy) * W + gx) : 0.f;
        sy[i] = in ? __ldg(tp + static_cast<long long>(gy) * W + gx) : 0.f;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < SL_IN * SL_MID; i += 256) {   // horizontal pass over all 52 rows, 42 columns
        const int r = i / SL_MID, c = i - r * SL_MID;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f, a4 = 0.f;
#pragma unroll
        for (int k = 0; k <= 2 * SL_R; ++k) {
            const float xv = sx[r * SL_IN + c + k], yv = sy[r * SL_IN + c + k], w = gw.g[k];
            a0 = fmaf(w, xv, a0); a1 = fmaf(w, yv, a1);
            a2 = fmaf(w, xv * xv, a2); a3 = fmaf(w, yv * yv, a3); a4 = fmaf(w, xv * yv, a4);
        }
        hb[i] = a0; hb[SL_IN * SL_MID + i] = a1; hb[2 * SL_IN * SL_MID + i] = a2;
        hb[3 * SL_IN * SL_MID + i] = a3; hb[4 * SL_IN * SL_MID + i] = a4;
    }
    __syncthreads();
    const float C1 = 0.01f * 0.01f, C2 = 0.03f * 0.03f;
    float ssim_part = 0.f, mse_part = 0.f;
    for (int i = threadIdx.x; i < SL_MID * SL_MID; i += 256) {  // vertical pass -> SSIM and its partial derivatives
        const int r = i / SL_MID, c = i - r * SL_MID;
        const int gy = ty0 - SL_R + r, gx = tx0 - SL_R + c;
        float m[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k <= 2 * SL_R; ++k) {
            const float w = gw.g[k];
#pragma unroll
            for (int q = 0; q < 5; ++q) m[q] = fmaf(w, hb[q * SL_IN * SL_MID + (r + k) * SL_MID + c], m[q]);
        }
        float d_mu = 0.f, d_11 = 0.f, d_12 = 0.f;
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
            const float mu1 = m[0], mu2 = m[1];
            const float A1 = 2.f * mu1 * mu2 + C1, A2 = 2.f * (m[4] - mu1 * mu2) + C2;
            const float B1 = mu1 * mu1 + mu2 * mu2 + C1, B2 = (m[2] - mu1 * mu1) + (m[3] - mu2 * mu2) + C2;
            const float inv = 1.f / (B1 * B2);
            const float S = A1 * A2 * inv;
            d_mu = 2.f * mu2 * (A2 - A1) * inv - 2.f * mu1 * S * (1.f / B1 - 1.f / B2);
            d_11 = -S / B2;
            d_12 = 2.f * A1 * inv;
            if (r >= SL_R && r < SL_R + SL_TILE && c >= SL_R && c < SL_R + SL_TILE) ssim_part += S;   // own tile only
        }
        dm[i] = d_mu; dm[SL_MID * SL_MID + i] = d_11; dm[2 * SL_MID * SL_MID + i] = d_12;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < SL_MID * SL_TILE; i += 256) {  // horizontal pass of the derivative maps
        const int r = i / SL_TILE, c = i - r * SL_TILE;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
        for (int k = 0; k <= 2 * SL_R; ++k) {
            const float w = gw.g[k];
            a0 = fmaf(w, dm[r * SL_MID + c + k], a0);
            a1 = fmaf(w, dm[SL_MID * SL_MID + r * SL_MID + c + k], a1);
            a2 = fmaf(w, dm[2 * SL_MID * SL_MID + r * SL_MID + c + k], a2);
        }
        hb2[i] = a0; hb2[SL_MID * SL_TILE + i] = a1; hb2[2 * SL_MID * SL_TILE + i] = a2;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < SL_TILE * SL_TILE; i += 256) {  // vertical pass -> gradient
        const int r = i / SL_TILE, c = i - r * SL_TILE;
        const int gy = ty0 + r, gx = tx0 + c;
        if (gy >= H || gx >= W) continue;
        float g0 = 0.f, g1 = 0.f, g2 = 0.f;
#pragma unroll
        for (int k = 0; k <= 2 * SL_R; ++k) {
            const float w = gw.g[k];
            g0 = fmaf(w, hb2[(r + k) * SL_TILE + c], g0);
            g1 = fmaf(w, hb2[SL_MID * SL_TILE + (r + k) * SL_TILE + c], g1);
            g2 = fmaf(w, hb2[2 * SL_MID * SL_TILE + (r + k) * SL_TILE + c], g2);
        }
        const float xv = sx[(r + 2 * SL_R) * SL_IN + c + 2 * SL_R], yv = sy[(r + 2 * SL_R) * SL_IN + c + 2 * SL_R];
        const float diff = xv - yv;
        mse_part = fmaf(diff, diff, mse_part);
        // d/dy [ mse_scale * sum diff^2 - ssim_scale * sum S ]
        dy[plane + static_cast<long long>(gy) * W + gx] =
            2.f * mse_scale * diff - ssim_scale * (g0 + 2.f * xv * g1 + yv * g2);
    }
    float part = mse_scale * mse_part - ssim_scale * ssim_part;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_down_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(loss, part);
}

// da[n][pix][c] = sum_k dy[n][k][pix] w[k][c];  dw[k][c] += sum dy * a;  db[k] += sum dy
template <int NCLS>
__global__ void __launch_bounds__(256)
head_backward_kernel(const uint4* __restrict__ a, const float* __restrict__ dy, long long P, long long HW,
                     const float* __restrict__ w, uint4* __restrict__ da, float* __restrict__ dw,
                     float* __restrict__ db) {
    constexpr int ncls = NCLS;
    __shared__ float ws[4 * 64];
    __shared__ float acc_w[4 * 64];
    __shared__ float acc_b[4];
    for (int i = threadIdx.x; i < ncls * 64; i += blockDim.x) { ws[i] = w[i]; acc_w[i] = 0.f; }
    if (threadIdx.x < 4) acc_b[threadIdx.x] = 0.f;
    __syncthreads();
    // thread = (pixel, 8-channel group): 8 consecutive threads share a pixel
    const int cg = threadIdx.x & 7;
    float lw[4][8];
    float lb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int j = 0; j < 8; ++j) lw[k][j] = 0.f;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < P * 8;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long p = i >> 3;
        const long long n = p / HW, pix = p - n * HW;
        float g[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < ncls; ++k) g[k] = __ldg(dy + (n * ncls + k) * HW + pix);
        const uint4 v = __ldg(a + i);
        const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
        float av[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float2 f = unpack2(wv[k]); av[2 * k] = f.x; av[2 * k + 1] = f.y; }
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float s = 0.f;
#pragma unroll
            for (int k = 0; k < ncls; ++k) { s = fmaf(g[k], ws[k * 64 + cg * 8 + j], s); lw[k][j] = fmaf(g[k], av[j], lw[k][j]); }
            o[j] = s;
        }
        if (cg == 0) {
#pragma unroll
            for (int k = 0; k < ncls; ++k) lb[k] += g[k];
        }
        da[i] = make_uint4(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]), pack_bf16x2(o[4], o[5]), pack_bf16x2(o[6], o[7]));
    }
#pragma unroll
    for (int k = 0; k < ncls; ++k) {
#pragma unroll
        for (int j = 0; j < 8; ++j) atomicAdd(&acc_w[k * 64 + cg * 8 + j], lw[k][j]);
        if (cg == 0) atomicAdd(&acc_b[k], lb[k]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < ncls * 64; i += blockDim.x) atomicAdd(dw + i, acc_w[i]);
    if (threadIdx.x < ncls) atomicAdd(db + threadIdx.x, acc_b[threadIdx.x]);
}

// ------------------------------------------------------------------------------------------------ BN + ReLU backward
// dy = dA * (a > 0); dbeta[c] += sum dy; dgamma[c] += sum dy * zhat, zhat = (z - mean) * rstd.   (same walk as bn_stats)
// The ReLU mask is recomputed from z with the forward's own expression (scale * z + shift > 0) instead of reading the
// stored activation: one tensor less to stream in both backward kernels.
__global__ void __launch_bounds__(256, 3)
bn_relu_bwd_reduce_kernel(const uint4* __restrict__ dA, const uint4* __restrict__ z, long long P, int c8,
                          const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ scale,
                          const float* __restrict__ shift, float* __restrict__ dbeta, float* __restrict__ dgamma) {
    __shared__ float sh[2][RED_MAX_C];
    const int C = 8 * c8;
    for (int i = threadIdx.x; i < C; i += 256) sh[0][i] = sh[1][i] = 0.f;
    __syncthreads();
    bool any_smem = false;
    channel_reduce_walk(P, c8, [&](int g, long long p, long long step, bool via_smem) {
        float m[8], sc[8], sf[8], b[8], gsum[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            m[j] = mean[8 * g + j]; sc[j] = scale[8 * g + j]; sf[j] = shift[8 * g + j];
            b[j] = gsum[j] = 0.f;
        }
        auto add = [&](const uint4& dv, const uint4& zv) {
            float d[8], zf[8];
            unpack8(dv, d); unpack8(zv, zf);
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float dd = fmaf(zf[j], sc[j], sf[j]) > 0.f ? d[j] : 0.f;
                b[j] += dd;
                gsum[j] = fmaf(dd, zf[j] - m[j], gsum[j]);
            }
        };
        for (; p + 2 * step < P; p += 3 * step) {
            const long long i0 = p * c8 + g, i1 = (p + step) * c8 + g, i2 = (p + 2 * step) * c8 + g;
            const uint4 d0 = __ldg(dA + i0), z0 = __ldg(z + i0), d1 = __ldg(dA + i1), z1 = __ldg(z + i1);
            const uint4 d2 = __ldg(dA + i2), z2 = __ldg(z + i2);
            add(d0, z0); add(d1, z1); add(d2, z2);
        }
        for (; p < P; p += step) { const long long i0 = p * c8 + g; add(__ldg(dA + i0), __ldg(z + i0)); }
#pragma unroll
        for (int j = 0; j < 8; ++j) gsum[j] *= rstd[8 * g + j];
        flush_group(sh[0], dbeta, g, b, via_smem);
        flush_group(sh[1], dgamma, g, gsum, via_smem);
        any_smem = via_smem;
    });
    if (any_smem) {
        __syncthreads();
        for (int i = threadIdx.x; i < C; i += 256) { atomicAdd(dbeta + i, sh[0][i]); atomicAdd(dgamma + i, sh[1][i]); }
    }
}

// dz = gamma * rstd * (dy - dbeta/P - zhat * dgamma/P)
__global__ void __launch_bounds__(256)
bn_relu_bwd_apply_kernel(const uint4* __restrict__ dA, const uint4* __restrict__ z, long long n8, int c8, float inv_p,
                         const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ gamma,
                         const float* __restrict__ beta, const float* __restrict__ dbeta, const float* __restrict__ dgamma,
                         uint4* __restrict__ dz) {
    // gridDim.x * 256 is a multiple of c8 (launcher): per-channel constants live in registers
    const long long i0 = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long step = static_cast<long long>(gridDim.x) * blockDim.x;
    const int c = static_cast<int>(i0 % c8) * 8;
    float k1[8], k2[8], k3[8], m[8], sf[8];   // dz = k1 * (dy - k2 - (z - m) * k3); mask: k1 * z + sf > 0 (the forward's fma)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float r = rstd[c + j];
        k1[j] = gamma[c + j] * r;
        k2[j] = dbeta[c + j] * inv_p;
        k3[j] = r * dgamma[c + j] * inv_p;
        m[j] = mean[c + j];
        sf[j] = beta[c + j] - m[j] * k1[j];
    }
    auto one = [&](long long i, const uint4& dv, const uint4& zv) {
        float d[8], zf[8], r[8];
        unpack8(dv, d); unpack8(zv, zf);
#pragma unroll
        for (int j = 0; j < 8; ++j)
            r[j] = k1[j] * ((fmaf(zf[j], k1[j], sf[j]) > 0.f ? d[j] : 0.f) - k2[j] - (zf[j] - m[j]) * k3[j]);
        dz[i] = make_uint4(pack_bf16x2(r[0], r[1]), pack_bf16x2(r[2], r[3]), pack_bf16x2(r[4], r[5]), pack_bf16x2(r[6], r[7]));
    };
    long long i = i0;
    for (; i + step < n8; i += 2 * step) {
        const uint4 d0 = __ldg(dA + i), z0 = __ldg(z + i);
        const uint4 d1 = __ldg(dA + i + step), z1 = __ldg(z + i + step);
        one(i, d0, z0);
        one(i + step, d1, z1);
    }
    if (i < n8) one(i, __ldg(dA + i), __ldg(z + i));
}

// ------------------------------------------------------------------------------------------------ pool / upsample backward
// d_full[n,y,x,c] = (d_skip ? d_skip : 0) + (a_full == a_pool[y/2,x/2] and first such position in the 2x2 window ? d_pool : 0)
__global__ void __launch_bounds__(256)
maxpool_bwd_add_kernel(const uint4* __restrict__ a_full, const uint4* __restrict__ a_pool, const uint4* __restrict__ d_pool,
                       const uint4* __restrict__ d_skip, uint4* __restrict__ d_full, int N, int H, int W, int c8) {
    const int oh = H / 2, ow = W / 2;
    const long long total = static_cast<long long>(N) * oh * ow * c8;  // one thread per pooled element group
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int cg = static_cast<int>(i % c8);
        long long r = i / c8;
        const int ox = static_cast<int>(r % ow);
        r /= ow;
        const int oy = static_cast<int>(r % oh);
        const int n = static_cast<int>(r / oh);
        const uint4 pv = __ldg(a_pool + i), gv = __ldg(d_pool + i);
        const uint32_t pw[4] = {pv.x, pv.y, pv.z, pv.w}, gw[4] = {gv.x, gv.y, gv.z, gv.w};
        uint32_t taken[4] = {0, 0, 0, 0};  // per half-word: gradient already routed (ties go to the first position)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int y = 2 * oy + (q >> 1), x = 2 * ox + (q & 1);
            const long long idx = ((static_cast<long long>(n) * H + y) * W + x) * c8 + cg;
            const uint4 fv = __ldg(a_full + idx);
            const uint32_t fw[4] = {fv.x, fv.y, fv.z, fv.w};
            uint4 sk = make_uint4(0, 0, 0, 0);
            if (d_skip) sk = __ldg(d_skip + idx);
            const uint32_t sw[4] = {sk.x, sk.y, sk.z, sk.w};
            uint32_t o[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float2 s = unpack2(sw[k]), g = unpack2(gw[k]);
                const bool lo = ((fw[k] & 0xffffu) == (pw[k] & 0xffffu)) && !(taken[k] & 1u);
                const bool hi = ((fw[k] >> 16) == (pw[k] >> 16)) && !(taken[k] & 2u);
                taken[k] |= (lo ? 1u : 0u) | (hi ? 2u : 0u);
                o[k] = pack_bf16x2(s.x + (lo ? g.x : 0.f), s.y + (hi ? g.y : 0.f));
            }
            d_full[idx] = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
    // odd trailing row / column (dropped by the floor pooling) only carries the skip gradient
    if ((H & 1) || (W & 1)) {
        const long long edge = static_cast<long long>(N) * H * W * c8;
        for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < edge;
             i += static_cast<long long>(gridDim.x) * blockDim.x) {
            long long r = i / c8;
            const int x = static_cast<int>(r % W);
            const int y = static_cast<int>((r / W) % H);
            if (y >= 2 * oh || x >= 2 * ow) d_full[i] = d_skip ? __ldg(d_skip + i) : make_uint4(0, 0, 0, 0);
        }
    }
}

// Backward of bilinear x2 (align_corners=True) with the F.pad offset of Up: d_lo[n,y,x,c] = sum over the output pixels
// whose taps include (y,x) of weight * d_up_padded. Gather form (deterministic): an input pixel can only be referenced
// by output rows in [2y-2, 2y+2] / columns likewise.
__global__ void __launch_bounds__(256)
upsample2x_bwd_kernel(const uint4* __restrict__ d_up, uint4* __restrict__ d_lo, int N, int h, int w, int c8) {
    const int oh = 2 * h, ow = 2 * w;
    const float rh = oh > 1 ? static_cast<float>(h - 1) / static_cast<float>(oh - 1) : 0.f;
    const float rw = ow > 1 ? static_cast<float>(w - 1) / static_cast<float>(ow - 1) : 0.f;
    const long long total = static_cast<long long>(N) * h * w * c8;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int cg = static_cast<int>(i % c8);
        long long r = i / c8;
        const int x = static_cast<int>(r % w);
        r /= w;
        const int y = static_cast<int>(r % h);
        const int n = static_cast<int>(r / h);
        float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        // weights of the five candidate output rows / columns 2y-2 .. 2y+2 (none further away can reference (y, x):
        // the source coordinate is o * (h-1)/(2h-1), just under o/2)
        float wy[5], wx[5];
#pragma unroll
        for (int d = 0; d < 5; ++d) {
            const int oy = 2 * y - 2 + d, ox = 2 * x - 2 + d;
            wy[d] = wx[d] = 0.f;
            if (oy >= 0 && oy < oh) {
                const float fy = rh * oy;
                const int y0 = static_cast<int>(fy);
                const int y1 = y0 + (y0 < h - 1 ? 1 : 0);
                const float ly = fy - y0;
                wy[d] = (y0 == y ? 1.f - ly : 0.f) + (y1 == y ? ly : 0.f);
            }
            if (ox >= 0 && ox < ow) {
                const float fx = rw * ox;
                const int x0 = static_cast<int>(fx);
                const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
                const float lx = fx - x0;
                wx[d] = (x0 == x ? 1.f - lx : 0.f) + (x1 == x ? lx : 0.f);
            }
        }
#pragma unroll
        for (int dy = 0; dy < 5; ++dy) {
            if (wy[dy] == 0.f) continue;
            const uint4* row = d_up + (static_cast<long long>(n) * oh + (2 * y - 2 + dy)) * ow * c8 + cg;
#pragma unroll
            for (int dx = 0; dx < 5; ++dx) {
                if (wx[dx] == 0.f) continue;
                float f[8];
                unpack8(__ldg(row + static_cast<long long>(2 * x - 2 + dx) * c8), f);
                const float wt = wy[dy] * wx[dx];
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] = fmaf(wt, f[k], acc[k]);
            }
        }
        d_lo[i] = make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]), pack_bf16x2(acc[4], acc[5]),
                             pack_bf16x2(acc[6], acc[7]));
    }
}

// Stem weight gradient (K = 9*C_in): dW[co][ci][tap] += sum_px dz[px,co] * x[px+tap, ci]; x in NCHW fp32.
// A block walks 128-pixel row segments: the 3 x 130 input window of a segment is staged in shared memory, each warp
// takes 16 consecutive pixels and slides a 3x3xCIN register window along them (3*CIN shared loads per pixel); a thread
// owns one channel pair of dz, so its 2 x 9*CIN partial sums stay in registers (CIN is a template parameter: the
// accumulator array is never indexed dynamically). Partials are combined per block with shared-memory atomics and leave
// the block as one global atomic per weight.
constexpr int STEM_WG_TILE = 128;

template <int CIN>
__global__ void __launch_bounds__(256)
stem_wgrad_kernel(const uint32_t* __restrict__ dz, const float* __restrict__ x, int N, int H, int W,
                  float* __restrict__ dW) {
    constexpr int K = 9 * CIN;
    constexpr int XS = STEM_WG_TILE + 2;
    __shared__ float xs[CIN][3][XS];
    __shared__ float part[64 * K];
    for (int i = threadIdx.x; i < 64 * K; i += 256) part[i] = 0.f;
    const int cp = threadIdx.x & 31, wp = threadIdx.x >> 5;
    float acc[2][K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[0][k] = acc[1][k] = 0.f;
    const int tiles_per_row = (W + STEM_WG_TILE - 1) / STEM_WG_TILE;
    const int total = N * H * tiles_per_row;
    for (int tile = blockIdx.x; tile < total; tile += gridDim.x) {
        const int tr = tile % tiles_per_row;
        const int ny = tile / tiles_per_row;
        const int y = ny % H, n = ny / H;
        const int x0 = tr * STEM_WG_TILE;
        // this warp's 16 dz values first: all loads of the segment are in flight while the window is staged
        const int px0 = wp * 16;                        // this warp's first pixel inside the segment
        const uint32_t* dzp = dz + (static_cast<long long>(ny) * W + x0 + px0) * 32 + cp;
        uint32_t gz[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) gz[j] = x0 + px0 + j < W ? __ldg(dzp + j * 32) : 0u;   // bf16 zeros past the row end
        __syncthreads();   // the previous segment's readers are done (and `part` is zeroed on the first pass)
        for (int i = threadIdx.x; i < CIN * 3 * XS; i += 256) {
            const int c = i % XS;
            const int r = (i / XS) % 3, ci = i / (3 * XS);
            const int yy = y + r - 1, xq = x0 + c - 1;
            (&xs[0][0][0])[i] = (yy >= 0 && yy < H && xq >= 0 && xq < W)
                                    ? __ldg(x + ((static_cast<long long>(n) * CIN + ci) * H + yy) * W + xq) : 0.f;
        }
        __syncthreads();
        float win[CIN][3][3];
#pragma unroll
        for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                win[ci][r][1] = xs[ci][r][px0];
                win[ci][r][2] = xs[ci][r][px0 + 1];
            }
#pragma unroll
        for (int j = 0; j < 16; ++j) {
#pragma unroll
            for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    win[ci][r][0] = win[ci][r][1];
                    win[ci][r][1] = win[ci][r][2];
                    win[ci][r][2] = xs[ci][r][px0 + j + 2];
                }
            const float2 g = unpack2(gz[j]);
#pragma unroll
            for (int ci = 0; ci < CIN; ++ci)
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                    const float v = win[ci][t / 3][t % 3];
                    acc[0][ci * 9 + t] = fmaf(g.x, v, acc[0][ci * 9 + t]);
                    acc[1][ci * 9 + t] = fmaf(g.y, v, acc[1][ci * 9 + t]);
                }
        }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < K; ++k) {   // 8-way contention at most (the 8 warps)
        atomicAdd(&part[(2 * cp) * K + k], acc[0][k]);
        atomicAdd(&part[(2 * cp + 1) * K + k], acc[1][k]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 64 * K; i += 256) atomicAdd(dW + i, part[i]);
}

// fiWgrad's dW[tap][co][ci] -> the parameter layout grad[co][ci][tap] (accumulated): thread = one (co, ci)
__global__ void __launch_bounds__(256)
unpack_conv_grad_kernel(const float* __restrict__ dW, long long n, float* __restrict__ grad) {
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        float v[9];
#pragma unroll
        for (int t = 0; t < 9; ++t) v[t] = __ldg(dW + t * n + i);
#pragma unroll
        for (int t = 0; t < 9; ++t) grad[i * 9 + t] += v[t];
    }
}

// ------------------------------------------------------------------------------------------------ optimizer / packing
// torch.optim.Adam defaults (reference model/train.py:160): p -= lr * mhat / (sqrt(vhat) + eps)
// hyper (optional, device): {lr, step} read at run time, so a captured CUDA graph of the step can be replayed while
// the learning-rate schedule and the step count advance. The bias corrections are computed here on both paths, so that
// the two give the same bits.
__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
            float lr, float b1, float b2, float eps, float step, const float* __restrict__ hyper) {
    if (hyper) {
        lr = hyper[0];
        step = hyper[1];
    }
    const float bc1 = 1.f - powf(b1, step), bc2 = 1.f - powf(b2, step);
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const float gi = g[i];
        const float mi = b1 * m[i] + (1.f - b1) * gi;
        const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        p[i] -= lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);
    }
}

// Device twin of stem_pack_weights (stem_mma.cu): fp32 [64][cin][3][3] -> bf16 [64][kp] = [w_hi | w_lo | w_hi | 0]
__global__ void __launch_bounds__(256)
stem_pack_kernel(const float* __restrict__ w, int cin, int kp, __nv_bfloat16* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 64 * kp) return;
    const bool chunked = cin > 4;            // tap-major rows with the channels padded to 8 (stem_mma.cu)
    const int group = chunked ? 8 : cin;
    const int co = i / kp, k = i - co * kp, kt = 9 * group;
    const int seg = k / kt, idx = k - seg * kt;
    const int tap = idx / group, c = idx - tap * group;
    __nv_bfloat16 r = __float2bfloat16(0.f);
    if (seg < 3 && c < cin) {
        const float v = w[(co * cin + c) * 9 + tap];
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        r = seg == 1 ? __float2bfloat16_rn(v - __bfloat162float(h)) : h;
    }
    out[i] = r;
}

// w fp32 [co][ci][3][3] -> fwd bf16 [co][tap*ci_tot + ci] and bwd bf16 [ci][(8-tap)*co_tot + co] (data-gradient weights:
// dX = conv3x3(dz, Wb) with Wb[ci][tap'][co] = w[co][ci][8 - tap']). A thread owns the nine taps of one (co, ci) pair
// (36 contiguous bytes); blockIdx.y picks the output: 0 walks pairs with ci fastest (coalesced fwd rows), 1 walks them
// with co fastest (coalesced bwd rows).
__global__ void __launch_bounds__(256)
pack_conv_kernel(const float* __restrict__ w, int co, int ci, __nv_bfloat16* __restrict__ fwd,
                 __nv_bfloat16* __restrict__ bwd) {
    const bool backward = blockIdx.y == 1;
    __nv_bfloat16* out = backward ? bwd : fwd;
    if (!out) return;
    const long long total = static_cast<long long>(co) * ci;
    for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int o = static_cast<int>(backward ? i % co : i / ci);
        const int c = static_cast<int>(backward ? i / co : i % ci);
        const float* src = w + (static_cast<long long>(o) * ci + c) * 9;
        float v[9];
#pragma unroll
        for (int t = 0; t < 9; ++t) v[t] = __ldg(src + t);
        if (backward) {
#pragma unroll
            for (int t = 0; t < 9; ++t) out[(static_cast<long long>(c) * 9 + (8 - t)) * co + o] = __float2bfloat16(v[t]);
        } else {
#pragma unroll
            for (int t = 0; t < 9; ++t) out[(static_cast<long long>(o) * 9 + t) * ci + c] = __float2bfloat16(v[t]);
        }
    }
}

}  // namespace

#define FI_REQUIRE(cond, msg) do { if (!(cond)) return msg; } while (0)

namespace {
// grid of a per-channel reduction: every block covers 256/c8 pixel lanes (or one when c8 does not divide 256)
int reduce_blocks(long long P, int c8, int blocks_per_sm = 4) {
    const int rows_par = (c8 <= 256 && 256 % c8 == 0) ? 256 / c8 : 1;
    return blocks_for(P, rows_par * 4, 148 * blocks_per_sm);   // one resident wave
}
// grid of an elementwise per-channel kernel: gridDim * 256 must be a multiple of c8 so threads keep their channel group
int apply_blocks(long long n8, int c8) {
    int b = blocks_for(n8, 512, 148 * 8);
    int unit = 1;                      // smallest block count with (unit * 256) % c8 == 0
    while ((static_cast<long long>(unit) * 256) % c8) ++unit;
    b = (b + unit - 1) / unit * unit;
    return b;
}
}  // namespace

const char* bn_stats_launch(const void* z, long long P, int C, float* sum, float* sumsq, float* pivot, cudaStream_t st) {
    FI_REQUIRE(z && sum && sumsq && P > 0 && C > 0 && C % 8 == 0 && C <= RED_MAX_C, "bn_stats: bad arguments");
    bn_stats_kernel<<<reduce_blocks(P, C / 8), 256, 0, st>>>(static_cast<const uint4*>(z), P, C / 8, sum, sumsq, pivot);
    return last_error();
}
const char* bn_finalize_launch(const float* sum, const float* sumsq, const float* pivot, int C, long long P, float eps,
                               float momentum, const float* gamma, const float* beta, float* mean, float* rstd,
                               float* scale, float* shift, float* running_mean, float* running_var, cudaStream_t st) {
    FI_REQUIRE(sum && sumsq && gamma && beta && mean && rstd && scale && shift && C > 0 && P > 0, "bn_finalize: bad arguments");
    bn_finalize_kernel<<<(C + 255) / 256, 256, 0, st>>>(sum, sumsq, pivot, C, 1.0f / static_cast<float>(P),
                                                        P > 1 ? static_cast<float>(P) / static_cast<float>(P - 1) : 1.f, eps,
                                                        momentum, gamma, beta, mean, rstd, scale, shift, running_mean,
                                                        running_var);
    return last_error();
}
const char* bn_apply_relu_launch(const void* z, long long P, int C, const float* scale, const float* shift, void* a,
                                 cudaStream_t st) {
    FI_REQUIRE(z && a && scale && shift && P > 0 && C % 8 == 0, "bn_apply: bad arguments");
    const long long n8 = P * (C / 8);
    bn_apply_relu_kernel<<<apply_blocks(n8, C / 8), 256, 0, st>>>(static_cast<const uint4*>(z), n8, C / 8, scale, shift,
                                                                  static_cast<uint4*>(a));
    return last_error();
}
const char* head_forward_launch(const void* a, int N, long long HW, const float* w, const float* b, int ncls, float* y,
                                cudaStream_t st) {
    FI_REQUIRE(a && w && b && y && ncls >= 1 && ncls <= 4 && N > 0 && HW > 0, "head_forward: bad arguments");
    const int grid = blocks_for(N * HW * 8, 256 * 2, 148 * 8);
    const uint4* ap = static_cast<const uint4*>(a);
    switch (ncls) {
        case 1: head_forward_kernel<1><<<grid, 256, 0, st>>>(ap, N * HW, HW, w, b, y); break;
        case 2: head_forward_kernel<2><<<grid, 256, 0, st>>>(ap, N * HW, HW, w, b, y); break;
        case 3: head_forward_kernel<3><<<grid, 256, 0, st>>>(ap, N * HW, HW, w, b, y); break;
        default: head_forward_kernel<4><<<grid, 256, 0, st>>>(ap, N * HW, HW, w, b, y); break;
    }
    return last_error();
}
const char* mse_launch(const float* y, const float* t, long long n, float* loss, float* dy, cudaStream_t st) {
    FI_REQUIRE(y && t && loss && dy && n > 0, "mse: bad arguments");
    mse_kernel<<<blocks_for(n, 256), 256, 0, st>>>(y, t, n, 1.0f / static_cast<float>(n), loss, dy);
    return last_error();
}
const char* combined_loss_launch(const float* y, const float* t, int planes, int H, int W, float mse_w, float ssim_w,
                                 float* loss, float* dy, cudaStream_t st) {
    FI_REQUIRE(y && t && loss && dy && planes > 0 && H > 0 && W > 0 && planes <= 65535, "combined_loss: bad arguments");
    GaussWindow gw;   // the reference's window: exp(-(i-5)^2 / (2 * 1.5^2)) normalised in fp32
    float sum = 0.f;
    for (int i = 0; i <= 2 * SL_R; ++i) {
        gw.g[i] = static_cast<float>(exp(-static_cast<double>((i - SL_R) * (i - SL_R)) / (2.0 * 1.5 * 1.5)));
        sum += gw.g[i];
    }
    for (int i = 0; i <= 2 * SL_R; ++i) gw.g[i] /= sum;
    static std::atomic<uint64_t> configured{0};
    const int smem = SL_SMEM_FLOATS * static_cast<int>(sizeof(float));
    if (!smem_opt_in(combined_loss_kernel, smem, configured)) return "combined_loss: cudaFuncSetAttribute failed";
    const float inv_n = 1.0f / (static_cast<float>(planes) * H * W);
    const int tiles = ((W + SL_TILE - 1) / SL_TILE) * ((H + SL_TILE - 1) / SL_TILE);
    // loss = mse_w * mean(diff^2) + ssim_w * (1 - mean(S)): the constant ssim_w is added by the first block's caller
    ssim_offset_kernel<<<1, 1, 0, st>>>(loss, ssim_w);
    combined_loss_kernel<<<dim3(tiles, planes), 256, smem, st>>>(y, t, H, W, gw, mse_w * inv_n, ssim_w * inv_n, loss, dy);
    return last_error();
}
const char* head_backward_launch(const void* a, const float* dy, int N, long long HW, const float* w, int ncls, void* da,
                                 float* dw, float* db, cudaStream_t st) {
    FI_REQUIRE(a && dy && w && da && dw && db && ncls >= 1 && ncls <= 4, "head_backward: bad arguments");
    const int grid = blocks_for(N * HW * 8, 256, 148 * 8);
    const uint4* ap = static_cast<const uint4*>(a);
    uint4* dap = static_cast<uint4*>(da);
    switch (ncls) {
        case 1: head_backward_kernel<1><<<grid, 256, 0, st>>>(ap, dy, N * HW, HW, w, dap, dw, db); break;
        case 2: head_backward_kernel<2><<<grid, 256, 0, st>>>(ap, dy, N * HW, HW, w, dap, dw, db); break;
        case 3: head_backward_kernel<3><<<grid, 256, 0, st>>>(ap, dy, N * HW, HW, w, dap, dw, db); break;
        default: head_backward_kernel<4><<<grid, 256, 0, st>>>(ap, dy, N * HW, HW, w, dap, dw, db); break;
    }
    return last_error();
}
const char* bn_relu_bwd_reduce_launch(const void* dA, const void* z, long long P, int C, const float* mean,
                                      const float* rstd, const float* scale, const float* shift, float* dbeta,
                                      float* dgamma, cudaStream_t st) {
    FI_REQUIRE(dA && z && mean && rstd && scale && shift && dbeta && dgamma && C % 8 == 0 && C <= RED_MAX_C,
               "bn_bwd_reduce: bad arguments");
    bn_relu_bwd_reduce_kernel<<<reduce_blocks(P, C / 8, 3), 256, 0, st>>>(
        static_cast<const uint4*>(dA), static_cast<const uint4*>(z), P, C / 8, mean, rstd, scale, shift, dbeta, dgamma);
    return last_error();
}
const char* bn_relu_bwd_apply_launch(const void* dA, const void* z, long long P, int C, const float* mean,
                                     const float* rstd, const float* gamma, const float* beta, const float* dbeta,
                                     const float* dgamma, void* dz, cudaStream_t st) {
    FI_REQUIRE(dA && z && dz && mean && rstd && gamma && beta && dbeta && dgamma && C % 8 == 0, "bn_bwd_apply: bad arguments");
    const long long n8 = P * (C / 8);
    bn_relu_bwd_apply_kernel<<<apply_blocks(n8, C / 8), 256, 0, st>>>(
        static_cast<const uint4*>(dA), static_cast<const uint4*>(z), n8, C / 8, 1.0f / static_cast<float>(P), mean, rstd,
        gamma, beta, dbeta, dgamma, static_cast<uint4*>(dz));
    return last_error();
}
const char* maxpool_bwd_add_launch(const void* a_full, const void* a_pool, const void* d_pool, const void* d_skip,
                                   void* d_full, int N, int H, int W, int C, cudaStream_t st) {
    FI_REQUIRE(a_full && a_pool && d_pool && d_full && C % 8 == 0 && H >= 2 && W >= 2, "maxpool_bwd: bad arguments");
    maxpool_bwd_add_kernel<<<blocks_for(static_cast<long long>(N) * (H / 2) * (W / 2) * (C / 8), 256), 256, 0, st>>>(
        static_cast<const uint4*>(a_full), static_cast<const uint4*>(a_pool), static_cast<const uint4*>(d_pool),
        static_cast<const uint4*>(d_skip), static_cast<uint4*>(d_full), N, H, W, C / 8);
    return last_error();
}
const char* upsample2x_bwd_launch(const void* d_up, void* d_lo, int N, int h, int w, int C, cudaStream_t st) {
    FI_REQUIRE(d_up && d_lo && C % 8 == 0, "upsample_bwd: bad arguments");
    upsample2x_bwd_kernel<<<blocks_for(static_cast<long long>(N) * h * w * (C / 8), 256), 256, 0, st>>>(
        static_cast<const uint4*>(d_up), static_cast<uint4*>(d_lo), N, h, w, C / 8);
    return last_error();
}
const char* stem_wgrad_launch(const void* dz, const float* x, int N, int H, int W, int cin, float* dW, cudaStream_t st) {
    FI_REQUIRE(dz && x && dW && cin >= 1 && cin <= 6 && static_cast<long long>(N) * H * W < (1LL << 31), "stem_wgrad: bad arguments");
    const int grid = blocks_for(static_cast<long long>(N) * H * ((W + STEM_WG_TILE - 1) / STEM_WG_TILE), 2, 148 * 4);
    const uint32_t* g = static_cast<const uint32_t*>(dz);
    switch (cin) {
        case 1: stem_wgrad_kernel<1><<<grid, 256, 0, st>>>(g, x, N, H, W, dW); break;
        case 2: stem_wgrad_kernel<2><<<grid, 256, 0, st>>>(g, x, N, H, W, dW); break;   // grayscale frame pair
        case 3: stem_wgrad_kernel<3><<<grid, 256, 0, st>>>(g, x, N, H, W, dW); break;
        case 4: stem_wgrad_kernel<4><<<grid, 256, 0, st>>>(g, x, N, H, W, dW); break;
        case 6: stem_wgrad_kernel<6><<<grid, 256, 0, st>>>(g, x, N, H, W, dW); break;   // RGB frame pair
        default: return "stem_wgrad: built for 1, 2, 3, 4 or 6 input channels";
    }
    return last_error();
}
const char* unpack_conv_grad_launch(const float* dW, int cout, int cin, float* grad, cudaStream_t st) {
    FI_REQUIRE(dW && grad && cout > 0 && cin > 0, "unpack_conv_grad: bad arguments");
    const long long n = static_cast<long long>(cout) * cin;
    unpack_conv_grad_kernel<<<blocks_for(n, 256), 256, 0, st>>>(dW, n, grad);
    return last_error();
}
const char* adam_launch(float* p, const float* g, float* m, float* v, long long n, float lr, float b1, float b2, float eps,
                        int step, const float* hyper, cudaStream_t st) {
    FI_REQUIRE(p && g && m && v && n > 0 && (step >= 1 || hyper), "adam: bad arguments");
    adam_kernel<<<blocks_for(n, 256), 256, 0, st>>>(p, g, m, v, n, lr, b1, b2, eps, static_cast<float>(step), hyper);
    return last_error();
}
const char* stem_pack_device_launch(const float* w, int cin, void* out, cudaStream_t st) {
    FI_REQUIRE(w && out && cin >= 1 && cin <= 8, "stem_pack: bad arguments");
    const int kp = stem_packed_k(cin);
    stem_pack_kernel<<<(64 * kp + 255) / 256, 256, 0, st>>>(w, cin, kp, static_cast<__nv_bfloat16*>(out));
    return last_error();
}
const char* pack_conv_launch(const float* w, int co, int ci, void* fwd, void* bwd, cudaStream_t st) {
    FI_REQUIRE(w && (fwd || bwd) && co > 0 && ci > 0, "pack_conv: bad arguments");
    pack_conv_kernel<<<dim3(blocks_for(static_cast<long long>(co) * ci, 256), 2), 256, 0, st>>>(
        w, co, ci, static_cast<__nv_bfloat16*>(fwd), static_cast<__nv_bfloat16*>(bwd));
    return last_error();
}

}  // namespace fi
