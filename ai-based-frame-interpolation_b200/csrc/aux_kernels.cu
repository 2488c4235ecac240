// CUDA-core kernels of the frame-synthesis path (the stem convolution lives in stem_mma.cu): the bilinear
// decoder upsample, frame-pair packing, output post-processing, the fused SSIM+PSNR metric kernel, the
// frame-pair SAD of scene-cut detection and the training-batch gather from the device frame cache.
#include "aux_kernels.cuh"
#include "ptx.cuh"

namespace fi {

namespace {

__device__ __forceinline__ float div255_u8(uint32_t u) {
    // image.astype(float32)/255.0 rounded to fp32 (reference model/train.py:138, model/inference.py:32).
    // u/255 is formed as u*(1/255) plus one FMA residual correction, which is the correctly rounded quotient for all
    // 256 inputs (checked exhaustively by tests/test_gpu_aux_kernels.py::test_pack_pair_bit_exact and
    // tests/test_gpu_frame_cache.py) at a third of the instruction count of an IEEE division.
    const float x = static_cast<float>(u);
    const float r = 1.0f / 255.0f;
    const float q = __fmul_rn(x, r);
    return __fmaf_rn(__fmaf_rn(-q, 255.0f, x), r, q);
}

__device__ __forceinline__ float norm_u8(uint32_t u) {
    // then 2.0*image-1.0, rounded to fp32 (reference model/inference.py:32-35)
    return __fmaf_rn(2.0f, div255_u8(u), -1.0f);  // 2*q is exact, so this is fl(2*q - 1)
}

// ------------------------------------------------------------------------------------------------ bilinear x2
__device__ __forceinline__ float bf_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }

// Packed fp32 pairs (FFMA2 on sm_100): one instruction per two lanes of arithmetic, same IEEE results as scalar fma.
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
    return static_cast<uint64_t>(__float_as_uint(lo)) | (static_cast<uint64_t>(__float_as_uint(hi)) << 32);
}
__device__ __forceinline__ uint64_t bf16x2_to_f32x2(uint32_t v) {   // (lo, hi) bf16 -> (lo, hi) fp32, exact
    return static_cast<uint64_t>(v << 16) | (static_cast<uint64_t>(v & 0xffff0000u) << 32);
}
__device__ __forceinline__ uint64_t mul_f32x2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ uint32_t f32x2_to_bf16x2(uint64_t v) {
    return pack_bf16x2(__uint_as_float(static_cast<uint32_t>(v)), __uint_as_float(static_cast<uint32_t>(v >> 32)));
}

// One block row = one output row (blockIdx.y = n*2h + oy): the vertical taps/weights are block-uniform, index math is
// 32-bit (a shift when the channel-group count is a power of two), and consecutive threads walk (ox, channel-group) so
// both the 16-byte gathers and the store are coalesced. The bf16 path blends with the four tap weights
// w = (hy|ly) * (hx|lx) on packed fp32 pairs: 4 FFMA2 per 32-bit word of output.
__global__ void __launch_bounds__(256)
upsample2x_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int h, int w, int c8,
                  const uint4* __restrict__ src_lo, uint4* __restrict__ dst_lo) {
    pdl_launch_dependents();
    pdl_wait();  // launched with programmatic stream serialization: the layer below is complete from here on
    const int oh = 2 * h, ow = 2 * w;
    const int n = blockIdx.y / oh, oy = blockIdx.y - n * oh;
    const float rh = oh > 1 ? static_cast<float>(h - 1) / static_cast<float>(oh - 1) : 0.f;
    const float rw = ow > 1 ? static_cast<float>(w - 1) / static_cast<float>(ow - 1) : 0.f;
    const float fy = rh * oy;
    const int y0 = static_cast<int>(fy);
    const int y1 = y0 + (y0 < h - 1 ? 1 : 0);
    const float ly = fy - y0, hy = 1.f - ly;
    const uint4* row0 = src + (static_cast<size_t>(n) * h + y0) * w * c8;
    const uint4* row1 = src + (static_cast<size_t>(n) * h + y1) * w * c8;
    uint4* out = dst + (static_cast<size_t>(n) * oh + oy) * ow * c8;
    const int items = ow * c8;
    const int c8_shift = (c8 & (c8 - 1)) == 0 ? __ffs(c8) - 1 : -1;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < items; i += gridDim.x * 256) {
        const int ox = c8_shift >= 0 ? i >> c8_shift : i / c8, cg = i - ox * c8;
        const float fx = rw * ox;
        const int x0 = static_cast<int>(fx);
        const int x1 = x0 + (x0 < w - 1 ? 1 : 0);
        const float lx = fx - x0, hx = 1.f - lx;
        const uint4 p00 = __ldg(row0 + x0 * c8 + cg);
        const uint4 p01 = __ldg(row0 + x1 * c8 + cg);
        const uint4 p10 = __ldg(row1 + x0 * c8 + cg);
        const uint4 p11 = __ldg(row1 + x1 * c8 + cg);
        const uint32_t a[4] = {p00.x, p00.y, p00.z, p00.w}, b[4] = {p01.x, p01.y, p01.z, p01.w};
        const uint32_t c[4] = {p10.x, p10.y, p10.z, p10.w}, e[4] = {p11.x, p11.y, p11.z, p11.w};
        uint32_t o[4];
        if (src_lo == nullptr) {
            const float w00 = hy * hx, w01 = hy * lx, w10 = ly * hx, w11 = ly * lx;
            const uint64_t p00w = pack_f32x2(w00, w00), p01w = pack_f32x2(w01, w01);
            const uint64_t p10w = pack_f32x2(w10, w10), p11w = pack_f32x2(w11, w11);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                uint64_t acc = mul_f32x2(bf16x2_to_f32x2(a[k]), p00w);
                acc = fma_f32x2(bf16x2_to_f32x2(b[k]), p01w, acc);
                acc = fma_f32x2(bf16x2_to_f32x2(c[k]), p10w, acc);
                acc = fma_f32x2(bf16x2_to_f32x2(e[k]), p11w, acc);
                o[k] = f32x2_to_bf16x2(acc);
            }
            out[i] = make_uint4(o[0], o[1], o[2], o[3]);
        } else {
            // precise mode: every value is hi + lo (exact in fp32); the result is split again
            const size_t d0 = (static_cast<size_t>(n) * h + y0) * w * c8, d1 = (static_cast<size_t>(n) * h + y1) * w * c8;
            const uint4 q00 = __ldg(src_lo + d0 + x0 * c8 + cg), q01 = __ldg(src_lo + d0 + x1 * c8 + cg);
            const uint4 q10 = __ldg(src_lo + d1 + x0 * c8 + cg), q11 = __ldg(src_lo + d1 + x1 * c8 + cg);
            const uint32_t al[4] = {q00.x, q00.y, q00.z, q00.w}, bl[4] = {q01.x, q01.y, q01.z, q01.w};
            const uint32_t cl[4] = {q10.x, q10.y, q10.z, q10.w}, el[4] = {q11.x, q11.y, q11.z, q11.w};
            uint32_t ol[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const float lo = hy * (hx * (bf_lo(a[k]) + bf_lo(al[k])) + lx * (bf_lo(b[k]) + bf_lo(bl[k]))) +
                                 ly * (hx * (bf_lo(c[k]) + bf_lo(cl[k])) + lx * (bf_lo(e[k]) + bf_lo(el[k])));
                const float hi = hy * (hx * (bf_hi(a[k]) + bf_hi(al[k])) + lx * (bf_hi(b[k]) + bf_hi(bl[k]))) +
                                 ly * (hx * (bf_hi(c[k]) + bf_hi(cl[k])) + lx * (bf_hi(e[k]) + bf_hi(el[k])));
                o[k] = pack_bf16x2(lo, hi);
                ol[k] = pack_bf16x2(lo - bf_lo(o[k]), hi - bf_hi(o[k]));
            }
            out[i] = make_uint4(o[0], o[1], o[2], o[3]);
            (dst_lo + (static_cast<size_t>(n) * oh + oy) * ow * c8)[i] = make_uint4(ol[0], ol[1], ol[2], ol[3]);
        }
    }
}

// ------------------------------------------------------------------------------------------------ max pool 2x2
// nn.MaxPool2d(2) on bf16 NHWC (floor semantics). Inside the network the pool is fused into the producing conv's
// epilogue; this kernel serves the stand-alone Down module only.
__global__ void __launch_bounds__(256)
maxpool2x2_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int H, int W, int c8) {
    const int oh = H / 2, ow = W / 2;
    const int n = blockIdx.y / oh, oy = blockIdx.y - n * oh;
    const uint4* r0 = src + (static_cast<size_t>(n) * H + 2 * oy) * W * c8;
    const uint4* r1 = r0 + static_cast<size_t>(W) * c8;
    uint4* out = dst + (static_cast<size_t>(n) * oh + oy) * ow * c8;
    for (int i = blockIdx.x * 256 + threadIdx.x; i < ow * c8; i += gridDim.x * 256) {
        const int ox = i / c8, cg = i - ox * c8;
        const uint4 a = __ldg(r0 + (2 * ox) * c8 + cg), b = __ldg(r0 + (2 * ox + 1) * c8 + cg);
        const uint4 c = __ldg(r1 + (2 * ox) * c8 + cg), d = __ldg(r1 + (2 * ox + 1) * c8 + cg);
        uint4 m;
        m.x = bf16x2_max(bf16x2_max(a.x, b.x), bf16x2_max(c.x, d.x));
        m.y = bf16x2_max(bf16x2_max(a.y, b.y), bf16x2_max(c.y, d.y));
        m.z = bf16x2_max(bf16x2_max(a.z, b.z), bf16x2_max(c.z, d.z));
        m.w = bf16x2_max(bf16x2_max(a.w, b.w), bf16x2_max(c.w, d.w));
        out[i] = m;
    }
}

// ------------------------------------------------------------------------------------------------ pack / post
// out[n, k, :, :] = 2*(f[n, k mod C]/255) - 1 with f = f0 for k < C else f1: 16 pixels (one 128-bit load) per thread.
__global__ void __launch_bounds__(256)
pack_pair_kernel(const uint8_t* __restrict__ f0, const uint8_t* __restrict__ f1, float* __restrict__ out, int N, int C,
                 size_t plane, int vec) {
    if (vec) {
        const size_t plane16 = plane / 16;
        const size_t total = static_cast<size_t>(N) * 2 * C * plane16;
        for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
             i += static_cast<size_t>(gridDim.x) * blockDim.x) {
            const size_t pi = i % plane16;
            const size_t nk = i / plane16;
            const int k = static_cast<int>(nk % (2 * C));
            const size_t n = nk / (2 * C);
            const uint8_t* srcp = (k < C ? f0 : f1) + (n * C + (k < C ? k : k - C)) * plane;
            const uint4 v = __ldg(reinterpret_cast<const uint4*>(srcp) + pi);
            const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
            float4* o = reinterpret_cast<float4*>(out + nk * plane) + pi * 4;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float4 r;
                r.x = norm_u8(wv[q] & 0xff);
                r.y = norm_u8((wv[q] >> 8) & 0xff);
                r.z = norm_u8((wv[q] >> 16) & 0xff);
                r.w = norm_u8(wv[q] >> 24);
                o[q] = r;
            }
        }
    } else {
        const size_t total = static_cast<size_t>(N) * 2 * C * plane;
        for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
             i += static_cast<size_t>(gridDim.x) * blockDim.x) {
            const size_t pi = i % plane;
            const size_t nk = i / plane;
            const int k = static_cast<int>(nk % (2 * C));
            const size_t n = nk / (2 * C);
            const uint8_t* srcp = (k < C ? f0 : f1) + (n * C + (k < C ? k : k - C)) * plane;
            out[i] = norm_u8(srcp[pi]);
        }
    }
}

__device__ __forceinline__ uint32_t post_u8(float t) {
    float u = __fmul_rn(__fadd_rn(t, 1.0f), 0.5f);  // (tensor + 1.0) / 2.0
    u = fminf(fmaxf(u, 0.0f), 1.0f);                // clamp(0, 1)
    return static_cast<uint32_t>(__fmul_rn(u, 255.0f)) & 0xff;  // *255 -> astype(uint8) truncates
}

__global__ void __launch_bounds__(256)
head_post_kernel(const float* __restrict__ y, uint8_t* __restrict__ out, size_t n, int vec) {
    const size_t n16 = vec ? n / 16 : 0;
    for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n16;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        const float4* p = reinterpret_cast<const float4*>(y) + i * 4;
        uint32_t o[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 v = __ldg(p + q);
            o[q] = post_u8(v.x) | (post_u8(v.y) << 8) | (post_u8(v.z) << 16) | (post_u8(v.w) << 24);
        }
        reinterpret_cast<uint4*>(out)[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
    for (size_t i = n16 * 16 + blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n;
         i += static_cast<size_t>(gridDim.x) * blockDim.x) {
        out[i] = static_cast<uint8_t>(post_u8(y[i]));
    }
}

// ------------------------------------------------------------------------------------------------ SSIM + PSNR
// compute_ssim / compute_psnr of the reference (model/evaluation.py:194-218) call scikit-image with data_range=255:
// 7x7 uniform window, sample covariance (x49/48), K1=.01, K2=.03, mean over the image cropped by 3; PSNR from the MSE.
// Colour images are scored as structural_similarity(..., channel_axis=-1): the mean over channels of each channel's
// grey SSIM (each with its own 3-pixel crop), and PSNR over all C*H*W samples.
// All 49-pixel window sums of u8 data are exact in int32, so the per-pixel ratio is formed from exact integers:
//   S = (2 Sx Sy + C1 49^2)(2(49 Sxy - Sx Sy) + C2 48 49) / ((Sx^2 + Sy^2 + C1 49^2)(49 Sqq - Sx^2 - Sy^2 + C2 48 49))
// with Sx = sum x, Sy = sum y, Sqq = sum (x^2 + y^2), Sxy = sum x y over the window.
// Block = one channel of one image (blockIdx.z = n*C + c) x SS_COLS columns x SS_ROWS rows. Thread = 4 adjacent
// columns, sliding down SS_ROWS rows: horizontal window sums slide along x, vertical along y.
constexpr int SS_THREADS = 128;
constexpr int SS_COLS = 4 * SS_THREADS;  // columns per block
constexpr int SS_ROWS = 36;              // owned rows per block (+6 halo rows streamed)

// Pixels c0 .. c0+3 of one channel of a row, packed little-endian into a word (0 outside [0, W)). PS is the pixel
// stride: 1 = planar (one word load when aligned), 3 = interleaved BGR, where rowp points at pixel 0 of channel 0 and
// the 12 bytes of pixels c0 .. c0+3 are three aligned words; __byte_perm picks channel `ch`'s bytes 3k + ch out of
// them (sel1 from words 0-1, sel2 adds word 2), so the window arithmetic below sees the same word either way.
template <int PS>
__device__ __forceinline__ uint32_t load_word_guarded(const uint8_t* rowp, int c0, int W, bool aligned, int ch,
                                                      uint32_t sel1, uint32_t sel2) {
    if (c0 >= 0 && c0 + 3 < W && aligned) {
        if (PS == 1) return __ldg(reinterpret_cast<const uint32_t*>(rowp + c0));
        const uint32_t* p = reinterpret_cast<const uint32_t*>(rowp + 3 * c0);
        return __byte_perm(__byte_perm(__ldg(p), __ldg(p + 1), sel1), __ldg(p + 2), sel2);
    }
    uint32_t v = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = c0 + k;
        if (c >= 0 && c < W) v |= static_cast<uint32_t>(__ldg(rowp + PS * c + (PS == 1 ? 0 : ch))) << (8 * k);
    }
    return v;
}

// One operand: channel plane (n, c) starts at ptr + n*batch + c*chan, rows are `row` bytes apart. Interleaved
// operands (PS = 3) keep chan = 1 and are addressed from channel 0 (the loader adds the channel).
struct SsimOperand {
    const uint8_t* ptr;
    long long batch, chan, row;
    int aligned;  // every word the loader reads is 4-byte aligned
};

template <int PA, int PB>
__global__ void __launch_bounds__(SS_THREADS, 4)
ssim_psnr_kernel(SsimOperand a, SsimOperand b, int C, int H, int W, double* __restrict__ part_ssim,
                 unsigned long long* __restrict__ part_ssd) {
    const int tid = threadIdx.x;
    const int n = blockIdx.z / C, ch = blockIdx.z - n * C;
    const int xb = blockIdx.x * SS_COLS + 4 * tid;  // first owned column
    const int ty0 = blockIdx.y * SS_ROWS;
    const uint8_t* ia = a.ptr + n * a.batch + (PA == 1 ? ch * a.chan : 0);
    const uint8_t* ib = b.ptr + n * b.batch + (PB == 1 ? ch * b.chan : 0);
    // __byte_perm selectors of channel ch in an interleaved span: bytes ch, ch+3 from words 0-1 (+ ch+6 when < 8),
    // then the rest from word 2
    const uint32_t sel1 = ch | (ch + 3) << 4 | (ch + 6 < 8 ? (ch + 6) << 8 : 0u);
    const uint32_t sel2 = 0x10u | (ch + 6 < 8 ? 2u : static_cast<uint32_t>(ch + 2)) << 8 | static_cast<uint32_t>(ch + 5) << 12;

    uint32_t ring1[7][4], ringq[7][4], ringp[7][4];
    uint32_t v1[4] = {0, 0, 0, 0}, vq[4] = {0, 0, 0, 0}, vp[4] = {0, 0, 0, 0};
#pragma unroll
    for (int s = 0; s < 7; ++s)
#pragma unroll
        for (int j = 0; j < 4; ++j) ring1[s][j] = ringq[s][j] = ringp[s][j] = 0;

    float ssim_acc = 0.f;
    uint32_t ssd = 0;
    const float K1 = 6.5025f * 2401.0f;   // C1 * 49^2
    const float K2 = 58.5225f * 2352.0f;  // C2 * 48 * 49

    // The six words of row i+1 are requested before row i is reduced, so their latency overlaps the arithmetic.
    // Rows are fetched in order, so the two row pointers advance by their strides (32-bit: a row is < 2 GB).
    uint32_t na[3], nb[3];
    const int row_a = static_cast<int>(a.row), row_b = static_cast<int>(b.row);
    const bool aligned = a.aligned && b.aligned;
    ia += static_cast<long long>(ty0 - 3) * a.row;
    ib += static_cast<long long>(ty0 - 3) * b.row;
    auto fetch_row = [&](int yin) {
#pragma unroll
        for (int k = 0; k < 3; ++k) na[k] = nb[k] = 0;
        if (yin >= 0 && yin < H && xb - 4 < W) {
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                na[k] = load_word_guarded<PA>(ia, xb - 4 + 4 * k, W, aligned, ch, sel1, sel2);
                nb[k] = load_word_guarded<PB>(ib, xb - 4 + 4 * k, W, aligned, ch, sel1, sel2);
            }
        }
        ia += row_a;
        ib += row_b;
    };
    fetch_row(ty0 - 3);
    for (int rb = 0; rb < SS_ROWS + 6; rb += 7) {
#pragma unroll
        for (int s = 0; s < 7; ++s) {
            const int i = rb + s;
            if (i < SS_ROWS + 6) {
                const int yin = ty0 - 3 + i;
                const uint32_t wa[3] = {na[0], na[1], na[2]}, wb[3] = {nb[0], nb[1], nb[2]};
                if (i + 1 < SS_ROWS + 6) fetch_row(yin + 1);
                // Pixels xb-3 .. xb+6 are bytes 1..10 of the 12-byte span {w0,w1,w2}; the 7-pixel window of owned column j
                // is bytes j+1 .. j+7. Two funnel shifts align it into (4 bytes, 3 bytes) and __dp4a forms the five
                // window sums directly on packed bytes (no per-pixel unpack / multiply):
                uint32_t h1[4], hq[4], hp[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t sh = 8 * (j + 1);
                    const uint32_t xa = j < 3 ? __funnelshift_r(wa[0], wa[1], sh) : wa[1];
                    const uint32_t xb2 = (j < 3 ? __funnelshift_r(wa[1], wa[2], sh) : wa[2]) & 0x00ffffffu;
                    const uint32_t ya = j < 3 ? __funnelshift_r(wb[0], wb[1], sh) : wb[1];
                    const uint32_t yb2 = (j < 3 ? __funnelshift_r(wb[1], wb[2], sh) : wb[2]) & 0x00ffffffu;
                    const uint32_t sx = __dp4a(xa, 0x01010101u, __dp4a(xb2, 0x01010101u, 0u));
                    const uint32_t sy = __dp4a(ya, 0x01010101u, __dp4a(yb2, 0x01010101u, 0u));
                    h1[j] = sx | (sy << 16);  // each <= 7*255: the two 16-bit halves never interact
                    hq[j] = __dp4a(xa, xa, __dp4a(xb2, xb2, __dp4a(ya, ya, __dp4a(yb2, yb2, 0u))));
                    hp[j] = __dp4a(xa, ya, __dp4a(xb2, yb2, 0u));
                }
                if (yin >= ty0 && yin < ty0 + SS_ROWS) {
                    // squared error of the 4 owned pixels (= bytes of w1): sum (x-y)^2 = x.x + y.y - 2 x.y
                    ssd += __dp4a(wa[1], wa[1], __dp4a(wb[1], wb[1], 0u)) - 2u * __dp4a(wa[1], wb[1], 0u);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    v1[j] += h1[j] - ring1[s][j];
                    vq[j] += hq[j] - ringq[s][j];
                    vp[j] += hp[j] - ringp[s][j];
                    ring1[s][j] = h1[j];
                    ringq[s][j] = hq[j];
                    ringp[s][j] = hp[j];
                }
                const int yo = yin - 3;  // window centre row of the sums now held
                if (i >= 6 && yo >= 3 && yo < H - 3) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int xo = xb + j;
                        if (xo >= 3 && xo < W - 3) {
                            const int sx = static_cast<int>(v1[j] & 0xffff), sy = static_cast<int>(v1[j] >> 16);
                            const int sxsy = sx * sy;
                            const int sq2 = sx * sx + sy * sy;
                            const float a1 = static_cast<float>(2 * sxsy) + K1;
                            const float b1 = static_cast<float>(sq2) + K1;
                            const float a2 = static_cast<float>(2 * (49 * static_cast<int>(vp[j]) - sxsy)) + K2;
                            const float b2 = static_cast<float>(49 * static_cast<int>(vq[j]) - sq2) + K2;
                            ssim_acc += __fdividef(a1 * a2, b1 * b2);  // |S| <= 1, operands ~1e17: well inside range
                        }
                    }
                }
            }
        }
    }

    // block reduction (fixed order -> deterministic partials)
    double ds = static_cast<double>(ssim_acc);
    unsigned long long du = ssd;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ds += __shfl_down_sync(0xffffffffu, ds, o);
        du += __shfl_down_sync(0xffffffffu, du, o);
    }
    __shared__ double sh_s[SS_THREADS / 32];
    __shared__ unsigned long long sh_u[SS_THREADS / 32];
    if ((tid & 31) == 0) {
        sh_s[tid >> 5] = ds;
        sh_u[tid >> 5] = du;
    }
    __syncthreads();
    if (tid == 0) {
        double ts = 0.0;
        unsigned long long tu = 0;
        for (int k = 0; k < SS_THREADS / 32; ++k) {
            ts += sh_s[k];
            tu += sh_u[k];
        }
        const size_t slot = (static_cast<size_t>(blockIdx.z) * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        part_ssim[slot] = ts;
        part_ssd[slot] = tu;
    }
}

// One block per image: each channel's partials are summed in a fixed order (so C = 1 is the grey result bit for bit),
// the channel SSIMs are averaged in channel order and the squared errors of all channels are summed in 64 bit.
__global__ void __launch_bounds__(256)
ssim_psnr_finalize_kernel(const double* __restrict__ part_ssim, const unsigned long long* __restrict__ part_ssd,
                          int nblk, int C, int H, int W, double* __restrict__ out) {
    const int n = blockIdx.x;
    __shared__ double sh_s[256];
    __shared__ unsigned long long sh_u[256];
    double ssim_sum = 0.0;
    unsigned long long sse = 0;
    for (int ch = 0; ch < C; ++ch) {
        const size_t base = (static_cast<size_t>(n) * C + ch) * nblk;
        double s = 0.0;
        unsigned long long u = 0;
        for (int i = threadIdx.x; i < nblk; i += 256) {
            s += part_ssim[base + i];
            u += part_ssd[base + i];
        }
        sh_s[threadIdx.x] = s;
        sh_u[threadIdx.x] = u;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if (threadIdx.x < o) {
                sh_s[threadIdx.x] += sh_s[threadIdx.x + o];
                sh_u[threadIdx.x] += sh_u[threadIdx.x + o];
            }
            __syncthreads();
        }
        ssim_sum += sh_s[0] / (static_cast<double>(H - 6) * (W - 6));
        sse += sh_u[0];
        __syncthreads();  // sh_s / sh_u are rewritten by the next channel
    }
    if (threadIdx.x == 0) {
        const double mse = static_cast<double>(sse) / (static_cast<double>(H) * W * C);
        // skimage peak_signal_noise_ratio: 10*log10(data_range^2 / mse); identical images -> inf
        out[2 * n + 0] = sse == 0 ? __longlong_as_double(0x7ff0000000000000LL) : 10.0 * log10(65025.0 / mse);
        out[2 * n + 1] = ssim_sum / C;
    }
}

// ------------------------------------------------------------------------------------------------ pair SAD
// sad[p] = sum_k |f[p+1][k] - f[p][k]| over all frame_bytes bytes of every consecutive frame pair (scene-cut statistic).
// blockIdx.y = group of PS_GROUP consecutive pairs; a thread walks its 16-byte chunks through the group's frames with
// the previous frame's chunk in registers, so each frame is read once per group (group edges twice: +1/PS_GROUP).
// Per-pair sums stay in 32-bit registers (a chunk adds at most 16*255; the launcher keeps <= 2^20 chunks per thread)
// and are reduced in 64 bit: one integer atomic per block and pair, exact and independent of the launch shape.
constexpr int PS_THREADS = 256;
constexpr int PS_GROUP = 8;

__global__ void __launch_bounds__(PS_THREADS)
pair_sad_kernel(const uint8_t* __restrict__ frames, long long frame_stride, long long frame_bytes, int n_pairs, int vec,
                unsigned long long* __restrict__ sad) {
    const int p0 = blockIdx.y * PS_GROUP;
    const int cnt = min(PS_GROUP, n_pairs - p0);
    const uint8_t* base = frames + p0 * frame_stride;
    uint32_t acc[PS_GROUP];
#pragma unroll
    for (int k = 0; k < PS_GROUP; ++k) acc[k] = 0;
    const long long tid = static_cast<long long>(blockIdx.x) * PS_THREADS + threadIdx.x;
    const long long nthr = static_cast<long long>(gridDim.x) * PS_THREADS;
    const long long n16 = vec ? frame_bytes / 16 : 0;
    for (long long c = tid; c < n16; c += nthr) {
        uint4 prev = __ldg(reinterpret_cast<const uint4*>(base) + c);
#pragma unroll
        for (int k = 0; k < PS_GROUP; ++k) {
            // past the group's last frame the same chunk is loaded again (an L1 hit) and adds 0: no predicated loads
            const int f = k + 1 < cnt ? k + 1 : cnt;
            const uint4 cur = __ldg(reinterpret_cast<const uint4*>(base + f * frame_stride) + c);
            acc[k] += __vsadu4(prev.x, cur.x) + __vsadu4(prev.y, cur.y) + __vsadu4(prev.z, cur.z) +
                      __vsadu4(prev.w, cur.w);
            prev = cur;
        }
    }
    // bytes not covered by 16-byte chunks: the tail of an aligned frame, or every byte of an unaligned one
    for (long long i = n16 * 16 + tid; i < frame_bytes; i += nthr) {
        int prev = __ldg(base + i);
#pragma unroll
        for (int k = 0; k < PS_GROUP; ++k) {
            const int f = k + 1 < cnt ? k + 1 : cnt;
            const int cur = __ldg(base + f * frame_stride + i);
            acc[k] += static_cast<uint32_t>(abs(cur - prev));
            prev = cur;
        }
    }
    __shared__ unsigned long long part[PS_THREADS / 32][PS_GROUP];
#pragma unroll
    for (int k = 0; k < PS_GROUP; ++k) {
        unsigned long long v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < cnt) {
        unsigned long long s = 0;
#pragma unroll
        for (int w = 0; w < PS_THREADS / 32; ++w) s += part[w][threadIdx.x];
        if (s) atomicAdd(sad + p0 + threadIdx.x, s);
    }
}

// ------------------------------------------------------------------------------------------------ triplet gather
// Training batches from the device-resident u8 frame cache: output row r = 3*b + k is
// out_k[b] = frames[triplets[samples[b]][k]] / 255 (FrameTripletDataset's img.astype(float32) / 255.0, bit for bit).
// blockIdx.y walks the rows (grid-stride), blockIdx.x the plane; a row's indices are block-uniform. A sample whose index
// or any of whose three frame indices is out of range has all three outputs written as NaN and nothing of it is read.
// Vector path: 16 pixels per thread, one 16-byte load and four 16-byte stores; the byte path covers any H*W.
constexpr int GT_THREADS = 256;

__global__ void __launch_bounds__(GT_THREADS)
gather_triplets_u8_kernel(const uint8_t* __restrict__ frames, long long n_frames, const int* __restrict__ triplets,
                          long long n_triplets, const long long* __restrict__ samples, long long rows, long long plane,
                          int vec, float* __restrict__ out0, float* __restrict__ out1, float* __restrict__ out2) {
    const float nan = __int_as_float(0x7fc00000);
    const long long tid = static_cast<long long>(blockIdx.x) * GT_THREADS + threadIdx.x;
    const long long nthr = static_cast<long long>(gridDim.x) * GT_THREADS;
    const long long n16 = vec ? plane / 16 : 0;
    for (long long row = blockIdx.y; row < rows; row += gridDim.y) {
        const long long b = row / 3;
        const int k = static_cast<int>(row - 3 * b);
        float* out = (k == 0 ? out0 : k == 1 ? out1 : out2) + b * plane;
        const long long s = __ldg(samples + b);
        bool ok = s >= 0 && s < n_triplets;
        long long f = 0;
        if (ok) {
            const int t0 = __ldg(triplets + 3 * s), t1 = __ldg(triplets + 3 * s + 1), t2 = __ldg(triplets + 3 * s + 2);
            ok = t0 >= 0 && t0 < n_frames && t1 >= 0 && t1 < n_frames && t2 >= 0 && t2 < n_frames;
            f = k == 0 ? t0 : k == 1 ? t1 : t2;
        }
        const uint8_t* src = frames + f * plane;
        for (long long i = tid; i < n16; i += nthr) {
            float4* o = reinterpret_cast<float4*>(out) + i * 4;
            if (ok) {
                const uint4 v = __ldg(reinterpret_cast<const uint4*>(src) + i);
                const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    o[q] = make_float4(div255_u8(wv[q] & 0xff), div255_u8((wv[q] >> 8) & 0xff),
                                       div255_u8((wv[q] >> 16) & 0xff), div255_u8(wv[q] >> 24));
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) o[q] = make_float4(nan, nan, nan, nan);
            }
        }
        for (long long i = n16 * 16 + tid; i < plane; i += nthr) out[i] = ok ? div255_u8(__ldg(src + i)) : nan;
    }
}

// ------------------------------------------------------------------------------------------------ crop gather
// Training batches of random windows from a cache of frames of different sizes (FrameTripletDataset(crop=S)):
// out_k[b][c][y][x] = frames[off[f] + (c*H + y0 + y)*W + x0 + (mirror ? S-1-x : x)] / 255 with f = rows[b][k], k < 3.
// One thread writes 4 consecutive output pixels of one output row with a 16-byte store; a warp covers 128 pixels of a
// row, so a 256-wide row is two coalesced warps. Source rows start at any byte: the 4 source bytes are funnel-shifted
// out of the (at most two) aligned 32-bit words that hold them, which never reads a word without a byte of the window;
// mirroring reverses the bytes of the same 4-byte run read from the mirrored position. A row whose frame indices,
// sizes or window are out of range is written as NaN (all three outputs) and none of its bytes are read.
constexpr int GC_THREADS = 256;

struct CropSrc {
    const uint8_t* base;   // first byte of the window's top-left pixel in plane 0
    long long plane;       // H*W
    int w;                 // row stride
};

__device__ __forceinline__ bool crop_src(const uint8_t* frames, long long frames_bytes, const long long* offsets,
                                         const int* sizes, long long n_frames, int C, int S, int f, int y0, int x0,
                                         CropSrc* out) {
    if (f < 0 || f >= n_frames) return false;
    const long long off = __ldg(offsets + f);
    const int h = __ldg(sizes + 2 * f), w = __ldg(sizes + 2 * f + 1);
    if (h < 1 || w < 1 || y0 < 0 || x0 < 0 || y0 > h - S || x0 > w - S) return false;
    const long long plane = static_cast<long long>(h) * w;
    if (off < 0 || off > frames_bytes - C * plane) return false;
    out->base = frames + off + static_cast<long long>(y0) * w + x0;
    out->plane = plane;
    out->w = w;
    return true;
}

__device__ __forceinline__ uint32_t load4_unaligned(const uint8_t* p) {
    // bytes p[0..3] as a little-endian word, from the aligned words that hold them
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~static_cast<uintptr_t>(3));
    const uint32_t sh = static_cast<uint32_t>(a & 3) * 8;
    const uint32_t lo = __ldg(w);
    if (sh == 0) return lo;
    return __funnelshift_r(lo, __ldg(w + 1), sh);
}

__global__ void __launch_bounds__(GC_THREADS)
gather_crops_u8_kernel(const uint8_t* __restrict__ frames, long long frames_bytes, const long long* __restrict__ offsets,
                       const int* __restrict__ sizes, long long n_frames, int C, const int* __restrict__ rows,
                       int S, long long units, float* __restrict__ out0, float* __restrict__ out1,
                       float* __restrict__ out2) {
    const float nan = __int_as_float(0x7fc00000);
    const int q = S / 4;                       // 4-pixel units per output row
    for (long long u = static_cast<long long>(blockIdx.x) * GC_THREADS + threadIdx.x; u < units;
         u += static_cast<long long>(gridDim.x) * GC_THREADS) {
        const long long r = u / q;             // output row: ((b*3 + k)*C + c)*S + y
        const int j = static_cast<int>(u - r * q);
        const int y = static_cast<int>(r % S);
        const long long bkc = r / S;
        const int c = static_cast<int>(bkc % C);
        const long long bk = bkc / C;
        const long long b = bk / 3;
        const int k = static_cast<int>(bk - 3 * b);
        const int* row = rows + 6 * b;
        const int y0 = __ldg(row + 3), x0 = __ldg(row + 4), mirror = __ldg(row + 5);
        CropSrc s0, s1, s2;
        const bool ok = crop_src(frames, frames_bytes, offsets, sizes, n_frames, C, S, __ldg(row), y0, x0, &s0) &&
                        crop_src(frames, frames_bytes, offsets, sizes, n_frames, C, S, __ldg(row + 1), y0, x0, &s1) &&
                        crop_src(frames, frames_bytes, offsets, sizes, n_frames, C, S, __ldg(row + 2), y0, x0, &s2);
        float* out = (k == 0 ? out0 : k == 1 ? out1 : out2) + ((b * C + c) * S + y) * static_cast<long long>(S) + 4 * j;
        float4 v = make_float4(nan, nan, nan, nan);
        if (ok) {
            const CropSrc& s = k == 0 ? s0 : k == 1 ? s1 : s2;
            const uint8_t* src = s.base + c * s.plane + static_cast<long long>(y) * s.w;
            uint32_t b4 = load4_unaligned(src + (mirror ? S - 4 - 4 * j : 4 * j));
            if (mirror) b4 = __byte_perm(b4, 0, 0x0123);
            v = make_float4(div255_u8(b4 & 0xff), div255_u8((b4 >> 8) & 0xff), div255_u8((b4 >> 16) & 0xff),
                            div255_u8(b4 >> 24));
        }
        *reinterpret_cast<float4*>(out) = v;
    }
}

int grid_for(size_t work_items, int threads) {
    size_t g = (work_items + threads - 1) / threads;
    const size_t cap = 148 * 16;  // grid-stride loops: a few waves of the 148 SMs is enough
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return static_cast<int>(g);
}

const char* last_launch_error() {
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

}  // namespace

const char* upsample2x_launch(const void* src, void* dst, int N, int h, int w, int C, cudaStream_t stream,
                              const void* src_lo, void* dst_lo) {
    if ((src_lo == nullptr) != (dst_lo == nullptr)) return "upsample: src_lo and dst_lo go together";
    if (C % 8) return "upsample: channels must be a multiple of 8";
    if (N <= 0 || h <= 0 || w <= 0) return "upsample: empty shape";
    if (static_cast<long long>(N) * 2 * h > 65535) return "upsample: N*2h must be <= 65535 (grid.y)";
    const int items = 2 * w * (C / 8);
    const int gx = (items + 1023) / 1024;  // 4 items per thread
    launch_kernel(upsample2x_kernel, dim3(gx, N * 2 * h), dim3(256), 0, stream, static_cast<const uint4*>(src),
                  static_cast<uint4*>(dst), h, w, C / 8, static_cast<const uint4*>(src_lo), static_cast<uint4*>(dst_lo));
    return last_launch_error();
}

const char* maxpool2x2_launch(const void* src, void* dst, int N, int H, int W, int C, cudaStream_t stream) {
    if (C % 8) return "maxpool: channels must be a multiple of 8";
    if (N <= 0 || H < 2 || W < 2) return "maxpool: needs at least a 2x2 image";
    if (static_cast<long long>(N) * (H / 2) > 65535) return "maxpool: N*(H/2) must be <= 65535 (grid.y)";
    const int items = (W / 2) * (C / 8);
    maxpool2x2_kernel<<<dim3((items + 1023) / 1024, N * (H / 2)), 256, 0, stream>>>(
        static_cast<const uint4*>(src), static_cast<uint4*>(dst), H, W, C / 8);
    return last_launch_error();
}

const char* pack_pair_launch(const uint8_t* f0, const uint8_t* f1, float* out, int N, int C, int H, int W,
                             cudaStream_t stream) {
    if (N <= 0 || C <= 0 || H <= 0 || W <= 0) return "pack: empty shape";
    const size_t plane = static_cast<size_t>(H) * W;
    const int vec = (plane % 16 == 0) && ((reinterpret_cast<uintptr_t>(f0) | reinterpret_cast<uintptr_t>(f1) |
                                           reinterpret_cast<uintptr_t>(out)) % 16 == 0);
    const size_t items = static_cast<size_t>(N) * 2 * C * (vec ? plane / 16 : plane);
    pack_pair_kernel<<<grid_for(items, 256), 256, 0, stream>>>(f0, f1, out, N, C, plane, vec);
    return last_launch_error();
}

const char* head_post_launch(const float* y, uint8_t* out, size_t n, cudaStream_t stream) {
    if (n == 0) return nullptr;
    const int vec = (reinterpret_cast<uintptr_t>(y) % 16 == 0) && (reinterpret_cast<uintptr_t>(out) % 16 == 0);
    head_post_kernel<<<grid_for(vec ? (n + 15) / 16 : n, 256), 256, 0, stream>>>(y, out, n, vec);
    return last_launch_error();
}

static void ssim_grid(int H, int W, int* gx, int* gy) {
    *gx = (W + SS_COLS - 1) / SS_COLS;
    *gy = (H + SS_ROWS - 1) / SS_ROWS;
}

size_t ssim_psnr_workspace_bytes(int N, int C, int H, int W) {
    int gx, gy;
    ssim_grid(H, W, &gx, &gy);
    return static_cast<size_t>(N) * C * gx * gy * 16;
}

// Pixel stride of a supported layout (1 planar, 3 interleaved BGR), or 0.
static int ssim_layout(const PlaneSrc& p) {
    if (p.batch_stride < 0 || p.chan_stride < 0 || p.row_stride < 0 || p.row_stride > 0x7fffffff) return 0;
    if (p.px_stride == 1) return 1;
    if (p.px_stride == 3 && p.chan_stride == 1 && p.channels == 3) return 3;
    return 0;
}

static SsimOperand ssim_operand(const PlaneSrc& p, int ps, int N) {
    const uint8_t* ptr = static_cast<const uint8_t*>(p.ptr);
    long long bits = static_cast<long long>(reinterpret_cast<uintptr_t>(ptr)) | p.row_stride;
    if (N > 1) bits |= p.batch_stride;
    if (ps == 1 && p.channels > 1) bits |= p.chan_stride;
    return SsimOperand{ptr, p.batch_stride, p.chan_stride, p.row_stride, static_cast<int>(bits % 4 == 0)};
}

const char* ssim_psnr_launch(const PlaneSrc& pred, const PlaneSrc& target, int N, int H, int W, double* out,
                             void* workspace, cudaStream_t stream) {
    if (N <= 0) return "ssim: empty batch (N < 1)";
    if (H < 7 || W < 7) return "ssim: win_size 7 exceeds image extent: H and W must be >= 7 (skimage raises ValueError here too)";
    if (!pred.ptr || !target.ptr) return "ssim: null pred or target pointer";
    if (!out || !workspace) return "ssim: null out or workspace";
    if (pred.channels != target.channels) return "ssim: pred and target channel counts differ";
    const int C = pred.channels;
    if (C != 1 && C != 3) return "ssim: channels must be 1 or 3";
    const int pa = ssim_layout(pred), pb = ssim_layout(target);
    if (!pa) return "ssim: pred layout is neither planar (px_stride 1) nor interleaved (px_stride 3, chan_stride 1, 3 channels)";
    if (!pb) return "ssim: target layout is neither planar (px_stride 1) nor interleaved (px_stride 3, chan_stride 1, 3 channels)";
    if (static_cast<long long>(N) * C > 65535) return "ssim: too many planes: N * channels must be <= 65535";
    int gx, gy;
    ssim_grid(H, W, &gx, &gy);
    const int nblk = gx * gy;
    double* part_ssim = static_cast<double*>(workspace);
    unsigned long long* part_ssd = reinterpret_cast<unsigned long long*>(part_ssim + static_cast<size_t>(N) * C * nblk);
    const SsimOperand a = ssim_operand(pred, pa, N), b = ssim_operand(target, pb, N);
    const dim3 grid(gx, gy, N * C);
    if (pa == 1 && pb == 1) ssim_psnr_kernel<1, 1><<<grid, SS_THREADS, 0, stream>>>(a, b, C, H, W, part_ssim, part_ssd);
    if (pa == 1 && pb == 3) ssim_psnr_kernel<1, 3><<<grid, SS_THREADS, 0, stream>>>(a, b, C, H, W, part_ssim, part_ssd);
    if (pa == 3 && pb == 1) ssim_psnr_kernel<3, 1><<<grid, SS_THREADS, 0, stream>>>(a, b, C, H, W, part_ssim, part_ssd);
    if (pa == 3 && pb == 3) ssim_psnr_kernel<3, 3><<<grid, SS_THREADS, 0, stream>>>(a, b, C, H, W, part_ssim, part_ssd);
    const char* e = last_launch_error();
    if (e) return e;
    ssim_psnr_finalize_kernel<<<N, 256, 0, stream>>>(part_ssim, part_ssd, nblk, C, H, W, out);
    return last_launch_error();
}

const char* pair_sad_launch(const uint8_t* frames, int64_t frame_stride, int64_t frame_bytes, int n_frames,
                            uint64_t* sad, cudaStream_t stream) {
    if (!frames || !sad) return "pair_sad: null operand";
    if (n_frames < 2 || frame_bytes < 1 || frame_stride < frame_bytes)
        return "pair_sad: needs >= 2 frames of >= 1 byte, frame_stride >= frame_bytes";
    const int n_pairs = n_frames - 1;
    const int gy = (n_pairs + PS_GROUP - 1) / PS_GROUP;
    if (gy > 65535) return "pair_sad: at most 524280 pairs per call";
    const int vec = (reinterpret_cast<uintptr_t>(frames) % 16 == 0) && (frame_stride % 16 == 0);
    const long long units = vec ? frame_bytes / 16 : frame_bytes;
    long long gx = (units + PS_THREADS - 1) / PS_THREADS;
    const long long fill = (148 * 8 + gy - 1) / gy;  // about one wave of 8 blocks per SM over all groups
    if (gx > fill) gx = fill;
    // 32-bit per-thread sums: at most 2^20 units (16*255 each) per thread, plus < 16 tail bytes of 255
    const long long min_gx = (units + (static_cast<long long>(PS_THREADS) << 20) - 1) / (static_cast<long long>(PS_THREADS) << 20);
    if (gx < min_gx) gx = min_gx;
    if (gx < 1) gx = 1;
    if (gx > 0x7fffffffLL) return "pair_sad: frame too large";
    const cudaError_t e = cudaMemsetAsync(sad, 0, static_cast<size_t>(n_pairs) * sizeof(uint64_t), stream);
    if (e != cudaSuccess) return cudaGetErrorString(e);
    pair_sad_kernel<<<dim3(static_cast<unsigned>(gx), gy), PS_THREADS, 0, stream>>>(
        frames, frame_stride, frame_bytes, n_pairs, vec, reinterpret_cast<unsigned long long*>(sad));
    return last_launch_error();
}

const char* gather_triplets_u8_launch(const uint8_t* frames, int64_t n_frames, const int32_t* triplets,
                                      int64_t n_triplets, const int64_t* samples, int n, int H, int W, float* frame1,
                                      float* frame2, float* target, cudaStream_t stream) {
    if (!frames || !triplets || !samples || !frame1 || !frame2 || !target) return "gather: null operand";
    if (n < 1 || H < 1 || W < 1) return "gather: needs n, H, W >= 1";
    if (n_frames < 0 || n_triplets < 0) return "gather: negative frame or triplet count";
    const long long plane = static_cast<long long>(H) * W;
    const int vec = plane % 16 == 0 && ((reinterpret_cast<uintptr_t>(frames) | reinterpret_cast<uintptr_t>(frame1) |
                                         reinterpret_cast<uintptr_t>(frame2) | reinterpret_cast<uintptr_t>(target)) %
                                        16) == 0;
    const long long units = vec ? plane / 16 : plane;
    const long long rows = 3LL * n;
    long long gx = (units + GT_THREADS - 1) / GT_THREADS;
    if (gx > 148 * 16) gx = 148 * 16;
    const long long gy = rows < 65535 ? rows : 65535;
    gather_triplets_u8_kernel<<<dim3(static_cast<unsigned>(gx), static_cast<unsigned>(gy)), GT_THREADS, 0, stream>>>(
        frames, n_frames, triplets, n_triplets, reinterpret_cast<const long long*>(samples), rows, plane, vec, frame1,
        frame2, target);
    return last_launch_error();
}

const char* gather_crops_u8_launch(const uint8_t* frames, int64_t frames_bytes, const int64_t* offsets,
                                   const int32_t* sizes, int64_t n_frames, int C, const int32_t* rows, int n, int S,
                                   float* frame1, float* frame2, float* target, cudaStream_t stream) {
    if (!frames || !offsets || !sizes || !rows || !frame1 || !frame2 || !target) return "gather_crops: null operand";
    if (n < 1 || S < 4 || S % 4) return "gather_crops: needs n >= 1 and S a positive multiple of 4";
    if (C != 1 && C != 3) return "gather_crops: C must be 1 or 3";
    if (n_frames < 0 || frames_bytes < 0) return "gather_crops: negative frame count or size";
    if ((reinterpret_cast<uintptr_t>(frame1) | reinterpret_cast<uintptr_t>(frame2) |
         reinterpret_cast<uintptr_t>(target)) % 16)
        return "gather_crops: outputs must be 16-byte aligned";
    const long long units = 3LL * n * C * S * (S / 4);
    gather_crops_u8_kernel<<<grid_for(static_cast<size_t>(units), GC_THREADS), GC_THREADS, 0, stream>>>(
        frames, frames_bytes, reinterpret_cast<const long long*>(offsets), sizes, n_frames, C, rows, S, units, frame1,
        frame2, target);
    return last_launch_error();
}

}  // namespace fi
