// Epilogue of one 64-column chunk of an 8x16-pixel accumulator tile (the per-tap kernels of conv_gemm.cu):
// TMEM -> registers, bias (+ReLU), then by mode: bf16 (or hi/lo) tile -> swizzled staging -> TMA store (+ 2x2 max-pooled
// tile), the transposed-conv pixel scatter, or the fused 1x1 head + postprocess.
#pragma once
#include "conv_gemm.cuh"
#include "ptx.cuh"

namespace fi {

struct EpiTile {
    int nb, img, y0, x0;
};

// DOUBLE_BUF as in epilogue_chunk_halo below: two alternating staging tiles per warp, or a single one.
template <int BLOCK_N, int MODE, bool SPLIT, bool DOUBLE_BUF = true>
__device__ __forceinline__ void epilogue_chunk_8x16(const ConvMaps& maps, const ConvKernelParams& p, const EpiTile& tc,
                                                    uint32_t taddr, int c, int q, int lane, uint32_t my_stage,
                                                    uint32_t my_pool, int& buf, bool store_enabled) {
    uint32_t v0[32], v1[32];
    tmem_ld_32x32b_x32(taddr + c * 64, v0);
    tmem_ld_32x32b_x32(taddr + c * 64 + 32, v1);
    tmem_ld_wait();
    const int n_glob = tc.nb * BLOCK_N + c * 64;
    const float4* bias4 = reinterpret_cast<const float4*>(p.bias + n_glob);
    float f[64];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(bias4 + j);
        f[4 * j + 0] = __uint_as_float(v0[4 * j + 0]) + b.x;
        f[4 * j + 1] = __uint_as_float(v0[4 * j + 1]) + b.y;
        f[4 * j + 2] = __uint_as_float(v0[4 * j + 2]) + b.z;
        f[4 * j + 3] = __uint_as_float(v0[4 * j + 3]) + b.w;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(bias4 + 8 + j);
        f[32 + 4 * j + 0] = __uint_as_float(v1[4 * j + 0]) + b.x;
        f[32 + 4 * j + 1] = __uint_as_float(v1[4 * j + 1]) + b.y;
        f[32 + 4 * j + 2] = __uint_as_float(v1[4 * j + 2]) + b.z;
        f[32 + 4 * j + 3] = __uint_as_float(v1[4 * j + 3]) + b.w;
    }
    if (p.relu) {
#pragma unroll
        for (int j = 0; j < 64; ++j) f[j] = fmaxf(f[j], 0.0f);
    }

    if constexpr (MODE == EPI_HEAD) {
        // 1x1 head on the fp32 (un-rounded) activations; thread = pixel.
        const int y = tc.y0 + 2 * q + (lane >> 4);
        const int x = tc.x0 + (lane & 15);
        const bool inside = store_enabled && (y < p.H) && (x < p.W);
        for (int k = 0; k < p.n_classes; ++k) {
            const float4* w4 = reinterpret_cast<const float4*>(p.head_w + k * 64);
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float4 w = __ldg(w4 + j);
                a0 = fmaf(f[4 * j + 0], w.x, a0);
                a1 = fmaf(f[4 * j + 1], w.y, a1);
                a2 = fmaf(f[4 * j + 2], w.z, a2);
                a3 = fmaf(f[4 * j + 3], w.w, a3);
            }
            const float yv = (a0 + a1) + (a2 + a3) + __ldg(p.head_b + k);
            if (inside) {
                const size_t o = ((static_cast<size_t>(tc.img) * p.n_classes + k) * p.H + y) * p.W + x;
                if (p.out_f32) p.out_f32[o] = yv;
                if (p.out_u8) {
                    // postprocess_image (reference model/inference.py:54-61): (t+1)/2, clamp, *255, truncate
                    float u = __fmul_rn(__fadd_rn(yv, 1.0f), 0.5f);
                    u = fminf(fmaxf(u, 0.0f), 1.0f);
                    p.out_u8[o] = static_cast<uint8_t>(__fmul_rn(u, 255.0f));
                }
            }
        }
    } else if constexpr (!SPLIT) {
        uint32_t pk[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) pk[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
        // The staging buffer used two chunks ago must have been read by its TMA store.
        if (elect_one()) {
            if (DOUBLE_BUF) tma_store_wait_read<1>();
            else tma_store_wait_read<0>();
        }
        __syncwarp();
        const uint32_t sbuf = my_stage + (DOUBLE_BUF ? buf * 4096 : 0);
        const uint32_t row = sbuf + lane * 128;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            st_shared_v4(row + ((j ^ (lane & 7)) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2],
                         pk[4 * j + 3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (store_enabled && elect_one()) {
            if constexpr (MODE == EPI_CONVT) {
                const int a = n_glob / p.cout2;
                tma_store_5d(&maps.out[0], sbuf, n_glob - a * p.cout2, tc.x0, a, tc.y0 + 2 * q, tc.img);
            } else {
                tma_store_4d(&maps.out[0], sbuf, n_glob, tc.x0, tc.y0 + 2 * q, tc.img);
            }
        }
        if constexpr (MODE == EPI_STORE_POOL) {
            // 2x2 max over (rows 2q,2q+1) x (cols 2p,2p+1): bf16 max commutes with the rounding above.
            const uint32_t pbuf = my_pool + (DOUBLE_BUF ? buf * 1024 : 0);
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int pp = lane >> 2;
                const int j = (lane & 3) * 2 + i;
                const int r0 = 2 * pp, r1 = 2 * pp + 1, r2 = 16 + 2 * pp, r3 = 17 + 2 * pp;
                const uint4 m0 = ld_shared_v4(sbuf + r0 * 128 + ((j ^ (r0 & 7)) << 4));
                const uint4 m1 = ld_shared_v4(sbuf + r1 * 128 + ((j ^ (r1 & 7)) << 4));
                const uint4 m2 = ld_shared_v4(sbuf + r2 * 128 + ((j ^ (r2 & 7)) << 4));
                const uint4 m3 = ld_shared_v4(sbuf + r3 * 128 + ((j ^ (r3 & 7)) << 4));
                uint4 m;
                m.x = bf16x2_max(bf16x2_max(m0.x, m1.x), bf16x2_max(m2.x, m3.x));
                m.y = bf16x2_max(bf16x2_max(m0.y, m1.y), bf16x2_max(m2.y, m3.y));
                m.z = bf16x2_max(bf16x2_max(m0.z, m1.z), bf16x2_max(m2.z, m3.z));
                m.w = bf16x2_max(bf16x2_max(m0.w, m1.w), bf16x2_max(m2.w, m3.w));
                st_shared_v4(pbuf + pp * 128 + ((j ^ (pp & 7)) << 4), m.x, m.y, m.z, m.w);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (store_enabled && elect_one()) {
                tma_store_4d(&maps.pool[0], pbuf, n_glob, tc.x0 >> 1, (tc.y0 >> 1) + q, tc.img);
            }
        }
        if (elect_one()) tma_store_commit();
        buf ^= 1;
    } else {
        // precise mode: value = hi + lo, both bf16; the two staging buffers hold the hi and the lo tile
        uint32_t pk[32], pl[32];
        split_hi_lo(f, pk, pl);
        if (elect_one()) tma_store_wait_read<0>();
        __syncwarp();
        const uint32_t shi = my_stage, slo = my_stage + 4096;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t o = lane * 128 + ((j ^ (lane & 7)) << 4);
            st_shared_v4(shi + o, pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
            st_shared_v4(slo + o, pl[4 * j], pl[4 * j + 1], pl[4 * j + 2], pl[4 * j + 3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (store_enabled && elect_one()) {
            if constexpr (MODE == EPI_CONVT) {
                const int a = n_glob / p.cout2;
                tma_store_5d(&maps.out[0], shi, n_glob - a * p.cout2, tc.x0, a, tc.y0 + 2 * q, tc.img);
                tma_store_5d(&maps.out[1], slo, n_glob - a * p.cout2, tc.x0, a, tc.y0 + 2 * q, tc.img);
            } else {
                tma_store_4d(&maps.out[0], shi, n_glob, tc.x0, tc.y0 + 2 * q, tc.img);
                tma_store_4d(&maps.out[1], slo, n_glob, tc.x0, tc.y0 + 2 * q, tc.img);
            }
        }
        if constexpr (MODE == EPI_STORE_POOL) {
            const uint32_t phi = my_pool, plo = my_pool + 1024;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int pp = lane >> 2;
                const int j = (lane & 3) * 2 + i;
                const int rows[4] = {2 * pp, 2 * pp + 1, 16 + 2 * pp, 17 + 2 * pp};
                uint4 mh, ml;
                pool4_hi_lo(shi, slo, rows, j, mh, ml);
                const uint32_t o = pp * 128 + ((j ^ (pp & 7)) << 4);
                st_shared_v4(phi + o, mh.x, mh.y, mh.z, mh.w);
                st_shared_v4(plo + o, ml.x, ml.y, ml.z, ml.w);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (store_enabled && elect_one()) {
                tma_store_4d(&maps.pool[0], phi, n_glob, tc.x0 >> 1, (tc.y0 >> 1) + q, tc.img);
                tma_store_4d(&maps.pool[1], plo, n_glob, tc.x0 >> 1, (tc.y0 >> 1) + q, tc.img);
            }
        }
        if (elect_one()) tma_store_commit();
    }
}

// Epilogue of one 64-column chunk of a halo-kernel accumulator (super tile 16x16 pixels = two 16x8 column halves; warp q
// owns tile rows 4q..4q+3 of each half; TMA store boxes {64, 8, 4, 1}, pooled {64, 4, 2, 1}).
struct HaloTile {
    int img, y0, x0;
};

// DOUBLE_BUF: two staging tiles per warp alternate (wait for the store before last); otherwise one tile per warp (eight
// epilogue warps share the same 40 KB) and the previous store must have drained.
template <int COUT, int MODE, bool SPLIT, bool DOUBLE_BUF>
__device__ __forceinline__ void epilogue_chunk_halo(const ConvMaps& maps, const ConvKernelParams& p, const HaloTile& tc,
                                                    uint32_t taddr, int c, int q, int lane, uint32_t my_stage,
                                                    uint32_t my_pool, int& buf, bool store_enabled) {
    const int half = c / (COUT / 64);
    const int n_glob = (c % (COUT / 64)) * 64;
    const int xh = tc.x0 + 8 * half;  // first column of this half
    const int yq = tc.y0 + 4 * q;     // first row of this warp
    uint32_t v0[32], v1[32];
    tmem_ld_32x32b_x32(taddr + c * 64, v0);
    tmem_ld_32x32b_x32(taddr + c * 64 + 32, v1);
    tmem_ld_wait();
    const float4* bias4 = reinterpret_cast<const float4*>(p.bias + n_glob);
    float f[64];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(bias4 + j);
        f[4 * j + 0] = __uint_as_float(v0[4 * j + 0]) + b.x;
        f[4 * j + 1] = __uint_as_float(v0[4 * j + 1]) + b.y;
        f[4 * j + 2] = __uint_as_float(v0[4 * j + 2]) + b.z;
        f[4 * j + 3] = __uint_as_float(v0[4 * j + 3]) + b.w;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const float4 b = __ldg(bias4 + 8 + j);
        f[32 + 4 * j + 0] = __uint_as_float(v1[4 * j + 0]) + b.x;
        f[32 + 4 * j + 1] = __uint_as_float(v1[4 * j + 1]) + b.y;
        f[32 + 4 * j + 2] = __uint_as_float(v1[4 * j + 2]) + b.z;
        f[32 + 4 * j + 3] = __uint_as_float(v1[4 * j + 3]) + b.w;
    }
    if (p.relu) {
#pragma unroll
        for (int j = 0; j < 64; ++j) f[j] = fmaxf(f[j], 0.0f);
    }

    if constexpr (MODE == EPI_HEAD) {
        const int y = yq + (lane >> 3);
        const int x = xh + (lane & 7);
        const bool inside = store_enabled && (y < p.H) && (x < p.W);
        for (int k = 0; k < p.n_classes; ++k) {
            const float4* w4 = reinterpret_cast<const float4*>(p.head_w + k * 64);
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const float4 w = __ldg(w4 + j);
                a0 = fmaf(f[4 * j + 0], w.x, a0);
                a1 = fmaf(f[4 * j + 1], w.y, a1);
                a2 = fmaf(f[4 * j + 2], w.z, a2);
                a3 = fmaf(f[4 * j + 3], w.w, a3);
            }
            const float yv = (a0 + a1) + (a2 + a3) + __ldg(p.head_b + k);
            if (inside) {
                const size_t o = ((static_cast<size_t>(tc.img) * p.n_classes + k) * p.H + y) * p.W + x;
                if (p.out_f32) p.out_f32[o] = yv;
                if (p.out_u8) {
                    float u = __fmul_rn(__fadd_rn(yv, 1.0f), 0.5f);
                    u = fminf(fmaxf(u, 0.0f), 1.0f);
                    p.out_u8[o] = static_cast<uint8_t>(__fmul_rn(u, 255.0f));
                }
            }
        }
    } else if constexpr (!SPLIT) {
        uint32_t pk[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) pk[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
        if (elect_one()) {
            if (DOUBLE_BUF) tma_store_wait_read<1>();
            else tma_store_wait_read<0>();
        }
        __syncwarp();
        const uint32_t sbuf = my_stage + (DOUBLE_BUF ? buf * 4096 : 0);
        const uint32_t row = sbuf + lane * 128;  // lane = (row in 0..3) * 8 + column
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            st_shared_v4(row + ((j ^ (lane & 7)) << 4), pk[4 * j], pk[4 * j + 1], pk[4 * j + 2],
                         pk[4 * j + 3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (store_enabled && elect_one()) tma_store_4d(&maps.out[0], sbuf, n_glob, xh, yq, tc.img);  // box {64, 8, 4, 1}
        if constexpr (MODE == EPI_STORE_POOL) {
            // pooled 2 rows x 4 columns: max over lanes {2ph*8 + 2pw, +1, +8, +9}
            const uint32_t pbuf = my_pool + (DOUBLE_BUF ? buf * 1024 : 0);
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int pp = lane >> 2;  // pooled pixel 0..7 = ph*4 + pw
                const int j = (lane & 3) * 2 + i;
                const int r0 = (pp >> 2) * 16 + (pp & 3) * 2;
                const int r1 = r0 + 1, r2 = r0 + 8, r3 = r0 + 9;
                const uint4 m0 = ld_shared_v4(sbuf + r0 * 128 + ((j ^ (r0 & 7)) << 4));
                const uint4 m1 = ld_shared_v4(sbuf + r1 * 128 + ((j ^ (r1 & 7)) << 4));
                const uint4 m2 = ld_shared_v4(sbuf + r2 * 128 + ((j ^ (r2 & 7)) << 4));
                const uint4 m3 = ld_shared_v4(sbuf + r3 * 128 + ((j ^ (r3 & 7)) << 4));
                uint4 m;
                m.x = bf16x2_max(bf16x2_max(m0.x, m1.x), bf16x2_max(m2.x, m3.x));
                m.y = bf16x2_max(bf16x2_max(m0.y, m1.y), bf16x2_max(m2.y, m3.y));
                m.z = bf16x2_max(bf16x2_max(m0.z, m1.z), bf16x2_max(m2.z, m3.z));
                m.w = bf16x2_max(bf16x2_max(m0.w, m1.w), bf16x2_max(m2.w, m3.w));
                st_shared_v4(pbuf + pp * 128 + ((j ^ (pp & 7)) << 4), m.x, m.y, m.z, m.w);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (store_enabled && elect_one()) {
                tma_store_4d(&maps.pool[0], pbuf, n_glob, xh >> 1, yq >> 1, tc.img);  // box {64, 4, 2, 1}
            }
        }
        if (elect_one()) tma_store_commit();
        buf ^= 1;
    } else {
        // precise mode: hi tile in staging buffer 0, lo tile in buffer 1
        uint32_t pk[32], pl[32];
        split_hi_lo(f, pk, pl);
        if (elect_one()) tma_store_wait_read<0>();
        __syncwarp();
        const uint32_t shi = my_stage, slo = my_stage + 4096;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint32_t o = lane * 128 + ((j ^ (lane & 7)) << 4);
            st_shared_v4(shi + o, pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
            st_shared_v4(slo + o, pl[4 * j], pl[4 * j + 1], pl[4 * j + 2], pl[4 * j + 3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (store_enabled && elect_one()) {
            tma_store_4d(&maps.out[0], shi, n_glob, xh, yq, tc.img);
            tma_store_4d(&maps.out[1], slo, n_glob, xh, yq, tc.img);
        }
        if constexpr (MODE == EPI_STORE_POOL) {
            const uint32_t phi = my_pool, plo = my_pool + 1024;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int pp = lane >> 2;
                const int j = (lane & 3) * 2 + i;
                const int r0 = (pp >> 2) * 16 + (pp & 3) * 2;
                const int rows[4] = {r0, r0 + 1, r0 + 8, r0 + 9};
                uint4 mh, ml;
                pool4_hi_lo(shi, slo, rows, j, mh, ml);
                const uint32_t o = pp * 128 + ((j ^ (pp & 7)) << 4);
                st_shared_v4(phi + o, mh.x, mh.y, mh.z, mh.w);
                st_shared_v4(plo + o, ml.x, ml.y, ml.z, ml.w);
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (store_enabled && elect_one()) {
                tma_store_4d(&maps.pool[0], phi, n_glob, xh >> 1, yq >> 1, tc.img);
                tma_store_4d(&maps.pool[1], plo, n_glob, xh >> 1, yq >> 1, tc.img);
            }
        }
        if (elect_one()) tma_store_commit();
    }
}

}  // namespace fi
