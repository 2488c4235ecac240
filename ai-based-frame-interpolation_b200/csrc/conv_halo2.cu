// CTA-pair (cta_group::2) variant of the halo-reuse conv3x3 (conv_halo.cu) for the narrow layers (Cout = 64 / 128).
//
// The narrow layers are bound by shared-memory bandwidth: a single-CTA tcgen05.mma of N = 64 reads 4 KB of A and 2 KB
// of B per 32 tensor-pipe cycles (measured 50.8 cycles per instruction, tools/probe/mma_probe.cu), N = 128 reads 8 KB
// per 64 cycles while TMA fills compete for the same port. In a CTA pair each SM keeps its own super tile's halo (A)
// but only HALF of every weight slab (Cout/2 rows); the M256 x Cout instruction reads both halves. That halves the
// weight traffic per SM (fills and operand reads), and it lets the weights of two more layers stay resident
// (up4.conv.0: 144 KB -> 72 KB per SM; down1.conv.0: 144 KB -> 72 KB).
//
// Protocol: as conv_gemm2.cu. Both CTAs run the same code on adjacent super tiles (rank picks the tile); producers
// wait on local "empty" barriers and send completion bytes to the leader's "full" barriers; the leader issues every
// MMA and commits with a multicast to both CTAs; epilogue warps of both CTAs release the accumulator on the leader.
#include "conv_epilogue.cuh"
#include "conv_gemm.cuh"
#include "ptx.cuh"

#include <cstdio>

namespace fi {

namespace {

constexpr int H2_T = 16;
constexpr int H2_W = 24, H2_H = 18;
constexpr int H2_HALO_BYTES = H2_W * H2_H * 128;  // 55296
constexpr int H2_THREADS = 224;
constexpr int H2_THREADS_8 = 352;
constexpr int H2_A_STAGES = 2;
constexpr int H2_PREFETCH_DIST = 2;               // as conv_halo.cu: L2 prefetch this many cluster strides ahead
constexpr int H2_B_BYTES = 73728;                 // weight region: a ring, or up to 72 KB of resident half slabs
constexpr int H2_STAGING = 4 * (2 * 4096 + 2 * 1024);
constexpr int H2_SMEM = 1024 + H2_A_STAGES * H2_HALO_BYTES + H2_B_BYTES + H2_STAGING + 512;
static_assert(H2_SMEM <= 232448, "pair halo kernel exceeds shared memory");

__device__ __forceinline__ uint64_t halo2_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>(1) << 16;
    d |= static_cast<uint64_t>((H2_W * 128) >> 4) << 32;  // 3072 B between consecutive tile rows
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

struct PairHTile {
    HaloTile t;
    bool valid;
};
__device__ __forceinline__ PairHTile decode_pair_htile(int qi, uint32_t rank, const ConvKernelParams& p) {
    const int per_img = p.tiles_y * p.tiles_x;
    const int tiles = p.n_img * per_img;
    int m = 2 * qi + static_cast<int>(rank);
    PairHTile r;
    r.valid = m < tiles;
    if (!r.valid) m = tiles - 1;
    r.t.img = m / per_img;
    m -= r.t.img * per_img;
    const int ty = m / p.tiles_x;
    r.t.y0 = ty * H2_T;
    r.t.x0 = (m - ty * p.tiles_x) * H2_T;
    return r;
}

template <int COUT, int MODE, bool RESIDENT, bool SPLIT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(SPLIT ? H2_THREADS : H2_THREADS_8, 1)
conv_halo2_kernel(const __grid_constant__ ConvMaps maps, const ConvKernelParams p) {
    constexpr int B_HALF_BYTES = (COUT / 2) * 128;        // this CTA's half of one [Cout x 64] weight slab
    constexpr int B_STAGES = 65536 / B_HALF_BYTES;        // ring depth when streaming (16 or 8)
    constexpr int ACC_COLS = 2 * COUT;
    constexpr int TMEM_COLS = 2 * ACC_COLS;
    constexpr uint32_t IDESC = umma_idesc_bf16(256, COUT);
    static_assert(MODE != EPI_HEAD || COUT == 64, "head epilogue consumes exactly 64 channels");
    // bf16 mode: 8 epilogue warps, one set of 4 per column half, single staging tile each; precise mode: 4 warps
    constexpr int EPI_SETS = SPLIT ? 1 : 2;
    constexpr int STAGE_PER_WARP = SPLIT ? 2 * 4096 : 4096;
    constexpr int POOL_PER_WARP = SPLIT ? 2 * 1024 : 1024;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t smem_a = smem_base;
    const uint32_t smem_b = smem_a + H2_A_STAGES * H2_HALO_BYTES;
    const uint32_t smem_stage = smem_b + H2_B_BYTES;
    const uint32_t smem_pool = smem_stage + 4 * 2 * 4096;
    const uint32_t smem_bar = smem_pool + 4 * 2 * 1024;
    const uint32_t bar_afull = smem_bar;
    const uint32_t bar_aempty = bar_afull + 8 * H2_A_STAGES;
    const uint32_t bar_bfull = bar_aempty + 8 * H2_A_STAGES;
    const uint32_t bar_bempty = bar_bfull + 8 * B_STAGES;
    const uint32_t bar_tfull = bar_bempty + 8 * B_STAGES;
    const uint32_t bar_tempty = bar_tfull + 16;
    const uint32_t bar_bres = bar_tempty + 16;
    const uint32_t tmem_slot = bar_bres + 8;
    uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;
    const int cluster_id = blockIdx.x >> 1;
    const int n_clusters = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a[0]);
        tma_prefetch_desc(&maps.a[2]);
        tma_prefetch_desc(&maps.b);
        if (MODE != EPI_HEAD) tma_prefetch_desc(&maps.out[0]);
        if (MODE == EPI_STORE_POOL) tma_prefetch_desc(&maps.pool[0]);
        for (int s = 0; s < H2_A_STAGES; ++s) {
            mbar_init(bar_afull + 8 * s, 1);
            mbar_init(bar_aempty + 8 * s, 1);
        }
        for (int s = 0; s < B_STAGES; ++s) {
            mbar_init(bar_bfull + 8 * s, 1);
            mbar_init(bar_bempty + 8 * s, 1);
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(bar_tfull + 8 * a, 1);
            mbar_init(bar_tempty + 8 * a, 8 * EPI_SETS);
        }
        mbar_init(bar_bres, 1);
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc_2sm(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_launch_dependents();
    pdl_wait();

    const int tiles = p.n_img * p.tiles_y * p.tiles_x;
    const int total = (tiles + 1) >> 1;
    const int slabs = p.slabs;
    const int b_row0 = static_cast<int>(rank) * (COUT / 2);  // this CTA's rows of every weight slab

    if (warp == 0) {
        // ------------------------------------------------------------ A producer (both CTAs): own halo boxes
        int stage = 0;
        uint32_t phase = 0;
        for (int qi = cluster_id; qi < total; qi += n_clusters) {
            const PairHTile pt = decode_pair_htile(qi, rank, p);
            const int qp = qi + H2_PREFETCH_DIST * n_clusters;
            if (qp < total && lane == 0) {
                const PairHTile pc = decode_pair_htile(qp, rank, p);
                for (int g = 0; g < p.nseg; ++g) {
                    const int mid = p.seg_map[g];
                    if (g > 0 && p.seg_map[g - 1] == mid) continue;
                    const int ox = mid >= 2 ? p.off_x : 0, oy = mid >= 2 ? p.off_y : 0;
                    for (int c = 0; c < p.seg_slabs[g]; ++c)
                        tma_prefetch_l2_4d(&maps.a[mid], c * BLOCK_K, pc.t.x0 - 1 - ox, pc.t.y0 - 1 - oy, pc.t.img);
                }
            }
            int seg = 0, left = p.seg_slabs[0];
            for (int s = 0; s < slabs; ++s) {
                while (left == 0) left = p.seg_slabs[++seg];
                const int local = p.seg_slabs[seg] - left;
                --left;
                const int mid = p.seg_map[seg];
                mbar_wait(bar_aempty + 8 * stage, phase ^ 1);
                const uint32_t full = bar_afull + 8 * stage;
                if (elect_one()) {
                    if (leader) mbar_expect_tx(full, 2 * H2_HALO_BYTES);
                    const int ox = mid >= 2 ? p.off_x : 0, oy = mid >= 2 ? p.off_y : 0;
                    tma_load_4d_2sm(smem_a + stage * H2_HALO_BYTES, &maps.a[mid], full, local * BLOCK_K,
                                    pt.t.x0 - 1 - ox, pt.t.y0 - 1 - oy, pt.t.img);
                }
                __syncwarp();
                if (++stage == H2_A_STAGES) {
                    stage = 0;
                    phase ^= 1;
                }
            }
        }
    } else if (warp == 2) {
        // ------------------------------------------------------------ B producer (both CTAs): own half slabs
        if (RESIDENT) {
            if (lane == 0) {
                if (leader) mbar_expect_tx(bar_bres, 2 * 9 * slabs * B_HALF_BYTES);
                for (int s = 0; s < slabs; ++s)
                    for (int tap = 0; tap < 9; ++tap)
                        tma_load_2d_2sm(smem_b + (s * 9 + tap) * B_HALF_BYTES, &maps.b, bar_bres,
                                        (tap * slabs + s) * BLOCK_K, b_row0);
            }
        } else {
            int stage = 0;
            uint32_t phase = 0;
            for (int qi = cluster_id; qi < total; qi += n_clusters) {
                for (int s = 0; s < slabs; ++s) {
                    for (int tap = 0; tap < 9; ++tap) {
                        mbar_wait(bar_bempty + 8 * stage, phase ^ 1);
                        const uint32_t full = bar_bfull + 8 * stage;
                        if (elect_one()) {
                            if (leader) mbar_expect_tx(full, 2 * B_HALF_BYTES);
                            tma_load_2d_2sm(smem_b + stage * B_HALF_BYTES, &maps.b, full, (tap * slabs + s) * BLOCK_K,
                                            b_row0);
                        }
                        __syncwarp();
                        if (++stage == B_STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (leader CTA only)
        if (leader) {
            int a_stage = 0, b_stage = 0;
            uint32_t a_phase = 0, b_phase = 0;
            int it = 0;
            if (RESIDENT) mbar_wait(bar_bres, 0);
            for (int qi = cluster_id; qi < total; qi += n_clusters, ++it) {
                const int acc = it & 1;
                mbar_wait(bar_tempty + 8 * acc, ((it >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * ACC_COLS;
                for (int s = 0; s < slabs; ++s) {
                    mbar_wait(bar_afull + 8 * a_stage, a_phase);
                    const uint32_t a_base = smem_a + a_stage * H2_HALO_BYTES;
                    for (int tap = 0; tap < 9; ++tap) {
                        if (!RESIDENT) mbar_wait(bar_bfull + 8 * b_stage, b_phase);
                        tc_fence_after();
                        const int dy = tap / 3, dx = tap - 3 * dy;
                        const uint64_t db =
                            umma_desc_sw128(smem_b + (RESIDENT ? s * 9 + tap : b_stage) * B_HALF_BYTES);
                        const uint64_t da0 = halo2_desc(a_base + (dy * H2_W + dx) * 128);
                        if (elect_one()) {
#pragma unroll
                            for (int k = 0; k < BLOCK_K / 16; ++k) {
#pragma unroll
                                for (int half = 0; half < 2; ++half) {
                                    umma_bf16_ss_2sm(d_tmem + half * COUT, da0 + 64 * half + 2 * k, db + 2 * k, IDESC,
                                                     (s | tap | k) != 0);
                                }
                            }
                            if (!RESIDENT) umma_commit_2sm(bar_bempty + 8 * b_stage);
                            if (tap == 8) {
                                umma_commit_2sm(bar_aempty + 8 * a_stage);
                                if (s == slabs - 1) umma_commit_2sm(bar_tfull + 8 * acc);
                            }
                        }
                        __syncwarp();
                        if (!RESIDENT) {
                            if (++b_stage == B_STAGES) {
                                b_stage = 0;
                                b_phase ^= 1;
                            }
                        }
                    }
                    if (++a_stage == H2_A_STAGES) {
                        a_stage = 0;
                        a_phase ^= 1;
                    }
                }
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue warps 3..6 (both CTAs)
        const int q = warp & 3;
        const int ew = warp - 3;
        const int set = ew >> 2;
        const uint32_t my_stage = smem_stage + ew * STAGE_PER_WARP;
        const uint32_t my_pool = smem_pool + ew * POOL_PER_WARP;
        int buf = 0;
        int it = 0;
        for (int qi = cluster_id; qi < total; qi += n_clusters, ++it) {
            const PairHTile pt = decode_pair_htile(qi, rank, p);
            const int acc = it & 1;
            mbar_wait(bar_tfull + 8 * acc, (it >> 1) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * ACC_COLS;
#pragma unroll 1
            for (int c = set * (ACC_COLS / 64 / EPI_SETS); c < (set + 1) * (ACC_COLS / 64 / EPI_SETS); ++c) {
                epilogue_chunk_halo<COUT, MODE, SPLIT, SPLIT>(maps, p, pt.t, taddr, c, q, lane, my_stage, my_pool, buf,
                                                       pt.valid);
            }
            tc_fence_before();
            __syncwarp();
            if (elect_one()) {
                if (leader) mbar_arrive(bar_tempty + 8 * acc);
                else mbar_arrive_cluster(bar_tempty + 8 * acc, 0);
            }
        }
        __syncwarp();
        if (MODE != EPI_HEAD && elect_one()) tma_store_wait_all();
    }

    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    }
}

template <int COUT, int MODE, bool RESIDENT = false, bool SPLIT = false>
const char* launch_halo2_inst(const ConvLaunch& l, cudaStream_t stream) {
    if constexpr (!RESIDENT) {
        // all half slabs of the layer fit next to the two halo stages: keep them for the CTA's lifetime
        if (9 * l.p.slabs * (COUT / 2) * 128 <= H2_B_BYTES) return launch_halo2_inst<COUT, MODE, true, SPLIT>(l, stream);
    }
    auto kfn = conv_halo2_kernel<COUT, MODE, RESIDENT, SPLIT>;
    static std::atomic<uint64_t> configured{0};
    if (!smem_opt_in(kfn, H2_SMEM, configured)) return "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed";
    const cudaError_t e = launch_kernel(kfn, dim3(l.grid), dim3(SPLIT ? H2_THREADS : H2_THREADS_8), H2_SMEM, stream,
                                        l.maps, l.p);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

template <int COUT, int MODE>
const char* launch_halo2_split(const ConvLaunch& l, cudaStream_t stream) {
    if constexpr (MODE != EPI_HEAD) {
        if (l.split) return launch_halo2_inst<COUT, MODE, false, true>(l, stream);
    }
    return launch_halo2_inst<COUT, MODE, false, false>(l, stream);
}

}  // namespace

const char* conv_halo_pair_launch(const ConvLaunch& l, cudaStream_t stream) {
    switch (l.block_n * 4 + l.mode) {
        case 64 * 4 + EPI_STORE: return launch_halo2_split<64, EPI_STORE>(l, stream);
        case 64 * 4 + EPI_STORE_POOL: return launch_halo2_split<64, EPI_STORE_POOL>(l, stream);
        case 64 * 4 + EPI_HEAD: return launch_halo2_split<64, EPI_HEAD>(l, stream);
        case 128 * 4 + EPI_STORE: return launch_halo2_split<128, EPI_STORE>(l, stream);
        case 128 * 4 + EPI_STORE_POOL: return launch_halo2_split<128, EPI_STORE_POOL>(l, stream);
        default: return "conv(halo pair): no kernel instantiation for this (cout, mode)";
    }
}

}  // namespace fi
