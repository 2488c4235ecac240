// tcgen05 / TMEM / TMA implicit-GEMM convolution for the UNet frame-synthesis path.
//
// Replaces, per launch, what the reference runs as separate eager ops (reference model/unet.py):
//   conv3x3(pad 1, no bias) -> BatchNorm2d(eval) -> ReLU          unet.py:12-17  (BN folded into W / bias on the host)
//   MaxPool2d(2)                                                   unet.py:28     (EPI_STORE_POOL: dual store)
//   F.pad + torch.cat([skip, up], 1)                               unet.py:49-54  (second K-range source + OOB zero fill)
//   ConvTranspose2d(k=2, s=2) + bias                               unet.py:43     (EPI_CONVT: 1-tap GEMM, pixel-scatter store)
//   Conv2d(64, n_classes, 1) + bias and postprocess_image          unet.py:60, inference.py:54-61 (EPI_HEAD)
//
// GEMM view: M = pixels (one CTA tile = 8x16 pixels of one image), N = output channels, K = taps x input channels.
// A operand: for every (tap, 64-channel slab) one TMA box {64ch,16,8,1} of the NHWC activation, start coordinate
//            shifted by the tap; out-of-bounds elements are zero-filled by TMA = the conv zero padding (and F.pad).
// B operand: BN-folded weights, bf16 [N][K] K-major, one TMA box {64, BLOCK_N} per K slab.
// Both land in 128B-swizzled K-major smem tiles that tcgen05.mma reads through shared-memory descriptors.
// Accumulators: fp32 in TMEM, double buffered (2 x BLOCK_N columns) so the epilogue of tile i overlaps tile i+1.
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2..5 = epilogue
// (320 threads and warps 2..9 where two epilogue sets split the 64-column chunks of a tile).
//
// CTA pairs (conv_gemm2_kernel, cta_group::2) for the wide layers (Cout multiple of 256). Measured with
// tools/probe/mma_probe.cu, a tcgen05.mma costs max(N/2, operand bytes per SM / ~120) cycles, and the TMA fills compete
// for the same ~128 B/cycle of shared-memory bandwidth. A single CTA doing M128 x N256 reads 12 KB of operands and
// receives 12 KB of new tiles per MMA-time: 192 B/cycle of demand. In a CTA pair each SM keeps its own 128 pixel rows
// of A but only HALF of the weight slab (128 of the 256 rows); the pair's MMA is M256 x N256, the hardware reads both
// halves, and each SM's traffic drops to 8 KB + 8 KB per 128 cycles = 128 B/cycle.
// Protocol (cluster of 2, same code in both CTAs, rank 0 = leader, adjacent pixel tiles):
//   producers (warp 0 of both)   wait on their LOCAL empty barrier, load their own A tile and their half of B with
//                                cp.async.bulk.tensor...cta_group::2, completion bytes go to the LEADER's full barrier
//   MMA issuer (warp 1, leader)  waits on its full barrier (2 x 32 KB), issues tcgen05.mma.cta_group::2, and commits
//                                with a multicast to the empty / accumulator-full barriers of BOTH CTAs
//   epilogue (warps 2..5, both)  read their own TMEM lanes; release the accumulator by arriving (locally or through
//                                mapa) on the leader's accumulator-empty barrier (8 arrivals per phase)
#include "conv_epilogue.cuh"
#include "conv_gemm.cuh"
#include "ptx.cuh"

#include <cstdio>
#include <cstdlib>
#include <cstring>

namespace fi {

namespace {

constexpr int NUM_THREADS = 192;    // 2 role warps + 4 epilogue warps (precise mode, head, CTA pairs)
constexpr int NUM_THREADS_8 = 320;  // 2 role warps + 8 epilogue warps: two sets split the 64-column chunks of a tile
constexpr int A_STAGE_BYTES = BLOCK_M * 128;             // 16 KB
constexpr int STAGING_BYTES_PER_WARP = 2 * 4096;         // 2 x (32 rows x 128 B)
constexpr int POOL_BYTES_PER_WARP = 2 * 1024;            // 2 x (8 rows x 128 B)
constexpr int EPI_BYTES = 4 * (STAGING_BYTES_PER_WARP + POOL_BYTES_PER_WARP);
constexpr int BAR_BYTES = 256;
constexpr int SMEM_LIMIT = 232448;                       // 227 KB usable per CTA on sm_100

// Ring depth and shared memory follow from the B slab one CTA holds: BLOCK_N rows, or half of them in a CTA pair.
__host__ __device__ constexpr int b_stage_bytes(int block_n) { return block_n * 128; }
__host__ __device__ constexpr int num_stages(int block_n) {
    int s = (SMEM_LIMIT - 1024 - BAR_BYTES - EPI_BYTES) / (A_STAGE_BYTES + b_stage_bytes(block_n));
    return s > 8 ? 8 : s;
}
__host__ __device__ constexpr int smem_bytes(int block_n) {
    return 1024 + num_stages(block_n) * (A_STAGE_BYTES + b_stage_bytes(block_n)) + EPI_BYTES + BAR_BYTES;
}
__host__ __device__ constexpr int tmem_cols(int block_n) { return 2 * block_n < 32 ? 32 : 2 * block_n; }

struct Unit {
    EpiTile t;
    bool valid;  // false: odd tile count, the last pair's second CTA recomputes the last tile with its stores off
};
// Work unit u -> this CTA's tile. Units that share a weight block are adjacent in time across the grid so the B slabs
// stay hot in L2; the two CTAs of a pair take adjacent pixel tiles of the same weight block.
template <int CTAS>
__device__ __forceinline__ Unit decode_unit(int u, uint32_t rank, const ConvKernelParams& p) {
    const int per_img = p.tiles_y * p.tiles_x;
    const int m_tiles = p.n_img * per_img;
    const int per_nb = (m_tiles + CTAS - 1) / CTAS;
    Unit r;
    r.t.nb = u / per_nb;
    int m = CTAS * (u - r.t.nb * per_nb) + static_cast<int>(rank);
    r.valid = CTAS == 1 || m < m_tiles;
    if (!r.valid) m = m_tiles - 1;
    r.t.img = m / per_img;
    m -= r.t.img * per_img;
    const int ty = m / p.tiles_x;
    r.t.y0 = ty * TILE_H;
    r.t.x0 = (m - ty * p.tiles_x) * TILE_W;
    return r;
}

__host__ __device__ constexpr bool eight_epilogue_warps(int ctas, int block_n, int mode, bool split) {
    // needs >= 2 chunks per tile and single staging tiles; a pair's leader counts the arrivals of 4 warps per CTA
    return ctas == 1 && !split && mode != EPI_HEAD && block_n >= 128;
}
__host__ __device__ constexpr int num_threads(int ctas, int block_n, int mode, bool split) {
    return eight_epilogue_warps(ctas, block_n, mode, split) ? NUM_THREADS_8 : NUM_THREADS;
}

// CTAS = 1: one CTA per tile. CTAS = 2: a CTA pair (cluster of 2) computes two adjacent tiles as one M256 GEMM.
template <int CTAS, int BLOCK_N, int MODE, bool SPLIT>
__device__ __forceinline__ void conv_gemm_body(const ConvMaps& maps, const ConvKernelParams& p) {
    constexpr int STAGES = num_stages(BLOCK_N / CTAS);
    constexpr int B_STAGE_BYTES = b_stage_bytes(BLOCK_N / CTAS);  // this CTA's rows of the weight slab
    constexpr uint32_t STAGE_TX = A_STAGE_BYTES + B_STAGE_BYTES;
    constexpr int TMEM_COLS = tmem_cols(BLOCK_N);
    constexpr uint32_t IDESC = umma_idesc_bf16(BLOCK_M * CTAS, BLOCK_N);
    static_assert(MODE != EPI_HEAD || BLOCK_N == 64, "head epilogue consumes exactly 64 channels");
    constexpr bool EIGHT = eight_epilogue_warps(CTAS, BLOCK_N, MODE, SPLIT);
    constexpr int EPI_SETS = EIGHT ? 2 : 1;

    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t smem_a = smem_base;
    const uint32_t smem_b = smem_a + STAGES * A_STAGE_BYTES;
    const uint32_t smem_stage = smem_b + STAGES * B_STAGE_BYTES;
    const uint32_t smem_pool = smem_stage + 4 * STAGING_BYTES_PER_WARP;
    const uint32_t smem_bar = smem_pool + 4 * POOL_BYTES_PER_WARP;
    const uint32_t bar_full = smem_bar;                     // STAGES x 8 B
    const uint32_t bar_empty = smem_bar + 8 * STAGES;       // STAGES x 8 B
    const uint32_t bar_tfull = smem_bar + 16 * STAGES;      // 2 x 8 B
    const uint32_t bar_tempty = bar_tfull + 16;             // 2 x 8 B
    const uint32_t tmem_slot = bar_tempty + 16;             // 4 B
    uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = CTAS == 1 ? 0 : cluster_ctarank();
    const bool leader = CTAS == 1 || rank == 0;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&maps.a[0]);
        tma_prefetch_desc(&maps.a[2]);
        tma_prefetch_desc(&maps.b);
        if (MODE != EPI_HEAD) tma_prefetch_desc(&maps.out[0]);
        if (MODE == EPI_STORE_POOL) tma_prefetch_desc(&maps.pool[0]);
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(bar_full + 8 * s, 1);   // pair: the leader's own arrive.expect_tx; bytes arrive from both CTAs
            mbar_init(bar_empty + 8 * s, 1);  // one (multicast) commit per use
        }
        for (int a = 0; a < 2; ++a) {
            mbar_init(bar_tfull + 8 * a, 1);
            mbar_init(bar_tempty + 8 * a, 4 * EPI_SETS * CTAS);  // one arrive per epilogue warp (of both CTAs)
        }
        fence_mbar_init();
    }
    if (warp == 1) tmem_alloc<CTAS>(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    if constexpr (CTAS == 2) cluster_sync_all();  // both CTAs' barriers exist before any remote signal can arrive
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    pdl_launch_dependents();  // the next layer may run its prologue on SMs this grid vacates
    pdl_wait();               // the previous layer's output is complete and visible from here on

    const int units = p.n_blocks * ((p.n_img * p.tiles_y * p.tiles_x + CTAS - 1) / CTAS);
    const int unit0 = static_cast<int>(blockIdx.x / CTAS);
    const int unit_step = static_cast<int>(gridDim.x / CTAS);
    const int slabs = p.slabs;
    const int k_iters = p.taps * slabs;

    if (warp == 0) {
        // ------------------------------------------------------------ TMA producer (warp converged, one lane issues)
        {
            int stage = 0;
            uint32_t phase = 0;
            for (int u = unit0; u < units; u += unit_step) {
                const EpiTile tc = decode_unit<CTAS>(u, rank, p).t;
                for (int tap = 0; tap < p.taps; ++tap) {
                    const int dy = (p.taps == 9) ? tap / 3 - 1 : 0;
                    const int dx = (p.taps == 9) ? tap % 3 - 1 : 0;
                    int seg = 0, left = p.seg_slabs[0];
                    for (int s = 0; s < slabs; ++s) {
                        while (left == 0) left = p.seg_slabs[++seg];  // K segment (source tensor) of this slab
                        const int local = p.seg_slabs[seg] - left;
                        --left;
                        const int mid = p.seg_map[seg];
                        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                        const uint32_t full = bar_full + 8 * stage;
                        if (elect_one()) {
                            if (leader) mbar_expect_tx(full, CTAS * STAGE_TX);
                            const int ox = mid >= 2 ? p.off_x : 0, oy = mid >= 2 ? p.off_y : 0;  // F.pad of src1
                            tma_load_4d<CTAS>(smem_a + stage * A_STAGE_BYTES, &maps.a[mid], full, local * BLOCK_K,
                                              tc.x0 + dx - ox, tc.y0 + dy - oy, tc.img);
                            tma_load_2d<CTAS>(smem_b + stage * B_STAGE_BYTES, &maps.b, full,
                                              (tap * slabs + s) * BLOCK_K,
                                              tc.nb * BLOCK_N + static_cast<int>(rank) * (BLOCK_N / CTAS));
                        }
                        __syncwarp();
                        if (++stage == STAGES) {
                            stage = 0;
                            phase ^= 1;
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------ MMA issuer (warp converged, one lane issues;
        // a pair's MMAs are all issued by the leader CTA)
        if (leader) {
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            for (int u = unit0; u < units; u += unit_step, ++it) {
                const int acc = it & 1;
                const uint32_t acc_phase = (it >> 1) & 1;
                mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BLOCK_N;
                for (int kb = 0; kb < k_iters; ++kb) {
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    const uint64_t da = umma_desc_sw128(smem_a + stage * A_STAGE_BYTES);
                    const uint64_t db = umma_desc_sw128(smem_b + stage * B_STAGE_BYTES);
                    if (elect_one()) {
#pragma unroll
                        for (int k = 0; k < BLOCK_K / 16; ++k) {
                            // +32 bytes along K inside the 128B swizzle row = +2 in the (addr >> 4) field
                            umma_bf16_ss<CTAS>(d_tmem, da + 2 * k, db + 2 * k, IDESC, (kb | k) != 0);
                        }
                        umma_commit<CTAS>(bar_empty + 8 * stage);  // frees the smem slot once these MMAs retire
                        if (kb == k_iters - 1) umma_commit<CTAS>(bar_tfull + 8 * acc);  // accumulator complete
                    }
                    __syncwarp();
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else {
        // ------------------------------------------------------------ epilogue warps 2..5
        const int q = warp & 3;  // TMEM lanes [32q, 32q+32) <-> tile rows 2q, 2q+1
        const int ew = warp - 2;   // 0..3, or 0..7 with two epilogue sets
        const int set = EIGHT ? ew >> 2 : 0;
        const uint32_t my_stage = smem_stage + ew * (EIGHT ? 4096 : STAGING_BYTES_PER_WARP);
        const uint32_t my_pool = smem_pool + ew * (EIGHT ? 1024 : POOL_BYTES_PER_WARP);
        int buf = 0;
        int it = 0;
        for (int u = unit0; u < units; u += unit_step, ++it) {
            const Unit w = decode_unit<CTAS>(u, rank, p);
            const int acc = it & 1;
            const uint32_t acc_phase = (it >> 1) & 1;
            mbar_wait(bar_tfull + 8 * acc, acc_phase);
            tc_fence_after();
            const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + acc * BLOCK_N;
#pragma unroll 1
            for (int c = set; c < BLOCK_N / 64; c += EPI_SETS) {
                epilogue_chunk_8x16<BLOCK_N, MODE, SPLIT, !EIGHT>(maps, p, w.t, taddr, c, q, lane, my_stage, my_pool,
                                                                   buf, w.valid);
            }
            // All TMEM reads of this accumulator are complete (tmem_ld_wait above): hand it back to the MMA warp.
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
    if constexpr (CTAS == 2) cluster_sync_all();  // the peer may still be reading TMEM / receiving commits
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc<CTAS>(tmem_base, TMEM_COLS);
    }
}

template <int BLOCK_N, int MODE, bool SPLIT>
__global__ void __launch_bounds__(num_threads(1, BLOCK_N, MODE, SPLIT), 1)
conv_gemm_kernel(const __grid_constant__ ConvMaps maps, const ConvKernelParams p) {
    conv_gemm_body<1, BLOCK_N, MODE, SPLIT>(maps, p);
}

template <int MODE, bool SPLIT>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(num_threads(2, 256, MODE, SPLIT), 1)
conv_gemm2_kernel(const __grid_constant__ ConvMaps maps, const ConvKernelParams p) {
    conv_gemm_body<2, 256, MODE, SPLIT>(maps, p);
}

// ------------------------------------------------------------------------------------------------ host side

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess) {
            fn = reinterpret_cast<EncodeTiledFn>(p);
        }
    }
    return fn;
}

// bf16 tensor map, 128B swizzle, zero OOB fill. dims/box are innermost-first; strides in elements for dims 1..rank-1.
const char* encode_bf16_map(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                            const uint64_t* strides_elems, const uint32_t* box) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) return "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)";
    cuuint64_t gdim[5], gstr[4];
    cuuint32_t bdim[5], estr[5];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bdim[i] = box[i];
        estr[i] = 1;
    }
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_elems[i] * 2;  // bytes
    if ((reinterpret_cast<uintptr_t>(base) & 15) != 0) return "tensor base address must be 16-byte aligned";
    const CUresult r =
        fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim, gstr,
           bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        static thread_local char msg[96];
        snprintf(msg, sizeof msg, "cuTensorMapEncodeTiled failed (CUresult %d)", static_cast<int>(r));
        return msg;
    }
    return nullptr;
}

const char* encode_nhwc(CUtensorMap* map, const void* base, int n, int h, int w, int c, int box_w, int box_h) {
    const uint64_t dims[4] = {static_cast<uint64_t>(c), static_cast<uint64_t>(w), static_cast<uint64_t>(h),
                              static_cast<uint64_t>(n)};
    const uint64_t strides[3] = {static_cast<uint64_t>(c), static_cast<uint64_t>(w) * c,
                                 static_cast<uint64_t>(h) * w * c};
    const uint32_t box[4] = {64, static_cast<uint32_t>(box_w), static_cast<uint32_t>(box_h), 1};
    return encode_bf16_map(map, base, 4, dims, strides, box);
}

template <int CTAS, int BLOCK_N, int MODE, bool SPLIT = false>
const char* launch_inst(const ConvLaunch& l, cudaStream_t stream) {
    if constexpr (!SPLIT && MODE != EPI_HEAD) {
        if (l.split) return launch_inst<CTAS, BLOCK_N, MODE, true>(l, stream);
    }
    static_assert(CTAS == 1 || BLOCK_N == 256, "CTA pairs run 256-column blocks");
    void (*kfn)(ConvMaps, ConvKernelParams);
    if constexpr (CTAS == 1) kfn = conv_gemm_kernel<BLOCK_N, MODE, SPLIT>;
    else kfn = conv_gemm2_kernel<MODE, SPLIT>;
    static std::atomic<uint64_t> configured{0};  // per instantiation: devices with the shared-memory opt-in
    constexpr int smem = smem_bytes(BLOCK_N / CTAS);
    if (!smem_opt_in(kfn, smem, configured)) return "cudaFuncSetAttribute(MaxDynamicSharedMemorySize) failed";
    const cudaError_t e =
        launch_kernel(kfn, dim3(l.grid), dim3(num_threads(CTAS, BLOCK_N, MODE, SPLIT)), smem, stream, l.maps, l.p);
    return e == cudaSuccess ? nullptr : cudaGetErrorString(e);
}

template <int CTAS>
const char* launch_per_tap(const ConvLaunch& l, cudaStream_t stream) {
    switch (l.block_n * 4 + l.mode) {
        case 256 * 4 + EPI_STORE: return launch_inst<CTAS, 256, EPI_STORE>(l, stream);
        case 256 * 4 + EPI_STORE_POOL: return launch_inst<CTAS, 256, EPI_STORE_POOL>(l, stream);
        case 256 * 4 + EPI_CONVT: return launch_inst<CTAS, 256, EPI_CONVT>(l, stream);
    }
    if constexpr (CTAS == 1) {
        switch (l.block_n * 4 + l.mode) {
            case 64 * 4 + EPI_STORE: return launch_inst<1, 64, EPI_STORE>(l, stream);
            case 64 * 4 + EPI_STORE_POOL: return launch_inst<1, 64, EPI_STORE_POOL>(l, stream);
            case 64 * 4 + EPI_HEAD: return launch_inst<1, 64, EPI_HEAD>(l, stream);
            case 128 * 4 + EPI_STORE: return launch_inst<1, 128, EPI_STORE>(l, stream);
            case 128 * 4 + EPI_STORE_POOL: return launch_inst<1, 128, EPI_STORE_POOL>(l, stream);
        }
    }
    return "conv: no kernel instantiation for this (block_n, mode)";
}

}  // namespace

const char* encode_bf16_map_public(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                                   const uint64_t* strides_elems, const uint32_t* box) {
    return encode_bf16_map(map, base, rank, dims, strides_elems, box);
}

const char* conv_prepare(const ConvDesc& d, int num_sms, ConvLaunch* out) {
    if (d.N <= 0 || d.H <= 0 || d.W <= 0) return "conv: empty shape";
    if (d.taps != 9 && d.taps != 1) return "conv: taps must be 9 (3x3) or 1";
    if (d.c0 <= 0 || d.c0 % BLOCK_K) return "conv: c0 must be a positive multiple of 64";
    if (d.c1 < 0 || d.c1 % BLOCK_K) return "conv: c1 must be a multiple of 64";
    if (d.c1 > 0 && !d.src1) return "conv: src1 missing";
    if (!d.src0 || !d.wpack || !d.bias) return "conv: null operand";
    if (d.n_total % 64) return "conv: n_total must be a multiple of 64";
    const bool precise = d.precise != 0;
    if (precise && (!d.src0_lo || (d.c1 > 0 && !d.src1_lo))) return "conv: precise mode needs the lo source tensors";
    int block_n = d.n_total % 256 == 0 ? 256 : (d.n_total % 128 == 0 ? 128 : 64);
    if (d.mode == EPI_HEAD) {
        if (d.n_total != 64) return "conv: head epilogue needs exactly 64 GEMM columns";
        if (d.n_classes < 1 || !d.head_w || !d.head_b || (!d.out_f32 && !d.out_u8)) return "conv: head operands";
        block_n = 64;
    } else if (d.mode == EPI_CONVT) {
        if (d.taps != 1 || d.c1 != 0) return "conv: transposed conv is a 1-tap single-source GEMM";
        if (d.n_total % 256) return "conv: transposed conv needs 4*Cout to be a multiple of 256";
        if (!d.dst) return "conv: dst missing";
        block_n = 256;
    } else if (d.mode == EPI_STORE || d.mode == EPI_STORE_POOL) {
        if (!d.dst) return "conv: dst missing";
        if (d.mode == EPI_STORE_POOL && (!d.dst_pool || d.H < 2 || d.W < 2)) return "conv: pooled dst missing";
    } else {
        return "conv: unknown epilogue mode";
    }
    if (precise && d.mode != EPI_HEAD && (!d.dst_lo || (d.mode == EPI_STORE_POOL && !d.dst_pool_lo)))
        return "conv: precise mode needs the lo destination tensors";

    ConvLaunch l;
    memset(&l, 0, sizeof l);
    const char* e;
    // geometry of the CTA tile and of the TMA boxes: generic per-tap kernel, or the halo-reuse kernel
    int tile_w = TILE_W, tile_h = TILE_H, box_w = TILE_W, box_h = TILE_H, out_w = TILE_W, out_h = 2,
        pool_w = TILE_W / 2, pool_h = 1;
    const char* no_halo = getenv("FI_NO_HALO");
    l.halo = conv_halo_eligible(d) && !(no_halo && no_halo[0] == '1');
    if (l.halo) {
        int t;
        conv_halo_geometry(&t, &box_w, &box_h, &out_w, &out_h, &pool_w, &pool_h);
        tile_w = tile_h = t;
        block_n = d.n_total;
    }
    if (!l.halo && (d.mode == EPI_STORE || d.mode == EPI_STORE_POOL)) {
        // Column-block width of the per-tap kernel. N = 256 is the efficient shape (tensor-bound M128/M256 x N256 MMAs,
        // CTA pairs halve the weight traffic: 1500-1600 TFLOP/s), narrower blocks are bound by the A-operand reads
        // (~56 % tensor-pipe activity at N = 128 under ncu). But a small frame gives a wide layer very few tiles:
        // down4.conv.3 of ONE 256x256 pair is 2 pixel tiles x 4 column blocks = 8 CTAs on 148 SMs. Only when the
        // 256-wide tiling cannot even fill one wave are narrower blocks considered, by (waves x cycles per K16 step:
        // 128 / 80 / 56); anything with a full wave of 256-wide tiles keeps 256. FI_BLOCK_N forces one.
        const long long m_tiles = static_cast<long long>(d.N) * ((d.H + TILE_H - 1) / TILE_H) * ((d.W + TILE_W - 1) / TILE_W);
        const int widths[3] = {256, 128, 64};
        const double cycles[3] = {128.0, 80.0, 56.0};
        const char* force = getenv("FI_BLOCK_N");
        const bool small = d.n_total % 256 != 0 || m_tiles * (d.n_total / 256) < num_sms;
        double best = 0;
        for (int i = 0; i < 3; ++i) {
            if (d.n_total % widths[i]) continue;
            if (force && atoi(force) == widths[i]) {
                block_n = widths[i];
                break;
            }
            if (force && atoi(force) > 0) continue;
            const long long tiles = m_tiles * (d.n_total / widths[i]);
            const double est = static_cast<double>((tiles + num_sms - 1) / num_sms) * cycles[i];
            if (best == 0 || (small && est < best * 0.999)) {
                best = est;
                block_n = widths[i];
            }
        }
    }
    ConvMaps& m = l.maps;
    if ((e = encode_nhwc(&m.a[0], d.src0, d.N, d.H, d.W, d.c0, box_w, box_h))) return e;
    m.a[1] = m.a[2] = m.a[3] = m.a[0];
    if (precise && (e = encode_nhwc(&m.a[1], d.src0_lo, d.N, d.H, d.W, d.c0, box_w, box_h))) return e;
    if (d.c1 > 0) {
        if ((e = encode_nhwc(&m.a[2], d.src1, d.N, d.h1, d.w1, d.c1, box_w, box_h))) return e;
        m.a[3] = m.a[2];
        if (precise && (e = encode_nhwc(&m.a[3], d.src1_lo, d.N, d.h1, d.w1, d.c1, box_w, box_h))) return e;
    }
    const int kmul = precise ? 3 : 1;
    {
        // CTA pairs halve the weight traffic per SM. Not for the transposed convs with a short K: they are bound by
        // their scatter store, and the pair only adds synchronisation there (measured: up4.up 0.31 -> 0.42 ms).
        // Nor for the 64->64 layers (inc.3, up4.3): their weights are already resident in the single-CTA halo kernel
        // and they are HBM-heavy; coupling two CTAs in lockstep costs more than the halved B reads save
        // (measured: inc.3 0.62 -> 0.83 ms). FI_CTA2=0 forces the single-CTA kernels everywhere (tests use it).
        const char* cta2 = getenv("FI_CTA2");
        const bool want = cta2 ? cta2[0] != '0' : true;
        const bool narrow_resident = l.halo && d.n_total == 64 && kmul * (d.c0 + d.c1) == BLOCK_K;
        l.pair = want && ((l.halo && !narrow_resident) ||
                          (!l.halo && block_n == 256 && d.mode != EPI_HEAD && (d.mode != EPI_CONVT || d.c0 >= 1024)));
    }
    {
        const uint64_t k_total = static_cast<uint64_t>(d.taps) * kmul * (d.c0 + d.c1);
        const uint64_t dims[2] = {k_total, static_cast<uint64_t>(d.n_total)};
        const uint64_t strides[1] = {k_total};
        const uint32_t box[2] = {64, static_cast<uint32_t>(l.pair ? block_n / 2 : block_n)};  // pair: half a slab per CTA
        if ((e = encode_bf16_map(&m.b, d.wpack, 2, dims, strides, box))) return e;
    }
    m.out[0] = m.out[1] = m.pool[0] = m.pool[1] = m.a[0];
    if (d.mode == EPI_STORE || d.mode == EPI_STORE_POOL) {
        if ((e = encode_nhwc(&m.out[0], d.dst, d.N, d.H, d.W, d.n_total, out_w, out_h))) return e;
        if (precise && (e = encode_nhwc(&m.out[1], d.dst_lo, d.N, d.H, d.W, d.n_total, out_w, out_h))) return e;
        if (d.mode == EPI_STORE_POOL) {
            if ((e = encode_nhwc(&m.pool[0], d.dst_pool, d.N, d.H / 2, d.W / 2, d.n_total, pool_w, pool_h))) return e;
            if (precise &&
                (e = encode_nhwc(&m.pool[1], d.dst_pool_lo, d.N, d.H / 2, d.W / 2, d.n_total, pool_w, pool_h)))
                return e;
        }
    } else if (d.mode == EPI_CONVT) {
        // dst [N, 2H, 2W, Cout] viewed as (b*Cout+co : 2Cout, j : W, a : 2, i : H, n : N)
        const uint64_t cout = d.n_total / 4;
        const uint64_t dims[5] = {2 * cout, static_cast<uint64_t>(d.W), 2, static_cast<uint64_t>(d.H),
                                  static_cast<uint64_t>(d.N)};
        const uint64_t strides[4] = {2 * cout, 2 * static_cast<uint64_t>(d.W) * cout,
                                     4 * static_cast<uint64_t>(d.W) * cout,
                                     4 * static_cast<uint64_t>(d.H) * d.W * cout};
        const uint32_t box[5] = {64, TILE_W, 1, 2, 1};
        if ((e = encode_bf16_map(&m.out[0], d.dst, 5, dims, strides, box))) return e;
        if (precise && (e = encode_bf16_map(&m.out[1], d.dst_lo, 5, dims, strides, box))) return e;
    }

    ConvKernelParams& p = l.p;
    p.tiles_x = (d.W + tile_w - 1) / tile_w;
    p.tiles_y = (d.H + tile_h - 1) / tile_h;
    p.n_img = d.N;
    p.n_blocks = d.n_total / block_n;
    p.taps = d.taps;
    // K segments of one tap: [src0] (+[src1]); precise: [src0_hi, src0_hi, src0_lo] (+ the same for src1)
    p.nseg = 0;
    for (int src = 0; src < (d.c1 > 0 ? 2 : 1); ++src) {
        const int sl = (src == 0 ? d.c0 : d.c1) / BLOCK_K;
        const int ids[3] = {2 * src, 2 * src, 2 * src + 1};
        for (int k = 0; k < kmul; ++k) {
            p.seg_slabs[p.nseg] = sl;
            p.seg_map[p.nseg] = ids[k];
            ++p.nseg;
        }
    }
    p.slabs = kmul * (d.c0 + d.c1) / BLOCK_K;
    p.off_x = d.off_x;
    p.off_y = d.off_y;
    p.relu = d.relu;
    p.cout2 = d.mode == EPI_CONVT ? d.n_total / 2 : 0;
    p.H = d.H;
    p.W = d.W;
    p.n_classes = d.n_classes;
    p.bias = d.bias;
    p.head_w = d.head_w;
    p.head_b = d.head_b;
    p.out_f32 = d.out_f32;
    p.out_u8 = d.out_u8;
    l.block_n = block_n;
    l.mode = d.mode;
    l.split = precise ? 1 : 0;
    const long long total = static_cast<long long>(p.n_blocks) * p.n_img * p.tiles_y * p.tiles_x;
    if (total > 0x7fffffffLL) return "conv: too many tiles";
    l.grid = conv_grid(l, num_sms);
    l.flops = 2.0 * d.N * d.H * d.W * static_cast<double>(d.n_total) * d.taps * (d.c0 + d.c1);
    if (d.mode == EPI_HEAD) l.flops += 2.0 * d.N * d.H * d.W * 64.0 * d.n_classes;
    *out = l;
    return nullptr;
}

int conv_grid(const ConvLaunch& l, int num_sms) {
    const ConvKernelParams& p = l.p;
    const int ctas = l.pair ? 2 : 1;
    const long long m_tiles = static_cast<long long>(p.n_img) * p.tiles_y * p.tiles_x;
    const long long units = p.n_blocks * ((m_tiles + ctas - 1) / ctas);
    return static_cast<int>(ctas * (units < num_sms / ctas ? units : num_sms / ctas));
}

const char* conv_launch(const ConvLaunch& l, cudaStream_t stream) {
    if (l.halo) return conv_halo_launch(l, stream);
    return l.pair ? launch_per_tap<2>(l, stream) : launch_per_tap<1>(l, stream);
}

}  // namespace fi
