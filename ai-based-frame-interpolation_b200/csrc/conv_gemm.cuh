// Host-side interface of the tcgen05 implicit-GEMM convolution (conv_gemm.cu).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda.h>
#include <cuda_runtime.h>

namespace fi {

// Pixel tile of one CTA: 8 rows x 16 columns of one image = 128 GEMM rows (= 128 TMEM lanes).
constexpr int TILE_H = 8;
constexpr int TILE_W = 16;
constexpr int BLOCK_M = TILE_H * TILE_W;
constexpr int BLOCK_K = 64;  // 64 bf16 channels = one 128-byte swizzle row

enum EpiMode : int {
    EPI_STORE = 0,       // bias(+ReLU) -> bf16 NHWC
    EPI_STORE_POOL = 1,  // as above, plus the 2x2/stride-2 max-pooled tensor (floor semantics)
    EPI_CONVT = 2,       // GEMM columns are (a,b,co) of a 2x2/stride-2 transposed conv: pixel-scatter store
    EPI_HEAD = 3,        // 64-channel result stays in registers: 1x1 head + bias -> fp32 NCHW and/or u8
};

// One layer as the C ABI (include/fi_b200.h: fiConvDesc) describes it. Device pointers only.
struct ConvDesc {
    const void* src0;  // bf16 NHWC [N,H,W,c0]
    int c0;
    const void* src1;  // optional second K-range source, bf16 NHWC [N,h1,w1,c1] placed at (off_y,off_x) in the HxW frame
    int c1, h1, w1, off_y, off_x;
    const void* wpack;  // bf16 [n_total][taps*(c0+c1)], K index = tap*(c0+c1) + channel
    const float* bias;  // fp32 [n_total]
    int n_total;        // GEMM N: Cout, or 4*Cout for EPI_CONVT
    int taps;           // 9 (3x3, zero pad 1) or 1
    int mode;           // EpiMode
    int relu;
    void* dst;       // EPI_STORE*: [N,H,W,n_total]; EPI_CONVT: [N,2H,2W,n_total/4]
    void* dst_pool;  // EPI_STORE_POOL: [N,H/2,W/2,n_total]
    const float* head_w;  // EPI_HEAD: fp32 [n_classes][64]
    const float* head_b;  // fp32 [n_classes]
    int n_classes;
    float* out_f32;    // EPI_HEAD: fp32 NCHW [N,n_classes,H,W] or null
    uint8_t* out_u8;   // EPI_HEAD: u8  NCHW [N,n_classes,H,W] = trunc(clamp((y+1)/2,0,1)*255) or null
    int N, H, W;
    // precise mode ("fp32x3"): every activation is a bf16 hi + bf16 lo pair (value = hi + lo, ~16 mantissa bits) and
    // the GEMM accumulates x_hi*w_hi + x_hi*w_lo + x_lo*w_hi. K per tap = 3*(c0+c1), ordered
    // [src0_hi | src0_hi | src0_lo | src1_hi | src1_hi | src1_lo] against wpack rows [w0_hi | w0_lo | w0_hi | w1_hi | ...].
    int precise;
    const void* src0_lo;
    const void* src1_lo;
    void* dst_lo;       // lo halves of dst / dst_pool (EPI_STORE*, EPI_CONVT)
    void* dst_pool_lo;
};

constexpr int MAX_SEGS = 6;

struct ConvKernelParams {
    int tiles_x, tiles_y, n_img, n_blocks;
    int taps;
    int slabs;                 // 64-channel K slabs per tap = sum of seg_slabs
    int nseg;                  // K segments per tap, each read from one source tensor map
    int seg_slabs[MAX_SEGS];
    int seg_map[MAX_SEGS];     // index into ConvMaps::a: 0 = src0 (hi), 1 = src0 lo, 2 = src1 (hi), 3 = src1 lo
    int off_x, off_y;
    int relu;
    int cout2;  // EPI_CONVT: 2*Cout (columns per output-row parity a)
    int H, W;
    int n_classes;
    const float* bias;
    const float* head_w;
    const float* head_b;
    float* out_f32;
    uint8_t* out_u8;
};

// A fully prepared launch: tensor maps are encoded once per (layer, shape) and reused every forward.
struct alignas(64) ConvMaps {
    CUtensorMap a[4];     // src0, src0 lo, src1, src1 lo
    CUtensorMap b;        // packed weights
    CUtensorMap out[2];   // dst (hi), dst lo
    CUtensorMap pool[2];  // pooled dst (hi), lo
};

struct ConvLaunch {
    ConvMaps maps;
    ConvKernelParams p;
    int block_n;
    int mode;
    int split;  // 1: precise mode, epilogue writes hi + lo tensors
    int halo;  // 1: conv_halo.cu (halo-reuse kernel for Cout 64/128), 0: conv_gemm.cu (per-tap kernel)
    int pair;  // 1: the family's CTA-pair kernel (cta_group::2, cluster of 2)
    int grid;
    double flops;  // algorithmic FLOPs of this launch (2*MACs, no padding counted)
};

// Returns nullptr on success, else a static error string.
const char* conv_prepare(const ConvDesc& d, int num_sms, ConvLaunch* out);
const char* conv_launch(const ConvLaunch& l, cudaStream_t stream);
// Persistent grid of a prepared launch for its current l.p.n_img: one CTA (or CTA pair) per work item, at most one
// per SM (pair). conv_prepare sets l.grid with it; a forward on fewer images than the plan holds calls it again.
int conv_grid(const ConvLaunch& l, int num_sms);

// bf16 tensor map (128B swizzle, zero OOB fill); dims/box innermost first, strides in elements for dims 1..rank-1.
const char* encode_bf16_map_public(CUtensorMap* map, const void* base, int rank, const uint64_t* dims,
                                   const uint64_t* strides_elems, const uint32_t* box);

// conv_inc_fused.cu: inc.double_conv.0 (stem) computed inside inc.double_conv.3's kernel (grey network, bf16 mode)
struct StemDesc;
bool inc_fused_eligible(int cin, const ConvLaunch& conv);
const char* inc_fused_launch(const StemDesc& d, const ConvLaunch& conv, const float* host_bias, int n_img, int num_sms,
                             cudaStream_t stream);

// conv_halo.cu
bool conv_halo_eligible(const ConvDesc& d);
void conv_halo_geometry(int* tile, int* box_w, int* box_h, int* out_w, int* out_h, int* pool_w, int* pool_h);
const char* conv_halo_launch(const ConvLaunch& l, cudaStream_t stream);

}  // namespace fi
