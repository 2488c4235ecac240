// Host side of libfi_b200.so: the C ABI (include/fi_b200.h), BatchNorm folding / weight repacking, the per-shape
// activation arena + prepared launch list, and the forward schedule of the UNet (reference model/unet.py:84-95).
#include "../../include/fi_b200.h"
#include "aux_kernels.cuh"
#include "conv_gemm.cuh"
#include "train_kernels.cuh"

#include <nvtx3/nvToolsExt.h>  // header-only NVTX v3: ranges are no-ops unless a profiler is attached

#include <cmath>
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <list>
#include <map>
#include <string>
#include <vector>

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_TRY(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess) return fail(FI_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e));        \
    } while (0)
#define KERNEL_TRY(expr)                                            \
    do {                                                            \
        const char* _m = (expr);                                    \
        if (_m) return fail(FI_ERR_CUDA, "%s: %s", #expr, _m);      \
    } while (0)

uint16_t f32_to_bf16_rn(float f) {
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) return static_cast<uint16_t>((u >> 16) | 0x40);  // NaN
    u += 0x7fffu + ((u >> 16) & 1u);
    return static_cast<uint16_t>(u >> 16);
}

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        bytes = 0;
    }
    cudaError_t upload(const void* host, size_t n) {
        release();
        cudaError_t e = cudaMalloc(&p, n ? n : 16);
        if (e != cudaSuccess) return e;
        bytes = n;
        return cudaMemcpy(p, host, n, cudaMemcpyHostToDevice);
    }
};

struct ConvW {     // one conv3x3+BN (or the transposed conv) after folding/packing
    int cin = 0;   // K per tap
    int n_total = 0;
    DevBuf w;      // bf16 [n_total][taps*cin]
    DevBuf b;      // fp32 [n_total]
    std::vector<float> b_host;  // the same shifts on the host (conv3x3 only)
};

struct Act {  // bf16 NHWC activation inside the arena (precise mode: a second, lo tensor at off_lo)
    size_t off = 0;
    size_t off_lo = 0;
    int C = 0, H = 0, W = 0;
    size_t bytes(int N) const { return static_cast<size_t>(N) * H * W * C * 2; }
};

enum StepKind { STEP_STEM, STEP_CONV, STEP_UPSAMPLE, STEP_INC_FUSED };
struct Step {
    StepKind kind;
    fi::ConvLaunch conv;        // STEP_CONV
    const void* src = nullptr;  // STEP_UPSAMPLE
    void* dst = nullptr;        // STEP_STEM / STEP_UPSAMPLE
    const void* src_lo = nullptr;
    void* dst_lo = nullptr;
    int h = 0, w = 0, C = 0;
    char name[48] = "";
    double flops = 0;  // algorithmic FLOPs of the launch, per image
    double bytes = 0;  // algorithmic HBM bytes of the launch per image (activations in + out; weights excluded)
    double weight_bytes = 0;
};

struct Plan {
    int N = 0, H = 0, W = 0;  // N = batch CAPACITY of the arena / tensor maps; any batch <= N runs without re-planning
    DevBuf arena;
    std::map<std::string, Act> acts;
    std::vector<Step> steps;
    int head_step = -1;
    bool reuse = false;  // arena placed with liveness reuse: intermediate tensors are overwritten during the forward
    int last_n = 0;    // batch of the most recent forward
    double flops = 0;  // per image
    void reset() {
        steps.clear();
        acts.clear();
        arena.release();
        N = H = W = 0;
        head_step = -1;
        last_n = 0;
        flops = 0;
    }
};

}  // namespace

struct fiNet {
    int device = 0;
    int n_channels = 2, n_classes = 1, bilinear = 0;
    int precise = 0;  // FI_PRECISION_FP32X3: hi/lo-split activations and weights, three products per MAC
    int num_sms = 148;
    bool loaded = false;
    DevBuf stem_w, stem_b;  // bf16 [64][stem_packed_k] hi/lo split, fp32 [64]
    float inc_bias_host[128] = {};  // folded shifts of inc.double_conv.0 and .3 for the fused kernel's parameters
    ConvW convs[17];        // inc.3, down{1-4}.{0,3}, up{1-4}.{0,3}
    ConvW upT[4];           // ConvTranspose2d of up1..up4 (bilinear=False)
    DevBuf head_w, head_b;  // fp32 [n_classes][64], [n_classes]
    // Prepared plans (arena + tensor maps + launch list), one per frame size, most recently used first. A server that
    // alternates between shapes (256x256 API requests, 1080p video, the levels of a mixed clip) re-uses them instead of
    // re-allocating a multi-GB arena and re-encoding ~60 tensor maps on every switch. FI_PLAN_CACHE (default 4) bounds
    // the list; the least recently used plan is dropped first, and all idle plans are dropped when an arena does not fit.
    std::list<Plan> plans;
    int max_plans = 4;
    long long plan_builds = 0;  // how many plans were built so far (observability: fiNetPlanStats)
    Plan& plan() { return plans.front(); }
    bool has_plan() const { return !plans.empty(); }
    void drop_plans() { plans.clear(); }
    bool nvtx = false;  // FI_NVTX=1: one NVTX range per forward and per layer launch (named like the state-dict layer)
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;  // [call][step][2], resolved by fiNetGetProfile
    int prof_calls = 0;
    // host-clip pipeline (fiNetInterpolateDyadicHostU8): double-buffered pinned + device staging, copy streams, events
    struct ClipSlot {
        void* pin_in = nullptr;
        void* dev_in = nullptr;
        cudaEvent_t in_ready = nullptr, done = nullptr, out_ready = nullptr;
        uint64_t* pin_sad = nullptr;  // per-pair SAD of the group (when the caller asks for it)
        uint64_t* dev_sad = nullptr;
        DevBuf pool;                  // every node of the group's bisection tree
        void* pin_nodes = nullptr;    // ... and the requested nodes on their way to the host
        size_t pin_nodes_bytes = 0;
    } clip[2];
    size_t clip_in_bytes = 0;
    int clip_sad_pairs = 0;  // capacity of pin_sad / dev_sad
    cudaStream_t clip_h2d = nullptr, clip_d2h = nullptr;
    DevBuf dyadic_gather;    // in0 | in1 of one bisection forward: the parents of up to pairs_per_batch nodes
    // pinned staging for the host-buffer convenience call
    void* pin_in = nullptr;
    void* pin_out = nullptr;
    size_t pin_in_bytes = 0, pin_out_bytes = 0;
    DevBuf dev_in, dev_out;
};

namespace {

// conv index helpers: 0 = inc.3; 1,2 = down1.{0,3}; ... 7,8 = down4; 9,10 = up1.{0,3}; ... 15,16 = up4
struct ConvShape {
    int cin, cout;
};
void conv_shapes(const fiNet* net, ConvShape (&cs)[17], ConvShape& stem, int (&upc)[4][2]) {
    const int f = net->bilinear ? 2 : 1;
    stem = {net->n_channels, 64};
    cs[0] = {64, 64};
    const int enc[5] = {64, 128, 256, 512, 1024 / f};
    for (int i = 1; i <= 4; ++i) {
        cs[2 * i - 1] = {enc[i - 1], enc[i]};
        cs[2 * i] = {enc[i], enc[i]};
    }
    // Up(in, out): bilinear: DoubleConv(in, out, mid=in/2); else ConvT(in, in/2) + DoubleConv(in, out)
    const int up_in[4] = {1024, 512, 256, 128};
    const int up_out[4] = {512 / f, 256 / f, 128 / f, 64};
    for (int i = 0; i < 4; ++i) {
        const int mid = net->bilinear ? up_in[i] / 2 : up_out[i];
        cs[9 + 2 * i] = {up_in[i], mid};
        cs[10 + 2 * i] = {mid, up_out[i]};
        upc[i][0] = net->bilinear ? up_in[i] / 2 : up_in[i];  // channels entering the upsample
        upc[i][1] = up_in[i] / 2;                             // channels leaving it
    }
}

std::string conv_prefix(int idx) {
    char buf[64];
    if (idx == 0) return "inc.double_conv.3";
    if (idx <= 8) {
        snprintf(buf, sizeof buf, "down%d.maxpool_conv.1.double_conv.%d", (idx + 1) / 2, (idx % 2) ? 0 : 3);
        return buf;
    }
    const int u = (idx - 9) / 2 + 1;
    snprintf(buf, sizeof buf, "up%d.conv.double_conv.%d", u, ((idx - 9) % 2) ? 3 : 0);
    return buf;
}
std::string bn_of(const std::string& conv_key) {  // "...double_conv.0" -> "...double_conv.1"
    std::string s = conv_key;
    s.back() = static_cast<char>(s.back() + 1);
    return s;
}

struct StateDict {
    std::map<std::string, std::pair<const float*, int64_t>> m;
    const float* get(const std::string& key, int64_t numel, std::string* err) const {
        auto it = m.find(key);
        if (it == m.end()) it = m.find("unet." + key);
        if (it == m.end()) {
            *err = "missing state-dict entry '" + key + "'";
            return nullptr;
        }
        if (it->second.second != numel) {
            char b[160];
            snprintf(b, sizeof b, "size mismatch for '%s': got %lld elements, expected %lld", key.c_str(),
                     static_cast<long long>(it->second.second), static_cast<long long>(numel));
            *err = b;
            return nullptr;
        }
        return it->second.first;
    }
};

// BN(eval) fold, reference model/unet.py:13,16 (eps = 1e-5, nn.BatchNorm2d default).
bool bn_fold(const StateDict& sd, const std::string& bn, int c, std::vector<double>* scale, std::vector<float>* shift,
             std::string* err) {
    const float* g = sd.get(bn + ".weight", c, err);
    const float* b = g ? sd.get(bn + ".bias", c, err) : nullptr;
    const float* mu = b ? sd.get(bn + ".running_mean", c, err) : nullptr;
    const float* var = mu ? sd.get(bn + ".running_var", c, err) : nullptr;
    if (!var) return false;
    scale->resize(c);
    shift->resize(c);
    for (int i = 0; i < c; ++i) {
        const double s = static_cast<double>(g[i]) / std::sqrt(static_cast<double>(var[i]) + 1e-5);
        (*scale)[i] = s;
        (*shift)[i] = static_cast<float>(static_cast<double>(b[i]) - static_cast<double>(mu[i]) * s);
    }
    return true;
}

// One packed weight row: per tap, per source block [c_begin, c_end): bf16 [w] or, in precise mode, [w_hi | w_lo | w_hi].
void pack_row(const std::vector<double>& w_tap_ci /*[taps][cin]*/, int taps, int cin, const int* blocks, int nblocks,
              bool precise, uint16_t* row) {
    size_t o = 0;
    for (int t = 0; t < taps; ++t) {
        int c0 = 0;
        for (int b = 0; b < nblocks; ++b) {
            const int c1 = c0 + blocks[b];
            if (!precise) {
                for (int c = c0; c < c1; ++c) row[o++] = f32_to_bf16_rn(static_cast<float>(w_tap_ci[static_cast<size_t>(t) * cin + c]));
            } else {
                for (int pass = 0; pass < 3; ++pass)
                    for (int c = c0; c < c1; ++c) {
                        const float v = static_cast<float>(w_tap_ci[static_cast<size_t>(t) * cin + c]);
                        const uint16_t h = f32_to_bf16_rn(v);
                        uint32_t hb = static_cast<uint32_t>(h) << 16;
                        float hf;
                        memcpy(&hf, &hb, 4);
                        row[o++] = pass == 1 ? f32_to_bf16_rn(v - hf) : h;
                    }
            }
            c0 = c1;
        }
    }
}

int load_conv3x3(const StateDict& sd, const std::string& key, int cin, int cout, ConvW* out, bool precise = false,
                 int split_at = 0) {
    std::string err;
    const float* w = sd.get(key + ".weight", static_cast<int64_t>(cout) * cin * 9, &err);
    std::vector<double> scale;
    std::vector<float> shift;
    if (!w || !bn_fold(sd, bn_of(key), cout, &scale, &shift, &err)) return fail(FI_ERR_WEIGHTS, "%s", err.c_str());
    const size_t K = static_cast<size_t>(9) * cin * (precise ? 3 : 1);
    std::vector<uint16_t> packed(static_cast<size_t>(cout) * K);
    std::vector<double> wt(static_cast<size_t>(9) * cin);
    const int blocks[2] = {split_at > 0 ? split_at : cin, cin - split_at};  // fused concat: skip block, then up block
    for (int co = 0; co < cout; ++co) {
        for (int ci = 0; ci < cin; ++ci)
            for (int t = 0; t < 9; ++t)
                wt[static_cast<size_t>(t) * cin + ci] =
                    static_cast<double>(w[(static_cast<size_t>(co) * cin + ci) * 9 + t]) * scale[co];
        pack_row(wt, 9, cin, blocks, split_at > 0 ? 2 : 1, precise, packed.data() + co * K);
    }
    out->cin = cin;
    out->n_total = cout;
    CUDA_TRY(out->w.upload(packed.data(), packed.size() * 2));
    CUDA_TRY(out->b.upload(shift.data(), shift.size() * 4));
    out->b_host = shift;
    return FI_OK;
}

int load_convT(const StateDict& sd, const std::string& key, int cin, int cout, ConvW* out, bool precise = false) {
    std::string err;
    const float* w = sd.get(key + ".weight", static_cast<int64_t>(cin) * cout * 4, &err);  // [cin][cout][2][2]
    const float* b = w ? sd.get(key + ".bias", cout, &err) : nullptr;
    if (!b) return fail(FI_ERR_WEIGHTS, "%s", err.c_str());
    const size_t K = static_cast<size_t>(cin) * (precise ? 3 : 1);
    std::vector<uint16_t> packed(static_cast<size_t>(4) * cout * K);
    std::vector<float> bias4(static_cast<size_t>(4) * cout);
    std::vector<double> wt(cin);
    for (int ab = 0; ab < 4; ++ab)
        for (int co = 0; co < cout; ++co) {
            bias4[static_cast<size_t>(ab) * cout + co] = b[co];
            for (int ci = 0; ci < cin; ++ci) wt[ci] = w[(static_cast<size_t>(ci) * cout + co) * 4 + ab];
            pack_row(wt, 1, cin, &cin, 1, precise, packed.data() + (static_cast<size_t>(ab) * cout + co) * K);
        }
    out->cin = cin;
    out->n_total = 4 * cout;
    CUDA_TRY(out->w.upload(packed.data(), packed.size() * 2));
    CUDA_TRY(out->b.upload(bias4.data(), bias4.size() * 4));
    return FI_OK;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int fill_plan(fiNet* net, Plan& pl, int N, int H, int W);

// Makes the plan for (N, H, W) the current one (net->plan()): an existing plan of that frame size with enough batch
// capacity is moved to the front of the LRU list, otherwise a new one is built (replacing a smaller one of the same size).
int build_plan(fiNet* net, int N, int H, int W) {
    if ((H >> 4) < 1 || (W >> 4) < 1) return fail(FI_ERR_INVALID, "input %dx%d is smaller than 16x16 (4 poolings)", H, W);
    for (auto it = net->plans.begin(); it != net->plans.end(); ++it) {
        if (it->H != H || it->W != W || !it->arena.p) continue;
        if (it->N >= N) {
            if (it != net->plans.begin()) net->plans.splice(net->plans.begin(), net->plans, it);
            return FI_OK;
        }
        net->plans.erase(it);  // same frame size, smaller batch capacity: superseded
        break;
    }
    while (static_cast<int>(net->plans.size()) >= net->max_plans && !net->plans.empty()) net->plans.pop_back();
    net->plans.emplace_front();
    int rc = fill_plan(net, net->plans.front(), N, H, W);
    if (rc == FI_ERR_NOMEM && net->plans.size() > 1) {  // make room: drop every idle plan and try once more
        net->plans.resize(1);
        net->plans.front().reset();
        rc = fill_plan(net, net->plans.front(), N, H, W);
    }
    if (rc != FI_OK) {
        net->plans.pop_front();
        return rc;
    }
    ++net->plan_builds;
    return FI_OK;
}

int fill_plan(fiNet* net, Plan& pl, int N, int H, int W) {
    pl.reset();

    ConvShape cs[17], stem;
    int upc[4][2];
    conv_shapes(net, cs, stem, upc);

    int hs[5], ws[5];
    hs[0] = H;
    ws[0] = W;
    for (int i = 1; i < 5; ++i) {
        hs[i] = hs[i - 1] / 2;
        ws[i] = ws[i - 1] / 2;
    }
    // Activation tensors with the schedule steps that write / last read them (step numbering: 0 stem, 1 inc.3,
    // 2i / 2i+1 the two convs of down_i, 10+3k / +1 / +2 = up, conv.0, conv.3 of up_{k+1}).
    struct Item {
        std::string name;
        int C, h, w, first, last;
    };
    std::vector<Item> items;
    auto add = [&](const std::string& name, int C, int h, int w, int first, int last) {
        items.push_back({name, C, h, w, first, last});
    };
    const int enc_c[5] = {64, cs[2].cout, cs[4].cout, cs[6].cout, cs[8].cout};
    // Grey network in bf16 mode: inc.double_conv.0 is computed inside inc.double_conv.3's kernel (conv_inc_fused.cu) and
    // inc.mid does not exist: bit-identical to the two separate launches, 530 MB less HBM traffic per 1080p pair, +2.3 %
    // frames/s at the sustained (power-capped) clock. FI_FUSE_INC=0 keeps the two launches.
    const char* fuse_env = getenv("FI_FUSE_INC");
    const char* no_halo_env = getenv("FI_NO_HALO");
    const bool fuse_inc = net->n_channels <= 2 && !net->precise && !(fuse_env && fuse_env[0] == '0') &&
                          !(no_halo_env && no_halo_env[0] == '1');
    if (!fuse_inc) add("inc.mid", 64, hs[0], ws[0], 0, 1);
    add("inc", 64, hs[0], ws[0], 1, 20);
    for (int i = 1; i <= 4; ++i) {
        char nm[32];
        snprintf(nm, sizeof nm, "pool%d", i);
        add(nm, enc_c[i - 1], hs[i], ws[i], 2 * i - 1, 2 * i);
        snprintf(nm, sizeof nm, "down%d.mid", i);
        add(nm, enc_c[i], hs[i], ws[i], 2 * i, 2 * i + 1);
        snprintf(nm, sizeof nm, "down%d", i);
        add(nm, enc_c[i], hs[i], ws[i], 2 * i + 1, i == 4 ? 10 : 10 + 3 * (3 - i) + 1);  // skip read by up_{4-i}.conv.0
    }
    for (int i = 0; i < 4; ++i) {
        char nm[32];
        const int lvl = 3 - i;  // skip level of up(i+1)
        const int base = 10 + 3 * i;
        snprintf(nm, sizeof nm, "up%d.up", i + 1);
        add(nm, upc[i][1], 2 * hs[lvl + 1], 2 * ws[lvl + 1], base, base + 1);
        snprintf(nm, sizeof nm, "up%d.mid", i + 1);
        add(nm, cs[9 + 2 * i].cout, hs[lvl], ws[lvl], base + 1, base + 2);
        if (i < 3) {
            snprintf(nm, sizeof nm, "up%d", i + 1);
            add(nm, cs[10 + 2 * i].cout, hs[lvl], ws[lvl], base + 2, base + 3);
        }
    }
    // Placement. Default: every tensor has its own memory (fiNetReadActivation can tap any of them after the forward).
    // Liveness reuse (FI_ARENA_REUSE=1, or automatically when the plain layout would exceed 16 GiB — 4K frames x 8 pairs
    // is 74 GB): a tensor may take the memory of tensors whose last reader ran in an earlier step. Kernels of
    // consecutive steps never overlap in their memory accesses (programmatic dependent launch waits for the previous grid
    // to complete before touching memory), so step granularity is exact. First fit over the tensors alive in between.
    const size_t mult = net->precise ? 2 : 1;
    auto bytes_of = [&](const Item& it) { return align_up(static_cast<size_t>(N) * it.h * it.w * it.C * 2, 1024); };
    size_t plain = 0;
    for (const Item& it : items) plain += mult * bytes_of(it);
    const char* reuse_env = getenv("FI_ARENA_REUSE");
    pl.reuse = reuse_env ? reuse_env[0] == '1' : plain > (size_t(16) << 30);
    size_t cursor = 0;
    struct Placed {
        size_t off, bytes;
        int first, last;
    };
    std::vector<Placed> placed;
    for (const Item& it : items) {
        const size_t bytes = mult * bytes_of(it);
        size_t off = cursor;
        if (pl.reuse) {
            std::vector<Placed> live;
            for (const Placed& q : placed)
                if (!(q.last < it.first || it.last < q.first)) live.push_back(q);
            std::sort(live.begin(), live.end(), [](const Placed& a, const Placed& b) { return a.off < b.off; });
            off = 0;
            for (const Placed& q : live) {
                if (off + bytes <= q.off) break;
                if (q.off + q.bytes > off) off = q.off + q.bytes;
            }
        }
        placed.push_back({off, bytes, it.first, it.last});
        if (off + bytes > cursor) cursor = off + bytes;
        Act a;
        a.off = off;
        a.off_lo = net->precise ? off + bytes_of(it) : 0;
        a.C = it.C;
        a.H = it.h;
        a.W = it.w;
        pl.acts[it.name] = a;
    }
    if (fuse_inc) pl.acts["inc.mid"] = pl.acts.at("inc");   // only to describe the layer; the fused kernel never reads it
    {
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, cursor);
        if (e != cudaSuccess)
            return fail(FI_ERR_NOMEM, "activation arena of %zu bytes: %s", cursor, cudaGetErrorString(e));
        pl.arena.p = p;
        pl.arena.bytes = cursor;
    }
    auto ptr = [&](const std::string& name) -> void* {
        return static_cast<char*>(pl.arena.p) + pl.acts.at(name).off;
    };
    auto ptr_lo = [&](const std::string& name) -> void* {
        return net->precise ? static_cast<char*>(pl.arena.p) + pl.acts.at(name).off_lo : nullptr;
    };

    pl.flops = 2.0 * H * W * 64.0 * 9 * stem.cin;
    auto push_conv = [&](fi::ConvDesc d, const std::string& name) -> int {
        Step s;
        s.kind = STEP_CONV;
        d.N = N;
        const char* e = fi::conv_prepare(d, net->num_sms, &s.conv);
        if (e) return fail(FI_ERR_INVALID, "%s", e);
        pl.flops += s.conv.flops / N;
        snprintf(s.name, sizeof s.name, "%s", name.c_str());
        s.flops = s.conv.flops / N;
        const double px = static_cast<double>(d.H) * d.W;
        s.bytes = px * d.c0 * 2 + static_cast<double>(d.h1) * d.w1 * d.c1 * 2;
        s.weight_bytes = static_cast<double>(d.n_total) * d.taps * (d.c0 + d.c1) * 2;
        if (d.mode == fi::EPI_HEAD) s.bytes += px * d.n_classes * 4;
        else s.bytes += px * d.n_total * 2 * (d.mode == fi::EPI_STORE_POOL ? 1.25 : 1.0);
        pl.steps.push_back(s);
        return FI_OK;
    };
    auto conv3 = [&](int idx, const std::string& src, const std::string& src1, const std::string& dst,
                     const std::string& pool, int mode) -> int {
        const Act& a = pl.acts.at(src);
        fi::ConvDesc d;
        memset(&d, 0, sizeof d);
        d.src0 = ptr(src);
        d.src0_lo = ptr_lo(src);
        d.precise = net->precise;
        d.c0 = a.C;
        d.H = a.H;
        d.W = a.W;
        if (!src1.empty()) {
            const Act& b = pl.acts.at(src1);
            d.src1 = ptr(src1);
            d.src1_lo = ptr_lo(src1);
            d.c1 = b.C;
            d.h1 = b.H;
            d.w1 = b.W;
            d.off_y = (a.H - b.H) / 2;  // F.pad(x1, [dX//2, dX-dX//2, dY//2, dY-dY//2]) reference model/unet.py:49-53
            d.off_x = (a.W - b.W) / 2;
        }
        const ConvW& cw = net->convs[idx];
        if (cw.cin != d.c0 + d.c1) return fail(FI_ERR_STATE, "internal: conv %d expects %d channels, got %d", idx, cw.cin, d.c0 + d.c1);
        d.wpack = cw.w.p;
        d.bias = static_cast<const float*>(cw.b.p);
        d.n_total = cw.n_total;
        d.taps = 9;
        d.mode = mode;
        d.relu = 1;
        if (mode == fi::EPI_HEAD) {
            d.head_w = static_cast<const float*>(net->head_w.p);
            d.head_b = static_cast<const float*>(net->head_b.p);
            d.n_classes = net->n_classes;
            d.out_f32 = reinterpret_cast<float*>(16);  // patched per forward call
        } else {
            d.dst = ptr(dst);
            d.dst_lo = ptr_lo(dst);
            if (mode == fi::EPI_STORE_POOL) {
                d.dst_pool = ptr(pool);
                d.dst_pool_lo = ptr_lo(pool);
            }
        }
        return push_conv(d, conv_prefix(idx));
    };

    int rc;
    {
        Step s;
        s.kind = STEP_STEM;
        s.dst = ptr("inc.mid");
        s.dst_lo = ptr_lo("inc.mid");
        snprintf(s.name, sizeof s.name, "inc.double_conv.0");
        s.flops = 2.0 * H * W * 64.0 * 9 * stem.cin;
        s.bytes = static_cast<double>(H) * W * (stem.cin * 4.0 + 128.0);
        pl.steps.push_back(s);
    }
    if ((rc = conv3(0, "inc.mid", "", "inc", "pool1", fi::EPI_STORE_POOL))) return rc;
    {
        // the stem is computed inside inc.double_conv.3's kernel (conv_inc_fused.cu), inc.mid never reaches HBM
        // (FI_FUSE_INC=0: two launches; tests compare the two schedules bit for bit)
        Step& conv_step = pl.steps.back();
        if (fuse_inc && !fi::inc_fused_eligible(net->n_channels, conv_step.conv))
            return fail(FI_ERR_STATE, "internal: inc.double_conv.3 was not prepared as the resident halo kernel");
        if (fuse_inc) {
            Step fused = conv_step;
            fused.kind = STEP_INC_FUSED;
            snprintf(fused.name, sizeof fused.name, "inc.double_conv.0+3");
            fused.flops += pl.steps[0].flops;
            const double px = static_cast<double>(H) * W;
            fused.bytes = px * (stem.cin * 4.0 + 64 * 2 * 1.25);   // raw planes in, inc + pool1 out
            pl.steps.clear();
            pl.steps.push_back(fused);
        }
    }
    for (int i = 1; i <= 4; ++i) {
        char pool[32], mid[32], out[32], nextpool[32];
        snprintf(pool, sizeof pool, "pool%d", i);
        snprintf(mid, sizeof mid, "down%d.mid", i);
        snprintf(out, sizeof out, "down%d", i);
        snprintf(nextpool, sizeof nextpool, "pool%d", i + 1);
        if ((rc = conv3(2 * i - 1, pool, "", mid, "", fi::EPI_STORE))) return rc;
        if ((rc = conv3(2 * i, mid, "", out, nextpool, i < 4 ? fi::EPI_STORE_POOL : fi::EPI_STORE))) return rc;
    }
    const char* skips[4] = {"down3", "down2", "down1", "inc"};
    std::string below = "down4";
    for (int i = 0; i < 4; ++i) {
        char up[32], mid[32], out[32];
        snprintf(up, sizeof up, "up%d.up", i + 1);
        snprintf(mid, sizeof mid, "up%d.mid", i + 1);
        snprintf(out, sizeof out, "up%d", i + 1);
        const Act& lo = pl.acts.at(below);
        if (net->bilinear) {
            Step s;
            s.kind = STEP_UPSAMPLE;
            s.src = ptr(below);
            s.dst = ptr(up);
            s.src_lo = ptr_lo(below);
            s.dst_lo = ptr_lo(up);
            s.h = lo.H;
            s.w = lo.W;
            s.C = lo.C;
            snprintf(s.name, sizeof s.name, "up%d.up", i + 1);
            s.bytes = static_cast<double>(lo.H) * lo.W * lo.C * 2 * 5.0;
            pl.steps.push_back(s);
        } else {
            fi::ConvDesc d;
            memset(&d, 0, sizeof d);
            const ConvW& cw = net->upT[i];
            d.src0 = ptr(below);
            d.src0_lo = ptr_lo(below);
            d.precise = net->precise;
            d.c0 = lo.C;
            d.H = lo.H;
            d.W = lo.W;
            d.wpack = cw.w.p;
            d.bias = static_cast<const float*>(cw.b.p);
            d.n_total = cw.n_total;
            d.taps = 1;
            d.mode = fi::EPI_CONVT;
            d.relu = 0;
            d.dst = ptr(up);
            d.dst_lo = ptr_lo(up);
            if ((rc = push_conv(d, up))) return rc;
        }
        if ((rc = conv3(9 + 2 * i, skips[i], up, mid, "", fi::EPI_STORE))) return rc;
        if (i < 3) {
            if ((rc = conv3(10 + 2 * i, mid, "", out, "", fi::EPI_STORE))) return rc;
        } else {
            if ((rc = conv3(10 + 2 * i, mid, "", "", "", fi::EPI_HEAD))) return rc;
            pl.head_step = static_cast<int>(pl.steps.size()) - 1;
        }
        below = out;
    }
    pl.N = N;
    pl.H = H;
    pl.W = W;
    return FI_OK;
}

int check_planes(const fiNet* net, const fiPlanes* in0, const fiPlanes* in1) {
    if (!in0 || !in0->ptr) return fail(FI_ERR_INVALID, "in0 is required");
    const int c = in0->channels + (in1 ? in1->channels : 0);
    if (in1 && !in1->ptr) return fail(FI_ERR_INVALID, "in1 has no data pointer");
    if (c != net->n_channels)
        return fail(FI_ERR_INVALID, "input planes provide %d channels, network expects %d", c, net->n_channels);
    return FI_OK;
}

fi::PlaneSrc to_src(const fiPlanes* p) {
    fi::PlaneSrc s;
    memset(&s, 0, sizeof s);
    if (p) {
        s.ptr = p->ptr;
        s.batch_stride = p->batch_stride;
        s.chan_stride = p->chan_stride;
        s.row_stride = p->row_stride;
        s.px_stride = p->px_stride;
        s.channels = p->channels;
    }
    return s;
}

// Every entry point that works on a handle switches to the handle's device for the duration of the call and puts the
// caller's current device back on every exit path: a library must not leave cudaSetDevice side effects behind (torch's
// "current device" IS the runtime's, so a leaked switch silently re-targets the caller's next "cuda" tensor).
struct DeviceGuard {
    int prev = -1;
    int rc = FI_OK;
    explicit DeviceGuard(int device) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != device) {
            const cudaError_t e = cudaSetDevice(device);
            if (e != cudaSuccess) rc = fail(FI_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
        } else {
            prev = -1;  // nothing to restore
        }
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
    DeviceGuard(const DeviceGuard&) = delete;
    DeviceGuard& operator=(const DeviceGuard&) = delete;
};
#define ON_DEVICE(device)              \
    DeviceGuard _device_guard(device); \
    if (_device_guard.rc) return _device_guard.rc

// Copy streams, events and the double-buffered input staging of the pipelined host-clip call: per slot at least
// in_bytes of pinned and device input, and with `sad` B per-pair SAD values. Buffers only grow.
int clip_staging(fiNet* net, int B, size_t in_bytes, bool sad) {
    if (!net->clip_h2d) {
        CUDA_TRY(cudaStreamCreateWithFlags(&net->clip_h2d, cudaStreamNonBlocking));
        CUDA_TRY(cudaStreamCreateWithFlags(&net->clip_d2h, cudaStreamNonBlocking));
        for (auto& c : net->clip) {
            CUDA_TRY(cudaEventCreateWithFlags(&c.in_ready, cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&c.done, cudaEventDisableTiming));
            CUDA_TRY(cudaEventCreateWithFlags(&c.out_ready, cudaEventDisableTiming));
        }
    }
    if (net->clip_in_bytes < in_bytes) {
        CUDA_TRY(cudaDeviceSynchronize());
        for (auto& c : net->clip) {
            if (c.pin_in) cudaFreeHost(c.pin_in);
            if (c.dev_in) cudaFree(c.dev_in);
            c.pin_in = c.dev_in = nullptr;
        }
        net->clip_in_bytes = 0;
        for (auto& c : net->clip) {
            CUDA_TRY(cudaMallocHost(&c.pin_in, in_bytes));
            CUDA_TRY(cudaMalloc(&c.dev_in, in_bytes));
        }
        net->clip_in_bytes = in_bytes;
    }
    if (sad && net->clip_sad_pairs < B) {
        CUDA_TRY(cudaDeviceSynchronize());
        for (auto& c : net->clip) {
            if (c.pin_sad) cudaFreeHost(c.pin_sad);
            if (c.dev_sad) cudaFree(c.dev_sad);
            c.pin_sad = c.dev_sad = nullptr;
        }
        net->clip_sad_pairs = 0;
        for (auto& c : net->clip) {
            CUDA_TRY(cudaMallocHost(reinterpret_cast<void**>(&c.pin_sad), B * sizeof(uint64_t)));
            CUDA_TRY(cudaMalloc(reinterpret_cast<void**>(&c.dev_sad), B * sizeof(uint64_t)));
        }
        net->clip_sad_pairs = B;
    }
    return FI_OK;
}

// Planes of `n` planar u8 images of `channels` x H x W, `stride` bytes apart, starting at ptr.
fiPlanes u8_planes(const void* ptr, int channels, int H, int W, int64_t stride) {
    fiPlanes p;
    p.ptr = ptr;
    p.channels = channels;
    p.px_stride = 1;
    p.row_stride = W;
    p.chan_stride = static_cast<int64_t>(H) * W;
    p.batch_stride = stride;
    return p;
}

}  // namespace

extern "C" {

int fiVersion(void) { return 100; }
const char* fiLastError(void) { return g_err; }

int fiNetCreate(fiNet** out, int device, int n_channels, int n_classes, int bilinear) {
    if (!out) return fail(FI_ERR_INVALID, "out is null");
    *out = nullptr;
    if (n_channels < 1 || n_channels > 8) return fail(FI_ERR_INVALID, "n_channels must be in 1..8");
    if (n_classes < 1 || n_classes > 4) return fail(FI_ERR_INVALID, "n_classes must be in 1..4");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(FI_ERR_CUDA, "no CUDA device available (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(FI_ERR_INVALID, "device %d out of range (%d devices)", device, ndev);
    ON_DEVICE(device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(FI_ERR_CUDA, "device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major,
                    prop.minor);
    fiNet* net = new fiNet();
    net->device = device;
    net->n_channels = n_channels;
    net->n_classes = n_classes;
    net->bilinear = bilinear ? 1 : 0;
    net->num_sms = prop.multiProcessorCount;
    if (const char* e = getenv("FI_PLAN_CACHE")) net->max_plans = atoi(e) > 0 ? atoi(e) : 1;
    if (const char* e = getenv("FI_NVTX")) net->nvtx = e[0] == '1';
    *out = net;
    return FI_OK;
}

int fiNetSetPrecision(fiNet* net, int precision) {
    if (!net) return fail(FI_ERR_INVALID, "net is null");
    if (precision != FI_PRECISION_BF16 && precision != FI_PRECISION_FP32X3)
        return fail(FI_ERR_INVALID, "unknown precision %d", precision);
    if (net->precise != precision) {  // packed weights and the arena layout depend on it
        net->precise = precision;
        net->loaded = false;
        net->drop_plans();
    }
    return FI_OK;
}

int fiNetDestroy(fiNet* net) {
    if (!net) return FI_OK;
    DeviceGuard guard(net->device);
    if (net->pin_in) cudaFreeHost(net->pin_in);
    if (net->pin_out) cudaFreeHost(net->pin_out);
    for (cudaEvent_t e : net->prof_events) cudaEventDestroy(e);
    for (auto& c : net->clip) {
        if (c.pin_in) cudaFreeHost(c.pin_in);
        if (c.dev_in) cudaFree(c.dev_in);
        if (c.pin_sad) cudaFreeHost(c.pin_sad);
        if (c.dev_sad) cudaFree(c.dev_sad);
        if (c.pin_nodes) cudaFreeHost(c.pin_nodes);
        if (c.in_ready) cudaEventDestroy(c.in_ready);
        if (c.done) cudaEventDestroy(c.done);
        if (c.out_ready) cudaEventDestroy(c.out_ready);
    }
    if (net->clip_h2d) cudaStreamDestroy(net->clip_h2d);
    if (net->clip_d2h) cudaStreamDestroy(net->clip_d2h);
    delete net;
    return FI_OK;
}

int fiNetLoadWeights(fiNet* net, const char* const* names, const float* const* data_host, const int64_t* numel,
                     int count) {
    if (!net || !names || !data_host || !numel) return fail(FI_ERR_INVALID, "null argument");
    ON_DEVICE(net->device);
    int rc = FI_OK;
    StateDict sd;
    for (int i = 0; i < count; ++i) sd.m[names[i]] = {data_host[i], numel[i]};
    net->loaded = false;
    net->drop_plans();  // launches hold weight pointers

    ConvShape cs[17], stem;
    int upc[4][2];
    conv_shapes(net, cs, stem, upc);
    std::string err;
    {   // stem: BN folded in fp64 (inc.double_conv.0 / .1), then split into bf16 hi/lo rows for the tensor-core stem
        const float* w = sd.get("inc.double_conv.0.weight", static_cast<int64_t>(64) * stem.cin * 9, &err);
        std::vector<double> scale;
        std::vector<float> shift;
        if (!w || !bn_fold(sd, "inc.double_conv.1", 64, &scale, &shift, &err))
            return fail(FI_ERR_WEIGHTS, "%s", err.c_str());
        std::vector<float> ws(static_cast<size_t>(64) * stem.cin * 9);
        for (int co = 0; co < 64; ++co)
            for (size_t i = 0; i < static_cast<size_t>(stem.cin) * 9; ++i)
                ws[co * static_cast<size_t>(stem.cin) * 9 + i] = static_cast<float>(
                    static_cast<double>(w[co * static_cast<size_t>(stem.cin) * 9 + i]) * scale[co]);
        std::vector<uint16_t> packed(static_cast<size_t>(64) * fi::stem_packed_k(stem.cin));
        fi::stem_pack_weights(ws.data(), stem.cin, packed.data());
        CUDA_TRY(net->stem_w.upload(packed.data(), packed.size() * 2));
        CUDA_TRY(net->stem_b.upload(shift.data(), shift.size() * 4));
        memcpy(net->inc_bias_host, shift.data(), 64 * sizeof(float));
    }
    for (int i = 0; i < 17; ++i) {
        // up{k}.conv.double_conv.0 (indices 9, 11, 13, 15) reads [skip | up]: two K blocks of cin/2 channels each
        const int split_at = (i >= 9 && (i - 9) % 2 == 0) ? cs[i].cin / 2 : 0;
        if ((rc = load_conv3x3(sd, conv_prefix(i), cs[i].cin, cs[i].cout, &net->convs[i], net->precise != 0, split_at)))
            return rc;
    }
    if (net->convs[0].b_host.size() == 64) memcpy(net->inc_bias_host + 64, net->convs[0].b_host.data(), 64 * sizeof(float));
    if (!net->bilinear) {
        for (int i = 0; i < 4; ++i) {
            char key[32];
            snprintf(key, sizeof key, "up%d.up", i + 1);
            if ((rc = load_convT(sd, key, upc[i][0], upc[i][1], &net->upT[i], net->precise != 0))) return rc;
        }
    }
    {
        const float* w = sd.get("outc.conv.weight", static_cast<int64_t>(net->n_classes) * 64, &err);
        const float* b = w ? sd.get("outc.conv.bias", net->n_classes, &err) : nullptr;
        if (!b) return fail(FI_ERR_WEIGHTS, "%s", err.c_str());
        CUDA_TRY(net->head_w.upload(w, static_cast<size_t>(net->n_classes) * 64 * 4));
        CUDA_TRY(net->head_b.upload(b, static_cast<size_t>(net->n_classes) * 4));
    }
    net->loaded = true;
    return FI_OK;
}

int fiNetForward(fiNet* net, const fiPlanes* in0, const fiPlanes* in1, int in_dtype, float* out_f32, uint8_t* out_u8,
                 int N, int H, int W, void* stream) {
    if (!net) return fail(FI_ERR_INVALID, "net is null");
    if (!net->loaded) return fail(FI_ERR_STATE, "fiNetLoadWeights has not been called");
    if (N <= 0 || H <= 0 || W <= 0) return fail(FI_ERR_INVALID, "empty batch or image");
    if (!out_f32 && !out_u8) return fail(FI_ERR_INVALID, "no output buffer");
    if (in_dtype != FI_IN_F32 && in_dtype != FI_IN_U8) return fail(FI_ERR_INVALID, "unknown input dtype");
    int rc = check_planes(net, in0, in1);
    if (rc) return rc;
    ON_DEVICE(net->device);
    if ((rc = build_plan(net, N, H, W))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    Plan& pl = net->plan();
    pl.last_n = N;
    cudaEvent_t* evs = nullptr;
    if (net->profiling) {
        const size_t base = net->prof_events.size();
        net->prof_events.resize(base + 2 * pl.steps.size());
        for (size_t i = base; i < net->prof_events.size(); ++i) CUDA_TRY(cudaEventCreate(&net->prof_events[i]));
        evs = net->prof_events.data() + base;
        ++net->prof_calls;
    }
    struct NvtxScope {  // pops on every exit path (the launch macros return early on errors)
        bool on;
        NvtxScope(bool enable, const char* name) : on(enable) {
            if (on) nvtxRangePushA(name);
        }
        ~NvtxScope() {
            if (on) nvtxRangePop();
        }
    };
    char fwd_name[64];
    if (net->nvtx) snprintf(fwd_name, sizeof fwd_name, "fiNetForward %dx%dx%d", N, H, W);
    NvtxScope fwd_range(net->nvtx, fwd_name);
    for (size_t i = 0; i < pl.steps.size(); ++i) {
        Step& s = pl.steps[i];
        NvtxScope layer_range(net->nvtx, s.name);
        if (evs) CUDA_TRY(cudaEventRecord(evs[2 * i], st));
        if (s.kind == STEP_STEM) {
            fi::StemDesc d;
            memset(&d, 0, sizeof d);
            d.src[0] = to_src(in0);
            d.src[1] = to_src(in1);
            d.is_u8 = in_dtype == FI_IN_U8;
            d.cin = net->n_channels;
            d.N = N;
            d.H = H;
            d.W = W;
            d.wpack = net->stem_w.p;
            d.bias = static_cast<const float*>(net->stem_b.p);
            d.dst = s.dst;
            d.dst_lo = s.dst_lo;
            KERNEL_TRY(fi::stem_conv_launch(d, st));
        } else if (s.kind == STEP_INC_FUSED) {
            fi::StemDesc d;
            memset(&d, 0, sizeof d);
            d.src[0] = to_src(in0);
            d.src[1] = to_src(in1);
            d.is_u8 = in_dtype == FI_IN_U8;
            d.cin = net->n_channels;
            d.N = N;
            d.H = H;
            d.W = W;
            d.wpack = net->stem_w.p;
            d.bias = static_cast<const float*>(net->stem_b.p);
            KERNEL_TRY(fi::inc_fused_launch(d, s.conv, net->inc_bias_host, N, net->num_sms, st));
        } else if (s.kind == STEP_UPSAMPLE) {
            KERNEL_TRY(fi::upsample2x_launch(s.src, s.dst, N, s.h, s.w, s.C, st, s.src_lo, s.dst_lo));
        } else {
            if (static_cast<int>(i) == pl.head_step) {
                s.conv.p.out_f32 = out_f32;
                s.conv.p.out_u8 = out_u8;
            }
            // the plan's arena and tensor maps are sized for pl.N images; this call uses the first N of them
            s.conv.p.n_img = N;
            s.conv.grid = fi::conv_grid(s.conv, net->num_sms);
            KERNEL_TRY(fi::conv_launch(s.conv, st));
        }
        if (evs) CUDA_TRY(cudaEventRecord(evs[2 * i + 1], st));
    }
    return FI_OK;
}

int fiNetSetProfiling(fiNet* net, int enable) {
    if (!net) return fail(FI_ERR_INVALID, "net is null");
    for (cudaEvent_t e : net->prof_events) cudaEventDestroy(e);
    net->prof_events.clear();
    net->prof_calls = 0;
    net->profiling = enable != 0;
    return FI_OK;
}

int fiNetGetProfile(fiNet* net, fiLaunchProfile* out, int capacity, int* count) {
    if (!net || !count) return fail(FI_ERR_INVALID, "null argument");
    if (!net->has_plan()) return fail(FI_ERR_STATE, "no forward has run yet");
    const Plan& pl = net->plan();
    const int n = static_cast<int>(pl.steps.size());
    *count = n;
    if (!out) return FI_OK;
    if (capacity < n) return fail(FI_ERR_INVALID, "profile buffer too small: need %d entries", n);
    if (net->prof_calls == 0 || net->prof_events.size() != static_cast<size_t>(2) * n * net->prof_calls)
        return fail(FI_ERR_STATE, "no profiled forward of the current shape has run");
    ON_DEVICE(net->device);
    int rc = FI_OK;
    CUDA_TRY(cudaDeviceSynchronize());
    for (int i = 0; i < n; ++i) {
        const Step& s = pl.steps[i];
        memset(&out[i], 0, sizeof out[i]);
        snprintf(out[i].name, sizeof out[i].name, "%s", s.name);
        out[i].kind = (s.kind == STEP_CONV || s.kind == STEP_INC_FUSED) ? 1 : (s.kind == STEP_STEM ? 0 : 2);
        out[i].flops = s.flops * pl.last_n;
        out[i].bytes = s.bytes * pl.last_n + s.weight_bytes;
        out[i].calls = net->prof_calls;
        double ms = 0;
        for (int c = 0; c < net->prof_calls; ++c) {
            float t = 0;
            CUDA_TRY(cudaEventElapsedTime(&t, net->prof_events[(static_cast<size_t>(c) * n + i) * 2],
                                          net->prof_events[(static_cast<size_t>(c) * n + i) * 2 + 1]));
            ms += t;
        }
        out[i].ms_total = ms;
    }
    return FI_OK;
}

int fiNetInterpolateHostU8(fiNet* net, const uint8_t* frame1_host, const uint8_t* frame2_host, int channels_per_frame,
                           uint8_t* out_host, int N, int H, int W, void* stream) {
    if (!net || !frame1_host || !frame2_host || !out_host) return fail(FI_ERR_INVALID, "null argument");
    if (2 * channels_per_frame != net->n_channels)
        return fail(FI_ERR_INVALID, "2 x %d channels per frame != n_channels %d", channels_per_frame, net->n_channels);
    if (N <= 0 || H <= 0 || W <= 0) return fail(FI_ERR_INVALID, "empty batch or image");
    ON_DEVICE(net->device);
    int rc = FI_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t frame_bytes = static_cast<size_t>(N) * channels_per_frame * H * W;
    const size_t out_bytes = static_cast<size_t>(N) * net->n_classes * H * W;
    if (net->pin_in_bytes < 2 * frame_bytes) {
        if (net->pin_in) cudaFreeHost(net->pin_in);
        net->pin_in = nullptr;
        net->pin_in_bytes = 0;
        CUDA_TRY(cudaMallocHost(&net->pin_in, 2 * frame_bytes));
        net->pin_in_bytes = 2 * frame_bytes;
        net->dev_in.release();
        CUDA_TRY(cudaMalloc(&net->dev_in.p, 2 * frame_bytes));
        net->dev_in.bytes = 2 * frame_bytes;
    }
    if (net->pin_out_bytes < out_bytes) {
        if (net->pin_out) cudaFreeHost(net->pin_out);
        net->pin_out = nullptr;
        net->pin_out_bytes = 0;
        CUDA_TRY(cudaMallocHost(&net->pin_out, out_bytes));
        net->pin_out_bytes = out_bytes;
        net->dev_out.release();
        CUDA_TRY(cudaMalloc(&net->dev_out.p, out_bytes));
        net->dev_out.bytes = out_bytes;
    }
    memcpy(net->pin_in, frame1_host, frame_bytes);
    memcpy(static_cast<char*>(net->pin_in) + frame_bytes, frame2_host, frame_bytes);
    CUDA_TRY(cudaMemcpyAsync(net->dev_in.p, net->pin_in, 2 * frame_bytes, cudaMemcpyHostToDevice, st));
    fiPlanes p0, p1;
    p0.ptr = net->dev_in.p;
    p0.channels = channels_per_frame;
    p0.px_stride = 1;
    p0.row_stride = W;
    p0.chan_stride = static_cast<int64_t>(H) * W;
    p0.batch_stride = p0.chan_stride * channels_per_frame;
    p1 = p0;
    p1.ptr = static_cast<const uint8_t*>(net->dev_in.p) + frame_bytes;
    rc = fiNetForward(net, &p0, &p1, FI_IN_U8, nullptr, static_cast<uint8_t*>(net->dev_out.p), N, H, W, stream);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(net->pin_out, net->dev_out.p, out_bytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    memcpy(out_host, net->pin_out, out_bytes);
    return FI_OK;
}

int fiNetInterpolateDyadicHostU8(fiNet* net, const uint8_t* frames_host, int64_t frame_stride, int n_frames,
                                 int channels_per_frame, int H, int W, int depth, const int32_t* req_pair_host,
                                 const int32_t* req_num_host, int n_req, uint8_t* out_host, int64_t out_stride,
                                 int pairs_per_batch, void* stream, uint64_t* pair_sad_host, int64_t* n_forwards_host) {
    if (!net) return fail(FI_ERR_INVALID, "net is null");
    if (!frames_host) return fail(FI_ERR_INVALID, "frames_host is null");
    if (n_req < 0) return fail(FI_ERR_INVALID, "n_req %d is negative", n_req);
    if (n_req > 0 && (!req_pair_host || !req_num_host || !out_host))
        return fail(FI_ERR_INVALID, "req_pair_host, req_num_host and out_host are required when n_req > 0");
    if (2 * channels_per_frame != net->n_channels)
        return fail(FI_ERR_INVALID, "2 x %d channels per frame != n_channels %d", channels_per_frame, net->n_channels);
    if (depth < 1 || depth > 6) return fail(FI_ERR_INVALID, "depth %d is outside 1..6", depth);
    if (depth > 1 && net->n_classes != channels_per_frame)
        return fail(FI_ERR_INVALID, "n_classes %d != channels_per_frame %d: below depth 1 bisection feeds nodes back "
                    "into the network", net->n_classes, channels_per_frame);
    if (n_frames < 2) return fail(FI_ERR_INVALID, "n_frames %d: a clip needs at least two frames", n_frames);
    if (H < 16 || W < 16) return fail(FI_ERR_INVALID, "input %dx%d is smaller than 16x16 (4 poolings)", H, W);
    if (pairs_per_batch < 1) return fail(FI_ERR_INVALID, "pairs_per_batch %d < 1", pairs_per_batch);
    // bytes of a frame and of a node (an output of the network); the two are equal wherever a node is fed back
    const size_t fb = static_cast<size_t>(channels_per_frame) * H * W;
    const size_t nodeb = static_cast<size_t>(net->n_classes) * H * W;
    if (frame_stride < static_cast<int64_t>(fb)) return fail(FI_ERR_INVALID, "frame_stride is smaller than a frame");
    if (n_req > 0 && out_stride < static_cast<int64_t>(nodeb))
        return fail(FI_ERR_INVALID, "out_stride is smaller than a node");
    const int n_pairs = n_frames - 1, full = 1 << depth;
    for (int j = 0; j < n_req; ++j) {
        const int p = req_pair_host[j], v = req_num_host[j];
        if (p < 0 || p >= n_pairs) return fail(FI_ERR_INVALID, "req_pair[%d] = %d is outside [0, %d)", j, p, n_pairs);
        if (j > 0 && p < req_pair_host[j - 1])
            return fail(FI_ERR_INVALID, "req_pair is not sorted: req_pair[%d] = %d < req_pair[%d] = %d", j, p, j - 1,
                        req_pair_host[j - 1]);
        if (v <= 0 || v >= full)
            return fail(FI_ERR_INVALID, "req_num[%d] = %d is outside (0, 2^depth = %d)", j, v, full);
    }
    if (!net->loaded) return fail(FI_ERR_STATE, "fiNetLoadWeights has not been called");
    ON_DEVICE(net->device);
    int rc = FI_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int B = pairs_per_batch;

    // A node of local pair q is keyed (q << depth) | v with v in (0, 2^depth) its position in units of 2^-depth; v = 0
    // and v = 2^depth are the uploaded frames q and q+1. Marks the closure of requests [r0, r1) of the group starting at
    // pair `first`: a node at level l (v an odd multiple of 2^(depth-l)) needs its parents v -/+ 2^(depth-l).
    std::vector<uint8_t> need;
    std::vector<int> stack;
    auto closure = [&](int first, int cnt, int r0, int r1) {
        need.assign(static_cast<size_t>(cnt) << depth, 0);
        int nodes = 0;
        for (int r = r0; r < r1; ++r) stack.push_back(((req_pair_host[r] - first) << depth) | req_num_host[r]);
        while (!stack.empty()) {
            const int key = stack.back(), v = key & (full - 1), low = v & -v;
            stack.pop_back();
            if (need[key]) continue;
            need[key] = 1;
            ++nodes;
            if (v - low > 0) stack.push_back(key - low);
            if (v + low < full) stack.push_back(key + low);
        }
        return nodes;
    };
    struct Group {
        int first, cnt, r0, r1;
    };
    std::vector<Group> groups;  // groups of B pairs that have requests (all of them when the SAD is asked for)
    size_t max_nodes = 0, max_req = 0;
    bool gather = false;  // a forward gathers its parents: a node below level 1, or midpoints of non-consecutive pairs
    for (int first = 0, r = 0; first < n_pairs; first += B) {
        Group g{first, std::min(B, n_pairs - first), r, r};
        while (r < n_req && req_pair_host[r] < first + g.cnt) ++r;
        g.r1 = r;
        if (g.r0 == g.r1 && !pair_sad_host) continue;
        groups.push_back(g);
        const int nodes = closure(g.first, g.cnt, g.r0, g.r1);
        bool direct = nodes == 0 || req_pair_host[g.r1 - 1] - req_pair_host[g.r0] + 1 == nodes;
        for (int j = g.r0; j < g.r1 && direct; ++j) direct = req_num_host[j] == full / 2;
        gather = gather || !direct;
        max_nodes = std::max(max_nodes, static_cast<size_t>(nodes));
        max_req = std::max(max_req, static_cast<size_t>(g.r1 - g.r0));
    }
    if (groups.empty()) {
        if (n_forwards_host) *n_forwards_host = 0;
        return FI_OK;
    }
    if ((rc = clip_staging(net, B, (B + 1) * fb, pair_sad_host != nullptr))) return rc;
    const size_t gather_bytes = gather ? 2 * B * fb : 0, pool_bytes = max_nodes * nodeb, nodes_bytes = max_req * nodeb;
    bool grow = net->dyadic_gather.bytes < gather_bytes;
    for (auto& c : net->clip) grow = grow || c.pool.bytes < pool_bytes || c.pin_nodes_bytes < nodes_bytes;
    if (grow) {
        CUDA_TRY(cudaDeviceSynchronize());
        auto grow_dev = [](DevBuf& d, size_t bytes) {
            if (d.bytes >= bytes) return cudaSuccess;
            d.release();
            const cudaError_t e = cudaMalloc(&d.p, bytes);
            if (e == cudaSuccess) d.bytes = bytes;
            return e;
        };
        CUDA_TRY(grow_dev(net->dyadic_gather, gather_bytes));
        for (auto& c : net->clip) {
            CUDA_TRY(grow_dev(c.pool, pool_bytes));
            if (c.pin_nodes_bytes < nodes_bytes) {
                if (c.pin_nodes) cudaFreeHost(c.pin_nodes);
                c.pin_nodes = nullptr;
                c.pin_nodes_bytes = 0;
                CUDA_TRY(cudaMallocHost(&c.pin_nodes, nodes_bytes));
                c.pin_nodes_bytes = nodes_bytes;
            }
        }
    }
    // one plan serves every level's batches: none has more than B images or more than a group's nodes
    if (max_nodes > 0 && (rc = build_plan(net, static_cast<int>(std::min(static_cast<size_t>(B), max_nodes)), H, W)))
        return rc;

    auto collect = [&](size_t b) -> int {  // wait for group b's D2H and hand its requested nodes to the caller
        const Group& g = groups[b];
        fiNet::ClipSlot& c = net->clip[b & 1];
        CUDA_TRY(cudaEventSynchronize(c.out_ready));
        for (int r = g.r0; r < g.r1; ++r)
            memcpy(out_host + static_cast<int64_t>(r) * out_stride,
                   static_cast<const char*>(c.pin_nodes) + (r - g.r0) * nodeb, nodeb);
        if (pair_sad_host) memcpy(pair_sad_host + g.first, c.pin_sad, g.cnt * sizeof(uint64_t));
        return FI_OK;
    };
    uint8_t* const in0 = static_cast<uint8_t*>(net->dyadic_gather.p);
    uint8_t* const in1 = in0 + B * fb;
    const fiPlanes p0 = u8_planes(in0, channels_per_frame, H, W, fb);
    const fiPlanes p1 = u8_planes(in1, channels_per_frame, H, W, fb);
    std::vector<int> slot, todo;  // pool index of each needed node; the nodes of one level
    int64_t forwards = 0;
    for (size_t b = 0; b < groups.size(); ++b) {
        const Group& g = groups[b];
        fiNet::ClipSlot& c = net->clip[b & 1];
        // slot reuse is safe: group b-2 was collected (host-synchronised) in iteration b-1
        if (frame_stride == static_cast<int64_t>(fb)) {
            memcpy(c.pin_in, frames_host + static_cast<size_t>(g.first) * fb, (g.cnt + 1) * fb);
        } else {
            for (int i = 0; i <= g.cnt; ++i)
                memcpy(static_cast<char*>(c.pin_in) + i * fb, frames_host + static_cast<int64_t>(g.first + i) * frame_stride,
                       fb);
        }
        CUDA_TRY(cudaMemcpyAsync(c.dev_in, c.pin_in, (g.cnt + 1) * fb, cudaMemcpyHostToDevice, net->clip_h2d));
        CUDA_TRY(cudaEventRecord(c.in_ready, net->clip_h2d));
        CUDA_TRY(cudaStreamWaitEvent(st, c.in_ready, 0));
        if (pair_sad_host)
            KERNEL_TRY(fi::pair_sad_launch(static_cast<const uint8_t*>(c.dev_in), static_cast<int64_t>(fb),
                                           static_cast<int64_t>(fb), g.cnt + 1, c.dev_sad, st));
        closure(g.first, g.cnt, g.r0, g.r1);
        slot.assign(need.size(), -1);
        const uint8_t* frames_dev = static_cast<const uint8_t*>(c.dev_in);
        uint8_t* pool = static_cast<uint8_t*>(c.pool.p);
        auto node = [&](int q, int v) -> const uint8_t* {
            if (v == 0) return frames_dev + q * fb;
            if (v == full) return frames_dev + (q + 1) * fb;
            return pool + slot[(q << depth) | v] * nodeb;
        };
        int next = 0;  // pool slots in evaluation order, so that each forward's outputs are contiguous
        for (int level = 1; level <= depth; ++level) {
            const int half = 1 << (depth - level);  // a level-l node sits half-way between its parents
            todo.clear();
            for (int q = 0; q < g.cnt; ++q)
                for (int v = half; v < full; v += 2 * half)
                    if (need[(q << depth) | v]) todo.push_back((q << depth) | v);
            for (size_t k0 = 0; k0 < todo.size(); k0 += B) {
                const int nb = static_cast<int>(std::min(todo.size() - k0, static_cast<size_t>(B)));
                // the midpoints of consecutive pairs q0 .. q0+nb-1 read their parents where they were uploaded; any
                // other batch gathers them into in0 | in1
                const int q0 = todo[k0] >> depth;
                const bool direct = level == 1 && (todo[k0 + nb - 1] >> depth) - q0 == nb - 1;
                for (int k = 0; k < nb; ++k) {
                    const int key = todo[k0 + k], q = key >> depth, v = key & (full - 1);
                    if (!direct) {
                        CUDA_TRY(cudaMemcpyAsync(in0 + k * fb, node(q, v - half), fb, cudaMemcpyDeviceToDevice, st));
                        CUDA_TRY(cudaMemcpyAsync(in1 + k * fb, node(q, v + half), fb, cudaMemcpyDeviceToDevice, st));
                    }
                    slot[key] = next + k;
                }
                const fiPlanes d0 = u8_planes(frames_dev + q0 * fb, channels_per_frame, H, W, fb);
                const fiPlanes d1 = u8_planes(frames_dev + (q0 + 1) * fb, channels_per_frame, H, W, fb);
                rc = fiNetForward(net, direct ? &d0 : &p0, direct ? &d1 : &p1, FI_IN_U8, nullptr, pool + next * nodeb,
                                  nb, H, W, stream);
                if (rc) return rc;
                next += nb;
            }
        }
        forwards += next;
        CUDA_TRY(cudaEventRecord(c.done, st));
        CUDA_TRY(cudaStreamWaitEvent(net->clip_d2h, c.done, 0));
        for (int r = g.r0; r < g.r1;) {  // requested nodes, runs of consecutive pool slots in one copy
            const int s = slot[((req_pair_host[r] - g.first) << depth) | req_num_host[r]];
            int e = r + 1;
            while (e < g.r1 && slot[((req_pair_host[e] - g.first) << depth) | req_num_host[e]] == s + (e - r)) ++e;
            CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(c.pin_nodes) + (r - g.r0) * nodeb, pool + s * nodeb,
                                     (e - r) * nodeb, cudaMemcpyDeviceToHost, net->clip_d2h));
            r = e;
        }
        if (pair_sad_host)
            CUDA_TRY(cudaMemcpyAsync(c.pin_sad, c.dev_sad, g.cnt * sizeof(uint64_t), cudaMemcpyDeviceToHost, net->clip_d2h));
        CUDA_TRY(cudaEventRecord(c.out_ready, net->clip_d2h));
        if (b > 0 && (rc = collect(b - 1))) return rc;
    }
    if ((rc = collect(groups.size() - 1))) return rc;
    if (n_forwards_host) *n_forwards_host = forwards;
    return FI_OK;
}

int fiNetForwardCost(fiNet* net, int N, int H, int W, double* flops, int* launches) {
    if (!net) return fail(FI_ERR_INVALID, "net is null");
    if (!net->loaded) return fail(FI_ERR_STATE, "fiNetLoadWeights has not been called");
    ON_DEVICE(net->device);
    int rc = FI_OK;
    if ((rc = build_plan(net, N, H, W))) return rc;
    if (flops) *flops = net->plan().flops * N;
    if (launches) *launches = static_cast<int>(net->plan().steps.size());
    return FI_OK;
}

int fiNetPlanStats(fiNet* net, int* cached, long long* builds, size_t* arena_bytes) {
    if (!net) return fail(FI_ERR_INVALID, "net is null");
    if (cached) *cached = static_cast<int>(net->plans.size());
    if (builds) *builds = net->plan_builds;
    if (arena_bytes) {
        size_t total = 0;
        for (const Plan& p : net->plans) total += p.arena.bytes;
        *arena_bytes = total;
    }
    return FI_OK;
}

int fiNetReadActivation(fiNet* net, const char* name, float* out_host, int64_t capacity, int* C, int* H, int* W) {
    if (!net || !name || !out_host) return fail(FI_ERR_INVALID, "null argument");
    if (!net->has_plan()) return fail(FI_ERR_INVALID, "no activation named '%s': no forward has run yet", name);
    Plan& pl = net->plan();
    auto it = pl.acts.find(name);
    if (!pl.arena.p || it == pl.acts.end()) return fail(FI_ERR_INVALID, "no activation named '%s' in the current plan", name);
    if (pl.reuse)
        return fail(FI_ERR_STATE, "activation taps are unavailable: this plan's arena re-uses the memory of dead tensors "
                                  "(FI_ARENA_REUSE=0 keeps every tensor)");
    const Act& a = it->second;
    const int64_t n = static_cast<int64_t>(pl.last_n) * a.C * a.H * a.W;
    if (capacity < n) return fail(FI_ERR_INVALID, "buffer too small: need %lld floats", static_cast<long long>(n));
    ON_DEVICE(net->device);
    int rc = FI_OK;
    std::vector<uint16_t> raw(static_cast<size_t>(n)), raw_lo;
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(raw.data(), static_cast<char*>(pl.arena.p) + a.off, raw.size() * 2, cudaMemcpyDeviceToHost));
    if (net->precise) {
        raw_lo.resize(raw.size());
        CUDA_TRY(cudaMemcpy(raw_lo.data(), static_cast<char*>(pl.arena.p) + a.off_lo, raw.size() * 2,
                            cudaMemcpyDeviceToHost));
    }
    for (int nn = 0; nn < pl.last_n; ++nn)
        for (int y = 0; y < a.H; ++y)
            for (int c = 0; c < a.C; ++c)       // row-blocked transpose: one NHWC row stays in cache, NCHW writes are contiguous
                for (int x = 0; x < a.W; ++x) {
                    const size_t src_i = ((static_cast<size_t>(nn) * a.H + y) * a.W + x) * a.C + c;
                    const uint32_t bits = static_cast<uint32_t>(raw[src_i]) << 16;
                    float f;
                    memcpy(&f, &bits, 4);
                    if (net->precise) {
                        const uint32_t lb = static_cast<uint32_t>(raw_lo[src_i]) << 16;
                        float fl;
                        memcpy(&fl, &lb, 4);
                        f += fl;
                    }
                    out_host[((static_cast<size_t>(nn) * a.C + c) * a.H + y) * a.W + x] = f;
                }
    if (C) *C = a.C;
    if (H) *H = a.H;
    if (W) *W = a.W;
    return FI_OK;
}

int fiNetCopyActivation(fiNet* net, const char* name, void* dst, void* dst_lo, int64_t capacity_elems, int* C, int* H,
                        int* W, void* stream) {
    if (!net || !name) return fail(FI_ERR_INVALID, "null argument");
    if (!net->has_plan()) return fail(FI_ERR_INVALID, "no activation named '%s': no forward has run yet", name);
    Plan& pl = net->plan();
    auto it = pl.acts.find(name);
    if (!pl.arena.p || it == pl.acts.end()) return fail(FI_ERR_INVALID, "no activation named '%s' in the current plan", name);
    if (pl.reuse)
        return fail(FI_ERR_STATE, "activation taps are unavailable: this plan's arena re-uses the memory of dead tensors "
                                  "(FI_ARENA_REUSE=0 keeps every tensor)");
    const Act& a = it->second;
    if (C) *C = a.C;
    if (H) *H = a.H;
    if (W) *W = a.W;
    if (!dst) return FI_OK;  // shape query
    if (net->precise && !dst_lo) return fail(FI_ERR_INVALID, "fp32-grade mode: dst_lo is required for the lo half");
    const int64_t n = static_cast<int64_t>(pl.last_n) * a.C * a.H * a.W;
    if (capacity_elems < n) return fail(FI_ERR_INVALID, "buffer too small: need %lld elements", static_cast<long long>(n));
    ON_DEVICE(net->device);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    CUDA_TRY(cudaMemcpyAsync(dst, static_cast<char*>(pl.arena.p) + a.off, static_cast<size_t>(n) * 2,
                             cudaMemcpyDeviceToDevice, st));
    if (net->precise)
        CUDA_TRY(cudaMemcpyAsync(dst_lo, static_cast<char*>(pl.arena.p) + a.off_lo, static_cast<size_t>(n) * 2,
                                 cudaMemcpyDeviceToDevice, st));
    return FI_OK;
}

int fiConvGemm(const fiConvDesc* desc, void* stream) {
    if (!desc) return fail(FI_ERR_INVALID, "desc is null");
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    int sms = 0;
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    fi::ConvDesc d;
    memset(&d, 0, sizeof d);
    d.src0 = desc->src0;
    d.c0 = desc->c0;
    d.src1 = desc->src1;
    d.c1 = desc->c1;
    d.h1 = desc->h1;
    d.w1 = desc->w1;
    d.off_y = desc->off_y;
    d.off_x = desc->off_x;
    d.wpack = desc->wpack;
    d.bias = desc->bias;
    d.n_total = desc->n_total;
    d.taps = desc->taps;
    d.mode = desc->mode;
    d.relu = desc->relu;
    d.dst = desc->dst;
    d.dst_pool = desc->dst_pool;
    d.head_w = desc->head_w;
    d.head_b = desc->head_b;
    d.n_classes = desc->n_classes;
    d.out_f32 = desc->out_f32;
    d.out_u8 = desc->out_u8;
    d.N = desc->N;
    d.H = desc->H;
    d.W = desc->W;
    d.precise = desc->precise;
    d.src0_lo = desc->src0_lo;
    d.src1_lo = desc->src1_lo;
    d.dst_lo = desc->dst_lo;
    d.dst_pool_lo = desc->dst_pool_lo;
    fi::ConvLaunch l;
    const char* e = fi::conv_prepare(d, sms, &l);
    if (e) return fail(FI_ERR_INVALID, "%s", e);
    KERNEL_TRY(fi::conv_launch(l, static_cast<cudaStream_t>(stream)));
    return FI_OK;
}

int fiStemPackedK(int cin) { return cin >= 1 && cin <= 8 ? fi::stem_packed_k(cin) : 0; }

int fiStemPackWeights(const float* w_host, int cin, uint16_t* out_host) {
    if (!w_host || !out_host) return fail(FI_ERR_INVALID, "null argument");
    if (cin < 1 || cin > 8) return fail(FI_ERR_INVALID, "stem: 1..8 input channels supported");
    fi::stem_pack_weights(w_host, cin, out_host);
    return FI_OK;
}

static int stem_conv_impl(const fiPlanes* in0, const fiPlanes* in1, int in_dtype, const void* wpack, const float* bias,
                          void* dst, int N, int H, int W, void* stream, int linear);

int fiStemConv(const fiPlanes* in0, const fiPlanes* in1, int in_dtype, const void* wpack, const float* bias, void* dst,
               int N, int H, int W, void* stream) {
    return stem_conv_impl(in0, in1, in_dtype, wpack, bias, dst, N, H, W, stream, 0);
}

int fiStemConvLinear(const fiPlanes* in0, const fiPlanes* in1, int in_dtype, const void* wpack, const float* bias,
                     void* dst, int N, int H, int W, void* stream) {
    return stem_conv_impl(in0, in1, in_dtype, wpack, bias, dst, N, H, W, stream, 1);
}

static int stem_conv_impl(const fiPlanes* in0, const fiPlanes* in1, int in_dtype, const void* wpack, const float* bias,
                          void* dst, int N, int H, int W, void* stream, int linear) {
    if (!in0 || !wpack || !bias || !dst) return fail(FI_ERR_INVALID, "null argument");
    fi::StemDesc d;
    memset(&d, 0, sizeof d);
    d.src[0] = to_src(in0);
    d.src[1] = to_src(in1);
    d.is_u8 = in_dtype == FI_IN_U8;
    d.cin = in0->channels + (in1 ? in1->channels : 0);
    d.N = N;
    d.H = H;
    d.W = W;
    d.wpack = wpack;
    d.linear = linear;
    d.bias = bias;
    d.dst = dst;
    const char* e = fi::stem_conv_launch(d, static_cast<cudaStream_t>(stream));
    if (e) return fail(FI_ERR_INVALID, "%s", e);
    return FI_OK;
}

int fiUpsample2x(const void* src, void* dst, int N, int h, int w, int C, void* stream) {
    if (!src || !dst) return fail(FI_ERR_INVALID, "null argument");
    const char* e = fi::upsample2x_launch(src, dst, N, h, w, C, static_cast<cudaStream_t>(stream));
    if (e) return fail(FI_ERR_INVALID, "%s", e);
    return FI_OK;
}

int fiMaxPool2x2(const void* src, void* dst, int N, int H, int W, int C, void* stream) {
    if (!src || !dst) return fail(FI_ERR_INVALID, "null argument");
    const char* e = fi::maxpool2x2_launch(src, dst, N, H, W, C, static_cast<cudaStream_t>(stream));
    if (e) return fail(FI_ERR_INVALID, "%s", e);
    return FI_OK;
}

int fiPackPairU8(const uint8_t* frame1, const uint8_t* frame2, float* out, int N, int C, int H, int W, void* stream) {
    if (!frame1 || !frame2 || !out) return fail(FI_ERR_INVALID, "null argument");
    const char* e = fi::pack_pair_launch(frame1, frame2, out, N, C, H, W, static_cast<cudaStream_t>(stream));
    if (e) return fail(FI_ERR_INVALID, "%s", e);
    return FI_OK;
}

int fiHeadPostU8(const float* logits, uint8_t* out, size_t n, void* stream) {
    if (n && (!logits || !out)) return fail(FI_ERR_INVALID, "null argument");
    const char* e = fi::head_post_launch(logits, out, n, static_cast<cudaStream_t>(stream));
    if (e) return fail(FI_ERR_INVALID, "%s", e);
    return FI_OK;
}

size_t fiSsimPsnrWorkspaceBytes(int N, int H, int W) {
    if (N <= 0 || H <= 0 || W <= 0) return 0;
    return fi::ssim_psnr_workspace_bytes(N, H, W);
}

int fiSsimPsnrU8(const uint8_t* pred, const uint8_t* target, int N, int H, int W, double* out, void* workspace,
                 void* stream) {
    const char* e = fi::ssim_psnr_launch(pred, target, N, H, W, out, workspace, static_cast<cudaStream_t>(stream));
    if (e) return fail(FI_ERR_INVALID, "%s", e);
    return FI_OK;
}

int fiPairSadU8(const uint8_t* frames, int64_t frame_stride, int64_t frame_bytes, int n_frames, uint64_t* sad,
                void* stream) {
    if (!frames || !sad) return fail(FI_ERR_INVALID, "null argument");
    if (n_frames < 2 || frame_bytes < 1 || frame_stride < frame_bytes)
        return fail(FI_ERR_INVALID, "needs >= 2 frames of >= 1 byte and frame_stride >= frame_bytes");
    const char* e = fi::pair_sad_launch(frames, frame_stride, frame_bytes, n_frames, sad, static_cast<cudaStream_t>(stream));
    if (e) return fail(FI_ERR_CUDA, "%s", e);
    return FI_OK;
}

int fiGatherTripletsU8(const uint8_t* frames, int64_t n_frames, const int32_t* triplets, int64_t n_triplets,
                       const int64_t* samples, int n, int H, int W, float* frame1, float* frame2, float* target,
                       void* stream) {
    if (!frames || !triplets || !samples || !frame1 || !frame2 || !target) return fail(FI_ERR_INVALID, "null argument");
    if (n < 1 || H < 1 || W < 1) return fail(FI_ERR_INVALID, "needs n, H and W >= 1 (got %d, %d, %d)", n, H, W);
    if (n_frames < 0 || n_triplets < 0) return fail(FI_ERR_INVALID, "negative frame or triplet count");
    const char* e = fi::gather_triplets_u8_launch(frames, n_frames, triplets, n_triplets, samples, n, H, W, frame1,
                                                  frame2, target, static_cast<cudaStream_t>(stream));
    if (e) return fail(FI_ERR_CUDA, "%s", e);
    return FI_OK;
}


// ---------------------------------------------------------------------------------------------- training-step kernels
#define TRAIN_CALL(expr)                                        \
    do {                                                        \
        const char* _m = (expr);                                \
        if (_m) return fail(FI_ERR_INVALID, "%s", _m);          \
        return FI_OK;                                           \
    } while (0)
#define ST static_cast<cudaStream_t>(stream)

int fiBnStats(const void* z, int64_t P, int C, float* sum, float* sumsq, void* stream) {
    TRAIN_CALL(fi::bn_stats_launch(z, P, C, sum, sumsq, nullptr, ST));
}
int fiBnStatsShifted(const void* z, int64_t P, int C, float* pivot, float* sum, float* sumsq, void* stream) {
    if (!pivot) return fail(FI_ERR_INVALID, "bn_stats: null pivot");
    TRAIN_CALL(fi::bn_stats_launch(z, P, C, sum, sumsq, pivot, ST));
}
int fiBnApplyRelu(const void* z, int64_t P, int C, const float* scale, const float* shift, void* a, void* stream) {
    TRAIN_CALL(fi::bn_apply_relu_launch(z, P, C, scale, shift, a, ST));
}
int fiHeadForward(const void* a, int N, int64_t HW, const float* w, const float* b, int n_classes, float* y, void* stream) {
    TRAIN_CALL(fi::head_forward_launch(a, N, HW, w, b, n_classes, y, ST));
}
int fiMseLossGrad(const float* y, const float* target, int64_t n, float* loss, float* dy, void* stream) {
    TRAIN_CALL(fi::mse_launch(y, target, n, loss, dy, ST));
}
int fiCombinedLossGrad(const float* y, const float* target, int planes, int H, int W, float mse_weight, float ssim_weight,
                       float* loss, float* dy, void* stream) {
    TRAIN_CALL(fi::combined_loss_launch(y, target, planes, H, W, mse_weight, ssim_weight, loss, dy, ST));
}
int fiHeadBackward(const void* a, const float* dy, int N, int64_t HW, const float* w, int n_classes, void* da, float* dw,
                   float* db, void* stream) {
    TRAIN_CALL(fi::head_backward_launch(a, dy, N, HW, w, n_classes, da, dw, db, ST));
}
int fiBnReluBackwardReduce(const void* dA, const void* z, int64_t P, int C, const float* mean, const float* rstd,
                           const float* scale, const float* shift, float* dbeta, float* dgamma, void* stream) {
    TRAIN_CALL(fi::bn_relu_bwd_reduce_launch(dA, z, P, C, mean, rstd, scale, shift, dbeta, dgamma, ST));
}
int fiBnReluBackwardApply(const void* dA, const void* z, int64_t P, int C, const float* mean, const float* rstd,
                          const float* gamma, const float* beta, const float* dbeta, const float* dgamma, void* dz,
                          void* stream) {
    TRAIN_CALL(fi::bn_relu_bwd_apply_launch(dA, z, P, C, mean, rstd, gamma, beta, dbeta, dgamma, dz, ST));
}
int fiMaxPoolBackwardAdd(const void* a_full, const void* a_pool, const void* d_pool, const void* d_skip, void* d_full,
                         int N, int H, int W, int C, void* stream) {
    TRAIN_CALL(fi::maxpool_bwd_add_launch(a_full, a_pool, d_pool, d_skip, d_full, N, H, W, C, ST));
}
int fiUpsample2xBackward(const void* d_up, void* d_lo, int N, int h, int w, int C, void* stream) {
    TRAIN_CALL(fi::upsample2x_bwd_launch(d_up, d_lo, N, h, w, C, ST));
}
int fiStemWgrad(const void* dz, const float* x, int N, int H, int W, int cin, float* dW, void* stream) {
    TRAIN_CALL(fi::stem_wgrad_launch(dz, x, N, H, W, cin, dW, ST));
}
int fiWgrad(const void* dz, const void* x0, int c0, const void* x1, int c1, int N, int H, int W, int cout, float* dW,
            void* stream) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    TRAIN_CALL(fi::wgrad_launch(dz, x0, c0, x1, c1, N, H, W, cout, dW, sms, ST));
}
int fiWgradPointwise(const void* dz, const void* x, int cin, int N, int H, int W, int cout, float* dW, void* stream) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    TRAIN_CALL(fi::wgrad_launch(dz, x, cin, nullptr, 0, N, H, W, cout, dW, sms, ST, 1));
}
int fiBnFinalize(const float* sum, const float* sumsq, int C, int64_t P, float eps, float momentum, const float* gamma,
                 const float* beta, float* mean, float* rstd, float* scale, float* shift, float* running_mean,
                 float* running_var, void* stream) {
    TRAIN_CALL(fi::bn_finalize_launch(sum, sumsq, nullptr, C, P, eps, momentum, gamma, beta, mean, rstd, scale, shift,
                                      running_mean, running_var, ST));
}
int fiBnFinalizeShifted(const float* sum, const float* sumsq, const float* pivot, int C, int64_t P, float eps,
                        float momentum, const float* gamma, const float* beta, float* mean, float* rstd, float* scale,
                        float* shift, float* running_mean, float* running_var, void* stream) {
    if (!pivot) return fail(FI_ERR_INVALID, "bn_finalize: null pivot");
    TRAIN_CALL(fi::bn_finalize_launch(sum, sumsq, pivot, C, P, eps, momentum, gamma, beta, mean, rstd, scale, shift, running_mean,
                                      running_var, ST));
}
int fiUnpackConvGrad(const float* dW, int cout, int cin, float* grad, void* stream) {
    TRAIN_CALL(fi::unpack_conv_grad_launch(dW, cout, cin, grad, ST));
}
int fiAdamStep(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
               int step, const float* hyper_dev, void* stream) {
    TRAIN_CALL(fi::adam_launch(p, g, m, v, n, lr, beta1, beta2, eps, step, hyper_dev, ST));
}
int fiStemPackWeightsDevice(const float* w_dev, int cin, void* packed_dev, void* stream) {
    TRAIN_CALL(fi::stem_pack_device_launch(w_dev, cin, packed_dev, ST));
}
int fiPackConvWeights(const float* w, int cout, int cin, void* fwd, void* bwd, void* stream) {
    TRAIN_CALL(fi::pack_conv_launch(w, cout, cin, fwd, bwd, ST));
}
#undef ST
#undef TRAIN_CALL

}  // extern "C"
