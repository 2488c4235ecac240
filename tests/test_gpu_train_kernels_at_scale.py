"""The training-step kernels at the shapes TrainStep launches (batch 16 x 256^2), against plain float64 torch references
computed on the GPU from the same bf16-rounded operands the kernels read.

At batch 16 x 256^2 a per-channel reduction walks P = 1 048 576 pixels: the unrolled grid-stride loops run many trips
and end in tails, the grids hit their caps and hundreds of blocks combine through atomics. The small cases of
test_gpu_train_kernels.py run one trip on one or two blocks. The shapes here are read from TrainStep itself:
`record_train_step` wraps the library's entry points for the duration of one step, and
`test_every_recorded_configuration_has_a_row` fails when a configuration the step launches has no row in the tables
below, so these tests follow the step when its layers change.

Bars:
- bf16 outputs: 1 bf16 ulp, |got - ref| <= 2^-7 |ref| + a small absolute term;
- fp32 reductions: |got - ref| <= 1e-4 |ref| + 1e-5 sum|terms|. The second term is there because the rounding error of
  a signed sum scales with the sum of the magnitudes of its terms, not with the (possibly cancelling) result.
"""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from model import _engine as E

pytestmark = pytest.mark.gpu

N_B, SIZE = 16, 256                     # the training batch: 16 frame triplets at 256 x 256
P0 = N_B * SIZE * SIZE                  # pixels of a full-resolution layer
ULP = 2.0 ** -7
EPS = 1e-5                              # nn.BatchNorm2d default
MOMENTUM = 0.1                          # model/train.py BN_MOMENTUM


def p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def st():
    return E.current_stream()


def bf16_close(got, ref, what, abs_frac=1e-4, abs_min=0.0):
    """1 bf16 ulp per element, plus abs_frac of the largest reference value of the element's channel (the last
    dimension; fp32 noise next to zero) and abs_min."""
    got, ref = got.double(), ref.double()
    assert not torch.isnan(got).any(), f"{what}: NaN"
    tol = ULP * ref.abs() + abs_frac * ref.abs().reshape(-1, ref.shape[-1]).amax(0) + abs_min
    err = (got - ref).abs()
    bad = err > tol
    ratio = (err / tol.clamp_min(1e-30)).max().item()
    assert not bad.any(), f"{what}: {int(bad.sum())}/{bad.numel()} beyond 1 bf16 ulp, max err {err.max().item():.4g}, " \
                          f"max err/bar {ratio:.3g}"
    return ratio


def sum_close(got, ref, mag, what, rtol=1e-4, ktol=1e-5):
    """fp32 reduction against fp64: |got - ref| <= rtol |ref| + ktol * mag, mag = sum of |terms| per element."""
    got, ref, mag = got.double(), ref.double(), mag.double()
    tol = rtol * ref.abs() + ktol * mag
    err = (got - ref).abs()
    ratio = (err / tol.clamp_min(1e-30)).max().item()
    assert (err <= tol).all(), f"{what}: max err {err.max().item():.4g}, max err/bar {ratio:.3g}"
    return ratio


# ------------------------------------------------------------------------------------------------ shapes of TrainStep
def _v(x):
    return x.value if hasattr(x, "value") else x


def _gemm_key(a):
    d = a[0]._obj
    if d.taps == 1 and d.mode == E.EPI_STORE:     # the ConvTranspose2d data gradient; 3x3 convs: test_gpu_conv_layers
        return ("convt_dgrad", d.N, d.H, d.W, d.c0, d.n_total)
    return None


# entry point -> key of the configuration it was called with (None: covered by other test files)
_KEYS = {
    "fiBnStatsShifted": lambda a: ("bn", _v(a[1]), _v(a[2])),
    "fiBnFinalizeShifted": lambda a: ("bn", _v(a[4]), _v(a[3])),
    "fiBnApplyRelu": lambda a: ("bn", _v(a[1]), _v(a[2])),
    "fiBnReluBackwardReduce": lambda a: ("bn", _v(a[2]), _v(a[3])),
    "fiBnReluBackwardApply": lambda a: ("bn", _v(a[2]), _v(a[3])),
    "fiBnStats": lambda a: ("bias_sum", _v(a[1]), _v(a[2])),
    "fiConvGemm": _gemm_key,
    "fiWgradPointwise": lambda a: ("wgrad_pw", _v(a[3]), _v(a[4]), _v(a[5]), _v(a[2]), _v(a[6])),
    "fiStemConvLinear": lambda a: ("stem", a[0]._obj.channels + (a[1]._obj.channels if a[1] is not None else 0),
                                   _v(a[6]), _v(a[7]), _v(a[8])),
    "fiStemPackWeightsDevice": lambda a: ("stem_pack", _v(a[1])),
    "fiStemWgrad": lambda a: ("stem_wgrad", _v(a[5]), _v(a[2]), _v(a[3]), _v(a[4])),
    "fiHeadForward": lambda a: ("head", _v(a[1]) * _v(a[2]), _v(a[5])),
    "fiHeadBackward": lambda a: ("head", _v(a[2]) * _v(a[3]), _v(a[5])),
    "fiMseLossGrad": lambda a: ("mse", _v(a[2])),
    "fiCombinedLossGrad": lambda a: ("combined", _v(a[2]), _v(a[3]), _v(a[4])),
    "fiMaxPoolBackwardAdd": lambda a: ("maxpool_bwd", _v(a[5]), _v(a[6]), _v(a[7]), _v(a[8])),
    "fiUpsample2xBackward": lambda a: ("upsample_bwd", _v(a[2]), _v(a[3]), _v(a[4]), _v(a[5])),
}


def record_train_step(model, n=N_B, size=SIZE):
    """Configurations of the entry points in _KEYS that one TrainStep call on `model` launches."""
    from model.train import TrainStep
    lib, seen, saved = E.lib(), set(), {}
    dev = next(model.parameters()).device
    cin, ncls = model.inc.double_conv[0].in_channels, model.outc.conv.out_channels
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.rand(n, cin, size, size, generator=g, device=dev) * 2 - 1
    tgt = torch.rand(n, ncls, size, size, generator=g, device=dev)
    for name, key in _KEYS.items():
        fn = saved[name] = getattr(lib, name)

        def wrapped(*a, _fn=fn, _key=key):
            k = _key(a)
            if k is not None:
                seen.add(k)
            return _fn(*a)
        setattr(lib, name, wrapped)
    try:
        TrainStep(model, lr=0.0)(x, None, tgt)
        torch.cuda.synchronize()
    finally:
        for name, fn in saved.items():
            setattr(lib, name, fn)
    return seen


L = [P0 >> (2 * k) for k in range(5)]   # pixels per level: 1 048 576, 262 144, 65 536, 16 384, 4 096

# (P, C) of every BatchNorm layer of the three networks, then the edges of the reduction walk
BN_ROWS = [(L[0], 64), (L[1], 128), (L[2], 256), (L[3], 512), (L[4], 1024),    # ConvT nets
           (L[4], 512), (L[3], 256), (L[2], 128), (L[1], 64)]                   # bilinear decoder (factor 2)
BN_EDGE_ROWS = [(L[1] + 5, 192),        # C/8 = 24 does not divide 256: one pixel lane per block
                (L[4] * 4 + 3, 2048),   # RED_MAX_C: c8 = 256, one lane, no shared-memory combine; tails in both loops
                (L[0] + 7, 64),         # 4-way / 3-way unrolled walks end in a tail at the grid cap
                (L[3] + 1, 1024)]
# ConvTranspose2d levels (N, h, w, Cin, Cout): data-gradient GEMM c0 = 4 Cout -> n_total = Cin, pointwise wgrad
CONVT_ROWS = [(N_B, 16, 16, 1024, 512), (N_B, 32, 32, 512, 256), (N_B, 64, 64, 256, 128), (N_B, 128, 128, 128, 64)]
CONVT_RAGGED = [(2, 9, 13, 1024, 512), (3, 7, 20, 512, 256), (2, 11, 9, 256, 128), (1, 13, 17, 128, 64)]
STEM_ROWS = [(cin, N_B, SIZE, SIZE) for cin in (1, 2, 3, 6, 8)]
STEM_WGRAD_ROWS = [(cin, N_B, SIZE, SIZE) for cin in (1, 2, 3, 4, 6)] + [(cin, 4, 64, 200) for cin in (1, 2, 3, 4, 6)]
HEAD_ROWS = [(P0, k) for k in (1, 2, 3, 4)] + [(3 * 37 * 41, k) for k in (1, 2, 3, 4)]
MAXPOOL_ROWS = [(N_B, 256, 256, 64), (N_B, 128, 128, 128), (N_B, 64, 64, 256), (N_B, 32, 32, 512),
                (2, 33, 35, 64), (1, 17, 9, 128), (3, 5, 7, 256)]
UPSAMPLE_ROWS = [(N_B, 16, 16, 512), (N_B, 32, 32, 256), (N_B, 64, 64, 128), (N_B, 128, 128, 64),
                 (1, 1, 1, 64), (1, 1, 3, 64), (1, 3, 1, 64), (2, 37, 53, 64)]
MSE_ROWS = [N_B * SIZE * SIZE, 3 * N_B * SIZE * SIZE]

TABLE = {
    "bn": set(BN_ROWS + BN_EDGE_ROWS),
    "bias_sum": {(n * 4 * h * w, co) for n, h, w, ci, co in CONVT_ROWS + CONVT_RAGGED},
    "convt_dgrad": {(n, h, w, 4 * co, ci) for n, h, w, ci, co in CONVT_ROWS + CONVT_RAGGED},
    "wgrad_pw": {(n, h, w, ci, 4 * co) for n, h, w, ci, co in CONVT_ROWS + CONVT_RAGGED},
    "stem": set(STEM_ROWS),
    "stem_pack": {(cin,) for cin in range(1, 9)},
    "stem_wgrad": set(STEM_WGRAD_ROWS),
    "head": set(HEAD_ROWS),
    "mse": {(n,) for n in MSE_ROWS},
    "combined": {(planes, SIZE, SIZE) for planes in (N_B, 3 * N_B)},
    "maxpool_bwd": set(MAXPOOL_ROWS),
    "upsample_bwd": set(UPSAMPLE_ROWS),
}


def test_every_recorded_configuration_has_a_row(cuda_device):
    """One TrainStep at batch 16 x 256^2 on the grey bilinear net, the grey ConvTranspose2d net and UNet(6, 3): every
    configuration it launches must be a row of the tables above."""
    from model.unet import FrameInterpolationUNet, UNet
    nets = {"grey bilinear": lambda: FrameInterpolationUNet(bilinear=True).unet,
            "grey convt": lambda: FrameInterpolationUNet(bilinear=False).unet,
            "UNet(6, 3)": lambda: UNet(6, 3)}
    missing, seen_all = [], set()
    for tag, make in nets.items():
        torch.manual_seed(0)
        seen = record_train_step(make().to(cuda_device).train())
        print(f"{tag}: {len(seen)} configurations")
        for k in sorted(seen, key=str):
            row = k[1:]
            ok = row in TABLE[k[0]]
            print(f"   {k[0]:13s} {row}  {'-> row' if ok else 'NO ROW'}")
            if not ok:
                missing.append((tag, k))
        seen_all |= seen
    assert {k[0] for k in seen_all} == set(TABLE) - {"combined"}, "an entry point was not recorded"
    assert not missing, f"configurations TrainStep launches without a row in the tables: {missing}"


# ------------------------------------------------------------------------------------------------ BatchNorm
def run_bn(lib, z, dA, gamma, beta, rm, rv):
    """The forward and backward BatchNorm kernels the way TrainStep chains them. z, dA: bf16 [P, C]."""
    P, c = z.shape
    dev = z.device
    work = torch.zeros(7, c, device=dev)           # sum, sumsq, mean, rstd, scale, shift, pivot
    E.check(lib.fiBnStatsShifted(p(z), P, c, p(work[6]), p(work[0]), p(work[1]), st()))
    E.check(lib.fiBnFinalizeShifted(p(work[0]), p(work[1]), p(work[6]), c, P, EPS, MOMENTUM, p(gamma), p(beta), p(work[2]),
                             p(work[3]), p(work[4]), p(work[5]), p(rm), p(rv), st()))
    a = torch.full_like(z, float("nan"))
    E.check(lib.fiBnApplyRelu(p(z), P, c, p(work[4]), p(work[5]), p(a), st()))
    red = torch.zeros(2, c, device=dev)
    E.check(lib.fiBnReluBackwardReduce(p(dA), p(z), P, c, p(work[2]), p(work[3]), p(work[4]), p(work[5]), p(red[0]),
                                       p(red[1]), st()))
    dz = torch.full_like(z, float("nan"))
    E.check(lib.fiBnReluBackwardApply(p(dA), p(z), P, c, p(work[2]), p(work[3]), p(gamma), p(beta), p(red[0]),
                                      p(red[1]), p(dz), st()))
    torch.cuda.synchronize()
    return dict(sum=work[0], sumsq=work[1], mean=work[2], rstd=work[3], pivot=work[6], a=a, dbeta=red[0],
                dgamma=red[1], dz=dz, rm=rm, rv=rv)


def check_bn(z, dA, gamma, beta, rm0, rv0, got, var_bar=False):
    """fp64 reference of batch-statistics BatchNorm + ReLU, forward and backward, on the same bf16 z / dA. The ReLU
    mask of the backward is the kernel's own (a > 0): whether each element is positive is checked by `a` itself, and
    an element within fp32 rounding of zero must not decide the comparison of the sums."""
    P, c = z.shape
    zd, dd, gd, bd = z.double(), dA.double(), gamma.double(), beta.double()
    ratios = {}
    mean = zd.mean(0)
    var = ((zd - mean) ** 2).mean(0)
    rstd = (var + EPS).rsqrt()
    std = var.sqrt()
    ratios["mean"] = sum_close(got["mean"], mean, mean.abs() + std, "mean")
    ratios["rstd"] = sum_close(got["rstd"], rstd, rstd, "rstd", ktol=0)
    ratios["running_mean"] = sum_close(got["rm"], (1 - MOMENTUM) * rm0.double() + MOMENTUM * mean,
                                       rm0.double().abs() + mean.abs() + std, "running_mean")
    rv_ref = (1 - MOMENTUM) * rv0.double() + MOMENTUM * var * P / (P - 1)
    ratios["running_var"] = sum_close(got["rv"], rv_ref, torch.full_like(rv_ref, 1e-6), "running_var", ktol=1e-6)
    if var_bar:   # running_var started at 0: it is the kernel's variance times MOMENTUM * P / (P - 1)
        var_k = got["rv"].double() / MOMENTUM * (P - 1) / P
        err, tol = (var_k - var).abs(), 1e-4 * var + 1e-9
        ratios["var"] = (err / tol).max().item()
        assert (err <= tol).all(), f"variance: max err/bar {ratios['var']:.3g}, worst channel " \
                                   f"{int((err / tol).argmax())}: {var_k[(err / tol).argmax()].item():.6g} vs " \
                                   f"{var[(err / tol).argmax()].item():.6g}"
    k = zd[0]
    assert torch.equal(got["pivot"].double(), k), "pivot = the first pixel"
    dev_ = zd - k
    ratios["sum"] = sum_close(got["sum"], dev_.sum(0), dev_.abs().sum(0), "shifted sum")
    ratios["sumsq"] = sum_close(got["sumsq"], (dev_ * dev_).sum(0), (dev_ * dev_).sum(0), "shifted sum of squares")
    zhat = (zd - mean) * rstd
    a_ref = (zhat * gd + bd).clamp_min(0)
    ratios["a"] = bf16_close(got["a"], a_ref, "a = relu(bn(z))")
    mask = got["a"] > 0
    dy = torch.where(mask, dd, 0.0)
    dbeta, dgamma = dy.sum(0), (dy * zhat).sum(0)
    ratios["dbeta"] = sum_close(got["dbeta"], dbeta, dy.abs().sum(0), "dbeta")
    ratios["dgamma"] = sum_close(got["dgamma"], dgamma, (dy * zhat).abs().sum(0), "dgamma")
    dz = gd * rstd * (dy - dbeta / P - zhat * dgamma / P)
    ratios["dz"] = bf16_close(got["dz"], dz, "dz")
    return ratios


def bn_inputs(dev, P, c, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    mean = torch.randn(c, generator=g, device=dev) * 2
    spread = torch.rand(c, generator=g, device=dev) * 1.5 + 0.1
    z = (torch.randn(P, c, generator=g, device=dev) * spread + mean).to(torch.bfloat16)
    dA = torch.randn(P, c, generator=g, device=dev).to(torch.bfloat16)
    gamma = torch.rand(c, generator=g, device=dev) + 0.5
    beta = torch.randn(c, generator=g, device=dev) * 0.3
    rm0, rv0 = torch.randn(c, generator=g, device=dev), torch.rand(c, generator=g, device=dev) + 0.5
    return z, dA, gamma, beta, rm0, rv0


@pytest.mark.parametrize("P,c", BN_ROWS + BN_EDGE_ROWS)
def test_batchnorm_at_scale(cuda_device, P, c):
    z, dA, gamma, beta, rm0, rv0 = bn_inputs(cuda_device, P, c, P % 1000 + c)
    got = run_bn(E.lib(), z, dA, gamma, beta, rm0.clone(), rv0.clone())
    ratios = check_bn(z, dA, gamma, beta, rm0, rv0, got)
    print("err/bar", {k: f"{v:.3g}" for k, v in ratios.items()})


FLAT_MEANS, FLAT_SPREADS = (0.5, 1.3, 3.0), (0.0, 1e-3, 1e-2)


def flat_inputs(dev, P=P0, c=64):
    """Channels with a large mean against their spread (flat regions, dark frames, letterbox bars, the bias-free stem
    output): m in {0.5, 1.3, 3} x s in {0, 1e-3, 1e-2} and one ordinary channel, repeated with alternating sign."""
    g = torch.Generator(device=dev).manual_seed(11)
    designs = [(m, s) for m in FLAT_MEANS for s in FLAT_SPREADS] + [(0.2, 1.0)]
    mean = torch.tensor([designs[i % 10][0] * (-1) ** (i // 10) for i in range(c)], device=dev)
    spread = torch.tensor([designs[i % 10][1] for i in range(c)], device=dev)
    z = (torch.randn(P, c, generator=g, device=dev) * spread + mean).to(torch.bfloat16)
    dA = torch.randn(P, c, generator=g, device=dev).to(torch.bfloat16)
    gamma = torch.rand(c, generator=g, device=dev) + 0.5
    beta = torch.randn(c, generator=g, device=dev) * 0.3
    return z, dA, gamma, beta


def test_batchnorm_flat_channels(cuda_device):
    """var = Q/P - (S/P)^2 from plain fp32 sums of z and z^2 cancels on these channels (an 11.8 % rstd error at
    m = 1.3, s = 0 in an emulation of the kernel's summation order); the sums about the first pixel do not."""
    z, dA, gamma, beta = flat_inputs(cuda_device)
    c = z.shape[1]
    rm0, rv0 = torch.zeros(c, device=cuda_device), torch.zeros(c, device=cuda_device)
    got = run_bn(E.lib(), z, dA, gamma, beta, rm0.clone(), rv0.clone())
    ratios = check_bn(z, dA, gamma, beta, rm0, rv0, got, var_bar=True)
    print("err/bar", {k: f"{v:.3g}" for k, v in ratios.items()})


# ------------------------------------------------------------------------------------------------ ConvTranspose2d backward
@pytest.fixture(params=["auto", "single-64", "single-128", "single-256", "pair-256"])
def gemm_selection(request, monkeypatch):
    """The 1-tap data-gradient GEMM under every kernel selection: automatic, each FI_BLOCK_N on the single-CTA kernel,
    and the CTA-pair kernel (N = 256 only)."""
    sel = request.param
    if sel != "auto":
        kind, bn = sel.split("-")
        monkeypatch.setenv("FI_CTA2", "1" if kind == "pair" else "0")
        monkeypatch.setenv("FI_BLOCK_N", bn)
    return sel


def convt_case(dev, n, h, w, ci, co, seed=0):
    """Operands of one ConvTranspose2d(ci, co, 2, 2) backward: layer input x (bf16 NHWC [n,h,w,ci]), weight
    [ci, co, 2, 2] (bf16-valued fp32), output gradient d_up (bf16 NHWC [n,2h,2w,co])."""
    g = torch.Generator(device=dev).manual_seed(seed + ci + h)
    x = torch.randn(n, h, w, ci, generator=g, device=dev).clamp_min(0).to(torch.bfloat16)   # post-ReLU input
    wt = (torch.randn(ci, co, 2, 2, generator=g, device=dev) * (1.0 / (4 * co)) ** 0.5).to(torch.bfloat16).float()
    d_up = torch.randn(n, 2 * h, 2 * w, co, generator=g, device=dev).to(torch.bfloat16)
    return x, wt, d_up


_REF = {}


def convt_reference(dev, n, h, w, ci, co):
    """fp64 autograd of F.conv_transpose2d(stride=2) on the same bf16 operands: (d_lo, dW, db) plus the magnitudes
    sum |terms| of dW and db. Cached: the same operands serve every kernel selection."""
    key = (n, h, w, ci, co)
    if key not in _REF:
        x, wt, d_up = convt_case(dev, n, h, w, ci, co)
        xd = x.permute(0, 3, 1, 2).double().requires_grad_(True)
        wd = wt.double().requires_grad_(True)
        bd = torch.zeros(co, dtype=torch.float64, device=dev, requires_grad=True)
        F.conv_transpose2d(xd, wd, bd, stride=2).backward(d_up.permute(0, 3, 1, 2).double())
        wa = torch.zeros_like(wd, requires_grad=True)      # sum |terms| of dW: the same product on magnitudes
        F.conv_transpose2d(xd.detach().abs(), wa, stride=2).backward(d_up.permute(0, 3, 1, 2).double().abs())
        _REF[key] = (xd.grad.permute(0, 2, 3, 1).contiguous(), wd.grad, bd.grad, wa.grad,
                     d_up.double().abs().sum((0, 1, 2)))
    return _REF[key]


@pytest.mark.parametrize("n,h,w,ci,co", CONVT_ROWS + CONVT_RAGGED)
def test_convt_data_gradient_gemm(cuda_device, gemm_selection, n, h, w, ci, co):
    """d_lo = [N,h,w,(ky,kx,co)] x W^T as the 1-tap EPI_STORE GEMM, weights packed as TrainStep packs them."""
    if gemm_selection.endswith("256") and ci % 256:
        pytest.skip("n_total is not a multiple of 256")
    lib = E.lib()
    x, wt, d_up = convt_case(cuda_device, n, h, w, ci, co)
    d_s2d = d_up.view(n, h, 2, w, 2, co).permute(0, 1, 3, 2, 4, 5).contiguous().view(n, h, w, 4 * co)
    w_lo = wt.permute(0, 2, 3, 1).reshape(ci, 4 * co).to(torch.bfloat16).contiguous()
    zero = torch.zeros(ci, device=cuda_device)
    dst = torch.full((n, h, w, ci), float("nan"), dtype=torch.bfloat16, device=cuda_device)
    d = E.ConvDesc()
    d.src0, d.c0, d.N, d.H, d.W = d_s2d.data_ptr(), 4 * co, n, h, w
    d.wpack, d.bias, d.n_total, d.taps, d.mode, d.relu, d.dst = (w_lo.data_ptr(), zero.data_ptr(), ci, 1, E.EPI_STORE,
                                                                 0, dst.data_ptr())
    E.check(lib.fiConvGemm(C.byref(d), st()))
    torch.cuda.synchronize()
    d_lo = convt_reference(cuda_device, n, h, w, ci, co)[0]
    print("err/bar", f"{bf16_close(dst, d_lo, 'd_lo', abs_frac=0, abs_min=1e-3):.3g}")


@pytest.mark.parametrize("n,h,w,ci,co", CONVT_ROWS + CONVT_RAGGED + [(2, 12, 10, 384, 64), (1, 9, 7, 192, 128)])
def test_pointwise_weight_gradient(cuda_device, n, h, w, ci, co):
    """fiWgradPointwise accumulates dW[(ky,kx,co)][ci] = sum_q d[q][(ky,kx,co)] x[q][ci] into its output. Cin/64 =
    16/8/4 -> 4 column blocks per tile, 2 -> 2, 6 and 3 (cin 384 / 192) -> 3."""
    lib = E.lib()
    x, _, d_up = convt_case(cuda_device, n, h, w, ci, co)
    d_s2d = d_up.view(n, h, 2, w, 2, co).permute(0, 1, 3, 2, 4, 5).contiguous().view(n, h, w, 4 * co)
    g = torch.Generator(device=cuda_device).manual_seed(3)
    prior = torch.randn(4 * co, ci, generator=g, device=cuda_device)
    dW = prior.clone()
    E.check(lib.fiWgradPointwise(p(d_s2d), p(x), ci, n, h, w, 4 * co, p(dW), st()))
    torch.cuda.synchronize()
    dq, xq = d_s2d.reshape(-1, 4 * co).double(), x.reshape(-1, ci).double()
    ref, mag = dq.t() @ xq, dq.abs().t() @ xq.abs()
    r = sum_close(dW - prior, ref, mag + 1e-2 * prior.abs(), "pointwise dW")
    print("err/bar", f"{r:.3g}")


def test_pointwise_weight_gradient_refuses_odd_channel_blocks(cuda_device):
    lib = E.lib()
    for ci in (64, 320):   # 1 and 5 blocks of 64 input channels
        x = torch.zeros(1, 4, 4, ci, dtype=torch.bfloat16, device=cuda_device)
        d = torch.zeros(1, 4, 4, 256, dtype=torch.bfloat16, device=cuda_device)
        dW = torch.zeros(256, ci, device=cuda_device)
        assert lib.fiWgradPointwise(p(d), p(x), ci, 1, 4, 4, 256, p(dW), st()) != 0, ci


@pytest.mark.parametrize("n,h,w,ci,co", CONVT_ROWS + CONVT_RAGGED)
def test_convt_bias_gradient(cuda_device, n, h, w, ci, co):
    """fiBnStats as the bias gradient: plain per-channel sums ACCUMULATED into the gradient."""
    lib = E.lib()
    _, _, d_up = convt_case(cuda_device, n, h, w, ci, co)
    g = torch.Generator(device=cuda_device).manual_seed(4)
    prior, prior_q = torch.randn(co, generator=g, device=cuda_device), torch.rand(co, generator=g, device=cuda_device)
    s, q = prior.clone(), prior_q.clone()
    E.check(lib.fiBnStats(p(d_up), n * 4 * h * w, co, p(s), p(q), st()))
    torch.cuda.synchronize()
    dd = d_up.reshape(-1, co).double()
    r1 = sum_close(s - prior, dd.sum(0), dd.abs().sum(0) + prior.abs(), "bias gradient")
    r2 = sum_close(q - prior_q, (dd * dd).sum(0), (dd * dd).sum(0) + prior_q.abs(), "sum of squares")
    print("err/bar", f"{r1:.3g} {r2:.3g}")


@pytest.fixture(scope="module")
def convt_step(cuda_device):
    from model.train import TrainStep
    from model.unet import UNet
    return TrainStep(UNet(2, 1, bilinear=False).to(cuda_device).train(), lr=0.0)


@pytest.mark.parametrize("n,h,w,ci,co", CONVT_ROWS + CONVT_RAGGED)
def test_convt_backward_composition(cuda_device, convt_step, n, h, w, ci, co):
    """TrainStep._convt_backward (the (ky, kx, co) view of d_up, the GEMM, the pointwise weight gradient, its permute
    into [ci, co, ky, kx], the bias) against fp64 autograd of F.conv_transpose2d."""
    x, wt, d_up = convt_case(cuda_device, n, h, w, ci, co)
    w_lo = wt.permute(0, 2, 3, 1).reshape(ci, 4 * co).to(torch.bfloat16).contiguous()   # model/train.py forward
    gw, gb = torch.zeros(ci, co, 2, 2, device=cuda_device), torch.zeros(co, device=cuda_device)
    d_lo = convt_step._convt_backward(d_up, x, w_lo, gw, gb)
    torch.cuda.synchronize()
    ref_lo, ref_w, ref_b, mag_w, mag_b = convt_reference(cuda_device, n, h, w, ci, co)
    r = [bf16_close(d_lo, ref_lo, "d_lo", abs_frac=0, abs_min=1e-3), sum_close(gw, ref_w, mag_w, "dW"),
         sum_close(gb, ref_b, mag_b, "db")]
    print("err/bar", " ".join(f"{v:.3g}" for v in r))


# ------------------------------------------------------------------------------------------------ stem
def stem_pack(lib, w, cin):
    packed = torch.empty((64, lib.fiStemPackedK(cin)), dtype=torch.bfloat16, device=w.device)
    E.check(lib.fiStemPackWeightsDevice(p(w), cin, p(packed), st()))
    return packed


@pytest.mark.parametrize("cin,n,h,w", STEM_ROWS)
def test_stem_conv_linear(cuda_device, cin, n, h, w):
    """The training stem keeps negative outputs; hi/lo operand splitting leaves only the bf16 output cast."""
    lib = E.lib()
    g = torch.Generator(device=cuda_device).manual_seed(cin)
    x = torch.rand(n, cin, h, w, generator=g, device=cuda_device) * 2 - 1
    wt = torch.randn(64, cin, 3, 3, generator=g, device=cuda_device) * 0.3
    b = torch.randn(64, generator=g, device=cuda_device) * 0.1
    dst = torch.full((n, h, w, 64), float("nan"), dtype=torch.bfloat16, device=cuda_device)
    p0 = E.planes_of(x)
    E.check(lib.fiStemConvLinear(C.byref(p0), None, E.FI_IN_F32, p(stem_pack(lib, wt, cin)), p(b), p(dst), n, h, w,
                                 st()))
    torch.cuda.synchronize()
    ref = F.conv2d(x.double(), wt.double(), b.double(), padding=1).permute(0, 2, 3, 1)
    got = dst.double()
    assert (ref < -0.1).any() and (got < -0.1).any(), "negative outputs must survive"
    err, tol = (got - ref).abs(), 2.0 ** -8 * ref.abs() + 1e-4      # the bar of test_gpu_aux_kernels.test_stem_conv
    assert (err <= tol).all(), f"max err/bar {(err / tol).max().item():.3g}"
    print("err/bar", f"{(err / tol).max().item():.3g}")


def test_stem_pack_device_matches_host(cuda_device):
    lib = E.lib()
    for cin in range(1, 9):
        g = torch.Generator().manual_seed(cin)
        w = torch.randn(64, cin, 3, 3, generator=g) * 0.3
        host = torch.empty((64, lib.fiStemPackedK(cin)), dtype=torch.int16)
        E.check(lib.fiStemPackWeights(w.data_ptr(), cin, host.data_ptr()))
        dev = stem_pack(lib, w.to(cuda_device), cin)
        torch.cuda.synchronize()
        assert torch.equal(dev.view(torch.int16).cpu(), host), f"cin {cin}"


@pytest.mark.parametrize("cin,n,h,w", STEM_WGRAD_ROWS)
def test_stem_weight_gradient_at_scale(cuda_device, cin, n, h, w):
    """W = 256: two 128-pixel segments per row; W = 200: a partial second segment."""
    lib = E.lib()
    g = torch.Generator(device=cuda_device).manual_seed(cin + w)
    x = torch.rand(n, cin, h, w, generator=g, device=cuda_device) * 2 - 1
    dz = torch.randn(n, h, w, 64, generator=g, device=cuda_device).to(torch.bfloat16)
    prior = torch.randn(64, cin, 3, 3, generator=g, device=cuda_device)
    dW = prior.clone()
    E.check(lib.fiStemWgrad(p(dz), p(x), n, h, w, cin, p(dW), st()))
    torch.cuda.synchronize()
    dzd = dz.permute(0, 3, 1, 2).double()
    ref = torch.nn.grad.conv2d_weight(x.double(), (64, cin, 3, 3), dzd, padding=1)
    mag = torch.nn.grad.conv2d_weight(x.double().abs(), (64, cin, 3, 3), dzd.abs(), padding=1)
    print("err/bar", f"{sum_close(dW - prior, ref, mag + prior.abs(), 'stem dW'):.3g}")


# ------------------------------------------------------------------------------------------------ head and loss
@pytest.mark.parametrize("P,ncls", HEAD_ROWS)
def test_head_forward_backward_at_scale(cuda_device, P, ncls):
    lib = E.lib()
    n = N_B if P == P0 else 3
    hw = P // n
    g = torch.Generator(device=cuda_device).manual_seed(P % 977 + ncls)
    a = torch.randn(P, 64, generator=g, device=cuda_device).clamp_min(0).to(torch.bfloat16)
    wt = torch.randn(ncls, 64, generator=g, device=cuda_device) * 0.3
    b = torch.randn(ncls, generator=g, device=cuda_device)
    dy = torch.randn(n, ncls, hw, generator=g, device=cuda_device) * 1e-3
    y = torch.full((n, ncls, hw), float("nan"), device=cuda_device)
    E.check(lib.fiHeadForward(p(a), n, hw, p(wt), p(b), ncls, p(y), st()))
    da = torch.full_like(a, float("nan"))
    dw, db = torch.zeros(ncls, 64, device=cuda_device), torch.zeros(ncls, device=cuda_device)
    E.check(lib.fiHeadBackward(p(a), p(dy), n, hw, p(wt), ncls, p(da), p(dw), p(db), st()))
    torch.cuda.synchronize()
    ad, wd = a.double().view(n, hw, 64), wt.double()
    y_ref = torch.einsum("npc,kc->nkp", ad, wd) + b.double()[None, :, None]
    r = [sum_close(y, y_ref, torch.einsum("npc,kc->nkp", ad.abs(), wd.abs()) + b.double().abs()[None, :, None], "y")]
    dyd = dy.double()
    r.append(bf16_close(da.view(n, hw, 64), torch.einsum("nkp,kc->npc", dyd, wd), "da", abs_min=1e-9))
    r.append(sum_close(dw, torch.einsum("nkp,npc->kc", dyd, ad), torch.einsum("nkp,npc->kc", dyd.abs(), ad.abs()), "dw"))
    r.append(sum_close(db, dyd.sum((0, 2)), dyd.abs().sum((0, 2)), "db"))
    print("err/bar", " ".join(f"{v:.3g}" for v in r))


@pytest.mark.parametrize("n", MSE_ROWS)
def test_mse_loss_at_scale(cuda_device, n):
    lib = E.lib()
    g = torch.Generator(device=cuda_device).manual_seed(n % 1000)
    y = torch.randn(n, generator=g, device=cuda_device)
    t = torch.rand(n, generator=g, device=cuda_device)
    loss, dy = torch.zeros(1, device=cuda_device), torch.full_like(y, float("nan"))
    E.check(lib.fiMseLossGrad(p(y), p(t), n, p(loss), p(dy), st()))
    torch.cuda.synchronize()
    d = y.double() - t.double()
    r1 = sum_close(loss, (d * d).mean().reshape(1), (d * d).mean().reshape(1), "loss")
    r2 = sum_close(dy, 2 * d / n, 2 * (y.double().abs() + t.double().abs()) / n, "dy", ktol=1e-6)
    print("err/bar", f"{r1:.3g} {r2:.3g}")


@pytest.mark.parametrize("planes", [N_B, 3 * N_B])
def test_combined_loss_at_scale(cuda_device, planes):
    """fiCombinedLossGrad at 16 grey planes and 16 x 3 RGB planes of 256^2 against fp64 autograd of CombinedLoss."""
    from model.train import CombinedLoss
    lib = E.lib()
    g = torch.Generator(device=cuda_device).manual_seed(planes)
    pred = torch.rand(planes, 1, SIZE, SIZE, generator=g, device=cuda_device)
    target = (pred + 0.15 * torch.randn(pred.shape, generator=g, device=cuda_device)).clamp(0, 1)
    pr = pred.double().requires_grad_(True)
    loss_ref = CombinedLoss(0.5, 0.5)(pr, target.double())
    loss_ref.backward()
    loss, dy = torch.zeros(1, device=cuda_device), torch.full_like(pred, float("nan"))
    E.check(lib.fiCombinedLossGrad(p(pred), p(target), planes, SIZE, SIZE, 0.5, 0.5, p(loss), p(dy), st()))
    torch.cuda.synchronize()
    err = abs(loss.item() - loss_ref.item())
    assert err < 2e-6 + 1e-5 * abs(loss_ref.item()), err           # the bars of test_combined_loss_kernel_matches_torch
    gerr = (dy.double() - pr.grad).abs().max().item()
    assert gerr <= 2e-3 * pr.grad.abs().max().item() + 1e-9, gerr
    print("err/bar", f"{err / (2e-6 + 1e-5 * abs(loss_ref.item())):.3g} {gerr / (2e-3 * pr.grad.abs().max().item()):.3g}")


# ------------------------------------------------------------------------------------------------ pool / upsample backward
def _torch_routes_ties_to_first():
    a = torch.zeros(1, 1, 2, 2, requires_grad=True)
    F.max_pool2d(a, 2).backward(torch.ones(1, 1, 1, 1))
    return a.grad.flatten().tolist() == [1.0, 0.0, 0.0, 0.0]


@pytest.mark.parametrize("skip", [True, False], ids=["skip", "no-skip"])
@pytest.mark.parametrize("n,h,w,c", MAXPOOL_ROWS)
def test_maxpool_backward_ties(cuda_device, n, h, w, c, skip):
    """Post-ReLU activations: many all-zero and tied windows. The kernel routes the gradient to the first maximum in
    scan order, as torch's CPU max_pool2d does; both sides add two bf16 values and round once, so the result is
    compared bit for bit."""
    if not _torch_routes_ties_to_first():
        pytest.skip("torch's max_pool2d does not route ties to the first maximum here")
    lib = E.lib()
    g = torch.Generator(device=cuda_device).manual_seed(h * w + c)
    a = torch.randn(n, h, w, c, generator=g, device=cuda_device).clamp_min(0).to(torch.bfloat16)
    d_pool = torch.randn(n, h // 2, w // 2, c, generator=g, device=cuda_device).to(torch.bfloat16)
    d_skip = torch.randn(n, h, w, c, generator=g, device=cuda_device).to(torch.bfloat16) if skip else None
    pooled = torch.empty((n, h // 2, w // 2, c), dtype=torch.bfloat16, device=cuda_device)
    E.check(lib.fiMaxPool2x2(p(a), p(pooled), n, h, w, c, st()))
    out = torch.full((n, h, w, c), float("nan"), dtype=torch.bfloat16, device=cuda_device)
    E.check(lib.fiMaxPoolBackwardAdd(p(a), p(pooled), p(d_pool), p(d_skip), p(out), n, h, w, c, st()))
    torch.cuda.synchronize()
    ar = a.cpu().float().permute(0, 3, 1, 2).requires_grad_(True)
    F.max_pool2d(ar, 2).backward(d_pool.cpu().float().permute(0, 3, 1, 2))
    ref = ar.grad.permute(0, 2, 3, 1)
    if skip:
        ref = ref + d_skip.cpu().float()
    ref = ref.to(torch.bfloat16)
    got = out.cpu()
    bad = got.view(torch.int16) != ref.view(torch.int16)
    assert not bad.any(), f"{int(bad.sum())} elements differ, first at {bad.nonzero()[0].tolist()}"


@pytest.mark.parametrize("n,h,w,c", UPSAMPLE_ROWS)
def test_upsample_backward_at_scale(cuda_device, n, h, w, c):
    lib = E.lib()
    g = torch.Generator(device=cuda_device).manual_seed(h * 7 + w)
    d_up = torch.randn(n, 2 * h, 2 * w, c, generator=g, device=cuda_device).to(torch.bfloat16)
    out = torch.full((n, h, w, c), float("nan"), dtype=torch.bfloat16, device=cuda_device)
    E.check(lib.fiUpsample2xBackward(p(d_up), p(out), n, h, w, c, st()))
    torch.cuda.synchronize()
    x = torch.zeros(n, c, h, w, dtype=torch.float64, device=cuda_device, requires_grad=True)
    F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True).backward(d_up.permute(0, 3, 1, 2).double())
    print("err/bar", f"{bf16_close(out, x.grad.permute(0, 2, 3, 1), 'd_lo', abs_frac=0, abs_min=1e-3):.3g}")


# ------------------------------------------------------------------------------------------------ optimizer and packing
@pytest.mark.parametrize("step", [1, 10000])
def test_adam_beyond_the_grid_cap(cuda_device, step):
    """31 M + 7 parameters: 1 184 blocks of 256 threads walk ~107 grid strides and a tail. The device-hyper path
    ({lr, step} read at run time) must give the same bits as the host arguments."""
    lib = E.lib()
    n = 31 * 2 ** 20 + 7
    g = torch.Generator(device=cuda_device).manual_seed(step)
    prm, grad = torch.randn(n, generator=g, device=cuda_device), torch.randn(n, generator=g, device=cuda_device) * 1e-2
    if step == 1:
        m0, v0 = torch.zeros(n, device=cuda_device), torch.zeros(n, device=cuda_device)
    else:
        m0 = torch.randn(n, generator=g, device=cuda_device) * 1e-2
        v0 = torch.rand(n, generator=g, device=cuda_device) * 1e-4
    lr, b1, b2, eps = 1e-3, 0.9, 0.999, 1e-8
    outs = []
    for hyper in (None, torch.tensor([lr, float(step)], device=cuda_device)):
        pp, m, v = prm.clone(), m0.clone(), v0.clone()
        E.check(lib.fiAdamStep(p(pp), p(grad), p(m), p(v), n, 0.0 if hyper is not None else lr, b1, b2, eps,
                               step, p(hyper), st()))
        outs.append((pp, m, v))
    torch.cuda.synchronize()
    lr, b1, b2, eps = (torch.tensor(x, dtype=torch.float32).item() for x in (lr, b1, b2, eps))   # as the kernel reads them
    gd = grad.double()
    m_ref = b1 * m0.double() + (1 - b1) * gd
    v_ref = b2 * v0.double() + (1 - b2) * gd * gd
    upd = lr * (m_ref / (1 - b1 ** step)) / ((v_ref / (1 - b2 ** step)).sqrt() + eps)
    p_ref = prm.double() - upd
    pp, m, v = outs[0]
    r = [sum_close(m, m_ref, b1 * m0.double().abs() + (1 - b1) * gd.abs(), "m", rtol=1e-6, ktol=1e-6),
         sum_close(v, v_ref, v_ref, "v", rtol=1e-6, ktol=1e-6),
         sum_close(pp, p_ref, 1e-3 * upd.abs() + 2.4e-7 * prm.double().abs(), "parameters", rtol=0, ktol=1)]
    print("err/bar", " ".join(f"{x:.3g}" for x in r))
    for name, a, b in zip(("p", "m", "v"), outs[0], outs[1]):
        assert torch.equal(a, b), f"{name}: hyper_dev path differs from the host arguments"


@pytest.mark.parametrize("co,ci", [(1024, 512), (512, 1024)])
def test_pack_and_unpack_at_scale(cuda_device, co, ci):
    lib = E.lib()
    g = torch.Generator(device=cuda_device).manual_seed(co)
    w = torch.randn(co, ci, 3, 3, generator=g, device=cuda_device)
    fwd = torch.empty((co, 9 * ci), dtype=torch.bfloat16, device=cuda_device)
    bwd = torch.empty((ci, 9 * co), dtype=torch.bfloat16, device=cuda_device)
    E.check(lib.fiPackConvWeights(p(w), co, ci, p(fwd), p(bwd), st()))
    dW = torch.randn(9, co, ci, generator=g, device=cuda_device)
    grad = torch.randn(co, ci, 3, 3, generator=g, device=cuda_device)
    want = grad + dW.permute(1, 2, 0).reshape(co, ci, 3, 3)
    E.check(lib.fiUnpackConvGrad(p(dW), co, ci, p(grad), st()))
    torch.cuda.synchronize()
    wb = w.to(torch.bfloat16)
    assert torch.equal(fwd, wb.permute(0, 2, 3, 1).reshape(co, -1))
    assert torch.equal(bwd, wb.flip(2, 3).permute(1, 2, 3, 0).reshape(ci, -1))
    assert torch.equal(grad, want)
