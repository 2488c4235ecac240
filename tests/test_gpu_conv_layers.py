"""Layer-level parity of the tcgen05 implicit-GEMM kernel (through the C ABI, fiConvGemm) against an fp64-accumulated
CPU convolution of the same bf16-rounded operands. Tolerance: the kernel accumulates in fp32 and rounds once to bf16,
so it may land on the bf16 neighbour of the rounded fp64 result: |err| <= 1 bf16 ulp <= 2^-7 * |ref| (+1e-3 near 0)."""
import pytest
import torch
import torch.nn.functional as F

from model import _engine as E
from layer_utils import bf16_round, ref_conv3x3, run_conv, run_conv_precise

pytestmark = pytest.mark.gpu


@pytest.fixture(params=["halo", "per-tap", "pair"], autouse=True)
def kernel_variant(request, monkeypatch):
    """Cout 64/128 layers have two kernel families (halo reuse in conv_halo.cu, per tap in conv_gemm.cu), and the halo
    family and the Cout-multiple-of-256 per-tap kernels each run as one CTA or as a CTA pair; run every case through
    all selections."""
    monkeypatch.setenv("FI_NO_HALO", "1" if request.param == "per-tap" else "0")
    monkeypatch.setenv("FI_CTA2", "1" if request.param == "pair" else "0")
    return request.param


def close(a, b, what):
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert not torch.isnan(a).any(), f"{what}: NaN in output (unwritten elements?)"
    err = (a - b).abs()
    tol = 2.0 ** -7 * b.abs() + 1e-3
    bad = (err > tol)
    assert not bad.any(), f"{what}: {int(bad.sum())}/{bad.numel()} mismatches, max err {err.max():.4g}, " \
                          f"first at {bad.nonzero()[0].tolist()}"


def rnd(g, *shape, scale=1.0):
    return torch.randn(*shape, generator=g) * scale


@pytest.mark.parametrize("n,cin,cout,h,w", [
    (1, 64, 64, 16, 16),       # two tiles, BLOCK_N 64
    (2, 128, 128, 24, 40),     # ragged tiles in both dims, BLOCK_N 128
    (1, 256, 256, 16, 32),     # BLOCK_N 256
    (1, 512, 512, 8, 16),      # 72 K iterations: smem ring wraps 24x
    (1, 64, 64, 200, 208),     # 325 tiles on <=148 CTAs: TMEM double buffering and barrier phases
    (1, 128, 64, 5, 7),        # image smaller than one tile
    (3, 192, 320, 9, 17),      # odd everything; cout 320 -> BLOCK_N 64 x 5 blocks
    (2, 64, 64, 13, 95),       # ragged halo tiles in both dims, two images
    (1, 128, 64, 9, 61),       # ... with two K slabs from one source
])
def test_conv3x3_store(cuda_device, n, cin, cout, h, w):
    g = torch.Generator().manual_seed(n * 1000 + cin + cout + h + w)
    x = rnd(g, n, cin, h, w)
    wt = rnd(g, cout, cin, 3, 3, scale=(2.0 / (9 * cin)) ** 0.5)
    b = rnd(g, cout, scale=0.1)
    got = run_conv(cuda_device, x, wt, b, relu=True)["dst"]
    close(got, bf16_round(ref_conv3x3(x, wt, b)), f"conv3x3 {cin}->{cout} {h}x{w}")


def test_conv3x3_no_relu(cuda_device):
    g = torch.Generator().manual_seed(5)
    x, wt, b = rnd(g, 1, 64, 16, 16), rnd(g, 64, 64, 3, 3, scale=0.06), rnd(g, 64, scale=0.1)
    got = run_conv(cuda_device, x, wt, b, relu=False)["dst"]
    ref = ref_conv3x3(x, wt, b, relu=False)
    assert (ref < 0).any()
    close(got, bf16_round(ref), "conv3x3 no relu")


@pytest.mark.parametrize("n,c,cout,h,w", [(1, 64, 64, 16, 32), (2, 64, 128, 18, 34), (1, 128, 256, 135, 30),
                                          (1, 64, 64, 7, 9)])
def test_conv3x3_pool(cuda_device, n, c, cout, h, w):
    g = torch.Generator().manual_seed(h * w + c)
    x, wt, b = rnd(g, n, c, h, w), rnd(g, cout, c, 3, 3, scale=(2.0 / (9 * c)) ** 0.5), rnd(g, cout, scale=0.1)
    out = run_conv(cuda_device, x, wt, b, mode=E.EPI_STORE_POOL)
    ref = bf16_round(ref_conv3x3(x, wt, b))
    close(out["dst"], ref, "pool: full-res store")
    # the pooled tensor must be EXACTLY max_pool2d(floor) of the stored full-res tensor
    assert torch.equal(out["pool"], F.max_pool2d(out["dst"], 2)), "pooled tensor != max_pool2d(stored tensor)"


@pytest.mark.parametrize("c0,c1,cout,h,w,h1,w1", [
    (64, 64, 64, 16, 32, 16, 32),        # plain concat
    (64, 64, 64, 17, 33, 16, 32),        # Cout 64 with F.pad
    (64, 64, 64, 70, 118, 70, 118),      # ... several tiles per CTA row
    (128, 128, 128, 17, 33, 16, 32),     # F.pad: one zero row at the bottom / column on the right
    (256, 256, 256, 19, 20, 16, 16),     # pad on both sides (diff 3 -> 1 before, 2 after; diff 4 -> 2, 2)
    (512, 512, 512, 135 // 8, 30, 16, 30),
])
def test_conv3x3_fused_concat(cuda_device, c0, c1, cout, h, w, h1, w1):
    g = torch.Generator().manual_seed(c0 + h + w)
    x, x1 = rnd(g, 1, c0, h, w), rnd(g, 1, c1, h1, w1)
    wt = rnd(g, cout, c0 + c1, 3, 3, scale=(2.0 / (9 * (c0 + c1))) ** 0.5)
    b = rnd(g, cout, scale=0.1)
    off = ((h - h1) // 2, (w - w1) // 2)
    got = run_conv(cuda_device, x, wt, b, x1=x1, off=off)["dst"]
    close(got, bf16_round(ref_conv3x3(x, wt, b, x1=x1, off=off)), "fused pad+concat conv")


@pytest.mark.parametrize("n,cin,cout,h,w", [(1, 128, 64, 8, 16), (2, 256, 128, 9, 20), (1, 1024, 512, 4, 7)])
def test_conv_transpose(cuda_device, n, cin, cout, h, w):
    g = torch.Generator().manual_seed(cin + h)
    x = rnd(g, n, cin, h, w)
    wt = rnd(g, cin, cout, 2, 2, scale=(1.0 / cin) ** 0.5)
    b = rnd(g, cout, scale=0.1)
    got = run_conv(cuda_device, x, wt, b, relu=False, mode=E.EPI_CONVT)["dst"]
    ref = F.conv_transpose2d(bf16_round(x).double(), bf16_round(wt).double(), b.double(), stride=2).float()
    close(got, bf16_round(ref), "conv transpose 2x2 s2")


@pytest.mark.parametrize("ncls,h,w", [(1, 16, 32), (3, 21, 37)])
def test_head_epilogue(cuda_device, ncls, h, w):
    g = torch.Generator().manual_seed(ncls + h)
    x, wt, b = rnd(g, 2, 64, h, w), rnd(g, 64, 64, 3, 3, scale=0.06), rnd(g, 64, scale=0.1)
    hw_, hb = rnd(g, ncls, 64, scale=0.4), rnd(g, ncls, scale=0.2)
    out = run_conv(cuda_device, x, wt, b, mode=E.EPI_HEAD, head_w=hw_, head_b=hb, want_u8=True)
    feat = ref_conv3x3(x, wt, b)  # fp32, NOT rounded to bf16: the head consumes the fp32 accumulators
    ref = F.conv2d(feat.double(), hw_.double()[:, :, None, None], hb.double()).float()
    err = (out["f32"] - ref).abs().max().item()
    assert err < 2e-4, f"head fp32 max err {err}"
    # u8 output == postprocess_image applied to the kernel's own fp32 output, bit for bit
    t = out["f32"]
    exp = (torch.clamp((t + 1.0) / 2.0, 0.0, 1.0).numpy() * 255).astype("uint8")
    assert (out["u8"].numpy() == exp).all()


# ------------------------------------------------------------------------------------------------ precise (fp32x3) mode
def ref_fp64(x, w, b, relu=True, x1=None, off=(0, 0)):
    xin = x
    if x1 is not None:
        h, wd = x.shape[2], x.shape[3]
        xin = torch.cat([x, F.pad(x1, [off[1], wd - x1.shape[3] - off[1], off[0], h - x1.shape[2] - off[0]])], 1)
    y = F.conv2d(xin.double(), w.double(), b.double(), padding=1)
    return (F.relu(y) if relu else y).float()


def close_precise(a, b, what):
    assert a.shape == b.shape and not torch.isnan(a).any(), what
    err = (a - b).abs().max().item()
    scale = b.abs().max().item()
    # three bf16 x bf16 products of hi/lo splits: ~2^-16 relative per operand; output re-split to 16 bits
    assert err <= 2.0 ** -13 * scale + 1e-6, f"{what}: max err {err:.3g} (scale {scale:.3g})"


@pytest.mark.parametrize("n,c0,c1,cout,h,w,mode", [
    (1, 64, 0, 64, 16, 32, E.EPI_STORE), (2, 128, 0, 128, 19, 23, E.EPI_STORE_POOL),
    (1, 256, 0, 256, 9, 17, E.EPI_STORE), (1, 64, 64, 64, 18, 34, E.EPI_STORE), (1, 256, 256, 256, 17, 20, E.EPI_STORE_POOL),
    (1, 128, 128, 128, 16, 48, E.EPI_STORE),
])
def test_precise_conv3x3(cuda_device, n, c0, c1, cout, h, w, mode):
    g = torch.Generator().manual_seed(c0 + c1 + cout + h)
    x = rnd(g, n, c0, h, w)
    x1 = rnd(g, n, c1, h - 1, w - 2) if c1 else None
    off = (0, 1)
    wt = rnd(g, cout, c0 + c1, 3, 3, scale=(2.0 / (9 * (c0 + c1))) ** 0.5)
    b = rnd(g, cout, scale=0.1)
    out = run_conv_precise(cuda_device, x, wt, b, mode=mode, x1=x1, off=off)
    ref = ref_fp64(x, wt, b, x1=x1, off=off)
    close_precise(out["dst"], ref, "precise conv")
    if mode == E.EPI_STORE_POOL:
        close_precise(out["pool"], F.max_pool2d(ref, 2), "precise pooled")
        assert (out["pool"] - F.max_pool2d(out["dst"], 2)).abs().max() <= 2.0 ** -15 * ref.abs().max()


def test_precise_conv_transpose_and_head(cuda_device):
    g = torch.Generator().manual_seed(77)
    x, wt, b = rnd(g, 1, 128, 9, 20), rnd(g, 128, 64, 2, 2, scale=0.09), rnd(g, 64, scale=0.1)
    got = run_conv_precise(cuda_device, x, wt, b, relu=False, mode=E.EPI_CONVT)["dst"]
    ref = F.conv_transpose2d(x.double(), wt.double(), b.double(), stride=2).float()
    close_precise(got, ref, "precise conv transpose")
    x, wt, b = rnd(g, 1, 64, 20, 24), rnd(g, 64, 64, 3, 3, scale=0.06), rnd(g, 64, scale=0.1)
    hw_, hb = rnd(g, 2, 64, scale=0.4), rnd(g, 2, scale=0.2)
    out = run_conv_precise(cuda_device, x, wt, b, mode=E.EPI_HEAD, head_w=hw_, head_b=hb)["f32"]
    ref = F.conv2d(ref_fp64(x, wt, b).double(), hw_.double()[:, :, None, None], hb.double()).float()
    assert (out - ref).abs().max() <= 2.0 ** -13 * ref.abs().max()
