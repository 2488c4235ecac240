"""Every conv launch of the forward at the shapes bench.py and the product run, per element against float64.

test_gpu_conv_layers.py checks each kernel selection per element, but at most 200x208 pixels: a persistent CTA walks a
handful of tiles, the TMEM double buffer and the mbarrier phases wrap a few times, and the CTA-pair clusters never see a
real layer's tile count. test_gpu_parity_baseline_sizes.py runs the real sizes, but under a relative-L2 bar that about
25 completely wrong tiles of `inc` would pass. This file closes the gap:

- `schedule()` derives every launch of fiNetForward from (network, N, H, W, precision), as engine.cu:fill_plan does.
  `test_every_forward_launch_has_a_row` compares it with Net.profile() for the seven configurations below, and
  `test_every_train_step_conv3x3_has_a_row` with the 3x3 fiConvGemm calls of TrainStep at 16 x 256^2. A schedule change
  (a fused layer, a new kernel) fails there until the derivation, and with it the per-layer rows, follows it.
- `test_layer_row` runs every distinct launch through fiConvGemm on random device operands (post-ReLU-like sources,
  signed upsampled and gradient sources, He-scaled weights) into NaN-filled outputs, and checks every element.
- The whole-forward tests check each conv step of the 4 x 1080p bench step against float64 computed from the step's own
  inputs as the plan stored them (fiNetCopyActivation), with the weights folded as engine.cu folds them: that covers
  the plan's wiring (tensor maps, arena offsets, concat and pad offsets, pooled outputs) at the benchmarked size. The
  stem, the fused `inc` kernel, the ragged last batch, arena reuse at 4K x 2 and the fp32-grade schedule follow.

The reference is float64 on the GPU: y = b + sum over the nine taps of shift(x, tap) @ W_tap (cuBLAS DGEMM), per image
and per band of rows, with the concat and F.pad built into the operand. Bars, per element:
- bf16 outputs: |got - ref| <= 2^-7 |ref| + 1e-5 A, A = |b| + sum |x||w|, the sum of the magnitudes of the output's
  terms, which fp32 accumulation error scales with. A is computed for every element (the same tap GEMMs on |x|, |w|),
  so the printed ratios are exact.
- the stem (bf16 hi/lo products): 2^-7 |ref| + 2^-14 A;
- fp32-grade (hi + lo) outputs: 2^-15 |ref| + 2^-14 A;
- head logits (fp32): 1e-5 (sum_c |hw_c| A_c + |hb|), on the unrounded conv result.
Pooled outputs must equal F.max_pool2d of the stored full-resolution tensor bit for bit, u8 outputs the postprocess of
the kernel's own logits. Each check prints its worst error/bar ratio.
"""
import ctypes as C
import time
from collections import OrderedDict, namedtuple

import pytest
import torch
import torch.nn.functional as F

from model import _engine as E
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu

ULP = 2.0 ** -7
K_BF16, K_STEM, K_FP32 = 1e-5, 2.0 ** -14, 2.0 ** -14      # coefficients of A
R_FP32 = 2.0 ** -15
BAND_ELEMS = 1 << 27                 # fp64 elements per band operand (1 GiB)
SELECTION_ENV = ("FI_CTA2", "FI_NO_HALO", "FI_BLOCK_N", "FI_FUSE_INC", "FI_ARENA_REUSE")


@pytest.fixture(autouse=True)
def default_selection(monkeypatch):
    """The kernels bench.py runs: no selection override from the environment."""
    for k in SELECTION_ENV:
        monkeypatch.delenv(k, raising=False)


@pytest.fixture(autouse=True)
def timed(request, cuda_device):
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    torch.cuda.synchronize()
    print(f"[{request.node.name}: {time.time() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB]")


# ------------------------------------------------------------------------------------------------ the schedules
Sched = namedtuple("Sched", "n_channels n_classes bilinear N H W precision")
SCHEDULES = {
    "video1080p": Sched(2, 1, False, 4, 1080, 1920, "bf16"),       # the step bench.py times
    "4k_eval": Sched(2, 1, False, 2, 2160, 3840, "bf16"),          # bench.py --workload 4k_eval, B = min(pairs, 2)
    "api256": Sched(2, 1, True, 1, 256, 256, "bf16"),              # load_model builds the bilinear network
    "config2_32x256": Sched(2, 1, False, 32, 256, 256, "bf16"),    # BASELINE config 2
    "bilinear1080p": Sched(2, 1, True, 4, 1080, 1920, "bf16"),     # bench.py --bilinear
    "rgb1080p": Sched(6, 3, False, 1, 1080, 1920, "bf16"),         # UNet(6, 3): the stand-alone stem
    "fp32_1080p": Sched(2, 1, False, 1, 1080, 1920, "fp32"),       # the fp32-grade mode
}
TRAIN_N, TRAIN_SIZE = 16, 256

# one fiConvGemm launch (the fields of fiConvDesc that select and shape it)
Row = namedtuple("Row", "c0 c1 h1 w1 off_y off_x n_total taps mode relu N H W precise n_classes")
# one step of the forward: name and kind as Net.profile() reports them, the conv row (None: stem / upsample), FLOPs
Launch = namedtuple("Launch", "name kind row flops")


def level_sizes(H, W):
    hs, ws = [H], [W]
    for _ in range(4):
        hs.append(hs[-1] // 2)
        ws.append(ws[-1] // 2)
    return hs, ws


def conv_names():
    """Step name -> (src0, src1, dst, pool) tensor names of the plan (engine.cu:fill_plan)."""
    t = {"inc.double_conv.3": ("inc.mid", None, "inc", "pool1")}
    for i in range(1, 5):
        t[f"down{i}.maxpool_conv.1.double_conv.0"] = (f"pool{i}", None, f"down{i}.mid", None)
        t[f"down{i}.maxpool_conv.1.double_conv.3"] = (f"down{i}.mid", None, f"down{i}", f"pool{i + 1}" if i < 4 else None)
    below, skips = "down4", ("down3", "down2", "down1", "inc")
    for k in range(1, 5):
        t[f"up{k}.up"] = (below, None, f"up{k}.up", None)
        t[f"up{k}.conv.double_conv.0"] = (skips[k - 1], f"up{k}.up", f"up{k}.mid", None)
        t[f"up{k}.conv.double_conv.3"] = (f"up{k}.mid", None, f"up{k}" if k < 4 else None, None)
        below = f"up{k}"
    return t


def schedule(s, fuse_inc=True):
    """Every launch of fiNetForward for schedule `s`, in order."""
    N, H, W = s.N, s.H, s.W
    precise = int(s.precision == "fp32")
    f = 2 if s.bilinear else 1
    hs, ws = level_sizes(H, W)
    enc = [64, 128, 256, 512, 1024 // f]
    out = []

    def conv(name, lvl, c0, n_total, mode, c1=0, h1=0, w1=0, taps=9, relu=1):
        h, w = hs[lvl], ws[lvl]
        off_y, off_x = ((h - h1) // 2, (w - w1) // 2) if c1 else (0, 0)
        row = Row(c0, c1, h1, w1, off_y, off_x, n_total, taps, mode, relu, N, h, w, precise,
                  s.n_classes if mode == E.EPI_HEAD else 0)
        fl = 2.0 * N * h * w * n_total * taps * (c0 + c1)
        if mode == E.EPI_HEAD:
            fl += 2.0 * N * h * w * 64 * s.n_classes
        return Launch(name, 1, row, fl)

    stem_fl = 2.0 * N * H * W * 64 * 9 * s.n_channels
    inc3 = conv("inc.double_conv.3", 0, 64, 64, E.EPI_STORE_POOL)
    if s.n_channels <= 2 and not precise and fuse_inc:
        out.append(Launch("inc.double_conv.0+3", 1, inc3.row, inc3.flops + stem_fl))
    else:
        out += [Launch("inc.double_conv.0", 0, None, stem_fl), inc3]
    for i in range(1, 5):
        out.append(conv(f"down{i}.maxpool_conv.1.double_conv.0", i, enc[i - 1], enc[i], E.EPI_STORE))
        out.append(conv(f"down{i}.maxpool_conv.1.double_conv.3", i, enc[i], enc[i],
                        E.EPI_STORE_POOL if i < 4 else E.EPI_STORE))
    up_in, up_out = [1024, 512, 256, 128], [512 // f, 256 // f, 128 // f, 64]
    below = enc[4]
    for i in range(4):
        lvl = 3 - i
        hl, wl = hs[lvl + 1], ws[lvl + 1]
        if s.bilinear:
            out.append(Launch(f"up{i + 1}.up", 2, None, 0.0))
        else:
            out.append(Launch(f"up{i + 1}.up", 1, Row(below, 0, 0, 0, 0, 0, 4 * (up_in[i] // 2), 1, E.EPI_CONVT, 0,
                                                      N, hl, wl, precise, 0), 2.0 * N * hl * wl * 4 * (up_in[i] // 2) * below))
        mid = up_in[i] // 2 if s.bilinear else up_out[i]
        out.append(conv(f"up{i + 1}.conv.double_conv.0", lvl, enc[lvl], mid, E.EPI_STORE, c1=up_in[i] // 2,
                        h1=2 * hl, w1=2 * wl))
        out.append(conv(f"up{i + 1}.conv.double_conv.3", lvl, mid, up_out[i], E.EPI_STORE if i < 3 else E.EPI_HEAD))
        below = up_out[i]
    return out


def train_rows(bilinear):
    """The 3x3 fiConvGemm launches of one TrainStep at 16 x 256^2: every conv but the stem with relu = 0 and a plain
    store, then the data gradient of each (flipped weights on dz, one launch per concat source)."""
    s = Sched(2, 1, bilinear, TRAIN_N, TRAIN_SIZE, TRAIN_SIZE, "bf16")
    fwd, dgrad = [], []
    for ln in schedule(s, fuse_inc=False):
        r = ln.row
        if r is None or r.taps != 9:
            continue
        fwd.append((ln.name, r._replace(mode=E.EPI_STORE, relu=0, off_y=0, off_x=0, n_classes=0)))
        for suffix, n_total in ((".dgrad", r.c0), (".dgrad1", r.c1)):
            if n_total:
                dgrad.append((ln.name + suffix, Row(r.n_total, 0, 0, 0, 0, 0, n_total, 9, E.EPI_STORE, 0, r.N, r.H, r.W,
                                                    0, 0)))
    return fwd, dgrad


def layer_params():
    """Distinct per-layer rows: (id, row, whether source 0 is signed)."""
    seen, params = set(), []
    for sname, s in SCHEDULES.items():
        for ln in schedule(s):
            if ln.row is not None and (ln.row, False) not in seen:
                seen.add((ln.row, False))
                params.append(pytest.param(ln.row, False, id=f"{sname}-{ln.name}"))
    for tag, bilinear in (("train-bilinear", True), ("train-convt", False)):
        fwd, dgrad = train_rows(bilinear)
        for signed, rows in ((False, fwd), (True, dgrad)):
            for name, row in rows:
                if (row, signed) not in seen:
                    seen.add((row, signed))
                    params.append(pytest.param(row, signed, id=f"{tag}-{name}"))
    return params


# ------------------------------------------------------------------------------------------------ guards
def _load_default(net, s):
    net.load_state_dict(O.init_state_dict(0, s.n_channels, s.n_classes, s.bilinear))


@pytest.mark.parametrize("sname", list(SCHEDULES))
def test_every_forward_launch_has_a_row(cuda_device, sname):
    s = SCHEDULES[sname]
    net = E.Net(cuda_device, s.n_channels, s.n_classes, s.bilinear, s.precision)
    _load_default(net, s)
    c = s.n_channels // 2
    x = torch.randint(0, 256, (s.N, c, s.H, s.W), dtype=torch.uint8, device=cuda_device)
    net.set_profiling(True)
    net.forward(x, x, want_f32=False, want_u8=True)
    prof = net.profile()
    net.close()
    derived = schedule(s)
    assert [p["name"] for p in prof] == [ln.name for ln in derived], "launch names or order differ from schedule()"
    for p, ln in zip(prof, derived):
        assert p["kind"] == ln.kind, (p["name"], p["kind"], ln.kind)
        assert p["flops"] == pytest.approx(ln.flops, rel=1e-12, abs=0), (p["name"], p["flops"], ln.flops)
    print(f"{sname}: {len(prof)} launches, {sum(ln.row is not None for ln in derived)} conv rows")


def test_every_train_step_conv3x3_has_a_row(cuda_device):
    """One TrainStep at 16 x 256^2 on the three networks of test_gpu_train_kernels_at_scale.py: every 3x3 fiConvGemm
    descriptor it launches must be one train_rows() derives."""
    from model.train import TrainStep
    from model.unet import FrameInterpolationUNet, UNet
    nets = {"grey bilinear": (lambda: FrameInterpolationUNet(bilinear=True).unet, True),
            "grey convt": (lambda: FrameInterpolationUNet(bilinear=False).unet, False),
            "UNet(6, 3)": (lambda: UNet(6, 3), False)}
    lib = E.lib()
    saved = lib.fiConvGemm
    for tag, (make, bilinear) in nets.items():
        torch.manual_seed(0)
        model = make().to(cuda_device).train()
        seen = []

        def wrapped(desc, stream):
            d = desc._obj
            if d.taps == 9:
                seen.append(Row(d.c0, d.c1, d.h1, d.w1, d.off_y, d.off_x, d.n_total, d.taps, d.mode, d.relu, d.N, d.H,
                                d.W, d.precise, d.n_classes))
            return saved(desc, stream)
        cin, ncls = model.inc.double_conv[0].in_channels, model.outc.conv.out_channels
        g = torch.Generator(device=cuda_device).manual_seed(0)
        x = torch.rand(TRAIN_N, cin, TRAIN_SIZE, TRAIN_SIZE, generator=g, device=cuda_device) * 2 - 1
        tgt = torch.rand(TRAIN_N, ncls, TRAIN_SIZE, TRAIN_SIZE, generator=g, device=cuda_device)
        lib.fiConvGemm = wrapped
        try:
            TrainStep(model, lr=0.0)(x, None, tgt)
            torch.cuda.synchronize()
        finally:
            lib.fiConvGemm = saved
        fwd, dgrad = train_rows(bilinear)
        want = sorted([r for _, r in fwd + dgrad])
        print(f"{tag}: {len(seen)} 3x3 launches")
        missing = [r for r in seen if r not in set(want)]
        assert not missing, f"{tag}: 3x3 launches without a row: {missing}"
        assert sorted(seen) == want, f"{tag}: the step launches {len(seen)} 3x3 convs, train_rows() derives {len(want)}"


# ------------------------------------------------------------------------------------------------ float64 reference
def split_bf16(t):
    hi = t.to(torch.bfloat16)
    return hi, (t - hi.float()).to(torch.bfloat16)


class Src:
    """One NHWC source of a conv: value = hi (+ lo), any float dtype; `off` places it in the output frame."""

    def __init__(self, hi, lo=None, off=(0, 0)):
        self.hi, self.lo, self.off = hi, lo, off
        self.c = hi.shape[3]

    def rows(self, img, a, b):
        v = self.hi[img, a:b].double()
        return v + self.lo[img, a:b].double() if self.lo is not None else v


def padded_band(srcs, img, r0, r1, H, W):
    """fp64 operand of output rows [r0, r1): rows r0-1 .. r1 of the zero-padded, concatenated input, flattened to
    [(R+2)*(W+2) + 2, Ctot] so that tap (dy, dx) is the contiguous slice starting at dy*(W+2) + dx."""
    R, ctot = r1 - r0, sum(s.c for s in srcs)
    dev = srcs[0].hi.device
    xp = torch.zeros((R + 2) * (W + 2) + 2, ctot, dtype=torch.float64, device=dev)
    view = xp[:(R + 2) * (W + 2)].view(R + 2, W + 2, ctot)
    c = 0
    for s in srcs:
        h, w = s.hi.shape[1], s.hi.shape[2]
        oy, ox = s.off
        lo, hi = max(r0 - 1, oy), min(r1 + 1, oy + h)        # frame rows of this source inside the band
        if hi > lo:
            view[lo - (r0 - 1):hi - (r0 - 1), 1 + ox:1 + ox + w, c:c + s.c] = s.rows(img, lo - oy, hi - oy)
        c += s.c
    return xp


def tap_gemms(xp, Wt, b, R, W):
    """b + sum_tap xp[shift] @ Wt[tap] over the padded width: [R, W, cout] (the two wrap-around columns dropped)."""
    y = b.expand(R * (W + 2), b.numel()).clone()
    for t in range(9):
        s = (t // 3) * (W + 2) + t % 3
        y.addmm_(xp[s:s + R * (W + 2)], Wt[t])
    return y.view(R, W + 2, -1)[:, :W]


class Worst:
    def __init__(self):
        self.ratio, self.where = 0.0, None

    def update(self, ratio, where):
        if ratio > self.ratio:
            self.ratio, self.where = ratio, where


def compare(what, got, ref, A, rel, kcoef, pos, worst):
    """Per element: |got - ref| <= rel |ref| + kcoef A; NaN fails. pos(idx) -> global positions for the message."""
    err = (got - ref).abs()
    bar = rel * ref.abs() + kcoef * A
    nan = torch.isnan(got)
    ratio = torch.where(err == 0, torch.zeros_like(err), err / bar.clamp_min(1e-300))
    ratio[nan] = float("inf")
    k = int(ratio.argmax())
    at = torch.stack(torch.unravel_index(torch.tensor(k), ratio.shape))[None]
    worst.update(ratio.flatten()[k].item(), pos(at)[0])
    fail = ratio > 1
    if fail.any():
        idx = fail.nonzero()[:5]
        first = [(pos(idx[j:j + 1])[0], got[tuple(idx[j])].item(), ref[tuple(idx[j])].item()) for j in range(len(idx))]
        raise AssertionError(f"{what}: {int(fail.sum())} elements beyond the bar (NaN: {int(nan.sum())}); "
                             f"first (image, y, x, channel) -> got, ref: {first}")
    return worst


def band_rows(H, W, width):
    return max(1, min(H, BAND_ELEMS // ((W + 2) * width)))


def check_conv3x3(what, srcs, Wt, b, got, *, relu=True, rel=ULP, kcoef=K_BF16, got_lo=None, worst=None):
    """got: [N, H, W, cout] (bf16, or hi with got_lo) against the fp64 conv of srcs. Returns the Worst record."""
    worst = worst or Worst()
    N, H, W, cout = got.shape
    Wabs, babs = Wt.abs(), b.abs()
    R = band_rows(H, W, max(Wt.shape[1], cout))
    for img in range(N):
        for r0 in range(0, H, R):
            r1 = min(H, r0 + R)
            xp = padded_band(srcs, img, r0, r1, H, W)
            ref = tap_gemms(xp, Wt, b, r1 - r0, W)
            if relu:
                ref = ref.clamp_min(0)
            g = got[img, r0:r1].double()
            if got_lo is not None:
                g = g + got_lo[img, r0:r1].double()

            A = tap_gemms(xp.abs_(), Wabs, babs, r1 - r0, W)
            del xp

            def pos(idx, img=img, r0=r0):
                return [(img, r0 + int(i[0]), int(i[1]), int(i[2])) for i in idx]
            compare(what, g, ref, A, rel, kcoef, pos, worst)
            del ref, g, A
    return worst


def check_convT(what, x, Wt, b, got, *, rel=ULP, kcoef=K_BF16, x_lo=None, got_lo=None, worst=None):
    """ConvTranspose2d(k=2, s=2) as the GEMM x[N,h,w,cin] @ Wt[(a,b,co), cin]^T scattered to [N, 2h, 2w, cout]."""
    worst = worst or Worst()
    N, h, w, cin = x.shape
    cout = Wt.shape[0] // 4
    Wabs, babs = Wt.abs(), b.abs().repeat(4)
    R = band_rows(h, w, max(cin, 4 * cout))
    for img in range(N):
        for r0 in range(0, h, R):
            r1 = min(h, r0 + R)
            X = x[img, r0:r1].double().reshape(-1, cin)
            if x_lo is not None:
                X = X + x_lo[img, r0:r1].double().reshape(-1, cin)
            y = (X @ Wt.t() + b.repeat(4)).view(r1 - r0, w, 2, 2, cout)
            ref = y.permute(0, 2, 1, 3, 4).reshape(2 * (r1 - r0), 2 * w, cout)
            g = got[img, 2 * r0:2 * r1].double()
            if got_lo is not None:
                g = g + got_lo[img, 2 * r0:2 * r1].double()

            A = (X.abs_() @ Wabs.t() + babs).view(r1 - r0, w, 2, 2, cout)
            A = A.permute(0, 2, 1, 3, 4).reshape(2 * (r1 - r0), 2 * w, cout)

            def pos(idx, img=img, r0=r0):
                return [(img, 2 * r0 + int(i[0]), int(i[1]), int(i[2])) for i in idx]
            compare(what, g, ref, A, rel, kcoef, pos, worst)
    return worst


def check_head(what, srcs, Wt, b, hw, hb, got_f32, got_u8=None, worst=None):
    """EPI_HEAD: fp32 logits [N, ncls, H, W] against the fp64 conv + ReLU (unrounded) and the fp64 1x1 head. Bar:
    1e-5 (sum_c |hw_c| A_c + |hb|). The u8 output must be postprocess of the kernel's own logits, bit for bit."""
    worst = worst or Worst()
    N, ncls, H, W = got_f32.shape
    hw64, hb64 = hw.double(), hb.double()
    R = band_rows(H, W, Wt.shape[1])
    for img in range(N):
        for r0 in range(0, H, R):
            r1 = min(H, r0 + R)
            xp = padded_band(srcs, img, r0, r1, H, W)
            y = tap_gemms(xp, Wt, b, r1 - r0, W).clamp_min(0)
            ref = y @ hw64.t() + hb64                                  # [R, W, ncls]
            A = tap_gemms(xp.abs_(), Wt.abs(), b.abs(), r1 - r0, W) @ hw64.abs().t() + hb64.abs()
            g = got_f32[img, :, r0:r1].permute(1, 2, 0).double()

            def pos(idx, img=img, r0=r0):
                return [(img, r0 + int(i[0]), int(i[1]), int(i[2])) for i in idx]
            compare(what, g, ref, A, 0.0, K_BF16, pos, worst)
    if got_u8 is not None:
        want = (((got_f32 + 1.0) / 2.0).clamp(0.0, 1.0) * 255).to(torch.uint8)
        bad = got_u8 != want
        assert not bad.any(), f"{what}: u8 output != postprocess(fp32 logits) at {int(bad.sum())} elements, first " \
                              f"(image, class, y, x) {bad.nonzero()[0].tolist()}"
    return worst


def check_pool(what, dst, pool, dst_lo=None, pool_lo=None):
    """The pooled tensor against F.max_pool2d (floor) of the stored full-resolution tensor: bit for bit in bf16; in
    the fp32-grade mode (hi + lo) within 2^-15 of the value."""
    if dst_lo is None:
        want = F.max_pool2d(dst.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        bad = pool.view(torch.int16) != want.view(torch.int16)
    else:
        full = dst.double() + dst_lo.double()
        want = F.max_pool2d(full.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        bad = ((pool.double() + pool_lo.double()) - want).abs() > R_FP32 * want.abs()
    assert pool.shape == want.shape, (what, pool.shape, want.shape)
    assert not bad.any(), f"{what}: pooled tensor != max_pool2d(stored tensor) at {int(bad.sum())} elements, first " \
                          f"(image, y, x, channel) {bad.nonzero()[0].tolist()}"


def report(what, worst):
    print(f"{what}: worst err/bar {worst.ratio:.3g} at {worst.where}")
    return worst.ratio


# ------------------------------------------------------------------------------------------------ per-layer rows
def launch_row(row, x0, x1, wpack, bias, x0_lo=None, x1_lo=None, head=None):
    """fiConvGemm of one row on device operands; outputs NaN-filled (fp32 logits) / zeroed (u8) before the launch."""
    dev = x0.device
    d = E.ConvDesc()
    for f in ("c0", "c1", "h1", "w1", "off_y", "off_x", "n_total", "taps", "mode", "relu", "N", "H", "W", "precise"):
        setattr(d, f, getattr(row, f))
    d.src0, d.wpack, d.bias = x0.data_ptr(), wpack.data_ptr(), bias.data_ptr()
    d.src1 = x1.data_ptr() if x1 is not None else None
    d.src0_lo = x0_lo.data_ptr() if x0_lo is not None else None
    d.src1_lo = x1_lo.data_ptr() if x1_lo is not None else None
    out = {}

    def nan_bf16(shape):
        return torch.full(shape, float("nan"), dtype=torch.bfloat16, device=dev)
    N, H, W = row.N, row.H, row.W
    if row.mode in (E.EPI_STORE, E.EPI_STORE_POOL, E.EPI_CONVT):
        shape = (N, 2 * H, 2 * W, row.n_total // 4) if row.mode == E.EPI_CONVT else (N, H, W, row.n_total)
        out["dst"] = nan_bf16(shape)
        d.dst = out["dst"].data_ptr()
        if row.precise:
            out["dst_lo"] = nan_bf16(shape)
            d.dst_lo = out["dst_lo"].data_ptr()
        if row.mode == E.EPI_STORE_POOL:
            out["pool"] = nan_bf16((N, H // 2, W // 2, row.n_total))
            d.dst_pool = out["pool"].data_ptr()
            if row.precise:
                out["pool_lo"] = nan_bf16((N, H // 2, W // 2, row.n_total))
                d.dst_pool_lo = out["pool_lo"].data_ptr()
    else:
        hw, hb = head
        out["f32"] = torch.full((N, hw.shape[0], H, W), float("nan"), dtype=torch.float32, device=dev)
        out["u8"] = torch.zeros((N, hw.shape[0], H, W), dtype=torch.uint8, device=dev)
        d.head_w, d.head_b, d.n_classes = hw.data_ptr(), hb.data_ptr(), hw.shape[0]
        d.out_f32, d.out_u8 = out["f32"].data_ptr(), out["u8"].data_ptr()
    with torch.cuda.device(dev):
        E.check(E.lib().fiConvGemm(C.byref(d), E.current_stream()))
    return out


def pack_weights(Wq, blocks, precise):
    """Wq: fp32 [rows, taps, Ctot] -> bf16 [rows, taps*K]; precise: per tap and source block [w_hi | w_lo | w_hi]."""
    if not precise:
        return Wq.reshape(Wq.shape[0], -1).to(torch.bfloat16).contiguous()
    parts, c = [], 0
    for nb in blocks:
        hi, lo = split_bf16(Wq[:, :, c:c + nb])
        parts.append(torch.cat([hi, lo, hi], 2))
        c += nb
    return torch.cat(parts, 2).reshape(Wq.shape[0], -1).contiguous()


def packed_value(Wq, precise):
    """fp64 value of the weights the kernel multiplies: bf16(w), or w_hi + w_lo."""
    hi, lo = split_bf16(Wq)
    return hi.double() + lo.double() if precise else hi.double()


def operand(g, shape, signed, precise, dev):
    x = torch.randn(shape, generator=g, device=dev)
    if not signed:
        x = x.clamp_min(0)
    return split_bf16(x) if precise else (x.to(torch.bfloat16), None)


def run_layer_row(row, signed0, seed=0):
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(seed + row.c0 + row.n_total + row.H + row.N)
    P = bool(row.precise)
    N, H, W = row.N, row.H, row.W
    x0, x0l = operand(g, (N, H, W, row.c0), signed0, P, dev)
    x1 = x1l = None
    if row.c1:
        x1, x1l = operand(g, (N, row.h1, row.w1, row.c1), True, P, dev)     # upsampled sources are signed
    ctot = row.c0 + row.c1
    Wq = torch.randn(row.n_total, row.taps, ctot, generator=g, device=dev) * (2.0 / (row.taps * ctot)) ** 0.5
    b = torch.randn(row.n_total, generator=g, device=dev) * 0.1
    head = None
    if row.mode == E.EPI_HEAD:
        ncls = row.n_classes
        head = (torch.randn(ncls, 64, generator=g, device=dev) * 0.3, torch.randn(ncls, generator=g, device=dev) * 0.2)
    if row.mode == E.EPI_CONVT:
        b = b[: row.n_total // 4].repeat(4).contiguous()
    blocks = [row.c0] + ([row.c1] if row.c1 else [])
    out = launch_row(row, x0, x1, pack_weights(Wq, blocks, P), b, x0l, x1l, head)
    torch.cuda.synchronize()
    rel, kc = (R_FP32, K_FP32) if P else (ULP, K_BF16)
    Wv, bv = packed_value(Wq, P), b.double()
    if row.mode == E.EPI_CONVT:
        w = check_convT("layer", x0, Wv[:, 0, :], bv[: row.n_total // 4], out["dst"], rel=rel, kcoef=kc, x_lo=x0l,
                        got_lo=out.get("dst_lo"))
        return w
    srcs = [Src(x0, x0l)] + ([Src(x1, x1l, (row.off_y, row.off_x))] if row.c1 else [])
    Wt = Wv.permute(1, 2, 0).contiguous()                                  # [9, Ctot, cout]
    if row.mode == E.EPI_HEAD:
        return check_head("layer", srcs, Wt, bv, head[0], head[1], out["f32"], out["u8"])
    w = check_conv3x3("layer", srcs, Wt, bv, out["dst"], relu=bool(row.relu), rel=rel, kcoef=kc,
                      got_lo=out.get("dst_lo"))
    if row.mode == E.EPI_STORE_POOL:
        check_pool("layer pool", out["dst"], out["pool"], out.get("dst_lo"), out.get("pool_lo"))
    return w


@pytest.mark.parametrize("row,signed0", layer_params())
def test_layer_row(cuda_device, request, row, signed0):
    """One distinct launch of the seven schedules or of the training step through fiConvGemm, every element checked."""
    try:
        w = run_layer_row(row, signed0)
    except AssertionError as e:
        raise AssertionError(f"{request.node.callspec.id}: {e}") from None
    report(request.node.callspec.id, w)


# ------------------------------------------------------------------------------------------------ whole forward
def sd_get(sd, key):
    return sd[key] if key in sd else sd["unet." + key]


def fold(sd, conv_key, precise, dev):
    """conv3x3 + BatchNorm(eval) as engine.cu folds them: s = gamma / sqrt(var + 1e-5) and w * s in fp64, then float,
    then bf16 (or the hi/lo pair); shift = float(beta - mu * s). Returns the fp32 weights [cout, tap, ci] to pack and
    the fp32 shift, on `dev`."""
    bn = conv_key[:-1] + str(int(conv_key[-1]) + 1)
    w = sd_get(sd, conv_key + ".weight").double()
    g, be = sd_get(sd, bn + ".weight").double(), sd_get(sd, bn + ".bias").double()
    mu, var = sd_get(sd, bn + ".running_mean").double(), sd_get(sd, bn + ".running_var").double()
    s = g / torch.sqrt(var + 1e-5)
    wf = (w * s[:, None, None, None]).float()                              # [cout, cin, 3, 3]
    Wq = wf.permute(0, 2, 3, 1).reshape(wf.shape[0], 9, wf.shape[1])     # [cout, tap, ci]
    return Wq.contiguous().to(dev), (be - mu * s).float().to(dev)


def convT_weights(sd, key, dev):
    """ConvTranspose2d weights fp32 [cin, cout, 2, 2] -> rows (a, b, co) [4 cout, 1, cin]; bias repeated per (a, b)."""
    w = sd_get(sd, key + ".weight").float()
    Wq = w.permute(2, 3, 1, 0).reshape(4 * w.shape[1], 1, w.shape[0])
    return Wq.contiguous().to(dev), sd_get(sd, key + ".bias").float().repeat(4).contiguous().to(dev)


def stressed_sd(n_channels, n_classes, x_first):
    """The stressed fixture (randomised BatchNorm, head calibrated to std 0.5 on the first pair); the calibration's
    oracle forward runs on the GPU."""
    sd = O.stress_state_dict(O.init_state_dict(0, n_channels, n_classes, False), seed=1)
    sd = O.calibrate_head(OrderedDict((k, v.to(x_first.device)) for k, v in sd.items()), x_first)
    return OrderedDict((k, v.cpu()) for k, v in sd.items())


def tap(net, name, n):
    t = net.activation(name, n)
    return t if isinstance(t, tuple) else (t, None)


def check_plan_steps(net, sd, s, n, out_f32, out_u8, tag, fused=True):
    """Every conv step of the current plan against fp64 from its own stored inputs. Each step's output must also be
    bit-identical to fiConvGemm of the same inputs with this file's fold, which pins the fold to the engine's."""
    P = s.precision == "fp32"
    rel, kc = (R_FP32, K_FP32) if P else (ULP, K_BF16)
    dev = out_f32.device
    names = conv_names()
    ratios = {}
    for ln in schedule(s, fuse_inc=fused):
        if ln.row is None or ln.name == "inc.double_conv.0+3":
            continue
        what = f"{tag} {ln.name}"
        src0, src1, dst, pool = names[ln.name]
        row = ln.row._replace(N=n)
        x0, x0l = tap(net, src0, n)
        x1, x1l = tap(net, src1, n) if src1 else (None, None)
        if row.mode == E.EPI_CONVT:
            Wq, bias = convT_weights(sd, ln.name, dev)
        else:
            Wq, bias = fold(sd, ln.name, P, dev)
        blocks = [row.c0] + ([row.c1] if row.c1 else [])
        Wv, bv = packed_value(Wq, P), bias.double()
        head = None
        if row.mode == E.EPI_HEAD:
            head = (sd_get(sd, "outc.conv.weight").reshape(-1, 64).float().to(dev),
                    sd_get(sd, "outc.conv.bias").float().to(dev))
        again = launch_row(row, x0, x1, pack_weights(Wq, blocks, P), bias, x0l, x1l, head)
        torch.cuda.synchronize()
        if row.mode == E.EPI_HEAD:
            assert torch.equal(again["f32"], out_f32), f"{what}: logits differ from fiConvGemm on the stored inputs"
            srcs = [Src(x0, x0l)] + ([Src(x1, x1l, (row.off_y, row.off_x))] if src1 else [])
            w = check_head(what, srcs, Wv.permute(1, 2, 0).contiguous(), bv, head[0], head[1], out_f32, out_u8)
            ratios[ln.name] = report(what, w)
            continue
        got, got_lo = tap(net, dst, n)
        assert torch.equal(again["dst"].view(torch.int16), got.view(torch.int16)), \
            f"{what}: the plan's output differs from fiConvGemm on its stored inputs with the test's fold"
        if P:
            assert torch.equal(again["dst_lo"].view(torch.int16), got_lo.view(torch.int16)), f"{what} (lo half)"
        if row.mode == E.EPI_CONVT:
            w = check_convT(what, x0, Wv[:, 0, :], bv[: row.n_total // 4], got, rel=rel, kcoef=kc, x_lo=x0l,
                            got_lo=got_lo)
        else:
            srcs = [Src(x0, x0l)] + ([Src(x1, x1l, (row.off_y, row.off_x))] if src1 else [])
            w = check_conv3x3(what, srcs, Wv.permute(1, 2, 0).contiguous(), bv, got, rel=rel, kcoef=kc, got_lo=got_lo)
        if pool:
            pv, pvl = tap(net, pool, n)
            check_pool(f"{what} pool", got, pv, got_lo, pvl)
        ratios[ln.name] = report(what, w)
    return ratios


def stem_reference_check(what, frames0, frames1, sd, got):
    """inc.mid (stem + BN + ReLU) against fp64 of the u8 frames normalised as preprocess_image, fp32 folded weights.
    Bar: 2^-7 |ref| + 2^-14 A (bf16 hi/lo products)."""
    w = sd_get(sd, "inc.double_conv.0.weight").double()
    g, be = sd_get(sd, "inc.double_conv.1.weight").double(), sd_get(sd, "inc.double_conv.1.bias").double()
    mu, var = sd_get(sd, "inc.double_conv.1.running_mean").double(), sd_get(sd, "inc.double_conv.1.running_var").double()
    s = g / torch.sqrt(var + 1e-5)
    wf = (w * s[:, None, None, None]).float().double()                    # fp32 folded weights
    shift = (be - mu * s).float().double()
    dev = got.device
    Wt = wf.permute(2, 3, 1, 0).reshape(9, wf.shape[1], 64).contiguous().to(dev)

    def norm(u8):   # preprocess_image: u8 / 255 in fp32, then 2a - 1
        return (2.0 * (u8.float() / 255.0) - 1.0).permute(0, 2, 3, 1).contiguous()
    x = torch.cat([norm(frames0), norm(frames1)], 3)
    return check_conv3x3(what, [Src(x)], Wt, shift.to(dev), got, kcoef=K_STEM)


@pytest.fixture(scope="module")
def bench_step(cuda_device):
    """The bench step (4 x 1080p, synthetic clip frames) on the stressed fixture, default (fused) schedule."""
    import bench
    fr = torch.from_numpy(bench.synthetic_frames(5)).to(cuda_device)
    f1, f2 = fr[:-1], fr[1:]
    xf = torch.cat([O.preprocess_u8(f1[:1].cpu().numpy()), O.preprocess_u8(f2[:1].cpu().numpy())], 1).to(cuda_device)
    sd = stressed_sd(2, 1, xf)
    return f1, f2, sd


def test_bench_step_every_conv_against_its_stored_inputs(cuda_device, bench_step):
    f1, f2, sd = bench_step
    s = SCHEDULES["video1080p"]
    net = E.Net(cuda_device, 2, 1, False)
    net.load_state_dict(sd)
    out_f, out_u = net.forward(f1, f2, want_f32=True, want_u8=True)
    assert out_f.min() < -1.0 and out_f.max() > 1.0, "the stressed fixture must reach both clamps"
    ratios = check_plan_steps(net, sd, s, 4, out_f, out_u, "video1080p")
    assert len(ratios) == 20
    net.close()


def test_bench_step_stem_and_fused_inc(cuda_device, bench_step, monkeypatch):
    """FI_FUSE_INC=0 runs the stem as its own launch: inc, pool1 and the output must be bit-identical to the fused
    kernel's; inc.mid must match the fp64 stem on the u8 frames, and inc fp64 from inc.mid."""
    f1, f2, sd = bench_step
    fused = E.Net(cuda_device, 2, 1, False)
    fused.load_state_dict(sd)
    want_f, want_u = fused.forward(f1, f2, want_f32=True, want_u8=True)
    fused_taps = {k: fused.activation(k, 4) for k in ("inc", "pool1")}
    monkeypatch.setenv("FI_FUSE_INC", "0")
    plain = E.Net(cuda_device, 2, 1, False)
    plain.load_state_dict(sd)
    got_f, got_u = plain.forward(f1, f2, want_f32=True, want_u8=True)
    assert plain.cost(4, 1080, 1920)[1] == 22 and fused.cost(4, 1080, 1920)[1] == 21
    for k, v in fused_taps.items():
        assert torch.equal(v.view(torch.int16), plain.activation(k, 4).view(torch.int16)), f"{k} differs"
    assert torch.equal(got_f, want_f) and torch.equal(got_u, want_u), "output differs"
    fused.close()
    mid = plain.activation("inc.mid", 4)
    report("video1080p stem inc.mid", stem_reference_check("video1080p stem", f1, f2, sd, mid))
    Wq, shift = fold(sd, "inc.double_conv.3", False, mid.device)
    inc = plain.activation("inc", 4)
    report("video1080p inc.double_conv.3", check_conv3x3("video1080p inc.double_conv.3", [Src(mid)],
                                                         packed_value(Wq, False).permute(1, 2, 0).contiguous(),
                                                         shift.double(), inc))
    check_pool("video1080p inc pool1", inc, plain.activation("pool1", 4))
    plain.close()


def test_rgb_stem(cuda_device):
    """UNet(6, 3): the stand-alone stem_mma_kernel<6, U8> on two BGR 1080p frames."""
    import bench
    fr = torch.from_numpy(bench.synthetic_frames(6)).to(cuda_device).view(2, 3, 1080, 1920)
    f1, f2 = fr[:1], fr[1:]
    xf = torch.cat([O.preprocess_u8(f1.cpu().numpy()), O.preprocess_u8(f2.cpu().numpy())], 1).to(cuda_device)
    sd = stressed_sd(6, 3, xf)
    net = E.Net(cuda_device, 6, 3, False)
    net.load_state_dict(sd)
    net.forward(f1, f2, want_f32=True)
    report("rgb1080p stem inc.mid", stem_reference_check("rgb1080p stem", f1, f2, sd, net.activation("inc.mid", 1)))
    net.close()


def test_ragged_last_batch_is_bit_identical(cuda_device, bench_step):
    """The video path's last batch: 3 pairs on the plan sized for 4 (fiNetForward recomputes the grids)."""
    f1, f2, sd = bench_step
    net = E.Net(cuda_device, 2, 1, False)
    net.load_state_dict(sd)
    want_f, want_u = (t.clone() for t in net.forward(f1, f2, want_f32=True, want_u8=True))
    got_f, got_u = net.forward(f1[:3], f2[:3], want_f32=True, want_u8=True)
    assert net.plan_stats()[:2] == (1, 1), "the 3-pair forward must run on the 4-pair plan"
    assert torch.equal(got_f, want_f[:3]) and torch.equal(got_u, want_u[:3])
    net.close()


def test_4k_arena_reuse_is_bit_identical(cuda_device, monkeypatch):
    """4K x 2 (bench.py --workload 4k_eval). With the fused inc the plain layout is 15.8 GiB, under the 16 GiB at which
    reuse switches on by itself; FI_FUSE_INC=0 adds inc.mid (17.7 GiB) and does switch it on. Every placement must give
    the same bytes."""
    import bench
    fr = torch.from_numpy(bench.synthetic_frames(3, h=2160, w=3840)).to(cuda_device)
    sd = O.stress_state_dict(O.init_state_dict(0, 2, 1, False), seed=1)

    def run(env):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        net = E.Net(cuda_device, 2, 1, False)
        net.load_state_dict(sd)
        out = [t.clone() for t in net.forward(fr[:2], fr[1:], want_f32=True, want_u8=True)]
        try:
            net.activation("pool4", 2)
            reuse = False
        except E.FiError as e:
            assert "taps are unavailable" in str(e)
            reuse = True
        nbytes = net.plan_stats()[2]
        net.close()
        for k in env:
            monkeypatch.delenv(k)
        return out, reuse, nbytes
    want, reuse, plain_bytes = run({})
    assert not reuse and plain_bytes < 16 * 2 ** 30
    for env in ({"FI_ARENA_REUSE": "1"}, {"FI_FUSE_INC": "0"}):
        got, reuse, nbytes = run(env)
        assert reuse and nbytes < plain_bytes, (env, nbytes, plain_bytes)
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), env
        print(f"4K x 2 {env}: arena {nbytes / 2 ** 30:.2f} GiB (plain, fused inc: {plain_bytes / 2 ** 30:.2f} GiB)")


def test_fp32_grade_schedule_every_conv(cuda_device):
    """fp32-grade 1 x 1080p: every conv step as hi + lo against fp64 from its stored hi + lo inputs."""
    import bench
    s = SCHEDULES["fp32_1080p"]
    fr = torch.from_numpy(bench.synthetic_frames(2)).to(cuda_device)
    xf = torch.cat([O.preprocess_u8(fr[:1].cpu().numpy()), O.preprocess_u8(fr[1:].cpu().numpy())], 1).to(cuda_device)
    sd = stressed_sd(2, 1, xf)
    net = E.Net(cuda_device, 2, 1, False, "fp32")
    net.load_state_dict(sd)
    out_f, out_u = net.forward(fr[:1], fr[1:], want_f32=True, want_u8=True)
    ratios = check_plan_steps(net, sd, s, 1, out_f, out_u, "fp32_1080p", fused=False)
    assert len(ratios) == 21
    net.close()


# ------------------------------------------------------------------------------------------------ the device tap
def test_copy_activation_matches_read_activation(cuda_device, monkeypatch):
    sd = O.stress_state_dict(O.init_state_dict(0, 2, 1, False), seed=2)
    g = torch.Generator(device=cuda_device).manual_seed(5)
    f1, f2 = (torch.randint(0, 256, (2, 1, 40, 72), generator=g, device=cuda_device, dtype=torch.uint8) for _ in "ab")
    for precision in ("bf16", "fp32"):
        net = E.Net(cuda_device, 2, 1, False, precision)
        net.load_state_dict(sd)
        net.forward(f1, f2, want_f32=True)
        for name in ("inc", "pool2", "down3.mid", "up1.up", "up2", "up4.mid"):
            t = net.activation(name, 2)
            hi, lo = t if precision == "fp32" else (t, None)
            v = hi.float() + (lo.float() if lo is not None else 0)
            want = net.read_activation(name, 2).to(cuda_device)
            assert torch.equal(v.permute(0, 3, 1, 2), want), (precision, name)
        with pytest.raises(E.FiError, match="no activation named"):
            net.activation("nope", 2)
        c, h, w = C.c_int(), C.c_int(), C.c_int()
        buf = torch.empty(10, dtype=torch.bfloat16, device=cuda_device)
        with pytest.raises(E.FiError, match="buffer too small"):
            E.check(E.lib().fiNetCopyActivation(net._h, b"inc", buf.data_ptr(), buf.data_ptr(), buf.numel(),
                                                C.byref(c), C.byref(h), C.byref(w), E.current_stream()))
        if precision == "fp32":
            with pytest.raises(E.FiError, match="dst_lo is required"):
                E.check(E.lib().fiNetCopyActivation(net._h, b"inc", buf.data_ptr(), None, buf.numel(), None, None,
                                                    None, E.current_stream()))
        net.close()
    monkeypatch.setenv("FI_ARENA_REUSE", "1")
    lean = E.Net(cuda_device, 2, 1, False)
    lean.load_state_dict(sd)
    lean.forward(f1, f2, want_f32=True)
    with pytest.raises(E.FiError, match="taps are unavailable"):
        lean.activation("inc", 2)
    lean.close()
