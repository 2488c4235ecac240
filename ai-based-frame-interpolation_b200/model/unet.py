"""Drop-in for the reference's model/unet.py: same class names, constructor signatures, state-dict keys and tensor
contracts, but forward() runs on the B200-native library (libfi_b200.so) instead of eager torch ops.

The nn.Module objects below are parameter containers only: they exist so that `.state_dict()`,
`.load_state_dict()`, `.parameters()`, `.to(device)` and `.eval()` behave exactly like the reference
(state-dict schema: SURVEY.md A.5 / reference model/unet.py:5-112). The arithmetic lives in csrc/:
  DoubleConv / Down / Up / OutConv   -> conv_gemm.cu (tcgen05 implicit GEMM, BN folded, pool / concat / head fused)
  first conv of `inc`                -> aux_kernels.cu stem kernel (frame-pair cat + normalisation fused)
There is no CPU fallback. forward() is the inference path (eval mode); the training-mode forward + backward + Adam
of the reference's train.py is model/train.py:TrainStep, which works on these same modules' parameters.
"""
from __future__ import annotations

import torch
import torch.nn as nn

try:  # imported as `model.unet` (main.py) or as top-level `unet` with model/ on sys.path (reference scripts)
    from . import _engine as _E
except ImportError:  # pragma: no cover - depends on how the caller set sys.path
    import _engine as _E


def _conv_bn_relu_slots(cin, cout):
    """Parameter slots of one conv3x3(no bias) + BatchNorm2d + ReLU stage (indices 0,1,2 / 3,4,5 of double_conv)."""
    return [nn.Conv2d(cin, cout, kernel_size=3, padding=1, bias=False), nn.BatchNorm2d(cout), nn.ReLU(inplace=True)]


# ----------------------------------------------------------------------------------------------------------------------
# Stand-alone use of the building blocks (DoubleConv / Down / Up / OutConv called on their own, as the reference allows).
# Inside UNet.forward none of this runs: the whole schedule is one fiNetForward call. Here each block is a handful of
# single-layer C-ABI calls (fiStemConv / fiConvGemm / fiMaxPool2x2 / fiUpsample2x); torch only converts the caller's
# NCHW fp32 tensors to the kernels' NHWC bf16 layout and back, and folds the (tiny) BatchNorm vectors.
# ----------------------------------------------------------------------------------------------------------------------
import ctypes as _C


def _to_nhwc(x):
    return x.detach().permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def _to_nchw(y):
    return y.permute(0, 3, 1, 2).contiguous().to(torch.float32)


def _fold_bn(conv, bn):
    """Eval-mode BatchNorm folded into the conv (reference model/unet.py:12-17): W*s, beta - mean*s."""
    scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
    w = conv.weight.detach().double() * scale[:, None, None, None]
    b = bn.bias.detach().double() - bn.running_mean.detach().double() * scale
    return w.float(), b.float().contiguous()


def _run_conv(x, w, bias, *, x1=None, off=(0, 0), taps=9, mode=_E.EPI_STORE, relu=True):
    """x (and x1): NHWC bf16 CUDA tensors; w: folded fp32 weight [cout, cin, k, k] (or packed rows for ConvT)."""
    n, h, wd, c0 = x.shape
    d = _E.ConvDesc()
    d.src0, d.c0, d.N, d.H, d.W = x.data_ptr(), c0, n, h, wd
    keep = [x]
    if x1 is not None:
        d.src1, d.c1, d.h1, d.w1 = x1.data_ptr(), x1.shape[3], x1.shape[1], x1.shape[2]
        d.off_y, d.off_x = off
        keep.append(x1)
    if mode == _E.EPI_CONVT:   # w: [cin, cout, 2, 2] -> rows (ky, kx, co), K = ci
        cout = w.shape[1]
        wp = w.permute(2, 3, 1, 0).reshape(4 * cout, w.shape[0])
        b = bias.repeat(4)
        n_total, out_shape = 4 * cout, (n, 2 * h, 2 * wd, cout)
    else:                      # w: [cout, cin, k, k] -> [cout, tap*cin + ci]
        wp = w.permute(0, 2, 3, 1).reshape(w.shape[0], -1)
        b = bias
        n_total, out_shape = w.shape[0], (n, h, wd, w.shape[0])
    wp = wp.contiguous().to(torch.bfloat16)
    b = b.contiguous().float()
    dst = torch.empty(out_shape, dtype=torch.bfloat16, device=x.device)
    keep += [wp, b]
    d.wpack, d.bias, d.n_total, d.taps, d.mode, d.relu, d.dst = (wp.data_ptr(), b.data_ptr(), n_total, taps, mode,
                                                                 int(relu), dst.data_ptr())
    with torch.cuda.device(x.device):
        _E.check(_E.lib().fiConvGemm(_C.byref(d), _E.current_stream()))
    return dst


def _check_standalone(x, module):
    _E.require_cuda(x.device)
    if module.training:
        raise _E.FiError("forward() is the inference path: call .eval() first (training: model.train.TrainStep)")
    if x.dtype != torch.float32 or x.dim() != 4:
        raise _E.FiError("expected an fp32 NCHW tensor")


def _double_conv_nhwc(dc, x_nchw=None, x_nhwc=None, x1_nhwc=None, off=(0, 0)):
    """The two conv+BN+ReLU stages of a DoubleConv. Input either NCHW fp32 with <= 8 channels (stem kernel) or NHWC
    bf16 with a multiple of 64 channels (optionally a second, padded source = the fused concat of Up)."""
    seq = dc.double_conv
    w1, b1 = _fold_bn(seq[0], seq[1])
    w2, b2 = _fold_bn(seq[3], seq[4])
    if w1.shape[0] % 64 or w2.shape[0] % 64:
        raise _E.FiError("stand-alone blocks need output channel counts that are multiples of 64")
    if x_nchw is not None:
        n, cin, h, w = x_nchw.shape
        if cin > 8 or w1.shape[0] != 64:
            raise _E.FiError("a raw-input DoubleConv needs <= 8 input channels and 64 mid channels (the stem kernel); "
                             "other inputs must have a multiple of 64 channels")
        kp = _E.lib().fiStemPackedK(cin)
        packed = torch.empty((64, kp), dtype=torch.int16)
        wc = w1.cpu().contiguous()
        _E.check(_E.lib().fiStemPackWeights(wc.data_ptr(), cin, packed.data_ptr()))
        packed = packed.to(x_nchw.device)
        mid = torch.empty((n, h, w, 64), dtype=torch.bfloat16, device=x_nchw.device)
        p0 = _E.planes_of(x_nchw)
        with torch.cuda.device(x_nchw.device):
            _E.check(_E.lib().fiStemConv(_C.byref(p0), None, _E.FI_IN_F32, packed.data_ptr(), b1.data_ptr(),
                                         mid.data_ptr(), n, h, w, _E.current_stream()))
    else:
        mid = _run_conv(x_nhwc, w1, b1, x1=x1_nhwc, off=off)
    return _run_conv(mid, w2, b2)


def _entry_nhwc(x, dc):
    """NCHW fp32 -> what _double_conv_nhwc wants for this channel count."""
    if x.shape[1] % 64 == 0:
        return dict(x_nhwc=_to_nhwc(x))
    return dict(x_nchw=x.detach().contiguous())


class _EngineBacked(nn.Module):
    """Mixin: lazily mirrors this module's parameters into a fiNet handle and re-uploads when they change.

    `module.precision` selects the arithmetic: "bf16" (default; bf16 operands, fp32 accumulate, <= 2e-2 pixel error) or
    "fp32" (hi/lo-split bf16 operands, three products per MAC: fp32-grade, <= 1e-3; about 3x slower)."""

    precision = "bf16"

    def _engine_spec(self):  # (n_channels, n_classes, bilinear)
        raise NotImplementedError

    def _fingerprint(self):
        return tuple((t.data_ptr(), t._version) for t in self.state_dict(keep_vars=True).values())

    def _engine(self, device):
        if self.training:
            raise _E.FiError("forward() is the inference path: call .eval() first; the training-mode forward, "
                             "backward and Adam step are model.train.TrainStep")
        net = self.__dict__.get("_fi_net")
        if net is None or net.device != device or net.precision != self.precision:
            if net is not None:
                net.close()
            n_ch, n_cls, bil = self._engine_spec()
            net = _E.Net(device, n_ch, n_cls, bil, self.precision)
            self.__dict__["_fi_net"] = net
            self.__dict__["_fi_print"] = None
        fp = self._fingerprint()
        if self.__dict__.get("_fi_print") != fp:
            net.load_state_dict(self.state_dict())
            self.__dict__["_fi_print"] = fp
        return net

    def _device_of(self, x):
        dev = _E.require_cuda(x.device)
        p = next(self.parameters())
        if p.device != x.device:
            raise _E.FiError(f"module parameters are on {p.device} but the input is on {x.device}")
        return torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())


class DoubleConv(nn.Module):
    """(conv3x3 => BatchNorm => ReLU) * 2 — reference model/unet.py:5-21."""

    def __init__(self, in_channels, out_channels, mid_channels=None):
        super().__init__()
        mid = mid_channels if mid_channels else out_channels
        self.double_conv = nn.Sequential(*(_conv_bn_relu_slots(in_channels, mid) + _conv_bn_relu_slots(mid, out_channels)))

    def forward(self, x):
        _check_standalone(x, self)
        return _to_nchw(_double_conv_nhwc(self, **_entry_nhwc(x, self)))


class Down(nn.Module):
    """MaxPool2d(2) then DoubleConv — reference model/unet.py:23-33 (the pool is fused into the producer's epilogue)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.maxpool_conv = nn.Sequential(nn.MaxPool2d(2), DoubleConv(in_channels, out_channels))

    def forward(self, x):
        _check_standalone(x, self)
        if x.shape[1] % 8:
            raise _E.FiError("stand-alone Down needs a multiple of 8 input channels")
        xs = _to_nhwc(x)
        n, h, w, c = xs.shape
        pooled = torch.empty((n, h // 2, w // 2, c), dtype=torch.bfloat16, device=x.device)
        with torch.cuda.device(x.device):
            _E.check(_E.lib().fiMaxPool2x2(xs.data_ptr(), pooled.data_ptr(), n, h, w, c, _E.current_stream()))
        dc = self.maxpool_conv[1]
        if c % 64:
            return _to_nchw(_double_conv_nhwc(dc, x_nchw=_to_nchw(pooled)))
        return _to_nchw(_double_conv_nhwc(dc, x_nhwc=pooled))


class Up(nn.Module):
    """Upscale, pad to the skip size, concat [skip, up], DoubleConv — reference model/unet.py:35-55."""

    def __init__(self, in_channels, out_channels, bilinear=True):
        super().__init__()
        if bilinear:
            self.up = nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True)
            self.conv = DoubleConv(in_channels, out_channels, in_channels // 2)
        else:
            self.up = nn.ConvTranspose2d(in_channels, in_channels // 2, kernel_size=2, stride=2)
            self.conv = DoubleConv(in_channels, out_channels)

    def forward(self, x1, x2):
        _check_standalone(x1, self)
        _check_standalone(x2, self)
        if x1.shape[1] % 64 or x2.shape[1] % 64:
            raise _E.FiError("stand-alone Up needs channel counts that are multiples of 64")
        lo = _to_nhwc(x1)
        n, h, w, c = lo.shape
        if isinstance(self.up, nn.ConvTranspose2d):
            up = _run_conv(lo, self.up.weight.detach().float(), self.up.bias.detach().float(), taps=1,
                           mode=_E.EPI_CONVT, relu=False)
        else:
            up = torch.empty((n, 2 * h, 2 * w, c), dtype=torch.bfloat16, device=x1.device)
            with torch.cuda.device(x1.device):
                _E.check(_E.lib().fiUpsample2x(lo.data_ptr(), up.data_ptr(), n, h, w, c, _E.current_stream()))
        skip = _to_nhwc(x2)
        off = ((skip.shape[1] - up.shape[1]) // 2, (skip.shape[2] - up.shape[2]) // 2)  # F.pad, unet.py:49-53
        return _to_nchw(_double_conv_nhwc(self.conv, x_nhwc=skip, x1_nhwc=up, off=off))


class OutConv(nn.Module):
    """1x1 output head — reference model/unet.py:57-63 (fused into the last conv's epilogue)."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.conv = nn.Conv2d(in_channels, out_channels, kernel_size=1)

    def forward(self, x):
        _check_standalone(x, self)
        if x.shape[1] % 64:
            raise _E.FiError("stand-alone OutConv needs a multiple of 64 input channels")
        ncls = self.conv.out_channels
        w = torch.zeros((64, x.shape[1], 1, 1), dtype=torch.float32, device=x.device)  # GEMM N is a multiple of 64
        b = torch.zeros(64, dtype=torch.float32, device=x.device)
        w[:ncls] = self.conv.weight.detach().float()
        b[:ncls] = self.conv.bias.detach().float()
        y = _run_conv(_to_nhwc(x), w, b, taps=1, relu=False)
        return _to_nchw(y[..., :ncls])


class UNet(_EngineBacked):
    """reference model/unet.py:65-95: widths 64-128-256-512-1024, four Down / four Up stages, 1x1 head."""

    def __init__(self, n_channels=2, n_classes=1, bilinear=False):
        super().__init__()
        self.n_channels, self.n_classes, self.bilinear = n_channels, n_classes, bilinear
        factor = 2 if bilinear else 1
        self.inc = DoubleConv(n_channels, 64)
        self.down1 = Down(64, 128)
        self.down2 = Down(128, 256)
        self.down3 = Down(256, 512)
        self.down4 = Down(512, 1024 // factor)
        self.up1 = Up(1024, 512 // factor, bilinear)
        self.up2 = Up(512, 256 // factor, bilinear)
        self.up3 = Up(256, 128 // factor, bilinear)
        self.up4 = Up(128, 64, bilinear)
        self.outc = OutConv(64, n_classes)

    def _engine_spec(self):
        return self.n_channels, self.n_classes, self.bilinear

    @torch.no_grad()
    def forward(self, x):
        """x: fp32 (normalised) or uint8 (raw) NCHW CUDA tensor -> fp32 logits [N, n_classes, H, W]."""
        net = self._engine(self._device_of(x))
        out, _ = net.forward(x, None, want_f32=True)
        return out

    @torch.no_grad()
    def forward_u8(self, x0, x1=None):
        """Raw uint8 planes in, post-processed uint8 frame out (normalisation and postprocess_image fused)."""
        net = self._engine(self._device_of(x0))
        _, out = net.forward(x0, x1, want_f32=False, want_u8=True)
        return out


class FrameInterpolationUNet(_EngineBacked):
    """reference model/unet.py:97-112: cat([frame1, frame2], 1) -> UNet(2, 1). The cat is fused into the stem loader."""

    def __init__(self, bilinear=False):
        super().__init__()
        self.unet = UNet(n_channels=2, n_classes=1, bilinear=bilinear)

    def _engine_spec(self):
        return 2, 1, self.unet.bilinear

    @torch.no_grad()
    def forward(self, frame1, frame2):
        """frame1, frame2: [B,1,H,W] fp32 in [-1,1] (or raw uint8) on the GPU -> [B,1,H,W] fp32."""
        net = self._engine(self._device_of(frame1))
        out, _ = net.forward(frame1, frame2, want_f32=True)
        return out

    @torch.no_grad()
    def forward_u8(self, frame1, frame2):
        net = self._engine(self._device_of(frame1))
        _, out = net.forward(frame1, frame2, want_f32=False, want_u8=True)
        return out


def model_from_state_dict(state):
    """The architecture a checkpoint's state dict was saved from, read off its keys and shapes: bilinear vs
    ConvTranspose2d decoder, input channels (2 grey, 6 colour) and classes. Returns (model, state) with a fresh module
    of that architecture, FrameInterpolationUNet for a wrapped 2->1 model, else UNet, and the state dict keyed for it
    (the `unet.` prefix of a wrapped colour model stripped); the weights are not loaded."""
    prefix = "unet." if any(k.startswith("unet.") for k in state) else ""
    bilinear = (prefix + "up1.up.weight") not in state
    n_channels = state[prefix + "inc.double_conv.0.weight"].shape[1]
    n_classes = state[prefix + "outc.conv.weight"].shape[0]
    if prefix and (n_channels, n_classes) == (2, 1):
        return FrameInterpolationUNet(bilinear=bilinear), state
    state = {k[len(prefix):]: v for k, v in state.items()} if prefix else state
    return UNet(n_channels, n_classes, bilinear), state


def architecture_name(model):
    """How `main.py info` names a model: FrameInterpolationUNet(bilinear=...) or UNet(n_channels, n_classes, ...)."""
    if isinstance(model, FrameInterpolationUNet):
        return f"FrameInterpolationUNet(bilinear={model.unet.bilinear})"
    return f"UNet(n_channels={model.n_channels}, n_classes={model.n_classes}, bilinear={model.bilinear})"


def count_parameters(model):
    """Number of trainable parameters — reference model/unet.py:114-116."""
    return sum(p.numel() for p in model.parameters() if p.requires_grad)
