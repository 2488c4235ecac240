"""Parity of the CUDA-core kernels (through the C ABI) against the oracle: stem conv, bilinear upsample, frame-pair
packing, post-processing (bit-exact byte work) and SSIM/PSNR (|err| <= 1e-4, north star)."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from model import _engine as E
from oracle import metrics_oracle as M
from oracle import unet_oracle as O

pytestmark = pytest.mark.gpu


def test_pack_pair_bit_exact(cuda_device):
    g = torch.Generator().manual_seed(0)
    allv = torch.arange(256, dtype=torch.uint8).view(1, 1, 16, 16)  # every input value, exhaustively
    got = E.pack_pair_u8(allv.to(cuda_device), allv.flip(3).to(cuda_device)).cpu()
    assert torch.equal(got, torch.cat([O.preprocess_u8(allv.numpy()), O.preprocess_u8(allv.flip(3).numpy())], 1))
    for shape in [(2, 1, 32, 48), (1, 3, 17, 19), (1, 1, 1080, 1920)]:
        f1 = torch.randint(0, 256, shape, generator=g, dtype=torch.uint8)
        f2 = torch.randint(0, 256, shape, generator=g, dtype=torch.uint8)
        got = E.pack_pair_u8(f1.to(cuda_device), f2.to(cuda_device)).cpu()
        exp = torch.cat([O.preprocess_u8(f1.numpy()), O.preprocess_u8(f2.numpy())], 1)
        assert torch.equal(got, exp)


def test_head_post_bit_exact(cuda_device):
    t = torch.cat([torch.linspace(-1.5, 1.5, 100003), torch.tensor([-1.0, 1.0, 0.0, 0.9999999, float(np.nextafter(1, 0))])])
    got = E.head_post_u8(t.to(cuda_device)).cpu().numpy()
    assert np.array_equal(got, O.postprocess(t))
    t2 = torch.randn(3, 1, 33, 35)  # unaligned tail
    assert np.array_equal(E.head_post_u8(t2.to(cuda_device)).cpu().numpy(), O.postprocess(t2))


@pytest.mark.parametrize("n,c,h,w", [(1, 64, 4, 7), (2, 128, 16, 15), (1, 512, 1, 1)])
def test_upsample2x(cuda_device, n, c, h, w):
    x = torch.randn(n, c, h, w).to(torch.bfloat16)
    src = x.permute(0, 2, 3, 1).contiguous().to(cuda_device)
    dst = torch.empty((n, 2 * h, 2 * w, c), dtype=torch.bfloat16, device=cuda_device)
    E.check(E.lib().fiUpsample2x(src.data_ptr(), dst.data_ptr(), n, h, w, c, E.current_stream()))
    torch.cuda.synchronize()
    ref = F.interpolate(x.float(), scale_factor=2, mode="bilinear", align_corners=True)
    got = dst.float().cpu().permute(0, 3, 1, 2)
    assert (got - ref).abs().max() <= 2.0 ** -7 * ref.abs().max() + 1e-6


@pytest.mark.parametrize("cin,u8,h,w", [(2, False, 33, 47), (2, True, 16, 64), (6, False, 20, 40), (1, True, 9, 9),
                                        (8, False, 17, 31), (3, True, 40, 200), (2, True, 270, 480)])
def test_stem_conv(cuda_device, cin, u8, h, w):
    g = torch.Generator().manual_seed(cin + h)
    n = 2
    if u8:
        frames = torch.randint(0, 256, (n, cin, h, w), generator=g, dtype=torch.uint8)
        x = O.preprocess_u8(frames.numpy())
        src = frames.to(cuda_device)
    else:
        x = torch.rand(n, cin, h, w, generator=g) * 2 - 1
        src = x.to(cuda_device)
    wt = torch.randn(64, cin, 3, 3, generator=g) * 0.3
    b = torch.randn(64, generator=g) * 0.1
    kp = E.lib().fiStemPackedK(cin)
    packed = torch.empty((64, kp), dtype=torch.int16)
    wc = wt.contiguous()
    E.check(E.lib().fiStemPackWeights(wc.data_ptr(), cin, packed.data_ptr()))
    wk = packed.to(cuda_device)  # bf16 bit patterns [64][kp]: [w_hi | w_lo | w_hi | 0]
    bd = b.to(cuda_device)
    dst = torch.empty((n, h, w, 64), dtype=torch.bfloat16, device=cuda_device)
    # split the channels over two plane groups like FrameInterpolationUNet.forward(frame1, frame2) does
    c_a = (cin + 1) // 2
    p0 = E.planes_of(src[:, :c_a])
    p1 = E.planes_of(src[:, c_a:]) if cin > c_a else None
    E.check(E.lib().fiStemConv(C.byref(p0), C.byref(p1) if p1 is not None else None, int(u8), wk.data_ptr(),
                               bd.data_ptr(), dst.data_ptr(), n, h, w, E.current_stream()))
    torch.cuda.synchronize()
    ref = F.relu(F.conv2d(x.double(), wt.double(), b.double(), padding=1)).float()
    got = dst.float().cpu().permute(0, 3, 1, 2)
    # hi/lo operand splitting keeps the pre-rounding value at fp32 grade: the only error left is the bf16 output cast
    assert ((got - ref).abs() <= 2.0 ** -8 * ref.abs() + 1e-4).all(), (got - ref).abs().max()


def degrade(a, rs, amp):
    return np.clip(a.astype(np.int32) + rs.randint(-amp, amp + 1, size=a.shape), 0, 255).astype(np.uint8)


@pytest.mark.parametrize("h,w", [(7, 7), (8, 13), (64, 64), (37, 530), (256, 256), (135, 241), (1080, 1920)])
def test_ssim_psnr_vs_oracle(cuda_device, h, w):
    rs = np.random.RandomState(h * 7 + w)
    yy, xx = np.mgrid[0:h, 0:w]
    base = (127 + 100 * np.sin(xx / 9.0) * np.cos(yy / 7.0)).astype(np.uint8)
    imgs_a = np.stack([base, rs.randint(0, 256, size=(h, w)).astype(np.uint8), np.full((h, w), 255, np.uint8)])
    imgs_b = np.stack([degrade(base, rs, 12), rs.randint(0, 256, size=(h, w)).astype(np.uint8),
                       np.zeros((h, w), np.uint8)])
    out = E.ssim_psnr_u8(torch.from_numpy(imgs_a).to(cuda_device), torch.from_numpy(imgs_b).to(cuda_device)).cpu().numpy()
    for i in range(3):
        assert abs(out[i, 0] - M.psnr_u8(imgs_a[i], imgs_b[i])) <= 1e-4, ("psnr", i)
        assert abs(out[i, 1] - M.ssim_u8(imgs_a[i], imgs_b[i])) <= 1e-4, ("ssim", i)


def test_ssim_psnr_identical_and_properties(cuda_device):
    rs = np.random.RandomState(1)
    a = rs.randint(0, 256, size=(2, 90, 130)).astype(np.uint8)
    ta = torch.from_numpy(a).to(cuda_device)
    out = E.ssim_psnr_u8(ta, ta).cpu().numpy()
    assert np.isinf(out[:, 0]).all() and np.allclose(out[:, 1], 1.0, atol=1e-6)
    # symmetry in the two arguments, and determinism
    b = torch.from_numpy(degrade(a, rs, 30)).to(cuda_device)
    o1 = E.ssim_psnr_u8(ta, b).cpu().numpy()
    o2 = E.ssim_psnr_u8(b, ta).cpu().numpy()
    o3 = E.ssim_psnr_u8(ta, b).cpu().numpy()
    assert np.allclose(o1, o2, atol=1e-12) and np.array_equal(o1, o3)
    from model._engine import FiError
    with pytest.raises(FiError):
        E.ssim_psnr_u8(ta[:, :6], ta[:, :6])


def test_host_buffer_entry_point(cuda_device):
    sd = O.init_state_dict(0, 2, 1, False)
    net = E.Net(cuda_device, 2, 1, False)
    net.load_state_dict(sd)
    rs = np.random.RandomState(0)
    f1 = rs.randint(0, 256, size=(2, 1, 48, 64)).astype(np.uint8)
    f2 = rs.randint(0, 256, size=(2, 1, 48, 64)).astype(np.uint8)
    out = net.interpolate_host_u8(f1, f2)
    _, dev = net.forward(torch.from_numpy(f1).to(cuda_device), torch.from_numpy(f2).to(cuda_device),
                         want_f32=False, want_u8=True)
    assert np.array_equal(out, dev.cpu().numpy())
    ref = O.postprocess(O.unet_forward(sd, torch.cat([O.preprocess_u8(f1), O.preprocess_u8(f2)], 1)))
    assert np.abs(out.astype(int) - ref.astype(int)).max() <= 2


def test_clip_pipeline_matches_pairwise_calls(cuda_device):
    """The midpoint clip (interpolate_clip_host_u8: the pipelined host-clip call at depth 1, as the video loop runs
    it) == the synchronous per-batch entry point, bit for bit, including a ragged last batch."""
    sd = O.init_state_dict(0, 2, 1, False)
    net = E.Net(cuda_device, 2, 1, False)
    net.load_state_dict(sd)
    rs = np.random.RandomState(3)
    clip = rs.randint(0, 256, size=(12, 1, 40, 56)).astype(np.uint8)
    ref = net.interpolate_host_u8(clip[:-1], clip[1:])
    for b in (1, 3, 4, 16):
        out = net.interpolate_clip_host_u8(clip, pairs_per_batch=b)
        assert out.shape == (11, 1, 40, 56) and np.array_equal(out, ref), b


def _metrics_golden():
    import json
    from pathlib import Path
    return json.loads((Path(__file__).parent / "golden" / "metrics_golden.json").read_text())


@pytest.mark.parametrize("row", _metrics_golden()["cases"], ids=lambda r: r["name"])
def test_ssim_psnr_kernel_against_closed_forms(cuda_device, row):
    """fiSsimPsnrU8 and the compute_psnr / compute_ssim drop-ins against the hand-derived exact values of
    tests/golden/metrics_golden.json (north-star bar: within 1e-4 of model/evaluation.py:194-218)."""
    from model import evaluation
    pred, target = np.array(row["pred"], np.uint8), np.array(row["target"], np.uint8)
    out = E.ssim_psnr_u8(torch.from_numpy(pred).to(cuda_device), torch.from_numpy(target).to(cuda_device)).cpu().numpy()[0]
    want_psnr = float("inf") if row["psnr"] == "inf" else row["psnr"]
    if want_psnr == float("inf"):
        assert out[0] == float("inf") and evaluation.compute_psnr(pred, target) == float("inf")
        assert abs(out[1] - 1.0) <= 1e-6
    else:
        assert abs(out[0] - want_psnr) <= 1e-4
        assert abs(evaluation.compute_psnr(pred, target) - want_psnr) <= 1e-4
    assert abs(out[1] - row["ssim"]) <= 1e-4
    assert abs(evaluation.compute_ssim(pred, target) - row["ssim"]) <= 1e-4
    # batched with a second, different pair: results do not leak between images
    both = E.ssim_psnr_u8(torch.from_numpy(np.stack([pred, target])).to(cuda_device),
                          torch.from_numpy(np.stack([target, target])).to(cuda_device)).cpu().numpy()
    assert abs(both[0, 1] - row["ssim"]) <= 1e-4 and abs(both[1, 1] - 1.0) <= 1e-6 and both[1, 0] == float("inf")


def test_ssim_error_rows(cuda_device):
    from model import evaluation
    for row in _metrics_golden()["errors"]:
        z = np.zeros(row["shape"], np.uint8)
        with pytest.raises((E.FiError, ValueError)):
            evaluation.compute_ssim(z, z)
