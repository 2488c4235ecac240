"""GPU tier of the colour metric: fiSsimPsnrPlanesU8 against the colour restatement of scikit-image's metrics at every
size and in all four layout combinations (planar / interleaved for each operand, bit-identical to each other), the C = 1
call bit for bit against fiSsimPsnrU8, C = 3 against fiSsimPsnrU8 on the extracted planes, the colour closed forms,
every argument error, and compute_* on BGR arrays."""
import ctypes as C

import numpy as np
import pytest
import torch

from model import _engine as E
from oracle import metrics_oracle as M
from test_color_metrics import ALL_ROWS, CASES, psnr_color, ssim_color

pytestmark = pytest.mark.gpu

SIZES = [(7, 7), (16, 16), (135, 241), (256, 256), (1080, 1920), (2160, 3840)]


def bgr_pair(h, w, n, seed):
    """n BGR pairs [n,H,W,3]: a smooth pattern against a noisy copy, a random pair, and 0 / 255 extremes."""
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    a, b = [], []
    for i in range(n):
        base = np.stack([(127 + 100 * np.sin(xx / (7.0 + 3 * c + i)) * np.cos(yy / 9.0)) for c in range(3)], -1)
        base = base.astype(np.uint8)
        noisy = np.clip(base.astype(np.int16) + rs.randint(-20, 21, base.shape), 0, 255).astype(np.uint8)
        a.append(base)
        b.append(noisy)
    a[-1][..., 2] = rs.randint(0, 256, (h, w))
    b[-1][..., 1] = 255
    return np.stack(a), np.stack(b)


def layouts(x_hwc, dev):
    """The same pixels [n,H,W,3] as a planar [n,3,H,W] tensor and as the interleaved view of a channels-last one."""
    t = torch.from_numpy(x_hwc).to(dev)
    return {"planar": t.permute(0, 3, 1, 2).contiguous(), "interleaved": t.permute(0, 3, 1, 2)}


@pytest.mark.parametrize("h,w", SIZES)
def test_planes_kernel_against_oracle_in_every_layout(cuda_device, h, w):
    pred, target = bgr_pair(h, w, 2, h * 31 + w)
    lp, lt = layouts(pred, cuda_device), layouts(target, cuda_device)
    assert lt["interleaved"].stride()[3] == 3 and lt["planar"].stride()[3] == 1
    outs = {(a, b): E.ssim_psnr_planes_u8(lp[a], lt[b]).cpu().numpy() for a in lp for b in lt}
    first = outs[("planar", "interleaved")]
    for k, o in outs.items():
        assert np.array_equal(o.view(np.int64), first.view(np.int64)), k     # bit-identical across layouts
    for i in range(2):
        assert abs(first[i, 1] - ssim_color(pred[i], target[i])) <= 1e-4, ("ssim", i)
        assert abs(first[i, 0] - psnr_color(pred[i], target[i])) <= 1e-9, ("psnr", i)


def grey_call(a, b):
    return E.ssim_psnr_u8(a, b).cpu().numpy()


def test_one_channel_is_the_grey_call_bit_for_bit(cuda_device):
    rs = np.random.RandomState(5)
    for h, w in [(7, 7), (37, 530), (135, 241), (1080, 1920)]:
        a = torch.from_numpy(rs.randint(0, 256, (3, h, w)).astype(np.uint8)).to(cuda_device)
        b = torch.from_numpy(rs.randint(0, 256, (3, h, w)).astype(np.uint8)).to(cuda_device)
        b[0] = a[0]
        got = E.ssim_psnr_planes_u8(a[:, None], b[:, None]).cpu().numpy()
        assert np.array_equal(got.view(np.int64), grey_call(a, b).view(np.int64)), (h, w)
    for row in CASES:
        p = torch.tensor(row["pred"], dtype=torch.uint8, device=cuda_device)[None]
        t = torch.tensor(row["target"], dtype=torch.uint8, device=cuda_device)[None]
        got = E.ssim_psnr_planes_u8(p[:, None], t[:, None]).cpu().numpy()
        assert np.array_equal(got.view(np.int64), grey_call(p, t).view(np.int64)), row["name"]


@pytest.mark.parametrize("h,w", [(16, 16), (135, 241), (1080, 1920)])
def test_three_channels_are_the_mean_of_the_plane_calls(cuda_device, h, w):
    pred, target = bgr_pair(h, w, 2, 7 * h + w)
    got = E.ssim_psnr_planes_u8(layouts(pred, cuda_device)["planar"], layouts(target, cuda_device)["interleaved"])
    got = got.cpu().numpy()
    planes_p = torch.from_numpy(np.ascontiguousarray(pred.transpose(0, 3, 1, 2).reshape(-1, h, w))).to(cuda_device)
    planes_t = torch.from_numpy(np.ascontiguousarray(target.transpose(0, 3, 1, 2).reshape(-1, h, w))).to(cuda_device)
    per_plane = grey_call(planes_p, planes_t).reshape(2, 3, 2)
    for i in range(2):
        assert abs(got[i, 1] - per_plane[i, :, 1].mean()) <= 1e-12
        sse = sum(h * w * 255.0 ** 2 / 10 ** (p / 10) for p in per_plane[i, :, 0])
        assert abs(got[i, 0] - 10 * np.log10(255.0 ** 2 * 3 * h * w / sse)) <= 1e-9


@pytest.mark.parametrize("name,pred,target,ssim,psnr", ALL_ROWS, ids=[r[0] for r in ALL_ROWS])
def test_colour_closed_forms(cuda_device, name, pred, target, ssim, psnr):
    lp, lt = layouts(pred[None], cuda_device), layouts(target[None], cuda_device)
    got = E.ssim_psnr_planes_u8(lp["planar"], lt["interleaved"]).cpu().numpy()[0]
    assert abs(got[1] - ssim) <= 1e-4
    assert (got[0] == psnr == np.inf) or abs(got[0] - psnr) <= 1e-4


def test_invalid_arguments_name_the_argument_and_write_nothing(cuda_device):
    n, h, w = 2, 16, 24
    p = torch.zeros((n, 3, h, w), dtype=torch.uint8, device=cuda_device)
    t = torch.zeros((n, h, w, 3), dtype=torch.uint8, device=cuda_device)
    ws = torch.empty(E.lib().fiSsimPsnrPlanesWorkspaceBytes(n, 3, h, w), dtype=torch.uint8, device=cuda_device)
    out = torch.full((n, 2), float("nan"), dtype=torch.float64, device=cuda_device)
    good_p, good_t = E.planes_of(p), E.planes_of(t.permute(0, 3, 1, 2))

    def call(pp, tt, nn=n, hh=h, ww=w, o=out.data_ptr(), wsp=ws.data_ptr()):
        return E.check(E.lib().fiSsimPsnrPlanesU8(pp, tt, nn, hh, ww, o, wsp, E.current_stream()))

    def planes(base, **kw):
        q = E.Planes(base.ptr, base.batch_stride, base.chan_stride, base.row_stride, base.px_stride, base.channels)
        for k, v in kw.items():
            setattr(q, k, v)
        return C.byref(q)

    cases = [
        ((None, C.byref(good_t)), {}, "null pred or target descriptor"),
        ((planes(good_p, ptr=None), C.byref(good_t)), {}, "null pred or target pointer"),
        ((C.byref(good_p), C.byref(good_t)), {"o": None}, "null out or workspace"),
        ((C.byref(good_p), C.byref(good_t)), {"wsp": None}, "null out or workspace"),
        ((planes(good_p, channels=1), C.byref(good_t)), {}, "channel counts differ"),
        ((planes(good_p, channels=2), planes(good_t, channels=2, px_stride=1)), {}, "channels must be 1 or 3"),
        ((planes(good_p, px_stride=2), C.byref(good_t)), {}, "pred layout"),
        ((C.byref(good_p), planes(good_t, chan_stride=2)), {}, "target layout"),
        ((C.byref(good_p), planes(good_t, row_stride=-72)), {}, "target layout"),
        ((C.byref(good_p), C.byref(good_t)), {"hh": 6}, "H and W must be >= 7"),
        ((C.byref(good_p), C.byref(good_t)), {"ww": 6}, "H and W must be >= 7"),
        ((C.byref(good_p), C.byref(good_t)), {"nn": 21846}, "too many planes"),
        ((C.byref(good_p), C.byref(good_t)), {"nn": 0}, "empty batch"),
    ]
    for (pp, tt), kw, msg in cases:
        with pytest.raises(E.FiError, match=msg):
            call(pp, tt, **kw)
    torch.cuda.synchronize()
    assert torch.isnan(out).all()
    call(C.byref(good_p), C.byref(good_t))
    assert torch.isinf(out[:, 0]).all() and (out[:, 1] == 1.0).all()


def test_compute_functions_on_bgr_arrays(cuda_device):
    from model import evaluation
    pred, target = bgr_pair(40, 57, 3, 11)
    psnr, ssim = evaluation.compute_metrics(pred, target)
    for i in range(3):
        assert abs(ssim[i] - ssim_color(pred[i], target[i])) <= 1e-4
        assert abs(psnr[i] - psnr_color(pred[i], target[i])) <= 1e-9
    assert abs(evaluation.compute_ssim(pred[0], target[0]) - ssim_color(pred[0], target[0])) <= 1e-4
    assert abs(evaluation.compute_psnr(pred[0], target[0]) - psnr_color(pred[0], target[0])) <= 1e-9
    # grey inputs still take the grey path, unchanged
    g = grey_call(torch.from_numpy(pred[..., 0]).to(cuda_device), torch.from_numpy(target[..., 0]).to(cuda_device))
    assert np.array_equal(np.stack(evaluation.compute_metrics(pred[..., 0], target[..., 0]), 1), g)
    assert evaluation.compute_ssim(pred[0, ..., 0], target[0, ..., 0]) == g[0, 1]
    assert abs(evaluation.compute_ssim(pred[0, ..., 0], target[0, ..., 0]) - M.ssim_u8(pred[0, ..., 0], target[0, ..., 0])) <= 1e-4
