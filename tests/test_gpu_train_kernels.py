"""Unit parity of the training-step kernels (through the C ABI) against torch autograd on identical bf16 inputs."""
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

from model import _engine as E

pytestmark = pytest.mark.gpu


def nhwc(t, dev):
    return t.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16).to(dev)


def nchw(t):
    return t.float().cpu().permute(0, 3, 1, 2).contiguous()


def p(t):
    return C.c_void_p(t.data_ptr())


@pytest.mark.parametrize("n,c,h,w", [(2, 64, 9, 11), (1, 256, 8, 8), (3, 1024, 3, 5)])
def test_bn_relu_forward_backward(cuda_device, n, c, h, w):
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(c + h)
    z = (torch.randn(n, c, h, w, generator=g) * 1.5 + 0.3).to(torch.bfloat16).float()
    dA = (torch.randn(n, c, h, w, generator=g)).to(torch.bfloat16).float()
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g) * 0.1
    # torch reference
    zr = z.clone().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    a_ref = F.relu(F.batch_norm(zr, None, None, gr, br, True, 0.0, 1e-5))
    a_ref.backward(dA)
    # kernels
    P = n * h * w
    zd, dAd = nhwc(z, cuda_device), nhwc(dA, cuda_device)
    stats = torch.zeros(2, c, device=cuda_device)
    E.check(lib.fiBnStats(p(zd), P, c, p(stats[0]), p(stats[1]), st))
    mean = stats[0] / P
    var = stats[1] / P - mean * mean
    assert torch.allclose(mean.cpu(), z.mean((0, 2, 3)), atol=1e-4)
    assert torch.allclose(var.cpu(), z.var((0, 2, 3), unbiased=False), rtol=1e-3, atol=1e-4)
    rstd = torch.rsqrt(var + 1e-5)
    gd, bd = gamma.to(cuda_device), beta.to(cuda_device)
    scale, shift = gd * rstd, bd - mean * gd * rstd
    a = torch.empty_like(zd)
    E.check(lib.fiBnApplyRelu(p(zd), P, c, p(scale), p(shift), p(a), st))
    assert (nchw(a) - a_ref.detach()).abs().max() <= 2.0 ** -7 * a_ref.abs().max() + 1e-3
    # backward recomputes the ReLU mask from z with the forward's scale / shift
    red = torch.zeros(2, c, device=cuda_device)
    E.check(lib.fiBnReluBackwardReduce(p(dAd), p(zd), P, c, p(mean), p(rstd), p(scale), p(shift), p(red[0]), p(red[1]), st))
    dz = torch.empty_like(zd)
    E.check(lib.fiBnReluBackwardApply(p(dAd), p(zd), P, c, p(mean), p(rstd), p(gd), p(bd), p(red[0]), p(red[1]), p(dz), st))
    torch.cuda.synchronize()
    assert torch.allclose(red[0].cpu(), br.grad, rtol=2e-3, atol=2e-3), "dbeta"
    assert torch.allclose(red[1].cpu(), gr.grad, rtol=2e-3, atol=2e-3), "dgamma"
    err = (nchw(dz) - zr.grad).abs().max().item()
    assert err <= 2.0 ** -7 * zr.grad.abs().max().item() + 1e-3, err


@pytest.mark.parametrize("n,c,h,w", [(2, 64, 8, 10), (1, 128, 9, 7)])
def test_maxpool_backward_with_skip(cuda_device, n, c, h, w):
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(h * w)
    a = torch.randn(n, c, h, w, generator=g).to(torch.bfloat16).float()
    d_pool = torch.randn(n, c, h // 2, w // 2, generator=g).to(torch.bfloat16).float()
    d_skip = torch.randn(n, c, h, w, generator=g).to(torch.bfloat16).float()
    ar = a.clone().requires_grad_(True)
    F.max_pool2d(ar, 2).backward(d_pool)
    ref = ar.grad + d_skip
    ad = nhwc(a, cuda_device)
    pooled = torch.empty((n, h // 2, w // 2, c), dtype=torch.bfloat16, device=cuda_device)
    E.check(lib.fiMaxPool2x2(p(ad), p(pooled), n, h, w, c, st))
    out = torch.full((n, h, w, c), float("nan"), dtype=torch.bfloat16, device=cuda_device)
    dpd, dsd = nhwc(d_pool, cuda_device), nhwc(d_skip, cuda_device)
    E.check(lib.fiMaxPoolBackwardAdd(p(ad), p(pooled), p(dpd), p(dsd), p(out), n, h, w, c, st))
    torch.cuda.synchronize()
    assert (nchw(out) - ref).abs().max() <= 2.0 ** -7 * ref.abs().max() + 1e-3


@pytest.mark.parametrize("n,c,h,w", [(2, 64, 4, 6), (1, 128, 1, 3), (1, 64, 8, 8)])
def test_upsample_backward(cuda_device, n, c, h, w):
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(h + w)
    d_up = torch.randn(n, c, 2 * h, 2 * w, generator=g).to(torch.bfloat16).float()
    x = torch.zeros(n, c, h, w, requires_grad=True)
    F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True).backward(d_up)
    out = torch.empty((n, h, w, c), dtype=torch.bfloat16, device=cuda_device)
    dud = nhwc(d_up, cuda_device)
    E.check(lib.fiUpsample2xBackward(p(dud), p(out), n, h, w, c, st))
    torch.cuda.synchronize()
    assert (nchw(out) - x.grad).abs().max() <= 2.0 ** -7 * x.grad.abs().max() + 1e-3


def test_head_forward_backward_and_mse(cuda_device):
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(1)
    n, h, w, ncls = 2, 6, 9, 2
    a = torch.randn(n, 64, h, w, generator=g).to(torch.bfloat16).float()
    wt, b = torch.randn(ncls, 64, generator=g) * 0.3, torch.randn(ncls, generator=g)
    tgt = torch.randn(n, ncls, h, w, generator=g)
    ar, wr, br = a.clone().requires_grad_(True), wt.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y_ref = F.conv2d(ar, wr[:, :, None, None], br)
    loss_ref = F.mse_loss(y_ref, tgt)
    loss_ref.backward()
    ad = nhwc(a, cuda_device)
    wd, bd, td = wt.to(cuda_device), b.to(cuda_device), tgt.to(cuda_device)
    y = torch.empty((n, ncls, h, w), device=cuda_device)
    E.check(lib.fiHeadForward(p(ad), n, h * w, p(wd), p(bd), ncls, p(y), st))
    loss = torch.zeros(1, device=cuda_device)
    dy = torch.empty_like(y)
    E.check(lib.fiMseLossGrad(p(y), p(td), y.numel(), p(loss), p(dy), st))
    da = torch.empty_like(ad)
    dw, db = torch.zeros(ncls, 64, device=cuda_device), torch.zeros(ncls, device=cuda_device)
    E.check(lib.fiHeadBackward(p(ad), p(dy), n, h * w, p(wd), ncls, p(da), p(dw), p(db), st))
    torch.cuda.synchronize()
    assert torch.allclose(y.cpu(), y_ref.detach(), atol=1e-4)
    assert abs(loss.item() - loss_ref.item()) < 1e-5
    assert torch.allclose(dw.cpu(), wr.grad, rtol=1e-3, atol=1e-5) and torch.allclose(db.cpu(), br.grad, rtol=1e-3, atol=1e-6)
    assert (nchw(da) - ar.grad).abs().max() <= 2.0 ** -7 * ar.grad.abs().max() + 1e-6


def test_adam_and_weight_packing(cuda_device):
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(2)
    prm = torch.randn(1000, generator=g)
    ref = prm.clone().requires_grad_(True)
    opt = torch.optim.Adam([ref], lr=1e-2)
    pd, m, v = prm.to(cuda_device), torch.zeros(1000, device=cuda_device), torch.zeros(1000, device=cuda_device)
    for step in range(1, 4):
        grad = torch.randn(1000, generator=g)
        ref.grad = grad.clone()
        opt.step()
        gd = grad.to(cuda_device)
        E.check(lib.fiAdamStep(p(pd), p(gd), p(m), p(v), 1000, 1e-2, 0.9, 0.999, 1e-8, step, None, st))
    assert torch.allclose(pd.cpu(), ref.detach(), rtol=1e-5, atol=1e-6)
    w = torch.randn(128, 64, 3, 3, generator=g)
    fwd = torch.empty((128, 9 * 64), dtype=torch.bfloat16, device=cuda_device)
    bwd = torch.empty((64, 9 * 128), dtype=torch.bfloat16, device=cuda_device)
    wd = w.to(cuda_device)
    E.check(lib.fiPackConvWeights(p(wd), 128, 64, p(fwd), p(bwd), st))
    wb = w.to(torch.bfloat16)
    assert torch.equal(fwd.cpu(), wb.permute(0, 2, 3, 1).reshape(128, -1))
    assert torch.equal(bwd.cpu(), wb.flip(2, 3).permute(1, 2, 3, 0).reshape(64, -1))


def test_data_gradient_is_a_conv_with_flipped_weights(cuda_device):
    """dX = conv_transpose(dz, W) computed by the forward conv kernel on fiPackConvWeights' bwd rows."""
    from layer_utils import from_nhwc
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(4)
    n, cin, cout, h, w = 2, 128, 64, 10, 12
    wt = torch.randn(cout, cin, 3, 3, generator=g) * 0.05
    dz = torch.randn(n, cout, h, w, generator=g).to(torch.bfloat16).float()
    bwd = torch.empty((cin, 9 * cout), dtype=torch.bfloat16, device=cuda_device)
    wtd = wt.to(cuda_device)
    E.check(lib.fiPackConvWeights(p(wtd), cout, cin, None, p(bwd), st))
    dzd = nhwc(dz, cuda_device)
    dst = torch.empty((n, h, w, cin), dtype=torch.bfloat16, device=cuda_device)
    zero = torch.zeros(cin, device=cuda_device)
    d = E.ConvDesc()
    d.src0, d.c0, d.N, d.H, d.W = dzd.data_ptr(), cout, n, h, w
    d.wpack, d.bias, d.n_total, d.taps, d.mode, d.relu, d.dst = bwd.data_ptr(), zero.data_ptr(), cin, 9, 0, 0, dst.data_ptr()
    E.check(lib.fiConvGemm(C.byref(d), st))
    torch.cuda.synchronize()
    ref = F.conv_transpose2d(dz.double(), wt.to(torch.bfloat16).double(), padding=1).float()
    assert (from_nhwc(dst) - ref).abs().max() <= 2.0 ** -7 * ref.abs().max() + 1e-3


@pytest.mark.parametrize("n,cin,h,w", [(2, 2, 9, 12), (1, 6, 8, 8), (3, 1, 5, 7)])
def test_stem_weight_gradient(cuda_device, n, cin, h, w):
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(cin * 10 + h)
    x = torch.rand(n, cin, h, w, generator=g) * 2 - 1
    dz = torch.randn(n, 64, h, w, generator=g).to(torch.bfloat16).float()
    wt = torch.zeros(64, cin, 3, 3, requires_grad=True)
    F.conv2d(x, wt, padding=1).backward(dz)
    xd, dzd = x.to(cuda_device), nhwc(dz, cuda_device)
    prior = torch.randn(64, cin, 3, 3, generator=g).to(cuda_device)
    dW = prior.clone()
    E.check(lib.fiStemWgrad(p(dzd), p(xd), n, h, w, cin, p(dW), st))
    torch.cuda.synchronize()
    assert torch.allclose((dW - prior).cpu(), wt.grad, rtol=1e-4, atol=1e-4)
    assert lib.fiStemWgrad(p(dzd), p(xd), n, h, w, 5, p(dW), st) != 0


def test_bn_finalize_and_running_statistics(cuda_device):
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(8)
    n, c, h, w = 3, 192, 5, 6   # C/8 = 24 does not divide 256: the unpacked reduction walk
    z = (torch.randn(n, c, h, w, generator=g) * 2 + 0.5).to(torch.bfloat16).float()
    bn = torch.nn.BatchNorm2d(c)
    bn.weight.data, bn.bias.data = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g)
    bn.running_mean.data, bn.running_var.data = torch.randn(c, generator=g), torch.rand(c, generator=g) + 0.5
    rm, rv = bn.running_mean.clone().to(cuda_device), bn.running_var.clone().to(cuda_device)
    bn.train()
    ref = bn(z)
    P = n * h * w
    zd = nhwc(z, cuda_device)
    work = torch.zeros(6, c, device=cuda_device)
    gd, bd = bn.weight.detach().to(cuda_device), bn.bias.detach().to(cuda_device)
    E.check(lib.fiBnStats(p(zd), P, c, p(work[0]), p(work[1]), st))
    E.check(lib.fiBnFinalize(p(work[0]), p(work[1]), c, P, bn.eps, 0.1, p(gd), p(bd), p(work[2]), p(work[3]), p(work[4]),
                             p(work[5]), p(rm), p(rv), st))
    torch.cuda.synchronize()
    assert torch.allclose(rm.cpu(), bn.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(rv.cpu(), bn.running_var, rtol=1e-3, atol=1e-5)
    got = nchw(zd.float() * work[4] + work[5])
    assert torch.allclose(got, ref.detach(), rtol=1e-3, atol=2e-3)


def test_bn_shifted_finalize_and_running_statistics(cuda_device):
    """The pair TrainStep runs: sums about each channel's first pixel, then the finalize that adds it back."""
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(8)
    n, c, h, w = 3, 192, 5, 6   # C/8 = 24 does not divide 256: the unpacked reduction walk
    z = (torch.randn(n, c, h, w, generator=g) * 2 + 0.5).to(torch.bfloat16).float()
    bn = torch.nn.BatchNorm2d(c)
    bn.weight.data, bn.bias.data = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g)
    bn.running_mean.data, bn.running_var.data = torch.randn(c, generator=g), torch.rand(c, generator=g) + 0.5
    rm, rv = bn.running_mean.clone().to(cuda_device), bn.running_var.clone().to(cuda_device)
    bn.train()
    ref = bn(z)
    P = n * h * w
    zd = nhwc(z, cuda_device)
    work = torch.zeros(7, c, device=cuda_device)   # sum, sumsq, mean, rstd, scale, shift, pivot
    gd, bd = bn.weight.detach().to(cuda_device), bn.bias.detach().to(cuda_device)
    E.check(lib.fiBnStatsShifted(p(zd), P, c, p(work[6]), p(work[0]), p(work[1]), st))
    E.check(lib.fiBnFinalizeShifted(p(work[0]), p(work[1]), p(work[6]), c, P, bn.eps, 0.1, p(gd), p(bd), p(work[2]),
                                    p(work[3]), p(work[4]), p(work[5]), p(rm), p(rv), st))
    torch.cuda.synchronize()
    assert torch.equal(work[6].cpu(), z[0, :, 0, 0]), "pivot = the first pixel"
    assert torch.allclose(rm.cpu(), bn.running_mean, rtol=1e-4, atol=1e-5)
    assert torch.allclose(rv.cpu(), bn.running_var, rtol=1e-3, atol=1e-5)
    got = nchw(zd.float() * work[4] + work[5])
    assert torch.allclose(got, ref.detach(), rtol=1e-3, atol=2e-3)


def test_unpack_conv_grad(cuda_device):
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(6)
    dW = torch.randn(9, 128, 64, generator=g).to(cuda_device)
    grad = torch.randn(128, 64, 3, 3, generator=g).to(cuda_device)
    want = grad + dW.permute(1, 2, 0).reshape(128, 64, 3, 3)
    E.check(lib.fiUnpackConvGrad(p(dW), 128, 64, p(grad), st))
    torch.cuda.synchronize()
    assert torch.allclose(grad, want, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("planes,h,w,mw,sw", [(2, 40, 56, 0.5, 0.5), (3, 32, 32, 0.3, 0.7), (1, 7, 9, 1.0, 1.0),
                                               (4, 70, 33, 0.0, 1.0)])
def test_combined_loss_kernel_matches_torch(cuda_device, planes, h, w, mw, sw):
    """fiCombinedLossGrad against autograd of the CombinedLoss mirror (itself pinned to the reference by
    tests/test_train_loss.py)."""
    from model.train import CombinedLoss
    lib, st = E.lib(), E.current_stream()
    g = torch.Generator().manual_seed(planes * 100 + h)
    pred = torch.rand(planes, 1, h, w, generator=g).requires_grad_(True)
    target = (pred.detach() + 0.15 * torch.randn(planes, 1, h, w, generator=g)).clamp(0, 1)
    loss_ref = CombinedLoss(mw, sw)(pred, target)
    loss_ref.backward()
    yd, td = pred.detach().to(cuda_device), target.to(cuda_device)
    loss = torch.zeros(1, device=cuda_device)
    dy = torch.full_like(yd, float("nan"))
    E.check(lib.fiCombinedLossGrad(p(yd), p(td), planes, h, w, mw, sw, p(loss), p(dy), st))
    torch.cuda.synchronize()
    assert abs(loss.item() - loss_ref.item()) < 2e-6 + 1e-5 * abs(loss_ref.item())
    err = (dy.cpu() - pred.grad).abs().max().item()
    assert err <= 2e-3 * pred.grad.abs().max().item() + 1e-9, (err, pred.grad.abs().max().item())
