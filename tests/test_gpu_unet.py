"""Whole-network parity: the drop-in UNet (CUDA path through the C ABI) against the CPU oracle on identical random-init
weights and synthetic inputs.

Tolerances (BASELINE.json north_star): bf16 path max |err| <= 2e-2 in [0,1] pixel units and PSNR >= 45 dB. The reference
output is in [-1,1] units (postprocess maps (y+1)/2), so logits are compared at half scale. The default-init fixture is
nearly constant (SURVEY.md D8), hence the additional relative-error bounds per tapped layer and the stressed fixture."""
import numpy as np
import pytest
import torch

from oracle import unet_oracle as O
from model.unet import UNet, FrameInterpolationUNet

pytestmark = pytest.mark.gpu


def psnr_unit(a, b):
    mse = float(((a - b) ** 2).mean())
    return 99.0 if mse == 0 else 10 * np.log10(1.0 / mse)


def build(sd, device, n_channels=2, n_classes=1, bilinear=False, wrapper=True):
    m = FrameInterpolationUNet(bilinear=bilinear) if wrapper else UNet(n_channels, n_classes, bilinear)
    m.load_state_dict(sd)
    return m.to(device).eval()


def frames(seed, n, c, h, w):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (n, c, h, w), generator=g, dtype=torch.uint8)


@pytest.mark.parametrize("bilinear", [False, True])
@pytest.mark.parametrize("n,h,w", [(1, 64, 64), (2, 48, 80), (1, 70, 54), (1, 135, 240)])
def test_default_init_parity(cuda_device, bilinear, n, h, w):
    sd = O.init_state_dict(0, 2, 1, bilinear)
    m = build(sd, cuda_device, bilinear=bilinear)
    f1, f2 = frames(1, n, 1, h, w), frames(2, n, 1, h, w)
    x1, x2 = O.preprocess_u8(f1.numpy()), O.preprocess_u8(f2.numpy())
    taps = {}
    ref = O.unet_forward(sd, torch.cat([x1, x2], 1), taps)
    got = m(x1.to(cuda_device), x2.to(cuda_device)).cpu()
    assert got.shape == ref.shape == (n, 1, h, w)
    err = (got - ref).abs().max().item() / 2
    assert err <= 2e-2, f"max abs pixel error {err}"
    assert psnr_unit(got / 2, ref / 2) >= 45.0
    # per-layer relative error (the end-to-end bound alone is vacuous on this fixture)
    net = m._fi_net
    names = {"inc": "inc", "down1": "down1", "down2": "down2", "down3": "down3", "down4": "down4", "up1": "up1",
             "up2": "up2", "up3": "up3", "up1.up": "up1.up", "up4.up": "up4.up"}
    for ours, theirs in names.items():
        a = net.read_activation(ours, n)
        b = taps[theirs]
        assert a.shape == b.shape, (ours, a.shape, b.shape)
        rel = (a - b).norm() / (b.norm() + 1e-12)
        assert rel < 2e-2, f"layer {ours}: relative L2 error {rel:.4f}"
    rel_out = (got - ref).norm() / ref.norm()
    assert rel_out < 2e-2, f"output relative L2 error {rel_out:.4f}"


@pytest.mark.parametrize("bilinear", [False, True])
def test_stressed_fixture(cuda_device, bilinear):
    """Randomised BN statistics + rescaled head: output spans both clamps (SURVEY.md A.6 ii)."""
    n, h, w = 1, 96, 128
    f1, f2 = frames(3, n, 1, h, w), frames(4, n, 1, h, w)
    x = torch.cat([O.preprocess_u8(f1.numpy()), O.preprocess_u8(f2.numpy())], 1)
    sd = O.calibrate_head(O.stress_state_dict(O.init_state_dict(0, 2, 1, bilinear), seed=1), x)
    ref = O.unet_forward(sd, x)
    assert ref.min() < -1.2 and ref.max() > 1.2
    m = build(sd, cuda_device, bilinear=bilinear)
    got = m(x[:, :1].to(cuda_device), x[:, 1:].to(cuda_device)).cpu()
    err = (got - ref).abs().max().item() / 2
    psnr = psnr_unit(got / 2, ref / 2)
    print(f"stressed bilinear={bilinear}: max abs {err:.4f} psnr {psnr:.1f} dB")
    # the all-bf16 torch pipeline measures 0.025-0.038 / 39-46 dB on this fixture (SURVEY.md A.6); we keep fp32
    # accumulators, an fp32 stem and an fp32 head, and must meet the stated bf16 bar
    assert err <= 2e-2, f"max abs pixel error {err}"
    assert psnr >= 45.0, f"PSNR {psnr:.2f} dB"
    # u8 path: same network fed raw uint8 frames, post-processing fused
    out_u8 = m.forward_u8(f1.to(cuda_device), f2.to(cuda_device)).cpu().numpy()
    exp_u8 = O.postprocess(ref)
    d = np.abs(out_u8.astype(np.int32) - exp_u8.astype(np.int32))
    assert d.max() <= 6, d.max()  # 2e-2 * 255 = 5.1 grey levels (+1 for the truncating cast)


def test_u8_and_f32_inputs_agree(cuda_device):
    sd = O.init_state_dict(0, 2, 1, False)
    m = build(sd, cuda_device)
    f1, f2 = frames(5, 2, 1, 32, 48), frames(6, 2, 1, 32, 48)
    a = m(O.preprocess_u8(f1.numpy()).to(cuda_device), O.preprocess_u8(f2.numpy()).to(cuda_device))
    b = m(f1.to(cuda_device), f2.to(cuda_device))
    assert torch.equal(a, b), "in-kernel normalisation must be bit-identical to preprocess_image's"


def test_unet_6_in_3_out(cuda_device):
    """UNet(6, 3): the RGB-pair variant the README describes (SURVEY.md D1)."""
    sd = O.init_state_dict(7, 6, 3, False, prefix="")
    m = build(sd, cuda_device, 6, 3, False, wrapper=False)
    x = O.preprocess_u8(frames(8, 1, 6, 40, 56).numpy())
    ref = O.unet_forward(sd, x)
    got = m(x.to(cuda_device)).cpu()
    assert got.shape == (1, 3, 40, 56)
    assert (got - ref).abs().max().item() / 2 <= 2e-2
    assert (got - ref).norm() / ref.norm() < 2e-2


def test_weight_update_is_picked_up(cuda_device):
    sd = O.init_state_dict(0, 2, 1, False)
    m = build(sd, cuda_device)
    x1 = torch.rand(1, 1, 32, 32, device=cuda_device) * 2 - 1
    x2 = torch.rand(1, 1, 32, 32, device=cuda_device) * 2 - 1
    a = m(x1, x2)
    with torch.no_grad():
        m.unet.outc.conv.bias.add_(0.5)
    b = m(x1, x2)
    assert torch.allclose(b, a + 0.5, atol=1e-6)


def test_errors_are_loud(cuda_device):
    from model._engine import FiError
    m = FrameInterpolationUNet().eval()
    with pytest.raises(FiError):  # CPU tensors: no fallback
        m(torch.zeros(1, 1, 32, 32), torch.zeros(1, 1, 32, 32))
    m = m.to(cuda_device)
    with pytest.raises(FiError):  # smaller than 16x16
        m(torch.zeros(1, 1, 8, 8, device=cuda_device), torch.zeros(1, 1, 8, 8, device=cuda_device))
    m.train()
    with pytest.raises(FiError):
        m(torch.zeros(1, 1, 32, 32, device=cuda_device), torch.zeros(1, 1, 32, 32, device=cuda_device))


@pytest.mark.parametrize("bilinear", [False, True])
def test_fp32_path_meets_1e_3(cuda_device, bilinear):
    """precision='fp32' (hi/lo-split operands, 3 products per MAC): north-star bar max |err| <= 1e-3 in [0,1] pixel units
    on the STRESSED fixture (the default-init fixture would pass even in bf16), PSNR far above 45 dB, per-layer taps
    at fp32-grade relative error."""
    n, h, w = 1, 70, 118  # odd sizes: F.pad path in two decoder levels
    f1, f2 = frames(11, n, 1, h, w), frames(12, n, 1, h, w)
    x = torch.cat([O.preprocess_u8(f1.numpy()), O.preprocess_u8(f2.numpy())], 1)
    sd = O.calibrate_head(O.stress_state_dict(O.init_state_dict(0, 2, 1, bilinear), seed=1), x)
    taps = {}
    ref = O.unet_forward(sd, x, taps)
    m = build(sd, cuda_device, bilinear=bilinear)
    m.precision = "fp32"
    got = m(x[:, :1].to(cuda_device), x[:, 1:].to(cuda_device)).cpu()
    err = (got - ref).abs().max().item() / 2
    psnr = psnr_unit(got / 2, ref / 2)
    print(f"fp32 path bilinear={bilinear}: max abs {err:.2e} psnr {psnr:.1f} dB")
    assert err <= 1e-3, f"max abs pixel error {err}"
    assert psnr >= 80.0
    net = m._fi_net
    for name in ("inc", "down2", "down4", "up1.up", "up2", "up3"):
        a, b = net.read_activation(name, n), taps[name]
        rel = (a - b).norm() / (b.norm() + 1e-12)
        assert rel < 1e-4, f"layer {name}: relative L2 error {rel:.2e}"
    # same module back in bf16: engine is rebuilt, result changes but stays inside the bf16 bar
    m.precision = "bf16"
    got16 = m(x[:, :1].to(cuda_device), x[:, 1:].to(cuda_device)).cpu()
    assert 1e-3 < (got16 - ref).abs().max().item() / 2 <= 2e-2
    # the u8 output of the fp32 path equals the oracle's post-processed frame except at truncation boundaries
    m.precision = "fp32"
    out_u8 = m.forward_u8(f1.to(cuda_device), f2.to(cuda_device)).cpu().numpy()
    d = np.abs(out_u8.astype(np.int32) - O.postprocess(ref).astype(np.int32))
    assert d.max() <= 1 and (d > 0).mean() < 0.02


def test_all_modes_small_clip(cuda_device):
    """Every kernel variant on one odd-sized clip: ConvT/bilinear x bf16/fp32, pipelined clip entry point, metrics."""
    from model import _engine as E
    rs = np.random.RandomState(0)
    f = rs.randint(0, 256, size=(4, 1, 38, 54)).astype(np.uint8)
    for bilinear in (False, True):
        sd = O.init_state_dict(0, 2, 1, bilinear)
        ref = O.postprocess(O.unet_forward(sd, torch.cat([O.preprocess_u8(f[:-1]), O.preprocess_u8(f[1:])], 1)))
        for precision, tol in (("bf16", 6), ("fp32", 1)):
            net = E.Net(cuda_device, 2, 1, bilinear, precision)
            net.load_state_dict(sd)
            out = net.interpolate_clip_host_u8(f, pairs_per_batch=2)
            assert np.abs(out.astype(int) - ref.astype(int)).max() <= tol, (bilinear, precision)
            net.close()


def test_batch_sizes_share_one_plan(cuda_device):
    """The arena / tensor maps are sized for the largest batch seen; smaller batches reuse them (ragged last batch of a
    clip, API requests of varying size) and give bit-identical per-image results."""
    from model import _engine as E
    sd = O.init_state_dict(0, 2, 1, False)
    net = E.Net(cuda_device, 2, 1, False)
    net.load_state_dict(sd)
    f = frames(21, 5, 1, 48, 80).to(cuda_device)
    full = net.forward(f[:4], f[1:5], want_f32=True)[0].clone()
    one = net.forward(f[2:3], f[3:4], want_f32=True)[0].clone()
    two = net.forward(f[1:3], f[2:4], want_f32=True)[0].clone()
    assert torch.equal(one[0], full[2]) and torch.equal(two, full[1:3])
    fl4, launches = net.cost(4, 48, 80)
    fl1, _ = net.cost(1, 48, 80)
    # 21 launches: the grey bf16 network computes inc.double_conv.0 inside inc.double_conv.3's kernel (22 without)
    assert abs(fl4 - 4 * fl1) < 1 and abs(fl1 - O.flops_per_forward(1, 48, 80)) < 1 and launches == 21
    again = net.forward(f[:4], f[1:5], want_f32=True)[0]
    assert torch.equal(again, full)


def test_random_shape_fuzz(cuda_device):
    """Seeded shape fuzz (the reference pins nothing but one output shape): random odd/even sizes down to the 16x16
    minimum, batches 1-3, both decoders, compared with the oracle on the output and on the deepest tap."""
    from model import _engine as E
    rs = np.random.RandomState(2024)
    nets = {}
    for case in range(14):
        bilinear = bool(case % 2)
        n, h, w = int(rs.randint(1, 4)), int(rs.randint(16, 90)), int(rs.randint(16, 130))
        if case == 0:
            n, h, w = 1, 16, 16
        if case == 1:
            n, h, w = 2, 17, 31
        if bilinear not in nets:
            sd = O.init_state_dict(0, 2, 1, bilinear)
            net = E.Net(cuda_device, 2, 1, bilinear)
            net.load_state_dict(sd)
            nets[bilinear] = (sd, net)
        sd, net = nets[bilinear]
        f1 = torch.from_numpy(rs.randint(0, 256, size=(n, 1, h, w)).astype(np.uint8))
        f2 = torch.from_numpy(rs.randint(0, 256, size=(n, 1, h, w)).astype(np.uint8))
        taps = {}
        ref = O.unet_forward(sd, torch.cat([O.preprocess_u8(f1.numpy()), O.preprocess_u8(f2.numpy())], 1), taps)
        got = net.forward(f1.to(cuda_device), f2.to(cuda_device), want_f32=True)[0].cpu()
        assert got.shape == ref.shape, (n, h, w)
        rel = ((got - ref).norm() / ref.norm()).item()
        deep = net.read_activation("down4", n)
        rel_deep = ((deep - taps["down4"]).norm() / (taps["down4"].norm() + 1e-12)).item()
        assert rel < 2e-2 and rel_deep < 2e-2, (bilinear, n, h, w, rel, rel_deep)


def test_building_blocks_stand_alone(cuda_device):
    """DoubleConv / Down / Up / OutConv called on their own (reference model/unet.py:5-63) against the same torch ops."""
    import torch.nn as nn
    import torch.nn.functional as F
    from model.unet import DoubleConv, Down, Up, OutConv
    g = torch.Generator().manual_seed(3)

    def randomise(m):
        for mod in m.modules():
            if isinstance(mod, nn.BatchNorm2d):
                mod.weight.data = torch.rand(mod.num_features, generator=g) + 0.5
                mod.bias.data = torch.randn(mod.num_features, generator=g) * 0.1
                mod.running_mean.data = torch.randn(mod.num_features, generator=g) * 0.1
                mod.running_var.data = torch.rand(mod.num_features, generator=g) + 0.5
        return m.eval()

    def ref_double(dc, x):
        s = dc.double_conv
        for conv, bn in ((s[0], s[1]), (s[3], s[4])):
            x = F.relu(F.batch_norm(F.conv2d(x, conv.weight, None, padding=1), bn.running_mean, bn.running_var,
                                    bn.weight, bn.bias, False, 0.0, bn.eps))
        return x

    def check(got, ref, what):
        assert got.shape == ref.shape, what
        rel = ((got.cpu() - ref).norm() / ref.norm()).item()
        assert rel < 1.5e-2, f"{what}: relative L2 error {rel:.4f}"

    with torch.no_grad():
        dc = randomise(DoubleConv(2, 64))
        x = torch.rand(2, 2, 21, 30, generator=g) * 2 - 1
        check(dc.to(cuda_device)(x.to(cuda_device)), ref_double(dc.cpu(), x), "DoubleConv(2,64)")
        dc = randomise(DoubleConv(64, 128))
        x = torch.randn(1, 64, 18, 20, generator=g)
        check(dc.to(cuda_device)(x.to(cuda_device)), ref_double(dc.cpu(), x), "DoubleConv(64,128)")
        dn = randomise(Down(64, 128))
        x = torch.randn(1, 64, 19, 26, generator=g)
        check(dn.to(cuda_device)(x.to(cuda_device)), ref_double(dn.cpu().maxpool_conv[1], F.max_pool2d(x, 2)), "Down")
        for bilinear in (False, True):
            up = randomise(Up(128, 64, bilinear))
            x1, x2 = torch.randn(1, 128 if not bilinear else 64, 9, 12, generator=g), torch.randn(1, 64, 19, 25, generator=g)
            u = up.cpu().up(x1)
            dy, dx = x2.shape[2] - u.shape[2], x2.shape[3] - u.shape[3]
            cat = torch.cat([x2, F.pad(u, [dx // 2, dx - dx // 2, dy // 2, dy - dy // 2])], 1)
            ref = ref_double(up.conv, cat)
            check(up.to(cuda_device)(x1.to(cuda_device), x2.to(cuda_device)), ref, f"Up(bilinear={bilinear})")
        oc = OutConv(64, 3).eval()
        x = torch.randn(2, 64, 10, 11, generator=g)
        check(oc.to(cuda_device)(x.to(cuda_device)), oc.cpu().conv(x), "OutConv")


@pytest.mark.parametrize("env", [{"FI_CTA2": "0"}, {"FI_CTA2": "0", "FI_NO_HALO": "1"},
                                 {"FI_BLOCK_N": "256"}, {"FI_BLOCK_N": "128"}, {"FI_BLOCK_N": "64"}, {"FI_PDL": "0"},
                                 {"FI_FUSE_INC": "0"}])
def test_kernel_selection_fallbacks_give_same_network(cuda_device, monkeypatch, env):
    """The single-CTA kernels (FI_CTA2=0), the per-tap kernel for narrow layers (FI_NO_HALO=1), every column-block
    width of the per-tap kernel (the default picks it from the tile count) and plain stream order instead of
    programmatic dependent launch compute the same network as the default selection (CTA pairs + halo reuse):
    identical per-layer inputs and fp32 accumulation orders differ only in how K is walked, so outputs agree to bf16
    noise."""
    from model import _engine as E
    sd = O.init_state_dict(0, 2, 1, False)
    f1, f2 = frames(31, 2, 1, 70, 118).to(cuda_device), frames(32, 2, 1, 70, 118).to(cuda_device)
    base = E.Net(cuda_device, 2, 1, False)
    base.load_state_dict(sd)
    ref = base.forward(f1, f2, want_f32=True)[0].clone()
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    alt = E.Net(cuda_device, 2, 1, False)
    alt.load_state_dict(sd)
    got = alt.forward(f1, f2, want_f32=True)[0]
    assert ((got - ref).norm() / ref.norm()).item() < 5e-3
    oracle = O.unet_forward(sd, torch.cat([O.preprocess_u8(f1.cpu().numpy()), O.preprocess_u8(f2.cpu().numpy())], 1))
    assert ((got.cpu() - oracle).norm() / oracle.norm()).item() < 2e-2


def test_c_abi_error_paths(cuda_device):
    """Errors come back as negative codes + message, never as a crash (SURVEY.md §8b error convention)."""
    import ctypes as C
    from model import _engine as E
    lib = E.lib()
    net = E.Net(cuda_device, 2, 1, False)
    x = torch.zeros(1, 1, 32, 32, device=cuda_device)
    with pytest.raises(E.FiError, match="fiNetLoadWeights has not been called"):
        net.forward(x, x)
    sd = O.init_state_dict(0, 2, 1, False)
    bad = {k: v for k, v in sd.items() if "up2.up.weight" not in k}
    with pytest.raises(E.FiError, match="missing state-dict entry 'up2.up.weight'"):
        net.load_state_dict(bad)
    bilinear_sd = O.init_state_dict(0, 2, 1, True)     # what the reference's load_model would reject as well
    with pytest.raises(E.FiError, match="size mismatch|missing"):
        net.load_state_dict(bilinear_sd)
    net.load_state_dict(sd)
    with pytest.raises(E.FiError, match="provide 3 channels"):
        net.forward(torch.zeros(1, 2, 32, 32, device=cuda_device), x)
    with pytest.raises(E.FiError, match="smaller than 16x16"):
        net.forward(x[:, :, :8, :8], x[:, :, :8, :8])
    with pytest.raises(E.FiError):
        net.forward(x.double(), x.double())
    d = E.ConvDesc()
    assert lib.fiConvGemm(C.byref(d), None) == -1 and b"conv:" in lib.fiLastError()
    assert lib.fiSsimPsnrU8(None, None, 1, 8, 8, None, None, None) == -1
    with pytest.raises(E.FiError, match="precision"):
        E.Net(cuda_device, 2, 1, False, "fp64")
    out = net.forward(x, x)[0]  # the handle is still usable after the failed calls
    assert torch.isfinite(out).all()


def test_plan_cache_keeps_alternating_shapes(cuda_device, monkeypatch):
    """A server alternates between frame sizes (256x256 API requests between video batches): each size gets its plan once
    and switching back neither rebuilds nor changes results; the cache is LRU-bounded ($FI_PLAN_CACHE)."""
    from model import _engine as E
    sd = O.init_state_dict(0, 2, 1, False)
    net = E.Net(cuda_device, 2, 1, False)
    net.load_state_dict(sd)
    shapes = [(1, 64, 64), (2, 48, 80), (1, 96, 128)]
    inputs = {s: (frames(40 + i, s[0], 1, s[1], s[2]).to(cuda_device), frames(50 + i, s[0], 1, s[1], s[2]).to(cuda_device))
              for i, s in enumerate(shapes)}
    first = {s: net.forward(*inputs[s], want_f32=True)[0].clone() for s in shapes}
    cached, builds, nbytes = net.plan_stats()
    assert (cached, builds) == (3, 3) and nbytes > 0
    for _ in range(3):
        for s in shapes:
            assert torch.equal(net.forward(*inputs[s], want_f32=True)[0], first[s])
    assert net.plan_stats()[:2] == (3, 3), "alternating shapes must not rebuild plans"
    # a smaller batch of a cached size reuses its plan; a larger one supersedes it (one plan per frame size)
    net.forward(inputs[(2, 48, 80)][0][:1], inputs[(2, 48, 80)][1][:1])
    assert net.plan_stats()[:2] == (3, 3)
    big = frames(60, 3, 1, 48, 80).to(cuda_device)
    net.forward(big, big)
    assert net.plan_stats()[:2] == (3, 4)
    # the read-back tap follows the most recent forward's plan
    net.forward(*inputs[(1, 64, 64)])
    assert net.read_activation("inc", 1).shape == (1, 64, 64, 64)
    # LRU bound
    monkeypatch.setenv("FI_PLAN_CACHE", "2")
    small = E.Net(cuda_device, 2, 1, False)
    small.load_state_dict(sd)
    for s in shapes:
        small.forward(*inputs[s])
    assert small.plan_stats()[:2] == (2, 3)
    small.forward(*inputs[shapes[0]])          # evicted earlier: rebuilt, same result
    assert small.plan_stats()[:2] == (2, 4)
    assert torch.equal(small.forward(*inputs[shapes[0]], want_f32=True)[0], first[shapes[0]])


@pytest.mark.parametrize("bilinear,precision", [(False, "bf16"), (True, "bf16"), (False, "fp32")])
def test_arena_liveness_reuse(cuda_device, monkeypatch, bilinear, precision):
    """FI_ARENA_REUSE=1 (automatic for plans above 16 GiB: 4K frames x 8 pairs) places dead tensors' memory under later
    ones: same bytes out, a much smaller arena, and the debug taps refuse to read overwritten tensors."""
    from model import _engine as E
    sd = O.init_state_dict(0, 2, 1, bilinear)
    f1, f2 = frames(71, 3, 1, 70, 118).to(cuda_device), frames(72, 3, 1, 70, 118).to(cuda_device)
    plain = E.Net(cuda_device, 2, 1, bilinear, precision)
    plain.load_state_dict(sd)
    want_f, want_u = plain.forward(f1, f2, want_f32=True, want_u8=True)
    plain_bytes = plain.plan_stats()[2]
    monkeypatch.setenv("FI_ARENA_REUSE", "1")
    lean = E.Net(cuda_device, 2, 1, bilinear, precision)
    lean.load_state_dict(sd)
    for _ in range(2):      # the second forward runs over an arena full of the first one's leftovers
        got_f, got_u = lean.forward(f1, f2, want_f32=True, want_u8=True)
        assert torch.equal(got_f, want_f) and torch.equal(got_u, want_u)
    lean_bytes = lean.plan_stats()[2]
    assert lean_bytes < 0.55 * plain_bytes, (lean_bytes, plain_bytes)
    with pytest.raises(E.FiError, match="taps are unavailable"):
        lean.read_activation("inc", 3)
    assert plain.read_activation("inc", 3).shape == (3, 64, 70, 118)


@pytest.mark.parametrize("n,h,w", [(1, 16, 16), (3, 70, 118), (2, 135, 240), (1, 257, 97)])
def test_fused_inc_kernel_is_bit_identical_to_stem_plus_conv(cuda_device, monkeypatch, n, h, w):
    """conv_inc_fused.cu (the default for the grey bf16 network: stem computed inside inc.double_conv.3's kernel, inc.mid
    never in HBM) against the two separate kernels (FI_FUSE_INC=0): same arithmetic in the same order, so the `inc`
    tensor, the pooled tensor's consumer (`down1`) and the network output must be bit-identical — u8 and fp32 inputs,
    partial tiles on every border."""
    from model import _engine as E
    sd = O.stress_state_dict(O.init_state_dict(0, 2, 1, False), seed=3)
    f1, f2 = frames(81, n, 1, h, w).to(cuda_device), frames(82, n, 1, h, w).to(cuda_device)
    x1 = O.preprocess_u8(f1.cpu().numpy()).to(cuda_device)
    x2 = O.preprocess_u8(f2.cpu().numpy()).to(cuda_device)
    monkeypatch.delenv("FI_FUSE_INC", raising=False)
    fused = E.Net(cuda_device, 2, 1, False)
    fused.load_state_dict(sd)
    assert fused.cost(n, h, w)[1] == 21
    got_u8 = fused.forward(f1, f2, want_f32=True, want_u8=True)
    taps_fused = {k: fused.read_activation(k, n) for k in ("inc", "down1")}
    got_f32 = fused.forward(x1, x2, want_f32=True)[0].clone()
    monkeypatch.setenv("FI_FUSE_INC", "0")
    plain = E.Net(cuda_device, 2, 1, False)
    plain.load_state_dict(sd)
    assert plain.cost(n, h, w)[1] == 22
    want_u8 = plain.forward(f1, f2, want_f32=True, want_u8=True)
    for k, v in taps_fused.items():
        assert torch.equal(v, plain.read_activation(k, n)), f"tap {k} differs"
    assert torch.equal(got_u8[0], want_u8[0]) and torch.equal(got_u8[1], want_u8[1])
    assert torch.equal(got_f32, plain.forward(x1, x2, want_f32=True)[0])
    # and both agree with the oracle
    ref = O.unet_forward(sd, torch.cat([x1.cpu(), x2.cpu()], 1))
    assert ((got_f32.cpu() - ref).norm() / ref.norm()).item() < 2e-2


@pytest.mark.parametrize("n_channels,n_classes,bilinear", [(1, 2, True), (1, 1, False), (4, 1, True), (3, 3, False)])
def test_other_channel_counts(cuda_device, n_channels, n_classes, bilinear):
    """UNet is channel-generic (reference model/unet.py:66): one input channel (the fused inc kernel's other
    instantiation), three and four (the stand-alone stem kernel with two K slabs), several output classes."""
    sd = O.init_state_dict(5, n_channels, n_classes, bilinear, prefix="")
    m = build(sd, cuda_device, n_channels, n_classes, bilinear, wrapper=False)
    x = O.preprocess_u8(frames(9, 2, n_channels, 37, 52).numpy())
    ref = O.unet_forward(sd, x)
    got = m(x.to(cuda_device)).cpu()
    assert got.shape == (2, n_classes, 37, 52)
    assert (got - ref).abs().max().item() / 2 <= 2e-2
    assert ((got - ref).norm() / ref.norm()).item() < 2e-2
