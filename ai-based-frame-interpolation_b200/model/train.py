"""Training step of the reference's model/train.py (train_model's inner loop, :183-199: forward in training mode,
loss, backward, Adam) on the B200 kernels — SURVEY.md §8f row 2 / BASELINE config "MSE + Adam, batch 16 at 256x256".

What runs where
  conv3x3 forward, conv3x3 data gradient   tcgen05 implicit-GEMM kernels (fiConvGemm; dgrad = conv with flipped weights)
  conv3x3 weight gradient                  tcgen05 split-K GEMM over the pixel dimension (fiWgrad), operands read as NHWC
  BatchNorm (batch statistics) fwd / bwd, ReLU, max-pool / bilinear-upsample backward, 1x1 head, MSE, Adam: CUDA-core
                                           kernels in csrc/train_kernels.cu
  gradient all-reduce                      torch.distributed (NCCL) on one flat fp32 gradient buffer
PyTorch holds the fp32 master parameters (the module's own nn.Parameters), the flat gradient / Adam buffers and does
per-channel vector arithmetic of BatchNorm (C-sized tensors); every per-pixel FLOP is in the library.

Scope: FrameInterpolationUNet / UNet with either decoder — bilinear=True (what the reference's train.py builds,
model/train.py:299) or the class default ConvTranspose2d (model/unet.py:43: forward = the EPI_CONVT GEMM, data gradient =
a per-pixel GEMM on the output gradient viewed as [N,h,w,(ky,kx,co)], weight gradient = fiWgradPointwise) —
H and W multiples of 16 (the reference trains at 256x256, model/train.py:138), bf16 activations and activation
gradients, fp32 master parameters / gradients / Adam state. Loss: criterion=None is the fused MSE kernel (BASELINE
config 5); a CombinedLoss instance (the reference's 0.5*MSE + 0.5*(1-SSIM), model/train.py:75-87) is the fused
fiCombinedLossGrad kernel; any other torch callable on the [N,1,H,W] fp32 network output is differentiated by torch
autograd on that one tensor and its gradient enters the library backward.

Also here, mirroring the reference file: SSIMLoss / CombinedLoss, FrameTripletDataset, train_model (same checkpoint
keys, ReduceLROnPlateau(factor 0.5, patience 10) schedule) and main().
"""
from __future__ import annotations

import argparse
import copy
import ctypes as C
import math
import os

import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

try:
    from . import _engine as E
    from . import crops
    from .unet import FrameInterpolationUNet, UNet
except ImportError:  # model/ on sys.path, like the reference's scripts
    import _engine as E
    import crops
    from unet import FrameInterpolationUNet, UNet

BN_MOMENTUM = 0.1


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


class _Layer:
    """One conv3x3 + BatchNorm + ReLU stage: parameters, packed weights and what the backward needs."""

    def __init__(self, name, conv, bn, src, src1=None):
        self.name, self.conv, self.bn, self.src, self.src1 = name, conv, bn, src, src1
        self.cout, self.cin = conv.weight.shape[0], conv.weight.shape[1]


class TrainStep:
    """loss = TrainStep(model, lr=1e-4)(frame1, frame2, target) — one optimisation step in place on `model`."""

    def __init__(self, model, lr=1e-4, betas=(0.9, 0.999), eps=1e-8, criterion=None, cuda_graph=False,
                 overlap_wgrad=True):
        """cuda_graph=True: after two eager steps the step is captured once per input shape
        (forward + backward, about 200 launches; the all-reduce and the Adam launch stay eager) and replayed; the Adam
        launch stays outside the graphs and takes learning rate and step count by value. With several data-parallel replicas the
        capture is two graphs and the decoder's gradients are all-reduced while the second one (the encoder half of
        the backward pass) runs.
        overlap_wgrad=True: weight gradients run on a second stream, beside the BatchNorm-backward / data-gradient
        chain of the layers below (tensor-core-bound and HBM-bound kernels share the SMs)."""
        self.criterion, self.cuda_graph, self.overlap_wgrad = criterion, cuda_graph, overlap_wgrad
        self._graphs, self._eager_steps = {}, 0
        self.keep_activations = False
        unet = model.unet if isinstance(model, FrameInterpolationUNet) else model
        if not isinstance(unet, UNet):
            raise E.FiError("TrainStep needs a UNet / FrameInterpolationUNet")
        # decoder variant: nn.Upsample (what reference train.py:299 builds) or the class default ConvTranspose2d
        self.convt = not unet.bilinear
        self.model, self.unet = model, unet
        self.lr, self.betas, self.eps, self.step_count = lr, betas, eps, 0
        p0 = next(model.parameters())
        self.device = E.require_cuda(p0.device)
        self.params = [p for p in model.parameters() if p.requires_grad]
        n = sum(p.numel() for p in self.params)
        self.flat_grad = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.flat_param = torch.empty(n, dtype=torch.float32, device=self.device)
        self.m = torch.zeros_like(self.flat_grad)
        self.v = torch.zeros_like(self.flat_grad)
        off = 0
        self.grad_view = {}
        # parameters() order is inc, down1-4, up1-4, outc: the decoder's gradients (finished first by the backward pass)
        # are the tail of the flat buffer starting at the first parameter of up1
        names = {id(p): nm for nm, p in model.named_parameters()}
        self._decoder_offset = None
        with torch.no_grad():  # parameters become views of one flat buffer: Adam and the all-reduce see one vector
            for p in self.params:
                if self._decoder_offset is None and ".up1." in "." + names[id(p)]:
                    self._decoder_offset = off
                k = p.numel()
                self.flat_param[off:off + k] = p.detach().reshape(-1)
                p.data = self.flat_param[off:off + k].view_as(p)
                self.grad_view[p] = self.flat_grad[off:off + k].view_as(p)
                off += k
        u = unet
        dc = lambda m: m.double_conv  # noqa: E731
        L = []
        L.append(_Layer("inc.0", dc(u.inc)[0], dc(u.inc)[1], "input"))
        L.append(_Layer("inc.3", dc(u.inc)[3], dc(u.inc)[4], "inc.0"))
        for i, d in enumerate((u.down1, u.down2, u.down3, u.down4), 1):
            blk = dc(d.maxpool_conv[1])
            L.append(_Layer(f"down{i}.0", blk[0], blk[1], f"pool{i}"))
            L.append(_Layer(f"down{i}.3", blk[3], blk[4], f"down{i}.0"))
        skips = ["down3.3", "down2.3", "down1.3", "inc.3"]
        for i, up in enumerate((u.up1, u.up2, u.up3, u.up4), 1):
            blk = dc(up.conv)
            L.append(_Layer(f"up{i}.0", blk[0], blk[1], skips[i - 1], f"up{i}.up"))
            L.append(_Layer(f"up{i}.3", blk[3], blk[4], f"up{i}.0"))
        self.layers = L
        self.up_mods = {f"up{i}.0": up.up for i, up in enumerate((u.up1, u.up2, u.up3, u.up4), 1)}
        self.lib = E.lib()
        self._side = torch.cuda.Stream(device=self.device)
        self._sync_replicas()

    def _sync_replicas(self):
        """Data-parallel replicas must start from the same point: parameters, Adam moments and the BatchNorm running
        estimates of rank 0 are broadcast once (torch DDP does the same for parameters and buffers at construction).
        Afterwards only gradients are exchanged; the running estimates stay per replica (DDP default) and are averaged
        by `average_bn_buffers()` before validation / checkpointing."""
        if not self._distributed():
            return
        for t in (self.flat_param, self.m, self.v):
            dist.broadcast(t, 0)
        for l in self.layers:
            dist.broadcast(l.bn.running_mean, 0)
            dist.broadcast(l.bn.running_var, 0)
        self._invalidate_inference_mirror()

    def average_bn_buffers(self):
        """Mean over the replicas of every BatchNorm running_mean / running_var (no-op on one replica)."""
        if not self._distributed():
            return
        bufs = [b for l in self.layers for b in (l.bn.running_mean, l.bn.running_var)]
        flat = torch.cat([b.reshape(-1) for b in bufs])
        dist.all_reduce(flat, op=dist.ReduceOp.AVG)
        off = 0
        for b in bufs:
            b.copy_(flat[off:off + b.numel()].view_as(b))
            off += b.numel()
        self._invalidate_inference_mirror()

    def state_dict(self):
        """torch.optim.Adam-shaped state: per-parameter step / exp_avg / exp_avg_sq plus the param group."""
        state, off = {}, 0
        for i, p in enumerate(self.params):
            k = p.numel()
            state[i] = {"step": torch.tensor(float(self.step_count)), "exp_avg": self.m[off:off + k].view_as(p).clone(),
                        "exp_avg_sq": self.v[off:off + k].view_as(p).clone()}
            off += k
        return {"state": state, "param_groups": [{"lr": self.lr, "betas": self.betas, "eps": self.eps,
                                                  "weight_decay": 0, "amsgrad": False,
                                                  "params": list(range(len(self.params)))}]}

    def load_state_dict(self, sd):
        off = 0
        for i, p in enumerate(self.params):
            k = p.numel()
            st = sd["state"].get(i)
            if st is not None:
                self.m[off:off + k] = st["exp_avg"].reshape(-1).to(self.device)
                self.v[off:off + k] = st["exp_avg_sq"].reshape(-1).to(self.device)
                self.step_count = int(st["step"])
            off += k
        g = sd["param_groups"][0]
        self.lr, self.betas, self.eps = g["lr"], tuple(g["betas"]), g["eps"]

    # ------------------------------------------------------------------------------------------------ helpers
    def _conv(self, src, wpack, n_total, src1=None, taps=9, mode=E.EPI_STORE, bias=None):
        """bf16 NHWC conv3x3 (no bias, no ReLU) through the tcgen05 kernels. taps=1: a per-pixel GEMM (the transposed
        conv's data gradient); mode=EPI_CONVT: ConvTranspose2d(k=2, s=2) with its bias, n_total = 4*Cout columns ordered
        (ky, kx, co), output [N, 2H, 2W, Cout]."""
        n, h, w, c0 = src.shape
        d = E.ConvDesc()
        d.src0, d.c0, d.N, d.H, d.W = src.data_ptr(), c0, n, h, w
        if src1 is not None:
            d.src1, d.c1, d.h1, d.w1 = src1.data_ptr(), src1.shape[3], src1.shape[1], src1.shape[2]
        shape = (n, 2 * h, 2 * w, n_total // 4) if mode == E.EPI_CONVT else (n, h, w, n_total)
        dst = torch.empty(shape, dtype=torch.bfloat16, device=self.device)
        b = bias if bias is not None else self._zero_bias(n_total)
        d.wpack, d.bias, d.n_total, d.taps, d.mode, d.relu, d.dst = (wpack.data_ptr(), b.data_ptr(), n_total, taps,
                                                                     mode, 0, dst.data_ptr())
        E.check(self.lib.fiConvGemm(C.byref(d), E.current_stream()))
        return dst

    def _zero_bias(self, n):
        z = getattr(self, "_zeros", None)
        if z is None or z.numel() < n:
            z = self._zeros = torch.zeros(max(n, 1024), dtype=torch.float32, device=self.device)
        return z

    def _bn_forward(self, layer, z, work):
        """Batch statistics -> a = relu(bn(z)); returns (a, work) and updates the running statistics.
        work: zeroed fp32 [7, C] scratch (sum, sumsq, mean, rstd, scale, shift, pivot). The sums are taken about the
        pivot (the channel's first pixel) so that flat channels keep their variance in fp32."""
        n, h, w, c = z.shape
        P = n * h * w
        st = E.current_stream()
        E.check(self.lib.fiBnStatsShifted(_ptr(z), P, c, _ptr(work[6]), _ptr(work[0]), _ptr(work[1]), st))
        bn = layer.bn
        E.check(self.lib.fiBnFinalizeShifted(_ptr(work[0]), _ptr(work[1]), _ptr(work[6]), c, P, bn.eps, BN_MOMENTUM,
                                             _ptr(bn.weight), _ptr(bn.bias), _ptr(work[2]), _ptr(work[3]), _ptr(work[4]),
                                             _ptr(work[5]), _ptr(bn.running_mean), _ptr(bn.running_var), st))
        a = torch.empty_like(z)
        E.check(self.lib.fiBnApplyRelu(_ptr(z), P, c, _ptr(work[4]), _ptr(work[5]), _ptr(a), st))
        return a, work

    # ------------------------------------------------------------------------------------------------ one step
    @torch.no_grad()
    def loss_value(self, y, target):
        """The criterion on a finished network output (validation loop of reference model/train.py:204-219) as a 1-element
        device tensor: the same fused loss kernel as the training step (its gradient output goes to a scratch buffer),
        no host synchronisation."""
        lib, st = E.lib(), lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731
        y, tgt = y.contiguous().float(), target.contiguous().float()
        crit = self.criterion
        fused = (isinstance(crit, CombinedLoss) and crit.ssim_loss.window_size == 11 and crit.ssim_loss.size_average)
        if crit is not None and not fused:
            return crit(y, tgt).detach().reshape(1).float()
        loss, dy = torch.zeros(1, dtype=torch.float32, device=y.device), torch.empty_like(y)
        if crit is None:
            E.check(lib.fiMseLossGrad(_ptr(y), _ptr(tgt), y.numel(), _ptr(loss), _ptr(dy), st()))
        else:
            n, c, h, w = y.shape
            E.check(lib.fiCombinedLossGrad(_ptr(y), _ptr(tgt), n * c, h, w, float(crit.mse_weight),
                                           float(crit.ssim_weight), _ptr(loss), _ptr(dy), st()))
        return loss

    @torch.no_grad()
    def __call__(self, frame1, frame2, target):
        self.step_count += 1
        with torch.cuda.device(self.device):
            self._invalidate_inference_mirror()
            if not self.cuda_graph:
                return self._eager_step(frame1, frame2, target)
            key = (tuple(frame1.shape), None if frame2 is None else tuple(frame2.shape), tuple(target.shape))
            entry = self._graphs.get(key)
            if entry is None:
                if self._eager_steps < 2:       # warm-up: kernel attributes, allocator pools, autograd of the criterion
                    self._eager_steps += 1
                    return self._eager_step(frame1, frame2, target)
                static = [frame1.clone(), None if frame2 is None else frame2.clone(), target.clone()]
                torch.cuda.synchronize()
                phases = self._phases(*static)
                graphs = [torch.cuda.CUDAGraph()]
                with torch.cuda.graph(graphs[0]):
                    loss = next(phases)
                    if not self._distributed():
                        next(phases)            # one replica: the whole backward pass is one graph
                if self._distributed():         # second graph = the encoder half of the backward pass (same pool)
                    graphs.append(torch.cuda.CUDAGraph())
                    with torch.cuda.graph(graphs[1], pool=graphs[0].pool()):
                        next(phases)
                entry = self._graphs[key] = (graphs, static, loss, phases)   # `phases` keeps the tensors alive
            graphs, static, loss = entry[:3]
            static[0].copy_(frame1)
            if frame2 is not None:
                static[1].copy_(frame2)
            static[2].copy_(target)
            graphs[0].replay()
            if len(graphs) == 2:
                early = self._reduce_decoder_async()
                graphs[1].replay()
                self._finish(early)
            else:
                self._finish(None)
            return loss

    @staticmethod
    def _distributed():
        return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1

    def _eager_step(self, frame1, frame2, target):
        phases = self._phases(frame1, frame2, target)
        loss = next(phases)
        early = self._reduce_decoder_async() if self._distributed() else None
        next(phases)
        self._finish(early)
        return loss

    def _reduce_decoder_async(self):
        """All-reduce (mean) of the decoder + head gradients, enqueued while the encoder half of the backward pass is
        still to run: NCCL works on its own stream behind the kernels enqueued so far."""
        return dist.all_reduce(self.flat_grad[self._decoder_offset:], op=dist.ReduceOp.AVG, async_op=True)

    def _phases(self, frame1, frame2, target):
        """The step as a two-phase generator: forward + loss + backward through the decoder, then the encoder half of
        the backward pass. Both phases yield the loss tensor; data-parallel runs reduce the decoder's gradients between
        the two."""
        lib, st = self.lib, E.current_stream
        x = torch.cat([frame1, frame2], 1).contiguous().float() if frame2 is not None else frame1.contiguous().float()
        n, cin0, h, w = x.shape
        if h % 16 or w % 16:
            raise E.FiError("the training step needs H and W to be multiples of 16 (the reference trains at 256x256)")
        with torch.cuda.device(self.device):
            self.flat_grad.zero_()
            acts, zs, stats, packs = {}, {}, {}, {}
            # one zeroed scratch for every layer's BatchNorm reductions / affine and weight-gradient accumulators
            bn_total = sum(7 * l.cout for l in self.layers)
            dw_total = sum(9 * l.cout * l.cin for l in self.layers[1:])
            scratch = torch.zeros(bn_total + dw_total, dtype=torch.float32, device=self.device)
            bn_work, dw_work, off = {}, {}, 0
            for l in self.layers:
                bn_work[l.name] = scratch[off:off + 7 * l.cout].view(7, l.cout)
                off += 7 * l.cout
            for l in self.layers[1:]:
                dw_work[l.name] = scratch[off:off + 9 * l.cout * l.cin]
                off += 9 * l.cout * l.cin
            # ---- pack weights (bf16 forward rows, flipped/transposed rows for the data gradient)
            for l in self.layers:
                wt = l.conv.weight.detach()
                if l.name == "inc.0":
                    packed = torch.empty((64, lib.fiStemPackedK(l.cin)), dtype=torch.bfloat16, device=self.device)
                    E.check(lib.fiStemPackWeightsDevice(_ptr(wt), l.cin, _ptr(packed), st()))
                    packs[l.name] = (packed, None)
                else:
                    fwd = torch.empty((l.cout, 9 * l.cin), dtype=torch.bfloat16, device=self.device)
                    bwd = torch.empty((l.cin, 9 * l.cout), dtype=torch.bfloat16, device=self.device)
                    E.check(lib.fiPackConvWeights(_ptr(wt), l.cout, l.cin, _ptr(fwd), _ptr(bwd), st()))
                    packs[l.name] = (fwd, bwd)
            # ---- forward (training-mode BatchNorm)
            for l in self.layers:
                if l.name == "inc.0":
                    z = torch.empty((n, h, w, 64), dtype=torch.bfloat16, device=self.device)
                    p0 = E.planes_of(x)
                    E.check(lib.fiStemConvLinear(C.byref(p0), None, E.FI_IN_F32, _ptr(packs[l.name][0]),
                                                 _ptr(self._zero_bias(64)), _ptr(z), n, h, w, st()))
                else:
                    if l.src.startswith("pool"):
                        full = acts[self.layers[self.layers.index(l) - 1].name]
                        fn, fh, fw, fc = full.shape
                        pooled = torch.empty((fn, fh // 2, fw // 2, fc), dtype=torch.bfloat16, device=self.device)
                        E.check(lib.fiMaxPool2x2(_ptr(full), _ptr(pooled), fn, fh, fw, fc, st()))
                        acts[l.src] = pooled
                    if l.src1 is not None:
                        lo = acts[self.layers[self.layers.index(l) - 1].name]
                        ln, lh, lw, lc = lo.shape
                        if self.convt:
                            # nn.ConvTranspose2d(lc, lc/2, 2, 2) (reference model/unet.py:43): weight [ci, co, ky, kx]
                            # -> GEMM rows (ky, kx, co) for the forward, rows ci / K = (ky, kx, co) for the data gradient
                            tw = self.up_mods[l.name].weight.detach()
                            cup = tw.shape[1]
                            fwd_t = tw.permute(2, 3, 1, 0).reshape(4 * cup, lc).to(torch.bfloat16).contiguous()
                            packs[l.src1] = tw.permute(0, 2, 3, 1).reshape(lc, 4 * cup).to(torch.bfloat16).contiguous()
                            bias4 = self.up_mods[l.name].bias.detach().float().repeat(4).contiguous()
                            up = self._conv(lo, fwd_t, 4 * cup, taps=1, mode=E.EPI_CONVT, bias=bias4)
                        else:
                            up = torch.empty((ln, 2 * lh, 2 * lw, lc), dtype=torch.bfloat16, device=self.device)
                            E.check(lib.fiUpsample2x(_ptr(lo), _ptr(up), ln, lh, lw, lc, st()))
                        acts[l.src1] = up
                    z = self._conv(acts[l.src], packs[l.name][0], l.cout, acts.get(l.src1) if l.src1 else None)
                zs[l.name] = z
                acts[l.name], stats[l.name] = self._bn_forward(l, z, bn_work[l.name])
            last = acts["up4.3"]
            hw_, hb = self.unet.outc.conv.weight.detach().reshape(-1, 64).contiguous(), self.unet.outc.conv.bias.detach()
            ncls = hw_.shape[0]
            y = torch.empty((n, ncls, h, w), dtype=torch.float32, device=self.device)
            E.check(lib.fiHeadForward(_ptr(last), n, h * w, _ptr(hw_), _ptr(hb), ncls, _ptr(y), st()))
            tgt = target.contiguous().float()
            if self.criterion is None:
                loss = torch.zeros(1, dtype=torch.float32, device=self.device)
                dy = torch.empty_like(y)
                E.check(lib.fiMseLossGrad(_ptr(y), _ptr(tgt), y.numel(), _ptr(loss), _ptr(dy), st()))
            elif (isinstance(self.criterion, CombinedLoss) and self.criterion.ssim_loss.window_size == 11
                  and self.criterion.ssim_loss.size_average):   # the reference's loss: one fused kernel
                loss = torch.zeros(1, dtype=torch.float32, device=self.device)
                dy = torch.empty_like(y)
                E.check(lib.fiCombinedLossGrad(_ptr(y), _ptr(tgt), n * ncls, h, w, float(self.criterion.mse_weight),
                                               float(self.criterion.ssim_weight), _ptr(loss), _ptr(dy), st()))
            else:  # any other torch loss on the network output: autograd on this one [N,ncls,H,W] tensor only
                with torch.enable_grad():
                    y_req = y.detach().requires_grad_(True)
                    loss_t = self.criterion(y_req, tgt)
                    dy, = torch.autograd.grad(loss_t, y_req)
                loss, dy = loss_t.detach().reshape(1), dy.contiguous().float()
            # ---- backward
            main_stream = torch.cuda.current_stream()
            side_handle = lambda: C.c_void_p(self._side.cuda_stream)  # noqa: E731
            grads = {}  # gradient w.r.t. the activation named by the key
            dA = torch.empty_like(last)
            gw = self.grad_view[self.unet.outc.conv.weight].view(ncls, 64)
            gb = self.grad_view[self.unet.outc.conv.bias]
            E.check(lib.fiHeadBackward(_ptr(last), _ptr(dy), n, h * w, _ptr(hw_), ncls, _ptr(dA), _ptr(gw), _ptr(gb), st()))
            grads["up4.3"] = dA
            for l in reversed(self.layers):
                if l.name == "down4.3":        # every decoder layer is done: its gradients may be reduced now
                    if self.overlap_wgrad:
                        main_stream.wait_stream(self._side)
                    self.last_output = y
                    yield loss
                a, z = acts[l.name], zs[l.name]
                ln, lh, lw, lc = z.shape
                P = ln * lh * lw
                wk = stats[l.name]       # rows: sum, sumsq, mean, rstd, scale, shift, pivot
                dA = grads.pop(l.name)
                dbeta, dgamma = self.grad_view[l.bn.bias], self.grad_view[l.bn.weight]   # zeroed with flat_grad
                E.check(lib.fiBnReluBackwardReduce(_ptr(dA), _ptr(z), P, lc, _ptr(wk[2]), _ptr(wk[3]), _ptr(wk[4]),
                                                   _ptr(wk[5]), _ptr(dbeta), _ptr(dgamma), st()))
                dz = torch.empty_like(z)
                E.check(lib.fiBnReluBackwardApply(_ptr(dA), _ptr(z), P, lc, _ptr(wk[2]), _ptr(wk[3]), _ptr(l.bn.weight),
                                                  _ptr(l.bn.bias), _ptr(dbeta), _ptr(dgamma), _ptr(dz), st()))
                # weight gradient: on the side stream once dz exists
                srcs = [] if l.name == "inc.0" else [acts[l.src]] + ([acts[l.src1]] if l.src1 else [])
                wst = st
                if self.overlap_wgrad:
                    self._side.wait_stream(main_stream)
                    for t in (dz, *srcs):
                        t.record_stream(self._side)
                    wst = side_handle
                if l.name == "inc.0":
                    E.check(lib.fiStemWgrad(_ptr(dz), _ptr(x), n, h, w, l.cin, _ptr(self.grad_view[l.conv.weight]), wst()))
                    continue
                dW = dw_work[l.name]
                x1 = srcs[1] if len(srcs) > 1 else None
                E.check(lib.fiWgrad(_ptr(dz), _ptr(srcs[0]), srcs[0].shape[3], _ptr(x1), x1.shape[3] if x1 is not None else 0,
                                    ln, lh, lw, l.cout, _ptr(dW), wst()))
                E.check(lib.fiUnpackConvGrad(_ptr(dW), l.cout, l.cin, _ptr(self.grad_view[l.conv.weight]), wst()))
                # data gradient(s): conv3x3 of dz with the flipped, transposed weights
                bwd = packs[l.name][1]
                c0 = srcs[0].shape[3]
                d_src = self._conv(dz, bwd[:c0], c0)
                if l.src1:
                    d_up = self._conv(dz, bwd[c0:], l.cin - c0)
                    below = self.layers[self.layers.index(l) - 1].name   # the tensor that was upsampled
                    bn_, bh, bw_, bc = acts[below].shape
                    if self.convt:
                        tmod = self.up_mods[l.name]
                        d_lo = self._convt_backward(d_up, acts[below], packs[l.src1], self.grad_view[tmod.weight],
                                                    self.grad_view[tmod.bias])
                    else:
                        d_lo = torch.empty_like(acts[below])
                        E.check(lib.fiUpsample2xBackward(_ptr(d_up), _ptr(d_lo), bn_, bh, bw_, bc, st()))
                    grads[below] = d_lo
                    grads["skip:" + l.src] = d_src       # joins the encoder-side gradient at the pool backward
                elif l.src.startswith("pool"):
                    full_name = self.layers[self.layers.index(l) - 1].name
                    full = acts[full_name]
                    fn, fh, fw, fc = full.shape
                    d_full = torch.empty_like(full)
                    skip = grads.pop("skip:" + full_name, None)
                    E.check(lib.fiMaxPoolBackwardAdd(_ptr(full), _ptr(acts[l.src]), _ptr(d_src), _ptr(skip), _ptr(d_full),
                                                     fn, fh, fw, fc, st()))
                    grads[full_name] = d_full
                else:
                    grads[l.src] = d_src
            if self.overlap_wgrad:
                main_stream.wait_stream(self._side)
        self.last_output = y
        self.last_activations = acts if self.keep_activations else None   # diagnostics only: pins GBs of HBM
        yield loss

    def _convt_backward(self, d_up, x, w_lo, grad_w, grad_b):
        """ConvTranspose2d(k=2, s=2) backward. Per low-resolution pixel the output gradient is a vector over
        (ky, kx, co): d_lo = that vector times W (a per-pixel GEMM, K = 4*Cout), dW = sum over pixels of the outer
        product with the layer input (fiWgradPointwise), dbias = per-channel sum.
        d_up: bf16 [N,2h,2w,Cout] output gradient; x: bf16 [N,h,w,Cin] layer input; w_lo: bf16 [Cin][(ky,kx,co)] rows
        of the data-gradient GEMM. dW and dbias are ADDED into grad_w (fp32 [Cin,Cout,2,2]) and grad_b (fp32 [Cout]).
        Returns d_lo: bf16 [N,h,w,Cin]."""
        lib, st = self.lib, E.current_stream
        bn_, bh, bw_, bc = x.shape
        cup = d_up.shape[3]
        d_s2d = d_up.view(bn_, bh, 2, bw_, 2, cup).permute(0, 1, 3, 2, 4, 5).contiguous().view(bn_, bh, bw_, 4 * cup)
        d_lo = self._conv(d_s2d, w_lo, bc, taps=1)
        sumsq = torch.zeros(cup, dtype=torch.float32, device=self.device)
        E.check(lib.fiBnStats(_ptr(d_up), bn_ * bh * bw_ * 4, cup, _ptr(grad_b), _ptr(sumsq), st()))
        dwt = torch.zeros((4 * cup, bc), dtype=torch.float32, device=self.device)
        E.check(lib.fiWgradPointwise(_ptr(d_s2d), _ptr(x), bc, bn_, bh, bw_, 4 * cup, _ptr(dwt), st()))
        grad_w.add_(dwt.view(2, 2, cup, bc).permute(3, 2, 0, 1))
        return d_lo

    def _finish(self, early):
        """Rest of the gradient all-reduce across data-parallel replicas (NCCL over NVLink; `early` is the handle of
        the decoder bucket already in flight), BatchNorm counters, Adam. Kept outside the captured graphs: collectives
        are enqueued eagerly on every rank."""
        if self._distributed():
            rest = dist.all_reduce(self.flat_grad[:self._decoder_offset], op=dist.ReduceOp.AVG, async_op=True)
            early.wait()
            rest.wait()
        torch._foreach_add_([l.bn.num_batches_tracked for l in self.layers], 1)
        E.check(self.lib.fiAdamStep(_ptr(self.flat_param), _ptr(self.flat_grad), _ptr(self.m), _ptr(self.v),
                                    self.flat_param.numel(), self.lr, self.betas[0], self.betas[1], self.eps,
                                    self.step_count, None, E.current_stream()))  # eager launch: lr / step by value

    def _invalidate_inference_mirror(self):
        # the inference engine mirrors the parameters lazily: force a re-upload on the next eval forward
        for mod in (self.model, self.unet):
            mod.__dict__["_fi_print"] = None


# ---------------------------------------------------------------------------------------------------- reference surface
class SSIMLoss(nn.Module):
    """1 - SSIM with an 11x11 Gaussian window (sigma 1.5), zero-padded 'same' filtering, C1 = 0.01^2, C2 = 0.03^2 —
    the loss of reference model/train.py:18-73 (torch ops on the network output; see the module docstring)."""

    def __init__(self, window_size=11, size_average=True, channel=1):
        super().__init__()
        self.window_size, self.size_average, self.channel = window_size, size_average, channel
        self.window = self._create_window(window_size, channel)

    @staticmethod
    def _gaussian(window_size, sigma):
        x = torch.arange(window_size, dtype=torch.float64) - window_size // 2
        g = torch.exp(-x * x / (2.0 * sigma * sigma))
        return (g / g.sum()).float()

    def _create_window(self, window_size, channel):
        g = self._gaussian(window_size, 1.5)
        return torch.outer(g, g).expand(channel, 1, window_size, window_size).contiguous()

    def forward(self, img1, img2):
        c = img1.shape[1]
        if c != self.channel or self.window.device != img1.device or self.window.dtype != img1.dtype:
            self.window, self.channel = self._create_window(self.window_size, c).to(img1), c
        win, pad = self.window, self.window_size // 2
        blur = lambda t: F.conv2d(t, win, padding=pad, groups=c)  # noqa: E731
        mu1, mu2 = blur(img1), blur(img2)
        s11, s22, s12 = blur(img1 * img1) - mu1 * mu1, blur(img2 * img2) - mu2 * mu2, blur(img1 * img2) - mu1 * mu2
        c1, c2 = 0.01 ** 2, 0.03 ** 2
        ssim = ((2 * mu1 * mu2 + c1) * (2 * s12 + c2)) / ((mu1 * mu1 + mu2 * mu2 + c1) * (s11 + s22 + c2))
        return 1 - (ssim.mean() if self.size_average else ssim.mean((1, 2, 3)))


class CombinedLoss(nn.Module):
    """mse_weight * MSE + ssim_weight * (1 - SSIM) (reference model/train.py:75-87)."""

    def __init__(self, mse_weight=0.5, ssim_weight=0.5):
        super().__init__()
        self.mse_weight, self.ssim_weight = mse_weight, ssim_weight
        self.mse_loss, self.ssim_loss = nn.MSELoss(), SSIMLoss()

    def forward(self, pred, target):
        return self.mse_weight * self.mse_loss(pred, target) + self.ssim_weight * self.ssim_loss(pred, target)


class FrameTripletDataset(torch.utils.data.Dataset):
    """(frame_t0, frame_t1, ground_truth_mid) from <data_dir>/<video>/<sorted frames>: frames i and i+2 are the inputs,
    i+1 the target; grayscale, resized to 256x256, [0,1] fp32 [1,H,W] (reference model/train.py:89-151).

    color=True: BGR frames as planes [3,H,W] in cv2's B, G, R order (what FrameInterpolator feeds a colour model),
    for UNet(6, 3). crop=S: S x S windows of the frames at their native size instead of the resize; training samples
    take the random window, left-right mirror and frame1/frame2 swap of model/crops.py for (seed, epoch, triplet),
    the copy returned by `for_validation()` the centre window without either. `set_epoch(e)` selects the draws."""

    EXTENSIONS = (".jpg", ".png", ".bmp")

    def __init__(self, data_dir, sequence_length=3, color=False, crop=None, seed=0):
        self.data_dir, self.sequence_length = data_dir, sequence_length
        self.color, self.crop = bool(color), None if crop is None else crops.check_size(crop)
        self.seed, self.epoch, self.augment = int(seed), 0, True
        self.triplets = []
        for video in os.listdir(data_dir):
            path = os.path.join(data_dir, video)
            if not os.path.isdir(path):
                continue
            frames = sorted(f for f in os.listdir(path) if f.endswith(self.EXTENSIONS))
            for i in range(len(frames) - 2):
                self.triplets.append({"video_dir": path, "frame_t0": frames[i], "frame_t1": frames[i + 2],
                                      "ground_truth": frames[i + 1]})

    def __len__(self):
        return len(self.triplets)

    def set_epoch(self, epoch):
        """The epoch of the crop draws (train_model calls it at the start of every epoch)."""
        self.epoch = int(epoch)

    def for_validation(self):
        """The same triplets with centre windows and no mirror or swap (a shallow copy; only matters with crop)."""
        v = copy.copy(self)
        v.augment = False
        return v

    def __getitem__(self, idx):
        import cv2
        import numpy as np
        t = self.triplets[idx]
        if not self.color and self.crop is None:
            out = []
            for key in ("frame_t0", "frame_t1", "ground_truth"):
                img = cv2.imread(os.path.join(t["video_dir"], t[key]), cv2.IMREAD_GRAYSCALE)
                img = cv2.resize(img, (256, 256)).astype(np.float32) / 255.0
                out.append(torch.from_numpy(img).unsqueeze(0))
            return tuple(out)
        planes = []
        for key in ("frame_t0", "frame_t1", "ground_truth"):
            path = os.path.join(t["video_dir"], t[key])
            img = cv2.imread(path, cv2.IMREAD_COLOR if self.color else cv2.IMREAD_GRAYSCALE)
            if img is None:
                raise ValueError(f"cannot read frame {path!r}")
            if self.crop is None:
                img = cv2.resize(img, (256, 256))
            elif img.shape[0] < self.crop or img.shape[1] < self.crop:
                raise ValueError(f"frame {path!r} is {img.shape[1]}x{img.shape[0]}, smaller than the "
                                 f"{self.crop}x{self.crop} crop")
            planes.append((path, img.transpose(2, 0, 1) if self.color else img[None]))
        if self.crop is not None:
            s = self.crop
            for path, p in planes[1:]:
                if p.shape != planes[0][1].shape:
                    raise ValueError(f"frame {path!r} differs in size from {planes[0][0]!r} of the same triplet")
            h, w = planes[0][1].shape[1:]
            if self.augment:
                y0, x0, mirror, swap = (v[0] for v in crops.draw(self.seed, self.epoch, [idx], h, w, s))
            else:
                (y0, x0), mirror, swap = crops.centre(h, w, s), False, False
            y0, x0 = int(y0), int(x0)
            planes = [(path, p[:, y0:y0 + s, x0:x0 + s][:, :, ::-1] if mirror else p[:, y0:y0 + s, x0:x0 + s])
                      for path, p in planes]
            if swap:                     # the midpoint of (t1, t0) is the same target
                planes[0], planes[1] = planes[1], planes[0]
        return tuple(torch.from_numpy(p.astype(np.float32) / 255.0) for _, p in planes)


class _PlateauSchedule:
    """optim.lr_scheduler.ReduceLROnPlateau(mode='min', factor=0.5, patience=10) with torch's default relative
    threshold 1e-4 (reference model/train.py:163-165), acting on TrainStep.lr."""

    def __init__(self, step, factor=0.5, patience=10, threshold=1e-4):
        self.step_obj, self.factor, self.patience, self.threshold = step, factor, patience, threshold
        self.best, self.bad = math.inf, 0

    def step(self, metric):
        if metric < self.best * (1 - self.threshold):
            self.best, self.bad = metric, 0
        else:
            self.bad += 1
        if self.bad > self.patience:
            self.step_obj.lr *= self.factor
            self.bad = 0


def train_model(model, train_loader, val_loader, num_epochs=100, device="cuda", criterion="combined", lr=1e-4,
                checkpoint_path="best_model.pth", cuda_graph=True):
    """The reference's train_model (model/train.py:153-249): Adam(lr=1e-4), CombinedLoss, plateau schedule, best
    checkpoint by validation loss with the same dictionary keys. The optimisation step is TrainStep (B200 kernels,
    captured in CUDA graphs per batch shape); validation runs the eval-mode inference path. criterion: "combined" |
    "mse" | a torch callable.

    Under an initialised process group (torchrun: see main) every rank calls this with its own shard of the training
    data; gradients are averaged by TrainStep, the validation loss is averaged over ranks, and rank 0 alone prints and
    writes the checkpoint."""
    crit = CombinedLoss() if criterion == "combined" else (None if criterion == "mse" else criterion)
    step = TrainStep(model, lr=lr, criterion=crit, cuda_graph=cuda_graph)
    sched = _PlateauSchedule(step)
    distributed = TrainStep._distributed()
    rank0 = not distributed or dist.get_rank() == 0
    say = print if rank0 else (lambda *a, **k: None)
    train_losses, val_losses, best = [], [], math.inf

    def mean_over_ranks(total, count):
        if distributed:
            t = torch.tensor([total, float(count)], dtype=torch.float64, device=device)
            dist.all_reduce(t)
            total, count = t[0].item(), t[1].item()
        return total / max(count, 1)

    say(f"Starting training for {num_epochs} epochs...")
    say(f"Using device: {device}")
    for epoch in range(num_epochs):
        sampler = getattr(train_loader, "sampler", None)
        if hasattr(sampler, "set_epoch"):
            sampler.set_epoch(epoch)
        data = getattr(train_loader, "dataset", None)
        while isinstance(data, torch.utils.data.Subset):
            data = data.dataset
        if hasattr(data, "set_epoch"):    # the crop draws of FrameTripletDataset (DataLoader and frame cache alike)
            data.set_epoch(epoch)
        model.train()
        total = torch.zeros((), dtype=torch.float32, device=device)   # summed on the device: no sync per step
        for f0, f1, gt in train_loader:
            total += step(f0.to(device, non_blocking=True), f1.to(device, non_blocking=True),
                          gt.to(device, non_blocking=True)).detach().reshape(())
        train_losses.append(mean_over_ranks(total.item(), len(train_loader)))
        step.average_bn_buffers()
        model.eval()
        total = torch.zeros(1, dtype=torch.float32, device=device)
        with torch.no_grad():
            for f0, f1, gt in val_loader:
                f0, f1 = f0.to(device, non_blocking=True), f1.to(device, non_blocking=True)
                y = model(torch.cat([f0, f1], 1)) if isinstance(model, UNet) else model(f0, f1)   # UNet takes one tensor
                total += step.loss_value(y, gt.to(device, non_blocking=True))
        val_losses.append(mean_over_ranks(total.item(), len(val_loader)))
        sched.step(val_losses[-1])
        say(f"Epoch {epoch + 1}/{num_epochs}:\n  Train Loss: {train_losses[-1]:.6f}\n  Val Loss: {val_losses[-1]:.6f}\n"
            f"  Learning Rate: {step.lr:.2e}")
        if val_losses[-1] < best:
            best = val_losses[-1]
            if rank0:
                torch.save({"epoch": epoch, "model_state_dict": model.state_dict(),
                            "optimizer_state_dict": step.state_dict(), "train_loss": train_losses[-1],
                            "val_loss": val_losses[-1], "train_losses": train_losses, "val_losses": val_losses},
                           checkpoint_path)
            say(f"  New best model saved! (Val Loss: {best:.6f})")
        say("-" * 50)
    say(f"Training completed! Best validation loss: {best:.6f}")
    return train_losses, val_losses


def crop_size(text):
    """argparse type of --crop: a multiple of 16, at least 16."""
    try:
        return crops.check_size(int(text))
    except ValueError:
        raise argparse.ArgumentTypeError(f"crop size must be a multiple of 16 and at least 16, got {text!r}") from None


def main(argv=None):
    """python model/train.py --data-dir D [--epochs 100 --batch-size 8 --device auto --val-split 0.2]
    (reference model/train.py:251-313); --frame-cache, --color and --crop S are opt-in additions (see
    FrameTripletDataset and model/framecache.py). Data parallel over the GPUs of a box:

        torchrun --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 model/train.py --data-dir D ...

    one process per GPU, NCCL all-reduce of the gradients (the only collective), --batch-size is per GPU."""
    ap = argparse.ArgumentParser(description="Train Frame Interpolation UNet (B200 training step)")
    ap.add_argument("--data-dir", required=True)
    ap.add_argument("--epochs", type=int, default=100)
    ap.add_argument("--batch-size", type=int, default=8)
    ap.add_argument("--device", default="auto")
    ap.add_argument("--val-split", type=float, default=0.2)
    ap.add_argument("--lr", type=float, default=1e-4)
    ap.add_argument("--no-cuda-graph", action="store_true", help="run the step eagerly instead of replaying CUDA graphs")
    ap.add_argument("--frame-cache", action="store_true",
                    help="decode every frame once into GPU memory (64 KB a frame) and build batches there instead of "
                         "decoding three files per sample in DataLoader workers")
    ap.add_argument("--color", action="store_true",
                    help="train UNet(6, 3) on BGR frames, the colour model FrameInterpolator runs once per frame pair")
    ap.add_argument("--crop", type=crop_size, default=None, metavar="S",
                    help="train on random S x S windows of frames at their native size (S a multiple of 16), mirrored "
                         "and with the input pair swapped at random, instead of resizing every frame to 256x256")
    args = ap.parse_args(argv)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1:
        local = int(os.environ.get("LOCAL_RANK", "0"))
        device = torch.device("cuda", local)
        torch.cuda.set_device(device)
        dist.init_process_group("nccl", device_id=device)
    else:
        device = torch.device("cuda" if args.device == "auto" else args.device)
    E.require_cuda(device)
    rank0 = world == 1 or dist.get_rank() == 0
    data = FrameTripletDataset(args.data_dir, color=args.color, crop=args.crop)
    n_val = int(len(data) * args.val_split)
    split_gen = torch.Generator().manual_seed(0) if world > 1 else None     # every rank must draw the same split
    train_set, val_set = torch.utils.data.random_split(data, [len(data) - n_val, n_val], generator=split_gen)
    if args.crop is not None:      # validation: centre windows, no mirror or swap
        val_set = torch.utils.data.Subset(data.for_validation(), val_set.indices)
    if rank0:
        print(f"Dataset split: {len(train_set)} train, {len(val_set)} validation")
    cache = None
    if args.frame_cache:
        try:
            from .framecache import CachedTripletLoader, FrameCache, build_info
        except ImportError:
            from framecache import CachedTripletLoader, FrameCache, build_info
        cache = FrameCache.build(data, device)        # one cache: train and validation triplets share its frames
        if rank0:
            print(build_info(cache))

    def mk(d, shuffle):
        sampler = None
        if world > 1:
            sampler = torch.utils.data.distributed.DistributedSampler(d, shuffle=shuffle, drop_last=shuffle)
        if cache is not None:
            return CachedTripletLoader(d, cache, args.batch_size, sampler=sampler, shuffle=shuffle and sampler is None)
        return torch.utils.data.DataLoader(d, batch_size=args.batch_size, shuffle=shuffle and sampler is None,
                                           sampler=sampler, num_workers=4, pin_memory=True)

    model = (UNet(6, 3, bilinear=True) if args.color else FrameInterpolationUNet(bilinear=True)).to(device)
    if rank0:
        print(f"Model parameters: {sum(p.numel() for p in model.parameters()):,} total")
    try:
        train_model(model, mk(train_set, True), mk(val_set, False), num_epochs=args.epochs, device=device, lr=args.lr,
                    cuda_graph=not args.no_cuda_graph)
    finally:
        if world > 1:
            dist.destroy_process_group()
    if rank0:
        print("Training completed successfully!")


if __name__ == "__main__":
    main()
