"""Test-only stand-in for engine.builder.Builder that executes each lowered op with plain torch
fp32 ops on CPU.  It lets the CPU suite check the LOWERING (graph wiring, BN folding, static
padding, concat order, skip routing) against the oracle without a GPU; kernel arithmetic itself
is covered by tests/test_conv_plan.py (emulated) and the -m gpu tests (real)."""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oct_segmentation_b200.engine.conv import Act, pad8
from tests.conv_cases import act_fn


def _nchw(a: Act) -> torch.Tensor:
    return a.t[..., :a.C].permute(0, 3, 1, 2).float()


def _act(x_nchw: torch.Tensor) -> Act:
    n, c, h, w = x_nchw.shape
    t = torch.zeros(n, h, w, pad8(c), device=x_nchw.device)
    t[..., :c] = x_nchw.permute(0, 2, 3, 1)
    return Act(t, c)


class CpuBuilder:
    def __init__(self, N, device='cpu'):
        self.N, self.device, self.macs, self.launches = N, torch.device(device), 0, 0

    def _d(self, t):
        return None if t is None else t.detach().float().to(self.device)

    def stem(self, x, in_dtype, w, b, *, name, k, stride, pad, out_hw, act, mean=None, std=None):
        x, w, b = x.float(), self._d(w), self._d(b)
        if mean is not None:
            x = (x - torch.tensor(mean, device=x.device).view(1, 3, 1, 1)) / torch.tensor(std, device=x.device).view(1, 3, 1, 1)
        H, W = x.shape[2:]
        pb = (out_hw[0] - 1) * stride + k - H - pad[0]
        pr = (out_hw[1] - 1) * stride + k - W - pad[1]
        y = F.conv2d(F.pad(x, (pad[1], max(pr, 0), pad[0], max(pb, 0))), w, b, stride=stride)
        return _act(act_fn(y[:, :, :out_hw[0], :out_hw[1]], act))

    def maxpool(self, x, *, name):
        return _act(F.max_pool2d(_nchw(x), 3, 2, 1))

    def conv(self, srcs, w, b, *, name, stride=1, pad=(0, 0), groups=1, transposed=False, act='none', res=None,
             res_mode='none', out_hw=None, out_mode='bf16_nhwc', out_tensor=None, head=None):
        w, b = self._d(w), self._d(b)
        parts = [F.interpolate(_nchw(a), scale_factor=2, mode='nearest') if up else _nchw(a) for a, up in srcs]
        x = torch.cat(parts, 1)
        if transposed:
            y = F.conv_transpose2d(x, w, b, stride=2, padding=1)
        else:
            y = F.conv2d(x, w, b, stride=stride, padding=pad, groups=groups)
        if res_mode == 'before_act':
            y = y + _nchw(res)
        y = act_fn(y, act)
        if res_mode == 'after_act':
            y = y + _nchw(res)
        if head is not None:                           # fused 1x1 segmentation head: fp32 on the activated output
            y = F.conv2d(y, self._d(head[0]).float().reshape(head[0].shape[0], -1, 1, 1), self._d(head[1]))
        if out_mode == 'bf16_nhwc':
            return _act(y)
        out_tensor.copy_(y if out_mode == 'f32_nchw' else (y > 0))
        return None

    def dwconv(self, x, w, b, *, name, k, stride, pad, out_hw, act, pool):
        xin, w, b = _nchw(x), self._d(w), self._d(b)
        H, W = xin.shape[2:]
        pb = (out_hw[0] - 1) * stride + k - H - pad[0]
        pr = (out_hw[1] - 1) * stride + k - W - pad[1]
        y = act_fn(F.conv2d(F.pad(xin, (pad[1], max(pr, 0), pad[0], max(pb, 0))), w, b, stride=stride, groups=x.C), act)
        pool.zero_()
        pool[:, 0].copy_(y.sum(dim=(2, 3)))
        return _act(y)

    def new_pool(self, C, out_hw):
        return torch.zeros(self.N, 1, C, device=self.device)

    def se_project(self, x, pool, w1, b1, w2, b2, wp, bp, *, name, res):
        xin = _nchw(x)
        w1, b1, w2, b2, wp, bp = (self._d(t) for t in (w1, b1, w2, b2, wp, bp))
        mean = pool.sum(1) / float(x.H * x.W)
        h = F.linear(mean, w1.flatten(1), b1)
        h = h * torch.sigmoid(h)
        gate = torch.sigmoid(F.linear(h, w2.flatten(1), b2))
        y = F.conv2d(xin * gate[:, :, None, None], wp, bp)
        if res is not None:
            y = y + _nchw(res)
        return _act(y)


def _r16(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).float()


class Bf16Builder(CpuBuilder):
    """Same ops with the engine's storage precision: folded weights of tensor-core convs rounded
    to bf16, every activation rounded to bf16 when it is written, fp32 accumulation.  The GPU
    kernels must match this pipeline tightly; its distance to the fp32 oracle is the price of
    bf16 storage, not a kernel property."""

    def stem(self, x, in_dtype, w, b, **k):
        a = super().stem(x, in_dtype, w, b, **k)
        a.t = _r16(a.t)
        return a

    def conv(self, srcs, w, b, **k):
        a = super().conv(srcs, _r16(w.detach().float()), b, **k)
        if a is not None:
            a.t = _r16(a.t)
        return a

    def dwconv(self, x, w, b, **k):
        a = super().dwconv(x, _r16(w.detach().float()), b, **k)        # the kernel keeps dw weights in bf16
        a.t = _r16(a.t)
        k['pool'].zero_()
        k['pool'][:, 0].copy_(a.t[..., :a.C].sum(dim=(1, 2)))
        return a

    def se_project(self, x, pool, w1, b1, w2, b2, wp, bp, **k):
        xin = _nchw(x)
        w1, b1, w2, b2, wp, bp = (self._d(t) for t in (w1, b1, w2, b2, wp, bp))
        mean = pool.sum(1) / float(x.H * x.W)
        h = F.linear(mean, w1.flatten(1), b1)
        h = h * torch.sigmoid(h)
        gate = torch.sigmoid(F.linear(h, w2.flatten(1), b2))
        # gate folded into per-image bf16 weights, exactly like octseg_scale_weights
        wn = _r16(wp.flatten(1)[None] * gate[:, None, :])                      # [N, cout, cmid]
        y = torch.einsum('nchw,noc->nohw', xin, wn) + bp.view(1, -1, 1, 1)
        if k.get('res') is not None:
            y = y + _nchw(k['res'])
        a = _act(y)
        a.t = _r16(a.t)
        return a


def run_lowered(model, x_nchw: torch.Tensor, norm=None, bf16: bool = False, return_stages: bool = False):
    """Run a product smp model's lowering through the torch-op builder; returns fp32 logits NCHW."""
    from oct_segmentation_b200.engine.lower import ENCODER_LOWERING, lower_decoder_and_head
    b = (Bf16Builder if bf16 else CpuBuilder)(x_nchw.shape[0], x_nchw.device)
    feats = ENCODER_LOWERING[model.encoder.kind](b, model.encoder, x_nchw, 'f32', norm)
    out = torch.zeros(x_nchw.shape[0], model.segmentation_head[0].out_channels, x_nchw.shape[2], x_nchw.shape[3],
                      device=x_nchw.device)
    y = lower_decoder_and_head(b, model, feats, out, 'f32_nchw')
    if return_stages:
        return out, [_nchw(f) for f in feats], (_nchw(y) if y is not None else None)      # y None: head fused (LinkNet)
    return out
