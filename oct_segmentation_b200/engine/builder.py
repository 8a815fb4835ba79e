"""Op-list builder: turns layer calls into device buffers + C-ABI launches.

A ``Builder`` is used once per (network, batch, resolution, input dtype): lowering code
(engine/lower.py) calls ``conv`` / ``stem`` / ``maxpool`` / ``dwconv`` / ``se_project`` in
network order; each call records one op: the activations it reads and writes (symbolic ``Act``
buffers) and a ``make`` closure.  ``finalize()`` then places every activation in ONE arena by
liveness (a buffer's bytes are reused as soon as its last reader has run -- only feature taps that
a test wants to inspect are pinned), binds the tensors and calls every ``make`` (which creates the
kernel plan with the final device pointers).  ``run()`` replays the op list on the current stream;
``CompiledNet`` (engine/network.py) captures that replay in a CUDA graph.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Sequence, Tuple

import torch

from .. import _lib
from .conv import (Act, ConvGeom, ConvPlan, d2s_weights, dense_macs, pad8, pad_bias, pixel_pack_factor, plan_conv,
                   plan_pixel_packed)


def fold_bn(w: torch.Tensor, bn: Optional[torch.nn.BatchNorm2d], conv_bias: Optional[torch.Tensor] = None,
            out_dim: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """Eval-mode BatchNorm folded into the preceding conv in fp32 (SURVEY.md App. B.4):
    w' = w*g/sqrt(v+eps);  b' = (b - mean)*g/sqrt(v+eps) + beta."""
    w = w.detach().float().cpu()
    cout = w.shape[out_dim]
    b = conv_bias.detach().float().cpu() if conv_bias is not None else torch.zeros(cout)
    if bn is None:
        return w, b
    scale = bn.weight.detach().float().cpu() / torch.sqrt(bn.running_var.detach().float().cpu() + bn.eps)
    shape = [1] * w.dim()
    shape[out_dim] = cout
    return w * scale.view(shape), (b - bn.running_mean.detach().float().cpu()) * scale + bn.bias.detach().float().cpu()


def stem_s2d_weights(w: torch.Tensor, k: int, pad: Tuple[int, int]) -> Tuple[torch.Tensor, Tuple[int, int]]:
    """Weights of the stride-1 conv on the 2x2 space-to-depth input that equals a stride-2 k x k conv with
    top/left padding ``pad``: returns (w2 [Cout, 12, kq_h, kq_w], (q0_h, q0_w)) where q0 <= 0 is the first
    tap offset (so the new conv pads -q0 at the top/left).  Input row 2*oy + ky - pad = 2*(oy + q) + d."""
    w = w.detach().float().cpu()
    cout = w.shape[0]
    qs = [[((t - p) // 2, (t - p) % 2) for t in range(k)] for p in pad]          # per axis: tap -> (q, d)
    q0 = tuple(min(q for q, _ in axis) for axis in qs)
    kq = tuple(max(q for q, _ in axis) - q0[i] + 1 for i, axis in enumerate(qs))
    w2 = torch.zeros(cout, 12, kq[0], kq[1])
    for ky, (qy, dy) in enumerate(qs[0]):
        for kx, (qx, dx) in enumerate(qs[1]):
            c0 = (dy * 2 + dx) * 3
            w2[:, c0:c0 + 3, qy - q0[0], qx - q0[1]] = w[:, :, ky, kx]
    return w2, q0


class _Op:
    """One recorded op.  kind: kernel family (conv_tc | dwconv | se | pack | maxpool); macs: algorithmic MACs of a
    tensor-core launch, None otherwise; nbytes: algorithmic HBM bytes (activations read + written once, + weights)."""
    __slots__ = ('name', 'kind', 'make', 'reads', 'writes', 'macs', 'nbytes')

    def __init__(self, name, kind, make, reads, writes, macs, nbytes):
        self.name, self.kind, self.make, self.reads, self.writes = name, kind, make, reads, writes
        self.macs, self.nbytes = macs, nbytes


def plan_arena(items: Sequence[Tuple[int, int, int]], align: int = 256) -> Tuple[List[int], int]:
    """items: (nbytes, first_op, last_op) with inclusive op-index intervals.  Returns (offsets, arena bytes).
    Greedy first-fit over the buffers sorted by size: each buffer takes the lowest offset that is free of every
    already-placed buffer whose lifetime overlaps its own."""
    order = sorted(range(len(items)), key=lambda i: (-items[i][0], items[i][1]))
    offsets = [0] * len(items)
    placed: List[int] = []
    top = 0
    for i in order:
        size, lo, hi = items[i]
        size = (size + align - 1) // align * align
        busy = sorted((offsets[j], offsets[j] + (items[j][0] + align - 1) // align * align) for j in placed
                      if not (items[j][2] < lo or hi < items[j][1]))
        off = 0
        for b0, b1 in busy:
            if off + size <= b0:
                break
            off = max(off, b1)
        offsets[i] = off
        placed.append(i)
        top = max(top, off + size)
    return offsets, top


class Builder:
    def __init__(self, device: torch.device, N: int, reuse: bool = True):
        self.lib = _lib.load()
        self.device = torch.device(device)
        self.N = N
        self.reuse = reuse           # False: every activation keeps its own bytes (in-situ checks read dead inputs)
        self.ops: List[Callable[[], None]] = []   # one launch function per record, created by finalize()
        self.op_fused_macs = {}                  # always empty; kept because bench.py reads it (op_fused_macs.get)
        self.macs = 0              # algorithmic MACs of the reference graph (dense count)
        self.launches = 0
        self.act_bytes = 0         # sum of all activation buffers (what a no-reuse allocation would take)
        self.arena_bytes = 0       # bytes actually allocated for them
        self._records: List[_Op] = []
        self._acts: List[Act] = []
        self._pinned: List[Act] = []
        self._keep: List[object] = []
        self._final = False

    # per-op views of the op records (see _Op)
    @property
    def op_names(self) -> Tuple[str, ...]:
        return tuple(op.name for op in self._records)

    @property
    def op_kinds(self) -> Tuple[str, ...]:
        return tuple(op.kind for op in self._records)

    @property
    def op_macs(self) -> Tuple[Optional[int], ...]:
        return tuple(op.macs for op in self._records)

    @property
    def op_bytes(self) -> Tuple[int, ...]:
        return tuple(op.nbytes for op in self._records)

    # ------------------------------------------------------------------ buffers
    def new_act(self, H: int, W: int, C: int) -> Act:
        a = Act.symbolic((self.N, H, W, pad8(C)), C)
        self._acts.append(a)
        self.act_bytes += a.nbytes
        return a

    def new_scratch(self, shape: Tuple[int, ...], dtype: torch.dtype) -> Act:
        """Arena-resident temporary that is not an activation (e.g. the per-image projection weights)."""
        a = Act.symbolic(tuple(shape), 0, dtype)
        self._acts.append(a)
        self.act_bytes += a.nbytes
        return a

    def pin(self, acts: Sequence[Act]) -> None:
        """Keep these buffers intact until the end of the network (feature taps read by diagnostics)."""
        self._pinned += list(acts)

    def _add(self, name: str, make: Callable[[], Callable[[], None]], reads: Sequence[Optional[Act]] = (),
             writes: Sequence[Act] = (), *, kind: str, macs: Optional[int] = None, launches: int = 1,
             extra_bytes: int = 0) -> None:
        assert not self._final, 'builder already finalized'
        reads, writes = [a for a in reads if a is not None], list(writes)
        nbytes = sum(a.nbytes for a in reads + writes) + int(extra_bytes)
        self._records.append(_Op(name, kind, make, reads, writes, macs, nbytes))
        self.launches += launches

    def plan_buffers(self) -> Tuple[List[Act], List[int], int]:
        """Liveness of every arena buffer over the recorded op list -> (buffers, byte offsets, arena bytes).
        Pure host arithmetic (no device needed)."""
        n_ops = len(self._records)
        first, last = {}, {}
        for i, op in enumerate(self._records):
            for a in op.writes:
                first.setdefault(id(a), i)
                last[id(a)] = max(last.get(id(a), i), i)
            for a in op.reads:
                if a._t is None:
                    assert id(a) in first, f'{op.name} reads a buffer nobody wrote'
                    last[id(a)] = i
        for a in self._pinned:
            if id(a) in first:
                last[id(a)] = n_ops
        acts = [a for a in self._acts if id(a) in first]
        if not self.reuse:
            items = [(a.nbytes, 0, n_ops) for a in acts]
        else:
            items = [(a.nbytes, first[id(a)], last[id(a)]) for a in acts]
        offsets, total = plan_arena(items)
        return acts, offsets, total

    def finalize(self) -> None:
        """Place the activations (liveness-based arena), bind them and create every kernel plan."""
        if self._final:
            return
        acts, offsets, total = self.plan_buffers()
        self.arena_bytes = total
        with torch.cuda.device(self.device):
            self._arena = torch.zeros(max(total, 256), dtype=torch.uint8, device=self.device)
        for a, off in zip(acts, offsets):
            a.t = self._arena[off:off + a.nbytes].view(a.dtype).view(a.shape)
        self._final = True
        self.ops = [op.make() for op in self._records]
        for op in self._records:
            op.make = None           # the plans hold what they launch; free the host-side packed weights

    def run(self) -> None:
        self.finalize()
        for op in self.ops:
            op()

    # ------------------------------------------------------------------ tensor-core conv
    def _add_conv(self, name: str, srcs: List[Act], geom: ConvGeom, packed: torch.Tensor | Act,
                  bias_rows: torch.Tensor, macs: int,
                  out_hw: Tuple[int, int], cout: int, f: int = 0, *, act: str, res: Optional[Act] = None,
                  res_mode: str = 'none', out_mode: str = 'bf16_nhwc', out_tensor: Optional[torch.Tensor] = None,
                  **plan_kw) -> Optional[Act]:
        """Records one planned tensor-core conv: allocates its bf16 NHWC output (or checks the NCHW `out_tensor`),
        counts its MACs and bytes and creates its ConvPlan at finalize().  f > 1: sources, output and residual are
        seen through their f-pixel packed view.  `packed` is the weight tensor, or the arena buffer of per-image
        weights (se_project); `plan_kw` are the form's extra ConvPlan arguments."""
        out, out_bytes = None, 0
        if out_mode == 'bf16_nhwc':
            out = self.new_act(out_hw[0], out_hw[1], cout)
        else:
            planes = plan_kw['head'][0].shape[0] if 'head' in plan_kw else cout
            assert out_tensor is not None and tuple(out_tensor.shape) == (self.N, planes) + tuple(out_hw) and res is None
            out_bytes = out_tensor.numel() * out_tensor.element_size()
        arena_w = packed if isinstance(packed, Act) else None

        def view(t):        # the pixel-packed view of an NHWC tensor (same memory, f pixels per row)
            return t.view(t.shape[0], t.shape[1], t.shape[2] // f, f * t.shape[3]) if f > 1 else t

        def make():
            plan = ConvPlan(geom, arena_w.t if arena_w is not None else packed, bias_rows, [view(a.t) for a in srcs],
                            view(out.t) if out is not None else out_tensor, out_mode=out_mode, act=act,
                            res=view(res.t) if res is not None else None, res_mode=res_mode, name=name, **plan_kw)
            self._keep.append(plan)
            return plan.run
        self.macs += macs
        wbytes = geom.phases * geom.n_tiles_n * geom.BN * geom.Ktot * 2
        self._add(name, make, srcs + [res, arena_w], [out] if out is not None else [], kind='conv_tc', macs=macs,
                  extra_bytes=out_bytes + wbytes)
        return out

    def conv(self, srcs: Sequence[Tuple[Act, bool]], w: torch.Tensor, b: Optional[torch.Tensor], *, name: str,
             stride: int = 1, pad: Tuple[int, int] = (0, 0), groups: int = 1, transposed: bool = False,
             act: str = 'none', res: Optional[Act] = None, res_mode: str = 'none',
             out_hw: Optional[Tuple[int, int]] = None, out_mode: str = 'bf16_nhwc',
             out_tensor: Optional[torch.Tensor] = None,
             head: Optional[Tuple[torch.Tensor, Optional[torch.Tensor]]] = None) -> Optional[Act]:
        """head = (weight [classes, cout, 1, 1], bias | None) of a 1x1 segmentation head: it is applied to this conv's
        activated output inside the epilogue (fp32, octseg.h `head_classes`), `out_tensor` (N, classes, H, W) receives the
        head's logits / masks and the conv's own output is never stored."""
        cout = w.shape[1] if transposed else w.shape[0]
        bf16_out = out_mode == 'bf16_nhwc'
        cout_store = pad8(cout) if bf16_out else cout        # channels per output pixel in memory
        acts, ups = [a for a, _ in srcs], [up for _, up in srcs]
        a0 = acts[0]

        # narrow decoder conv over cat([up(x), skips...]): the half-resolution tile grid of the fused form
        # reads the full-resolution skips through stride-2 boxes, 9 per tile and phase, and is bound by
        # that activation feed.  Split it: depth-to-space conv of the upsampled part (no bias/act), then a
        # plain 3x3 conv of the skips (wide boxes: 3x less feed) that adds the first part before the
        # activation.  Costs one extra bf16 round trip of the (narrow) output.
        if (bf16_out and not transposed and len(srcs) > 1 and ups[0] and not any(ups[1:]) and groups == 1
                and res is None and cout <= 64 and acts[1].W >= 112):
            part = self.conv([srcs[0]], w[:, :a0.C], None, name=name + '.up', pad=(1, 1), act='none')
            return self.conv(list(srcs[1:]), w[:, a0.C:], b, name=name, pad=(1, 1), act=act, res=part,
                             res_mode='before_act')

        f, plan_kw = 0, {}
        if (not transposed and groups == 1 and stride == 1 and not any(ups) and out_hw is None
                and pad[0] == (w.shape[2] - 1) // 2 and pad[1] == (w.shape[3] - 1) // 2):
            # the fused-head epilogue packs at most 4 pixels per row
            f = pixel_pack_factor([a.Cp for a in acts], a0.W, w.shape[3], cout_store, 8 if head is None else 4)
        if f:
            # narrow stride-1 convs: pack f adjacent pixels into one GEMM row (same memory, wider view)
            geom, packed, bias_rows = plan_pixel_packed(acts, w, b, f, pad, cout_store, out_bf16=bf16_out)
            out_hw = (a0.H, a0.W)
            if not bf16_out:
                plan_kw['out_pack'] = f
        elif (bf16_out and len(srcs) == 1 and (transposed or ups[0]) and res is None and 4 * cout_store <= 256
                and groups == 1):
            # single-source upsample+conv / ConvTranspose with few output channels: one depth-to-space conv
            # on the half-resolution grid (N = 4*Cout) instead of four N = Cout phase problems
            wp, bp = d2s_weights(w, b, transposed, cout_store)
            geom, packed = plan_conv([((a0.N, a0.H, a0.W, a0.C, a0.Cp), False)], wp, pad=(1, 1))
            bias_rows = pad_bias(bp, geom, 4 * cout_store)
            out_hw = (2 * a0.H, 2 * a0.W)
            plan_kw['d2s'] = cout_store
        else:
            geom, packed = plan_conv([((a.N, a.H, a.W, a.C, a.Cp), up) for a, up in srcs], w, out_hw=out_hw,
                                     stride=stride, pad=pad, groups=groups, transposed=transposed, out_bf16=bf16_out)
            bias_rows = pad_bias(b, geom, cout, groups)
            out_hw = (geom.out_H, geom.out_W)
        macs = dense_macs(w, self.N, out_hw, transposed)

        if head is not None:
            hw = head[0].detach().float().cpu().reshape(head[0].shape[0], -1)
            assert (not bf16_out and res is None and not transposed and hw.shape[1] == cout and cout % 16 == 0
                    and hw.shape[0] <= 4)
            assert cout <= 64, 'a fused head reads at most 64 channels per pixel'
            assert geom.n_tiles_n == 1, 'a fused head needs all of a pixel\'s channels in one tile'
            hb = head[1].detach().float().cpu() if head[1] is not None else torch.zeros(hw.shape[0])
            cb = b.detach().float().cpu() if b is not None else torch.zeros(cout)
            plan_kw['head'] = (hw, hb, cb)
            macs += dense_macs(hw, self.N, out_hw)
        return self._add_conv(name, acts, geom, packed, bias_rows, macs, out_hw, cout, f, act=act, res=res,
                              res_mode=res_mode, out_mode=out_mode, out_tensor=out_tensor, **plan_kw)

    # ------------------------------------------------------------------ CUDA-core kernels
    def stem(self, x: torch.Tensor, in_dtype: str, w: torch.Tensor, b: torch.Tensor, *, name: str, k: int,
             stride: int, pad: Tuple[int, int], out_hw: Tuple[int, int], act: str,
             mean: Optional[Sequence[float]] = None, std: Optional[Sequence[float]] = None) -> Act:
        """Stride-2 k x k stem conv on the 3-channel input, as a tensor-core conv over the input's
        space-to-depth form.  x: logical (N,3,H,W) view of the static input buffer (any strides).

        in[2(oy+qy)+dy] with ky = 2qy + dy + pad: the k taps of a row fold into ceil-ish k/2 taps qy of the
        2x2-packed tensor (12 channels, padded to 16); weights move to w2[co][(dy*2+dx)*3+c][qy-q0][qx-q0]."""
        assert stride == 2
        if in_dtype == 's2d':
            N, H, W = x.shape[0], 2 * x.shape[1], 2 * x.shape[2]
        else:
            assert x.shape[1] == 3
            N, _, H, W = x.shape
        cout = w.shape[0]
        if in_dtype == 's2d':
            # the caller (pipeline: octseg_preprocess_resize_s2d) writes the packed input itself: `x` IS the
            # (N, H/2, W/2, 16) bf16 tensor, an external buffer that never enters the arena
            assert x.dtype == torch.bfloat16 and tuple(x.shape) == (N, H // 2, W // 2, 16) and (mean is None and std is None)
            x2 = Act(x, 12)
            self._keep += [x]
        else:
            x2 = self.new_act(H // 2, W // 2, 12)
            sn, sc, sh, sw = x.stride()
            mean_a = (C.c_float * 3)(*mean) if mean is not None else None
            istd_a = (C.c_float * 3)(*[1.0 / s for s in std]) if std is not None else None
            self._keep += [x]
            lib, dt = self.lib, {'f32': 0, 'u8': 1}[in_dtype]

            def pack_op():
                _lib.check(lib.octseg_stem_pack(x.data_ptr(), dt, sn, sc, sh, sw, N, H, W, mean_a, istd_a,
                                                x2.t.data_ptr(), _lib.stream_ptr()), name + '.pack')
            self._add(name + '.pack', lambda: pack_op, [], [x2], kind='pack', extra_bytes=N * H * W * 3 * (1 if in_dtype == 'u8' else 4))
        w2, q0 = stem_s2d_weights(w, k, pad)
        assert q0[0] <= 0 and q0[1] <= 0
        geom, packed = plan_conv([((x2.N, x2.H, x2.W, x2.C, x2.Cp), False)], w2, out_hw=out_hw, pad=(-q0[0], -q0[1]))
        return self._add_conv(name, [x2], geom, packed, pad_bias(b, geom, cout), dense_macs(w, N, out_hw), out_hw, cout,
                              act=act)

    def maxpool(self, x: Act, *, name: str) -> Act:
        Ho, Wo = (x.H + 2 - 3) // 2 + 1, (x.W + 2 - 3) // 2 + 1
        out = self.new_act(Ho, Wo, x.C)
        lib = self.lib

        def op():
            _lib.check(lib.octseg_maxpool3x3s2(x.t.data_ptr(), out.t.data_ptr(), x.N, x.H, x.W, x.Cp, Ho, Wo,
                                               _lib.stream_ptr()), name)
        self._add(name, lambda: op, [x], [out], kind='maxpool')
        return out

    def new_pool(self, C: int, out_hw: Tuple[int, int]) -> torch.Tensor:
        """Squeeze-excite partial-sum buffer fp32 [N][slots][C] for a depthwise launch of this shape: every slot is
        written exactly once per launch and octseg_se_hidden adds them in order (no atomics)."""
        slots = self.lib.octseg_dwconv_pool_slots(C, out_hw[0], out_hw[1])
        return torch.zeros(self.N, slots, C, dtype=torch.float32, device=self.device)

    def dwconv(self, x: Act, w: torch.Tensor, b: torch.Tensor, *, name: str, k: int, stride: int,
               pad: Tuple[int, int], out_hw: Tuple[int, int], act: str, pool: Optional[torch.Tensor]) -> Act:
        assert x.C % 8 == 0
        out = self.new_act(out_hw[0], out_hw[1], x.C)
        wk = w.detach().float().reshape(x.C, k, k).permute(1, 2, 0).contiguous().to(torch.bfloat16).to(self.device)  # [kh][kw][C]
        bk = b.detach().float().contiguous().to(self.device)
        self._keep += [wk, bk]
        lib, a = self.lib, _lib.ACT[act]

        def op():   # `pool` (new_pool): write-once slots, summed by octseg_se_hidden
            _lib.check(lib.octseg_dwconv(x.t.data_ptr(), wk.data_ptr(), bk.data_ptr(), out.t.data_ptr(), x.N, x.H,
                                         x.W, x.C, k, stride, pad[0], pad[1], out_hw[0], out_hw[1], a,
                                         pool.data_ptr() if pool is not None else None,
                                         pool.shape[1] if pool is not None else 0, _lib.stream_ptr()), name)
        self.macs += x.N * out_hw[0] * out_hw[1] * x.C * k * k
        self._add(name, lambda: op, [x], [out], kind='dwconv')
        return out

    def se_project(self, x: Act, pool: torch.Tensor, w1, b1, w2, b2, wp: torch.Tensor, bp: torch.Tensor, *,
                   name: str, res: Optional[Act]) -> Act:
        """Squeeze-excite gate folded into the projection 1x1: per-image weights
        bf16(w[:, k] * gate[n, k]) feed the tensor-core conv (octseg_scale_weights)."""
        N, C_mid, cr = x.N, x.C, w1.shape[0]
        dev = self.device
        w1d = w1.detach().float().reshape(cr, C_mid).contiguous().to(dev)
        b1d = b1.detach().float().contiguous().to(dev)
        w2d = w2.detach().float().reshape(C_mid, cr).t().contiguous().to(dev)      # [Cr][C]
        b2d = b2.detach().float().contiguous().to(dev)
        hidden = torch.empty(N, cr, dtype=torch.float32, device=dev)
        gate = torch.empty(N, C_mid, dtype=torch.float32, device=dev)
        cout = wp.shape[0]
        cs = pad8(cout)
        # narrow projections (<= 32 output channels, the 448 x 448 stage): two adjacent pixels per GEMM row, so the
        # output rows are 128 bytes and K is a whole 64-channel chunk (same memory, wider view; block-diagonal weights)
        f = 2 if (cs <= 32 and x.Cp <= 64 and x.C == x.Cp and x.W % 2 == 0 and (res is None or res.Cp == cs)) else 1
        if f > 1:
            geom, packed32, bias_rows = plan_pixel_packed([x], wp, bp, f, (0, 0), cs, packed_dtype=torch.float32)
        else:
            geom, packed32 = plan_conv([((N, x.H, x.W, x.C, x.Cp), False)], wp, packed_dtype=torch.float32)
            bias_rows = pad_bias(bp, geom, cout)
        rows, Ktot = packed32.shape[1], packed32.shape[2]
        base = packed32[0].contiguous().to(dev)                                    # fp32 [rows][Ktot]
        wn = self.new_scratch((N, rows, Ktot), torch.bfloat16)                     # per-image weights: dead after the conv
        self._keep += [w1d, b1d, w2d, b2d, hidden, gate, base]
        lib, inv_hw = self.lib, 1.0 / float(x.H * x.W)

        def gate_op():
            st = _lib.stream_ptr()
            _lib.check(lib.octseg_se_hidden(pool.data_ptr(), pool.shape[1], gate.data_ptr(), inv_hw, w1d.data_ptr(), b1d.data_ptr(),
                                            hidden.data_ptr(), N, C_mid, cr, st), name + '.se_hidden')   # `gate` doubles as the [N][C] sums scratch
            _lib.check(lib.octseg_se_gate(hidden.data_ptr(), w2d.data_ptr(), b2d.data_ptr(), gate.data_ptr(),
                                          None, N, C_mid, cr, st), name + '.se_gate')
            _lib.check(lib.octseg_se_scale_weights(gate.data_ptr(), base.data_ptr(), wn.t.data_ptr(), N, rows, Ktot,
                                                   f * C_mid, C_mid, st), name + '.se_scale_weights')
        self.macs += N * 2 * C_mid * cr
        self._add(name + '.se', lambda: gate_op, [], [wn], launches=3 + int(pool.shape[1] > 1), kind='se')
        return self._add_conv(name, [x], geom, wn, bias_rows, dense_macs(wp, N, (x.H, x.W)), (x.H, x.W), cout, f,
                              act='none', res=res, res_mode='before_act' if res is not None else 'none',
                              per_image_weights=True)
