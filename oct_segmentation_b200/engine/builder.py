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
from .conv import Act, ConvPlan, d2s_weights, pack_conv_weights, pad8, pad_bias, pixel_pack_factor, plan_conv


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
    __slots__ = ('name', 'make', 'reads', 'writes', 'tc_macs')

    def __init__(self, name, make, reads, writes, tc_macs):
        self.name, self.make, self.reads, self.writes, self.tc_macs = name, make, reads, writes, tc_macs


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
        self.ops: List[Callable[[], None]] = []
        self.op_names: List[str] = []
        self.op_macs: List[Optional[int]] = []   # algorithmic MACs of tensor-core launches, None otherwise
        self.op_bytes: List[int] = []            # algorithmic HBM bytes per op: activations read + written once, + weights
        self.op_kinds: List[str] = []            # kernel family per op: conv_tc | dwconv | se | pack | maxpool
        self.op_fused_macs = {}                  # always empty; kept because bench.py reads it (op_fused_macs.get)
        self.macs = 0              # algorithmic MACs of the reference graph (dense count)
        self.tc_launches = 0
        self.launches = 0
        self.act_bytes = 0         # sum of all activation buffers (what a no-reuse allocation would take)
        self.arena_bytes = 0       # bytes actually allocated for them
        self._records: List[_Op] = []
        self._acts: List[Act] = []
        self._pinned: List[Act] = []
        self._keep: List[object] = []
        self._final = False

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

    def _add(self, name: str, make: Callable[[], Callable[[], None]], reads: Sequence[Act] = (),
             writes: Sequence[Act] = (), tc_macs: Optional[int] = None, launches: int = 1, extra_bytes: int = 0,
             kind: str = '') -> None:
        assert not self._final, 'builder already finalized'
        self.op_kinds.append(kind or ('conv_tc' if tc_macs is not None else 'other'))
        self._records.append(_Op(name, make, [a for a in reads if a is not None], list(writes), tc_macs))
        self.op_names.append(name)
        self.op_macs.append(tc_macs)
        self.op_bytes.append(sum(a.nbytes for a in list(reads) + list(writes) if a is not None) + int(extra_bytes))
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
        self._records = []

    def run(self) -> None:
        self.finalize()
        for op in self.ops:
            op()

    # ------------------------------------------------------------------ tensor-core conv
    def _add_conv(self, name: str, geom, make_plan: Callable[[], ConvPlan], reads, writes, extra_bytes: int = 0) -> None:
        def make():
            plan = make_plan()
            self._keep.append(plan)
            return plan.run
        self.macs += geom.macs
        self.tc_launches += 1
        wbytes = geom.phases * geom.n_tiles_n * geom.BN * geom.Ktot * 2
        self._add(name, make, reads, writes, tc_macs=geom.macs, extra_bytes=extra_bytes + wbytes)

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
        reads = [a for a, _ in srcs] + [res]
        head_t, n_planes = None, cout
        if head is not None:
            hw = head[0].detach().float().cpu().reshape(head[0].shape[0], -1)
            assert not bf16_out and res is None and not transposed and hw.shape[1] == cout and cout % 16 == 0 and hw.shape[0] <= 4
            hb = head[1].detach().float().cpu() if head[1] is not None else torch.zeros(hw.shape[0])
            cb = b.detach().float().cpu() if b is not None else torch.zeros(cout)
            assert cout <= 64, 'a fused head reads at most 64 channels per pixel'
            head_t, n_planes = (hw, hb, cb), hw.shape[0]
        # narrow stride-1 convs: pack f adjacent pixels into one GEMM row (same memory, wider view)
        f = 0
        if (not transposed and groups == 1 and stride == 1 and not any(up for _, up in srcs) and out_hw is None
                and pad[0] == (w.shape[2] - 1) // 2 and pad[1] == (w.shape[3] - 1) // 2):
            f = pixel_pack_factor([a.Cp for a, _ in srcs], srcs[0][0].W, w.shape[3], pad8(cout) if bf16_out else cout)
            if head_t is not None and f > 4:
                f = 4                                         # the fused-head epilogue packs at most 4 pixels per row
        if f:
            a0 = srcs[0][0]
            cout_store = pad8(cout) if bf16_out else cout
            wp, bp = pack_conv_weights(w, b, [a.C for a, _ in srcs], [a.Cp for a, _ in srcs], f, pad[1], cout_store)
            spec = [((a.N, a.H, a.W // f, f * a.Cp, f * a.Cp), False) for a, _ in srcs]
            geom, packed = plan_conv(spec, wp, stride=1, pad=(pad[0], 1 if w.shape[3] > 1 else 0), out_bf16=bf16_out)
            geom.macs = a0.N * a0.H * a0.W * cout * w.shape[1] * w.shape[2] * w.shape[3]     # dense count of the real op
            bias_rows = pad_bias(bp, geom, f * cout_store)
            out_act = None
            if bf16_out:
                out_act = self.new_act(a0.H, a0.W, cout)
            else:
                assert out_tensor is not None and tuple(out_tensor.shape) == (self.N, n_planes, a0.H, a0.W) and res is None
            if head_t is not None:
                geom.macs += a0.N * a0.H * a0.W * cout * n_planes

            def make_plan():
                views = [a.t.view(a.N, a.H, a.W // f, f * a.Cp) for a, _ in srcs]
                if bf16_out:
                    out_t = out_act.t.view(a0.N, a0.H, a0.W // f, f * cout_store)
                    res_t = res.t.view(a0.N, a0.H, a0.W // f, f * cout_store) if res is not None else None
                    return ConvPlan(geom, packed, bias_rows, views, out_t, out_mode=out_mode, act=act, res=res_t,
                                    res_mode=res_mode, name=name)
                return ConvPlan(geom, packed, bias_rows, views, out_tensor, out_mode=out_mode, act=act, name=name,
                                out_pack=f, out_ldc=n_planes, head=head_t)
            self._add_conv(name, geom, make_plan, reads, [out_act] if out_act is not None else [],
                           extra_bytes=0 if bf16_out else out_tensor.numel() * out_tensor.element_size())
            return out_act

        # narrow decoder conv over cat([up(x), skips...]): the half-resolution tile grid of the fused form
        # reads the full-resolution skips through stride-2 boxes, 9 per tile and phase, and is bound by
        # that activation feed.  Split it: depth-to-space conv of the upsampled part (no bias/act), then a
        # plain 3x3 conv of the skips (wide boxes: 3x less feed) that adds the first part before the
        # activation.  Costs one extra bf16 round trip of the (narrow) output.
        if (bf16_out and not transposed and len(srcs) > 1 and srcs[0][1] and not any(up for _, up in srcs[1:])
                and groups == 1 and res is None and cout <= 64 and srcs[1][0].W >= 112):
            cup = srcs[0][0].C
            part = self.conv([srcs[0]], w[:, :cup], None, name=name + '.up', pad=(1, 1), act='none')
            return self.conv(list(srcs[1:]), w[:, cup:], b, name=name, pad=(1, 1), act=act, res=part,
                             res_mode='before_act')

        # single-source upsample+conv / ConvTranspose with few output channels: one depth-to-space conv
        # on the half-resolution grid (N = 4*Cout) instead of four N = Cout phase problems
        if (bf16_out and len(srcs) == 1 and (transposed or srcs[0][1]) and res is None and 4 * pad8(cout) <= 256
                and groups == 1):
            a0 = srcs[0][0]
            cs = pad8(cout)
            wp, bp = d2s_weights(w, b, transposed, cs)
            geom, packed = plan_conv([((a0.N, a0.H, a0.W, a0.C, a0.Cp), False)], wp, pad=(1, 1))
            cin = w.shape[0] if transposed else w.shape[1]
            geom.macs = a0.N * a0.H * a0.W * cin * cout * (16 if transposed else 36)   # dense count of the real op
            out_act = self.new_act(2 * a0.H, 2 * a0.W, cout)
            bias_rows = pad_bias(bp, geom, 4 * cs)
            self._add_conv(name, geom, lambda: ConvPlan(geom, packed, bias_rows, [a0.t], out_act.t, act=act, name=name,
                                                        out_ldc=out_act.Cp, d2s=cs), reads, [out_act])
            return out_act

        spec = [((a.N, a.H, a.W, a.C, a.Cp), up) for a, up in srcs]
        geom, packed = plan_conv(spec, w, out_hw=out_hw, stride=stride, pad=pad, groups=groups,
                                 transposed=transposed, out_bf16=bf16_out)
        bias_rows = pad_bias(b, geom, cout, groups)
        out_act = None
        if bf16_out:
            out_act = self.new_act(geom.out_H, geom.out_W, cout)
        else:
            assert out_tensor is not None and tuple(out_tensor.shape) == (self.N, n_planes, geom.out_H, geom.out_W)
        if head_t is not None:
            assert geom.n_tiles_n == 1, 'a fused head needs all of a pixel\'s channels in one tile'
            geom.macs += self.N * geom.out_H * geom.out_W * cout * n_planes

        def make_plan():
            return ConvPlan(geom, packed, bias_rows, [a.t for a, _ in srcs], out_act.t if bf16_out else out_tensor,
                            out_mode=out_mode, act=act, res=res.t if res is not None else None, res_mode=res_mode,
                            name=name, out_ldc=None if head_t is None else n_planes, head=head_t)
        self._add_conv(name, geom, make_plan, reads, [out_act] if out_act is not None else [],
                       extra_bytes=0 if bf16_out else out_tensor.numel() * out_tensor.element_size())
        return out_act

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
        out = self.conv([(x2, False)], w2, b, name=name, pad=(-q0[0], -q0[1]), out_hw=out_hw, act=act)
        real = N * out_hw[0] * out_hw[1] * cout * 3 * k * k        # algorithmic MACs: the dense count of the real op
        self.macs += real - self.op_macs[-1]
        self.op_macs[-1] = real
        self._records[-1].tc_macs = real
        return out

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
            wpk, bpk = pack_conv_weights(wp, bp, [x.C], [x.Cp], f, 0, cs)
            spec = [((N, x.H, x.W // f, f * x.Cp, f * x.Cp), False)]
            geom, packed32 = plan_conv(spec, wpk, out_hw=(x.H, x.W // f), packed_dtype=torch.float32)
            geom.macs = N * x.H * x.W * cout * C_mid                                # dense count of the real op
            bias_rows = pad_bias(bpk, geom, f * cs)
        else:
            spec = [((N, x.H, x.W, x.C, x.Cp), False)]
            geom, packed32 = plan_conv(spec, wp, out_hw=(x.H, x.W), packed_dtype=torch.float32)
            bias_rows = pad_bias(bp, geom, cout)
        rows, Ktot = packed32.shape[1], packed32.shape[2]
        base = packed32[0].contiguous().to(dev)                                    # fp32 [rows][Ktot]
        wn = self.new_scratch((N, rows, Ktot), torch.bfloat16)                     # per-image weights: dead after the conv
        out = self.new_act(x.H, x.W, cout)
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
        def make_plan():
            def pk(t):      # the pixel-packed view of an NHWC tensor
                return t.view(t.shape[0], t.shape[1], t.shape[2] // f, f * t.shape[3]) if f > 1 else t
            return ConvPlan(geom, wn.t, bias_rows, [pk(x.t)], pk(out.t), act='none',
                            res=pk(res.t) if res is not None else None,
                            res_mode='before_act' if res is not None else 'none', per_image_weights=True, name=name)
        self._add_conv(name, geom, make_plan, [x, res, wn], [out])
        return out
