"""Host-side planning of one fused tensor-core convolution launch.

Turns a layer description (sources of the fused concat, folded fp32 weights, geometry) into
the explicit K-segment / tile / packed-weight form that ``octseg_conv_plan_create`` consumes
(include/octseg.h).  Everything here is shape arithmetic + weight re-layout and runs on CPU;
``ConvPlan`` uploads the packed weights and creates the device plan.

Replaces (reference call sites src/models/smp/model.py:70,192): conv2d / conv_transpose2d +
folded BatchNorm + activation (+ nearest-x2 upsample, channel concat, residual add) of the
smp 0.3.3 graphs.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import torch

from .. import _lib

KC = 64  # K elements per pipeline stage (one 128-byte swizzle atom of bf16)
HALO_B_BYTES = 80 * 1024   # resident-weight budget of halo mode (shared memory)


def choose_kc(c_eff: int, taps: int = 9) -> int:
    """Channel-chunk width of a K-segment: 64 (128B swizzle), 32 (64B) or 16 (32B).  Narrow sources
    use narrow chunks so neither TMA nor the MMAs spend time on zero padding; 64/kc consecutive
    (tap, chunk) sub-blocks share one pipeline stage.  A 1x1 conv over 33..48 channels is output-bound: one
    zero-padded 64-channel chunk (one TMA box of 128-byte rows) beats three 16-channel boxes of 32-byte rows
    (measured 48 -> 288 @224^2: 0.23 ms vs 0.34 ms, tools/bench_expand.py)."""
    if c_eff > 48 or (taps == 1 and c_eff > 32):
        return 64
    if c_eff > 32:
        return 16
    if c_eff > 16:
        return 32
    return 16


def pad8(c: int) -> int:
    return (c + 7) // 8 * 8


class Act:
    """NHWC bf16 activation of shape (N, H, W, Cp) with Cp = pad8(C); pad channels are 0.

    ``Act(tensor, C)`` wraps an existing tensor.  ``Act.symbolic(shape, C)`` is a buffer the Builder places in
    its activation arena later (engine/builder.py: liveness-based reuse); ``t`` is bound by ``Builder.finalize``."""

    def __init__(self, t: Optional[torch.Tensor], C: int, shape: Optional[Tuple[int, ...]] = None,
                 dtype: torch.dtype = torch.bfloat16):
        self._t = t
        self.C = C
        self.shape = tuple(t.shape) if t is not None else tuple(shape)
        self.dtype = t.dtype if t is not None else dtype

    @classmethod
    def symbolic(cls, shape: Tuple[int, ...], C: int, dtype: torch.dtype = torch.bfloat16) -> 'Act':
        return cls(None, C, shape, dtype)

    @property
    def t(self) -> torch.Tensor:
        if self._t is None:
            raise RuntimeError('activation buffer is not placed yet (Builder.finalize() binds arena buffers)')
        return self._t

    @t.setter
    def t(self, value: torch.Tensor) -> None:
        self._t = value
        self.shape = tuple(value.shape)

    @property
    def nbytes(self) -> int:
        n = 1
        for d in self.shape:
            n *= d
        return n * torch.empty((), dtype=self.dtype).element_size()

    @property
    def N(self): return self.shape[0]
    @property
    def H(self): return self.shape[1]
    @property
    def W(self): return self.shape[2]
    @property
    def Cp(self): return self.shape[3]


@dataclass
class SegSpec:
    """One K-segment (source tensor) in kernel terms; see octseg_conv_seg."""
    N: int
    H: int
    W: int
    C: int
    ldc: int
    kh: int
    kw: int
    mul: int
    off_h: Tuple[int, int]
    off_w: Tuple[int, int]
    c_per_tile: int
    cchunks: int
    kc: int = 64
    wide: int = 0


@dataclass
class ConvGeom:
    """Everything octseg_conv_desc holds except device pointers."""
    segs: List[SegSpec]
    phases: int
    N: int
    Hq: int
    Wq: int
    TH: int
    TW: int
    BN: int
    n_tiles_n: int
    cout_per_tile: int
    Cout: int            # channels written (padded to 8 for bf16 NHWC)
    Ktot: int
    out_H: int
    out_W: int
    halo: int = 0        # 1: 16x8 tiles, one halo-box A load per channel chunk, weights resident in smem


def dense_macs(w: torch.Tensor, N: int, out_hw: Tuple[int, int], transposed: bool = False) -> int:
    """Algorithmic MACs of the reference op (dense count, for rooflines) from its un-transformed weights
    ([Cout, Cin/groups, kh, kw], or [Cin, Cout, 4, 4] when ``transposed``) and its output extent: one MAC per weight
    element and output pixel; a ConvTranspose2d(k4, s2, p1) uses a quarter of its taps for each output pixel."""
    macs = N * out_hw[0] * out_hw[1] * w.numel()
    return macs // 4 if transposed else macs


def choose_tile(Hq: int, Wq: int) -> Tuple[int, int]:
    """TH x TW <= 128 output pixels maximising the useful fraction of the 128-row MMA."""
    best, best_key = (1, 1), None
    for tw in range(1, min(Wq, 128) + 1):
        th = min(Hq, 128 // tw)
        covered = -(-Hq // th) * th * -(-Wq // tw) * tw
        eff = (Hq * Wq) / covered * (th * tw) / 128.0
        key = (round(eff, 6), tw)
        if best_key is None or key > best_key:
            best, best_key = (th, tw), key
    return best


def choose_bn(cout_p: int, k_total: int = 1 << 30) -> Tuple[int, int]:
    """(n_tiles_n, BN): BN multiple of 16, <= 256, tiles cover cout_p channels.

    Output-bound layers (short K) get BN in whole 64-channel chunks: every chunk then leaves through the
    TMA-store epilogue (a partial chunk is only allowed at the very end of the tensor, where TMA clips
    it); the extra zero columns cost MMA time that such layers have to spare.  Long-K layers keep the
    tightest BN."""
    n_tiles = -(-cout_p // 256)
    if k_total <= 512 and cout_p > 64:
        chunks = -(-cout_p // 64)
        n_tiles = -(-chunks // 4)
        return n_tiles, 64 * -(-chunks // n_tiles)
    bn = -(-cout_p // n_tiles)
    bn = (bn + 15) // 16 * 16
    return n_tiles, bn


def _phase_tap_groups(ph: int, a: int) -> List[int]:
    """3x3 taps (pad 1) of a conv over a nearest-x2-upsampled tensor that land on low-res
    offset ``ph - 1 + a`` for output-row parity ``ph``: floor((ph + k - 1) / 2) == ph - 1 + a."""
    return [k for k in range(3) if (ph + k - 1) // 2 == ph - 1 + a]


def plan_conv(srcs: Sequence[Tuple[Tuple[int, int, int, int, int], bool]], weight: torch.Tensor,
              out_hw: Optional[Tuple[int, int]] = None, stride: int = 1, pad: Tuple[int, int] = (0, 0),
              groups: int = 1, transposed: bool = False, out_bf16: bool = True,
              packed_dtype: torch.dtype = torch.bfloat16) -> Tuple[ConvGeom, torch.Tensor]:
    """Plan one conv.

    srcs: [((N, H, W, C, ldc), upsampled)] in concat order; ``upsampled`` sources are at half the
          output resolution and are read through a fused nearest-x2 upsample.
    weight: fp32 [Cout, Cin_total/groups, kh, kw] (BN folded), or [Cin, Cout, 4, 4] when
          ``transposed`` (ConvTranspose2d k4 s2 p1).
    out_hw: output extent; derived from ``pad`` (top, left; assumed symmetric) when omitted.
          efficientnet_pytorch's static "same" padding is asymmetric, so it passes out_hw.
    Returns (geometry, packed weights bf16 [phases, n_tiles_n*BN, Ktot]).
    """
    w = weight.detach().to(torch.float32).cpu()
    any_up = any(up for _, up in srcs)
    N = srcs[0][0][0]
    if transposed:
        assert len(srcs) == 1 and groups == 1 and tuple(w.shape[2:]) == (4, 4) and not any_up
        (_, H, W, cin, _), _ = srcs[0]
        assert w.shape[0] == cin
        cout = w.shape[1]
        phases, Hq, Wq, out_H, out_W = 4, H, W, 2 * H, 2 * W
    else:
        cout, cin_g, kh, kw = w.shape
        cin_total = sum(s[3] for s, _ in srcs)
        assert cin_g * groups == cin_total, (tuple(w.shape), groups, cin_total)
        if any_up:
            assert (kh, kw) == (3, 3) and stride == 1 and tuple(pad) == (1, 1) and groups == 1
            up_src = next(s for s, up in srcs if up)
            out_H, out_W = 2 * up_src[1], 2 * up_src[2]
            for s, up in srcs:
                assert (s[1], s[2]) == ((out_H // 2, out_W // 2) if up else (out_H, out_W)), 'source extent mismatch'
            phases, Hq, Wq = 4, out_H // 2, out_W // 2
        else:
            (_, H, W, _, _), _ = srcs[0]
            if out_hw is None:
                out_hw = ((H + 2 * pad[0] - kh) // stride + 1, (W + 2 * pad[1] - kw) // stride + 1)
            out_H, out_W = out_hw
            phases, Hq, Wq = 1, out_H, out_W
    cout_w = pad8(cout) if out_bf16 else cout          # channels the kernel writes
    TH, TW = choose_tile(Hq, Wq)
    if groups > 1:
        assert len(srcs) == 1 and phases == 1
        cout_g = cout // groups
        assert cout_g % 8 == 0, 'grouped conv needs cout/groups % 8 == 0'
        n_tiles_n, BN, cout_per_tile = groups, (cout_g + 15) // 16 * 16, cout_g
    else:
        k_est = sum((2 * 2 if (transposed or up) else (3 * 3 if phases == 4 else w.shape[2] * w.shape[3])) * sC
                    for (_, _, _, sC, _), up in srcs)
        n_tiles_n, BN = choose_bn(max(cout_w, 16), k_est)
        cout_per_tile = BN
    rows = n_tiles_n * BN

    segs: List[SegSpec] = []
    blocks: List[List[torch.Tensor]] = [[] for _ in range(phases)]  # per phase: K column blocks [rows, 64]
    c_lo = 0
    for (sN, sH, sW, sC, ldc), up in srcs:
        assert sN == N
        if transposed or up:
            # half-resolution source: 2x2 taps per output phase
            kc = choose_kc(sC)
            seg = SegSpec(N, sH, sW, sC, ldc, 2, 2, 1, (-1, 0), (-1, 0), 0, -(-sC // kc), kc)
        elif phases == 4:
            # full-resolution skip tensor seen from the half-resolution tile grid
            kc = choose_kc(sC)
            seg = SegSpec(N, sH, sW, sC, ldc, 3, 3, 2, (-1, 0), (-1, 0), 0, -(-sC // kc), kc)
        else:
            cg = sC // groups
            kc = choose_kc(cg if groups > 1 else sC, kh * kw)
            seg = SegSpec(N, sH, sW, sC, ldc, kh, kw, stride, (-pad[0], -pad[0]), (-pad[1], -pad[1]),
                          cg if groups > 1 else 0, -(-(cg if groups > 1 else sC) // kc), kc)
        segs.append(seg)

        for phase in range(phases):
            ph, pw = phase >> 1, phase & 1
            for ty in range(seg.kh):
                for tx in range(seg.kw):
                    # effective [cout, sC_slice] weight of this tap for this phase
                    if transposed:
                        wt = w[:, :, 3 - ph - 2 * ty, 3 - pw - 2 * tx].t()          # [cout, cin]
                    elif up:
                        khs, kws = _phase_tap_groups(ph, ty), _phase_tap_groups(pw, tx)
                        wt = w[:, c_lo:c_lo + sC][:, :, khs][:, :, :, kws].sum(dim=(2, 3))
                    elif groups > 1:
                        wt = w[:, :, ty, tx]                                         # [cout, cin_g]
                    else:
                        wt = w[:, c_lo:c_lo + sC, ty, tx]
                    for cc in range(seg.cchunks):
                        blk = torch.zeros(rows, seg.kc)
                        if groups > 1:
                            cg, cout_g = sC // groups, cout // groups
                            lo, hi = cc * seg.kc, min((cc + 1) * seg.kc, cg)
                            for g in range(groups):
                                blk[g * BN:g * BN + cout_g, :hi - lo] = wt[g * cout_g:(g + 1) * cout_g, lo:hi]
                        else:
                            lo, hi = cc * seg.kc, min((cc + 1) * seg.kc, sC)
                            blk[:cout, :hi - lo] = wt[:, lo:hi]
                        blocks[phase].append(blk)
        c_lo += sC
    packed = torch.stack([torch.cat(b, dim=1) for b in blocks]).to(packed_dtype).contiguous()
    Ktot = packed.shape[2]
    # Halo-tile mode for narrow single-source k x k convs (stride 1): the tile is 16 x 8 pixels, its
    # (16+kh-1) x (8+kw-1) halo is ONE TMA box per channel chunk and the taps are shifted views of it
    # (8-pixel rows keep the UMMA 8-row groups at a uniform stride); the channel tile's whole weight
    # slice stays resident in shared memory.  Cuts the L2->smem traffic of such layers ~9x.
    halo = 0
    if len(segs) == 1 and phases == 1 and not transposed:
        sg = segs[0]
        b_bytes = sg.kh * sg.kw * sg.cchunks * BN * sg.kc * 2
        cover = (-(-Hq // 16) * 16) * (-(-Wq // 8) * 8)
        if (sg.mul == 1 and sg.kh * sg.kw >= 4 and sg.kh <= 7 and sg.kw <= 7 and b_bytes <= HALO_B_BYTES
                and Hq * Wq >= 0.75 * cover):
            halo, TH, TW = 1, 16, 8

    def wide_boxes(sg: SegSpec) -> bool:
        """Under a row tile, the kw taps of a tap row of this segment can share one A box."""
        return sg.kc == 64 and sg.mul == 1 and sg.kw >= 2 and BN <= 128 and (sg.c_per_tile == 0 or sg.cchunks == 1)
    if TH != 1 and not halo and phases == 1 and not transposed and all(wide_boxes(sg) for sg in segs):
        # k x k conv over wide sources with few output channels and no resident-weight (halo) form: L2 -> shared-memory
        # traffic bounds it (every tap re-reads its A tile).  A ROW tile lets the kw taps of a tap row share one box
        # (wide boxes below: 3x less A traffic), which pays even when the row does not fill the 128 MMA rows:
        # 168 -> 64 @224^2 (U-Net decoder skip conv): 0.86 ms with 4 x 32 tiles, 0.43 ms with 1 x 112 (tools/ab/tile_test.py)
        kw_max = max(sg.kw for sg in segs)
        best_tw, best_eff = 0, 0.0
        for tw in range(16, min(Wq, 128) + 1):
            if tw + kw_max - 1 > 136:
                break
            eff = Wq / (-(-Wq // tw) * tw) * tw / 128.0
            if eff >= best_eff:
                best_tw, best_eff = tw, eff
        if best_eff >= 0.8:
            TH, TW = 1, best_tw
    if TH == 1 and not halo:
        # activation-traffic saver for L2-bound shapes: the B stage then holds kw weight tiles
        for sg in segs:
            if wide_boxes(sg) and TW + sg.kw - 1 <= 136:
                sg.wide = 1
    geom = ConvGeom(segs, phases, N, Hq, Wq, TH, TW, BN, n_tiles_n, cout_per_tile, cout_w, Ktot, out_H, out_W, halo)
    return geom, packed


def pixel_pack_factor(src_cps: Sequence[int], W: int, kw: int, cout_p: int, max_f: int = 8) -> int:
    """Pixels packed along W per GEMM row for narrow tensors (0 = do not pack).  A pixel of a
    16-channel tensor is a 32-byte TMA row; packing f adjacent pixels into one f*C-channel
    "super pixel" (same memory, different view) gives 128-byte rows and an MMA N of f*Cout."""
    cmax = max(src_cps)
    if cmax > 32:
        return 0
    f = 64 // cmax
    while f > 1 and (f > max_f or W % f or kw > f + 1 or f * cout_p > 256):
        f //= 2
    return f if f > 1 else 0


def pack_conv_weights(w: torch.Tensor, b: Optional[torch.Tensor], src_cs: Sequence[int], src_cps: Sequence[int],
                      f: int, pad_l: int, cout_store: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Weights of the equivalent conv on the packed view.  Input channel (r, ci) of source s is pixel
    r of the super pixel; output channel (q, co) is pixel q.  Original tap tx maps to super-pixel tap
    tx' in {0,1,2} (offset tx'-1) with tx = (tx'-1)*f + r - q + pad_l.  cout_store = channels per
    output pixel in memory (padded for bf16 NHWC, exact for NCHW heads)."""
    w = w.detach().float().cpu()
    cout, _, kh, kw = w.shape
    kwp = 3 if kw > 1 else 1
    cin_p = sum(f * cp for cp in src_cps)
    wp = torch.zeros(f * cout_store, cin_p, kh, kwp)
    base_in, base_w = 0, 0
    for c, cp in zip(src_cs, src_cps):
        for q in range(f):
            for r in range(f):
                for txp in range(kwp):
                    tx = (txp - (1 if kwp == 3 else 0)) * f + r - q + pad_l
                    if 0 <= tx < kw:
                        wp[q * cout_store:q * cout_store + cout, base_in + r * cp:base_in + r * cp + c, :, txp] = \
                            w[:, base_w:base_w + c, :, tx]
        base_in += f * cp
        base_w += c
    bp = torch.zeros(f * cout_store)
    if b is not None:
        for q in range(f):
            bp[q * cout_store:q * cout_store + cout] = b.detach().float().cpu()
    return wp, bp


def plan_pixel_packed(srcs: Sequence[Act], w: torch.Tensor, b: Optional[torch.Tensor], f: int, pad: Tuple[int, int],
                      cout_store: int, **kw) -> Tuple[ConvGeom, torch.Tensor, torch.Tensor]:
    """Plan a stride-1 "same" conv over NHWC activations on their f-pixel packed view (pixel_pack_factor).  Returns
    (geometry, packed weights, bias rows); ``kw`` goes to plan_conv."""
    wp, bp = pack_conv_weights(w, b, [a.C for a in srcs], [a.Cp for a in srcs], f, pad[1], cout_store)
    spec = [((a.N, a.H, a.W // f, f * a.Cp, f * a.Cp), False) for a in srcs]
    geom, packed = plan_conv(spec, wp, pad=(pad[0], 1 if w.shape[3] > 1 else 0), **kw)
    return geom, packed, pad_bias(bp, geom, f * cout_store)


def d2s_weights(w: torch.Tensor, b: Optional[torch.Tensor], transposed: bool, cout_store: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Depth-to-space form of `nearest-x2 upsample + 3x3 conv` (w: [Cout, Cin, 3, 3]) or of
    ConvTranspose2d(k4,s2,p1) (w: [Cin, Cout, 4, 4]) with a single source: ONE 3x3 conv (pad 1) on the
    half-resolution tensor whose 4*cout_store output channels, ordered (ph, pw, co), are the 2x2
    output block of each low-res pixel.  Phase (ph, pw) only uses taps dy in {ph-1, ph}, dx in
    {pw-1, pw}; the other taps of its rows are zero."""
    w = w.detach().float().cpu()
    cout = w.shape[1] if transposed else w.shape[0]
    cin = w.shape[0] if transposed else w.shape[1]
    wp = torch.zeros(4 * cout_store, cin, 3, 3)
    for ph in range(2):
        for pw in range(2):
            q = ph * 2 + pw
            for a in range(2):
                for bb in range(2):
                    if transposed:
                        wt = w[:, :, 3 - ph - 2 * a, 3 - pw - 2 * bb].t()
                    else:
                        wt = w[:, :, _phase_tap_groups(ph, a)][:, :, :, _phase_tap_groups(pw, bb)].sum(dim=(2, 3))
                    wp[q * cout_store:q * cout_store + cout, :, ph + a, pw + bb] = wt
    bp = torch.zeros(4 * cout_store)
    if b is not None:
        for q in range(4):
            bp[q * cout_store:q * cout_store + cout] = b.detach().float().cpu()
    return wp, bp


def pad_bias(bias: Optional[torch.Tensor], geom: ConvGeom, cout: int, groups: int = 1) -> torch.Tensor:
    """fp32 bias laid out like the packed weight rows: [n_tiles_n * BN], zero padded."""
    out = torch.zeros(geom.n_tiles_n * geom.BN + 64, dtype=torch.float32)   # +64: the epilogue reads whole 64-wide chunks
    if bias is not None:
        b = bias.detach().to(torch.float32).cpu()
        if groups > 1:
            cg = cout // groups
            for g in range(groups):
                out[g * geom.BN:g * geom.BN + cg] = b[g * cg:(g + 1) * cg]
        else:
            out[:cout] = b
    return out


class ConvPlan:
    """Device-resident plan: packed weights + bias + the C-side TMA/launch plan."""

    def __init__(self, geom: ConvGeom, packed: torch.Tensor, bias: torch.Tensor, seg_tensors: Sequence[torch.Tensor],
                 out: torch.Tensor, out_mode: str = 'bf16_nhwc', act: str = 'none',
                 res: Optional[torch.Tensor] = None, res_mode: str = 'none', per_image_weights: bool = False,
                 name: str = '', out_pack: int = 1, out_ldc: Optional[int] = None, d2s: int = 0,
                 head: Optional[Tuple[torch.Tensor, torch.Tensor, torch.Tensor]] = None):
        """head: (weight fp32 [classes][cmid], bias fp32 [classes], conv bias fp32 [cmid]) of a 1x1 segmentation head
        fused into the epilogue (octseg.h, `head_classes`): `out` is then the head's NCHW output and the conv's own
        output is never stored.  The descriptor's `out_c_off` stays 0: the output starts at channel 0."""
        lib = _lib.load()
        dev = out.device
        self.geom, self.name = geom, name
        self.weight = packed.to(dev) if packed.device != dev else packed
        self.bias = bias.to(dev)
        self.keep = (list(seg_tensors), out, res)  # keep buffers alive as long as the plan
        d = _lib.ConvDesc()
        d.nseg = len(geom.segs)
        for i, (sg, t) in enumerate(zip(geom.segs, seg_tensors)):
            s = d.seg[i]
            s.ptr = t.data_ptr()
            s.N, s.H, s.W, s.C, s.ldc = sg.N, sg.H, sg.W, sg.C, sg.ldc
            s.kh, s.kw, s.mul = sg.kh, sg.kw, sg.mul
            s.off_h[0], s.off_h[1] = sg.off_h
            s.off_w[0], s.off_w[1] = sg.off_w
            s.c_per_tile, s.cchunks, s.kc, s.wide = sg.c_per_tile, sg.cchunks, sg.kc, sg.wide
        d.phases, d.N, d.Hq, d.Wq, d.TH, d.TW = geom.phases, geom.N, geom.Hq, geom.Wq, geom.TH, geom.TW
        d.BN, d.n_tiles_n, d.cout_per_tile, d.Cout = geom.BN, geom.n_tiles_n, geom.cout_per_tile, geom.Cout
        d.weight, d.Ktot, d.per_image_weights = self.weight.data_ptr(), geom.Ktot, int(per_image_weights)
        d.bias = self.bias.data_ptr()
        d.act, d.res_mode = _lib.ACT[act], _lib.RES[res_mode]
        d.res = res.data_ptr() if res is not None else None
        d.res_ldc = res.shape[-1] if res is not None else 0
        d.out, d.out_mode = out.data_ptr(), _lib.OUT[out_mode]
        d.out_H, d.out_W = geom.out_H, geom.out_W
        d.out_ldc = out_ldc if out_ldc is not None else (out.shape[-1] if out_mode == 'bf16_nhwc' else out.shape[1])
        d.out_pack = out_pack
        d.d2s = d2s
        d.halo = geom.halo
        if head is not None:       # host arrays, copied into the plan's parameter block by plan_create
            hw, hb, cb = (t.detach().to('cpu', torch.float32).contiguous() for t in head)
            d.head_classes, d.head_cmid = hw.shape
            assert hb.numel() == hw.shape[0] and cb.numel() == hw.shape[1]
            d.head_weight, d.head_bias, d.head_conv_bias = hw.data_ptr(), hb.data_ptr(), cb.data_ptr()
        handle = C.c_void_p()
        _lib.check(lib.octseg_conv_plan_create(C.byref(d), C.byref(handle)), f'conv_plan_create({name})')
        self._lib, self._h = lib, handle

    def run(self, stream: Optional[int] = None) -> None:
        _lib.check(self._lib.octseg_conv_run(self._h, stream if stream is not None else _lib.stream_ptr()),
                   f'conv_run({self.name})')

    def info(self) -> dict:
        """The library's launch decisions for this plan (octseg_conv_plan_info): grid, tiles, ring sizes, mode flags."""
        out = _lib.ConvPlanInfo()
        _lib.check(self._lib.octseg_conv_plan_info(self._h, C.byref(out)), f'conv_plan_info({self.name})')
        return {n: getattr(out, n) for n, _ in out._fields_}

    def __del__(self):
        h = getattr(self, '_h', None)
        if h:
            self._lib.octseg_conv_plan_destroy(h)
            self._h = None
