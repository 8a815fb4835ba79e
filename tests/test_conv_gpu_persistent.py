"""The tensor-core conv at production tile counts, in every epilogue and scheduling mode, element by element.

conv_tc_kernel is persistent: grid = min(total_tiles, SMs) and each CTA walks its tiles through the TMEM accumulator
ring (n_acc slots, the phase flips on each wrap), the shared-memory stage ring, the TMA-store staging buffers, the
resident halo weights (reloaded when a CTA moves to another channel tile), own_spatial dealing and per-image weights
(the weight slice switches when a CTA's tiles cross an image boundary).  test_conv_gpu's cases plan one tile per CTA,
so none of that machinery runs there; the product runs up to 170 tiles per CTA (batch 16 at 896 x 896).

Each case below drives one Builder op, exactly as lowering calls it, at a size where every CTA runs more tiles than
the accumulator ring has slots, and asserts:
  - the plan reaches the mode the case is named for, as the library decided it (ConvPlan.info());
  - every output element is written: the arena is filled with 0xFF bytes (bf16 NaN) after finalize(), NCHW outputs
    with NaN / 7, no sentinel survives and the pad channels are exactly 0;
  - nothing outside the outputs is written: arena bytes outside the op's outputs and scratch still read 0xFF, and
    the guard bands around NCHW outputs are unchanged;
  - every element is within `conv_bound` of a float64 reference of the same op, and the rel-L2 error is <= 4e-3;
  - a second run is bit-identical.
A whole-tensor rel-L2 cannot see a defect confined to one tile, one ring wrap or one image: its error is diluted by
the norm of everything else.  test_checker_* shows, on the CPU, that the element checks reject such defects.

The sizes target 148 SMs (B200).  On a device with another SM count the tile-count assertion fails with the numbers
instead of silently covering less.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, replace
from typing import Callable, Optional, Sequence, Tuple

import pytest
import torch
import torch.nn.functional as F

from tests.conv_cases import ConvCase, act_fn, make_inputs, reference

U = 2.0 ** -8        # bf16 unit roundoff: 8 significant bits, round to nearest
SLACK = 2.0 ** -12   # fp32 accumulation over K <= 4096 terms (K * 2^-24) and second-order rounding terms
SMS = 148            # the SM count the case sizes below are chosen for (B200)
NAN_BF16 = 0xFF      # arena fill byte: 0xFFFF is a bf16 NaN


# ----------------------------------------------------------------------------------------------- the checker
def lipschitz(act: str) -> float:
    return 1.1 if act == 'swish' else 1.0          # max |d swish / dx| = 1.0998; relu and identity: 1


def conv_bound(ref: torch.Tensor, M: torch.Tensor, pre: torch.Tensor, act: str, rounded: bool = True,
               extra: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Largest |got - ref| a correct kernel can produce, per element.

    ref: float64 reference output; pre: its pre-activation (bias and residual included); M: the same op on |x| and
    |w| without bias, residual or activation.
      - bf16 weights: |sum x (w - bf16(w))| <= U M.  The planner's transformed weights (upsample tap sums, depth-to-space
        and pixel-packed layouts, SE-gated weights) round sums or products of w; still <= U M.
      - fp32 accumulation (K <= 4096) and U times the errors above: < SLACK M.
      - the activation passes a pre-activation error on at most lipschitz(act) times.
      - swish is h tanh(h) + h, h = x / 2, with tanh.approx (relative error 2^-11): |h dtanh| <= 2^-12 |pre|; the
        bound allows 2^-10 |pre|.
      - bf16 output rounding (`rounded`): U |ref|.
    `extra`: further absolute error of the pre-activation (e.g. the bf16 round trip of a split conv's first part)."""
    e = (U + SLACK) * M
    if extra is not None:
        e = e + extra
    b = lipschitz(act) * e
    if act == 'swish':
        b = b + 2.0 ** -10 * pre.abs()
    if rounded:
        b = b + U * ref.abs()
    return b


def head_bound(act_ref: torch.Tensor, M: torch.Tensor, pre: torch.Tensor, act: str, hw: torch.Tensor,
               hb: torch.Tensor) -> torch.Tensor:
    """Bound of a fused 1x1 head's fp32 logits: the conv's activated fp32 outputs (no bf16 rounding) carry
    conv_bound(rounded=False) each and the head sums them with weights hw; its own fp32 sum adds < 2^-16 of the
    magnitude sum."""
    e = conv_bound(act_ref, M, pre, act, rounded=False)
    return F.conv2d(e, hw.abs()) + 2.0 ** -16 * (F.conv2d(act_ref.abs(), hw.abs()) + hb.abs().view(1, -1, 1, 1))


def _index(t: torch.Tensor, flat: int) -> Tuple[int, ...]:
    return tuple(int(i) for i in torch.unravel_index(torch.tensor(flat), t.shape))


def check_elements(got: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor, what: str,
                   where: Callable[[Tuple[int, ...]], str] = lambda i: str(i)) -> float:
    """Every element of `got` (float64, NCHW) is written and within `bound` of `ref`.  Returns max |got - ref| / bound.
    `where` turns an (n, c, y, x) index into a description of where the kernel computed it."""
    nan = torch.isnan(got)
    if nan.any():
        i = _index(got, int(nan.flatten().nonzero()[0]))
        raise AssertionError(f'{what}: {int(nan.sum())} elements unwritten (sentinel NaN), first {where(i)}')
    diff = (got - ref).abs()
    ratio = torch.where(diff == 0, torch.zeros_like(diff), diff / bound)
    worst = float(ratio.max())
    if worst > 1:
        i = _index(ratio, int(ratio.flatten().argmax()))
        raise AssertionError(
            f'{what}: {int((ratio > 1).sum())} elements outside the bound; worst {worst:.3g} x bound {where(i)}: '
            f'got {float(got[i]):.6g}, ref {float(ref[i]):.6g}, bound {float(bound[i]):.3g}')
    return worst


def check_rel_l2(got: torch.Tensor, ref: torch.Tensor, what: str, tol: float = 4e-3) -> None:
    err = float((got - ref).norm() / ref.norm())
    assert err <= tol, f'{what}: rel-L2 {err:.3e} > {tol}'


def check_mask(got: torch.Tensor, logit: torch.Tensor, bound: torch.Tensor, what: str,
               where: Callable[[Tuple[int, ...]], str] = lambda i: str(i)) -> None:
    """u8 output: {0, 1} everywhere (the 7 sentinel never survives), and == logit > 0 wherever |logit| > bound."""
    assert int(got.max()) <= 1, f'{what}: {int((got > 1).sum())} mask bytes unwritten or not 0/1'
    sure = logit.abs() > bound
    bad = sure & (got.bool() != (logit > 0))
    if bad.any():
        i = _index(bad, int(bad.flatten().nonzero()[0]))
        raise AssertionError(f'{what}: {int(bad.sum())} mask bytes wrong, first {where(i)}: logit {float(logit[i]):.4g}')
    assert float(sure.double().mean()) > 0.9, f'{what}: the bound leaves too few elements decided'


def check_untouched(buf: torch.Tensor, regions: Sequence[Tuple[int, int]], what: str, fill: int = NAN_BF16) -> None:
    """Every byte of `buf` (uint8) outside the (offset, nbytes) regions still reads `fill`."""
    inside = torch.zeros(buf.numel(), dtype=torch.bool, device=buf.device)
    for off, n in regions:
        inside[off:off + n] = True
    bad = (~inside) & (buf != fill)
    if bad.any():
        raise AssertionError(f'{what}: {int(bad.sum())} bytes outside the outputs were written, first at byte '
                             f'{int(bad.nonzero()[0])} of {buf.numel()}')


def guarded(shape: Tuple[int, ...], dtype: torch.dtype, fill: float, guard_bytes: int = 4096,
            device: str = 'cuda') -> Tuple[torch.Tensor, torch.Tensor]:
    """(buffer, view): a `shape` view with `guard_bytes` of guard band on both sides, everything filled with `fill`."""
    g = guard_bytes // torch.empty((), dtype=dtype).element_size()
    n = math.prod(shape)
    buf = torch.full((n + 2 * g,), fill, dtype=dtype, device=device)
    return buf, buf[g:g + n].view(shape)


def as_bytes(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(-1).view(torch.uint8)


# ----------------------------------------------------------------------------------------------- float64 references
def se_gate64(pool, w1, b1, w2, b2, hw: int) -> torch.Tensor:
    """efficientnet_pytorch squeeze-excite gate from the depthwise kernel's partial sums: fp64 [N][C]."""
    mean = pool.sum(1) / hw
    z = mean @ w1.t() + b1
    h = z * torch.sigmoid(z)
    return torch.sigmoid(h @ w2.t() + b2)


@dataclass
class Ref:
    out: torch.Tensor      # reference output (NCHW; a head's logits)
    bound: torch.Tensor
    rounded: bool          # bf16 output


def reference64(case: ConvCase, xs, w, b, res, *, gate=None, split_c: int = 0, head=None) -> Ref:
    """Reference and per-element bound of one case, in float64 on the tensors' device.  gate: SE gate [N][C] applied
    to the input channels (per-image weights); split_c: channels of the first (upsampled) source when the op runs as
    a split decoder conv (its part is stored as bf16 before it is added); head: (hw, hb) of a fused 1x1 head."""
    lin = replace(case, act='none', out_mode='f32_nchw')
    g = gate[:, :, None, None] if gate is not None else 1.0
    pre = reference(lin, [xs[0] * g] + list(xs[1:]), w, b, res)
    M = reference(replace(lin, res_mode='none'), [(xs[0] * g).abs()] + [x.abs() for x in xs[1:]], w.abs(), None, None)
    extra = None
    if split_c:
        part = replace(lin, srcs=case.srcs[:1], res_mode='none')
        extra = U * reference(part, [xs[0].abs()], w[:, :split_c].abs(), None, None)
    out = act_fn(pre, case.act)
    if head is not None:
        hw, hb = head
        logits = F.conv2d(out, hw, hb)
        return Ref(logits, head_bound(out, M, pre, case.act, hw, hb), False)
    rounded = case.out_mode == 'bf16_nhwc'
    return Ref(out, conv_bound(out, M, pre, case.act, rounded=rounded, extra=extra), rounded)


def to_bf16_64(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).double()


# ----------------------------------------------------------------------------------------------- CPU self-test
def _small_case():
    case = ConvCase('self', [(64, 16, 16, False)], 64, N=2, act='relu')
    xs, w, b, _ = make_inputs(case, seed=5)
    xs, w, b = [x.double() for x in xs], w.double(), b.double()
    return case, xs, w, b


def test_checker_accepts_a_correct_output():
    """The float64 reference rounded to bf16 is what a correct kernel may return: the checker accepts it."""
    case, xs, w, b = _small_case()
    r = reference64(case, xs, w, b, None)
    ratio = check_elements(to_bf16_64(r.out), r.out, r.bound, 'bf16-rounded reference')
    assert 0.05 < ratio <= 1, ratio            # output rounding alone uses a visible share of the bound
    check_rel_l2(to_bf16_64(r.out), r.out, 'bf16-rounded reference')


def test_checker_rejects_a_neighbours_channel_group():
    """One 8-channel group of one pixel holds its neighbour's values (a mis-addressed 16-byte store)."""
    case, xs, w, b = _small_case()
    r = reference64(case, xs, w, b, None)
    got = to_bf16_64(r.out)
    got[1, 8:16, 5, 7] = got[1, 8:16, 5, 8]
    with pytest.raises(AssertionError, match='outside the bound'):
        check_elements(got, r.out, r.bound, 'swapped group')


def test_checker_rejects_a_tile_missing_its_last_k_chunk():
    """One 128-pixel tile (8 rows x 16) lacks the contribution of the last K chunk (tap (2, 2), channels 0..63)."""
    case, xs, w, b = _small_case()
    r = reference64(case, xs, w, b, None)
    w_last = torch.zeros_like(w)
    w_last[:, :, 2, 2] = w[:, :, 2, 2]
    pre = reference(replace(case, act='none'), xs, w, b, None)
    chunk = reference(replace(case, act='none'), xs, w_last, None, None)
    got = to_bf16_64(r.out)
    got[0, :, 8:16, :] = to_bf16_64(F.relu(pre - chunk))[0, :, 8:16, :]
    with pytest.raises(AssertionError, match='outside the bound'):
        check_elements(got, r.out, r.bound, 'missing K chunk')


def test_checker_rejects_a_tile_without_its_bias():
    case, xs, w, b = _small_case()
    r = reference64(case, xs, w, b, None)
    pre = reference(replace(case, act='none'), xs, w, b, None)
    got = to_bf16_64(r.out)
    got[1, :, 0:8, :] = to_bf16_64(F.relu(pre - b.view(1, -1, 1, 1)))[1, :, 0:8, :]
    with pytest.raises(AssertionError, match='outside the bound'):
        check_elements(got, r.out, r.bound, 'no bias')


def test_checker_rejects_another_images_se_gate():
    """Per-image weights: image 1 computed with image 0's gate (a CTA that did not switch its weight slice)."""
    g = torch.Generator().manual_seed(7)
    N, C, Cr, cout, H, W, slots = 2, 32, 4, 16, 8, 8, 3
    case = ConvCase('se', [(C, H, W, False)], cout, k=1, pad=(0, 0), act='none', N=N)
    xs, w, b, _ = make_inputs(case, seed=7)
    xs, w, b = [x.double() for x in xs], w.double(), b.double()
    pool = torch.randn(N, slots, C, generator=g, dtype=torch.float64) * H * W / slots ** 0.5
    w1, b1 = torch.randn(Cr, C, generator=g, dtype=torch.float64) / C ** 0.5, torch.randn(Cr, generator=g, dtype=torch.float64) * 0.1
    w2, b2 = torch.randn(C, Cr, generator=g, dtype=torch.float64) / Cr ** 0.5, torch.randn(C, generator=g, dtype=torch.float64) * 0.1
    gate = se_gate64(pool, w1, b1, w2, b2, H * W)
    r = reference64(case, xs, w, b, None, gate=gate)
    check_elements(to_bf16_64(r.out), r.out, r.bound, 'SE, correct gates')
    wrong = reference64(case, xs, w, b, None, gate=gate[[0, 0]])
    got = to_bf16_64(r.out)
    got[1] = to_bf16_64(wrong.out[1])
    with pytest.raises(AssertionError, match='outside the bound'):
        check_elements(got, r.out, r.bound, 'SE, image 1 with image 0 gate')


def test_checker_rejects_an_unwritten_element():
    case, xs, w, b = _small_case()
    r = reference64(case, xs, w, b, None)
    got = to_bf16_64(r.out)
    got[0, 3, 4, 5] = float('nan')
    with pytest.raises(AssertionError, match='unwritten'):
        check_elements(got, r.out, r.bound, 'sentinel')
    with pytest.raises(AssertionError, match='unwritten'):
        check_mask(torch.tensor([0, 1, 7], dtype=torch.uint8), torch.tensor([-1.0, 1.0, 1.0]), torch.zeros(3), 'u8')


def test_checker_rejects_a_byte_in_a_guard_band():
    buf, view = guarded((2, 3, 5, 7), torch.uint8, 7, guard_bytes=64, device='cpu')
    view.fill_(1)
    regions = [(64, view.numel())]
    check_untouched(buf, regions, 'guards', fill=7)
    buf[64 + view.numel()] = 0                       # first byte after the output
    with pytest.raises(AssertionError, match='outside the outputs'):
        check_untouched(buf, regions, 'guards', fill=7)
    buf[64 + view.numel()] = 7
    buf[63] = 1                                      # last byte before it
    with pytest.raises(AssertionError, match='outside the outputs'):
        check_untouched(buf, regions, 'guards', fill=7)


# ----------------------------------------------------------------------------------------------- GPU cases
@dataclass
class PCase:
    conv: ConvCase
    expect: dict                      # ConvPlan.info() / geometry values the op's plan must have
    f: int = 1                        # pixels packed per GEMM row
    d2s: int = 0                      # depth-to-space output channels
    head: int = 0                     # classes of a fused 1x1 head
    se: bool = False                  # Builder.se_project (per-image weights)
    expect_up: Optional[dict] = None  # split decoder conv: the `.up` plan

    @property
    def name(self):
        return self.conv.name


PCASES = [
    PCase(ConvCase('simple_1x1', [(64, 304, 304, False)], 64, k=1, pad=(0, 0), N=2),
          dict(use_tma_store=1, halo=0, own_spatial=0, BN=64, n_acc=8)),
    PCase(ConvCase('own_spatial', [(48, 224, 224, False)], 288, k=1, pad=(0, 0), act='swish', N=2),
          dict(own_spatial=1, use_tma_store=1, n_tiles_n=2, BN=192, n_acc=2)),
    PCase(ConvCase('halo_grouped', [(392, 112, 112, False)], 392, groups=7, N=2),
          dict(halo=1, out_grouped=1, use_tma_store=1, n_tiles_n=7)),
    PCase(ConvCase('grouped_stride2', [(392, 224, 224, False)], 392, groups=7, stride=2, N=2),
          dict(halo=0, out_grouped=1, use_tma_store=1, n_tiles_n=7)),
    PCase(ConvCase('halo_partial_tiles', [(64, 200, 600, False)], 64, N=2), dict(halo=1, use_tma_store=1)),
    PCase(ConvCase('wide_row_tiles', [(128, 28, 1024, False)], 128, N=4), dict(wide=1, halo=0, TH=1)),
    PCase(ConvCase('phase4_tma_store', [(256, 64, 64, True), (128, 128, 128, False)], 128, N=6),
          dict(phases=4, use_tma_store=1)),
    PCase(ConvCase('phase4_direct_store', [(96, 40, 40, True), (64, 80, 80, False)], 96, N=16),
          dict(phases=4, use_tma_store=0)),
    PCase(ConvCase('d2s_tma', [(64, 224, 224, True)], 16, N=4), dict(d2s_tma=1, use_tma_store=1), d2s=16),
    PCase(ConvCase('d2s_direct_24', [(64, 112, 112, True)], 24, N=8), dict(d2s_tma=0, use_tma_store=0), d2s=24),
    PCase(ConvCase('d2s_direct_convT_40', [(48, 112, 112, False)], 40, k=4, transposed=True, N=6),
          dict(d2s_tma=0, use_tma_store=0), d2s=40),
    PCase(ConvCase('packed_bf16_residual', [(16, 448, 448, False), (16, 448, 448, False)], 16, res_mode='before_act',
                   N=3), dict(use_tma_store=1), f=4),
    PCase(ConvCase('packed_nchw_u8', [(16, 448, 448, False)], 2, act='none', out_mode='u8_nchw', N=4),
          dict(use_tma_store=0), f=4),
    PCase(ConvCase('packed_nchw_f32', [(16, 448, 448, False)], 2, act='none', out_mode='f32_nchw', N=4),
          dict(use_tma_store=0), f=4),
    PCase(ConvCase('fused_head_f32', [(32, 448, 448, False)], 32, k=1, pad=(0, 0), out_mode='f32_nchw', N=2),
          dict(use_tma_store=0), f=2, head=3),
    PCase(ConvCase('fused_head_u8', [(32, 448, 448, False)], 32, k=1, pad=(0, 0), out_mode='u8_nchw', N=2),
          dict(use_tma_store=0), f=2, head=3),
    PCase(ConvCase('split_decoder', [(128, 112, 112, True), (64, 224, 224, False)], 32, N=6),
          dict(halo=1, use_tma_store=1), expect_up=dict(d2s_tma=1)),
    PCase(ConvCase('se_projection', [(192, 112, 112, False)], 64, k=1, pad=(0, 0), act='none', N=16),
          dict(use_tma_store=1), se=True),
    PCase(ConvCase('se_projection_packed', [(64, 224, 224, False)], 32, k=1, pad=(0, 0), act='none',
                   res_mode='before_act', N=16), dict(use_tma_store=1), f=2, se=True),
]


def dev_nhwc(x: torch.Tensor) -> torch.Tensor:
    n, c, h, w = x.shape
    out = torch.zeros(n, h, w, (c + 7) // 8 * 8, dtype=torch.bfloat16, device='cuda')
    out[..., :c] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    return out


def facts(plan) -> dict:
    g = plan.geom
    return {**plan.info(), 'phases': g.phases, 'BN': g.BN, 'TH': g.TH, 'n_tiles_n': g.n_tiles_n}


def locate(plan, info: dict, f: int, d2s: int, idx: Tuple[int, ...]) -> str:
    """Where the kernel computed output element (n, c, y, x): tile, CTA, position in the CTA's tile list, ring slot."""
    n, c, y, x = idx
    g = plan.geom
    if g.phases == 4:
        yq, xq, phase, col = y // 2, x // 2, (y % 2) * 2 + x % 2, c
    elif d2s:
        yq, xq, phase, col = y // 2, x // 2, 0, ((y % 2) * 2 + x % 2) * d2s + c
    else:
        yq, xq, phase, col = y, x // f, 0, (x % f) * (g.Cout // f) + c
    th, tw, nt = yq // g.TH, xq // g.TW, col // g.cout_per_tile
    tiles_h, tiles_w = -(-g.Hq // g.TH), -(-g.Wq // g.TW)
    if info['halo']:
        t = ((nt * g.N + n) * tiles_h + th) * tiles_w + tw
    else:
        t = (((n * tiles_h + th) * tiles_w + tw) * g.phases + phase) * g.n_tiles_n + nt
    grid = info['grid']
    if info['own_spatial']:
        s, r = divmod(t, g.n_tiles_n)
        cta, i = s % grid, (s // grid) * g.n_tiles_n + r
    else:
        cta, i = t % grid, t // grid
    return (f'at image {n} channel {c} pixel ({y}, {x}): tile {t} (row {th}, column {tw}, channel tile {nt}, '
            f'phase {phase}) = tile {i} of CTA {cta}, accumulator slot {i % info["n_acc"]}')


def run_case(pc: PCase, seed: int = 0):
    from oct_segmentation_b200 import _lib
    from oct_segmentation_b200.engine.builder import Builder
    from oct_segmentation_b200.engine.conv import Act, ConvPlan

    case = pc.conv
    N, dev = case.N, torch.device('cuda')
    xs, w, b, res = make_inputs(case, seed)
    g = torch.Generator().manual_seed(seed + 1)
    bld = Builder(dev, N, reuse=False)
    srcs = [(Act(dev_nhwc(x), C), up) for x, (C, _, _, up) in zip(xs, case.srcs)]
    res_act = Act(dev_nhwc(res), case.cout) if res is not None else None
    nchw_buf = out_view = head = gate = None
    if case.out_mode != 'bf16_nhwc':
        planes = pc.head or case.cout
        Ho, Wo = case.srcs[0][1], case.srcs[0][2]
        dtype, fill = (torch.float32, float('nan')) if case.out_mode == 'f32_nchw' else (torch.uint8, 7)
        nchw_buf, out_view = guarded((N, planes, Ho, Wo), dtype, fill)
    if pc.head:
        head = (torch.randn(pc.head, case.cout, 1, 1, generator=g) / case.cout ** 0.5, torch.randn(pc.head, generator=g) * 0.1)
    if pc.se:
        C, H, W, _ = case.srcs[0]
        cr = C // 24 if C > 96 else C // 16
        slots = bld.lib.octseg_dwconv_pool_slots(C, H, W)
        assert slots > 1
        pool = torch.randn(N, slots, C, generator=g) * H * W / slots ** 0.5
        w1, b1 = torch.randn(cr, C, generator=g) / C ** 0.5, torch.randn(cr, generator=g) * 0.1
        w2, b2 = torch.randn(C, cr, generator=g) / cr ** 0.5, torch.randn(C, generator=g) * 0.1
        out = bld.se_project(srcs[0][0], pool.to(dev), w1, b1, w2, b2, w, b, name=case.name, res=res_act)
        gate = se_gate64(*(t.double().to(dev) for t in (pool, w1, b1, w2, b2)), H * W)
    else:
        out = bld.conv(srcs, w, b, name=case.name, stride=case.stride, pad=case.pad, groups=case.groups,
                       transposed=case.transposed, act=case.act, res=res_act, res_mode=case.res_mode,
                       out_mode=case.out_mode, out_tensor=out_view, head=head)
    # guard bands in the arena: with reuse=False every buffer stays live, so first-fit stacks them by size -- the
    # larger guard first, then the op's buffers, then the smaller guard (an op with only an NCHW output has none)
    biggest = max((a.nbytes for a in bld._acts), default=0)
    guards = [bld.new_scratch((biggest + 4096,), torch.uint8), bld.new_scratch((4096,), torch.uint8)]
    bld._add('guards', lambda: (lambda: None), [], guards, kind='pack')
    bld.finalize()
    arena = bld._arena
    own = [a for a in bld._acts if a not in guards and a._t is not None and a._t.data_ptr() >= arena.data_ptr()
           and a._t.data_ptr() < arena.data_ptr() + arena.numel()]
    regions = [(a.t.data_ptr() - arena.data_ptr(), a.nbytes) for a in own]
    plans = [p for p in bld._keep if isinstance(p, ConvPlan)]
    sms = _lib.load().octseg_sm_count()

    def fill():
        arena.fill_(NAN_BF16)
        if nchw_buf is not None:
            nchw_buf.fill_(float('nan') if nchw_buf.dtype == torch.float32 else 7)

    fill()
    bld.run()
    torch.cuda.synchronize()
    first = (arena.clone(), nchw_buf.clone() if nchw_buf is not None else None)
    return dict(case=case, xs=xs, w=w, b=b, res=res, head=head, gate=gate, out=out, out_view=out_view,
                nchw_buf=nchw_buf, arena=arena, regions=regions, own=own, plans=plans, sms=sms, bld=bld, fill=fill,
                first=first)


@pytest.mark.gpu
@pytest.mark.parametrize('pc', PCASES, ids=lambda pc: pc.name)
def test_conv_persistent_element_by_element(pc):
    r = run_case(pc)
    case, plans, sms = r['case'], r['plans'], r['sms']

    # ---- the plan reaches its mode, with more tiles per CTA than accumulator slots
    assert plans and plans[-1].name == case.name, [p.name for p in plans]
    main = plans[-1]
    want = {main.name: pc.expect}
    if pc.expect_up is not None:
        assert [p.name for p in plans] == [case.name + '.up', case.name]
        want[case.name + '.up'] = pc.expect_up
    else:
        assert len(plans) == 1, [p.name for p in plans]
    report = []
    for p in plans:
        fa = facts(p)
        per_cta = -(-fa['total_tiles'] // fa['grid'])
        report.append(f'{p.name}: grid {fa["grid"]}, {fa["total_tiles"]} tiles, {per_cta} per CTA, n_acc '
                      f'{fa["n_acc"]}, nstages {fa["nstages"]}, ' +
                      ', '.join(f'{k} {fa[k]}' for k in ('phases', 'BN', 'n_tiles_n', 'use_tma_store', 'out_grouped',
                                                        'd2s_tma', 'own_spatial', 'halo', 'wide')))
        assert per_cta >= fa['n_acc'] + 1, (
            f'{report[-1]}: the accumulator ring does not wrap (sizes chosen for {SMS} SMs, this device has {sms})')
        bad = {k: (fa[k], v) for k, v in want[p.name].items() if fa[k] != v}
        assert not bad, f'{report[-1]}: plan differs from the mode the case is named for (got, want): {bad}'
    info = main.info()
    g = main.geom
    src_W = case.srcs[0][2]
    if pc.f > 1:
        assert g.segs[0].W * pc.f == src_W and g.Cout % pc.f == 0, 'not planned on the pixel-packed view'
    if pc.d2s:
        assert g.phases == 1 and g.Cout == 4 * pc.d2s and g.BN >= g.Cout, 'not planned as a depth-to-space conv'
    if info['halo'] and g.n_tiles_n > 1:      # channel tile slowest: CTA 0 must move on to another channel tile
        assert info['grid'] * (-(-info['total_tiles'] // info['grid']) - 1) >= info['total_tiles'] // g.n_tiles_n
    if pc.se:                                  # per-image weights: CTA 0 must cross an image boundary
        assert info['grid'] * (-(-info['total_tiles'] // info['grid']) - 1) >= info['total_tiles'] // case.N
        assert case.N > 8, 'se_hidden_kernel takes 8 images per block: N > 8 runs its second image group'

    # ---- nothing outside the outputs and scratch was written, and every output element was
    check_untouched(as_bytes(r['arena']), r['regions'], f'{case.name}: arena')
    if r['nchw_buf'] is not None:
        buf, view = r['nchw_buf'], r['out_view']
        gb = (buf.numel() - view.numel()) // 2
        sent = torch.isnan(buf) if buf.dtype == torch.float32 else buf == 7
        assert sent[:gb].all() and sent[gb + view.numel():].all(), f'{case.name}: guard band around the NCHW output written'
    for a in r['own']:
        t = a.t
        if t.dtype == torch.bfloat16:
            assert not torch.isnan(t).any(), f'{case.name}: {int(torch.isnan(t).sum())} elements of {tuple(t.shape)} unwritten'
        if t.dtype == torch.bfloat16 and a.C and t.dim() == 4 and t.shape[3] > a.C:
            assert (t[..., a.C:] == 0).all(), f'{case.name}: pad channels {a.C}..{t.shape[3]} not zero'

    # ---- every element within the bound of a float64 reference
    dev = 'cuda'
    xs64 = [x.double().to(dev) for x in r['xs']]
    w64, b64 = r['w'].double().to(dev), r['b'].double().to(dev) if r['b'] is not None else None
    res64 = r['res'].double().to(dev) if r['res'] is not None else None
    head64 = tuple(t.double().to(dev) for t in r['head']) if r['head'] is not None else None
    ref = reference64(case, xs64, w64, b64, res64, gate=r['gate'], head=head64,
                      split_c=case.srcs[0][0] if pc.expect_up is not None else 0)
    where = lambda i: locate(main, info, pc.f, pc.d2s, i if not pc.head else (i[0], 0) + i[2:])
    if case.out_mode == 'bf16_nhwc':
        got = r['out'].t[..., :case.cout].permute(0, 3, 1, 2).double()
    else:
        got = r['out_view'].double()
    if case.out_mode == 'u8_nchw':
        check_mask(r['out_view'], ref.out, ref.bound, case.name, where)
        ratio = float('nan')
    else:
        ratio = check_elements(got, ref.out, ref.bound, case.name, where)
        check_rel_l2(got, ref.out, case.name)

    # ---- a second run gives bit-identical output
    r['fill']()
    r['bld'].run()
    torch.cuda.synchronize()
    assert torch.equal(r['arena'], r['first'][0]), f'{case.name}: second run differs'
    if r['nchw_buf'] is not None:
        assert torch.equal(as_bytes(r['nchw_buf']), as_bytes(r['first'][1])), f'{case.name}: second run differs'
    print(f'\n{case.name}: ' + '; '.join(report) + f'; max |got - ref| / bound {ratio:.3f}')


# ----------------------------------------------------------------------------------------------- the SE launches
@pytest.mark.gpu
@pytest.mark.parametrize('N', [16, 11])
def test_se_hidden_and_gate_match_float64(N):
    """octseg_se_hidden (slot sums, then 8 images per block: N > 8 runs a second image group) and octseg_se_gate,
    each on its own inputs, against float64 at a relative 1e-5 of the terms' magnitude."""
    from oct_segmentation_b200 import _lib
    lib, dev = _lib.load(), 'cuda'
    g = torch.Generator().manual_seed(N)
    C, Cr, slots, hw = 192, 8, 14, 112 * 112
    pool = torch.randn(N, slots, C, generator=g) * hw / slots ** 0.5
    w1, b1 = torch.randn(Cr, C, generator=g) / C ** 0.5, torch.randn(Cr, generator=g) * 0.1
    w2, b2 = torch.randn(C, Cr, generator=g) / Cr ** 0.5, torch.randn(C, generator=g) * 0.1
    pd, w1d, b1d, b2d = (t.to(dev) for t in (pool, w1, b1, b2))
    w2t = w2.t().contiguous().to(dev)
    sums = torch.full((N, C), float('nan'), device=dev)
    hidden = torch.full((N, Cr), float('nan'), device=dev)
    gate = torch.full((N, C), float('nan'), device=dev)
    st = _lib.stream_ptr()
    _lib.check(lib.octseg_se_hidden(pd.data_ptr(), slots, sums.data_ptr(), 1.0 / hw, w1d.data_ptr(), b1d.data_ptr(),
                                    hidden.data_ptr(), N, C, Cr, st), 'se_hidden')
    _lib.check(lib.octseg_se_gate(hidden.data_ptr(), w2t.data_ptr(), b2d.data_ptr(), gate.data_ptr(), None, N, C, Cr, st),
               'se_gate')
    torch.cuda.synchronize()

    p64, w164, b164, w264, b264 = (t.double() for t in (pool, w1, b1, w2, b2))
    mean, mean_mag = p64.sum(1) / hw, p64.abs().sum(1) / hw
    z = mean @ w164.t() + b164
    h_ref = z * torch.sigmoid(z)
    h_tol = 1e-5 * (h_ref.abs() + 1.1 * (mean_mag @ w164.abs().t() + b164.abs()))
    h_got = hidden.double().cpu()
    bad = (h_got - h_ref).abs() > h_tol
    assert not bad.any(), f'se_hidden wrong for (image, unit) {bad.nonzero()[:8].tolist()}'

    hg = hidden.double().cpu()                       # se_gate on its own input
    t = hg @ w264.t() + b264
    g_ref = torch.sigmoid(t)
    g_tol = 1e-5 * (g_ref.abs() + 0.25 * (hg.abs() @ w264.abs().t() + b264.abs()))
    bad = (gate.double().cpu() - g_ref).abs() > g_tol
    assert not bad.any(), f'se_gate wrong for (image, channel) {bad.nonzero()[:8].tolist()}'


@pytest.mark.gpu
@pytest.mark.parametrize('rows,Ktot,C,period', [(64, 256, 200, 200), (32, 128, 80, 40)],
                         ids=['plain_k_padding', 'pixel_packed'])
def test_se_scale_weights_bit_exact(rows, Ktot, C, period):
    """octseg_se_scale_weights == torch's (w * gate[k % period]).to(bf16) bit for bit at N = 16, and the K padding
    columns are exactly 0.  Ties first: pack8 must round to nearest even, as torch does."""
    from oct_segmentation_b200 import _lib
    lib, dev, N = _lib.load(), 'cuda', 16
    g = torch.Generator().manual_seed(rows + C)
    w = torch.randn(rows, Ktot, generator=g)
    gate = torch.rand(N, period, generator=g) + 0.01
    ties = torch.tensor([1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8), 2 ** -20 * (1 + 2 ** -8), 3 + 2 ** -7, 255.5 + 0.25,
                         0.0, -0.0])
    # bf16 round-to-nearest-even of the values above (1 + 2^-8 -> 1, 1 + 3 * 2^-8 -> 1 + 2^-6, ...)
    want_ties = torch.tensor([0x3F80, 0x3F82, 0xBF80, 0x3580, 0x4040, 0x4380, 0x0000, 0x8000], dtype=torch.int32)
    w[:, :8] = ties
    gate[:, :8] = 1.0
    out = torch.full((N, rows, Ktot), float('nan'), dtype=torch.bfloat16, device=dev)
    gd, wd = gate.to(dev), w.to(dev)
    _lib.check(lib.octseg_se_scale_weights(gd.data_ptr(), wd.data_ptr(), out.data_ptr(), N, rows, Ktot, C, period,
                                           _lib.stream_ptr()), 'se_scale_weights')
    torch.cuda.synchronize()
    got = out.cpu().view(torch.int16).int() & 0xFFFF
    assert (got[:, :, :8] == want_ties).all(), f'pack8 is not round-to-nearest-even: {got[0, 0, :8].tolist()}'
    k = torch.arange(C)
    want = torch.zeros(N, rows, Ktot, dtype=torch.bfloat16)
    want[:, :, :C] = (w[None, :, :C] * gate[:, None, k % period]).to(torch.bfloat16)
    assert (want.view(torch.int16)[:, :, :8].int() & 0xFFFF == want_ties).all()   # torch rounds the same way
    diff = got != (want.view(torch.int16).int() & 0xFFFF)
    assert not diff.any(), f'{int(diff.sum())} weights differ, first at (image, row, k) {diff.nonzero()[0].tolist()}'
    assert (got[:, :, C:] == 0).all(), 'K padding columns not zero'
