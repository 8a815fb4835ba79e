import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from oct_segmentation_b200.engine import conv as C
N = 32
def run(srcs, cout, k, tile=None, tag=''):
    orig = C.choose_tile
    if tile: C.choose_tile = lambda h, w: tile
    try:
        spec = [((N, s[1], s[2], s[0], C.pad8(s[0])), False) for s in srcs]
        w = torch.randn(cout, sum(s[0] for s in srcs), k, k) * 0.02
        geom, packed = C.plan_conv(spec, w, pad=(k // 2, k // 2))
    finally:
        C.choose_tile = orig
    seg_t = [torch.randn(N, s[1], s[2], C.pad8(s[0]), device='cuda').to(torch.bfloat16) for s in srcs]
    out = torch.empty(N, geom.out_H, geom.out_W, geom.Cout, dtype=torch.bfloat16, device='cuda')
    plan = C.ConvPlan(geom, packed, C.pad_bias(torch.zeros(cout), geom, cout), seg_t, out, act='relu', name='x')
    for _ in range(3): plan.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): plan.run()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    print(json.dumps(dict(tag=tag, tile=(geom.TH, geom.TW), BN=geom.BN, halo=geom.halo, wide=[s.wide for s in geom.segs], ms=round(ms, 4),
                          tflops=round(2 * geom.macs / ms / 1e9, 1))), flush=True)
for tile in (None, (1, 112), (2, 56), (1, 128), (8, 16)):
    run([(168, 224, 224)], 64, 3, tile, 'vv dec2 skip 168->64 @224')
for tile in (None, (1, 112), (1, 128)):
    run([(32, 448, 448)], 32, 3, tile, '32->32 @448')
    run([(64, 448, 448)], 32, 3, tile, '64->32 @448')
for tile in (None, (1, 128), (4, 32), (8,16)):
    run([(64, 256, 256), (64, 256, 256), (64, 256, 256), (64, 256, 256)], 32, 3, tile, 'lm x_0_3 skips 256->32 @256')
    run([(64, 256, 256), (64, 256, 256), (64, 256, 256)], 64, 3, tile, 'lm x_1_3 skips 192->64 @256')
