"""Small-K / output-bound conv layers through the C-ABI (for ncu captures and quick timing)."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oct_segmentation_b200.engine import conv as C

LAYERS = [
    ('effnet expand 32->192 @448 swish', [(32, 448, 448)], 192, 1, 16, 'swish'),
    ('effnet expand 48->288 @224 swish', [(48, 224, 224)], 288, 1, 16, 'swish'),
    ('resnet l1.conv3 64->256 @128 relu', [(64, 128, 128)], 256, 1, 32, 'relu'),
    ('resnet l1.conv1 256->64 @128 relu', [(256, 128, 128)], 64, 1, 32, 'relu'),
    ('regnet 1x1 784->784 @56', [(784, 56, 56)], 784, 1, 16, 'relu'),
    ('effnet project 1344->224 @56', [(1344, 56, 56)], 224, 1, 16, 'none'),
    ('3x3 64->64 @256', [(64, 256, 256)], 64, 3, 32, 'relu'),
]


def main():
    only = int(sys.argv[1]) if len(sys.argv) > 1 else None
    for li, (name, srcs, cout, k, n, act) in enumerate(LAYERS):
        if only is not None and li != only:
            continue
        spec = [((n, s[1], s[2], s[0], C.pad8(s[0])), False) for s in srcs]
        w = torch.randn(cout, sum(s[0] for s in srcs), k, k) * 0.05
        geom, packed = C.plan_conv(spec, w, pad=(k // 2, k // 2))
        macs = C.dense_macs(w, n, (geom.out_H, geom.out_W))
        bias = C.pad_bias(torch.zeros(cout), geom, cout)
        seg_t = [torch.randn(n, s[1], s[2], C.pad8(s[0]), device='cuda').to(torch.bfloat16) for s in srcs]
        out = torch.empty(n, geom.out_H, geom.out_W, geom.Cout, dtype=torch.bfloat16, device='cuda')
        plan = C.ConvPlan(geom, packed, bias, seg_t, out, act=act, name=name)
        for _ in range(3):
            plan.run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            plan.run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        bytes_io = sum(t.numel() * 2 for t in seg_t) + out.numel() * 2
        tiles = geom.phases * geom.N * -(-geom.Hq // geom.TH) * -(-geom.Wq // geom.TW) * geom.n_tiles_n
        print(json.dumps(dict(layer=name, ms=round(ms, 4), TBps=round(bytes_io / ms / 1e9, 2),
                              tflops=round(2 * macs / ms / 1e9, 1), tile=(geom.TH, geom.TW), BN=geom.BN,
                              ntn=geom.n_tiles_n, kc=[s.kc for s in geom.segs], tiles=tiles,
                              clk_per_tile_per_sm=round(ms * 1e-3 * 1.9e9 / (tiles / 148)))), flush=True)


if __name__ == '__main__':
    main()
