"""Micro-benchmark of representative conv layers through the C-ABI (CUDA events, TFLOP/s of the
reference's dense FLOP count).  Usage: python tools/bench_layers.py [batch]"""
import json
import sys
import os

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oct_segmentation_b200.engine import conv as C

N = int(sys.argv[1]) if len(sys.argv) > 1 else 32

LAYERS = [
    # name, srcs (C,H,W,up), cout, k, stride, pad, groups
    ('x_1_2.conv1', [(512, 64, 64, True), (256, 128, 128, False), (256, 128, 128, False)], 256, 3, 1, 1, 1),
    ('x_1_2.conv2', [(256, 128, 128, False)], 256, 3, 1, 1, 1),
    ('x_1_1.conv1', [(1024, 32, 32, True), (512, 64, 64, False)], 512, 3, 1, 1, 1),
    ('x_3_3.conv1', [(256, 128, 128, True), (64, 256, 256, False)], 64, 3, 1, 1, 1),
    ('x_0_4.conv2', [(16, 512, 512, False)], 16, 3, 1, 1, 1),
    ('l3.conv2 3x3 256', [(256, 32, 32, False)], 256, 3, 1, 1, 1),
    ('l3.conv3 1x1 256->1024', [(256, 32, 32, False)], 1024, 1, 1, 0, 1),
    ('l3.conv1 1x1 1024->256', [(1024, 32, 32, False)], 256, 1, 1, 0, 1),
    ('l1.conv1 1x1 256->64 @128', [(256, 128, 128, False)], 64, 1, 1, 0, 1),
    ('regnet 1x1 784', [(784, 56, 56, False)], 784, 1, 1, 0, 1),
    ('regnet g3x3 784 g14', [(784, 56, 56, False)], 784, 3, 1, 1, 14),
    ('effnet 1x1 224->1344 @56', [(224, 56, 56, False)], 1344, 1, 1, 0, 1),
    ('effnet 1x1 1344->224 @56', [(1344, 56, 56, False)], 224, 1, 1, 0, 1),
]


def main():
    dev = 'cuda'
    results = []
    for name, srcs, cout, k, stride, pad, groups in LAYERS:
        n = N if 'regnet' not in name and 'effnet' not in name else max(1, N // 2)
        spec = [((n, s[1], s[2], s[0], C.pad8(s[0])), s[3]) for s in srcs]
        cin = sum(s[0] for s in srcs)
        w = torch.randn(cout, cin // groups, k, k) * 0.02
        geom, packed = C.plan_conv(spec, w, stride=stride, pad=(pad, pad), groups=groups)
        bias = C.pad_bias(torch.zeros(cout), geom, cout, groups)
        seg_t = [torch.randn(n, s[1], s[2], C.pad8(s[0]), device=dev).to(torch.bfloat16) for s in srcs]
        out = torch.empty(n, geom.out_H, geom.out_W, geom.Cout, dtype=torch.bfloat16, device=dev)
        plan = C.ConvPlan(geom, packed, bias, seg_t, out, act='relu', name=name)
        for _ in range(3):
            plan.run()
        torch.cuda.synchronize()
        reps = 10
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            plan.run()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        tflops = 2 * C.dense_macs(w, n, (geom.out_H, geom.out_W)) / (ms * 1e-3) / 1e12
        executed = 2.0 * n * geom.phases * geom.Hq * geom.Wq * geom.n_tiles_n * geom.BN * geom.Ktot / (ms * 1e-3) / 1e12
        r = dict(layer=name, batch=n, ms=round(ms, 4), tflops_algorithmic=round(tflops, 1),
                 tflops_executed=round(executed, 1), tile=(geom.TH, geom.TW), BN=geom.BN, ntn=geom.n_tiles_n,
                 k_iters=geom.Ktot // 64)
        print(json.dumps(r), flush=True)
        results.append(r)
    return results


if __name__ == '__main__':
    main()
