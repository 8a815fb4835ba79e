import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from oct_segmentation_b200.engine import conv as C
N=32
def run(cin, cout, H, act, ldc_out=None):
    w = torch.randn(cout, cin, 1, 1) * 0.05
    geom, packed = C.plan_conv([((N, H, H, cin, C.pad8(cin)), False)], w)
    x = torch.randn(N, H, H, C.pad8(cin), device='cuda').to(torch.bfloat16)
    ldc = ldc_out or geom.Cout
    out = torch.empty(N, H, H, ldc, dtype=torch.bfloat16, device='cuda')
    plan = C.ConvPlan(geom, packed, C.pad_bias(torch.zeros(cout), geom, cout), [x], out, act=act, name='x', out_ldc=ldc)
    for _ in range(3): plan.run()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): plan.run()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    byt = (x.numel() + N*H*H*cout) * 2
    print(json.dumps(dict(cin=cin, cout=cout, ldc=ldc, H=H, act=act, BN=geom.BN, ntn=geom.n_tiles_n, ms=round(ms,4), GBs=round(byt/ms/1e6))), flush=True)
for act in ('relu','swish'):
    run(48,288,224,act); run(48,288,224,act,320); run(48,320,224,act); run(48,256,224,act)
    run(80,480,112,act); run(80,480,112,act,512); run(80,512,112,act)
