"""Pre/post-processing kernels in isolation (CUDA events around graph replays, 4 rotating buffer sets > L2): achieved GB/s of
ALGORITHMIC bytes (DESIGN.md 4.4) against the measured HBM peak."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from oct_segmentation_b200 import prepost


def timeit(fns, reps=5):
    """The calls are captured into ONE CUDA graph (the Python wrappers cost more host time than the
    kernels run), then the graph replay is timed with CUDA events."""
    for f in fns:
        f()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for f in fns:
            f()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (reps * len(fns))


def main():
    N, SRC, HO = 32, 512, 1000
    peak = 6533.8
    try:
        peak = json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'MEASURED_PEAKS.json')))['hbm_gbs']
    except Exception:
        pass
    sets = 4
    frames = [torch.randint(0, 255, (N, SRC, SRC, 3), dtype=torch.uint8, device='cuda') for _ in range(sets)]
    for S in (512, 896):
        outs = [torch.empty(N, S, S, 3, dtype=torch.uint8, device='cuda') for _ in range(sets)]
        ms = timeit([lambda i=i: prepost.preprocess(frames[i], S, outs[i]) for i in range(sets)])
        b = N * (3 * SRC * SRC + 3 * S * S)
        print(json.dumps(dict(kernel='preprocess_resize_bgr', S_src=SRC, S=S, frames=N, ms=round(ms, 4),
                              GBps=round(b / ms / 1e6, 1), frac_of_hbm=round(b / ms / 1e6 / peak, 3))), flush=True)
    planes = [{0: (torch.rand(N, 512, 512, device='cuda') > 0.5).to(torch.uint8),
               1: (torch.rand(N, 896, 896, device='cuda') > 0.5).to(torch.uint8),
               2: (torch.rand(N, 896, 896, device='cuda') > 0.5).to(torch.uint8),
               3: (torch.rand(N, 896, 896, device='cuda') > 0.5).to(torch.uint8)} for _ in range(sets)]
    masks = [torch.empty(N, HO, HO, 4, dtype=torch.uint8, device='cuda') for _ in range(sets)]
    labels = [torch.empty(N, HO, HO, dtype=torch.uint8, device='cuda') for _ in range(sets)]
    counts = [torch.zeros(N, 4, dtype=torch.int32, device='cuda') for _ in range(sets)]
    ms = timeit([lambda i=i: prepost.postprocess(planes[i], [0, 1, 2, 3], HO, HO, N, 'cuda', masks[i], labels[i], counts[i])
                 for i in range(sets)])
    b = N * (512 * 512 + 3 * 896 * 896 + 5 * HO * HO)
    print(json.dumps(dict(kernel='postprocess (+counts.zero_)', Ho=HO, frames=N, ms=round(ms, 4), GBps=round(b / ms / 1e6, 1),
                          frac_of_hbm=round(b / ms / 1e6 / peak, 3))), flush=True)
    ms = timeit([lambda i=i: prepost.radial_thickness(masks[i]) for i in range(sets)])
    print(json.dumps(dict(kernel='radial_thickness', frames=N, ms=round(ms, 4))), flush=True)
    big = [torch.randint(0, 255, (N, HO, HO, 3), dtype=torch.uint8, device='cuda') for _ in range(sets)]
    overs = [torch.empty_like(b_) for b_ in big]
    # OCT-shaped masks: lumen disc, fibrous-cap arc, lipid wedge behind it, a few vasa-vasorum blobs (the noise
    # masks left by the post-processing bench above are the worst case: every pixel is an object boundary)
    yy, xx = torch.meshgrid(torch.arange(HO, device='cuda'), torch.arange(HO, device='cuda'), indexing='ij')
    rr = ((yy - HO / 2) ** 2 + (xx - HO / 2) ** 2).float().sqrt()
    ang = torch.atan2((yy - HO / 2).float(), (xx - HO / 2).float())
    shaped = torch.zeros(N, HO, HO, 4, dtype=torch.uint8, device='cuda')
    shaped[..., 0] = (rr < 0.22 * HO).to(torch.uint8)
    shaped[..., 1] = ((rr >= 0.22 * HO) & (rr < 0.26 * HO) & (ang.abs() < 1.0)).to(torch.uint8)
    shaped[..., 2] = ((rr >= 0.26 * HO) & (rr < 0.36 * HO) & (ang.abs() < 0.9)).to(torch.uint8)
    shaped[..., 3] = (((yy - 0.2 * HO) ** 2 + (xx - 0.3 * HO) ** 2 < 64) | ((yy - 0.75 * HO) ** 2 + (xx - 0.7 * HO) ** 2 < 100)).to(torch.uint8)
    b = N * HO * HO * (3 + 4 + 3)
    for what, mm in (('OCT-shaped masks', [shaped] * sets), ('noise masks (worst case)', masks)):
        ms = timeit([lambda i=i: prepost.overlay(big[i], mm[i], [0, 1, 2, 3], overs[i]) for i in range(sets)])
        print(json.dumps(dict(kernel='overlay', masks=what, Ho=HO, frames=N,
                              ms=round(ms, 4), GBps=round(b / ms / 1e6, 1), frac_of_hbm=round(b / ms / 1e6 / peak, 3))), flush=True)
    for what, mm in (('OCT-shaped masks', shaped), ('noise masks (worst case)', masks[0])):
        ms = timeit([lambda: prepost.contour_largest(mm)], reps=3)
        print(json.dumps(dict(kernel='contour_largest', masks=what, frames=N, ms=round(ms, 4))), flush=True)
    K = 5
    folds = [[torch.randn(N, 1, 896, 896, device='cuda') for _ in range(K)] for _ in range(2)]
    fouts = [torch.empty(N, 1, 896, 896, dtype=torch.uint8, device='cuda') for _ in range(2)]
    ms = timeit([lambda i=i: prepost.fold_average_threshold(folds[i], fouts[i]) for i in range(2)])
    b = N * 896 * 896 * (4 * K + 1)
    print(json.dumps(dict(kernel='fold_average_threshold', K=K, S=896, frames=N, ms=round(ms, 4), GBps=round(b / ms / 1e6, 1),
                          frac_of_hbm=round(b / ms / 1e6 / peak, 3))), flush=True)

if __name__ == '__main__':
    main()
