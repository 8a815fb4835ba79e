"""Per-layer table of one network at the bench batch, sorted by lost time: joins the per-launch CUDA-event times that
tools/bench_net.py wrote on the GPU box (gpurun_out/ops_<KEY>.json) with the algorithmic MACs / bytes of every launch,
recomputed here on the CPU by lowering the same network (no GPU needed).

  python tools/layer_table.py KEY [BATCH] [out.md]

"ideal" = the larger of (algorithmic FLOPs / sustained bf16 peak) and (algorithmic bytes / measured HBM peak) from
MEASURED_PEAKS.json; "lost" = measured - ideal.  Algorithmic bytes = activations read + written once + weights."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch

from oct_segmentation_b200 import synthetic
from oct_segmentation_b200.engine.builder import Builder
from oct_segmentation_b200.engine.lower import ENCODER_LOWERING, lower_decoder_and_head
from oct_segmentation_b200.model import OCTSegmentationModel


def main():
    key = sys.argv[1]
    NB = int(sys.argv[2]) if len(sys.argv) > 2 else 32
    dst = sys.argv[3] if len(sys.argv) > 3 else None
    peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    peak_tf, peak_gbs = peaks['bf16_tflops_sustained'], peaks['hbm_gbs']
    cfg = synthetic.MODEL_CONFIGS[key]
    S = cfg['input_size']
    m = OCTSegmentationModel(arch=cfg['architecture'], encoder_name=cfg['encoder'], model_name=cfg['model_name'], in_channels=3,
                             classes=cfg['classes'], encoder_weights=None).model
    b = Builder('cpu', 1)
    x = torch.zeros(1, S, S, 3, dtype=torch.uint8).permute(0, 3, 1, 2)
    feats = ENCODER_LOWERING[m.encoder.kind](b, m.encoder, x, 'u8', None)
    lower_decoder_and_head(b, m, feats, torch.zeros(1, len(cfg['classes']), S, S, dtype=torch.uint8), 'u8_nchw')
    times = json.load(open(os.path.join(ROOT, 'gpurun_out', f'ops_{key}.json')))
    rows = []
    for name, kind, macs, byt in zip(b.op_names, b.op_kinds, b.op_macs, b.op_bytes):
        ms = times.get(name)
        if ms is None:
            continue
        macs = macs or 0
        tf =2 * macs * NB / ms / 1e9 if macs else 0.0
        gbs = byt * NB / ms / 1e6
        ideal = max(2 * macs * NB / 1e9 / peak_tf, byt * NB / 1e6 / peak_gbs)
        rows.append((ms - ideal, name, kind, ms, tf, gbs, ideal))
    rows.sort(reverse=True)
    tot = sum(r[3] for r in rows)
    out = [f'# {key} ({cfg["architecture"]}/{cfg["encoder"]} @{S}) per-launch table, batch {NB}, one B200', '',
           f'{len(rows)} launches, {tot:.3f} ms summed (eager, one CUDA-event pair per launch: `tools/bench_net.py {key} {NB}`); '
           f'peaks: {peak_tf} TFLOP/s sustained bf16, {peak_gbs} GB/s (MEASURED_PEAKS.json).  Sorted by lost time.', '',
           '| launch | kernel | ms | TFLOP/s (algorithmic) | GB/s (algorithmic) | ideal ms | lost ms |', '|---|---|---|---|---|---|---|']
    for lost, name, kind, ms, tf, gbs, ideal in rows:
        out.append(f'| {name} | {kind} | {ms:.3f} | {tf:.0f} | {gbs:.0f} | {ideal:.3f} | {lost:.3f} |')
    text = '\n'.join(out) + '\n'
    if dst:
        open(dst, 'w').write(text)
    print('\n'.join(out[:30]))


if __name__ == '__main__':
    main()
