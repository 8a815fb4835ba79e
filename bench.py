#!/usr/bin/env python
"""bench.py — frames/s of the hybrid-ensemble inference hot path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--config C] [--impl ours|reference] [--dump-outputs DIR]

A step = one pass of the hot path over one batch of B synthetic RGB frames per GPU.  `--config`:
  ensemble (default, BASELINE config 4, the workload the metric is quoted on): bilinear resize+BGR -> LM (U-Net++/
      resnet101 @512) + FC_LC (LinkNet/efficientnet-b7 @896) + VV (U-Net/regnetx_064 @896) -> threshold -> nearest
      resize to 1000x1000 + class routing + label map + per-class pixel counts + radial thickness; B = 32
  lm (config 2): the U-Net++ LM network alone, B = 32;   fc_lc (config 3): LinkNet FC_LC + threshold + areas, B = 16
  ensemble1024 (config 5): all three networks at 1024x1024 on 1024x1024 frames, B = 32
One process per GPU (torchrun for N > 1), frames sharded by rank, no data-path collective; one final gather of the
per-frame counts table.

Output: ONE JSON line on rank 0 (contract in the task statement): `value` = device-resident throughput, `e2e` = same
metric through EnsemblePipeline.stream_host (host frames in, host masks/labels/counts out, copies inside the timed
region), `roofline` for the dominant kernel (conv_tc_kernel, tensor-bound) plus `kernels` (every kernel family: the
fused MBConv kernel, depthwise, SE, stem pack, maxpool against the tensor and HBM peaks), `per_network` (LM / FC_LC /
VV: ms per frame, algorithmic TFLOP/s, fraction of peak, activation arena) and `prepost` (HBM fractions of the
pre/post kernels), `cpu_baseline` = the CPU oracle port on host cores.

`--impl reference` times the reference's own CPU implementation of the path restated in oracle/ (the original cannot
be installed offline: smp/timm/efficientnet_pytorch/lightning/hydra are absent, see DESIGN.md) on all host threads,
batch 1 per call as src/predict.py does.

`--dump-outputs DIR` writes what the last timed step returned on rank 0 (mask, label, counts, radii of
EnsemblePipeline.run_device) as DIR/<name>.npy, so that two builds run with the same arguments, and hence the same
seeded frames and weights, can be compared output for output (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch
import torch.distributed as dist

CLASSES = ['Lumen', 'Fibrous cap', 'Lipid core', 'Vasa vasorum']
METRIC = 'frames/s, LM+FC_LC+VV ensemble inference'

# BASELINE.json configs[1..4] (configs[0] is the reference's own CPU case = `--impl reference`)
CONFIGS = {
    # config 4 (the one the metric is quoted on): full hybrid ensemble, reference-shipped sizes
    'ensemble': dict(classes=CLASSES, src=512, out=[1000, 1000], input_size=None, batch=32, keys=('LM', 'FC_LC', 'VV'),
                     workload='hybrid ensemble LM(UnetPlusPlus/resnet101@512)+FC_LC(LinkNet/efficientnet-b7@896)+'
                              'VV(Unet/timm-regnetx_064@896), routing+label map+pixel counts+radial thickness at 1000x1000, '
                              'synthetic 512x512 RGB frames'),
    # config 1 (the reference's CPU-runnable case; `--impl reference --config unet` times exactly that): plain U-Net on
    # resnet101, single-class lumen, 512 x 512
    'unet': dict(classes=['Lumen'], src=512, out=[1000, 1000], input_size=None, batch=32, keys=('LM',),
                 arch={'LM': dict(architecture='Unet', encoder='resnet101', model_name='Unet_resnet101')},
                 workload='LM only: Unet/resnet101@512 single-class (BASELINE configs[0] on the GPU), threshold+nearest '
                          'resize+pixel counts at 1000x1000, synthetic 512x512 RGB frames'),
    # config 2: U-Net++ LM single class, batch 32
    'lm': dict(classes=['Lumen'], src=512, out=[1000, 1000], input_size=None, batch=32, keys=('LM',),
               workload='LM only: UnetPlusPlus/resnet101@512 single-class, threshold+nearest resize+pixel counts at 1000x1000, '
                        'synthetic 512x512 RGB frames'),
    # config 3: LinkNet FC_LC two classes + threshold + per-class area
    'fc_lc': dict(classes=['Fibrous cap', 'Lipid core'], src=512, out=[1000, 1000], input_size=None, batch=16, keys=('FC_LC',),
                  workload='FC_LC only: LinkNet/efficientnet-b7@896 two-class, threshold+per-class pixel area at 1000x1000, '
                           'synthetic 512x512 RGB frames'),
    # config 5: every model at 1024x1024 (fully convolutional), 1024x1024 sources and outputs, large batch
    'ensemble1024': dict(classes=CLASSES, src=1024, out=[1024, 1024], input_size=1024, batch=32, keys=('LM', 'FC_LC', 'VV'),
                         workload='hybrid ensemble with all three models at 1024x1024 (LM UnetPlusPlus/resnet101, FC_LC '
                                  'LinkNet/efficientnet-b7, VV Unet/timm-regnetx_064), routing+label map+pixel counts+radial '
                                  'thickness at 1024x1024, synthetic 1024x1024 RGB frames'),
}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('bf16_tflops_sustained', 1409.7), d.get('hbm_gbs', 6533.8), 'measured (MEASURED_PEAKS.json, sustained)'
    return 1400.0, 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 200 ms during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(nm)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


def cpu_oracle_frames_per_s(n_frames: int, warmup: int, cfg: dict):
    """The reference path restated in oracle/ (batch 1 per call, FC_LC run once per class exactly like
    src/predict.py:70-100), timed on the host cores.  Returns (frames/s, seconds per frame list)."""
    from oracle import model_ref, synth
    torch.set_num_threads(os.cpu_count() or 1)
    models = {}
    for key in cfg['keys']:
        over = cfg.get('arch', {}).get(key)
        m = synth.make_model('U_LM' if over else key, calib_size=128, calib_frames=1)
        mc = dict(synth.MODEL_CONFIGS[key], **(over or {}))
        if cfg['input_size']:
            mc['input_size'] = cfg['input_size']
        models[key] = (m, mc)
    from PIL import Image
    times = []
    for i in range(warmup + n_frames):
        rgb = synth.synthetic_frame(10_000 + i, cfg['src'])
        img = Image.fromarray(rgb).resize(tuple(cfg['out']))          # data_processing (PIL bicubic)
        mask = np.zeros((cfg['out'][1], cfg['out'][0], 4))
        t0 = time.perf_counter()
        model_ref.segment_with_models([img], [mask], cfg['out'], cfg['classes'], models, 'cpu')
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    return len(times) / sum(times), times


def reference_arm(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    cfg = CONFIGS[args.config]
    WORKLOAD = cfg['workload']
    fps, times = cpu_oracle_frames_per_s(args.steps, args.warmup, cfg)
    ms = 1e3 * float(np.mean(times))
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'name': args.config, 'batch_per_step': 1, 'note': 'reference-as-written: batch 1 per call, each class '
                   'loops its model (FC_LC runs twice), cv2 pre/post on CPU; runs on rank 0 host cores only'},
        'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                         'sample': f'{args.steps} frames (1 frame per step) through the oracle restatement of src/predict.py'},
        'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


DUMP_MAX_ELEMENTS = 1 << 22          # per output: 16 MB as float32, so the four outputs stay well under 64 MB
DUMP_SEED = 0


def dump_outputs(dst: str, outputs: dict) -> None:
    """Each device tensor becomes dst/<name>.npy: float64 for 32/64-bit integers and float64 data, float32 otherwise
    (both exact for these outputs).  A tensor of more than DUMP_MAX_ELEMENTS elements is stored as a sample of its
    flattened elements: one position in each of DUMP_MAX_ELEMENTS equal strides, drawn by a generator seeded with
    DUMP_SEED and the tensor's size, so the same shape always yields the same positions."""
    os.makedirs(dst, exist_ok=True)
    for name, t in outputs.items():
        n, k = t.numel(), DUMP_MAX_ELEMENTS
        if n > k:
            stride = n // k
            idx = np.arange(k, dtype=np.int64) * stride + np.random.default_rng([DUMP_SEED, n]).integers(0, stride, size=k)
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        wide = t.dtype in (torch.int32, torch.int64, torch.float64)
        np.save(os.path.join(dst, f'{name}.npy'), t.cpu().numpy().astype(np.float64 if wide else np.float32))


def lib_sha16() -> str:
    import hashlib
    path = os.path.join(ROOT, 'oct_segmentation_b200', 'liboctseg.so')
    return hashlib.sha1(open(path, 'rb').read()).hexdigest()[:16] if os.path.exists(path) else ''


def kernel_rooflines(pipe, B, peak_tf, peak_hbm):
    """Per-launch CUDA-event timing of every op of every network (instrumented eager passes after the timed region),
    aggregated by kernel family and by network.  Algorithmic FLOPs = 2 x dense MACs of the smp graph; algorithmic
    bytes = activations read + written once + weights (DESIGN.md section 4)."""
    fam, per_net = {}, {}
    for d in pipe.model_dirs:
        net = pipe.nets[d]
        b = net.builder
        for _ in range(3):                               # standalone graph replay of this network
            net.run()
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(3):
            net.run()
        g1.record()
        torch.cuda.synchronize()
        ms_batch = g0.elapsed_time(g1) / 3
        flops = 2.0 * net.macs
        per_net[d] = {'ms_per_frame': ms_batch / B, 'gflop_per_frame': flops / B / 1e9, 'tflops_algorithmic': flops / ms_batch / 1e9,
                      'frac_of_tensor_peak': flops / ms_batch / 1e9 / peak_tf, 'launches': net.launches,
                      'arena_gb': net.arena_bytes / 1e9, 'activations_without_reuse_gb': net.act_bytes / 1e9}
        for rep in range(2):
            evs = []
            for op in b.ops:
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                op()
                e.record()
                evs.append((s, e))
            torch.cuda.synchronize()
            for (s, e), name, kind, macs, byt in zip(evs, b.op_names, b.op_kinds, b.op_macs, b.op_bytes):
                f = fam.setdefault(kind, {'ms': 0.0, 'flops': 0.0, 'bytes': 0.0, 'launches': 0})
                f['ms'] += s.elapsed_time(e)
                f['flops'] += 2.0 * (macs or b.op_fused_macs.get(name, 0))
                f['bytes'] += byt
                f['launches'] += 1
    total_ms = sum(f['ms'] for f in fam.values())
    out = {}
    for kind, f in fam.items():
        tf, gbs = f['flops'] / (f['ms'] * 1e-3) / 1e12, f['bytes'] / (f['ms'] * 1e-3) / 1e9
        out[kind] = {'launches_per_batch': f['launches'] // 2, 'ms_per_batch': f['ms'] / 2, 'share_of_network_time': f['ms'] / total_ms,
                     'tflops_algorithmic': tf, 'frac_of_tensor_peak': tf / peak_tf, 'gbs_algorithmic': gbs,
                     'frac_of_hbm_peak': gbs / peak_hbm, 'avg_launch_ms': f['ms'] / max(f['launches'], 1),
                     'flops_per_launch': f['flops'] / max(f['launches'], 1), 'bytes_per_launch': f['bytes'] / max(f['launches'], 1)}
    return out, per_net


def prepost_rooflines(pipe, frames_dev, B, peak_hbm):
    """HBM roofline of the pre/post kernels on algorithmic bytes (SURVEY.md section 8d), CUDA events, 5 repetitions."""
    from oct_segmentation_b200 import prepost as P

    def timed(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps
    out = {}
    Hs, Ws = pipe.src_hw
    pre_ms, pre_bytes = 0.0, 0.0
    for d in pipe.model_dirs:
        S = pipe.sizes[d]
        net = pipe.nets[d]
        pre_ms += timed(lambda: P.preprocess_s2d(frames_dev, S, out=net.x_s2d))     # resize + BGR + stem packing, one pass
        pre_bytes += B * (3.0 * Hs * Ws + 6.0 * S * S)                              # SURVEY 8d: uint8 source in, bf16 NHWC out
    out['preprocess'] = {'ms_per_batch': pre_ms, 'gbs_algorithmic': pre_bytes / pre_ms / 1e6, 'frac_of_hbm_peak': pre_bytes / pre_ms / 1e6 / peak_hbm}
    planes = {}
    from oct_segmentation_b200.pipeline import MODELS_META
    from oct_segmentation_b200.model import CLASS_IDS
    in_bytes = 0.0
    for name in pipe.classes:
        meta = MODELS_META[name]
        o = pipe.nets[meta['model_dir']].out
        planes[CLASS_IDS[name] - 1] = o[:, meta['index']]
        in_bytes += B * o.shape[2] * o.shape[3]
    post_ms = timed(lambda: P.postprocess(planes, pipe.order, pipe.Ho, pipe.Wo, B, pipe.device, mask=pipe.mask, label=pipe.label,
                                          counts=pipe.counts))
    post_bytes = in_bytes + B * 5.0 * pipe.Ho * pipe.Wo
    out['postprocess'] = {'ms_per_batch': post_ms, 'gbs_algorithmic': post_bytes / post_ms / 1e6, 'frac_of_hbm_peak': post_bytes / post_ms / 1e6 / peak_hbm}
    return out


def ours_arm(args):
    from oct_segmentation_b200 import synthetic
    from oct_segmentation_b200.parallel import gather_table, shard_range
    from oct_segmentation_b200.pipeline import EnsemblePipeline

    cfg = CONFIGS[args.config]
    world = int(os.environ.get('WORLD_SIZE', 1))
    rank = int(os.environ.get('RANK', 0))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    B, K, W = args.batch or cfg['batch'], args.steps, args.warmup
    SRC, OUT_SIZE = cfg['src'], cfg['out']

    models = synthetic.random_models(dev, keys=cfg['keys'], input_size=cfg['input_size'], arch=cfg.get('arch'))
    pipe = EnsemblePipeline(models, cfg['classes'], OUT_SIZE, dev, B, src_hw=(SRC, SRC), thickness=True)

    # this rank's slice of the global synthetic frame list (weak scaling: B*(K+W) frames per rank)
    total = world * B * (K + W)
    lo, hi = shard_range(total, rank, world)
    n_distinct = min(hi - lo, 4 * B)                                     # 4 distinct batches, cycled
    host = torch.from_numpy(synthetic.synthetic_frames(lo, n_distinct, SRC)).pin_memory()
    dev_batches = [host[i:i + B].to(dev) for i in range(0, n_distinct, B)]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- device-resident throughput
    for i in range(W):
        pipe.run_device(dev_batches[i % len(dev_batches)])
    counts_log = []
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(K):
        outputs = pipe.run_device(dev_batches[i % len(dev_batches)])
        counts_log.append(outputs[2].clone())
    table = gather_table(torch.cat(counts_log), world * B * K) if world > 1 else torch.cat(counts_log)
    e1.record()
    barrier()
    t_ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    t_ms = t_ms.item()
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * K / (t_ms * 1e-3)
    if args.dump_outputs and rank == 0:             # before the passes below overwrite the pipeline's output buffers
        dump_outputs(args.dump_outputs, {k: v for k, v in zip(('mask', 'label', 'counts', 'radii'), outputs) if v is not None})

    # ---------------------------------------------------------------- end to end (host buffers)
    host_np = host.numpy()
    for _ in pipe.stream_host((host_np[:B] for _ in range(max(min(W, 3), 2))), copy=False):
        pass
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    starts = [(i % (n_distinct // B)) * B for i in range(K)]
    for mask, label, counts, radii in pipe.stream_host((host_np[j:j + B] for j in starts), copy=False):
        pass                                   # every batch's results are on the host when it is yielded
    e3.record()
    barrier()
    e2e_ms = torch.tensor([e2.elapsed_time(e3)], device=dev)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / (e2e_ms.item() * 1e-3)
    h2d = B * SRC * SRC * 3
    d2h = int(mask.nbytes + label.nbytes + counts.nbytes + radii.nbytes)

    # ---------------------------------------------------------------- rooflines (rank 0, after the timed regions)
    roof = kernels = per_net = prepost = None
    if rank == 0 and not args.no_rooflines:
        peak_tf, peak_hbm, peak_src = peaks()
        kernels, per_net = kernel_rooflines(pipe, B, peak_tf, peak_hbm)
        prepost = prepost_rooflines(pipe, dev_batches[0], B, peak_hbm)
        tc = kernels['conv_tc']
        traffic, traffic_src = None, None
        tpath = os.path.join(ROOT, 'profiles', 'launches_r2_traffic.json')
        if os.path.exists(tpath):                       # dram__bytes_read+write per conv_tc_kernel launch (ncu pass)
            tj = json.load(open(tpath))
            if tj.get('batch') == B and tj.get('config', 'ensemble') == args.config and tj.get('lib_sha16') == lib_sha16():
                traffic, traffic_src = tj['dram_bytes_per_launch'], 'profiles/launches_r2_traffic.json'
            else:
                traffic_src = 'profiles/launches_r2_traffic.json is from another build/config/batch: not used'
        roof = {'bound': 'tensor', 'kernel': 'conv_tc_kernel', 'achieved': tc['tflops_algorithmic'], 'peak': peak_tf,
                'unit': 'TFLOP/s', 'frac': tc['frac_of_tensor_peak'], 'traffic': traffic, 'traffic_source': traffic_src,
                'peak_source': peak_src, 'algorithmic_flops_per_launch': tc['flops_per_launch'],
                'launches_measured': 2 * tc['launches_per_batch'], 'avg_launch_ms': tc['avg_launch_ms'],
                'share_of_network_time': tc['share_of_network_time'],
                'how': 'algorithmic FLOPs (2 x dense MACs of the smp graph, DESIGN.md) of every conv_tc_kernel launch in one '
                       'batch divided by the sum of their CUDA-event durations (eager pass after the timed region); the other '
                       'kernel families and the per-network figures are under "kernels" / "per_network" / "prepost"'}

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': t_ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16',
            'data': 'synthetic',
            'config': {'workload': cfg['workload'], 'name': args.config, 'batch_per_gpu_per_step': B, 'frames_total': world * B * K,
                       'weights': 'seeded random init of the shipped architectures',
                       'l2': 'inputs cycle over 4 distinct batches; per-step activations (several GB) exceed the 126 MB L2',
                       'parallelism': f'frame-sharded x{world}, final all_gather of the counts table'},
            'clocks': clocks,
            'e2e': {'value': e2e_value, 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h},
            'gpu_launches': int(pipe.launches_per_batch * K),
            'roofline': roof,
            'kernels': kernels,
            'per_network': per_net,
            'prepost': prepost,
            'gflop_per_frame_algorithmic': 2 * pipe.macs_per_frame / 1e9,
        }
        if not args.no_cpu_baseline and world == 1:
            fps, times = cpu_oracle_frames_per_s(args.cpu_frames, 1, cfg)
            line['cpu_baseline'] = {'value': fps, 'unit': 'frames/s', 'cores': os.cpu_count() or 1, 'kind': 'port',
                                    'sample': f'{args.cpu_frames} frames through the oracle restatement of src/predict.py '
                                              f'(batch 1 per call, FC_LC run per class, cv2 pre/post), {sum(times):.1f} s'}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def files_arm(args):
    """SURVEY.md section 8f.1: frames/s of the WHOLE entry point on files -- N synthetic PNGs on disk -> predict.main with
    stream_chunk (decode + bicubic resize on host threads, GPU pipeline, overlay kernel, PNG encode of mask + overlay on
    host threads, all overlapped) -> 2 PNGs per frame + quantities.json.  Each stage is also timed alone on the same
    files, so the line shows what the overlap hides; the reference's own flow (oracle restatement of src/predict.py:
    PIL decode, CPU networks, cv2 morphology, PNG encode, single thread of control) is timed on a small sample."""
    import shutil
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    from PIL import Image
    from oct_segmentation_b200 import config as cfgmod, predict as P, synthetic
    n, chunk, B = args.e2e_files, args.stream_chunk, args.batch or 32
    root = tempfile.mkdtemp(prefix='octseg_files_')
    src, dst, mdir = os.path.join(root, 'in'), os.path.join(root, 'out'), os.path.join(root, 'models')
    os.makedirs(src)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(8) as io:
        list(io.map(lambda i: Image.fromarray(synthetic.synthetic_frame(30_000 + i, 512)).save(os.path.join(src, f'f{i:05d}.png')), range(n)))
    gen_s = time.perf_counter() - t0
    dev = torch.device('cuda:0')
    models = synthetic.random_models(dev)
    out_size = [1000, 1000]
    workers = int(args.io_workers)
    cfg = cfgmod.Config({'data_dir': src, 'models_dir': mdir, 'save_dir': dst, 'output_size': out_size, 'device': 'cuda',
                         'classes': CLASSES, 'batch_size': B, 'stream_chunk': chunk, 'io_workers': workers, 'quantities': False})
    orig_load = P.load_models
    P.load_models = lambda *a, **k: models                     # seeded random-init checkpoints (no trained weights offline)
    try:
        P.main(cfgmod.Config(dict(cfg, data_dir=src, save_dir=os.path.join(root, 'warm'), stream_chunk=chunk)))   # warm-up: compile + graphs
        shutil.rmtree(os.path.join(root, 'warm'), ignore_errors=True)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        P.main(cfg)
        torch.cuda.synchronize()
        total_s = time.perf_counter() - t0
    finally:
        P.load_models = orig_load
    n_png = len([f for f in os.listdir(dst) if f.endswith('.png')])
    # the three stages alone, on the same files
    paths = P.list_images(src)
    with ThreadPoolExecutor(workers) as io:
        t0 = time.perf_counter()
        images, masks, names = P.open_images(paths[:min(n, 4 * chunk)], out_size, pool=io)
        decode_s = (time.perf_counter() - t0) * n / len(images)
        pipe = P.make_pipeline(models, CLASSES, out_size, B, (out_size[1], out_size[0]), False)
        P.segment(images, masks, out_size, CLASSES, '', 'cuda', batch_size=B, models=models, pipe=pipe)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        P.segment(images, masks, out_size, CLASSES, '', 'cuda', batch_size=B, models=models, pipe=pipe)
        torch.cuda.synchronize()
        gpu_s = (time.perf_counter() - t0) * n / len(images)
        os.makedirs(os.path.join(root, 'enc'), exist_ok=True)
        t0 = time.perf_counter()
        P.save_results(images, masks, names, CLASSES, os.path.join(root, 'enc'), B, 'cuda', io)
        encode_s = (time.perf_counter() - t0) * n / len(images)
    # the reference flow (CPU oracle restatement), a small sample
    ref_fps = None
    if not args.no_cpu_baseline:
        from oracle import model_ref, prepost_ref, synth
        torch.set_num_threads(os.cpu_count() or 1)
        rm = {k: (synth.make_model(k, calib_size=128, calib_frames=1), synth.MODEL_CONFIGS[k]) for k in ('LM', 'FC_LC', 'VV')}
        k = max(1, args.cpu_frames)
        t0 = time.perf_counter()
        imgs = [Image.open(q_).resize(tuple(out_size)) for q_ in paths[:k]]
        mks = [np.zeros((out_size[1], out_size[0], 4)) for _ in imgs]
        model_ref.segment_with_models(imgs, mks, out_size, CLASSES, rm, 'cpu')
        os.makedirs(os.path.join(root, 'ref'), exist_ok=True)
        for im, mk, nm in zip(imgs, mks, names):
            Image.fromarray(prepost_ref.overlay(np.asarray(im), (mk != 0).astype(np.uint8), CLASSES)).save(os.path.join(root, 'ref', nm + '_overlay.png'))
            Image.fromarray(prepost_ref.color_mask(mk, CLASSES)).save(os.path.join(root, 'ref', nm + '_mask.png'))
        ref_fps = k / (time.perf_counter() - t0)
    shutil.rmtree(root, ignore_errors=True)
    slowest = max(decode_s, gpu_s, encode_s)
    emit({'metric': 'frames/s, PNG files in -> segmentation -> mask + overlay PNGs out (src/predict.py main, stream_chunk)',
          'value': n / total_s, 'unit': 'frames/s', 'n_gpus': 1, 'frames': n, 'seconds': total_s, 'higher_is_better': True,
          'config': {'workload': CONFIGS['ensemble']['workload'], 'files': f'{n} synthetic 512x512 PNGs', 'stream_chunk': chunk,
                     'batch_size': B, 'io_workers': workers, 'host_cores': os.cpu_count(), 'pngs_written': n_png},
          'stages_alone_s': {'decode+bicubic (host threads)': decode_s, 'gpu pipeline incl. copies': gpu_s,
                             'overlay kernel + PNG encode (host threads)': encode_s, 'frame generation (not timed)': gen_s},
          'overlap': {'sum_of_stages_s': decode_s + gpu_s + encode_s, 'slowest_stage_s': slowest,
                      'total_over_slowest': total_s / slowest},
          'cpu_baseline': None if ref_fps is None else {'value': ref_fps, 'unit': 'frames/s', 'cores': os.cpu_count() or 1, 'kind': 'port',
                                                        'sample': f'{max(1, args.cpu_frames)} files through the oracle restatement of the whole src/predict.py flow'},
          'data': 'synthetic'})


_RESULT_FD = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries (NCCL prints its version banner there) must not add
    to it: everything written to fd 1 from here on goes to stderr; emit() writes the result line to the real one."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line: dict) -> None:
    data = (json.dumps(line) + '\n').encode()
    sys.stdout.flush()
    if _RESULT_FD is None:
        os.write(1, data)
    else:
        os.write(_RESULT_FD, data)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--batch', type=int, default=0, help='frames per GPU per step (0 = the config default)')
    ap.add_argument('--config', default='ensemble', choices=sorted(CONFIGS),
                    help='ensemble = BASELINE config 4 (the metric); lm / fc_lc / ensemble1024 = configs 2 / 3 / 5')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--e2e-files', type=int, default=0, help='file-to-file mode: N synthetic PNGs -> predict.main(stream_chunk) -> PNGs')
    ap.add_argument('--stream-chunk', type=int, default=64)
    ap.add_argument('--io-workers', type=int, default=os.cpu_count() or 8)
    ap.add_argument('--cpu-frames', type=int, default=3)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-rooflines', action='store_true',
                    help='skip the instrumented per-launch passes (for the ncu launch list: only the timed steps run)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (a seeded sample of the large ones)')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and (args.e2e_files > 0 or args.impl == 'reference'):
        ap.error('--dump-outputs applies to the device-resident timed path (--impl ours without --e2e-files)')
    _claim_stdout()
    if args.e2e_files > 0:
        files_arm(args)
    elif args.impl == 'reference':
        reference_arm(args)
    else:
        ours_arm(args)


if __name__ == '__main__':
    main()
