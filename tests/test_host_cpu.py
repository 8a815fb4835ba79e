"""CPU: host logic of the boundary — C-ABI exports, config composition, sharding + gloo gather,
state-dict compatibility, error behaviour of the reference-facing surface."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oct_segmentation_b200 import _lib, config, parallel, smp
from oct_segmentation_b200.model import OCTSegmentationModel
from oct_segmentation_b200 import predict as pred

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol_at_abi_4():
    """ABI 4 added octseg_conv_plan_info; the header, the library and the binding must agree on it."""
    header = open(os.path.join(ROOT, 'include', 'octseg.h')).read()
    declared = set(re.findall(r'\b(octseg_[a-z0-9_]+)\s*\(', header))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    assert 'octseg_conv_plan_info' in declared
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert re.search(r'#define OCTSEG_ABI_VERSION 4\b', header)
    assert _lib.load().octseg_abi_version() == 4


def test_conv_plan_rejects_bad_arguments_without_a_gpu():
    lib = _lib.load()
    d = _lib.ConvDesc()
    d.nseg = 0
    h = ctypes.c_void_p()
    assert lib.octseg_conv_plan_create(ctypes.byref(d), ctypes.byref(h)) == -1
    assert b'nseg' in lib.octseg_last_error()
    d.nseg, d.phases, d.BN = 1, 3, 64
    assert lib.octseg_conv_plan_create(ctypes.byref(d), ctypes.byref(h)) == -1
    assert b'phases' in lib.octseg_last_error()


def test_config_composition_and_overrides():
    cfg = config.compose(os.path.join(ROOT, 'configs'), 'predict', ['device=cpu', 'output_size=[512,512]', 'classes=[Lumen]'])
    assert cfg.device == 'cpu' and cfg.output_size == [512, 512] and cfg.classes == ['Lumen']
    assert cfg.data_dir == 'data/demo/input' and cfg.models_dir == 'models' and cfg.save_dir == 'data/demo/output'
    assert cfg.hydra.job.chdir is False                     # from configs/main.yaml via `defaults`
    base = config.compose(os.path.join(ROOT, 'configs'), 'predict')
    assert base.classes == ['Lumen', 'Fibrous cap', 'Lipid core', 'Vasa vasorum'] and base.output_size == [1000, 1000]
    with pytest.raises(ValueError):
        config.compose(os.path.join(ROOT, 'configs'), 'predict', ['oops'])
    with pytest.raises(FileNotFoundError):
        config.compose(os.path.join(ROOT, 'configs'), 'nope')


def test_pick_device_and_errors():
    assert pred.pick_device('cpu') == 'cpu' and pred.pick_device('cuda') == 'cuda'
    assert pred.pick_device('auto') in ('cpu', 'cuda')
    with pytest.raises(ValueError):
        pred.pick_device('tpu')
    with pytest.raises(KeyError):
        smp.create_model('NoSuchArch', 'resnet101')
    with pytest.raises(KeyError):
        smp.create_model('Unet', 'resnet18')
    with pytest.raises(FileNotFoundError):
        pred.load_model('/nonexistent/dir', 'cpu')
    assert pred.MODELS_META['Lipid core'] == {'model_dir': 'FC_LC', 'index': 0}
    assert pred.MODELS_META['Fibrous cap'] == {'model_dir': 'FC_LC', 'index': 1}


def test_model_surface_and_cpu_refusal():
    m = OCTSegmentationModel(arch='Unet', encoder_name='timm-regnetx_064', model_name='x', in_channels=3,
                             classes=['Vasa vasorum'], encoder_weights=None)
    assert hasattr(m.model, 'encoder') and hasattr(m.model, 'decoder') and hasattr(m.model, 'segmentation_head')
    assert set(k.split('.')[0] for k in m.state_dict()) == {'model', 'mean', 'std'}
    assert m.mean.shape == (1, 3, 1, 1) and abs(m.std[0, 0, 0, 0].item() - 0.229) < 1e-6
    with pytest.raises(RuntimeError):                        # H, W must be divisible by 32
        m.model(torch.zeros(1, 3, 100, 128))
    with pytest.raises(RuntimeError):                        # no CPU fallback
        m.model(torch.zeros(1, 3, 64, 64))
    with pytest.raises(RuntimeError):
        m.predict(np.zeros((1, 64, 64, 3), np.uint8), 'cpu')


def test_checkpoint_roundtrip(tmp_path):
    from oracle import synth
    ref = synth.make_model('VV', calib_size=64, calib_frames=1)
    synth.save_checkpoint(ref, str(tmp_path / 'weights.ckpt'))
    cfg = synth.MODEL_CONFIGS['VV']
    import json
    json.dump(cfg, open(tmp_path / 'config.json', 'w'))
    model, got_cfg = pred.load_model(str(tmp_path), 'cpu')
    assert got_cfg == cfg
    sd = model.state_dict()
    for k, v in ref.state_dict().items():
        assert torch.equal(sd[k], v), k


def test_shard_range_partitions_exactly():
    for n in (0, 1, 7, 16, 25698):
        for world in (1, 2, 3, 4, 8):
            spans = [parallel.shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [hi - lo for lo, hi in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        parallel.shard_range(10, 2, 2)


def _gather_worker(rank, world, n_total, port, q):
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    lo, hi = parallel.shard_range(n_total, rank, world)
    local = torch.arange(lo, hi, dtype=torch.int32)[:, None] * torch.tensor([[1, 10, 100, 1000]], dtype=torch.int32)
    table = parallel.gather_table(local, n_total)
    if rank == 0:
        q.put(table.numpy())
    dist.destroy_process_group()


@pytest.mark.parametrize('n_total', [7, 16])
def test_gather_table_world_size_2_gloo(n_total):
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 500) + n_total
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, n_total, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    table = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    want = np.arange(n_total, dtype=np.int32)[:, None] * np.array([[1, 10, 100, 1000]], dtype=np.int32)
    assert np.array_equal(table, want)           # frame order preserved across ranks == single-rank result


@pytest.mark.parametrize('k,pad,H,W', [(7, (3, 3), 32, 64), (3, (1, 1), 32, 32), (3, (0, 0), 64, 32)])
def test_stem_space_to_depth_weights_equal_the_stride2_conv(k, pad, H, W):
    """engine.builder.stem_s2d_weights: the stride-1 conv on the 2x2 space-to-depth input (what the
    tensor-core stem runs) equals the stride-2 k x k stem conv, incl. efficientnet's bottom/right-only padding."""
    import torch.nn.functional as F
    from oct_segmentation_b200.engine.builder import stem_s2d_weights
    g = torch.Generator().manual_seed(k)
    x = torch.randn(2, 3, H, W, generator=g)
    w = torch.randn(8, 3, k, k, generator=g)
    Ho, Wo = H // 2, W // 2
    pb, pr = (Ho - 1) * 2 + k - H - pad[0], (Wo - 1) * 2 + k - W - pad[1]
    want = F.conv2d(F.pad(x, (pad[1], max(pr, 0), pad[0], max(pb, 0))), w, stride=2)[:, :, :Ho, :Wo]
    w2, q0 = stem_s2d_weights(w, k, pad)
    # channel (dy*2+dx)*3 + c of the packed tensor = pixel (2y+dy, 2x+dx), channel c
    x2 = x.view(2, 3, Ho, 2, Wo, 2).permute(0, 3, 5, 1, 2, 4).reshape(2, 12, Ho, Wo)
    kq = w2.shape[2:]
    xp = F.pad(x2, (-q0[1], kq[1] - 1 + q0[1], -q0[0], kq[0] - 1 + q0[0]))
    got = F.conv2d(xp, w2)
    assert got.shape == want.shape
    assert torch.allclose(got, want, atol=1e-4, rtol=1e-4)


def test_objects_table_follows_get_analysis():
    """prepost.objects_table vs the oracle's restatement of analysis.py:185-207 (object ids of consecutive slices,
    area, contour thickness) on the reference's demo masks, with rows built the way the product builds them."""
    import os
    from oct_segmentation_b200 import prepost as P
    from oracle import prepost_ref as R
    from tests.test_oracle_prepost import G, unpack
    d = np.load(os.path.join(G, 'masks_app_demo.npz'))
    masks = [unpack(p, d['shape']) for p in d['packed']]
    masks = masks[:3] + [np.zeros_like(masks[0])] + masks[3:6]          # a gap starts new objects
    H, W = masks[0].shape[:2]
    ratio = P.dicom_ratio(H)
    rows = []
    for m in masks:
        row = {}
        for c, name in enumerate(P.CLASS_NAMES):
            ch = np.ascontiguousarray(m[:, :, c])
            nnz = int(np.count_nonzero(ch))
            q = {'nnz': nnz, 'present': 0 < nnz < H * W}
            if q['present']:
                t = R.thickness_contour(ch)
                q.update(area=pow(nnz // ratio, 0.5), contour_thickness_mean=t['median'] / ratio, contour_thickness_min=t['min'] / ratio)
            row[name] = q
        rows.append(row)
    got = P.objects_table(rows, [f's{i}' for i in range(len(masks))])
    for c, name in enumerate(P.CLASS_NAMES):
        present = [R.class_present(np.ascontiguousarray(m[:, :, c])) for m in masks]
        assert got[name]['slice'] == [i for i, p in enumerate(present) if p]
        assert got[name]['object_id'] == R.object_ids(present)
        want = [R.frame_quantities(m, ratio)[name] for m, p in zip(masks, present) if p]
        assert got[name]['area'] == [w['area'] for w in want]
        assert got[name]['thickness_mean'] == [w['thickness_mean'] for w in want]
        assert got[name]['thickness_min'] == [w['thickness_min'] for w in want]
        assert got[name]['img_name'] == [f's{i}' for i, p in enumerate(present) if p]
    assert any(len(set(got[n]['object_id'])) > 1 for n in P.CLASS_NAMES)


def _objects_worker(rank, world, counts_all, port, q):
    os.environ['MASTER_ADDR'], os.environ['MASTER_PORT'] = '127.0.0.1', str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    from oct_segmentation_b200 import prepost as P
    n_total = counts_all.shape[0]
    lo, hi = parallel.shard_range(n_total, rank, world)
    table = parallel.gather_table(torch.from_numpy(counts_all[lo:hi].copy()), n_total)     # each rank: its own frames
    if rank == 0:
        rows = P.quantities_from_counts(table.numpy(), 100, 100, P.dicom_ratio(100))
        q.put(P.objects_table(rows))
    dist.destroy_process_group()


def test_object_ids_continue_across_the_shard_boundary_world_size_2_gloo():
    """Frame-sharded ranks gather their per-frame counts; object-id run tracking (analysis.py:191-198) runs on the
    gathered table, so a plaque spanning the shard boundary keeps one id -- identical to the single-rank table."""
    from oct_segmentation_b200 import prepost as P
    from oracle import prepost_ref as R
    n_total = 9
    counts = np.zeros((n_total, 4), np.int32)
    counts[2:7, 0] = 500                       # frames 2..6: crosses the boundary between rank 0 ([0, 5)) and rank 1
    counts[[0, 1, 5, 8], 2] = 40               # three runs
    counts[:, 3] = 100 * 100                   # full plane: not "present" (analysis.py:189)
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 500) + 77
    procs = [ctx.Process(target=_objects_worker, args=(r, 2, counts, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert got['Lumen']['slice'] == [2, 3, 4, 5, 6] and got['Lumen']['object_id'] == [0] * 5
    assert got['Lipid core']['slice'] == [0, 1, 5, 8] and got['Lipid core']['object_id'] == [0, 0, 1, 2]
    assert got['Vasa vasorum']['slice'] == [] and got['Fibrous cap']['slice'] == []
    for c, name in enumerate(P.CLASS_NAMES):
        present = [0 < int(v) < 100 * 100 for v in counts[:, c]]
        assert got[name]['object_id'] == R.object_ids(present)
    assert got == P.objects_table(P.quantities_from_counts(counts, 100, 100, P.dicom_ratio(100)))


def test_contour_fits_matches_the_c_abi_limit():
    from oct_segmentation_b200 import prepost as P
    assert P.contour_fits(1000, 1000) and P.contour_fits(1024, 1024) and not P.contour_fits(2048, 2048)
    lib = _lib.load()
    one = ctypes.c_void_p(16)         # never dereferenced: the size check comes first and no kernel is launched
    rc = lib.octseg_contour_largest(one, 1, 2048, 2048, one, one, one, 8, None)
    assert rc != 0 and b'shared memory' in lib.octseg_last_error()


def test_arena_planner_never_overlaps_live_buffers():
    """engine.builder.plan_arena: buffers whose op intervals intersect never share bytes; the arena stays
    close to the peak of live bytes."""
    import random
    from oct_segmentation_b200.engine.builder import plan_arena
    rnd = random.Random(0)
    items = []
    for _ in range(200):
        lo = rnd.randint(0, 300)
        items.append((rnd.randint(1, 1000) * 1000, lo, lo + rnd.randint(0, 25)))
    offs, total = plan_arena(items)
    for i in range(len(items)):
        assert offs[i] % 256 == 0
        for j in range(i):
            if not (items[i][2] < items[j][1] or items[j][2] < items[i][1]):
                a0, a1, b0, b1 = offs[i], offs[i] + items[i][0], offs[j], offs[j] + items[j][0]
                assert a1 <= b0 or b1 <= a0, (i, j)
    peak = max(sum(s for s, lo, hi in items if lo <= t <= hi) for t in range(330))
    assert peak <= total <= 1.5 * peak


def test_activation_arena_of_a_lowered_network_reuses_dead_buffers():
    """Lowering records reads/writes per op; plan_buffers places the VV network's activations by liveness:
    the arena is several times smaller than one-buffer-per-activation, pinned feature taps keep their bytes,
    and no two simultaneously live buffers overlap."""
    import torch
    from oct_segmentation_b200 import synthetic
    from oct_segmentation_b200.engine.builder import Builder
    from oct_segmentation_b200.engine.lower import ENCODER_LOWERING, lower_decoder_and_head
    from oct_segmentation_b200.model import OCTSegmentationModel
    cfg = synthetic.MODEL_CONFIGS['VV']
    m = OCTSegmentationModel(arch=cfg['architecture'], encoder_name=cfg['encoder'], model_name=cfg['model_name'],
                             in_channels=3, classes=cfg['classes'], encoder_weights=None).model
    b = Builder('cpu', 1)
    S = 64
    x = torch.zeros(1, S, S, 3, dtype=torch.uint8).permute(0, 3, 1, 2)
    feats = ENCODER_LOWERING[m.encoder.kind](b, m.encoder, x, 'u8', None)
    y = lower_decoder_and_head(b, m, feats, torch.zeros(1, 1, S, S, dtype=torch.uint8), 'u8_nchw')
    b.pin(list(feats) + [y])
    acts, offs, total = b.plan_buffers()
    assert len(acts) == len(b._acts) and total < 0.4 * b.act_bytes
    # recompute liveness independently and check the placement
    first, last = {}, {}
    for i, op in enumerate(b._records):
        for a in op.writes:
            first.setdefault(id(a), i)
        for a in list(op.reads) + list(op.writes):
            last[id(a)] = i
    for a in list(feats) + [y]:
        last[id(a)] = len(b._records)
    spans = [(offs[k], offs[k] + a.nbytes, first[id(a)], last[id(a)]) for k, a in enumerate(acts)]
    for i in range(len(spans)):
        for j in range(i):
            a0, a1, alo, ahi = spans[i]
            b0, b1, blo, bhi = spans[j]
            if not (ahi < blo or bhi < alo):
                assert a1 <= b0 or b1 <= a0


def test_dicom_front_end_normalises_like_the_reference_and_needs_pydicom_only_for_files():
    """analysis.normalise_slice = the reference's two cv2 calls (src/app/tools/analysis.py:166-177); a file path needs
    pydicom (absent offline: a clear ImportError), an in-memory pixel array does not."""
    import cv2
    from oct_segmentation_b200 import analysis
    rng = np.random.default_rng(0)
    g16 = rng.integers(100, 4000, (40, 48), dtype=np.uint16)
    want = cv2.cvtColor(cv2.cvtColor(cv2.normalize(g16, None, alpha=0, beta=255, norm_type=cv2.NORM_MINMAX, dtype=cv2.CV_8U),
                                     cv2.COLOR_GRAY2BGR), cv2.COLOR_BGR2RGB)
    got = analysis.normalise_slice(g16)
    assert got.dtype == np.uint8 and got.shape == (40, 48, 3) and np.array_equal(got, want)
    assert got.min() == 0 and got.max() == 255
    c8 = rng.integers(0, 200, (32, 32, 3), dtype=np.uint8)
    want = cv2.cvtColor(cv2.normalize(c8, None, alpha=0, beta=255, norm_type=cv2.NORM_MINMAX, dtype=cv2.CV_8U), cv2.COLOR_BGR2RGB)
    assert np.array_equal(analysis.normalise_slice(c8), want)
    try:
        import pydicom  # noqa: F401
    except ImportError:
        with pytest.raises(ImportError, match='pydicom'):
            analysis.analyse_volume('/nonexistent/study.dcm', models={})
    with pytest.raises(ValueError):
        analysis.analyse_volume(np.zeros((4, 4), np.uint8), models={})


def test_normalisation_constants_match_the_reference_encoders():
    """smp.encoders.get_preprocessing_params (model.py:60-63) gives the ImageNet statistics for all three shipped
    encoders; the product returns what the oracle's restatement does, and OCTSegmentationModel registers them."""
    from oracle import smp_ref, synth
    for key, cfg in synth.MODEL_CONFIGS.items():
        ours = smp.encoders.get_preprocessing_params(cfg['encoder'])
        ref = smp_ref.get_preprocessing_params(cfg['encoder'])
        assert ours['mean'] == ref['mean'] == [0.485, 0.456, 0.406], key
        assert ours['std'] == ref['std'] == [0.229, 0.224, 0.225], key
    cfg = synth.MODEL_CONFIGS['VV']
    m = OCTSegmentationModel(cfg['architecture'], cfg['encoder'], 'VV', 3, cfg['classes'])
    assert m.mean.flatten().tolist() == pytest.approx([0.485, 0.456, 0.406])
    assert m.std.flatten().tolist() == pytest.approx([0.229, 0.224, 0.225])
    with pytest.raises(KeyError):
        smp.encoders.get_preprocessing_params('resnet18')


def test_ctypes_conv_desc_layout_matches_the_c_header(tmp_path):
    """The host side fills octseg_conv_desc through a ctypes mirror: its size and every field offset must equal what a C
    compiler makes of include/octseg.h (a silent mismatch would hand the planner shifted fields)."""
    import shutil
    import subprocess
    if shutil.which('gcc') is None:
        pytest.skip('no gcc')
    names = [n for n, _ in _lib.ConvDesc._fields_]
    seg_names = [n for n, _ in _lib.ConvSeg._fields_]
    info_names = [n for n, _ in _lib.ConvPlanInfo._fields_]
    src = ['#include <stddef.h>', '#include <stdio.h>', '#include "octseg.h"', 'int main(void) {',
           '  printf("sizeof %zu %zu %zu\\n", sizeof(octseg_conv_desc), sizeof(octseg_conv_seg),',
           '         sizeof(struct octseg_conv_plan_info));']
    src += [f'  printf("d {n} %zu\\n", offsetof(octseg_conv_desc, {n}));' for n in names]
    src += [f'  printf("s {n} %zu\\n", offsetof(octseg_conv_seg, {n}));' for n in seg_names]
    src += [f'  printf("i {n} %zu\\n", offsetof(struct octseg_conv_plan_info, {n}));' for n in info_names]
    src += ['  return 0;', '}']
    c = tmp_path / 'layout.c'
    c.write_text('\n'.join(src))
    exe = tmp_path / 'layout'
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include')
    subprocess.run(['gcc', '-I', inc, '-o', str(exe), str(c)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split('\n')
    assert out[0] == (f'sizeof {ctypes.sizeof(_lib.ConvDesc)} {ctypes.sizeof(_lib.ConvSeg)} '
                      f'{ctypes.sizeof(_lib.ConvPlanInfo)}')
    for line in out[1:]:
        if not line:
            continue
        kind, name, off = line.split()
        cls = {'d': _lib.ConvDesc, 's': _lib.ConvSeg, 'i': _lib.ConvPlanInfo}[kind]
        assert getattr(cls, name).offset == int(off), (kind, name)
