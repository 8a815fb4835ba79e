"""GPU parity of the three lowered networks (through the engine + C-ABI kernels) on the same seeded
synthetic checkpoint + frames as the oracle.

  (1) every launch, in situ (tests/checked_builder.py): each of the network's kernels is compared
      with torch fp32 ops applied to the kernel's own input buffers; rel-L2 <= 1e-2 per launch
      (bf16 output rounding is ~2e-3).  This is the kernel-correctness bar.
  (2) end to end against the fp32 oracle (oracle/smp_ref.py): logits rel-L2 <= 0.12.  The
      synthetic checkpoints are BN-calibrated random networks, which amplify rounding noise far
      more than a trained net (a CPU replay of pure bf16 storage gives 0.04-0.08, DESIGN.md);
      masks must agree on the pixels whose |logit| exceeds 4x the measured logit RMS error.
"""
import numpy as np
import pytest
import torch

from oct_segmentation_b200.model import OCTSegmentationModel
from oracle import synth
from oct_segmentation_b200.engine.network import CompiledNet
from tests.checked_builder import CheckedBuilder

pytestmark = pytest.mark.gpu

SIZES = {'LM': 256, 'VV': 256, 'FC_LC': 256, 'U_LM': 256, 'LINK_R101': 192, 'UPP_REGNET': 192}
# U_LM = BASELINE.json configs[0] (plain U-Net on resnet101); LINK_R101 / UPP_REGNET = cross pairings of the shipped
# decoders and encoders (smp.create_model accepts any pairing, model.py:38-44)
ALL_KEYS = ['LM', 'VV', 'FC_LC', 'U_LM', 'LINK_R101', 'UPP_REGNET']


def rel_l2(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-12)).item()


def build_pair(key):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = synth.make_model(key)
    cfg = synth.model_config(key)
    ours = OCTSegmentationModel(arch=cfg['architecture'], encoder_name=cfg['encoder'], model_name=cfg['model_name'],
                                in_channels=3, classes=cfg['classes'], encoder_weights=None)
    ours.load_state_dict(ref.state_dict(), strict=True)
    return ref.cuda().eval(), ours.cuda().eval()


def frames_bgr(n, size):
    f = synth.synthetic_frames(100, n, size)[..., ::-1].copy()
    return f


@pytest.mark.parametrize('key', ALL_KEYS)
def test_every_launch_matches_torch_in_situ(key):
    ref, ours = build_pair(key)
    size = SIZES[key]
    x = torch.from_numpy(frames_bgr(2, size)).cuda()
    net = CompiledNet(ours.model, 2, size, size, x.device, 'u8', 'f32_nchw', use_graph=False, builder_cls=CheckedBuilder)
    net.x_nhwc.copy_(x)
    errs = net.builder.run_checked()
    worst = sorted(errs, key=lambda e: -e[1])[:5]
    print(f'\n{key}: {len(errs)} launches checked; worst: ' + ', '.join(f'{n}={e:.1e}' for n, e in worst))
    bad = [(n, e) for n, e in errs if not e <= 1e-2]
    assert not bad, f'{key}: launches off by more than 1e-2: {bad[:8]}'


@pytest.mark.parametrize('key,H,W,N', [('LM', 96, 160, 3), ('VV', 224, 160, 3), ('FC_LC', 160, 224, 1)])
def test_every_launch_matches_torch_in_situ_non_square(key, H, W, N):
    """Same per-launch check on non-square inputs and odd batch sizes: feature maps such as 7x5, 14x10, 28x20
    exercise partial tiles of every tiling mode (row tiles, 16x8 halo tiles, depthwise 8x16 / 4x32 tiles)."""
    ref, ours = build_pair(key)
    fr = synth.synthetic_frames(101, N, max(H, W))[:, :H, :W, ::-1].copy()
    x = torch.from_numpy(fr).cuda()
    net = CompiledNet(ours.model, N, H, W, x.device, 'u8', 'f32_nchw', use_graph=False, builder_cls=CheckedBuilder)
    net.x_nhwc.copy_(x)
    errs = net.builder.run_checked()
    bad = [(n, e) for n, e in errs if not e <= 1e-2]
    assert not bad, f'{key} {H}x{W}: launches off by more than 1e-2: {bad[:8]}'


@pytest.mark.parametrize('key', ['LM', 'VV', 'FC_LC', 'U_LM'])
def test_network_matches_oracle(key):
    ref, ours = build_pair(key)
    size = SIZES[key]
    fr = frames_bgr(2, size)
    x = torch.from_numpy(fr).cuda().permute(0, 3, 1, 2).float()          # NHWC-strided, like predict()
    with torch.no_grad():
        feats_ref = ref.model.encoder(x)
        dec_ref = ref.model.decoder(*feats_ref)
        want = ref.model.segmentation_head(dec_ref)
        got = ours.model(x)
    torch.cuda.synchronize()
    net = ours.model.compiled(2, size, size, x.device, 'f32', 'f32_nchw')
    rep = []
    for i, (a, r) in enumerate(zip(net.feats, feats_ref[1:]), start=1):
        rep.append(f'f{i}:{rel_l2(a.t[..., :a.C].permute(0, 3, 1, 2), r):.1e}')
    e32 = rel_l2(got, want)
    if net.dec_out is not None:              # (LinkNet: the head is fused into the decoder's last conv, no such tensor)
        g = net.dec_out.t[..., :net.dec_out.C].permute(0, 3, 1, 2)
        rep.append(f'dec:{rel_l2(g, dec_ref):.1e}')
    rep.append(f'logits:{e32:.1e}')
    print(f'\n{key} vs fp32 oracle : ' + ' '.join(rep))
    assert got.shape == want.shape and got.dtype == torch.float32
    assert torch.isfinite(got).all()
    assert e32 <= 0.12, f'{key}: logits vs fp32 oracle rel-L2 {e32:.3e} ({" ".join(rep)})'
    rms = (got - want).pow(2).mean().sqrt()
    conf = want.abs() > 4 * rms
    assert conf.float().mean() > 0.3
    agree = ((got > 0) == (want > 0))[conf].float().mean().item()
    assert agree >= 0.9995, f'{key}: confident-pixel mask agreement {agree:.5f}'


@pytest.mark.parametrize('key', ['LM', 'VV', 'FC_LC'])
def test_logits_are_bit_reproducible_and_independent_of_buffer_reuse(key):
    """(1) Two replays on the same input give identical bits -- including FC_LC, whose squeeze-excite sums are
    write-once slots added in a fixed order (round 1 accumulated them with fp32 atomics).  (2) The activation arena
    (buffers recycled by liveness, engine/builder.py) changes nothing: a plan whose every activation owns its bytes
    produces the same logits bit for bit."""
    ref, ours = build_pair(key)
    size = 192
    x = torch.from_numpy(frames_bgr(2, size)).cuda()
    outs = []
    for reuse in (True, False):
        net = CompiledNet(ours.model, 2, size, size, x.device, 'u8', 'f32_nchw', use_graph=reuse, reuse=reuse)
        net.x_nhwc.copy_(x)
        a = net.run().clone()
        net.x_nhwc.copy_(x)
        b = net.run().clone()
        torch.cuda.synchronize()
        assert torch.equal(a, b), f'{key}: two runs differ (reuse={reuse})'
        outs.append(a)
        if reuse:
            assert net.arena_bytes < 0.5 * net.act_bytes
    assert torch.equal(outs[0], outs[1]), f'{key}: logits depend on activation-buffer reuse'


def test_forward_normalises_like_reference():
    """OCTSegmentationModel.forward = (x - mean)/std then net (model.py:65-71)."""
    ref, ours = build_pair('LM')
    x = torch.from_numpy(frames_bgr(1, 128)).cuda().permute(0, 3, 1, 2).float()
    with torch.no_grad():
        want = ref(x)
        got = ours(x)
    assert rel_l2(got, want) <= 0.2       # off-calibration input scale: wiring check only (see test_lowering_cpu)


def test_predict_matches_reference_predict():
    """predict(): uint8 NHWC in, {0,1} float32 NHWC out, identical masks away from the zero crossing."""
    ref, ours = build_pair('VV')
    fr = frames_bgr(2, 128)
    want = ref.predict(fr, 'cuda')
    got = ours.predict(fr, 'cuda')
    assert got.shape == want.shape == (2, 128, 128, 1) and got.dtype == np.float32
    assert set(np.unique(got)) <= {0.0, 1.0}
    with torch.no_grad():
        logits = ref.model(torch.from_numpy(fr).cuda().permute(0, 3, 1, 2).float()).permute(0, 2, 3, 1).cpu().numpy()
    conf = np.abs(logits) > 0.3 * logits.std()
    assert (got[conf] == want[conf]).mean() >= 0.9995


def test_shape_not_divisible_by_32_raises():
    _, ours = build_pair('VV')
    with pytest.raises(RuntimeError):
        ours.model(torch.zeros(1, 3, 100, 128, device='cuda'))
