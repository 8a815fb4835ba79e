"""CPU: the lowering of each network (BN folding, fused upsample/concat/residual wiring, static
same padding, SE folding) reproduces the oracle's logits when every lowered op is executed with
plain torch fp32 ops (tests/cpu_builder.py)."""
import pytest
import torch

from oct_segmentation_b200 import smp
from oracle import synth
from tests.cpu_builder import run_lowered


# the shipped trio, BASELINE.json configs[0] (plain U-Net on resnet101) and two cross pairings of decoders and encoders
@pytest.mark.parametrize('key,size', [('LM', 64), ('VV', 64), ('FC_LC', 96), ('U_LM', 64), ('LINK_R101', 64), ('UPP_REGNET', 64)])
def test_lowering_matches_oracle(key, size):
    ref = synth.make_model(key, calib_size=size, calib_frames=4)
    cfg = synth.model_config(key)
    ours = smp.create_model(cfg['architecture'], cfg['encoder'], classes=len(cfg['classes']))
    ours.load_state_dict(ref.model.state_dict(), strict=True)
    x = torch.from_numpy(synth.synthetic_frames(7, 2, size)[..., ::-1].copy()).permute(0, 3, 1, 2).float()
    with torch.no_grad():
        want = ref.model(x)
        got = run_lowered(ours, x)
        err = ((got - want).norm() / want.norm()).item()
        assert err < 2e-3, f'{key}: rel-L2 {err:.3e}'
        want_n = ref(x)
        got_n = run_lowered(ours, x, norm=(ref.mean.flatten().tolist(), ref.std.flatten().tolist()))
        # inputs on the 0..255 scale divided by std ~0.23 are far from the calibration distribution:
        # the synthetic net is ill-conditioned there, so this only checks the wiring of the fold
        assert ((got_n - want_n).norm() / want_n.norm()).item() < 5e-2


@pytest.mark.parametrize('key,size', [('LM', 512), ('FC_LC', 896), ('VV', 896)])
def test_lowered_network_counts_the_oracles_macs(key, size):
    """Builder.macs (the algorithmic MACs behind bench.py's roofline figures) of a lowered shipped network equals the
    oracle's per-conv count exactly: the space-to-depth stem, pixel-packed, depth-to-space and split convs, the fused
    head and the SE-folded projections each count the reference op, not the launch it became."""
    from oct_segmentation_b200.engine.builder import Builder
    from oct_segmentation_b200.engine.lower import ENCODER_LOWERING, lower_decoder_and_head
    from oracle import smp_ref
    from tests.test_oracle_models import conv_macs
    cfg = synth.model_config(key)
    classes = len(cfg['classes'])
    want, _ = conv_macs(smp_ref.create_model(cfg['architecture'], cfg['encoder'], classes=classes).eval(),
                        torch.zeros(1, 3, size, size))
    m = smp.create_model(cfg['architecture'], cfg['encoder'], classes=classes)
    b = Builder('cpu', 1)
    x = torch.zeros(1, size // 2, size // 2, 16, dtype=torch.bfloat16)      # the pipeline's space-to-depth input
    feats = ENCODER_LOWERING[m.encoder.kind](b, m.encoder, x, 's2d', None)
    lower_decoder_and_head(b, m, feats, torch.zeros(1, classes, size, size, dtype=torch.uint8), 'u8_nchw')
    assert b.macs == want
