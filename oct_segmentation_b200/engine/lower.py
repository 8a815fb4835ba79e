"""Lowering of the smp 0.3.3 graphs (SURVEY.md App. A/B) onto the octseg kernels.

Each function walks a parameter schema from oct_segmentation_b200/smp/modules.py in the order
smp's forward executes it, folds BatchNorm (App. B.4) and emits fused launches:

  conv + BN + ReLU/swish            -> one tensor-core conv
  nearest-x2 upsample + cat + conv  -> one tensor-core conv (4 output phases, multi-segment K)
  ConvTranspose2d(k4,s2,p1)+BN+ReLU -> one tensor-core conv (4 output phases)
  bottleneck tail conv + add + ReLU -> residual in the conv epilogue
  SE gate * x -> project 1x1        -> gate folded into per-image weights of the projection
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import torch

from .builder import Builder, fold_bn
from .conv import Act


# ----------------------------------------------------------------------------------- encoders
def lower_resnet(b: Builder, enc, x: torch.Tensor, in_dtype: str, norm) -> List[Act]:
    """torchvision ResNet (Bottleneck, stride on the 3x3): feature taps at strides 2,4,8,16,32."""
    w, bias = fold_bn(enc.conv1.weight, enc.bn1)
    H, W = (2 * x.shape[1], 2 * x.shape[2]) if in_dtype == 's2d' else (x.shape[2], x.shape[3])
    f1 = b.stem(x, in_dtype, w, bias, name='encoder.conv1', k=7, stride=2, pad=(3, 3),
                out_hw=((H + 6 - 7) // 2 + 1, (W + 6 - 7) // 2 + 1), act='relu', mean=norm and norm[0], std=norm and norm[1])
    feats = [f1]
    cur = b.maxpool(f1, name='encoder.maxpool')
    for li in range(1, 5):
        layer = getattr(enc, f'layer{li}')
        for bi, blk in enumerate(layer):
            nm = f'encoder.layer{li}.{bi}'
            s = blk.conv2.stride[0]
            w1, b1 = fold_bn(blk.conv1.weight, blk.bn1)
            w2, b2 = fold_bn(blk.conv2.weight, blk.bn2)
            w3, b3 = fold_bn(blk.conv3.weight, blk.bn3)
            identity = cur
            if blk.downsample is not None:
                wd, bd = fold_bn(blk.downsample[0].weight, blk.downsample[1])
                identity = b.conv([(cur, False)], wd, bd, name=nm + '.downsample', stride=s, act='none')
            y = b.conv([(cur, False)], w1, b1, name=nm + '.conv1', act='relu')
            y = b.conv([(y, False)], w2, b2, name=nm + '.conv2', stride=s, pad=(1, 1), act='relu')
            cur = b.conv([(y, False)], w3, b3, name=nm + '.conv3', act='relu', res=identity, res_mode='before_act')
        feats.append(cur)
    return feats


def lower_regnet(b: Builder, enc, x: torch.Tensor, in_dtype: str, norm) -> List[Act]:
    """timm RegNetX: stem 3x3 s2, four stages of 1x1 -> grouped 3x3 (stride) -> 1x1 (+shortcut) -> ReLU."""
    w, bias = fold_bn(enc.stem.conv.weight, enc.stem.bn)
    H, W = (2 * x.shape[1], 2 * x.shape[2]) if in_dtype == 's2d' else (x.shape[2], x.shape[3])
    cur = b.stem(x, in_dtype, w, bias, name='encoder.stem', k=3, stride=2, pad=(1, 1),
                 out_hw=((H + 2 - 3) // 2 + 1, (W + 2 - 3) // 2 + 1), act='relu', mean=norm and norm[0], std=norm and norm[1])
    feats = [cur]
    for si in range(1, 5):
        for bname, blk in getattr(enc, f's{si}').named_children():
            nm = f'encoder.s{si}.{bname}'
            s = blk.stride
            w1, b1 = fold_bn(blk.conv1.conv.weight, blk.conv1.bn)
            w2, b2 = fold_bn(blk.conv2.conv.weight, blk.conv2.bn)
            w3, b3 = fold_bn(blk.conv3.conv.weight, blk.conv3.bn)
            shortcut = cur
            if blk.downsample is not None:
                wd, bd = fold_bn(blk.downsample.conv.weight, blk.downsample.bn)
                shortcut = b.conv([(cur, False)], wd, bd, name=nm + '.downsample', stride=s, act='none')
            y = b.conv([(cur, False)], w1, b1, name=nm + '.conv1', act='relu')
            y = b.conv([(y, False)], w2, b2, name=nm + '.conv2', stride=s, pad=(1, 1), groups=blk.conv2.conv.groups,
                       act='relu')
            cur = b.conv([(y, False)], w3, b3, name=nm + '.conv3', act='relu', res=shortcut, res_mode='before_act')
        feats.append(cur)
    return feats


def lower_efficientnet(b: Builder, enc, x: torch.Tensor, in_dtype: str, norm) -> List[Act]:
    """efficientnet_pytorch MBConv stack with static 'same' padding; taps after blocks 11/18/38/55."""
    H, W = (2 * x.shape[1], 2 * x.shape[2]) if in_dtype == 's2d' else (x.shape[2], x.shape[3])
    w, bias = fold_bn(enc._conv_stem.weight, enc._bn0)
    pt, pb = enc._conv_stem.pad
    oh, ow = (H + pt + pb - 3) // 2 + 1, (W + pt + pb - 3) // 2 + 1
    cur = b.stem(x, in_dtype, w, bias, name='encoder._conv_stem', k=3, stride=2, pad=(pt, pt), out_hw=(oh, ow),
                 act='swish', mean=norm and norm[0], std=norm and norm[1])
    feats = [cur]
    for i, blk in enumerate(enc._blocks):
        nm = f'encoder._blocks.{i}'
        inp = cur
        y = cur
        wd, bd = fold_bn(blk._depthwise_conv.weight, blk._bn1)
        pt, pb = blk._depthwise_conv.pad
        cmid = blk._depthwise_conv.weight.shape[0]
        oh = (y.H + pt + pb - blk.k) // blk.stride + 1
        ow = (y.W + pt + pb - blk.k) // blk.stride + 1
        pool = b.new_pool(cmid, (oh, ow))          # fp32 [N][slots][C] partial sums for the SE mean
        if blk.expand != 1:
            we, be = fold_bn(blk._expand_conv.weight, blk._bn0)
            y = b.conv([(y, False)], we, be, name=nm + '._expand_conv', act='swish')
        y = b.dwconv(y, wd, bd, name=nm + '._depthwise_conv', k=blk.k, stride=blk.stride, pad=(pt, pt),
                     out_hw=(oh, ow), act='swish', pool=pool)
        wp, bp = fold_bn(blk._project_conv.weight, blk._bn2)
        skip = inp if (blk.stride == 1 and blk.cin == blk.cout) else None
        cur = b.se_project(y, pool, blk._se_reduce.weight, blk._se_reduce.bias, blk._se_expand.weight,
                           blk._se_expand.bias, wp, bp, name=nm + '._project_conv', res=skip)
        if (i + 1) in enc.stage_idxs:
            feats.append(cur)
    return feats


ENCODER_LOWERING = {'resnet': lower_resnet, 'regnet': lower_regnet, 'efficientnet': lower_efficientnet}


# ----------------------------------------------------------------------------------- decoders
def _unet_block(b: Builder, blk, x: Act, skips: Sequence[Act], name: str) -> Act:
    """DecoderBlock: cat([up2(x), *skips]) -> conv1(3x3)+BN+ReLU -> conv2(3x3)+BN+ReLU."""
    w1, b1 = fold_bn(blk.conv1[0].weight, blk.conv1[1])
    w2, b2 = fold_bn(blk.conv2[0].weight, blk.conv2[1])
    y = b.conv([(x, True)] + [(s, False) for s in skips], w1, b1, name=name + '.conv1', pad=(1, 1), act='relu')
    return b.conv([(y, False)], w2, b2, name=name + '.conv2', pad=(1, 1), act='relu')


def lower_unet_decoder(b: Builder, dec, feats: List[Act]) -> Act:
    f = feats[::-1]                      # f5, f4, f3, f2, f1
    x = f[0]
    skips = f[1:]
    for i, blk in enumerate(dec.blocks):
        x = _unet_block(b, blk, x, [skips[i]] if i < len(skips) else [], f'decoder.blocks.{i}')
    return x


def lower_unetpp_decoder(b: Builder, dec, feats: List[Act]) -> Act:
    f = feats[::-1]
    depth = dec.depth
    dense = {}
    for layer_idx in range(depth):
        for depth_idx in range(depth - layer_idx):
            if layer_idx == 0:
                key = f'x_{depth_idx}_{depth_idx}'
                dense[key] = _unet_block(b, dec.blocks[key], f[depth_idx], [f[depth_idx + 1]], 'decoder.blocks.' + key)
            else:
                li = depth_idx + layer_idx
                key = f'x_{depth_idx}_{li}'
                cat = [dense[f'x_{idx}_{li}'] for idx in range(depth_idx + 1, li + 1)] + [f[li + 1]]
                dense[key] = _unet_block(b, dec.blocks[key], dense[f'x_{depth_idx}_{li - 1}'], cat, 'decoder.blocks.' + key)
    key = f'x_0_{depth}'
    return _unet_block(b, dec.blocks[key], dense[f'x_0_{depth - 1}'], [], 'decoder.blocks.' + key)


def lower_linknet_decoder(b: Builder, dec, feats: List[Act], head=None) -> Optional[Act]:
    """head = (segmentation_head, out tensor, out_mode): fuse the 1x1 head into the last block's final conv; returns
    None then (there is no decoder output tensor any more)."""
    f = feats[::-1]
    x = f[0]
    skips = f[1:]
    for i, blk in enumerate(dec.blocks):
        nm = f'decoder.blocks.{i}.block'
        c1, tr, c2 = blk.block[0], blk.block[1], blk.block[2]
        w1, b1 = fold_bn(c1[0].weight, c1[1])
        wt, bt = fold_bn(tr[0].weight, tr[1], conv_bias=tr[0].bias, out_dim=1)
        w2, b2 = fold_bn(c2[0].weight, c2[1])
        y = b.conv([(x, False)], w1, b1, name=nm + '.0', act='relu')
        y = b.conv([(y, False)], wt, bt, name=nm + '.1', transposed=True, act='relu')
        skip = skips[i] if i < len(skips) else None
        if head is not None and i == len(dec.blocks) - 1 and skip is None:
            hconv = head[0][0]
            b.conv([(y, False)], w2, b2, name=nm + '.2+segmentation_head.0', act='relu', out_mode=head[2], out_tensor=head[1],
                   head=(hconv.weight.detach().float().cpu(), hconv.bias))
            return None
        x = b.conv([(y, False)], w2, b2, name=nm + '.2', act='relu', res=skip,
                   res_mode='after_act' if skip is not None else 'none')
    return x


DECODER_LOWERING = {'unet': lower_unet_decoder, 'unetplusplus': lower_unetpp_decoder, 'linknet': lower_linknet_decoder}


def lower_head(b: Builder, head, x: Act, out: torch.Tensor, out_mode: str) -> None:
    conv = head[0]
    k = conv.kernel_size[0]
    b.conv([(x, False)], conv.weight.detach().float().cpu(), conv.bias, name='segmentation_head.0',
           pad=(k // 2, k // 2), act='none', out_mode=out_mode, out_tensor=out)


def lower_decoder_and_head(b: Builder, model, feats: List[Act], out: torch.Tensor, out_mode: str) -> Optional[Act]:
    """Decoder + segmentation head into ``out``.  Returns the decoder's output activation, or None when the head was
    fused into the decoder's last conv (LinkNet: its 1x1 head rides in that conv's epilogue)."""
    head = model.segmentation_head
    # LinkNet ends in conv1x1+BN+ReLU (16 -> 32 channels at full resolution) followed by a 1x1 segmentation head: fused,
    # the 32-channel full-resolution tensor (the largest activation of the network) is never written or read back.
    if model.decoder.kind == 'linknet' and tuple(head[0].kernel_size) == (1, 1) and head[0].out_channels <= 4:
        return lower_linknet_decoder(b, model.decoder, feats, head=(head, out, out_mode))
    y = DECODER_LOWERING[model.decoder.kind](b, model.decoder, feats)
    lower_head(b, head, y, out, out_mode)
    return y
