"""CPU oracle, seeded checkpoint and golden-vector loader of the ResNeSt-50 backbone variant.  TEST INFRASTRUCTURE ONLY.

``I2P`` builds ``resnest50()`` for any arch containing 'resnest' (reference model_building.py:48-49).  Like
``reference_port``, the forward pass is restated with ``torch.nn.functional`` in fp32 on the CPU, citing the reference
lines it follows (paths relative to the reference tree); ``tests/golden/make_golden_resnest.py`` pins it to the
reference's own module and ``tests/test_oracle_resnest.py`` checks it against those vectors.  Nothing in
``synergynet_b200/`` may import this module.
"""
from __future__ import annotations

import os
from typing import Dict

import torch
import torch.nn.functional as F

from oracle.golden import GOLDEN_DIR, _with_inputs
from oracle.reference_port import BN_EPS
from synergynet_b200 import synthetic

RESNEST_VECTORS = os.path.join(GOLDEN_DIR, 'resnest_vectors.npz')
_CACHE: Dict[int, Dict[str, torch.Tensor]] = {}


@torch.no_grad()
def resnest50_forward(sd: Dict[str, torch.Tensor], x: torch.Tensor, prefix: str = 'I2P.backbone.', bn=None,
                      return_stages: bool = False):
    """ResNet.forward of ``resnest50()`` (backbone_nets/ResNeSt/resnest.py:33-41: radix 2, cardinality 1, deep stem of
    width 32, avg_down, avd, avd_first=False), Bottleneck (ResNeSt/resnet.py:94-127) with SplAtConv2d (splat.py:47-98).
    Returns (out62 = ori|shape|exp, pooled 2048-d feature) -- the pair I2P unpacks -- and, with ``return_stages``, the
    four stage outputs.  ``bn(t, key)`` replaces the eval-mode BatchNorm (the synthetic checkpoint's calibration pass)."""
    sd = {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}

    if bn is None:
        def bn(t, key):
            return F.batch_norm(t, sd[key + '.running_mean'], sd[key + '.running_var'], sd[key + '.weight'],
                                sd[key + '.bias'], False, 0.0, BN_EPS)

    x = F.relu(bn(F.conv2d(x, sd['conv1.0.weight'], None, 2, 1), 'conv1.1'))                 # resnet.py:182-190
    x = F.relu(bn(F.conv2d(x, sd['conv1.3.weight'], None, 1, 1), 'conv1.4'))
    x = F.relu(bn(F.conv2d(x, sd['conv1.6.weight'], None, 1, 1), 'bn1'))                     # :299-301
    x = F.max_pool2d(x, 3, 2, 1)                                                              # :302
    stages = []
    for li, (blocks, stride) in enumerate(((3, 1), (4, 2), (6, 2), (3, 2)), 1):               # :197-219, :304-307
        for j in range(blocks):
            pre = f'layer{li}.{j}'
            out = F.relu(bn(F.conv2d(x, sd[f'{pre}.conv1.weight']), f'{pre}.bn1'))            # :97-101
            # SplAtConv2d (splat.py:47-82)
            sp = F.relu(bn(F.conv2d(out, sd[f'{pre}.conv2.conv.weight'], None, 1, 1, 1, 2), f'{pre}.conv2.bn0'))
            c = sp.shape[1] // 2
            x0, x1 = torch.split(sp, c, dim=1)
            gap = F.adaptive_avg_pool2d(x0 + x1, 1)
            gap = F.relu(bn(F.conv2d(gap, sd[f'{pre}.conv2.fc1.weight'], sd[f'{pre}.conv2.fc1.bias']), f'{pre}.conv2.bn1'))
            att = F.conv2d(gap, sd[f'{pre}.conv2.fc2.weight'], sd[f'{pre}.conv2.fc2.bias'])
            att = F.softmax(att.view(att.shape[0], 1, 2, -1).transpose(1, 2), dim=1).reshape(att.shape[0], -1, 1, 1)
            a0, a1 = torch.split(att, c, dim=1)
            out = a0 * x0 + a1 * x1
            if j == 0 and stride > 1:                                                          # avd_layer (:45-50, :113-114)
                out = F.avg_pool2d(out, 3, stride, 1)
            out = bn(F.conv2d(out, sd[f'{pre}.conv3.weight']), f'{pre}.bn3')                  # :116-117
            identity = x
            if j == 0:                                                                         # downsample (:246-261)
                if stride > 1:
                    identity = F.avg_pool2d(identity, stride, stride, ceil_mode=True, count_include_pad=False)
                identity = bn(F.conv2d(identity, sd[f'{pre}.downsample.1.weight']), f'{pre}.downsample.2')
            x = F.relu(out + identity)                                                         # :124-125
        stages.append(x)
    pooled = torch.flatten(F.adaptive_avg_pool2d(x, 1), 1)                                     # :309-312
    out62 = torch.cat([F.linear(pooled, sd[f'{k}.weight'], sd[f'{k}.bias']) for k in ('fc_ori', 'fc_shape', 'fc_exp')], 1)
    if return_stages:
        return out62, pooled, stages
    return out62, pooled                                                                       # :316-324


@torch.no_grad()
def build_resnest50_state_dict(seed: int = 0) -> Dict[str, torch.Tensor]:
    """Seeded, calibrated state dict of ``ResNeSt.resnest50()`` (reference backbone_nets/ResNeSt key schema, keys without
    prefix, 482 entries).  Convs and Linears are seeded like the reference's own initialiser, BatchNorm affine parameters
    randomised; then every BatchNorm's running statistics are set to the batch statistics of its own input over 16
    calibration crops -- what one train-mode pass with ``momentum=None`` leaves behind (mean, unbiased variance) -- in
    float64.  With random statistics the network nearly forgets its input and the split-attention weights all sit near
    0.5; calibrated, about half of out62 depends on the face and the attention weights span most of (0, 1)."""
    if seed in _CACHE:
        return _CACHE[seed]
    from synergynet_b200 import backbone
    m = backbone.resnest50()
    synthetic.seeded_init_(m, 400 + seed)
    synthetic.randomize_batchnorm_(m, 400 + seed)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    sd64 = {k: v.double() for k, v in sd.items()}
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(16, seed=500 + seed)).double()

    def calibrate(t, k):
        mean, var = t.mean(dim=(0, 2, 3)), t.var(dim=(0, 2, 3), unbiased=True)
        sd64[k + '.running_mean'], sd64[k + '.running_var'] = mean, var
        sd[k + '.running_mean'].copy_(mean.float())
        sd[k + '.running_var'].copy_(var.float())
        return F.batch_norm(t, mean, var, sd64[k + '.weight'], sd64[k + '.bias'], False, 0.0, 1e-5)

    resnest50_forward(sd64, x, prefix='', bn=calibrate)
    _CACHE[seed] = sd
    return sd


def resnest_inputs() -> dict:
    """The 8 structured crops ``tests/golden/make_golden_resnest.py`` runs the reference's ``resnest50()`` on (pure noise
    crops lie far outside what the synthetic checkpoint was calibrated on: its activations grow ~1000x there)."""
    return {'x_u8': synthetic.make_structured_crops_u8(8, seed=61).numpy()}


def load_resnest_vectors() -> dict:
    """``resnest_vectors.npz`` with its inputs rebuilt: the checkpoint schema (``keys``, ``key_shapes`` as 'AxBxC'
    strings), ``out62`` / ``pool2048`` of the 8 crops, ``stage{1..4}_sub`` (face 0, every 8th channel, spatially
    subsampled by ``stage_stride``) and ``lmk`` (the reference's landmarks of its own out62)."""
    return _with_inputs(RESNEST_VECTORS, resnest_inputs())
