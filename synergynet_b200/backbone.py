"""Parameter containers with the reference's checkpoint key schema, plus the layer plan.

The arithmetic of the hot path lives in the CUDA library (``csrc/``); the ``nn.Module`` classes
here only *hold* parameters under the same ``state_dict`` keys as the reference so that its
checkpoints load unchanged (SURVEY.md section 8(b); reference
``backbone_nets/mobilenetv2_backbone.py:33-74,104-158`` and
``backbone_nets/pointnet_backbone.py:7-29,67-88``).  None of them implements a torch forward:
there is deliberately no CPU/eager fallback for the product path.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List

import torch
from torch import nn

# (expand ratio t, out channels c, repeats n, first stride s) -- mobilenetv2_backbone.py:108-117
MBV2_STAGES = ((1, 16, 1, 1), (6, 24, 2, 2), (6, 32, 3, 2), (6, 64, 4, 2),
               (6, 96, 3, 1), (6, 160, 3, 2), (6, 320, 1, 1))
STEM_CH, LAST_CH = 32, 1280
HEAD_DIMS = (('classifier_ori', 12), ('classifier_shape', 40), ('classifier_exp', 10))
IMG = 120


@dataclass(frozen=True)
class ConvSpec:
    """One conv+BN(+ReLU6) of the backbone, in execution order."""
    index: int          # 0..51, the order the C-ABI expects (include/synergy_b200.h)
    conv_key: str       # state_dict prefix of the Conv2d ("...weight")
    bn_key: str         # state_dict prefix of the BatchNorm2d
    kind: str           # 'stem' | 'expand' | 'dw' | 'project' | 'last'
    block: int          # features index (0..18)
    cin: int
    cout: int
    ksize: int
    stride: int
    groups: int
    relu6: bool
    h_in: int
    h_out: int
    residual: bool = False   # project conv of a block with a skip connection


def _out_size(h: int, stride: int) -> int:
    return (h + 2 - 3) // stride + 1        # 3x3, padding 1


def conv_plan(prefix: str = 'features') -> List[ConvSpec]:
    """The 52 convolutions of MobileNetV2 @120x120 (SURVEY.md section 8(a) shape table)."""
    plan: List[ConvSpec] = []

    def add(**kw):
        plan.append(ConvSpec(index=len(plan), **kw))

    h = IMG
    ho = _out_size(h, 2)
    add(conv_key=f'{prefix}.0.0', bn_key=f'{prefix}.0.1', kind='stem', block=0, cin=3,
        cout=STEM_CH, ksize=3, stride=2, groups=1, relu6=True, h_in=h, h_out=ho)
    h, cin, blk = ho, STEM_CH, 1
    for t, c, n, s in MBV2_STAGES:
        for i in range(n):
            stride = s if i == 0 else 1
            hid = cin * t
            base = f'{prefix}.{blk}.conv'
            j = 0
            if t != 1:
                add(conv_key=f'{base}.0.0', bn_key=f'{base}.0.1', kind='expand', block=blk,
                    cin=cin, cout=hid, ksize=1, stride=1, groups=1, relu6=True, h_in=h, h_out=h)
                j = 1
            ho = _out_size(h, stride)
            add(conv_key=f'{base}.{j}.0', bn_key=f'{base}.{j}.1', kind='dw', block=blk, cin=hid,
                cout=hid, ksize=3, stride=stride, groups=hid, relu6=True, h_in=h, h_out=ho)
            add(conv_key=f'{base}.{j + 1}', bn_key=f'{base}.{j + 2}', kind='project', block=blk,
                cin=hid, cout=c, ksize=1, stride=1, groups=1, relu6=False, h_in=ho, h_out=ho,
                residual=(stride == 1 and cin == c))
            h, cin, blk = ho, c, blk + 1
    add(conv_key=f'{prefix}.{blk}.0', bn_key=f'{prefix}.{blk}.1', kind='last', block=blk, cin=cin,
        cout=LAST_CH, ksize=1, stride=1, groups=1, relu6=True, h_in=h, h_out=h)
    return plan


def _conv_bn_act(cin, cout, k, stride, groups):
    return nn.Sequential(nn.Conv2d(cin, cout, k, stride, (k - 1) // 2, groups=groups, bias=False),
                         nn.BatchNorm2d(cout), nn.ReLU6(inplace=True))


class _MBConvParams(nn.Module):
    """Holds ``conv.*`` of one inverted-residual block (keys as mobilenetv2_backbone.py:58-68)."""

    def __init__(self, cin, cout, stride, t):
        super().__init__()
        hid = cin * t
        mods = []
        if t != 1:
            mods.append(_conv_bn_act(cin, hid, 1, 1, 1))
        mods += [_conv_bn_act(hid, hid, 3, stride, hid), nn.Conv2d(hid, cout, 1, bias=False),
                 nn.BatchNorm2d(cout)]
        self.conv = nn.Sequential(*mods)


class MobileNetV2Params(nn.Module):
    """State-dict twin of the reference ``MobileNetV2`` (features + three heads)."""

    def __init__(self):
        super().__init__()
        feats = [_conv_bn_act(3, STEM_CH, 3, 2, 1)]
        cin = STEM_CH
        for t, c, n, s in MBV2_STAGES:
            for i in range(n):
                feats.append(_MBConvParams(cin, c, s if i == 0 else 1, t))
                cin = c
        feats.append(_conv_bn_act(cin, LAST_CH, 1, 1, 1))
        self.features = nn.Sequential(*feats)
        self.last_channel = LAST_CH
        self.num_ori, self.num_shape, self.num_exp = (d for _, d in HEAD_DIMS)
        for name, dim in HEAD_DIMS:
            setattr(self, name, nn.Sequential(nn.Dropout(0.2), nn.Linear(LAST_CH, dim)))
        for m in self.modules():      # same distributions as mobilenetv2_backbone.py:161-171
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode='fan_out')
            elif isinstance(m, nn.Linear):
                nn.init.normal_(m.weight, 0, 0.01)
                nn.init.zeros_(m.bias)

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError('MobileNetV2Params is a parameter container; the forward pass runs in '
                           'the sm_100a library via synergynet_b200.engine.Engine')


def mobilenet_v2(pretrained: bool = False, **_):
    return MobileNetV2Params()


class _PointMLPParams(nn.Module):
    """Parameter container in the reference's key schema; ``forward`` runs in the sm_100a library through the engine
    of the model that owns the module (``_engine_provider`` is installed by ``model_building._SynergyBase``)."""
    _NET = -1

    def __init__(self, num_pts, convs, bns):
        super().__init__()
        for name, (ci, co) in convs.items():
            setattr(self, name, nn.Conv1d(ci, co, 1))
        for name, c in bns.items():
            setattr(self, name, nn.BatchNorm1d(c))
        self.num_pts = num_pts
        object.__setattr__(self, '_engine_provider', None)

    def _engine(self, t):
        if self._engine_provider is None:
            raise RuntimeError(f'{type(self).__name__}: not attached to a SynergyNet model (its engine owns the GPU state)')
        if self.num_pts != 68:
            raise RuntimeError('the sm_100a PointNet heads are built for 68 landmarks (MLP_for(68) / MLP_rev(68))')
        return self._engine_provider(t, self._NET)


class MLP_for(_PointMLPParams):
    """pointnet_backbone.py:7-64 (forwardDirection.*, 63 keys)."""
    _NET = 0

    def __init__(self, num_pts):
        chans = [(3, 64), (64, 64), (64, 64), (64, 128), (128, 1024), (2418, 512), (512, 256),
                 (256, 128), (128, 3)]
        super().__init__(num_pts, {f'conv{i + 1}': c for i, c in enumerate(chans)},
                         {f'bn{i + 1}': c[1] for i, c in enumerate(chans)})

    def forward(self, x, other_input1=None, other_input2=None, other_input3=None):
        """point_residual (B,3,68) from landmarks x (B,3,68), avgpool (B,1280), shape code (B,40), expression code (B,10)
        (pointnet_backbone.py:31-64; eval-mode BatchNorm)."""
        import torch
        params = torch.zeros((x.shape[0], 62), device=x.device, dtype=torch.float32)
        params[:, 12:52] = other_input2
        params[:, 52:62] = other_input3
        res, _ = self._engine(x).mlp_for(x, other_input1, params)
        return res if x.is_cuda else res.to(x.device)


class MLP_rev(_PointMLPParams):
    """pointnet_backbone.py:67-106 (reverseDirection.*, 56 keys)."""
    _NET = 1

    def __init__(self, num_pts):
        chans = [(3, 64), (64, 64), (64, 64), (64, 128), (128, 1024)]
        convs = {f'conv{i + 1}': c for i, c in enumerate(chans)}
        bns = {f'bn{i + 1}': c[1] for i, c in enumerate(chans)}
        for tag, dim in (('6_1', 12), ('6_2', 40), ('6_3', 10)):
            convs[f'conv{tag}'] = (1024, dim)
            bns[f'bn{tag}'] = dim
        super().__init__(num_pts, convs, bns)

    def forward(self, x, other_input1=None, other_input2=None, other_input3=None):
        """(B,62) = [rot12 | shape40 | expr10] regressed back from landmarks x (B,3,68) (pointnet_backbone.py:90-106)."""
        out = self._engine(x).mlp_rev(x)
        return out if x.is_cuda else out.to(x.device)


# ---- ResNet-50 backbone variant (reference backbone_nets/resnet_backbone.py:120-249; BASELINE.json configs[4]) -------

class _Bottleneck(nn.Module):
    expansion = 4

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = nn.Conv2d(planes, planes, 3, stride, 1, bias=False)
        self.bn2 = nn.BatchNorm2d(planes)
        self.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.downsample = downsample


class ResNet50Params(nn.Module):
    """Key schema of ``resnet_backbone.resnet50()`` (conv1/bn1, layer1..4.{i}.conv{1,2,3}/bn{1,2,3}/downsample.{0,1},
    fc_tex/fc_ori/fc_shape/fc_exp); parameter container, the forward pass runs in the sm_100a library."""
    feature_dim = 2048

    def __init__(self):
        super().__init__()
        self.conv1 = nn.Conv2d(3, 64, 7, 2, 3, bias=False)
        self.bn1 = nn.BatchNorm2d(64)
        inplanes = 64
        for li, (planes, blocks, stride) in enumerate(((64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)), 1):
            layers = []
            for j in range(blocks):
                ds = None
                if j == 0:
                    ds = nn.Sequential(nn.Conv2d(inplanes, planes * 4, 1, stride, bias=False), nn.BatchNorm2d(planes * 4))
                layers.append(_Bottleneck(inplanes, planes, stride if j == 0 else 1, ds))
                inplanes = planes * 4
            setattr(self, f'layer{li}', nn.Sequential(*layers))
        self.fc_tex = nn.Linear(2048, 40)
        self.fc_ori = nn.Linear(2048, 12)
        self.fc_shape = nn.Linear(2048, 40)
        self.fc_exp = nn.Linear(2048, 10)
        for m in self.modules():                                            # resnet_backbone.py:184-189
            if isinstance(m, nn.Conv2d):
                nn.init.kaiming_normal_(m.weight, mode='fan_out', nonlinearity='relu')
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError('ResNet50Params is a parameter container; the forward pass runs in the sm_100a library')


def resnet50_conv_keys():
    """(conv key, bn key) of the 53 convolutions in the execution order of the C ABI (syn_resnet_set_conv)."""
    keys = [('conv1', 'bn1')]
    for li, blocks in enumerate((3, 4, 6, 3), 1):
        for j in range(blocks):
            pre = f'layer{li}.{j}'
            keys += [(f'{pre}.conv1', f'{pre}.bn1'), (f'{pre}.conv2', f'{pre}.bn2'), (f'{pre}.conv3', f'{pre}.bn3')]
            if j == 0:
                keys.append((f'{pre}.downsample.0', f'{pre}.downsample.1'))
    return keys


def resnet50(pretrained: bool = False, **_):
    return ResNet50Params()


# ---- ResNeSt-50 backbone variant (reference backbone_nets/ResNeSt/resnest.py:33-41, resnet.py:29-324, splat.py) ------

class _SplAtParams(nn.Module):
    """``SplAtConv2d`` with radix 2, cardinality 1 (splat.py:14-45): conv (groups 2), bn0, fc1 (+bias), bn1, fc2 (+bias)."""

    def __init__(self, gw):
        super().__init__()
        inter = max(gw * 2 // 4, 32)
        self.conv = nn.Conv2d(gw, gw * 2, 3, 1, 1, groups=2, bias=False)
        self.bn0 = nn.BatchNorm2d(gw * 2)
        self.fc1 = nn.Conv2d(gw, inter, 1)
        self.bn1 = nn.BatchNorm2d(inter)
        self.fc2 = nn.Conv2d(inter, gw * 2, 1)


class _SplAtBottleneck(nn.Module):
    expansion = 4

    def __init__(self, inplanes, planes, downsample=None):
        super().__init__()
        self.conv1 = nn.Conv2d(inplanes, planes, 1, bias=False)
        self.bn1 = nn.BatchNorm2d(planes)
        self.conv2 = _SplAtParams(planes)
        self.conv3 = nn.Conv2d(planes, planes * 4, 1, bias=False)
        self.bn3 = nn.BatchNorm2d(planes * 4)
        self.downsample = downsample


RESNEST_STAGES = ((64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2))     # (planes, blocks, stride), resnet.py:197-219


class ResNeSt50Params(nn.Module):
    """Key schema of ``ResNeSt.resnest50()`` (482 state-dict keys): the deep stem ``conv1.{0,1,3,4,6}`` + ``bn1``,
    ``layer1..4.{i}.conv1/bn1/conv2.{conv,bn0,fc1,bn1,fc2}/conv3/bn3/downsample.{1,2}``, fc_ori/fc_shape/fc_exp/fc_tex.
    Parameter container; the forward pass runs in the sm_100a library."""
    feature_dim = 2048

    def __init__(self):
        super().__init__()
        self.conv1 = nn.Sequential(nn.Conv2d(3, 32, 3, 2, 1, bias=False), nn.BatchNorm2d(32), nn.ReLU(inplace=True),
                                   nn.Conv2d(32, 32, 3, 1, 1, bias=False), nn.BatchNorm2d(32), nn.ReLU(inplace=True),
                                   nn.Conv2d(32, 64, 3, 1, 1, bias=False))
        self.bn1 = nn.BatchNorm2d(64)
        inplanes = 64
        for li, (planes, blocks, stride) in enumerate(RESNEST_STAGES, 1):
            layers = []
            for j in range(blocks):
                ds = None
                if j == 0:          # avg-down shortcut: AvgPool2d (identity in layer1), 1x1 conv, BN (resnet.py:246-261)
                    ds = nn.Sequential(nn.AvgPool2d(stride, stride, ceil_mode=True, count_include_pad=False),
                                       nn.Conv2d(inplanes, planes * 4, 1, bias=False), nn.BatchNorm2d(planes * 4))
                layers.append(_SplAtBottleneck(inplanes, planes, ds))
                inplanes = planes * 4
            setattr(self, f'layer{li}', nn.Sequential(*layers))
        self.fc_ori = nn.Linear(2048, 12)
        self.fc_shape = nn.Linear(2048, 40)
        self.fc_exp = nn.Linear(2048, 10)
        self.fc_tex = nn.Linear(2048, 40)
        for m in self.modules():                                            # resnet.py:235-241
            if isinstance(m, nn.Conv2d):
                m.weight.data.normal_(0, (2.0 / (m.kernel_size[0] * m.kernel_size[1] * m.out_channels)) ** 0.5)
            elif isinstance(m, nn.BatchNorm2d):
                m.weight.data.fill_(1)
                m.bias.data.zero_()

    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError('ResNeSt50Params is a parameter container; the forward pass runs in the sm_100a library')


def resnest50_layer_keys():
    """(conv key, BatchNorm key or None) of the 87 layers in the execution order of the C ABI (syn_resnest_set_layer)."""
    keys = [('conv1.0', 'conv1.1'), ('conv1.3', 'conv1.4'), ('conv1.6', 'bn1')]
    for li, (_, blocks, _) in enumerate(RESNEST_STAGES, 1):
        for j in range(blocks):
            pre = f'layer{li}.{j}'
            keys += [(f'{pre}.conv1', f'{pre}.bn1'), (f'{pre}.conv2.conv', f'{pre}.conv2.bn0'),
                     (f'{pre}.conv2.fc1', f'{pre}.conv2.bn1'), (f'{pre}.conv2.fc2', None), (f'{pre}.conv3', f'{pre}.bn3')]
            if j == 0:
                keys.append((f'{pre}.downsample.1', f'{pre}.downsample.2'))
    return keys


def resnest50(pretrained: bool = False, **_):
    return ResNeSt50Params()
