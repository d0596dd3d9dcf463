"""ResNeSt-50 backbone variant (I2P with arch 'resnest*'), CPU side: the oracle against the vectors recorded from the
reference's own ``resnest50()`` module, the parameter container's key schema, and the C ABI's layer plan."""
import ctypes as C
import types

import numpy as np
import pytest
import torch

from oracle import reference_port as rp
from oracle import resnest_port
from synergynet_b200 import _lib, backbone, synthetic

TOL = 2e-5


@pytest.fixture(scope='module')
def gold():
    return resnest_port.load_resnest_vectors()


@pytest.fixture(scope='module')
def sd():
    return resnest_port.build_resnest50_state_dict(0)


def test_oracle_matches_reference_module(gold, sd):
    x = synthetic.normalize_crops(torch.from_numpy(gold['x_u8']))
    out62, pooled, stages = resnest_port.resnest50_forward(sd, x, prefix='', return_stages=True)
    assert out62.shape == (8, 62) and pooled.shape == (8, 2048)
    e_out, e_pool = rp.max_rel_err(out62.numpy(), gold['out62']), rp.max_rel_err(pooled.numpy(), gold['pool2048'])
    print(f'oracle vs reference resnest50: out62 {e_out:.2e}, pool2048 {e_pool:.2e}')
    assert e_out < TOL and e_pool < TOL
    for i, (f, s) in enumerate(zip(stages, gold['stage_stride']), 1):
        assert rp.max_rel_err(f[0, ::8, ::s, ::s].numpy(), gold[f'stage{i}_sub']) < TOL, i
    # the calibrated checkpoint keeps the input alive: a large part of out62 differs from face to face
    spread = np.abs(gold['out62'] - gold['out62'].mean(0)).max()
    assert spread > 0.3 * np.abs(gold['out62']).max()


def test_landmarks_of_the_reference_parameters(gold, synth_pack):
    basis = rp.gather_sparse_basis(synthetic.make_3dmm(0))
    lmk = rp.reconstruct_vertex_62(gold['out62'], basis)
    assert rp.max_rel_err(lmk, gold['lmk']) < 1e-6


def test_container_matches_reference_schema(gold):
    sd = backbone.resnest50().state_dict()
    assert list(sd.keys()) == [str(k) for k in gold['keys']]
    assert ['x'.join(str(d) for d in v.shape) for v in sd.values()] == [str(s) for s in gold['key_shapes']]
    assert len(sd) == 482
    assert sum(p.numel() for p in backbone.resnest50().parameters()) == 25_643_238


def test_layer_desc_agrees_with_container():
    lib = _lib.load()
    keys = backbone.resnest50_layer_keys()
    assert lib.syn_resnest_num_layers() == len(keys) == 87
    mods = dict(backbone.resnest50().named_modules())
    d = _lib.ResNeStLayerDesc()
    for i, (ck, bk) in enumerate(keys):
        assert lib.syn_resnest_layer_desc(i, C.byref(d)) == 0
        conv = mods[ck]
        assert d.name.decode() == ck
        assert (d.bn_name.decode() if d.bn_name else None) == bk
        if bk is not None:
            assert mods[bk].num_features == conv.out_channels
        assert (d.cin, d.cout, d.ksize, d.stride, d.groups) == (conv.in_channels, conv.out_channels, conv.kernel_size[0],
                                                                conv.stride[0], conv.groups), ck
        assert d.has_bias == (conv.bias is not None), ck
    assert lib.syn_resnest_layer_desc(87, C.byref(d)) == 1
    assert lib.syn_resnest_layer_desc(-1, C.byref(d)) == 1
    # spatial sizes: the stem runs at 60, the stages at 30 / 15 / 8 / 4 (conv2 before the avd pool of block 0)
    assert lib.syn_resnest_layer_desc(0, C.byref(d)) == 0 and (d.h_in, d.h_out) == (120, 60)
    assert lib.syn_resnest_layer_desc(86, C.byref(d)) == 0 and (d.h_in, d.h_out) == (4, 4)
    i = [k for k, _ in keys].index('layer3.0.conv2.conv')
    assert lib.syn_resnest_layer_desc(i, C.byref(d)) == 0 and (d.h_in, d.h_out) == (15, 15)
    assert lib.syn_resnest_layer_desc(i + 3, C.byref(d)) == 0 and (d.h_in, d.h_out) == (8, 8)      # conv3 after the pool


def test_i2p_builds_resnest_on_cpu():
    from synergynet_b200.model_building import I2P
    for arch in ('resnest50', 'resnest101'):       # the reference builds resnest50() for any 'resnest' arch
        m = I2P(types.SimpleNamespace(arch=arch))
        assert isinstance(m.backbone, backbone.ResNeSt50Params)
        assert m._variant == 'resnest50'
    for arch in ('mobilenet_1', 'ghostnet'):
        with pytest.raises(RuntimeError, match='resnest50'):
            I2P(types.SimpleNamespace(arch=arch))
    with pytest.raises(RuntimeError, match='Please choose'):
        I2P(types.SimpleNamespace(arch='vgg16'))
