"""ResNeSt-50 backbone variant (I2P with arch 'resnest*') on the B200: the sm_100a path through the C ABI and the
drop-in model against the vectors recorded from the reference's own ``resnest50()`` module and the CPU oracle."""
import types

import numpy as np
import pytest
import torch

from oracle import reference_port as rp
from oracle import resnest_port
from synergynet_b200 import synthetic

pytestmark = pytest.mark.gpu
TOL = 1e-4
# stem conv + 2 stem GEMMs + max-pool; 16 blocks x (conv1, conv2, attention, apply, conv3); 4 shortcut convs and 3
# avg-down pools; global average pool + heads
LAUNCHES = 4 + 16 * 5 + 4 + 3 + 2


@pytest.fixture(scope='module')
def gold():
    return resnest_port.load_resnest_vectors()


@pytest.fixture(scope='module')
def sd():
    return {'I2P.backbone.' + k: v for k, v in resnest_port.build_resnest50_state_dict(0).items()}


@pytest.fixture(scope='module')
def model(synth_pack, sd):
    from synergynet_b200 import model_building
    m = model_building.SynergyNet(types.SimpleNamespace(arch='resnest50', img_size=120, devices_id=[0]))
    missing = m.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and all(not k.startswith('I2P.') for k in missing.missing_keys)
    return m.eval()


def test_matches_reference_module(model, gold, sd):
    x = synthetic.normalize_crops(torch.from_numpy(gold['x_u8'])).cuda()
    eng = model._engine(torch.device('cuda', 0))
    n0 = eng.launch_count
    out, pool = eng.forward_resnest50(x)
    torch.cuda.synchronize()
    assert eng.launch_count - n0 == LAUNCHES
    assert out.shape == (8, 62) and pool.shape == (8, 2048)
    want, want_pool = resnest_port.resnest50_forward(sd, x.cpu())
    errs = {'out62 vs reference': rp.max_rel_err(out.cpu().numpy(), gold['out62']),
            'pool2048 vs reference': rp.max_rel_err(pool.cpu().numpy(), gold['pool2048']),
            'out62 vs oracle': rp.max_rel_err(out.cpu().numpy(), want.numpy()),
            'pool2048 vs oracle': rp.max_rel_err(pool.cpu().numpy(), want_pool.numpy())}
    print('resnest50 max-rel errors: ' + ', '.join(f'{k} {v:.2e}' for k, v in errs.items()))
    assert all(v < TOL for v in errs.values()), errs
    # forward_test returns the backbone's own (params62, avgpool) pair, no adapter
    params = model.forward_test(x)
    assert torch.equal(params, out)
    p2, feat = model.I2P.forward_test(x)
    assert torch.equal(p2, out) and torch.equal(feat, pool)
    # landmarks from the reference's own parameters
    lmk = model.reconstruct_vertex_62(torch.from_numpy(np.ascontiguousarray(gold['out62'])).cuda())
    e_lmk = rp.max_rel_err(lmk.cpu().numpy(), gold['lmk'])
    print(f'resnest50 landmarks of the reference params: {e_lmk:.2e}')
    assert e_lmk < TOL
    with pytest.raises(RuntimeError, match='1280-d image feature'):
        model(x, params)
    eng.raise_if_error()


@pytest.mark.parametrize('batch', [1, 5, 37])
def test_ragged_batches_match_oracle(model, sd, batch):
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(batch, seed=90 + batch))
    want, want_pool = resnest_port.resnest50_forward(sd, x)
    eng = model._engine(torch.device('cuda', 0))
    got, gp = eng.forward_resnest50(x.cuda())
    e_out, e_pool = rp.max_rel_err(got.cpu().numpy(), want.numpy()), rp.max_rel_err(gp.cpu().numpy(), want_pool.numpy())
    print(f'resnest50 B={batch}: out62 {e_out:.2e}, pool2048 {e_pool:.2e} vs the oracle')
    assert e_out < TOL and e_pool < TOL
    k = batch // 2
    one, one_pool = eng.forward_resnest50(x[k:k + 1].cuda())
    assert rp.max_rel_err(one.cpu().numpy(), got[k:k + 1].cpu().numpy()) < 1e-6
    assert rp.max_rel_err(one_pool.cpu().numpy(), gp[k:k + 1].cpu().numpy()) < 1e-6
    eng.raise_if_error()


def test_c_abi_errors(model, sd):
    from synergynet_b200.backbone import resnest50_layer_keys
    eng = model._engine(torch.device('cuda', 0))       # a committed MobileNetV2 handle for the shared state
    from synergynet_b200.engine import Engine
    fresh = Engine(0)
    try:
        lib, h = fresh._lib, fresh._h
        x = torch.zeros((1, 3, 120, 120), device='cuda')
        o62, pool = torch.empty((1, 62), device='cuda'), torch.empty((1, 2048), device='cuda')
        # a forward on a handle whose ResNeSt weights were never committed (the MobileNetV2 path is)
        fresh.load_backbone(model.I2P._rt._mbv2_stub, prefix='')
        z = torch.zeros(62)
        fresh.load_3dmm(z, z + 1, torch.zeros(3, 1), torch.zeros(3, 40), torch.zeros(3, 10))
        fresh.commit()
        rc = lib.syn_resnest50_forward(h, x.data_ptr(), 1, o62.data_ptr(), pool.data_ptr(), None)
        assert rc == 3 and b'not committed' in lib.syn_last_error()                     # SYN_ERR_STATE
        keys = resnest50_layer_keys()
        w = sd[f'I2P.backbone.{keys[4][0]}.weight'].contiguous()                         # layer1.0.conv2.conv (groups 2)
        bn = [sd[f'I2P.backbone.{keys[4][1]}.{k}'].contiguous() for k in ('weight', 'bias', 'running_mean', 'running_var')]
        bnp = [t.data_ptr() for t in bn]
        assert lib.syn_resnest_set_layer(h, 4, w.data_ptr(), w.numel(), None, *bnp, 1e-5) == 0
        assert lib.syn_resnest_set_layer(h, 4, w.data_ptr(), w.numel() * 2, None, *bnp, 1e-5) == 4        # SYN_ERR_SHAPE
        assert lib.syn_resnest_set_layer(h, 4, w.data_ptr(), w.numel(), bn[0].data_ptr(), *bnp, 1e-5) == 1  # no bias here
        assert lib.syn_resnest_set_layer(h, 4, w.data_ptr(), w.numel(), None, None, None, None, None, 1e-5) == 1   # BN missing
        fc2 = keys[6][0]                                                                  # layer1.0.conv2.fc2: bias, no BN
        w2, b2 = sd[f'I2P.backbone.{fc2}.weight'].contiguous(), sd[f'I2P.backbone.{fc2}.bias'].contiguous()
        assert lib.syn_resnest_set_layer(h, 6, w2.data_ptr(), w2.numel(), b2.data_ptr(), None, None, None, None, 1e-5) == 0
        assert lib.syn_resnest_set_layer(h, 6, w2.data_ptr(), w2.numel(), None, None, None, None, None, 1e-5) == 1   # bias missing
        assert lib.syn_resnest_set_layer(h, 6, w2.data_ptr(), w2.numel(), b2.data_ptr(), *bnp, 1e-5) == 1           # has no BN
        assert lib.syn_resnest_set_layer(h, 87, w2.data_ptr(), w2.numel(), b2.data_ptr(), None, None, None, None, 1e-5) == 1
        assert lib.syn_resnest_commit(h) == 3                                             # layers missing
    finally:
        fresh.close()
    eng.raise_if_error()
