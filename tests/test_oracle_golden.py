"""Pin the CPU oracle (oracle/reference_port.py) to the vectors recorded from the live reference
(tests/golden/make_golden.py).  CPU only."""

import numpy as np
import pytest
import torch

from oracle import golden
from oracle import reference_port as rp
from oracle import synth_model
from synergynet_b200 import synthetic

TOL = 2e-5       # oracle and reference run the same ATen kernels; slack is for cross-host ISA paths


@pytest.fixture(scope='module')
def gold():
    return golden.load_ref_vectors()


@pytest.fixture(scope='module')
def sd():
    return synth_model.build_state_dict(0)


@pytest.fixture(scope='module')
def basis():
    return rp.gather_sparse_basis(synthetic.make_3dmm(0))


@pytest.fixture(scope='module')
def fwd(gold, sd):
    x = synthetic.normalize_crops(torch.from_numpy(gold['x_u8']))
    return rp.mobilenetv2_forward(sd, x, return_features=True)


def test_inputs_are_reproducible(gold):
    u8 = torch.cat([synthetic.make_structured_crops_u8(6, seed=11), synthetic.make_crops_u8(2, seed=0)])
    assert np.array_equal(u8.numpy(), gold['x_u8'])


def test_backbone_params_and_pool(gold, fwd):
    params, pool, _ = fwd
    assert rp.max_rel_err(params.numpy(), gold['params']) < TOL
    assert rp.max_rel_err(pool.numpy(), gold['pool']) < TOL


def test_backbone_block_activations(gold, fwd):
    _, _, feats = fwd
    assert len(feats) == 19
    for i, f in enumerate(feats):
        sub = f[0, :, ::5, ::5].numpy()
        assert sub.shape == gold[f'feat{i:02d}_sub'].shape
        assert rp.max_rel_err(sub, gold[f'feat{i:02d}_sub']) < TOL, i
        assert abs(float(f.abs().double().mean()) / float(gold[f'feat{i:02d}_absmean']) - 1) < 1e-5


def test_reconstruct_sparse(gold, basis):
    lmk = rp.reconstruct_vertex_62(gold['params'], basis)
    assert lmk.shape == (8, 3, 68)
    assert rp.max_rel_err(lmk, gold['lmk']) < 1e-6
    raw = rp.reconstruct_vertex_62(gold['params'], basis, transform=False)
    assert rp.max_rel_err(raw, gold['lmk_notransform']) < 1e-6
    assert rp.nme_vs_reference(lmk, gold['lmk']).max() < 1e-6


def test_reconstruct_dense(gold, basis):
    dense = rp.reconstruct_vertex_62(gold['params'][:3], basis, dense=True)
    assert dense.shape == (3, 3, synthetic.NVER)
    assert rp.max_rel_err(dense[:, :, ::53], gold['dense_sub']) < 1e-6
    kp_vert = basis['keypoints'][::3] // 3
    assert rp.max_rel_err(dense[:, :, kp_vert], gold['dense_kp']) < 1e-6
    assert np.allclose(dense.astype(np.float64).sum(2), gold['dense_sum64'], rtol=1e-6, atol=1.0)


def test_length_mismatch_raises(basis):
    with pytest.raises(RuntimeError, match='length of params mismatch'):
        rp.reconstruct_vertex_62(np.zeros((2, 61), np.float32), basis)


def test_per_face_numpy_api(gold, basis):
    p0 = gold['params'][0]
    roi = [30.2, 41.7, 211.4, 222.9, 0.99]
    lmk = rp.rescale_to_image(rp.reconstruct_vertex_62(p0[None], basis)[0], roi)
    assert rp.max_rel_err(lmk, gold['np_sparse']) < 1e-6
    dn = rp.rescale_to_image(rp.reconstruct_vertex_62(p0[None], basis, dense=True)[0], roi)
    assert rp.max_rel_err(dn[:, ::53], gold['np_dense_sub']) < 1e-6
    ang, t3d = rp.predict_pose(p0, basis, roi)
    assert np.allclose(ang, gold['np_pose_angles'], rtol=0, atol=1e-4)
    assert np.allclose(t3d, gold['np_pose_t3d'], rtol=1e-6)


def test_crop_img_bit_exact(gold):
    for i, box in enumerate(gold['crop_boxes']):
        assert np.array_equal(rp.crop_img(gold['crop_img'], list(box)), gold[f'crop_out{i}'])


def test_training_forward_losses_and_pointnet_heads(gold, sd, basis):
    """SynergyNet.forward (model_building.py:141-157): the oracle's MLP_for / MLP_rev / WingLoss / ParamLoss against the
    values recorded from the reference's own modules."""
    x = synthetic.normalize_crops(torch.from_numpy(gold['x_u8']))
    loss, t = rp.synergy_forward(sd, basis, x, torch.from_numpy(gold['fwd_target']))
    for k in ('loss_LMK_f0', 'loss_LMK_pointNet', 'loss_Param_In', 'loss_Param_S2', 'loss_Param_S1S2'):
        assert rp.max_rel_err(loss[k].numpy(), gold['fwd_' + k]) < TOL, k
    assert rp.max_rel_err(t['point_residual'].numpy(), gold['fwd_point_residual']) < TOL
    assert rp.max_rel_err(t['vertex_lmk_refined'].numpy(), gold['fwd_vertex_lmk_refined']) < TOL
    assert rp.max_rel_err(t['_3D_attr_S2'].numpy(), gold['fwd_3D_attr_S2']) < TOL
    assert float(np.abs(gold['fwd_point_residual']).max()) > 0.1          # the heads are alive in the synthetic checkpoint


def test_resnet50_variant(gold):
    """BASELINE.json configs[4]: the oracle's ResNet-50 against the reference's resnet_backbone.resnet50() module."""
    sd = {'I2P.backbone.' + k: v for k, v in synth_model.build_resnet50_state_dict(0).items()}
    x = synthetic.normalize_crops(torch.from_numpy(gold['x_u8']))[:4]
    out, pooled = rp.resnet50_forward(sd, x)
    assert out.shape == (4, 102) and pooled.shape == (4, 2048)
    assert rp.max_rel_err(out.numpy(), gold['resnet50_out102']) < TOL


def test_thousand_face_batch_sample(gold, sd, basis):
    """The 1024 distinct faces of the configs[1]-size golden batch: the oracle on a 16-face sample."""
    xs = synthetic.normalize_crops(synthetic.make_structured_crops_u8(1024, seed=77))
    idx = torch.arange(0, 1024, 64)
    p, _ = rp.mobilenetv2_forward(sd, xs[idx])
    assert rp.max_rel_err(p.numpy(), gold['params1024'][idx.numpy()]) < TOL
    assert rp.max_rel_err(rp.reconstruct_vertex_62(p.numpy(), basis), gold['lmk1024_even'][idx.numpy() // 2]) < TOL
    # the reconstruction of the reference's own parameters, which stands in for the landmarks not stored (odd faces)
    lmk = rp.reconstruct_vertex_62(gold['params1024'][::2], basis)
    assert rp.max_rel_err(lmk, gold['lmk1024_even']) < 1e-6
    assert rp.nme_vs_reference(lmk, gold['lmk1024_even']).max() < 1e-6
