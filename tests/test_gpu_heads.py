"""SURVEY.md section 8 rows a10 / f4 on the B200: MLP_for / MLP_rev, WingLoss / ParamLoss and SynergyNet.forward
(inference mode) through the C ABI, against the vectors recorded from the reference's own modules and the CPU oracle."""
import types

import numpy as np
import pytest
import torch

from oracle import golden
from oracle import reference_port as rp
from oracle import synth_model
from synergynet_b200 import synthetic

pytestmark = pytest.mark.gpu
TOL = 1e-4
# The PointNet heads are nine random, BatchNorm-calibrated layers in a row: they amplify a relative perturbation of their
# input ~50x (measured on the oracle: 1e-6 on the landmarks -> 4.8e-5 on point_residual), and the reference's own fp32 result
# moves by 5e-6 when the same layers run in float64.  The split-fp16 GEMMs carry 22-bit operands (8x fp32's unit
# round-off), so ~1e-4 on point_residual / the regressed parameters is the expected figure; the REFINED LANDMARKS
# (lmk + 0.05 * residual), which is what the path outputs, stay at ~1e-7.
HEAD_TOL = 3e-4
LOSS_KEYS = ('loss_LMK_f0', 'loss_LMK_pointNet', 'loss_Param_In', 'loss_Param_S2', 'loss_Param_S1S2')


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
def model(synth_pack, sd):
    from synergynet_b200 import model_building
    m = model_building.SynergyNet(types.SimpleNamespace(arch='mobilenet_v2', img_size=120, devices_id=[0]))
    m.load_state_dict(sd, strict=True)
    return m.eval()


def test_forward_matches_reference_losses(model, gold):
    x = synthetic.normalize_crops(torch.from_numpy(gold['x_u8'])).cuda()
    eng = model._engine(torch.device('cuda', 0))
    n0 = eng.launch_count
    loss = model(x, torch.from_numpy(gold['fwd_target']).cuda())
    torch.cuda.synchronize()
    assert eng.launch_count - n0 > 40                                    # backbone + 2 reconstructions + heads + losses
    assert set(loss.keys()) == set(LOSS_KEYS) == set(model.get_losses())
    for k in LOSS_KEYS:
        got = loss[k].cpu().numpy()
        assert got.shape == gold['fwd_' + k].shape, k
        err = rp.max_rel_err(got, gold['fwd_' + k])
        print(f'{k}: rel err {err:.2e}')
        assert err < HEAD_TOL, k
    t = model.last_forward
    assert rp.max_rel_err(t['point_residual'].cpu().numpy(), gold['fwd_point_residual']) < HEAD_TOL
    assert rp.max_rel_err(t['vertex_lmk_refined'].cpu().numpy(), gold['fwd_vertex_lmk_refined']) < 1e-5
    assert rp.max_rel_err(t['_3D_attr_S2'].cpu().numpy(), gold['fwd_3D_attr_S2']) < HEAD_TOL
    eng.raise_if_error()


def test_heads_as_modules_match_oracle_on_other_inputs(model, sd, basis):
    """forwardDirection / reverseDirection called like the reference calls them (model_building.py:149,153), on a
    batch that is not a multiple of the GEMM tile (37 faces x 68 points = 2516 rows)."""
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(37, seed=71))
    attr, pool = rp.mobilenetv2_forward(sd, x)
    lmk = torch.from_numpy(rp.reconstruct_vertex_62(attr.numpy(), basis))
    want_res = rp.mlp_for_forward(sd, lmk, pool, attr[:, 12:52], attr[:, 52:62])
    got_res = model.forwardDirection(lmk.cuda(), pool.cuda(), attr[:, 12:52].cuda(), attr[:, 52:62].cuda())
    assert got_res.shape == (37, 3, 68) and got_res.is_cuda
    assert rp.max_rel_err(got_res.cpu().numpy(), want_res.numpy()) < HEAD_TOL
    refined = lmk + 0.05 * want_res
    want_rev = rp.mlp_rev_forward(sd, refined)
    got_rev = model.reverseDirection(refined.cuda())
    assert got_rev.shape == (37, 62)
    assert rp.max_rel_err(got_rev.cpu().numpy(), want_rev.numpy()) < HEAD_TOL
    # single face and CPU tensors in -> CPU tensors out
    one = model.reverseDirection(refined[:1])
    assert not one.is_cuda and rp.max_rel_err(one.numpy(), want_rev[:1].numpy()) < HEAD_TOL


def test_losses_edge_cases(model):
    eng = model._engine(torch.device('cuda', 0))
    g = torch.Generator().manual_seed(9)
    a = torch.rand((5, 3, 68), generator=g) * 120
    b = a.clone()
    b[0, 0, 0] += 25.0                                                   # one coordinate in the linear branch (>= omega)
    b[1] += 0.5
    want = rp.wing_loss(a, b)
    assert abs(float(eng.wing_loss(a.cuda(), b.cuda()).cpu()) / float(want) - 1) < 1e-5
    assert float(eng.wing_loss(a.cuda(), a.cuda()).cpu()) == 0.0
    p, q = torch.randn((7, 62), generator=g), torch.randn((7, 62), generator=g)
    for mode in ('normal', 'only_3dmm'):
        assert rp.max_rel_err(eng.param_loss(p.cuda(), q.cuda(), mode=mode).cpu().numpy(), rp.param_loss(p, q, mode).numpy()) < 1e-6
    with pytest.raises(RuntimeError):
        eng.param_loss(p.cuda(), q.cuda(), mode='bogus')


def test_large_activations_do_not_saturate_the_heads(model, sd, basis):
    """The GEMM layers scale every row by its own power of two, so inputs far beyond the fixed-scale limit of the
    backbone engines (|x| ~ 937) stay exact: landmarks scaled 50x (values up to ~6000) through MLP_rev."""
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(4, seed=3))
    attr, _ = rp.mobilenetv2_forward(sd, x)
    lmk = torch.from_numpy(rp.reconstruct_vertex_62(attr.numpy(), basis)) * 50.0
    want = rp.mlp_rev_forward(sd, lmk)
    got = model.reverseDirection(lmk.cuda()).cpu()
    assert rp.max_rel_err(got.numpy(), want.numpy()) < HEAD_TOL


# ---- SURVEY.md section 8 f1: batched device pre/post-processing around the path ---------------------------------------

def test_pose_decode_matches_reference_numpy_path(model, gold):
    """parse_pose + predict_pose (utils/inference.py) on the device, against the reference's own numbers."""
    from synergynet_b200 import inference
    eng = model._engine(torch.device('cuda', 0))
    roi = [30.2, 41.7, 211.4, 222.9, 0.99]
    p0 = torch.from_numpy(gold['params'][:1]).cuda()
    ang, t3d = eng.pose_decode(p0, torch.from_numpy(inference.roi_affine([roi])).cuda())
    assert ang.dtype == torch.float64 and tuple(ang.shape) == (1, 3) and tuple(t3d.shape) == (1, 3)
    assert np.allclose(ang.cpu().numpy()[0], gold['np_pose_angles'], rtol=0, atol=1e-4)       # degrees
    assert np.allclose(t3d.cpu().numpy()[0].astype(np.float64), gold['np_pose_t3d'], rtol=1e-6, atol=1e-5)
    # batch of 8 against the oracle, crop coordinates (no box)
    p8 = torch.from_numpy(gold['params']).cuda()
    ang8, t8 = eng.pose_decode(p8)
    pack = rp.gather_sparse_basis(synthetic.make_3dmm(0))
    for i in range(8):
        a_ref, t_ref = rp.predict_pose(gold['params'][i], pack, [0.0, 0.0, 120.0, 120.0])
        assert np.allclose(ang8[i].cpu().numpy(), a_ref, atol=1e-4)
        assert np.allclose(t8[i].cpu().numpy(), t_ref, rtol=1e-6, atol=1e-5)


def test_reconstruct_image_equals_reference_rescale(model, gold, basis):
    from synergynet_b200 import inference
    eng = model._engine(torch.device('cuda', 0))
    boxes = [[30.2, 41.7, 211.4, 222.9, 0.99], [-10.5, 3.25, 95.0, 108.75, 0.5], [400.0, 300.0, 520.0, 420.0, 1.0]]
    p = torch.from_numpy(gold['params'][:3]).cuda()
    roi5 = torch.from_numpy(inference.roi_affine(boxes)).cuda()
    for dense in (False, True):
        got = eng.reconstruct_image(p, roi5, dense=dense).cpu().numpy()
        crop = model.reconstruct_vertex_62(p, dense=dense).cpu().numpy()
        for i, b in enumerate(boxes):
            want = rp.rescale_to_image(crop[i], b)                        # numpy arithmetic of utils/inference.py:127-138
            assert np.array_equal(got[i], want.astype(np.float32)), (dense, i)   # same fp32 operations in the same order
    assert rp.max_rel_err(eng.reconstruct_image(p[:1], roi5[:1]).cpu().numpy()[0], gold['np_sparse']) < TOL


def test_center_crop_border_on_uint8_loader(model):
    """CenterCrop(5, mode='test') + Normalize of benchmark.py:116 == uint8 entry point with a 5-pixel zero frame."""
    eng = model._engine(torch.device('cuda', 0))
    u8 = synthetic.make_structured_crops_u8(9, seed=14)
    framed = torch.zeros_like(u8)
    framed[:, :, 5:115, 5:115] = u8[:, :, 5:115, 5:115]                   # utils/ddfa.py:230-238 on the raw pixel values
    want = eng.forward_landmarks(synthetic.normalize_crops(framed).cuda())
    try:
        eng.set_center_crop(5)
        got = eng.forward_landmarks(u8.cuda())
        host = eng.forward_landmarks_host(u8.pin_memory())
    finally:
        eng.set_center_crop(0)
    assert torch.equal(got, want) and torch.equal(host, want.cpu())
    assert not torch.equal(eng.forward_landmarks(u8.cuda()), want)


# ---- SURVEY.md section 8 a11: ResNet-50 backbone variant (BASELINE.json configs[4]) ---------------------------------

@pytest.fixture(scope='module')
def resnet_model(synth_pack):
    from synergynet_b200 import model_building
    m = model_building.SynergyNet(types.SimpleNamespace(arch='resnet50', img_size=120, devices_id=[0]))
    rsd = synth_model.build_resnet50_state_dict(0)
    missing = m.load_state_dict({'I2P.backbone.' + k: v for k, v in rsd.items()}, strict=False)
    assert not missing.unexpected_keys and all(not k.startswith('I2P.') for k in missing.missing_keys)
    return m.eval()


def test_resnet50_matches_reference_module(resnet_model, gold, basis):
    x = synthetic.normalize_crops(torch.from_numpy(gold['x_u8']))[:4].cuda()
    eng = resnet_model._engine(torch.device('cuda', 0))
    n0 = eng.launch_count
    out, pool = eng.forward_resnet50(x)
    torch.cuda.synchronize()
    assert eng.launch_count - n0 == 2 + 52 + 2                           # stem, max-pool, 52 GEMM convs, avg-pool, heads
    assert out.shape == (4, 102) and pool.shape == (4, 2048)
    err = rp.max_rel_err(out.cpu().numpy(), gold['resnet50_out102'])
    print(f'resnet50 out102 rel err vs the reference module {err:.2e}')
    assert err < TOL
    # the (param62, avgpool) adapter and the landmark path behind it
    params = resnet_model.forward_test(x)
    assert torch.equal(params, out[:, :62])
    # landmarks behind the adapter: the random ResNet emits |params| ~ 200, i.e. 3DMM coefficients hundreds of sigmas out,
    # and the reconstruction amplifies a 5e-5 difference in them past 1e-4 of the (meaningless) landmark range -- so
    # the reconstruction is held to the reference on the reference's own parameters
    ref_params = torch.from_numpy(np.ascontiguousarray(gold['resnet50_out102'][:, :62])).cuda()
    lmk = resnet_model.reconstruct_vertex_62(ref_params)
    assert rp.max_rel_err(lmk.cpu().numpy(), gold['resnet50_lmk']) < TOL
    p2, feat = resnet_model.I2P.forward_test(x)
    assert torch.equal(p2, params) and torch.equal(feat, pool)
    with pytest.raises(RuntimeError, match='1280-d image feature'):
        resnet_model(x, params)
    eng.raise_if_error()


def test_resnet50_ragged_batch_and_oracle(resnet_model):
    sd = {'I2P.backbone.' + k: v for k, v in synth_model.build_resnet50_state_dict(0).items()}
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(5, seed=33))
    want, pooled = rp.resnet50_forward(sd, x)
    eng = resnet_model._engine(torch.device('cuda', 0))
    got, gp = eng.forward_resnet50(x.cuda())
    assert rp.max_rel_err(got.cpu().numpy(), want.numpy()) < TOL
    assert rp.max_rel_err(gp.cpu().numpy(), pooled.numpy()) < TOL
    one, _ = eng.forward_resnet50(x[2:3].cuda())
    assert rp.max_rel_err(one.cpu().numpy(), got[2:3].cpu().numpy()) < 1e-6
