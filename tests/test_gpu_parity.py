"""Parity of the sm_100a library against the CPU oracle and the reference's golden vectors.
All calls go through the C ABI (ctypes) via the reference-shaped Python API.  B200 only."""
import types

import numpy as np
import pytest
import torch

from oracle import golden
from oracle import reference_port as rp
from oracle import synth_model
from synergynet_b200 import _lib, synthetic
from synergynet_b200.backbone import conv_plan

pytestmark = pytest.mark.gpu

TOL = 1e-4            # north_star: 1e-4 relative fp32 on params / landmarks / vertices
# Intermediate activations are a diagnostic, not a north_star output: the calibrated synthetic network amplifies fp32
# ordering noise to ~3e-5 per layer already (engine 0 vs the oneDNN oracle); the split-fp16 tensor-core engines measure
# 7.9e-5 at the deepest layers.  DESIGN.md section 2 quotes the bound asserted here.
LAYER_TOL = {0: 1e-4, 1: 1.5e-4, 2: 1.5e-4}
ENGINES = [_lib.ENGINE_SIMT_FP32, _lib.ENGINE_TC_BF16X3, _lib.ENGINE_TC_FUSED]


def _engine_available(model, kind):
    try:
        model.set_engine(kind)
        return True
    except _lib.SynergyLibError as e:
        if e.code == 6:
            return False
        raise


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
    args = types.SimpleNamespace(arch='mobilenet_v2', img_size=120, devices_id=[0])
    m = model_building.SynergyNet(args)
    m.load_state_dict(sd, strict=True)
    m.eval()
    return m


@pytest.fixture(scope='module', params=ENGINES, ids=['simt_fp32', 'tc_bf16x3', 'tc_fused'])
def engine_kind(request, model):
    if not _engine_available(model, request.param):
        pytest.skip('engine not in this build')
    yield request.param
    model.set_engine(_lib.ENGINE_TC_FUSED)


def _x(gold):
    return synthetic.normalize_crops(torch.from_numpy(gold['x_u8']))


def test_native_library_is_what_runs(model):
    assert model.param_mean.is_cuda
    eng = model._engine(torch.device('cuda', 0))
    before = eng.launch_count
    eng.forward(torch.zeros(1, 3, 120, 120, device='cuda'))
    torch.cuda.synchronize()
    assert eng.launch_count - before >= 4
    with open('/proc/self/maps') as f:
        assert 'libsynergy_b200.so' in f.read()


def test_every_conv_layer_matches_oracle(model, sd, gold, engine_kind):
    x = _x(gold)[:3]
    _, _, convs = rp.mobilenetv2_forward(sd, x, return_convs=True)
    eng = model._engine(torch.device('cuda', 0))
    xd = x.cuda()
    worst = 0.0
    for spec in conv_plan():
        try:
            got = eng.debug_forward_until(xd, spec.index).cpu().permute(0, 3, 1, 2).numpy()
        except _lib.SynergyLibError as e:
            assert e.code == 6 and engine_kind == _lib.ENGINE_TC_FUSED      # fused away, never in HBM
            continue
        err = rp.max_rel_err(got, convs[spec.index].numpy())
        worst = max(worst, err)
        assert err < LAYER_TOL[engine_kind], f'conv {spec.index} ({spec.kind}, block {spec.block}): {err:.3e}'
    print(f'worst per-layer rel err {worst:.3e}')
    assert eng.poll_error() == 0


def test_forward_matches_golden_and_oracle(model, sd, gold, engine_kind):
    x = _x(gold)
    params = model.forward_test(x.cuda())
    assert params.shape == (8, 62) and params.is_cuda and params.dtype == torch.float32
    p_ref, pool_ref = rp.mobilenetv2_forward(sd, x)
    got = params.cpu().numpy()
    assert rp.max_rel_err(got, gold['params']) < TOL
    assert rp.max_rel_err(got, p_ref.numpy()) < TOL
    p2, pool = model.I2P.forward_test(x.cuda())
    assert torch.equal(p2, params)
    assert rp.max_rel_err(pool.cpu().numpy(), gold['pool']) < TOL
    lmk = model.reconstruct_vertex_62(params)
    assert lmk.shape == (8, 3, 68)
    assert rp.max_rel_err(lmk.cpu().numpy(), gold['lmk']) < TOL
    assert rp.nme_vs_reference(lmk.cpu().numpy(), gold['lmk']).max() < TOL
    fused = model.forward_landmarks(x.cuda())
    assert torch.equal(fused, lmk)
    print('params err %.3e  lmk err %.3e' % (rp.max_rel_err(got, gold['params']),
                                             rp.max_rel_err(lmk.cpu().numpy(), gold['lmk'])))


def test_reconstruct_flags_and_dense(model, gold, basis, engine_kind):
    p = torch.from_numpy(gold['params']).cuda()
    for whitening in (True, False):
        for transform in (True, False):
            pin = p if whitening else p * model.param_std + model.param_mean
            got = model.reconstruct_vertex_62(pin, whitening=whitening, transform=transform).cpu().numpy()
            want = rp.reconstruct_vertex_62(pin.cpu().numpy(), basis, whitening=whitening, transform=transform)
            assert rp.max_rel_err(got, want) < TOL
    dense = model.reconstruct_vertex_62(p[:3], dense=True)
    assert dense.shape == (3, 3, synthetic.NVER) and dense.is_contiguous()
    d = dense.cpu().numpy()
    assert rp.max_rel_err(d[:, :, ::53], gold['dense_sub']) < TOL
    assert rp.max_rel_err(d[:, :, basis['keypoints'][::3] // 3], gold['dense_kp']) < TOL
    assert np.allclose(d.astype(np.float64).sum(2), gold['dense_sum64'], rtol=1e-4, atol=50.0)
    want = rp.reconstruct_vertex_62(gold['params'][:3], basis, dense=True)
    assert rp.max_rel_err(d, want) < TOL


def test_dense_keypoint_columns_equal_sparse_bit_exact(model, gold, basis, engine_kind):
    p = torch.from_numpy(gold['params']).cuda()
    sparse = model.reconstruct_vertex_62(p)
    dense = model.reconstruct_vertex_62(p, dense=True)
    kp = torch.from_numpy(basis['keypoints'][::3] // 3).cuda()
    assert torch.equal(dense[:, :, kp], sparse)          # SURVEY.md section 4 invariant


def test_length_mismatch_raises(model):
    with pytest.raises(RuntimeError, match='length of params mismatch'):
        model.reconstruct_vertex_62(torch.zeros(2, 61, device='cuda'))
    with pytest.raises(RuntimeError, match=r'\(B,3,120,120\)'):
        model.forward_test(torch.zeros(2, 3, 64, 64, device='cuda'))


@pytest.mark.parametrize('batch', [1, 7, 33])
def test_ragged_batches_agree_with_single_face_calls(model, sd, engine_kind, batch):
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(batch, seed=50 + batch))
    got = model.forward_test(x.cuda()).cpu()
    want, _ = rp.mobilenetv2_forward(sd, x)
    assert rp.max_rel_err(got.numpy(), want.numpy()) < TOL
    single = torch.cat([model.forward_test(x[i:i + 1].cuda()).cpu() for i in range(min(batch, 3))])
    assert rp.max_rel_err(single.numpy(), got[:single.shape[0]].numpy()) < 1e-6


def test_full_size_batch_properties(model, sd, gold, basis, engine_kind):
    """BASELINE.json config 2/3 sizes: B=1024 is too slow for the CPU oracle end to end, so use
    size-independent properties: every row of a tiled batch reproduces the small-batch row, dense
    keypoint columns equal the sparse landmarks, reconstruction is affine in the pose offset."""
    x8 = _x(gold)
    ref8 = model.forward_test(x8.cuda())
    big = x8.repeat(128, 1, 1, 1).cuda()
    assert big.shape[0] == 1024
    lmk, params = model._engine(big.device).forward_landmarks(big, want_params=True)
    assert rp.max_rel_err(params.view(128, 8, 62).cpu().numpy(),
                          ref8.cpu().numpy()[None].repeat(128, 0)) < 1e-6
    assert rp.max_rel_err(lmk[:8].cpu().numpy(), gold['lmk']) < TOL
    # 1024 DISTINCT faces end to end against the values the reference itself produced for them (make_golden.py)
    xs = synthetic.normalize_crops(synthetic.make_structured_crops_u8(1024, seed=77))
    l_big, p_dev = model._engine(big.device).forward_landmarks(xs.cuda(), want_params=True)
    p_big = p_dev.cpu()
    assert rp.max_rel_err(p_big.numpy(), gold['params1024']) < TOL
    # landmarks: every face against the oracle's reconstruction of the reference's parameters (held to the reference's
    # landmarks by test_oracle_golden.py), the even-numbered faces against the reference's own landmarks
    l_np = l_big.cpu().numpy()
    for got, want in ((l_np, rp.reconstruct_vertex_62(gold['params1024'], basis)), (l_np[::2], gold['lmk1024_even'])):
        assert rp.max_rel_err(got, want) < TOL
        assert rp.nme_vs_reference(got, want).max() < TOL
    idx = torch.arange(0, 1024, 43)
    want, _ = rp.mobilenetv2_forward(sd, xs[idx])
    assert rp.max_rel_err(p_big[idx].numpy(), want.numpy()) < TOL
    dense = model.reconstruct_vertex_62(p_big.cuda(), dense=True)
    assert dense.shape == (1024, 3, synthetic.NVER)
    kp = torch.from_numpy(basis['keypoints'][::3] // 3).cuda()
    assert torch.equal(dense[:, :, kp], model.reconstruct_vertex_62(p_big.cuda()))
    want_d = rp.reconstruct_vertex_62(p_big[idx[:4]].numpy(), basis, dense=True)
    assert rp.max_rel_err(dense[idx[:4]].cpu().numpy(), want_d) < TOL
    # affine in the translation parameters (whitening off): shifting t by d shifts x,z by d, y by -d
    raw = (p_big[:64].cuda() * model.param_std + model.param_mean)
    shifted = raw.clone()
    shifted[:, [3, 7, 11]] += torch.tensor([2.0, 3.0, 4.0], device='cuda')
    a = model.reconstruct_vertex_62(raw, whitening=False)
    b = model.reconstruct_vertex_62(shifted, whitening=False)
    delta = (b - a).cpu().numpy()
    assert np.allclose(delta[:, 0], 2.0, atol=2e-3) and np.allclose(delta[:, 1], -3.0, atol=2e-3)
    assert np.allclose(delta[:, 2], 4.0, atol=2e-3)


def test_host_buffer_call_matches_device_call(model, gold, engine_kind):
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(300, seed=5))
    eng = model._engine(torch.device('cuda', 0))
    want = eng.forward_landmarks(x.cuda()).cpu()
    pinned = x.pin_memory()
    out = torch.empty((300, 3, 68), dtype=torch.float32).pin_memory()
    par = torch.empty((300, 62), dtype=torch.float32).pin_memory()
    got = eng.forward_landmarks_host(pinned, out, par)
    assert torch.equal(got, want)
    got2 = eng.forward_landmarks_host(x)                  # pageable memory also works
    assert torch.equal(got2, want)
    assert rp.max_rel_err(par.numpy(), model.forward_test(x.cuda()).cpu().numpy()) < 1e-6


def test_pipelined_host_calls_match_blocking_calls(model, engine_kind):
    """submit / wait with two calls in flight (the loader-loop form of the host call): every ticket returns exactly what
    the blocking call returns for its batch, whatever the interleaving, batch sizes and input types; a stream-ordered
    call in between sees a consistent workspace; a ticket cannot be collected twice."""
    eng = model._engine(torch.device('cuda', 0))
    batches = [synthetic.normalize_crops(synthetic.make_structured_crops_u8(n, seed=40 + i)).pin_memory()
               for i, n in enumerate((600, 130, 1024, 7))]
    batches.append(synthetic.make_structured_crops_u8(257, seed=77).pin_memory())          # uint8 batch in the mix
    want = [eng.forward_landmarks_host(b).clone() for b in batches]
    outs = [torch.empty((b.shape[0], 3, 68), dtype=torch.float32).pin_memory() for b in batches]
    pars = [torch.empty((b.shape[0], 62), dtype=torch.float32).pin_memory() for b in batches]
    prev = None
    for i, b in enumerate(batches):
        tk = eng.forward_landmarks_host_submit(b, outs[i], pars[i])
        if prev is not None:
            got = eng.host_wait(prev[0])
            assert got is outs[prev[1]] and torch.equal(got, want[prev[1]])
        prev = (tk, i)
    mid = eng.forward_landmarks(batches[1].cuda()).cpu()          # stream call while the last ticket is still open
    assert torch.equal(mid, want[1])
    assert torch.equal(eng.host_wait(prev[0]), want[prev[1]])
    with pytest.raises(RuntimeError):
        eng.host_wait(prev[0])
    for i, b in enumerate(batches):
        x = b.cuda() if b.dtype == torch.float32 else synthetic.normalize_crops(b).cuda()
        assert rp.max_rel_err(pars[i].numpy(), model.forward_test(x).cpu().numpy()) < 1e-6
    three = [eng.forward_landmarks_host_submit(batches[i], outs[i]) for i in (0, 1, 3)]   # third submit waits for the first
    for tk, i in zip(three, (0, 1, 3)):
        assert torch.equal(eng.host_wait(tk), want[i])
    assert eng.poll_error() == 0


def test_uint8_crops_match_host_normalised_floats(model, engine_kind):
    """`(img - 127.5) / 128` applied on the device (uint8 entry points) is the same fp32 arithmetic as
    the reference's host-side normalisation (synergy3DMM.py:192): outputs must be bit-identical."""
    u8 = synthetic.make_structured_crops_u8(70, seed=9)
    eng = model._engine(torch.device('cuda', 0))
    want = eng.forward_landmarks(synthetic.normalize_crops(u8).cuda())
    got = eng.forward_landmarks(u8.cuda())
    assert torch.equal(got, want)
    host = eng.forward_landmarks_host(u8.pin_memory())
    assert torch.equal(host, want.cpu())
    assert eng.poll_error() == 0


def test_get_all_outputs_matches_reference_api(model, gold, engine_kind):
    rects = [list(r) for r in gold['scene_rects']]
    pts, verts, poses = model.get_all_outputs(gold['scene'].copy(), rects=rects)
    assert len(pts) == len(verts) == len(poses) == 2
    assert pts[0].shape == (3, 68) and verts[0].shape == (3, synthetic.NVER)
    assert rp.max_rel_err(np.stack(pts), gold['scene_lmk']) < TOL
    assert rp.max_rel_err(np.stack([v[:, ::53] for v in verts]), gold['scene_dense_sub']) < TOL
    assert np.allclose([p[0] for p in poses], gold['scene_angles'], atol=2e-2)
    assert np.allclose([p[1] for p in poses], gold['scene_t3d'], rtol=1e-4, atol=1e-3)
    model.face_detector = lambda img: rects
    pts2, _, _ = model.get_all_outputs(gold['scene'].copy())
    assert np.array_equal(np.stack(pts2), np.stack(pts))
    model.face_detector = None
    with pytest.raises(RuntimeError, match='no face detector'):
        model.get_all_outputs(gold['scene'])


def test_per_launch_timing_api(model):
    eng = model._engine(torch.device('cuda', 0))
    model.set_engine(_lib.ENGINE_TC_FUSED)
    x = synthetic.make_inputs(16, 0).cuda()
    eng.set_timing(True)
    eng.forward_landmarks(x)
    t = eng.timings()
    eng.set_timing(False)
    names = [n for n, _ in t]
    assert names[0] == 'fused_stem_block1' and 'tail_conv_pool_kernel' in names and names[-1] == 'dense_recon_tc_kernel'
    assert len(t) == 21 and all(ms > 0 for _, ms in t)


def test_reload_of_weights_is_picked_up(model, sd, gold):
    x = _x(gold)[:2].cuda()
    before = model.forward_test(x)
    key = 'I2P.backbone.classifier_ori.1.bias'
    bumped = {k: v.clone() for k, v in sd.items()}
    bumped[key] += 1.0
    model.load_state_dict(bumped, strict=True)
    after = model.forward_test(x)
    assert torch.allclose(after[:, :12], before[:, :12] + 1.0, atol=1e-5)
    assert torch.equal(after[:, 12:], before[:, 12:])
    model.load_state_dict(sd, strict=True)
    assert torch.equal(model.forward_test(x), before)
