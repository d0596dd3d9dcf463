"""The drop-in boundary, exercised the way the reference's own scripts drive it (SURVEY.md section 8(b)):
benchmark.py:111-132 (DataParallel wrap + `module.`-prefixed checkpoint + `model.module.forward_test`) followed by
benchmark.py:76-97 (`reconstruct_vertex(param, model.module.data_param)`), singleImage.py:28-37 (state-dict
merge), the no-argument CPU-constructed wrapper of synergy3DMM.py:71-114, plus the error / saturation flags and
the single-pass engine.  B200 only."""
import threading
import types
import warnings

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import golden
from oracle import reference_port as rp
from oracle import synth_model
from synergynet_b200 import _lib, synthetic

pytestmark = pytest.mark.gpu
TOL = 1e-4


@pytest.fixture(scope='module')
def sd():
    return synth_model.build_state_dict(0)


@pytest.fixture(scope='module')
def basis():
    return rp.gather_sparse_basis(synthetic.make_3dmm(0))


def _args():
    return types.SimpleNamespace(arch='mobilenet_v2', img_size=120, devices_id=[0])


def _torch_reconstruct_vertex(param, data_param, std_size=120):
    """What benchmark.py:76-97 does with `model.module.data_param`: plain torch ops on the model's buffers."""
    param_mean, param_std, w_shp_base, u_base, w_exp_base = data_param
    param = param * param_std[:62] + param_mean[:62]
    cam = param[:, :12].reshape(-1, 3, 4)
    shape = u_base + w_shp_base @ param[:, 12:52].reshape(-1, 40, 1) + w_exp_base @ param[:, 52:62].reshape(-1, 10, 1)
    vertex = cam[:, :, :3] @ shape.contiguous().view(-1, 68, 3).transpose(1, 2) + cam[:, :, -1].reshape(-1, 3, 1)
    vertex[:, 1, :] = std_size + 1 - vertex[:, 1, :]
    return vertex


def test_benchmark_py_caller_sequence(synth_pack, sd, basis):
    """benchmark.py:111-132 then :153-166, line for line against the shim."""
    from synergynet_b200 import model_building
    checkpoint = {'module.' + k: v.clone() for k, v in sd.items()}         # trained under DataParallel
    device_ids = [0]
    torch.cuda.set_device(device_ids[0])
    model = model_building.SynergyNet(_args())
    model = nn.DataParallel(model, device_ids=device_ids).cuda()
    missing = model.load_state_dict(checkpoint, strict=False)
    assert not missing.missing_keys and not missing.unexpected_keys
    model.eval()
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(12, seed=21))
    with torch.no_grad():
        inputs = x.cuda()
        output = model.module.forward_test(inputs)
    assert output.shape == (12, 62) and output.is_cuda
    want, _ = rp.mobilenetv2_forward(sd, x)
    assert rp.max_rel_err(output.cpu().numpy(), want.numpy()) < TOL
    # per-row host extraction exactly like the loop of benchmark.py:128-131
    rows = np.array([output[i].cpu().numpy().flatten() for i in range(output.shape[0])], dtype=np.float32)
    assert rows.shape == (12, 62)
    # the reference's own reconstruct_vertex consumes data_param: tensors on the model's device, reference shapes
    dp = model.module.data_param
    assert [tuple(t.shape) for t in dp] == [(62,), (62,), (204, 40), (204, 1), (204, 10)] and all(t.is_cuda for t in dp)
    lmk_torch = _torch_reconstruct_vertex(output, dp)
    lmk_lib = model.module.reconstruct_vertex_62(output)
    assert rp.max_rel_err(lmk_lib.cpu().numpy(), lmk_torch.cpu().numpy()) < TOL
    assert rp.max_rel_err(lmk_lib.cpu().numpy(), rp.reconstruct_vertex_62(want.numpy(), basis)) < TOL
    # DataParallel.forward over replicas is the training path; forward_test on .module is what the script calls.
    # A second model on the same device gets its own engine state (no shared workspace between modules).
    other = model_building.SynergyNet(_args())
    other.load_state_dict(sd, strict=True)
    assert torch.equal(other.eval().forward_test(inputs), output)


def test_single_image_py_state_dict_merge(synth_pack, sd):
    """singleImage.py:28-37: build on the default device, merge a `module.`-prefixed checkpoint into state_dict(),
    load with strict=False, then .cuda().eval()."""
    from synergynet_b200 import model_building
    checkpoint = {'module.' + k: v.clone() for k, v in sd.items()}
    model = model_building.SynergyNet(_args())
    model_dict = model.state_dict()
    assert len(model_dict) == 445
    for k in checkpoint.keys():
        model_dict[k.replace('module.', '')] = checkpoint[k]
    model.load_state_dict(model_dict, strict=False)
    model = model.cuda()
    model.eval()
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(3, seed=4))
    want, _ = rp.mobilenetv2_forward(sd, x)
    assert rp.max_rel_err(model.forward_test(x.cuda()).cpu().numpy(), want.numpy()) < TOL


def test_cpu_constructed_wrapper_runs_like_the_reference(synth_pack, sd, basis):
    """synergy3DMM.SynergyNet() is constructed on the CPU and used without .cuda() (synergy3DMM.py:71-114,167-207):
    CPU tensors in -> the library runs on the current GPU -> CPU tensors out."""
    from synergynet_b200 import synergy3DMM
    model = synergy3DMM.SynergyNet()
    model.load_state_dict(sd, strict=True)
    assert not model.param_mean.is_cuda
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(4, seed=8))
    params = model.forward_test(x)
    assert not params.is_cuda and params.shape == (4, 62)
    want, _ = rp.mobilenetv2_forward(sd, x)
    assert rp.max_rel_err(params.numpy(), want.numpy()) < TOL
    lmk = model.reconstruct_vertex_62(params)
    assert not lmk.is_cuda
    assert rp.max_rel_err(lmk.numpy(), rp.reconstruct_vertex_62(want.numpy(), basis)) < TOL
    gold = golden.load_ref_vectors()
    rects = [list(r) for r in gold['scene_rects']]
    pts, verts, poses = model.get_all_outputs(gold['scene'].copy(), rects=rects)
    assert rp.max_rel_err(np.stack(pts), gold['scene_lmk']) < TOL
    assert len(verts) == 2 and len(poses) == 2


def test_single_pass_engine_reports_its_error(synth_pack, sd, basis):
    """Engine 3 (one fp16 MMA per product): same shapes / index work, measured error above the parity bar of the
    default engine but far below garbage; never the default."""
    from synergynet_b200 import model_building
    model = model_building.SynergyNet(_args())
    model.load_state_dict(sd, strict=True)
    model.eval()
    eng = model._engine(torch.device('cuda', 0))
    assert eng.engine == _lib.ENGINE_TC_FUSED
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(40, seed=31)).cuda()
    ref = model.forward_test(x)
    model.set_engine(_lib.ENGINE_TC_FUSED_1PASS)
    assert eng.engine == _lib.ENGINE_TC_FUSED_1PASS
    got = model.forward_test(x)
    lmk = model.reconstruct_vertex_62(got)
    dense = model.reconstruct_vertex_62(got[:2], dense=True)
    kp = torch.from_numpy(basis['keypoints'][::3] // 3).cuda()
    assert torch.equal(dense[:, :, kp], lmk[:2])                       # index work is engine independent
    err = rp.max_rel_err(got.cpu().numpy(), ref.cpu().numpy())
    print(f'single-pass fp16 engine: params rel err vs split-3 engine {err:.3e}')
    assert 1e-6 < err < 2e-2
    model.set_engine(_lib.ENGINE_TC_FUSED)
    assert torch.equal(model.forward_test(x), ref)
    assert eng.poll_error() == 0


def test_saturation_flag_is_raised_for_out_of_range_activations(synth_pack, sd):
    """The split-fp16 engines clamp block inputs beyond |x| ~ 937; a checkpoint that produces them must not pass
    silently: the flag is raised (and the fp32 engine is unaffected)."""
    from synergynet_b200 import model_building
    model = model_building.SynergyNet(_args())
    big = {k: v.clone() for k, v in sd.items()}
    big['I2P.backbone.features.1.conv.2.weight'] *= 4000.0            # BN scale of block 1's projection: huge block-2 input
    big['I2P.backbone.features.1.conv.2.bias'] *= 4000.0
    model.load_state_dict(big, strict=True)
    model.eval()
    eng = model._engine(torch.device('cuda', 0))
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(4, seed=2)).cuda()
    assert eng.poll_saturation(warn=False) == 0
    model.forward_test(x)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        assert eng.poll_saturation() == 1
    assert any('clamped' in str(i.message) for i in w)
    assert eng.poll_saturation(warn=False) == 0                        # cleared by the poll
    model.load_state_dict(sd, strict=True)
    model.forward_test(x)
    assert model._engine(torch.device('cuda', 0)).poll_saturation(warn=False) == 0


def test_engine_is_safe_across_threads_and_streams(synth_pack, sd):
    """One model driven from two host threads and from two CUDA streams: calls are serialised on the handle and
    ordered across streams, so every result equals the single-threaded one."""
    from synergynet_b200 import model_building
    model = model_building.SynergyNet(_args())
    model.load_state_dict(sd, strict=True)
    model.eval()
    xs = [synthetic.normalize_crops(synthetic.make_structured_crops_u8(64, seed=60 + i)).cuda() for i in range(2)]
    want = [model.forward_landmarks(x).clone() for x in xs]
    torch.cuda.synchronize()
    got = [[None] * 8 for _ in range(2)]

    def worker(t):
        torch.cuda.set_device(0)
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            for i in range(8):
                got[t][i] = model.forward_landmarks(xs[t]).clone()
        st.synchronize()

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(2)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    torch.cuda.synchronize()
    for t in range(2):
        for i in range(8):
            assert torch.equal(got[t][i], want[t])
    model._engine(torch.device('cuda', 0)).raise_if_error()


def test_host_call_validates_caller_buffers(synth_pack, sd):
    from synergynet_b200 import model_building
    model = model_building.SynergyNet(_args())
    model.load_state_dict(sd, strict=True)
    eng = model._engine(torch.device('cuda', 0))
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(4, seed=1))
    with pytest.raises(RuntimeError, match='lmk_host'):
        eng.forward_landmarks_host(x, torch.empty((3, 3, 68)))                 # too small
    with pytest.raises(RuntimeError, match='params_host'):
        eng.forward_landmarks_host(x, torch.empty((4, 3, 68)), torch.empty((4, 62), dtype=torch.float64))
    with pytest.raises(RuntimeError, match=r'\(B,3,120,120\)'):
        eng.forward_landmarks_host(torch.zeros(4, 3, 64, 64))
