#!/usr/bin/env python
"""Generate ``tests/golden/ref_vectors.npz`` by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

What it does (SURVEY.md section 8(c) recipe):
  1. copies the reference's Python tree to a scratch directory (the reference resolves
     ``3dmm_data/`` next to its own files and /root/reference is read-only);
  2. writes the seeded synthetic ``3dmm_data/`` (synergynet_b200/synthetic.py);
  3. stubs ``matplotlib`` (not installed) and shims the Cython ``cpu_nms`` (does not build with
     Cython 3 / numpy 2) with the reference's own pure-python NMS;
  4. imports the reference ``synergy3DMM``, loads the seeded calibrated checkpoint with
     ``strict=True`` (so the 445-key schema is checked on the way) and records the reference's
     outputs for fixed inputs.
Nothing from the reference is copied into the repository: only numbers are stored.
"""
import os
import shutil
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
REF = '/root/reference'

from synergynet_b200 import synthetic  # noqa: E402
from oracle import golden  # noqa: E402
from oracle import synth_model  # noqa: E402

DENSE_STRIDE = 53
FEAT_STRIDE = 5


def scratch_reference() -> str:
    tmp = tempfile.mkdtemp(prefix='synergy_ref_')
    dst = os.path.join(tmp, 'ref')
    shutil.copytree(REF, dst, ignore=shutil.ignore_patterns('*.ipynb', 'img', 'demo', '.git'))
    os.system(f'chmod -R u+w {dst}')
    synthetic.write_3dmm_dir(os.path.join(dst, '3dmm_data'), synthetic.make_3dmm(seed=0))
    stubs = os.path.join(tmp, 'stubs', 'matplotlib')
    os.makedirs(stubs)
    open(os.path.join(stubs, '__init__.py'), 'w').close()
    open(os.path.join(stubs, 'pyplot.py'), 'w').close()
    with open(os.path.join(dst, 'FaceBoxes/utils/nms/cpu_nms.py'), 'w') as f:
        f.write('from .py_cpu_nms import py_cpu_nms as cpu_nms\n'
                'def cpu_soft_nms(*a, **k):\n    raise NotImplementedError\n')
    sys.path.insert(0, os.path.join(tmp, 'stubs'))
    sys.path.insert(0, dst)
    os.chdir(dst)
    return dst


def main():
    torch.manual_seed(0)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sd = synth_model.build_state_dict(seed=0)
    scratch_reference()
    import synergy3DMM as ref_api          # the reference module, unmodified
    from utils import inference as ref_inf
    ref = ref_api.SynergyNet()
    missing = ref.load_state_dict(sd, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    ref.eval()
    out = {}

    # ---- batched hot path: forward_test + reconstruct_vertex_62 -------------------------------
    inputs = golden.ref_inputs()                 # stored as SHA-256 only: the tests rebuild them from their seeds
    u8 = torch.from_numpy(inputs['x_u8'])
    x = synthetic.normalize_crops(u8)
    feats = []
    hooks = [m.register_forward_hook(lambda _m, _i, o: feats.append(o.detach().clone()))
             for m in ref.I2P.backbone.features]
    with torch.no_grad():
        params, pool = ref.I2P.forward_test(x)
        params2 = ref.forward_test(x)
    for h in hooks:
        h.remove()
    feats = feats[:19]
    assert torch.equal(params, params2)
    with torch.no_grad():
        lmk = ref.reconstruct_vertex_62(params, dense=False)
        lmk_raw = ref.reconstruct_vertex_62(params, dense=False, transform=False)
        dense = ref.reconstruct_vertex_62(params[:3], dense=True)
    out['params'] = params.numpy()
    out['pool'] = pool.numpy()
    out['lmk'] = lmk.numpy()
    out['lmk_notransform'] = lmk_raw.numpy()
    kp_vert = (ref.keypoints[::3] // 3).numpy()
    out['dense_sub'] = dense[:, :, ::DENSE_STRIDE].numpy()
    out['dense_kp'] = dense[:, :, kp_vert].numpy()
    out['dense_absmax'] = dense.abs().amax(dim=(1, 2)).numpy()
    out['dense_sum64'] = dense.double().sum(dim=2).numpy()
    for i, f in enumerate(feats):                      # NCHW reference activations, face 0
        out[f'feat{i:02d}_sub'] = f[0, :, ::FEAT_STRIDE, ::FEAT_STRIDE].numpy()
        out[f'feat{i:02d}_absmean'] = np.float64(f.abs().double().mean().item())

    # ---- BASELINE.json configs[1] size: 1024 DISTINCT faces through the reference, end to end ----------------------
    x1024 = synthetic.normalize_crops(synthetic.make_structured_crops_u8(1024, seed=77))
    with torch.no_grad():
        p1024 = torch.cat([ref.forward_test(x1024[i:i + 64]) for i in range(0, 1024, 64)])
        l1024 = ref.reconstruct_vertex_62(p1024, dense=False)
    out['params1024'] = p1024.numpy()
    out['lmk1024_even'] = l1024[::2].numpy()           # every other face: keeps the file under 1 MB

    # ---- training-time forward (model_building.py:141-157) through the reference's own modules -------------
    # model_building.SynergyNet needs CUDA at construction; synergy3DMM.SynergyNet owns the same sub-modules
    # (I2P, forwardDirection, reverseDirection, LMKLoss_3D, ParamLoss), so the statements of forward() are executed
    # on them one by one (I2P.forward's `.type(torch.cuda.FloatTensor)` becomes `.float()`), eval-mode BatchNorm.
    g = torch.Generator().manual_seed(3)
    target = params + 0.3 * torch.randn(params.shape, generator=g)
    with torch.no_grad():
        _3D_attr, avgpool = ref.I2P.backbone(x)
        _3D_attr_GT = target.float()
        vertex_lmk = ref.reconstruct_vertex_62(_3D_attr, dense=False)
        vertex_GT_lmk = ref.reconstruct_vertex_62(_3D_attr_GT, dense=False)
        fwd = {'loss_LMK_f0': 0.05 * ref.LMKLoss_3D(vertex_lmk, vertex_GT_lmk, kp=True),
               'loss_Param_In': 0.02 * ref.ParamLoss(_3D_attr, _3D_attr_GT)}
        point_residual = ref.forwardDirection(vertex_lmk, avgpool, _3D_attr[:, 12:52], _3D_attr[:, 52:62])
        vertex_lmk_ref = vertex_lmk + 0.05 * point_residual
        fwd['loss_LMK_pointNet'] = 0.05 * ref.LMKLoss_3D(vertex_lmk_ref, vertex_GT_lmk, kp=True)
        _3D_attr_S2 = ref.reverseDirection(vertex_lmk_ref)
        fwd['loss_Param_S2'] = 0.02 * ref.ParamLoss(_3D_attr_S2, _3D_attr_GT, mode='only_3dmm')
        fwd['loss_Param_S1S2'] = 0.001 * ref.ParamLoss(_3D_attr_S2, _3D_attr, mode='only_3dmm')
    out['fwd_target'] = target.numpy()
    for k, v in fwd.items():
        out['fwd_' + k] = v.numpy()
    out['fwd_point_residual'] = point_residual.numpy()
    out['fwd_vertex_lmk_refined'] = vertex_lmk_ref.numpy()
    out['fwd_3D_attr_S2'] = _3D_attr_S2.numpy()
    assert float(point_residual.abs().max()) > 0.1 and float((_3D_attr_S2 != 0).float().mean()) > 0.2, 'dead PointNet heads'

    # ---- ResNet-50 backbone variant (BASELINE.json configs[4]): the reference module itself ------------------
    from backbone_nets import resnet_backbone as ref_resnet
    rn = ref_resnet.resnet50(pretrained=False)
    rn_sd = synth_model.build_resnet50_state_dict(0)
    res = rn.load_state_dict(rn_sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    rn.eval()
    with torch.no_grad():
        rn_out = rn(x[:4])                                  # (4,102) = ori | shape | exp | tex (resnet_backbone.py:242-246)
        lmk_rn = ref.reconstruct_vertex_62(rn_out[:, :62].contiguous(), dense=False)   # the adapter: first 62 = ori|shape|exp
    out['resnet50_out102'] = rn_out.numpy()
    out['resnet50_lmk'] = lmk_rn.numpy()

    # ---- numpy per-face path (utils/inference.py) and crop_img ------------------------------------
    p0 = params[0].numpy().astype(np.float32)
    roi = [30.2, 41.7, 211.4, 222.9, 0.99]
    out['np_sparse'] = ref_inf.predict_sparseVert(p0, roi, transform=True)
    out['np_dense_sub'] = ref_inf.predict_denseVert(p0, roi, transform=True)[:, ::DENSE_STRIDE]
    ang, t3d = ref_inf.predict_pose(p0, roi)
    out['np_pose_angles'] = np.asarray(ang, np.float64)
    out['np_pose_t3d'] = np.asarray(t3d, np.float64)
    img = inputs['crop_img']
    boxes = np.array([[10.4, 5.5, 60.6, 70.2, 1], [-12.3, -7.8, 40.5, 33.3, 1], [100.2, 60.1, 150.7, 120.9, 1],
                      [-5.5, -5.5, 140.4, 110.6, 1], [20.5, 30.5, 21.4, 31.6, 1]], np.float64)
    out['crop_boxes'] = boxes
    for i, b in enumerate(boxes):
        out[f'crop_out{i}'] = ref_inf.crop_img(img, list(b))

    # ---- get_all_outputs with a stub detector (FaceBoxes itself is out of scope) ------------------
    scene = inputs['scene']
    rects = [[60.3, 80.1, 200.9, 250.4, 0.98], [250.2, -20.0, 372.6, 140.7, 0.91]]

    class _StubDetector:
        def __call__(self, _img):
            return [list(r) for r in rects]

    ref_api.FaceBoxes = _StubDetector
    pts, verts, poses = ref.get_all_outputs(scene.copy())
    out['scene_rects'] = np.asarray(rects, np.float64)
    out['scene_lmk'] = np.stack(pts)
    out['scene_dense_sub'] = np.stack([v[:, ::DENSE_STRIDE] for v in verts])
    out['scene_angles'] = np.asarray([p[0] for p in poses], np.float64)
    out['scene_t3d'] = np.asarray([p[1] for p in poses], np.float64)

    out.update({k + '_sha256': np.array(golden.sha256(v)) for k, v in inputs.items()})
    out['meta'] = np.array([f'torch={torch.__version__}', f'numpy={np.__version__}',
                            'reference=choyingw/SynergyNet@9de11e2', 'seed=0',
                            f'dense_stride={DENSE_STRIDE}', f'feat_stride={FEAT_STRIDE}'])
    dst = os.path.join(ROOT, 'tests', 'golden', 'ref_vectors.npz')
    np.savez_compressed(dst, **out)
    print('wrote', dst, os.path.getsize(dst) // 1024, 'KiB;', len(out), 'arrays')
    print('params[0,:6]', params[0, :6].numpy(), 'lmk range', float(lmk.min()), float(lmk.max()))


if __name__ == '__main__':
    main()
