#!/usr/bin/env python
"""Tiny pass over every kernel family for `compute-sanitizer --tool memcheck` (B200 only; batches of 1-3 faces)."""
import os
import sys
import types

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import resnest_port, synth_model  # noqa: E402
from synergynet_b200 import inference, model_building, synthetic  # noqa: E402
from synergynet_b200.params import ParamsPack, set_param_pack  # noqa: E402


def main():
    set_param_pack(ParamsPack(arrays=synthetic.make_3dmm(seed=0)))
    sd = synth_model.build_state_dict(0)
    m = model_building.SynergyNet(types.SimpleNamespace(arch='mobilenet_v2', img_size=120, devices_id=[0]))
    m.load_state_dict(sd, strict=True)
    m.eval()
    dev = torch.device('cuda', 0)
    eng = m._engine(dev)
    u8 = synthetic.make_structured_crops_u8(3, seed=1)
    x = synthetic.normalize_crops(u8).cuda()
    for kind in (2, 0, 1, 3):
        m.set_engine(kind)
        lmk, params = eng.forward_landmarks(x, want_params=True)
        torch.cuda.synchronize()
    m.set_engine(2)
    eng.forward_landmarks(u8.cuda())
    eng.forward_landmarks_host(u8)
    dense = eng.reconstruct(params, dense=True)
    eng.reconstruct(params.repeat(24, 1)[:70], dense=True)          # two face tiles, the second one ragged; band edges
    tk = [eng.forward_landmarks_host_submit(u8.pin_memory()) for _ in range(3)]   # third submit waits for the first
    for t in tk:
        eng.host_wait(t)
    roi5 = torch.from_numpy(inference.roi_affine([[1.0, 2.0, 100.0, 110.0]] * 3)).cuda()
    eng.reconstruct_image(params, roi5, dense=True)
    eng.reconstruct_image(params, roi5, dense=False)
    eng.pose_decode(params, roi5)
    loss = m(x, params + 0.1)
    torch.cuda.synchronize()
    rn = model_building.SynergyNet(types.SimpleNamespace(arch='resnet50', img_size=120, devices_id=[0]))
    rn.load_state_dict({'I2P.backbone.' + k: v for k, v in synth_model.build_resnet50_state_dict(0).items()}, strict=False)
    rn.eval()
    rn.forward_test(x[:2])
    torch.cuda.synchronize()
    rs = model_building.SynergyNet(types.SimpleNamespace(arch='resnest50', img_size=120, devices_id=[0]))
    rs.load_state_dict({'I2P.backbone.' + k: v for k, v in resnest_port.build_resnest50_state_dict(0).items()}, strict=False)
    rs.eval()
    rs.forward_test(x[:2])
    torch.cuda.synchronize()
    eng.raise_if_error()
    print('sanitizer smoke done:', float(dense.abs().max()), {k: float(v.mean()) for k, v in loss.items()})


if __name__ == '__main__':
    main()
