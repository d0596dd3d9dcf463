#!/usr/bin/env python
"""Generate ``tests/golden/resnest_vectors.npz`` by running the UNMODIFIED reference ``resnest50()``.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden_resnest.py

It takes a scratch copy of the reference exactly as ``make_golden.py`` does, builds ``backbone_nets.ResNeSt.resnest50()``
(the backbone the reference's I2P builds for any arch containing 'resnest', model_building.py:48-49), loads the seeded,
calibrated synthetic state dict with ``strict=True`` (so the 482-key schema is checked on the way) and records, for 8
seeded crops, what ``I2P.forward_test`` would return -- (out62, avgpool) -- plus subsampled stage outputs and the
landmarks the reference's ``reconstruct_vertex_62`` makes of its own out62.  Only numbers are stored.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import make_golden  # noqa: E402  (puts the repository root on sys.path; scratch copy of the reference)

from synergynet_b200 import synthetic  # noqa: E402
from oracle import golden  # noqa: E402
from oracle import resnest_port  # noqa: E402

CH_STRIDE = 8


def main():
    torch.manual_seed(0)
    sd = resnest_port.build_resnest50_state_dict(0)
    make_golden.synth_model.build_state_dict(0)            # installs the synthetic 3DMM pack the landmarks use
    make_golden.scratch_reference()
    import synergy3DMM as ref_api                          # the reference modules, unmodified
    from backbone_nets.ResNeSt import resnest50
    net = resnest50()
    res = net.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    net.eval()
    inputs = resnest_port.resnest_inputs()
    x = synthetic.normalize_crops(torch.from_numpy(inputs['x_u8']))
    stages = []
    hooks = [getattr(net, f'layer{i}').register_forward_hook(lambda _m, _i, o: stages.append(o.detach().clone()))
             for i in range(1, 5)]
    with torch.no_grad():
        out62, pool = net(x)
    for h in hooks:
        h.remove()
    ref = ref_api.SynergyNet()
    with torch.no_grad():
        lmk = ref.reconstruct_vertex_62(out62, dense=False)
    out = {'keys': np.array(list(sd.keys())),
           'key_shapes': np.array(['x'.join(str(d) for d in v.shape) for v in sd.values()]),
           'out62': out62.numpy(), 'pool2048': pool.numpy(), 'lmk': lmk.numpy()}
    strides = []
    for i, f in enumerate(stages, 1):
        s = max(1, f.shape[2] // 10)
        strides.append(s)
        out[f'stage{i}_sub'] = f[0, ::CH_STRIDE, ::s, ::s].numpy()
    out['stage_stride'] = np.array(strides, np.int32)
    out.update({k + '_sha256': np.array(golden.sha256(v)) for k, v in inputs.items()})
    out['meta'] = np.array([f'torch={torch.__version__}', f'numpy={np.__version__}',
                            'reference=choyingw/SynergyNet@9de11e2', 'seed=0', f'channel_stride={CH_STRIDE}'])
    dst = os.path.join(make_golden.ROOT, 'tests', 'golden', 'resnest_vectors.npz')
    np.savez_compressed(dst, **out)
    spread = float((out62 - out62.mean(0)).abs().max())
    print('wrote', dst, os.path.getsize(dst) // 1024, 'KiB;', len(out), 'arrays; out62 |max|', float(out62.abs().max()),
          'face spread', spread)


if __name__ == '__main__':
    main()
