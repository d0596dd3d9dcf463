#!/usr/bin/env python
"""ResNeSt-50 backbone variant (I2P with arch 'resnest50') on one B200: one JSON line.

    python scripts/bench_resnest.py [--batch 512] [--steps 20] [--warmup 5]  > resnest_bench.json

Reports ms/step, faces/s and the algorithmic TFLOP/s of ``forward_resnest50`` (device-resident fp32 crops; the
activations of a 512-face step are ~0.2 GB per buffer, far beyond the 126 MB L2), the per-kernel-class breakdown of one
step from the library's own per-launch CUDA events (``syn_set_timing``), the same-box comparator -- the oracle's
``torch.nn.functional`` restatement on the GPU through cuDNN, with TF32 off and on -- and the card's name and power
limit read in the same run.  The algorithmic FLOP count comes from the layer plan of the C ABI (2 x MAC of every conv
and Linear at the size it runs at); pools, attention softmax and adds are not counted.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import types
from collections import OrderedDict

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import reference_port as rp  # noqa: E402
from oracle import resnest_port  # noqa: E402
from synergynet_b200 import _lib, model_building, synthetic  # noqa: E402
from synergynet_b200.params import ParamsPack, set_param_pack  # noqa: E402


def plan_macs() -> int:
    lib = _lib.load()
    d = _lib.ResNeStLayerDesc()
    macs = 62 * 2048                                                   # fc_ori | fc_shape | fc_exp
    for i in range(lib.syn_resnest_num_layers()):
        _lib.check(lib.syn_resnest_layer_desc(i, C.byref(d)))
        macs += d.cout * (d.cin // d.groups) * d.ksize * d.ksize * d.h_out * d.h_out
    return macs


def card_info(dev) -> dict:
    info = {'name': torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', str(dev.index), '--query-gpu=name,power.limit,clocks.max.sm',
                            '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [p.strip() for p in q.split(',')]
        info.update(smi_name=name, power_limit_w=float(power), sm_max_mhz=float(clk))
    except Exception as e:                                             # the number still stands with the torch name
        info['smi_error'] = str(e)
    return info


def time_steps(fn, steps: int, warmup: int) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=512)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--no-comparator', action='store_true')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_resnest.py measures the B200 path; no CUDA device is visible')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    set_param_pack(ParamsPack(arrays=synthetic.make_3dmm(seed=0)))
    sd = {'I2P.backbone.' + k: v for k, v in resnest_port.build_resnest50_state_dict(0).items()}
    m = model_building.SynergyNet(types.SimpleNamespace(arch='resnest50', img_size=120, devices_id=[0]))
    m.load_state_dict(sd, strict=False)
    m.eval()
    eng = m._engine(dev)
    B = a.batch
    x = synthetic.normalize_crops(synthetic.make_structured_crops_u8(B, seed=2024)).to(dev)
    macs = plan_macs()
    flop = 2 * macs * B

    n0 = eng.launch_count
    out, pool = eng.forward_resnest50(x)
    torch.cuda.synchronize()
    launches = eng.launch_count - n0
    ms = time_steps(lambda: eng.forward_resnest50(x), a.steps, a.warmup)
    eng.raise_if_error()

    # per-kernel-class breakdown of one step (events after every launch; serialises nothing, adds ~93 event records)
    eng.set_timing(True)
    eng.forward_resnest50(x)
    cap = 256
    tms, tnames, n = (C.c_float * cap)(), (C.c_char_p * cap)(), C.c_int(0)
    _lib.check(eng._lib.syn_get_timings(eng._h, tms, tnames, cap, C.byref(n)))
    eng.set_timing(False)
    classes = OrderedDict()
    for i in range(n.value):
        k = tnames[i].decode()
        c = classes.setdefault(k, {'launches': 0, 'ms': 0.0})
        c['launches'] += 1
        c['ms'] += float(tms[i])
    for c in classes.values():
        c['ms'] = round(c['ms'], 4)

    res = {'workload': 'resnest50_forward', 'batch': B, 'steps': a.steps, 'warmup': a.warmup,
           'input': 'device-resident fp32 (B,3,120,120) structured synthetic crops, calibrated synthetic checkpoint',
           'launches_per_step': launches, 'ms_per_step': round(ms, 4), 'faces_per_s': round(B / ms * 1e3, 1),
           'macs_per_face': macs, 'algorithmic_tflops': round(flop / (ms * 1e-3) / 1e12, 2),
           'kernel_classes': classes, 'timed_breakdown_ms': round(sum(c['ms'] for c in classes.values()), 4)}

    if not a.no_comparator:
        sd_dev = {k: v.to(dev) for k, v in sd.items() if k.startswith('I2P.backbone.')}
        comp = {}
        for tf32 in (False, True):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            with torch.no_grad():
                o_ref, p_ref = resnest_port.resnest50_forward(sd_dev, x)
                t = time_steps(lambda: resnest_port.resnest50_forward(sd_dev, x), a.steps, a.warmup)
            comp['cudnn_tf32' if tf32 else 'cudnn_fp32'] = {
                'ms_per_step': round(t, 4), 'faces_per_s': round(B / t * 1e3, 1),
                'algorithmic_tflops': round(flop / (t * 1e-3) / 1e12, 2),
                'ours_speedup': round(t / ms, 2),
                'out62_max_rel_diff_vs_ours': rp.max_rel_err(out.cpu().numpy(), o_ref.cpu().numpy()),
                'pool2048_max_rel_diff_vs_ours': rp.max_rel_err(pool.cpu().numpy(), p_ref.cpu().numpy())}
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
        res['comparator_torch_functional'] = comp
    res['card'] = card_info(dev)
    res['torch'] = torch.__version__
    print(json.dumps(res))


if __name__ == '__main__':
    main()
