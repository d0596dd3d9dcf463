#!/usr/bin/env python
"""Headline benchmark: faces/sec of the SynergyNet inference hot path on B200.

    python bench.py --gpus N --steps K --warmup W          # this framework (one process per GPU)
    python bench.py --impl reference --steps K --warmup W  # the reference algorithm on host cores

A step = one pass of the hot path (MobileNetV2 backbone -> 62 3DMM params -> 68 landmarks) over
one batch of 1024 synthetic 120x120 crops per GPU (BASELINE.json configs[1]); with N > 1 the batch
is sharded (weak scaling, 1024 faces per GPU) and the step ends with the single all-gather of
landmarks.  Prints ONE JSON line (see the task contract): `value` is device-resident throughput,
`e2e` goes through the host-buffer C-ABI call with H2D/D2H inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_FACE = 186_430_744            # SURVEY.md section 8(d): 2*(93,204,560 + 10,812) MAC
X_BYTES_PER_FACE = 3 * 120 * 120 * 4
LMK_BYTES_PER_FACE = 3 * 68 * 4
METRIC = 'faces/sec (120x120, batch 1024 per GPU, backbone + 3DMM params + 68 landmarks)'
# algorithmic MAC per face of every launch of the fused engine (SURVEY.md section 8(a) shape table)
KERNEL_MACS = {
    'fused_stem_block1': 3_110_400 + 1_036_800 + 1_843_200, 'fused_block2': 8_380_800, 'fused_block3': 7_387_200,
    'fused_block4': 4_438_800, 'fused_block5': 3_153_600, 'fused_block6': 3_153_600, 'fused_block7': 2_279_424,
    'fused_block8': 3_366_912, 'fused_block9': 3_366_912, 'fused_block10': 3_366_912, 'fused_block11': 4_153_344,
    'fused_block12': 7_409_664, 'fused_block13': 7_409_664, 'fused_block14': 5_096_448, 'fused_block15': 5_053_440,
    'fused_block16': 5_053_440, 'fused_block17': 7_511_040, 'tail_conv_pool_kernel': 6_553_600, 'heads_kernel': 79_360,
    'dense_recon_tc_kernel': 10_812, 'dense_alpha_kernel': 0,
}

# algorithmic HBM bytes per face of every launch: block input + output (NHWC fp32; the stem reads the NCHW crop,
# residual blocks read their input once: the skip comes from L2/smem); DESIGN.md section 5
def _io(cin, hin, cout, hout):
    return 4 * (cin * hin * hin + cout * hout * hout)


KERNEL_BYTES = {
    'fused_stem_block1': _io(3, 120, 16, 60), 'fused_block2': _io(16, 60, 24, 30), 'fused_block3': _io(24, 30, 24, 30),
    'fused_block4': _io(24, 30, 32, 15), 'fused_block5': _io(32, 15, 32, 15), 'fused_block6': _io(32, 15, 32, 15),
    'fused_block7': _io(32, 15, 64, 8), 'fused_block8': _io(64, 8, 64, 8), 'fused_block9': _io(64, 8, 64, 8),
    'fused_block10': _io(64, 8, 64, 8), 'fused_block11': _io(64, 8, 96, 8), 'fused_block12': _io(96, 8, 96, 8),
    'fused_block13': _io(96, 8, 96, 8), 'fused_block14': _io(96, 8, 160, 4), 'fused_block15': _io(160, 4, 160, 4),
    'fused_block16': _io(160, 4, 160, 4), 'fused_block17': _io(160, 4, 320, 4), 'tail_conv_pool_kernel': 4 * (320 * 16 + 1280),
    'heads_kernel': 4 * (1280 + 62), 'dense_recon_tc_kernel': 4 * (62 + 3 * 68), 'dense_alpha_kernel': 4 * 62,
}
DENSE_BYTES_PER_FACE = 3 * 53215 * 4          # SURVEY.md section 8(d): 638,580 B written per face
DUMP_MAX_BYTES = 64 << 20                     # --dump-outputs: above this a fixed sample of faces is written


def load_peaks():
    fp = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(fp):
        with open(fp) as f:
            p = json.load(f)
        return dict(bf16_sustained=p['bf16_tflops_sustained'], bf16_burst=p['bf16_tflops'],
                    hbm=p['hbm_gbs'], source='measured (MEASURED_PEAKS.json)')
    return dict(bf16_sustained=1400.0, bf16_burst=1590.0, hbm=6650.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, reasons, smax = [], set(), None
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ts, line in self.rows:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 7:
                continue
            try:
                smax = float(parts[1])
                if t0 - 0.05 <= ts <= t1 + 0.05:
                    sm.append(float(parts[0]))
                    for n, v in zip(names, parts[3:7]):
                        if v.lower().startswith('active'):
                            reasons.add(n)
            except ValueError:
                continue
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': smax, 'reasons': sorted(reasons), 'samples': 0}
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': smax, 'reasons': sorted(reasons), 'samples': len(sm)}


def dominant_roofline(kernel_ms: dict, batch: int, peaks: dict):
    """`roofline` of the launch that takes the largest share of the step, against BOTH ceilings: algorithmic FLOP
    of that launch / its CUDA-event duration vs the sustained bf16 peak (it runs inside a long step), and its
    algorithmic HBM bytes (block in + out) vs the measured HBM peak.  `bound` names the ceiling that is closer,
    i.e. the one that bounds the kernel.  `traffic` = DRAM bytes of one launch from the committed ncu capture
    (profiles/kernel_traffic.json)."""
    if not kernel_ms:
        return None
    name = max(kernel_ms, key=kernel_ms.get)
    flop = 2.0 * KERNEL_MACS.get(name, 0) * batch
    nbytes = float(KERNEL_BYTES.get(name, 0)) * batch
    ms = kernel_ms[name]
    tflops = flop / (ms * 1e-3) / 1e12
    gbs = nbytes / (ms * 1e-3) / 1e9
    f_tensor, f_hbm = tflops / peaks['bf16_sustained'], gbs / peaks['hbm']
    traffic = None
    fp = os.path.join(ROOT, 'profiles', 'kernel_traffic.json')
    if os.path.exists(fp):
        with open(fp) as f:
            traffic = json.load(f).get(name)
    hbm_bound = f_hbm >= f_tensor
    return {'kernel': name, 'bound': 'hbm' if hbm_bound else 'tensor',
            'achieved': gbs if hbm_bound else tflops, 'peak': peaks['hbm'] if hbm_bound else peaks['bf16_sustained'],
            'unit': 'GB/s' if hbm_bound else 'TFLOP/s', 'frac': f_hbm if hbm_bound else f_tensor,
            'frac_tensor': f_tensor, 'achieved_tflops': tflops, 'frac_hbm': f_hbm, 'achieved_gbs': gbs,
            'traffic': traffic, 'ms_per_launch': ms, 'share_of_step': ms / sum(kernel_ms.values()),
            'what': f'algorithmic {KERNEL_MACS.get(name, 0):,} MAC/face x 2 and {KERNEL_BYTES.get(name, 0):,} HBM B/face '
                    f'x {batch} faces / CUDA-event time of one launch; peaks = sustained bf16 and HBM copy of {peaks["source"]}'}


def dump_outputs(out_dir: str, lmk) -> None:
    """--dump-outputs: the landmarks the timed path returned in its last step, as DIR/landmarks.npy (float32), so that
    two builds run with the same arguments can be compared output for output.  Above DUMP_MAX_BYTES a seeded sample of
    faces (the same faces on every run) is written in their original order."""
    a = np.ascontiguousarray(lmk.cpu().numpy() if torch.is_tensor(lmk) else lmk, np.float32)
    n_max = DUMP_MAX_BYTES // a[:1].nbytes
    if a.shape[0] > n_max:
        a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], n_max, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'landmarks.npy'), a)


def build_model(device: str):
    """Random-init weights of the reference architecture + seeded synthetic 3DMM (no network)."""
    from synergynet_b200 import model_building, synthetic
    from synergynet_b200.params import ParamsPack, set_param_pack
    set_param_pack(ParamsPack(arrays=synthetic.make_3dmm(seed=0)))
    args = types.SimpleNamespace(arch='mobilenet_v2', img_size=120, devices_id=[0])
    model = model_building.SynergyNet(args, _device=device)
    synthetic.seeded_init_(model, 0)
    synthetic.randomize_batchnorm_(model, 0)
    return model.eval()


def cpu_reference_throughput(seconds: float, batch: int = 64):
    """The reference algorithm (oracle port: same ATen CPU kernels as the reference's nn.Modules)
    on the host cores: forward_test + reconstruct_vertex_62(dense=False).  The thread count is
    chosen by a short sweep (oneDNN convs of this size get slower with very many threads), so the
    baseline is the best the host can do, and `cores` is the count actually used."""
    from oracle import reference_port as rp
    from oracle import synth_model
    from synergynet_b200 import synthetic
    sd = synth_model.build_state_dict(0)
    basis = rp.gather_sparse_basis(synthetic.make_3dmm(0))
    x = synthetic.make_inputs(batch, 0)

    def step():
        p, _ = rp.mobilenetv2_forward(sd, x)
        return rp.reconstruct_vertex_62(p.numpy(), basis)

    ncpu = os.cpu_count() or 1
    best_t, best_n = None, ncpu
    for n in sorted({min(ncpu, c) for c in (4, 8, 12, 16, 24, 32, 64, ncpu)}):
        torch.set_num_threads(n)
        step()
        dt = None
        for _ in range(2):                      # best of two: the host is shared, single samples are noisy
            t0 = time.perf_counter()
            step()
            d1 = time.perf_counter() - t0
            dt = d1 if dt is None else min(dt, d1)
        if best_t is None or dt < best_t:
            best_t, best_n = dt, n
        if dt > 4.0:
            break
    torch.set_num_threads(best_n)
    step()
    n, t0 = 0, time.perf_counter()
    while True:
        step()
        n += 1
        el = time.perf_counter() - t0
        if el >= seconds and n >= 3:
            break
    # configs[0]: the reference's own CPU-runnable case, one face per call (latency, same thread count)
    x1 = x[:1]
    for _ in range(3):
        rp.reconstruct_vertex_62(rp.mobilenetv2_forward(sd, x1)[0].numpy(), basis)
    t1 = time.perf_counter()
    for _ in range(20):
        rp.reconstruct_vertex_62(rp.mobilenetv2_forward(sd, x1)[0].numpy(), basis)
    b1_ms = (time.perf_counter() - t1) / 20 * 1e3
    return {'value': n * batch / el, 'unit': 'faces/s', 'cores': best_n, 'kind': 'port',
            'batch1_ms_per_face': b1_ms,
            'sample': f'{n} batches of {batch} faces ({el:.1f} s), forward_test + 68-landmark reconstruction, '
                      f'torch {torch.__version__} CPU fp32, best of a thread sweep on {ncpu} logical CPUs; '
                      f'batch1_ms_per_face = configs[0] (one face per call, 20 calls)'}, step


def run_reference(args):
    """Reference arm: the reference algorithm on the host cores (oracle port = the same ATen CPU kernels the
    reference's nn.Modules dispatch to; the Python reference cannot travel to the GPU box), on the config
    BASELINE.md section 3 names for the CPU row: batches of 64 faces, best thread count of a short sweep.
    One step = one 64-face batch (a bounded sample of the 1024-face workload)."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    sample = 64
    base, step = cpu_reference_throughput(0.0, batch=sample)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        lmk = step()
    el = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, lmk)
    value = args.steps * sample / el
    line = {
        'metric': METRIC, 'value': value, 'unit': 'faces/s', 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * el / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
        'config': {'workload': 'configs[1]: batch=1024 synthetic 120x120 crops, MobileNetV2 + 3DMM params + '
                               '68-landmark reconstruction', 'sample_per_step': sample, 'device': 'host CPU',
                   'same_config': True, 'batch_note': 'BASELINE.md section 3 CPU row: batches of 64 faces (the '
                   'throughput-optimal CPU batch; per-face cost is flat beyond it), thread count = best of a sweep'},
        'cpu_baseline': {'value': value, 'unit': 'faces/s', 'cores': base['cores'], 'kind': 'port',
                         'batch1_ms_per_face': base.get('batch1_ms_per_face'),
                         'sample': f'{sample} faces per step (bounded sample of the 1024-face batch), '
                                   f'{args.steps} steps, {base["cores"]} threads of {os.cpu_count()} logical CPUs'},
        'e2e': {'value': value, 'unit': 'faces/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)


def _time_cuda(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def gpu_reference_comparator(dev, B):
    """Same-box comparator (SURVEY.md section 8(d)): the reference's PyTorch GPU path -- the conv / batch_norm /
    linear / matmul calls of its nn.Modules, restated in oracle/reference_port.py -- on this GPU at batch B with
    cudnn.benchmark, TF32 off (the fp32 parity path) and on (PyTorch's default, fact 7).  A reported comparator,
    not a target and not on the product path."""
    from oracle import reference_port as rp
    from oracle import synth_model
    from synergynet_b200 import synthetic
    sd = {k: v.to(dev) for k, v in synth_model.build_state_dict(0).items() if v.is_floating_point()}
    pack = rp.gather_sparse_basis(synthetic.make_3dmm(0))
    mean, std = (torch.from_numpy(pack[k][:62]).to(dev) for k in ('param_mean', 'param_std'))
    ub, ws, we = (torch.from_numpy(np.ascontiguousarray(pack[k])).to(dev) for k in ('u_base', 'w_shp_base', 'w_exp_base'))
    x = synthetic.make_inputs(B, seed=7).to(dev)

    def step():
        with torch.no_grad():
            param, _ = rp.mobilenetv2_forward(sd, x)
            p = param * std + mean                                     # model_building.py:117
            cam = p[:, :12].reshape(-1, 3, 4)
            S = (ub + ws @ p[:, 12:52].reshape(-1, 40, 1) + we @ p[:, 52:62].reshape(-1, 10, 1))
            v = cam[:, :, :3] @ S.reshape(-1, 68, 3).transpose(1, 2) + cam[:, :, 3:]
            v[:, 1, :] = 121 - v[:, 1, :]
        return v

    out = {}
    old = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    try:
        torch.backends.cudnn.benchmark = True
        for tf32 in (False, True):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            ms = _time_cuda(step, iters=10, warmup=5)
            out['tf32_on' if tf32 else 'tf32_off'] = {'ms_per_step': ms, 'faces_per_s': B / ms * 1e3}
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old
    out['what'] = (f'reference PyTorch GPU path (torch {torch.__version__} eager, cuDNN/cuBLAS, cudnn.benchmark=True), '
                   f'device-resident B={B}, forward_test + 68-landmark reconstruction; kind=port '
                   '(oracle/reference_port.py: the same functional ops the reference modules call)')
    return out


def config5_measurement(dev, peaks, B=512):
    """BASELINE.json configs[4]: ResNet-50 backbone variant (resnet_backbone.py:227-249) at batch 512 and the PointNet
    heads MLP_for / MLP_rev (pointnet_backbone.py:31-106) on 512 faces.  The reference cannot chain the two (I2P unpacks
    two values from a backbone that returns one, MLP_for.conv6 wants a 1280-d feature; SURVEY.md fact 4), so they are
    timed separately: ResNet-50 forward -> (B,102) + 68 landmarks from its first 62 outputs; MLP_for + MLP_rev fed with
    MobileNetV2 features.  Random-init weights of the reference architecture, synthetic crops."""
    from synergynet_b200 import model_building, synthetic
    from synergynet_b200.params import ParamsPack, set_param_pack
    set_param_pack(ParamsPack(arrays=synthetic.make_3dmm(seed=0)))
    rn = model_building.SynergyNet(types.SimpleNamespace(arch='resnet50', img_size=120, devices_id=[dev.index]), _device=str(dev))
    synthetic.seeded_init_(rn, 1)
    synthetic.randomize_batchnorm_(rn, 1)
    rn.eval()
    x = synthetic.make_inputs(B, seed=3).to(dev)
    eng = rn._engine(dev)
    ms_rn = _time_cuda(lambda: rn.reconstruct_vertex_62(rn.forward_test(x)), iters=5, warmup=2)
    flop_rn = 2.0 * 1_259_011_072 * B
    mb = build_model(str(dev))
    e2 = mb._engine(dev)
    params, pool = e2.forward(x, want_pool=True)
    lmk = e2.reconstruct(params)
    ef = mb._pointnet_engine(x, 0)
    mb._pointnet_engine(x, 1)
    ms_for = _time_cuda(lambda: ef.mlp_for(lmk, pool, params), iters=10, warmup=2)
    ms_rev = _time_cuda(lambda: ef.mlp_rev(lmk), iters=10, warmup=2)
    mac_for = 68 * (192 + 4096 + 4096 + 8192 + 131072 + 32768 + 131072 + 32768 + 384) + 2354 * 512
    mac_rev = 68 * (192 + 4096 + 4096 + 8192 + 131072) + 1024 * 62
    return {'workload': 'configs[4]: ResNet-50 backbone variant, batch 512 -> (B,102) + 68 landmarks; PointNet heads on 512 faces',
            'resnet50_ms': ms_rn, 'resnet50_faces_per_s': B / ms_rn * 1e3, 'resnet50_tflops': flop_rn / (ms_rn * 1e-3) / 1e12,
            'resnet50_frac_tensor': flop_rn / (ms_rn * 1e-3) / 1e12 / peaks['bf16_sustained'],
            'mlp_for_ms': ms_for, 'mlp_for_tflops': 2.0 * mac_for * B / (ms_for * 1e-3) / 1e12,
            'mlp_rev_ms': ms_rev, 'mlp_rev_tflops': 2.0 * mac_rev * B / (ms_rev * 1e-3) / 1e12,
            'note': 'general split-fp16 GEMM kernel (tc_gemm_kernel), not tuned: parity-grade coverage of the variant, '
                    'algorithmic FLOP (2 x MAC; the shared per-face part of conv6 counted once) / CUDA-event time'}


def render_detect_measurement(dev, peaks, cpu_too=True):
    """SURVEY.md section 8 rows f2 / f3, the stages either side of the 3DMM path.
    render: B = 8 meshes of 53 215 vertices / 105 408 triangles (synthetic.make_render_meshes: the dense stage's (B,3,N)
    layout, read in place) lit and drawn onto one 720 x 1080 x 3 uint8 canvas = utils/render.py:40-45 for 8 faces.
    detect: FaceBoxes.py:98-127 for a 720 x 1080 network input (16 680 priors), ~1 500 boxes above the score threshold.
    CPU legs: the reference's own rasterize_kernel.cpp compiled in place (oracle/_ref, kind "reference"; else the C port) +
    its numpy lighting; the torch / numpy post-processing with py_cpu_nms (the reference's Cython NMS does not build)."""
    from oracle import render_port as rp
    from synergynet_b200 import Sim3DR, detect, synthetic
    from synergynet_b200.inference import RENDER_CFG
    out = {}
    B, H, W = 8, 720, 1080
    tri = synthetic.make_render_topology()
    verts = synthetic.make_render_meshes(B, H, W, seed=0)
    r = Sim3DR.MeshRenderer(tri, verts.shape[2], dev)
    vd = torch.from_numpy(verts).to(dev)
    v = vd.transpose(1, 2)
    cfg = Sim3DR._light_cfg(**RENDER_CFG)
    bg = torch.zeros((H, W, 3), dtype=torch.uint8, device=dev)
    nrm = r.normals(v)
    col = r.colors(v, nrm, cfg)
    ms_n = _time_cuda(lambda: r.normals(v), iters=50, warmup=5)
    ms_l = _time_cuda(lambda: r.colors(v, nrm, cfg), iters=50, warmup=5)
    ms_r = _time_cuda(lambda: r.rasterize(bg, v, col), iters=50, warmup=5)
    ms_all = _time_cuda(lambda: r.render(bg, v, cfg), iters=50, warmup=5)
    vh = torch.from_numpy(verts).pin_memory()
    img_h = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
    bg_h = torch.zeros((H, W, 3), dtype=torch.uint8).pin_memory()

    def e2e():
        vd.copy_(vh, non_blocking=True)
        bg.copy_(bg_h, non_blocking=True)
        r.render(bg, v, cfg)
        img_h.copy_(bg, non_blocking=True)
    for _ in range(3):
        e2e()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(20):
        e2e()
        torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) / 20 * 1e3
    nver, ntri = verts.shape[2], tri.shape[0]
    alg_bytes = B * nver * 12 + ntri * 12 + 2 * H * W * 3
    try:      # DRAM bytes of one call from the committed ncu capture (profiles/r2_ncu_full_render.txt)
        with open(os.path.join(ROOT, 'profiles', 'kernel_traffic.json')) as f:
            render_traffic = json.load(f).get('render_call')
    except Exception:
        render_traffic = None
    out['render'] = {
        'workload': f'{B} meshes x {nver} vertices / {ntri} triangles -> one {H}x{W}x3 uint8 canvas (normals + lighting + z-buffer), '
                    'vertices read in place from the (B,3,N) layout of the dense stage',
        'normals_ms': ms_n, 'lighting_ms': ms_l, 'rasterize_ms': ms_r, 'total_ms': ms_all, 'meshes_per_s': B / ms_all * 1e3,
        'triangles_per_s': B * ntri / ms_r * 1e3, 'gpu_launches_per_call': 6,
        'e2e': {'ms': e2e_ms, 'meshes_per_s': B / e2e_ms * 1e3, 'h2d_bytes': int(verts.nbytes + H * W * 3), 'd2h_bytes': H * W * 3,
                'what': 'pinned host vertices + canvas in, image out, synchronised per call'},
        'roofline': {'bound': 'hbm', 'achieved': alg_bytes / (ms_all * 1e-3) / 1e9, 'peak': peaks['hbm'], 'unit': 'GB/s',
                     'frac': alg_bytes / (ms_all * 1e-3) / 1e9 / peaks['hbm'], 'traffic': render_traffic,
                     'what': f'algorithmic {alg_bytes} B per call (vertices + triangle list once + canvas in and out) / CUDA-event time of '
                             'the six launches; the stage is instruction-issue / atomic work (raster_depth_kernel: issue slots 82 % busy, '
                             'DRAM 3 %) far below the HBM ceiling; traffic is 13x the algorithmic bytes because the (B,H,W) 64-bit key '
                             'image is cleared and read back whole (100 MB of the 141 MB)'}}
    # ---- detect ---------------------------------------------------------------------------------------------------------------
    ih, iw = 720, 1080
    P = detect.num_priors(ih, iw)
    g = torch.Generator().manual_seed(21)
    loc_h = torch.randn((P, 4), generator=g) * 0.6
    logit = torch.randn((P, 2), generator=g) * 2.0
    logit[:, 0] += 3.4                                                         # ~9 % of the priors pass the 0.05 threshold
    conf_h = torch.softmax(logit, dim=-1)
    loc, conf = loc_h.to(dev), conf_h.to(dev)

    def post():
        dets, n = detect.decode_device(loc, conf, ih, iw)
        return detect.nms_device(dets, detect.nms_threshold, n=int(n.item()))
    n_cand = int((conf_h[:, 1] > detect.confidence_threshold).sum())
    ms_d = _time_cuda(lambda: detect.decode_device(loc, conf, ih, iw), iters=50, warmup=5)
    ms_p = _time_cuda(post, iters=50, warmup=5)
    keep, nk = post()
    out['detect'] = {'workload': f'FaceBoxes post-processing for a {ih}x{iw} input: {P} priors, {n_cand} above the score threshold -> '
                                 f'decode + order + greedy NMS(0.3) -> {int(nk.item())} boxes',
                     'decode_ms': ms_d, 'decode_plus_nms_ms': ms_p, 'images_per_s': 1e3 / ms_p, 'gpu_launches_per_call': 4}
    # the detector network itself (FaceBoxes/models/faceboxes.py) on one 720 x 1080 image: seeded synthetic checkpoint
    from synergynet_b200 import faceboxes
    fsd = synthetic.make_faceboxes_state_dict(0)
    fnet = faceboxes.FaceBoxesNet(fsd, dev)
    scene = synthetic.make_scene_u8(ih, iw, 0)
    scene_d = torch.from_numpy(scene).to(dev)
    ms_net = _time_cuda(lambda: fnet.forward(scene_d), iters=20, warmup=3)
    fb = faceboxes.FaceBoxes(weights=fsd, device=dev)
    fb(scene)
    t0 = time.perf_counter()
    for _ in range(10):
        boxes = fb(scene)
    ms_call = (time.perf_counter() - t0) / 10 * 1e3
    plan = faceboxes.layer_plan()
    g32 = [-(-ih // 32) * -(-iw // 32), -(-ih // 64) * -(-iw // 64), -(-ih // 128) * -(-iw // 128)]
    px = {0: -(-ih // 4) * -(-iw // 4), 1: -(-ih // 16) * -(-iw // 16)}
    mac = 0
    for L in plan:
        n = L['name']
        pix = px.get(L['index'], g32[0])
        if n in ('conv3_2', 'conv4_1', 'loc.1', 'conf.1'):
            pix = g32[1]
        if n in ('conv4_2', 'loc.2', 'conf.2'):
            pix = g32[2]
        mac += pix * L['cin'] * L['cout'] * L['ksize'] ** 2
    out['detect']['network'] = {'workload': f'FaceBoxesNet forward on one {ih}x{iw}x3 uint8 image (33 convs, pools, softmax; {mac / 1e6:.0f} MMAC)',
                                'ms': ms_net, 'tflops': 2.0 * mac / (ms_net * 1e-3) / 1e12, 'gpu_launches_per_call': 39,
                                'detector_call_ms': ms_call, 'detector_images_per_s': 1e3 / ms_call, 'boxes': len(boxes),
                                'note': 'fp32 CUDA-core implicit GEMM (first correct path, not tensor-core code); detector_call = '
                                        'FaceBoxes.__call__ from a host uint8 image to the box list (H2D, network, decode, NMS, D2H)'}
    if cpu_too:
        ver0 = [np.ascontiguousarray(verts[b].T) for b in range(B)]
        kind = 'ref' if rp.have_ref() else 'port'
        img = np.zeros((H, W, 3), np.uint8)
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 3.0:
            rp.render_faces(img, list(verts), tri, kind=kind)
            reps += 1
        cpu_ms = (time.perf_counter() - t0) / reps * 1e3
        out['render']['cpu_baseline'] = {'value': B / cpu_ms * 1e3, 'unit': 'meshes/s', 'cores': 1,
                                         'kind': 'reference' if kind == 'ref' else 'port', 'ms_per_call': cpu_ms,
                                         'sample': f'{reps} calls of utils/render.py:40-45 on the same {B} meshes: Sim3DR C++ '
                                                   '(single-threaded by construction) + numpy lighting'}
        del ver0
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 2.0:
            d = rp.faceboxes_dets(loc_h.numpy(), conf_h.numpy(), ih, iw)
            k = rp.py_cpu_nms(d, detect.nms_threshold)
            reps += 1
        cpu_ms = (time.perf_counter() - t0) / reps * 1e3
        assert len(k) == int(nk.item()), (len(k), int(nk.item()))
        t0 = time.perf_counter()
        reps = 0
        while time.perf_counter() - t0 < 2.0:
            rp.faceboxes_forward(fsd, scene)
            reps += 1
        out['detect']['network']['cpu_baseline'] = {'value': reps / (time.perf_counter() - t0), 'unit': 'images/s', 'cores': torch.get_num_threads(),
                                                    'kind': 'port', 'sample': f'{reps} forwards of the torch CPU restatement of FaceBoxesNet'}
        out['detect']['cpu_baseline'] = {'value': 1e3 / cpu_ms, 'unit': 'images/s', 'cores': torch.get_num_threads(), 'kind': 'port',
                                         'ms_per_call': cpu_ms, 'sample': f'{reps} calls: PriorBox + decode (torch CPU) + argsort + py_cpu_nms (numpy)'}
    return out


def run_b200(args):
    import torch.distributed as dist
    from synergynet_b200 import distributed as sdist
    rank, local_rank, world = sdist.env_rank_world()
    if world > 1:
        sdist.init_process_group('nccl')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    B = args.batch
    model = build_model(f'cuda:{local_rank}')
    if args.engine is not None:
        model.set_engine(args.engine)
    eng = model._engine(dev)
    peaks = load_peaks()

    from synergynet_b200 import synthetic
    n_rot = 3                                   # rotate 3 x 177 MB inputs: every step misses the 126 MB L2
    xs = [synthetic.make_inputs(B, seed=10 * rank + i).to(dev) for i in range(n_rot)]
    # two gather targets: the all-gather of step i runs on a side stream under the backbone of step i+1
    lmk_alls = [torch.empty((world * B, 3, 68), device=dev, dtype=torch.float32) for _ in range(2)]
    lmk_all = lmk_alls[0]
    og = sdist.OverlappedGather(dev) if world > 1 else None

    def step(i):
        lmk = eng.forward_landmarks(xs[i % n_rot])
        if world > 1:
            og.gather(lmk, lmk_alls[i & 1])
        return lmk

    def barrier():
        if world > 1:
            og.wait()                                   # every gather issued so far is part of the timed region
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        t_start = time.time()
        while sampler.proc is not None and not sampler.rows and time.time() - t_start < 5.0:
            time.sleep(0.01)                            # nvidia-smi's start-up stays out of the timed steps
    # the warm-up runs after the sampler's start-up, right before the timed steps, so that they do not begin on an idle
    # GPU whose clocks have dropped
    for i in range(max(args.warmup, 3)):
        step(i)
    barrier()
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    ev0.record()
    for i in range(args.steps):
        lmk = step(i)
    if world > 1:
        og.wait()                                       # the last gather ends inside the CUDA-event region
    ev1.record()
    barrier()
    t_wall1 = time.time()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, lmk_alls[(args.steps - 1) & 1] if world > 1 else lmk)
    ms = ev0.elapsed_time(ev1)
    launches = eng.launch_count - launches0
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    n_timed = args.steps
    eng.raise_if_error()

    # ---- multi-GPU correctness: the gathered tensor holds every rank's shard in rank order -----------------
    verify = None
    if world > 1:
        lmk = eng.forward_landmarks(xs[0])
        sdist.gather_landmarks(lmk, lmk_all)
        torch.cuda.synchronize(dev)
        if rank == 0:
            ok = torch.equal(lmk_all[:B], lmk)
            checked = []
            for rr in sorted({1, world - 1}):
                xr = synthetic.make_inputs(B, seed=10 * rr).to(dev)      # rank rr's first input, recomputed here
                ok = ok and torch.equal(lmk_all[rr * B:(rr + 1) * B], eng.forward_landmarks(xr))
                checked.append(rr)
            verify = {'all_gather_equals_single_gpu': bool(ok), 'remote_shards_recomputed_on_rank0': checked}

    # ---- per-kernel device times (CUDA events behind every launch, outside the timed region) -------------
    kernel_ms = {}
    eng.set_timing(True)
    n_t = 5
    for i in range(n_t):
        eng.forward_landmarks(xs[i % n_rot])
        for name, t_ms in eng.timings():
            kernel_ms[name] = kernel_ms.get(name, 0.0) + t_ms / n_t
    eng.set_timing(False)

    if args.profile:
        if rank == 0:
            emit({'profile_run': True, 'ms_per_step': ms / n_timed, 'gpu_launches': launches})
        return

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, H2D + D2H timed) ----
    # Every step copies ITS crops host -> device and reads ITS landmarks back, all inside the timed region.  `pipelined`
    # is how a loader loop calls the library (benchmark.py:119-132 iterates a pinned DataLoader with non_blocking
    # copies): submit batch k+1, then wait for batch k -- two calls in flight, so the copies of one batch run under the
    # kernels of the previous one.  `blocking` is one synchronous call per step (nothing overlaps across steps).
    def e2e_loop(bufs, steps, pipelined):
        outs = [torch.empty((B, 3, 68), dtype=torch.float32).pin_memory() for _ in range(2)]
        for i in range(3):
            eng.forward_landmarks_host(bufs[i % 2], outs[i % 2])
        barrier()
        t0 = time.perf_counter()
        if pipelined:
            prev = None
            for i in range(steps):
                tk = eng.forward_landmarks_host_submit(bufs[i % 2], outs[i % 2])
                if prev is not None:
                    eng.host_wait(prev)                      # landmarks of step i-1 are on the host
                prev = tk
            eng.host_wait(prev)
        else:
            for i in range(steps):
                eng.forward_landmarks_host(bufs[i % 2], outs[i % 2])   # returns when the landmarks are on the host
        torch.cuda.synchronize(dev)
        sec = time.perf_counter() - t0
        t = torch.tensor([sec], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    xh = [synthetic.make_inputs(B, seed=100 + 10 * rank + i).pin_memory() for i in range(2)]
    e2e_steps = max(3, min(args.steps, 20)) * 4
    e2e_s = e2e_loop(xh, e2e_steps, True)
    e2e_block_s = e2e_loop(xh, e2e_steps, False)

    # ---- same call fed with raw uint8 crops (normalised on the device; bit-identical outputs) --------
    uh = [synthetic.make_crops_u8(B, seed=100 + 10 * rank + i).pin_memory() for i in range(2)]
    u8_s = e2e_loop(uh, e2e_steps, True)
    u8_block_s = e2e_loop(uh, e2e_steps, False)

    extra = {}
    if rank == 0 and world == 1:
        # ---- configs[2]: params -> dense (B,3,53215) vertices, and image -> dense in one stream ---------
        params = eng.forward(xs[0])
        dense_out = [None]

        def dense_step():
            dense_out[0] = eng.reconstruct(params, dense=True)
        d_ms = _time_cuda(dense_step, iters=50, warmup=5)
        img_dense_ms = _time_cuda(lambda: eng.reconstruct(eng.forward(xs[1]), dense=True), iters=20, warmup=3)
        dbytes = float(B) * DENSE_BYTES_PER_FACE
        traffic = None
        fp = os.path.join(ROOT, 'profiles', 'kernel_traffic.json')
        if os.path.exists(fp):
            with open(fp) as f:
                traffic = json.load(f).get('dense_recon_fm_kernel')
        extra['dense'] = {
            'workload': 'configs[2]: batch=1024 params -> dense (B,3,53215) vertices', 'ms': d_ms,
            'faces_per_s': B / d_ms * 1e3, 'image_to_dense_ms': img_dense_ms, 'image_to_dense_faces_per_s': B / img_dense_ms * 1e3,
            'roofline': {'bound': 'hbm', 'achieved': dbytes / d_ms / 1e6, 'peak': peaks['hbm'], 'unit': 'GB/s',
                         'frac': dbytes / d_ms / 1e6 / peaks['hbm'], 'traffic': traffic,
                         'what': '638,580 B written per face x 1024 / CUDA-event time of alpha pre-pass + reconstruction kernel'}}
        del dense_out, params
        # ---- configs[0] shape on the GPU: one face per call, device-resident (eager launches vs one CUDA graph) ----
        x1 = xs[0][:1].contiguous()
        eager_ms = _time_cuda(lambda: eng.forward_landmarks(x1), iters=200, warmup=20)
        graph_ms = None
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                eng.forward_landmarks(x1)
            torch.cuda.current_stream(dev).wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                keep = eng.forward_landmarks(x1)
            graph_ms = _time_cuda(g.replay, iters=200, warmup=20)
            del keep
        except Exception as e:       # graph capture is an optimisation of the launch path, not a requirement
            graph_ms = f'capture failed: {type(e).__name__}: {e}'
        x1h = synthetic.make_inputs(1, seed=5).pin_memory()
        l1h = torch.empty((1, 3, 68), dtype=torch.float32).pin_memory()
        for _ in range(5):
            eng.forward_landmarks_host(x1h, l1h)
        t0 = time.perf_counter()
        for _ in range(100):
            eng.forward_landmarks_host(x1h, l1h)
        host1_ms = (time.perf_counter() - t0) / 100 * 1e3
        extra['latency_b1'] = {'workload': 'configs[0] shape on the GPU: one 120x120 crop -> 68 landmarks',
                               'device_resident_eager_ms': eager_ms, 'device_resident_cuda_graph_ms': graph_ms,
                               'host_call_ms': host1_ms, 'launches_per_call': 21}
        if not args.no_gpu_reference:
            try:
                extra['gpu_reference'] = gpu_reference_comparator(dev, B)
            except Exception as e:
                extra['gpu_reference'] = {'unavailable': f'{type(e).__name__}: {e}'}
        if not args.no_config5:
            # ---- configs[4]: ResNet-50 backbone variant + PointNet refinement heads, batch 512 ---------------
            try:
                extra['config5'] = config5_measurement(dev, peaks)
            except Exception as e:
                extra['config5'] = {'unavailable': f'{type(e).__name__}: {e}'}
        if not args.no_render:
            # ---- SURVEY.md section 8 rows f2 / f3: Sim3DR and FaceBoxes post-processing ---------------------------------------
            try:
                extra.update(render_detect_measurement(dev, peaks, cpu_too=not args.no_cpu_baseline))
            except Exception as e:
                extra['render'] = {'unavailable': f'{type(e).__name__}: {e}'}
        if args.engine is None and not args.no_single_pass:
            # ---- single-pass fp16 engine (NOT parity grade): how much of the step is the 3x precision tax ----
            ref_l, ref_p = eng.forward_landmarks(xs[0][:256], want_params=True)
            try:
                model.set_engine(3)
                one_ms = _time_cuda(lambda: eng.forward_landmarks(xs[1]), iters=50, warmup=5)
                l1, p1 = eng.forward_landmarks(xs[0][:256], want_params=True)
                extra['single_pass_fp16'] = {
                    'ms_per_step': one_ms, 'faces_per_s': B / one_ms * 1e3,
                    'params_max_rel_err_vs_split3': float((p1 - ref_p).abs().max() / ref_p.abs().max()),
                    'landmarks_max_rel_err_vs_split3': float((l1 - ref_l).abs().max() / ref_l.abs().max()),
                    'roofline_step_frac': FLOP_PER_FACE * B / (one_ms * 1e-3) / 1e12 / peaks['bf16_sustained'],
                    'note': 'engine 3 = the fused kernels with one fp16 MMA per product; misses the 1e-4 bar by design, never the default'}
            except Exception as e:
                extra['single_pass_fp16'] = {'unavailable': f'{type(e).__name__}: {e}'}
            finally:
                model.set_engine(2)

    if rank == 0:
        faces = world * B * n_timed
        value = faces / (ms * 1e-3)
        achieved = FLOP_PER_FACE * B * n_timed / (ms * 1e-3) / 1e12        # per GPU, TFLOP/s
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu, _ = cpu_reference_throughput(args.cpu_seconds)
        line = {
            'metric': METRIC, 'value': value, 'unit': 'faces/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': ms / n_timed, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': 'configs[1]: batch=1024 synthetic 120x120 crops, MobileNetV2 + 3DMM params + '
                                   '68-landmark reconstruction' + (' + all-gather of landmarks' if world > 1 else ''),
                       'batch_per_gpu': B, 'global_batch': world * B,
                       'engine': {0: 'simt_fp32', 1: 'tcgen05_f16x3_unfused', 2: 'tcgen05_f16x3_fused',
                                  3: 'tcgen05_f16x1_fused (not parity grade)'}.get(eng.engine, eng.engine),
                       'parallelism': f'dp{world}',
                       'collective': ('one all_gather_into_tensor of the (B,3,68) landmarks per step (NCCL), issued on a side '
                                      'stream under the next step\'s backbone; the last one completes inside the timed region'
                                      if world > 1 else None),
                       'timed_region': f'{args.steps} steps in one CUDA-event region ({ms / 1e3:.2f} s)',
                       'timed_steps': n_timed,
                       'l2': f'{n_rot} rotating device-resident input batches of {B * X_BYTES_PER_FACE / 1e6:.0f} MB '
                             '(> 126 MB L2) + >1 GB of activations written per step'},
            'e2e': {'value': world * B * e2e_steps / e2e_s, 'unit': 'faces/s',
                    'h2d_bytes_per_step': B * X_BYTES_PER_FACE, 'd2h_bytes_per_step': B * LMK_BYTES_PER_FACE,
                    'steps': e2e_steps, 'blocking_value': world * B * e2e_steps / e2e_block_s,
                    'call': 'syn_forward_landmarks_host_submit + syn_host_wait (pinned fp32 crops in, landmarks out), two '
                            'calls in flight: step k+1 is submitted before step k is waited for; blocking_value = one '
                            'synchronous syn_forward_landmarks_host per step'},
            'e2e_u8': {'value': world * B * e2e_steps / u8_s, 'unit': 'faces/s', 'h2d_bytes_per_step': B * X_BYTES_PER_FACE // 4,
                       'd2h_bytes_per_step': B * LMK_BYTES_PER_FACE, 'steps': e2e_steps,
                       'blocking_value': world * B * e2e_steps / u8_block_s,
                       'call': 'the same with pinned uint8 crops, (img-127.5)/128 on the device'},
            'gpu_launches': launches,
            'roofline': dominant_roofline(kernel_ms, B, peaks),
            'kernels_ms': {k: round(v, 4) for k, v in sorted(kernel_ms.items(), key=lambda kv: -kv[1])},
            'roofline_step': {'bound': 'tensor', 'achieved': achieved, 'peak': peaks['bf16_sustained'], 'unit': 'TFLOP/s',
                         'frac': achieved / peaks['bf16_sustained'], 'frac_issued_mma': 3 * achieved / peaks['bf16_sustained'],
                         'traffic': None,
                         'what': 'whole step (all kernels of the fused path): algorithmic 186,430,744 FLOP/face x '
                                 f'{B} faces / CUDA-event step time; peak = sustained bf16 of {peaks["source"]}; '
                                 'frac_issued_mma counts the three fp16 MMAs the split engine issues per product'},
            'cpu_baseline': cpu,
            'clocks': clocks,
        }
        if verify is not None:
            line['verify'] = verify
        line.update(extra)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def _protect_stdout():
    """Third-party code (NCCL banner, torchrun children) may print to fd 1; the contract is ONE JSON
    line on stdout.  Route fd 1 to stderr for the duration of the run and keep a private handle."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    return os.fdopen(saved, 'w')


_OUT = None


def emit(line: dict) -> None:
    _OUT.write(json.dumps(line) + '\n')
    _OUT.flush()


def main():
    global _OUT
    _OUT = _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=1024, help='faces per GPU per step')
    ap.add_argument('--engine', type=int, default=None, help='0 = fp32 CUDA cores, 1 = tcgen05 split-fp16 x3, 2 = 1 + fused blocks (default), 3 = 2 with one fp16 pass')
    ap.add_argument('--cpu-seconds', type=float, default=12.0)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--profile', action='store_true', help='device-resident steps only (for ncu runs)')
    ap.add_argument('--no-gpu-reference', action='store_true', help='skip the same-box PyTorch GPU comparator')
    ap.add_argument('--no-config5', action='store_true', help='skip the ResNet-50 / PointNet heads measurement')
    ap.add_argument('--no-render', action='store_true', help='skip the Sim3DR / FaceBoxes post-processing measurement')
    ap.add_argument('--no-single-pass', action='store_true', help='skip the single-pass fp16 engine measurement')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the landmarks of the last timed step to DIR/landmarks.npy (float32, at most 64 MB)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
