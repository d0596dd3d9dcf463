"""Per-device handle of the sm_100a library: weight hand-over and the compute entry points.

PyTorch is used for device memory, streams and (in bench.py) ``torch.distributed`` only; all
arithmetic of the path runs in ``libsynergy_b200.so``.
"""
from __future__ import annotations

import ctypes as C
import threading
import warnings
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from .backbone import HEAD_DIMS, conv_plan

N_PARAMS = 62


def _host_f32(t) -> torch.Tensor:
    if isinstance(t, np.ndarray):
        t = torch.from_numpy(np.ascontiguousarray(t))
    return t.detach().to(device='cpu', dtype=torch.float32).contiguous()


class Engine:
    """Owns one ``syn_handle_t`` bound to ``cuda:<device>``."""

    def __init__(self, device: int = 0):
        self._lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError('synergynet_b200 needs a CUDA device (B200, sm_100a); there is no '
                               'CPU fallback for the inference hot path')
        self.device = torch.device('cuda', int(device))
        h = C.c_void_p()
        _lib.check(self._lib.syn_create(int(device), C.byref(h)))
        self._h = h
        self.n_pts = 0
        self.n_vert = 0
        self._keep = []
        # The C handle is not re-entrant and all calls share one activation workspace: serialise the host threads
        # (nn.DataParallel replicas use one engine per device, but user threads may share a model) and order
        # consecutive calls that arrive on different CUDA streams with an event.
        self._lock = threading.RLock()
        self._host_inflight: Dict[int, tuple] = {}     # ticket -> tensors of a submitted host call (kept alive)
        self._last_stream = None
        self._last_event = None

    def close(self):
        if getattr(self, '_h', None):
            self._lib.syn_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    # ---- weights --------------------------------------------------------------------------------
    def load_backbone(self, sd: Dict[str, torch.Tensor], prefix: str = 'I2P.backbone.') -> None:
        """Hand the 52 conv+BN pairs and the three heads of a reference-schema state dict
        (SURVEY.md section 8(b)) to the library."""
        for spec in conv_plan():
            w = _host_f32(sd[f'{prefix}{spec.conv_key}.weight'])
            bn = [_host_f32(sd[f'{prefix}{spec.bn_key}.{k}'])
                  for k in ('weight', 'bias', 'running_mean', 'running_var')]
            _lib.check(self._lib.syn_set_conv_bn(self._h, spec.index, w.data_ptr(), w.numel(),
                                                 *[t.data_ptr() for t in bn], 1e-5))
        heads = []
        for name, _ in HEAD_DIMS:
            heads += [_host_f32(sd[f'{prefix}{name}.1.weight']), _host_f32(sd[f'{prefix}{name}.1.bias'])]
        _lib.check(self._lib.syn_set_heads(self._h, *[t.data_ptr() for t in heads]))

    def load_3dmm(self, param_mean, param_std, u_base, w_shp_base, w_exp_base, u=None, w_shp=None,
                  w_exp=None) -> None:
        mean, std = _host_f32(param_mean).reshape(-1)[:62].contiguous(), _host_f32(param_std).reshape(-1)[:62].contiguous()
        _lib.check(self._lib.syn_set_whitening(self._h, mean.data_ptr(), std.data_ptr()))
        ub, wsb, web = _host_f32(u_base), _host_f32(w_shp_base), _host_f32(w_exp_base)
        self.n_pts = ub.numel() // 3
        _lib.check(self._lib.syn_set_basis_sparse(self._h, ub.data_ptr(), wsb.data_ptr(), web.data_ptr(), self.n_pts))
        if u is not None:
            ud, wsd, wed = _host_f32(u), _host_f32(w_shp), _host_f32(w_exp)
            self.n_vert = ud.numel() // 3
            _lib.check(self._lib.syn_set_basis_dense(self._h, ud.data_ptr(), wsd.data_ptr(), wed.data_ptr(), self.n_vert))

    def commit(self) -> None:
        _lib.check(self._lib.syn_commit(self._h))

    def set_engine(self, engine: int) -> None:
        _lib.check(self._lib.syn_set_engine(self._h, int(engine)))

    @property
    def engine(self) -> int:
        return self._lib.syn_get_engine(self._h)

    @property
    def launch_count(self) -> int:
        return int(self._lib.syn_launch_count(self._h))

    def set_timing(self, on: bool) -> None:
        _lib.check(self._lib.syn_set_timing(self._h, int(on)))

    def timings(self):
        """[(kernel label, ms)] of the last device-buffer call (needs set_timing(True) before it)."""
        ms = (C.c_float * 64)()
        names = (C.c_char_p * 64)()
        n = C.c_int(0)
        _lib.check(self._lib.syn_get_timings(self._h, ms, names, 64, C.byref(n)))
        return [(names[i].decode(), float(ms[i])) for i in range(n.value)]

    def poll_error(self) -> int:
        """Device sync + sticky in-kernel timeout flag (0 = clean)."""
        flag = C.c_int(0)
        _lib.check(self._lib.syn_poll_error(self._h, C.byref(flag)))
        return int(flag.value)

    # ---- compute --------------------------------------------------------------------------------
    def _check_x(self, x: torch.Tensor) -> torch.Tensor:
        if x.dim() != 4 or tuple(x.shape[1:]) != (3, 120, 120):
            raise RuntimeError(f'expected (B,3,120,120) input, got {tuple(x.shape)}')
        if x.device != self.device:
            raise RuntimeError(f'input on {x.device}, engine on {self.device}')
        return x.to(torch.float32).contiguous()

    def _stream(self) -> int:
        """Current torch stream of the engine's device; if the previous call ran on another stream, that
        stream's work is ordered before this call (the workspace buffers are shared)."""
        st = torch.cuda.current_stream(self.device)
        if torch.cuda.is_current_stream_capturing():
            return st.cuda_stream            # CUDA-graph capture: no cross-stream events (they would join the graph)
        for ticket in list(self._host_inflight):     # submitted host calls run on the library's own streams and use the
            _lib.check(self._lib.syn_host_wait(self._h, ticket))   # same workspace: let them finish (tickets stay valid)
        if self._last_stream is not None and self._last_stream != st.cuda_stream and self._last_event is not None:
            st.wait_event(self._last_event)
        return st.cuda_stream

    def _done(self) -> None:
        if torch.cuda.is_current_stream_capturing():
            return
        st = torch.cuda.current_stream(self.device)
        if self._last_event is None:
            self._last_event = torch.cuda.Event()
        self._last_event.record(st)
        self._last_stream = st.cuda_stream

    def raise_if_error(self) -> None:
        """Cheap (no device sync) look at the sticky time-out flag of the bounded in-kernel waits; call it after a
        host-side synchronisation point (``.cpu()``, ``synchronize``) before trusting the outputs."""
        fn = getattr(self._lib, 'syn_peek_error', None)
        if fn is None:
            return
        flag = C.c_int(0)
        _lib.check(fn(self._h, C.byref(flag)))
        if flag.value:
            raise _lib.SynergyLibError(2, 'a kernel timed out in a pipeline wait; outputs are invalid '
                                          '(Engine.poll_error() reports and clears the flag)')

    def poll_saturation(self, warn: bool = True) -> int:
        """Device sync + sticky "a block input was clamped to the fp16 range" flag of the split-fp16 engines
        (|x| > ~937 at a block input).  Non-zero: use ``set_engine(0)`` (fp32) for this checkpoint."""
        fn = getattr(self._lib, 'syn_poll_saturation', None)
        if fn is None:
            return 0
        flag = C.c_int(0)
        _lib.check(fn(self._h, C.byref(flag)))
        if flag.value and warn:
            warnings.warn('synergynet_b200: an activation left the range of the split-fp16 tensor-core engines and was '
                          'clamped; results differ from fp32 -- use set_engine(0) for this checkpoint', RuntimeWarning)
        return int(flag.value)

    def forward(self, x: torch.Tensor, want_pool: bool = False):
        x = self._check_x(x)
        b = x.shape[0]
        params = torch.empty((b, N_PARAMS), device=self.device, dtype=torch.float32)
        pool = torch.empty((b, 1280), device=self.device, dtype=torch.float32) if want_pool else None
        with self._lock:
            _lib.check(self._lib.syn_forward(self._h, x.data_ptr(), b, params.data_ptr(),
                                             pool.data_ptr() if want_pool else None, self._stream()))
            self._done()
        return (params, pool) if want_pool else params

    def reconstruct(self, params: torch.Tensor, dense: bool = False, whitening: bool = True,
                    transform: bool = True) -> torch.Tensor:
        if params.dim() != 2 or params.shape[1] != N_PARAMS:
            raise RuntimeError('length of params mismatch')          # model_building.py:116-119
        params = params.to(device=self.device, dtype=torch.float32).contiguous()
        b = params.shape[0]
        n = self.n_vert if dense else self.n_pts
        if n == 0:
            raise RuntimeError('dense basis not loaded' if dense else 'sparse basis not loaded')
        out = torch.empty((b, 3, n), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_reconstruct(self._h, params.data_ptr(), b, int(dense), int(whitening),
                                                 int(transform), out.data_ptr(), self._stream()))
            self._done()
        return out

    def reconstruct_image(self, params: torch.Tensor, roi5: torch.Tensor, dense: bool = False) -> torch.Tensor:
        """reconstruct_vertex_62 + the crop -> image affine of _predict_vertices (utils/inference.py:127-138) in one
        kernel: (B,3,N) vertices in the coordinates of the original image.  ``roi5`` (B,5) fp32 = kx, sx, ky, sy, kz
        (``inference.roi_affine``)."""
        params, roi5 = self._dev_f32(params), self._dev_f32(roi5)
        b = params.shape[0]
        if params.dim() != 2 or params.shape[1] != N_PARAMS:
            raise RuntimeError('length of params mismatch')
        if tuple(roi5.shape) != (b, 5):
            raise RuntimeError(f'roi5 must be (B,5), got {tuple(roi5.shape)}')
        n = self.n_vert if dense else self.n_pts
        if n == 0:
            raise RuntimeError('dense basis not loaded' if dense else 'sparse basis not loaded')
        out = torch.empty((b, 3, n), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_reconstruct_image(self._h, params.data_ptr(), b, int(dense), roi5.data_ptr(), out.data_ptr(),
                                                       self._stream()))
            self._done()
        return out

    def pose_decode(self, params: torch.Tensor, roi5: Optional[torch.Tensor] = None):
        """Batched parse_pose + predict_pose (utils/inference.py:33-62,86-92,146-157): (angles (B,3) float64 degrees,
        t3d (B,3) float32 -- in image coordinates when ``roi5`` is given)."""
        params = self._dev_f32(params)
        b = params.shape[0]
        if roi5 is not None:
            roi5 = self._dev_f32(roi5)
            if tuple(roi5.shape) != (b, 5):
                raise RuntimeError(f'roi5 must be (B,5), got {tuple(roi5.shape)}')
        ang = torch.empty((b, 3), device=self.device, dtype=torch.float64)
        t3d = torch.empty((b, 3), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_pose_decode(self._h, params.data_ptr(), b, roi5.data_ptr() if roi5 is not None else None,
                                                 ang.data_ptr(), t3d.data_ptr(), self._stream()))
            self._done()
        return ang, t3d

    def set_center_crop(self, margin: int) -> None:
        """CenterCrop(margin, mode='test') of the reference loader for the uint8 entry points (0 = off)."""
        _lib.check(self._lib.syn_set_center_crop(self._h, int(margin)))

    def forward_landmarks(self, x: torch.Tensor, want_params: bool = False):
        """x: fp32 normalised crops, or raw uint8 crops (normalised on the device)."""
        if x.dtype == torch.uint8:
            return self._forward_landmarks_u8(x, want_params)
        x = self._check_x(x)
        b = x.shape[0]
        lmk = torch.empty((b, 3, self.n_pts), device=self.device, dtype=torch.float32)
        params = torch.empty((b, N_PARAMS), device=self.device, dtype=torch.float32) if want_params else None
        with self._lock:
            _lib.check(self._lib.syn_forward_landmarks(self._h, x.data_ptr(), b,
                                                       params.data_ptr() if want_params else None,
                                                       lmk.data_ptr(), self._stream()))
            self._done()
        return (lmk, params) if want_params else lmk

    def _forward_landmarks_u8(self, x: torch.Tensor, want_params: bool):
        if x.dim() != 4 or tuple(x.shape[1:]) != (3, 120, 120) or x.device != self.device:
            raise RuntimeError(f'expected uint8 (B,3,120,120) on {self.device}, got {tuple(x.shape)} on {x.device}')
        x = x.contiguous()
        b = x.shape[0]
        lmk = torch.empty((b, 3, self.n_pts), device=self.device, dtype=torch.float32)
        params = torch.empty((b, N_PARAMS), device=self.device, dtype=torch.float32) if want_params else None
        with self._lock:
            _lib.check(self._lib.syn_forward_landmarks_u8(self._h, x.data_ptr(), b,
                                                          params.data_ptr() if want_params else None,
                                                          lmk.data_ptr(), self._stream()))
            self._done()
        return (lmk, params) if want_params else lmk

    def forward_landmarks_host(self, x_host: torch.Tensor, lmk_host: Optional[torch.Tensor] = None,
                               params_host: Optional[torch.Tensor] = None) -> torch.Tensor:
        """End-to-end call on HOST tensors (pinned recommended): H2D, forward, landmarks, D2H.  Synchronous."""
        return self.host_wait(self.forward_landmarks_host_submit(x_host, lmk_host, params_host))

    def forward_landmarks_host_submit(self, x_host: torch.Tensor, lmk_host: Optional[torch.Tensor] = None,
                                      params_host: Optional[torch.Tensor] = None) -> int:
        """Enqueue the end-to-end call and return a ticket for :meth:`host_wait`.  Up to two calls may be in flight: the
        second one's host->device copies run under the first one's kernels (a loader loop: submit batch k+1, then wait
        for batch k).  The tensors are kept alive here until their ticket has been waited for."""
        if x_host.is_cuda or x_host.dtype not in (torch.float32, torch.uint8) or not x_host.is_contiguous():
            raise RuntimeError('x_host must be a contiguous fp32 (normalised) or uint8 (raw) CPU tensor')
        if x_host.dim() != 4 or tuple(x_host.shape[1:]) != (3, 120, 120):
            raise RuntimeError(f'expected (B,3,120,120) crops, got {tuple(x_host.shape)}')
        b = x_host.shape[0]
        if lmk_host is None:
            lmk_host = torch.empty((b, 3, self.n_pts), dtype=torch.float32)
        # the C side writes B*3*n_pts and B*62 floats through these pointers: refuse anything it could overrun
        for name, buf, need in (('lmk_host', lmk_host, b * 3 * self.n_pts), ('params_host', params_host, b * N_PARAMS)):
            if buf is None:
                continue
            if buf.is_cuda or buf.dtype != torch.float32 or not buf.is_contiguous() or buf.numel() < need:
                raise RuntimeError(f'{name} must be a contiguous CPU float32 tensor with at least {need} elements')
        ticket = C.c_int(0)
        with self._lock:
            if self._last_event is not None:         # stream-ordered calls share the workspace with the host pipeline
                self._last_event.synchronize()
            _lib.check(self._lib.syn_forward_landmarks_host_submit(
                self._h, x_host.data_ptr(), 1 if x_host.dtype == torch.uint8 else 0, b,
                params_host.data_ptr() if params_host is not None else None, lmk_host.data_ptr(), C.byref(ticket)))
            self._host_inflight[ticket.value] = (x_host, lmk_host, params_host)
        return ticket.value

    def host_wait(self, ticket: int) -> torch.Tensor:
        """Block until the call behind ``ticket`` has written its host outputs; returns its landmark tensor."""
        with self._lock:
            if ticket not in self._host_inflight:
                raise RuntimeError(f'unknown or already collected ticket {ticket}')
            try:
                _lib.check(self._lib.syn_host_wait(self._h, ticket))
            finally:
                _, lmk_host, _ = self._host_inflight.pop(ticket)
        return lmk_host

    # ---- PointNet refinement heads + losses (training-forward surface, model_building.py:141-157) --------------
    _FOR_LAYERS = [f'conv{i}' for i in range(1, 10)]
    _REV_LAYERS = ['conv1', 'conv2', 'conv3', 'conv4', 'conv5', 'conv6_1', 'conv6_2', 'conv6_3']

    def load_pointnet(self, net: int, sd: Dict[str, torch.Tensor]) -> None:
        """net 0: MLP_for state dict (conv1..conv9 + bn1..bn9), net 1: MLP_rev (conv1..5, conv6_1/2/3 + their BN);
        keys without prefix, as ``module.state_dict()`` returns them (pointnet_backbone.py:7-29,67-88)."""
        names = self._FOR_LAYERS if net == 0 else self._REV_LAYERS
        with self._lock:
            for i, cname in enumerate(names):
                bname = 'bn' + cname[4:]
                w = _host_f32(sd[f'{cname}.weight'])
                cb = _host_f32(sd[f'{cname}.bias'])
                bn = [_host_f32(sd[f'{bname}.{k}']) for k in ('weight', 'bias', 'running_mean', 'running_var')]
                _lib.check(self._lib.syn_pointnet_set_layer(self._h, net, i, w.data_ptr(), w.shape[0], w.shape[1], cb.data_ptr(),
                                                            *[t.data_ptr() for t in bn], 1e-5))
            _lib.check(self._lib.syn_pointnet_commit(self._h, net))

    def _dev_f32(self, t: torch.Tensor) -> torch.Tensor:
        return t.to(device=self.device, dtype=torch.float32).contiguous()

    def mlp_for(self, lmk: torch.Tensor, pool: torch.Tensor, params: torch.Tensor):
        """(point_residual (B,3,68), lmk + 0.05 * point_residual) -- MLP_for.forward + model_building.py:150."""
        lmk, pool, params = self._dev_f32(lmk), self._dev_f32(pool), self._dev_f32(params)
        b = lmk.shape[0]
        if tuple(lmk.shape[1:]) != (3, 68) or tuple(pool.shape) != (b, 1280) or tuple(params.shape) != (b, N_PARAMS):
            raise RuntimeError(f'mlp_for: expected (B,3,68), (B,1280), (B,62); got {tuple(lmk.shape)}, {tuple(pool.shape)}, {tuple(params.shape)}')
        res, ref = torch.empty_like(lmk), torch.empty_like(lmk)
        with self._lock:
            _lib.check(self._lib.syn_mlp_for(self._h, lmk.data_ptr(), pool.data_ptr(), params.data_ptr(), b, res.data_ptr(),
                                             ref.data_ptr(), self._stream()))
            self._done()
        return res, ref

    def mlp_rev(self, lmk: torch.Tensor) -> torch.Tensor:
        lmk = self._dev_f32(lmk)
        if lmk.dim() != 3 or tuple(lmk.shape[1:]) != (3, 68):
            raise RuntimeError(f'mlp_rev: expected (B,3,68), got {tuple(lmk.shape)}')
        out = torch.empty((lmk.shape[0], N_PARAMS), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_mlp_rev(self._h, lmk.data_ptr(), lmk.shape[0], out.data_ptr(), self._stream()))
            self._done()
        return out

    def wing_loss(self, pred: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
        """WingLoss(omega=10, epsilon=2) of two (B,3,N) tensors -> 0-d tensor (loss_definition.py:8-27)."""
        pred, target = self._dev_f32(pred), self._dev_f32(target)
        if pred.shape != target.shape or pred.dim() != 3 or pred.shape[1] != 3:
            raise RuntimeError(f'wing_loss: expected two (B,3,N) tensors, got {tuple(pred.shape)} and {tuple(target.shape)}')
        out = torch.empty((1,), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_wing_loss(self._h, pred.data_ptr(), target.data_ptr(), pred.shape[0], pred.shape[2],
                                               out.data_ptr(), self._stream()))
            self._done()
        return out[0]

    def param_loss(self, inp: torch.Tensor, target: torch.Tensor, mode: str = 'normal') -> torch.Tensor:
        """ParamLoss (loss_definition.py:29-42): per-sample (B,) tensor; mode 'normal' or 'only_3dmm'."""
        if mode not in ('normal', 'only_3dmm'):
            raise RuntimeError(f"param_loss: mode must be 'normal' or 'only_3dmm', got {mode!r}")
        inp, target = self._dev_f32(inp), self._dev_f32(target)
        if inp.dim() != 2 or inp.shape[1] != N_PARAMS or target.shape != inp.shape:
            raise RuntimeError('param_loss: expected two (B,62) tensors')
        out = torch.empty((inp.shape[0],), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_param_loss(self._h, inp.data_ptr(), target.data_ptr(), inp.shape[0],
                                                0 if mode == 'normal' else 1, out.data_ptr(), self._stream()))
            self._done()
        return out

    # ---- ResNet-50 backbone variant (BASELINE.json configs[4]) ---------------------------------------------------
    def load_resnet50(self, sd: Dict[str, torch.Tensor], prefix: str = '') -> None:
        """Hand a ``resnet_backbone.resnet50()`` state dict to the library (53 conv+BN pairs in execution order, the four
        Linear heads concatenated in the reference's output order ori | shape | exp | tex, resnet_backbone.py:242-246)."""
        from .backbone import resnet50_conv_keys
        with self._lock:
            for i, (ck, bk) in enumerate(resnet50_conv_keys()):
                w = _host_f32(sd[f'{prefix}{ck}.weight'])
                bn = [_host_f32(sd[f'{prefix}{bk}.{k}']) for k in ('weight', 'bias', 'running_mean', 'running_var')]
                _lib.check(self._lib.syn_resnet_set_conv(self._h, i, w.data_ptr(), w.numel(), *[t.data_ptr() for t in bn], 1e-5))
            order = ('fc_ori', 'fc_shape', 'fc_exp', 'fc_tex')
            w = torch.cat([_host_f32(sd[f'{prefix}{k}.weight']) for k in order]).contiguous()
            b = torch.cat([_host_f32(sd[f'{prefix}{k}.bias']) for k in order]).contiguous()
            _lib.check(self._lib.syn_resnet_set_heads(self._h, w.data_ptr(), b.data_ptr()))
            _lib.check(self._lib.syn_resnet_commit(self._h))

    def forward_resnet50(self, x: torch.Tensor):
        """ResNet._forward_impl (resnet_backbone.py:227-249): (B,3,120,120) -> ((B,102) ori|shape|exp|tex, (B,2048) pooled)."""
        x = self._check_x(x)
        b = x.shape[0]
        out = torch.empty((b, 102), device=self.device, dtype=torch.float32)
        pool = torch.empty((b, 2048), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_resnet50_forward(self._h, x.data_ptr(), b, out.data_ptr(), pool.data_ptr(), self._stream()))
            self._done()
        return out, pool

    # ---- ResNeSt-50 backbone variant (I2P with arch 'resnest*', model_building.py:48-49) ---------------------------------
    def load_resnest50(self, sd: Dict[str, torch.Tensor], prefix: str = '') -> None:
        """Hand a ``ResNeSt.resnest50()`` state dict to the library: the 87 layers in execution order (conv weight, conv
        bias where the layer has one, its BatchNorm where it has one) and the three evaluated Linear heads concatenated
        in the reference's output order ori | shape | exp (ResNeSt/resnet.py:316-320)."""
        from .backbone import resnest50_layer_keys
        bn_fields = ('weight', 'bias', 'running_mean', 'running_var')
        with self._lock:
            for i, (ck, bk) in enumerate(resnest50_layer_keys()):
                w = _host_f32(sd[f'{prefix}{ck}.weight'])
                b = sd.get(f'{prefix}{ck}.bias')
                b = _host_f32(b) if b is not None else None
                bn = [_host_f32(sd[f'{prefix}{bk}.{k}']) for k in bn_fields] if bk is not None else None
                ptrs = [t.data_ptr() for t in bn] if bn is not None else [None] * 4
                _lib.check(self._lib.syn_resnest_set_layer(self._h, i, w.data_ptr(), w.numel(),
                                                           b.data_ptr() if b is not None else None, *ptrs, 1e-5))
            order = ('fc_ori', 'fc_shape', 'fc_exp')
            w = torch.cat([_host_f32(sd[f'{prefix}{k}.weight']) for k in order]).contiguous()
            b = torch.cat([_host_f32(sd[f'{prefix}{k}.bias']) for k in order]).contiguous()
            _lib.check(self._lib.syn_resnest_set_heads(self._h, w.data_ptr(), b.data_ptr()))
            _lib.check(self._lib.syn_resnest_commit(self._h))

    def forward_resnest50(self, x: torch.Tensor):
        """ResNet.forward of ResNeSt-50 (ResNeSt/resnet.py:298-324): (B,3,120,120) -> ((B,62) ori|shape|exp, (B,2048) pooled)."""
        x = self._check_x(x)
        b = x.shape[0]
        out = torch.empty((b, N_PARAMS), device=self.device, dtype=torch.float32)
        pool = torch.empty((b, 2048), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_resnest50_forward(self._h, x.data_ptr(), b, out.data_ptr(), pool.data_ptr(), self._stream()))
            self._done()
        return out, pool

    def debug_forward_until(self, x: torch.Tensor, layer: int) -> torch.Tensor:
        x = self._check_x(x)
        spec = conv_plan()[layer]
        out = torch.empty((x.shape[0], spec.h_out, spec.h_out, spec.cout), device=self.device, dtype=torch.float32)
        with self._lock:
            _lib.check(self._lib.syn_debug_forward_until(self._h, x.data_ptr(), x.shape[0], layer,
                                                         out.data_ptr(), self._stream()))
            self._done()
        return out
