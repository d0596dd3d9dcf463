"""Drop-in twin of the reference ``model_building.py`` for the inference hot path.

Same class names, constructor arguments, attributes, ``state_dict`` keys and method signatures
(reference model_building.py:25-32,35-62,65-165,169-306); the arithmetic of ``forward_test`` and
``reconstruct_vertex_62`` runs in the sm_100a library through ``Engine`` -- no torch conv/matmul is
executed on the product path and nothing falls back to the CPU.
"""
from __future__ import annotations

import threading
import types
from typing import Callable, Dict, Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import backbone as mobilenetv2_backbone
from .backbone import MLP_for, MLP_rev
from .engine import Engine
from .inference import crop_img, roi_affine, square_roi
from .params import ParamsPack, get_param_pack, set_param_pack  # noqa: F401  (re-exported)

_LOSS_KEYS = ('loss_LMK_f0', 'loss_LMK_pointNet', 'loss_Param_In', 'loss_Param_S2', 'loss_Param_S1S2')


def parse_param_62(param):
    """Views of a (B,62) tensor: rotation (B,3,3), offset (B,3,1), alpha_shp (B,40,1),
    alpha_exp (B,10,1) (reference model_building.py:25-32; index work, bit-exact)."""
    cam = param[:, :12].reshape(-1, 3, 4)
    return (cam[:, :, :3], cam[:, :, -1].reshape(-1, 3, 1),
            param[:, 12:52].reshape(-1, 40, 1), param[:, 52:62].reshape(-1, 10, 1))


class _Runtime:
    """Per-device engines for one model; rebuilt when the parameters they were packed from change
    (``load_state_dict``, in-place edits, ``.cuda()``)."""

    def __init__(self):
        self._engines: Dict[int, Engine] = {}
        self._sig: Dict[int, tuple] = {}
        self._pn_sig: Dict[tuple, tuple] = {}
        self._lock = threading.RLock()
        self.engine_kind = None      # None: the library default (fused tcgen05 engine)

    @staticmethod
    def _signature(tensors) -> tuple:
        return tuple((t.data_ptr(), t._version) for t in tensors)

    def get(self, device: torch.device, backbone_sd: Callable[[], Dict[str, torch.Tensor]],
            basis: Optional[Callable[[], Dict[str, torch.Tensor]]]) -> Engine:
        if device.type != 'cuda':
            raise RuntimeError('synergynet_b200: the forward pass needs inputs on a CUDA device '
                               '(B200); there is no CPU fallback')
        idx = device.index if device.index is not None else torch.cuda.current_device()
        sd = backbone_sd()
        bs = basis() if basis is not None else {}
        sig = self._signature(list(sd.values()) + list(bs.values()))
        with self._lock:
            eng = self._engines.get(idx)
            if eng is None or self._sig.get(idx) != sig:
                if eng is None:
                    eng = Engine(idx)
                    self._engines[idx] = eng
                eng.load_backbone(sd, prefix='')
                if bs:
                    eng.load_3dmm(bs['param_mean'], bs['param_std'], bs['u_base'], bs['w_shp_base'],
                                  bs['w_exp_base'], bs.get('u'), bs.get('w_shp'), bs.get('w_exp'))
                else:   # backbone-only use: identity whitening, dummy one-point basis
                    z = torch.zeros(62)
                    eng.load_3dmm(z, z + 1, torch.zeros(3, 1), torch.zeros(3, 40), torch.zeros(3, 10))
                eng.commit()
                if self.engine_kind is not None:
                    eng.set_engine(self.engine_kind)
                self._sig[idx] = sig
                self._pn_sig.pop((idx, 0), None)          # a new commit rebuilds the library state: re-hand the heads
                self._pn_sig.pop((idx, 1), None)
        return eng

    def ensure_pointnet(self, eng: Engine, net: int, module: nn.Module) -> None:
        """Hand the PointNet head ``module`` (net 0 = MLP_for, 1 = MLP_rev) to ``eng`` when its parameters changed."""
        sd = {k: v for k, v in module.state_dict(keep_vars=True).items() if not k.endswith('num_batches_tracked')}
        sig = self._signature(list(sd.values()))
        key = (eng.device.index, net)
        with self._lock:
            if self._pn_sig.get(key) != sig:
                eng.load_pointnet(net, sd)
                self._pn_sig[key] = sig


class I2P(nn.Module):
    """Image-to-parameter module (reference model_building.py:35-62)."""

    def __init__(self, args):
        super().__init__()
        self.args = args
        if 'mobilenet_v2' in self.args.arch:
            self.backbone = getattr(mobilenetv2_backbone, args.arch)(pretrained=False)
        elif self.args.arch == 'resnet50':
            # BASELINE.json configs[4].  The reference's own I2P cannot run this backbone: ResNet._forward_impl returns
            # ONE (B,102) tensor (resnet_backbone.py:242-249) and I2P unpacks two (model_building.py:55,61; SURVEY.md
            # fact 4).  Adapter used here (and by the oracle / golden vectors): params = out[:, :62] (ori|shape|exp),
            # avgpool = the 2048-d pooled feature.
            self.backbone = mobilenetv2_backbone.resnet50(pretrained=False)
        elif 'resnest' in self.args.arch:
            # the reference builds resnest50() for ANY arch containing 'resnest' (model_building.py:48-49); it returns
            # (params62, avgpool2048) exactly as I2P unpacks (ResNeSt/resnet.py:298-324), so no adapter is needed.
            self.backbone = mobilenetv2_backbone.resnest50(pretrained=False)
        elif any(k in self.args.arch for k in ('mobilenet', 'resnet', 'ghostnet')):
            raise RuntimeError(f"arch '{args.arch}': mobilenet_v2, resnet50 and resnest50 are built for sm_100a "
                               '(SURVEY.md section 8; the other backbones are not on the hot path)')
        else:
            raise RuntimeError("Please choose [mobilenet_v2, mobilenet_1, resnet50, or ghostnet]")
        # the variant backbones run on their own library entry points (None: MobileNetV2, the fused default path)
        self._variant = 'resnet50' if self.args.arch == 'resnet50' else 'resnest50' if 'resnest' in self.args.arch else None
        self._is_resnet = self._variant is not None
        object.__setattr__(self, '_rt', _Runtime())
        object.__setattr__(self, '_basis_provider', None)

    def _backbone_sd(self):
        return {k: v for k, v in self.backbone.state_dict(keep_vars=True).items()
                if not k.endswith('num_batches_tracked')}

    def _engine(self, device) -> Engine:
        if self._is_resnet:
            return self._resnet_engine(device)
        return self._rt.get(device, self._backbone_sd, self._basis_provider)

    def _resnet_engine(self, device) -> Engine:
        """Engine with the weights of the variant backbone (ResNet-50 or ResNeSt-50): the shared library state (error flag,
        3DMM bases for reconstruct) comes from a commit of the MobileNetV2 path with a zero checkpoint of the right schema,
        then the variant's layers are handed over."""
        rt = self._rt
        if not hasattr(rt, '_mbv2_stub'):
            rt._mbv2_stub = {k: v for k, v in mobilenetv2_backbone.mobilenet_v2().state_dict().items()
                             if not k.endswith('num_batches_tracked')}
        eng = rt.get(device, lambda: rt._mbv2_stub, self._basis_provider)
        sd = self._backbone_sd()
        sig = rt._signature(list(sd.values()))
        key = (eng.device.index, self._variant)
        attr = f'_{self._variant}_commit_of'
        with rt._lock:
            if rt._pn_sig.get(key) != sig or getattr(eng, attr, None) is not rt._sig.get(eng.device.index):
                getattr(eng, f'load_{self._variant}')(sd)
                rt._pn_sig[key] = sig
                setattr(eng, attr, rt._sig.get(eng.device.index))
        return eng

    def _compute_device(self, t: Optional[torch.Tensor] = None) -> torch.device:
        """Where the library runs for tensor ``t``: its own GPU, else the GPU the backbone lives on, else the current
        CUDA device -- the reference wrappers are built on the CPU (synergy3DMM.py:71-77) and still usable as is."""
        if t is not None and t.is_cuda:
            return t.device
        w = next(self.backbone.parameters())
        if w.is_cuda:
            return w.device
        if not torch.cuda.is_available():
            raise RuntimeError('synergynet_b200: no CUDA device (B200) visible; there is no CPU fallback')
        return torch.device('cuda', torch.cuda.current_device())

    def forward_test(self, input):
        """Testing time forward -> (param62, avgpool1280) (model_building.py:59-62).  A CPU input is moved to the
        compute GPU and the results come back on the CPU, as the reference's CPU model would return them."""
        dev = self._compute_device(input)
        if self._variant == 'resnet50':
            out, pool = self._engine(dev).forward_resnet50(input.to(dev))
            params = out[:, :62].contiguous()
        elif self._variant == 'resnest50':
            params, pool = self._engine(dev).forward_resnest50(input.to(dev))
        else:
            params, pool = self._engine(dev).forward(input.to(dev), want_pool=True)
        if not input.is_cuda:
            params, pool = params.to(input.device), pool.to(input.device)
        return params, pool

    def forward(self, input, target):
        """Training time forward (model_building.py:53-57): same backbone pass, GT cast."""
        params, pool = self.forward_test(input)
        return params, target.to(device=input.device, dtype=torch.float32), pool


class _SynergyBase(nn.Module):
    """Everything the two reference wrappers share: buffers, ``data_param``,
    ``reconstruct_vertex_62``, ``forward_test``, ``load_weights``, ``get_all_outputs``."""

    resize_interpolation = 'lanczos4'          # synergy3DMM.py:188; singleImage.py:77 uses linear

    def _setup(self, args, pack: ParamsPack, device: Optional[str]):
        tri = pack.tri if pack.tri is not None else np.zeros((3, 0), np.int64)
        self.triangles = torch.from_numpy(np.asarray(tri).astype(np.int64) - 1).long()
        self.I2P = I2P(args)
        self.forwardDirection = MLP_for(68)
        self.reverseDirection = MLP_rev(68)
        self.loss = {k: 0.0 for k in _LOSS_KEYS}
        for name in ('param_mean', 'param_std', 'w_shp', 'u', 'w_exp', 'u_base', 'w_shp_base', 'w_exp_base'):
            self.register_buffer(name, torch.from_numpy(np.ascontiguousarray(getattr(pack, name))).float())
        self.keypoints = torch.from_numpy(np.asarray(pack.keypoints)).long()
        self.std_size = pack.std_size
        self.face_detector = None
        if device is not None:
            self.triangles = self.triangles.to(device)
            self.to(device)
        self._refresh_data_param()
        object.__setattr__(self.I2P, '_basis_provider', self._basis)
        object.__setattr__(self.forwardDirection, '_engine_provider', self._pointnet_engine)
        object.__setattr__(self.reverseDirection, '_engine_provider', self._pointnet_engine)

    def _refresh_data_param(self):
        self.data_param = [self.param_mean, self.param_std, self.w_shp_base, self.u_base, self.w_exp_base]

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        if hasattr(self, 'param_mean'):
            self._refresh_data_param()
        return out

    def _basis(self):
        return {n: getattr(self, n) for n in ('param_mean', 'param_std', 'u_base', 'w_shp_base',
                                              'w_exp_base', 'u', 'w_shp', 'w_exp')}

    def _engine(self, device) -> Engine:
        return self.I2P._engine(device)

    def set_engine(self, kind: int) -> None:
        """0 = fp32 CUDA-core engine, 1 = tcgen05 split-fp16 engine (unfused), 2 = fused tcgen05 engine (default);
        see include/synergy_b200.h."""
        for eng in self.I2P._rt._engines.values():
            eng.set_engine(int(kind))
        self.I2P._rt.engine_kind = int(kind)

    # ---- reference API ---------------------------------------------------------------------------
    def reconstruct_vertex_62(self, param, whitening=True, dense=False, transform=True, lmk_pts=68):
        """Whitened param (B,62) -> (B,3,68) landmarks or (B,3,53215) vertices in crop image
        space (reference model_building.py:106-139)."""
        if param.shape[1] != 62:
            raise RuntimeError('length of params mismatch')
        dev = self._compute_device(param)
        out = self._engine(dev).reconstruct(param.to(dev), dense=dense, whitening=whitening, transform=transform)
        return out if param.is_cuda else out.to(param.device)

    def _compute_device(self, t: Optional[torch.Tensor] = None) -> torch.device:
        """GPU the library runs on for tensor ``t``: t's own device, else the device of the buffers, else the current
        CUDA device (the no-argument reference wrappers are constructed on the CPU, synergy3DMM.py:71-114)."""
        if t is not None and t.is_cuda:
            return t.device
        if self.param_mean.is_cuda:
            return self.param_mean.device
        if not torch.cuda.is_available():
            raise RuntimeError('synergynet_b200: no CUDA device (B200) visible; there is no CPU fallback')
        return torch.device('cuda', torch.cuda.current_device())

    def forward_test(self, input):
        """test time forward (model_building.py:159-162): whitened (B,62) parameters (on the input's device)."""
        if self.I2P._is_resnet:
            return self.I2P.forward_test(input)[0]
        dev = self._compute_device(input)
        out = self._engine(dev).forward(input.to(dev))
        return out if input.is_cuda else out.to(input.device)

    def forward_landmarks(self, input):
        """forward_test + reconstruct_vertex_62(dense=False) in one library call."""
        if self.I2P._is_resnet:
            return self.reconstruct_vertex_62(self.forward_test(input))
        dev = self._compute_device(input)
        out = self._engine(dev).forward_landmarks(input.to(dev))
        return out if input.is_cuda else out.to(input.device)

    def _pointnet_engine(self, t: torch.Tensor, net: int) -> Engine:
        """Engine of the compute device with the weights of head ``net`` (0 = forwardDirection, 1 = reverseDirection)."""
        eng = self._engine(self._compute_device(t))
        self.I2P._rt.ensure_pointnet(eng, net, self.forwardDirection if net == 0 else self.reverseDirection)
        return eng

    def forward(self, input, target):
        """The reference's training-time forward (model_building.py:141-157) in inference mode (eval BatchNorm, no
        autograd): backbone -> landmarks of prediction and ground truth -> WingLoss / ParamLoss -> MLP_for refinement
        -> MLP_rev -> the two cycle losses.  Returns the same dict of five (weighted) losses; the intermediate
        tensors are kept in ``self.last_forward`` for inspection."""
        dev = self._compute_device(input)
        eng = self._engine(dev)
        _3D_attr, avgpool = self.I2P.forward_test(input.to(dev))
        if avgpool.shape[1] != 1280:
            raise RuntimeError('SynergyNet.forward: MLP_for.conv6 is hard-wired to a 1280-d image feature '
                               f'(pointnet_backbone.py:15,58: 2418 = 64 + 1024 + 1280 + 40 + 10); the {self.I2P.args.arch} backbone '
                               f'pools {avgpool.shape[1]} channels, so the refinement head cannot follow it (the reference fails '
                               f'here too, SURVEY.md fact 4).  Use forward_test() / reconstruct_vertex_62() with {self.I2P.args.arch}.')
        _3D_attr_GT = target.to(device=dev, dtype=torch.float32)
        vertex_lmk = eng.reconstruct(_3D_attr, dense=False)
        vertex_GT_lmk = eng.reconstruct(_3D_attr_GT, dense=False)
        self.loss['loss_LMK_f0'] = 0.05 * eng.wing_loss(vertex_lmk, vertex_GT_lmk)
        self.loss['loss_Param_In'] = 0.02 * eng.param_loss(_3D_attr, _3D_attr_GT)
        eng = self._pointnet_engine(input, 0)
        point_residual, refined = eng.mlp_for(vertex_lmk, avgpool, _3D_attr)      # refined = lmk + 0.05 * residual (:150)
        self.loss['loss_LMK_pointNet'] = 0.05 * eng.wing_loss(refined, vertex_GT_lmk)
        eng = self._pointnet_engine(input, 1)
        _3D_attr_S2 = eng.mlp_rev(refined)
        self.loss['loss_Param_S2'] = 0.02 * eng.param_loss(_3D_attr_S2, _3D_attr_GT, mode='only_3dmm')
        self.loss['loss_Param_S1S2'] = 0.001 * eng.param_loss(_3D_attr_S2, _3D_attr, mode='only_3dmm')
        self.last_forward = {'_3D_attr': _3D_attr, 'avgpool': avgpool, 'vertex_lmk': vertex_lmk, 'vertex_GT_lmk': vertex_GT_lmk,
                             'point_residual': point_residual, 'vertex_lmk_refined': refined, '_3D_attr_S2': _3D_attr_S2}
        return self.loss

    def get_losses(self):
        return self.loss.keys()

    def load_weights(self, path):
        ckpt = torch.load(path, map_location=lambda storage, loc: storage)['state_dict']
        merged = self.state_dict()
        for k, v in ckpt.items():
            merged[k.replace('module.', '')] = v     # trained under DataParallel (:259-263)
        self.load_state_dict(merged, strict=False)

    def get_all_outputs(self, input, rects: Optional[Sequence[Sequence[float]]] = None):
        """3d landmarks, dense meshes and poses of every face in a BGR uint8 image
        (model_building.py:266-306 / synergy3DMM.py:167-207), batched over faces.

        ``rects`` are detector boxes ``[x0,y0,x1,y1,score]``.  The FaceBoxes detector is outside
        the hot path (SURVEY.md section 8 f3): pass ``rects`` or set ``self.face_detector``.
        """
        import cv2
        if rects is None:
            if self.face_detector is None:
                raise RuntimeError('no face detector configured: pass rects=[[x0,y0,x1,y1,score],...] '
                                   'or set model.face_detector to a callable(img)->rects')
            rects = self.face_detector(input)
        boxes = [square_roi(list(r)) for r in rects]
        if not boxes:
            return [], [], []
        interp = cv2.INTER_LANCZOS4 if self.resize_interpolation == 'lanczos4' else cv2.INTER_LINEAR
        # integer ROI crop + cv2 resize stay on the host (bit-exact index work / OpenCV's fixed-point Lanczos); everything
        # after it is batched on the GPU: uint8 -> (v-127.5)/128, backbone, both reconstructions already mapped to image
        # coordinates, pose decode.  One H2D of the uint8 crops, one D2H per output, no per-face arithmetic in Python.
        crops = np.stack([cv2.resize(crop_img(input, b), dsize=(120, 120), interpolation=interp) for b in boxes])
        dev = self._compute_device()
        eng = self._engine(dev)
        batch = torch.from_numpy(crops).permute(0, 3, 1, 2).contiguous().to(dev)                 # uint8 (B,3,120,120)
        _, params = eng.forward_landmarks(batch, want_params=True)
        roi5 = torch.from_numpy(roi_affine(boxes)).to(dev)
        lmk = eng.reconstruct_image(params, roi5, dense=False).cpu().numpy()
        mesh = eng.reconstruct_image(params, roi5, dense=True).cpu().numpy()
        ang, t3d = eng.pose_decode(params, roi5)
        ang, t3d = ang.cpu().numpy(), t3d.cpu().numpy()
        eng.raise_if_error()
        return list(lmk), list(mesh), [[ang[i].tolist(), t3d[i]] for i in range(len(boxes))]


class SynergyNet(_SynergyBase):
    """``SynergyNet(args)`` of the reference benchmark/training scripts (model_building.py:65-165):
    buffers are placed on CUDA at construction like the reference (:69,87-101)."""

    def __init__(self, args, _device: Optional[str] = 'cuda'):
        super().__init__()
        self.img_size = args.img_size
        self._setup(args, get_param_pack(), _device)


class WrapUpSynergyNet(_SynergyBase):
    """No-argument CPU-constructible wrapper (model_building.py:169-306)."""

    def __init__(self, checkpoint_fp: str = 'pretrained/best.pth.tar'):
        super().__init__()
        args = types.SimpleNamespace(arch='mobilenet_v2', checkpoint_fp=checkpoint_fp)
        self._setup(args, get_param_pack(), None)
        try:
            print('loading weights from ', args.checkpoint_fp)
            self.load_weights(args.checkpoint_fp)
        except Exception:
            pass
        self.eval()
