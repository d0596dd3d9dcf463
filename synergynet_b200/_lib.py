"""ctypes binding of ``libsynergy_b200.so`` (include/synergy_b200.h).

There is no fallback: if the library is missing or cannot be loaded, importing the symbols
raises, and every product entry point above it fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('SYN_LIB_PATH') or os.path.join(_PKG, 'libsynergy_b200.so')   # override: A/B runs of two builds
HEADER_PATH = os.path.join(_PKG, '..', 'include', 'synergy_b200.h')

SYN_OK = 0
ERR_NAMES = {1: 'SYN_ERR_INVALID', 2: 'SYN_ERR_CUDA', 3: 'SYN_ERR_STATE', 4: 'SYN_ERR_SHAPE',
             5: 'SYN_ERR_NOMEM', 6: 'SYN_ERR_UNSUPPORTED'}
ENGINE_SIMT_FP32, ENGINE_TC_BF16X3, ENGINE_TC_FUSED, ENGINE_TC_FUSED_1PASS = 0, 1, 2, 3


class SynergyLibError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f'{ERR_NAMES.get(code, code)}: {msg}')
        self.code = code


class ConvDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ('cin', 'cout', 'ksize', 'stride', 'groups', 'relu6',
                                         'h_in', 'h_out', 'residual')]


class LightCfg(C.Structure):
    """``syn_light_cfg_t`` (Sim3DR/lighting.py:24-32)."""
    _fields_ = [('intensity_ambient', C.c_float), ('intensity_directional', C.c_float), ('intensity_specular', C.c_float),
                ('color_ambient', C.c_float * 3), ('color_directional', C.c_float * 3), ('light_pos', C.c_float * 3),
                ('view_pos', C.c_float * 3), ('specular_exp', C.c_int32)]


class FbLayerDesc(C.Structure):
    """``syn_fb_layer_desc_t``."""
    _fields_ = [('name', C.c_char_p)] + [(n, C.c_int32) for n in ('cin', 'cout', 'ksize', 'stride', 'pad', 'has_bn', 'activation')]


class ResNeStLayerDesc(C.Structure):
    """``syn_resnest_layer_desc_t``."""
    _fields_ = [('name', C.c_char_p), ('bn_name', C.c_char_p)] + [
        (n, C.c_int32) for n in ('cin', 'cout', 'ksize', 'stride', 'groups', 'has_bias', 'h_in', 'h_out')]


NMS_CPU_NMS, NMS_PY_CPU_NMS = 0, 1

_P, _F, _I, _L = C.c_void_p, C.c_void_p, C.c_int, C.c_int64
# name -> (restype, argtypes); float*/void* travel as integer addresses (tensor.data_ptr()).
SIGNATURES = {
    'syn_abi_version': (_I, []),
    'syn_last_error': (C.c_char_p, []),
    'syn_num_conv_layers': (_I, []),
    'syn_conv_desc': (_I, [_I, C.POINTER(ConvDesc)]),
    'syn_create': (_I, [_I, C.POINTER(_P)]),
    'syn_destroy': (None, [_P]),
    'syn_set_conv_bn': (_I, [_P, _I, _F, _L, _F, _F, _F, _F, C.c_float]),
    'syn_set_heads': (_I, [_P, _F, _F, _F, _F, _F, _F]),
    'syn_set_whitening': (_I, [_P, _F, _F]),
    'syn_set_basis_sparse': (_I, [_P, _F, _F, _F, _I]),
    'syn_set_basis_dense': (_I, [_P, _F, _F, _F, _L]),
    'syn_commit': (_I, [_P]),
    'syn_set_engine': (_I, [_P, _I]),
    'syn_get_engine': (_I, [_P]),
    'syn_forward': (_I, [_P, _F, _I, _F, _F, _P]),
    'syn_reconstruct': (_I, [_P, _F, _I, _I, _I, _I, _F, _P]),
    'syn_forward_landmarks': (_I, [_P, _F, _I, _F, _F, _P]),
    'syn_forward_landmarks_host': (_I, [_P, _F, _I, _F, _F]),
    'syn_forward_landmarks_u8': (_I, [_P, _F, _I, _F, _F, _P]),
    'syn_forward_landmarks_host_u8': (_I, [_P, _F, _I, _F, _F]),
    'syn_forward_landmarks_host_submit': (_I, [_P, _F, _I, _I, _F, _F, C.POINTER(C.c_int)]),
    'syn_host_wait': (_I, [_P, _I]),
    'syn_pointnet_set_layer': (_I, [_P, _I, _I, _F, _I, _I, _F, _F, _F, _F, _F, C.c_float]),
    'syn_pointnet_commit': (_I, [_P, _I]),
    'syn_mlp_for': (_I, [_P, _F, _F, _F, _I, _F, _F, _P]),
    'syn_mlp_rev': (_I, [_P, _F, _I, _F, _P]),
    'syn_wing_loss': (_I, [_P, _F, _F, _I, _I, _F, _P]),
    'syn_param_loss': (_I, [_P, _F, _F, _I, _I, _F, _P]),
    'syn_reconstruct_image': (_I, [_P, _F, _I, _I, _F, _F, _P]),
    'syn_pose_decode': (_I, [_P, _F, _I, _F, _F, _F, _P]),
    'syn_set_center_crop': (_I, [_P, _I]),
    'syn_resnet_num_convs': (_I, []),
    'syn_resnet_conv_desc': (_I, [_I, C.POINTER(ConvDesc)]),
    'syn_resnet_set_conv': (_I, [_P, _I, _F, _L, _F, _F, _F, _F, C.c_float]),
    'syn_resnet_set_heads': (_I, [_P, _F, _F]),
    'syn_resnet_commit': (_I, [_P]),
    'syn_resnet50_forward': (_I, [_P, _F, _I, _F, _F, _P]),
    'syn_resnest_num_layers': (_I, []),
    'syn_resnest_layer_desc': (_I, [_I, C.POINTER(ResNeStLayerDesc)]),
    'syn_resnest_set_layer': (_I, [_P, _I, _F, _L, _F, _F, _F, _F, _F, C.c_float]),
    'syn_resnest_set_heads': (_I, [_P, _F, _F]),
    'syn_resnest_commit': (_I, [_P]),
    'syn_resnest50_forward': (_I, [_P, _F, _I, _F, _F, _P]),
    'syn_debug_heads_buffer': (_I, [_P, _I, _F, _L]),
    'syn_mesh_incidence_host': (_I, [_F, _I, _I, _F, _F]),
    'syn_mesh_normals': (_I, [_F, _L, _I, _I, _I, _I, _F, _I, _F, _F, _F, _F, _P]),
    'syn_mesh_lighting': (_I, [_F, _L, _I, _I, _I, _I, _F, C.POINTER(LightCfg), _F, _F, _F, _P]),
    'syn_rasterize': (_I, [_F, _I, _I, _I, _F, _L, _I, _I, _I, _I, _F, _I, _F, C.c_float, _I, _F, _F, _P]),
    'syn_nms': (_I, [_F, _I, C.c_double, _I, _F, _F, _F, _P]),
    'syn_faceboxes_num_priors': (_I, [_I, _I]),
    'syn_fb_num_layers': (_I, []),
    'syn_fb_layer_desc': (_I, [_I, C.POINTER(FbLayerDesc)]),
    'syn_fb_create': (_I, [_I, C.POINTER(_P)]),
    'syn_fb_destroy': (None, [_P]),
    'syn_fb_set_layer': (_I, [_P, _I, _F, _L, _F, _F, _F, _F, _F, C.c_float]),
    'syn_fb_commit': (_I, [_P]),
    'syn_fb_forward': (_I, [_P, _F, _I, _I, _F, _F, _P]),
    'syn_fb_launch_count': (_L, [_P]),
    'syn_faceboxes_decode': (_I, [_F, _F, _I, _I, C.c_float, C.c_float, C.c_float, C.c_float, _I, _F, _F, _F, _P]),
    'syn_launch_count': (_L, [_P]),
    'syn_set_timing': (_I, [_P, _I]),
    'syn_get_timings': (_I, [_P, C.POINTER(C.c_float), C.POINTER(C.c_char_p), _I, C.POINTER(C.c_int)]),
    'syn_poll_error': (_I, [_P, C.POINTER(C.c_int)]),
    'syn_peek_error': (_I, [_P, C.POINTER(C.c_int)]),
    'syn_poll_saturation': (_I, [_P, C.POINTER(C.c_int)]),
    'syn_debug_forward_until': (_I, [_P, _F, _I, _I, _F, _P]),
    'syn_debug_tile_plan': (_I, [_I, _I, _I, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
}


# entry points every build must export (everything the compute path binds)
_CORE = {n for n in SIGNATURES if n not in ('syn_peek_error', 'syn_poll_saturation', 'syn_pointnet_set_layer',
                                             'syn_pointnet_commit', 'syn_mlp_for', 'syn_mlp_rev', 'syn_wing_loss',
                                             'syn_param_loss', 'syn_reconstruct_image', 'syn_pose_decode', 'syn_set_center_crop', 'syn_resnet_num_convs', 'syn_resnet_conv_desc',
                                             'syn_resnet_set_conv', 'syn_resnet_set_heads', 'syn_resnet_commit', 'syn_resnet50_forward', 'syn_debug_heads_buffer',
                                             'syn_resnest_num_layers', 'syn_resnest_layer_desc', 'syn_resnest_set_layer',
                                             'syn_resnest_set_heads', 'syn_resnest_commit', 'syn_resnest50_forward',
                                             'syn_mesh_incidence_host', 'syn_mesh_normals', 'syn_mesh_lighting', 'syn_rasterize', 'syn_nms',
                                             'syn_faceboxes_num_priors', 'syn_faceboxes_decode', 'syn_fb_num_layers', 'syn_fb_layer_desc', 'syn_fb_create',
                                             'syn_fb_destroy', 'syn_fb_set_layer', 'syn_fb_commit', 'syn_fb_forward', 'syn_fb_launch_count')}


def declared_symbols(header: str = HEADER_PATH):
    """Function names declared in include/synergy_b200.h (used by the symbol-export test)."""
    text = open(header).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(syn_[a-z0-9_]+)\s*\(', text)))


_lib = None


def load() -> C.CDLL:
    """Load the library once; raise (never fall back) if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f'{LIB_PATH} not found: build it with `python -m synergynet_b200.build` '
            '(nvcc, sm_100a). There is no CPU or eager fallback for this path.')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            # an older A/B build (SYN_LIB_PATH) may predate an introspection entry point; using it then raises
            # AttributeError at the call site.  tests/test_cabi_symbols.py holds the shipped library to the header.
            if name in _CORE:
                raise
            continue
        fn.restype, fn.argtypes = res, args
    if lib.syn_abi_version() != 1:
        raise RuntimeError('libsynergy_b200.so ABI version mismatch; rebuild')
    _lib = lib
    return lib


def check(code: int) -> None:
    if code != SYN_OK:
        raise SynergyLibError(code, load().syn_last_error().decode(errors='replace'))
