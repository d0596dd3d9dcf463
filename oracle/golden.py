"""Loaders of the golden vectors under ``tests/golden/`` and the seeded inputs they were recorded on.  TEST INFRASTRUCTURE.

The recording scripts (``tests/golden/make_golden*.py``) and the tests take their inputs from here, so that both sides
run on the same arrays.  Inputs that the seeded generators rebuild exactly are not stored: the ``.npz`` keeps their
SHA-256, and the loaders check the rebuilt arrays against it, so a generator that drifts fails loudly instead of
comparing the reference's outputs with the wrong inputs.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np
import torch

from synergynet_b200 import synthetic

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'tests', 'golden')
REF_VECTORS = os.path.join(GOLDEN_DIR, 'ref_vectors.npz')
SIM3DR_REF_VECTORS = os.path.join(GOLDEN_DIR, 'sim3dr_ref_vectors.npz')


def sha256(a: np.ndarray) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _with_inputs(path: str, inputs: dict) -> dict:
    gold = dict(np.load(path, allow_pickle=False))
    for k, v in inputs.items():
        if sha256(v) != str(gold[k + '_sha256']):
            raise AssertionError(f'{os.path.basename(path)}: the regenerated input {k!r} is not the one it was recorded on')
        gold[k] = v
    return gold


def ref_inputs() -> dict:
    """The inputs ``tests/golden/make_golden.py`` runs the reference on: 8 crops (6 structured, 2 noise), the image of
    the ``crop_img`` cases and the 360 x 360 scene of the ``get_all_outputs`` case."""
    x_u8 = torch.cat([synthetic.make_structured_crops_u8(6, seed=11), synthetic.make_crops_u8(2, seed=0)]).numpy()
    rng = np.random.default_rng(3)
    crop_img = rng.integers(0, 256, (97, 131, 3), dtype=np.uint8)
    scene = (np.clip(synthetic.make_structured_crops_u8(1, seed=21)[0].permute(1, 2, 0).numpy()
                     .repeat(3, 0).repeat(3, 1).astype(np.int32)
                     + rng.integers(-8, 9, (360, 360, 3)), 0, 255)).astype(np.uint8)
    return {'x_u8': x_u8, 'crop_img': crop_img, 'scene': scene}


def load_ref_vectors() -> dict:
    """``ref_vectors.npz`` with its inputs rebuilt.  Of the 1024-face batch it holds all parameters and the landmarks of
    the even-numbered faces (``lmk1024_even``)."""
    return _with_inputs(REF_VECTORS, ref_inputs())


def sim3dr_inputs() -> dict:
    """Two meshes on a 200 x 240 canvas with a few huge and degenerate triangles on top of the grid, and per mesh random
    vertex colours and a random background."""
    tri = synthetic.make_render_topology(60, 70)
    extra = np.array([[0, 4199, 2100], [10, 10, 500], [69, 4130, 35]], np.int32)
    tri = np.ascontiguousarray(np.concatenate([tri, extra]))
    verts = synthetic.make_render_meshes(2, 200, 240, seed=5, rows=60, cols=70, size=120)
    rng = np.random.default_rng(3)
    colors, bgs = [], []
    for b in range(verts.shape[0]):
        colors.append(rng.uniform(0, 1, (verts.shape[2], 3)).astype(np.float32))
        bgs.append(rng.integers(0, 256, (200, 240, 3), dtype=np.uint8))
    return {'tri': tri, 'verts': verts, 'colors': np.stack(colors), 'bg': np.stack(bgs)}


def load_sim3dr_ref_vectors() -> dict:
    """``sim3dr_ref_vectors.npz`` (the reference's own ``rasterize_kernel.cpp`` on :func:`sim3dr_inputs`) with its inputs
    rebuilt.  ``normals`` is (mesh, vertex, 3); ``image_minus_bg`` (uint8, modulo 256) and ``depth`` are indexed
    [mesh, reverse]."""
    return _with_inputs(SIM3DR_REF_VECTORS, sim3dr_inputs())
