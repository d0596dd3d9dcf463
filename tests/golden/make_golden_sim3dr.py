#!/usr/bin/env python
"""Generate ``tests/golden/sim3dr_ref_vectors.npz``: the reference's own ``Sim3DR/lib/rasterize_kernel.cpp``, compiled
unmodified into ``oracle/_ref/libsim3dr_ref.so`` by ``oracle/Makefile`` (so it needs the reference tree the Makefile's
``REF`` points at), run on ``oracle.golden.sim3dr_inputs()``:

    python tests/golden/make_golden_sim3dr.py

Stored: vertex normals, the depth buffer and the image minus its background (uint8, modulo 256: zero wherever no triangle
was drawn, so the file stays small) for both orientations of the depth test.  The inputs are rebuilt from their seeds
by the tests; only their SHA-256 is stored.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import golden  # noqa: E402
from oracle import render_port as rp  # noqa: E402


def main():
    rp.build()
    if not rp.have_ref():
        sys.exit(f'{rp.REF_LIB} was not built: no reference tree at the path oracle/Makefile expects')
    inp = golden.sim3dr_inputs()
    normals, diff, depth = [], [], []
    for b in range(inp['verts'].shape[0]):
        ver = np.ascontiguousarray(inp['verts'][b].T)
        normals.append(rp.get_normal(ver, inp['tri'], 'ref'))
        d_b, z_b = [], []
        for rev in (False, True):
            img, z = rp.rasterize(ver, inp['tri'], inp['colors'][b], inp['bg'][b].copy(), reverse=rev, kind='ref',
                                  return_depth=True)
            d_b.append(img - inp['bg'][b])
            z_b.append(z)
        diff.append(np.stack(d_b))
        depth.append(np.stack(z_b))
    out = {k + '_sha256': np.array(golden.sha256(v)) for k, v in inp.items()}
    out.update(normals=np.stack(normals), image_minus_bg=np.stack(diff), depth=np.stack(depth))
    np.savez_compressed(golden.SIM3DR_REF_VECTORS, **out)
    print('wrote', golden.SIM3DR_REF_VECTORS, os.path.getsize(golden.SIM3DR_REF_VECTORS) // 1024, 'KiB')


if __name__ == '__main__':
    main()
