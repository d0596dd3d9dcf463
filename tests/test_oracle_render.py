"""Pin the render / detection oracle (oracle/render_port.py, oracle/sim3dr_port.c) to the vectors recorded from the live
reference (tests/golden/make_golden_render.py) and from the reference's own C++ compiled unmodified
(tests/golden/make_golden_sim3dr.py).  CPU only."""
import os

import numpy as np
import pytest

from oracle import golden
from oracle import render_port as rp
from synergynet_b200 import synthetic

GOLD = os.path.join(os.path.dirname(__file__), 'golden', 'render_vectors.npz')
LIGHT_TOL = 2e-7      # absolute, on light in [0,1]: numpy's float32 pow differs by an ulp between hosts (SVML or libm)


@pytest.fixture(scope='module')
def gold():
    return dict(np.load(GOLD, allow_pickle=False))


def test_inputs_are_reproducible(gold):
    assert np.array_equal(synthetic.make_render_topology(40, 50), gold['render_tri'])
    assert np.array_equal(synthetic.make_render_meshes(3, 96, 128, seed=2, rows=40, cols=50, size=60), gold['render_verts'])


def test_normals_bit_exact(gold):
    for b in range(3):
        ver = np.ascontiguousarray(gold['render_verts'][b].T)
        assert np.array_equal(rp.get_normal(ver, gold['render_tri']), gold['render_normals'][b])


def test_lighting_matches_reference(gold):
    for b in range(3):
        ver = np.ascontiguousarray(gold['render_verts'][b].T)
        light = rp.lighting(ver, gold['render_normals'][b])
        assert np.abs(light - gold['render_light'][b]).max() <= LIGHT_TOL


def test_rasterize_bit_exact(gold):
    ver0 = np.ascontiguousarray(gold['render_verts'][0].T)
    for key, rev in (('raster_plain', False), ('raster_reverse', True)):
        out = rp.rasterize(ver0, gold['render_tri'], gold['raster_colors'], gold['render_bg'].copy(), reverse=rev)
        assert np.array_equal(out, gold[key])
    assert (gold['raster_plain'] != gold['render_bg']).any()


def test_pipeline_sequence(gold):
    """utils/render.py:40-45: meshes drawn one after the other; the light fed to the rasteriser is the recorded one, so the
    uint8 result is bit-exact."""
    img = gold['render_bg'].copy()
    for b in range(3):
        ver = np.ascontiguousarray(gold['render_verts'][b].T)
        img = rp.rasterize(ver, gold['render_tri'], gold['render_light'][b], img)
        assert np.array_equal(img, gold['render_steps'][b])


def test_port_equals_compiled_reference():
    """Bit for bit against the reference's own rasterize_kernel.cpp (tests/golden/make_golden_sim3dr.py), on meshes with
    a few huge and degenerate triangles on top of the grid."""
    ref = golden.load_sim3dr_ref_vectors()
    tri = ref['tri']
    for b in range(2):
        ver = np.ascontiguousarray(ref['verts'][b].T)
        assert np.array_equal(rp.get_normal(ver, tri, 'port'), ref['normals'][b], equal_nan=True)
        bg = ref['bg'][b]
        for rev in (False, True):
            a, da = rp.rasterize(ver, tri, ref['colors'][b], bg.copy(), reverse=rev, kind='port', return_depth=True)
            assert np.array_equal(a - bg, ref['image_minus_bg'][b, int(rev)]) and np.array_equal(da, ref['depth'][b, int(rev)])
    assert ref['image_minus_bg'].any()


def test_prior_boxes_bit_exact(gold):
    for (h, w) in ((96, 160), (250, 333)):
        assert np.array_equal(rp.prior_boxes(h, w), gold[f'priors_{h}x{w}'])


def test_decode(gold):
    boxes = rp.decode_boxes(gold['decode_loc'], gold['priors_250x333']).numpy()
    assert np.allclose(boxes, gold['decode_boxes'], rtol=1e-6, atol=1e-6)


def test_nms_restatements(gold):
    for thr, key in ((0.3, 'nms_keep_3'), (0.5, 'nms_keep_5')):
        want = gold[key].tolist()
        assert rp.py_cpu_nms(gold['nms_dets'], thr) == want
        assert rp.cpu_nms(gold['nms_dets'], thr, ge=False) == want
        # the .pyx convention differs from py_cpu_nms only when an overlap equals the threshold exactly
        assert rp.cpu_nms(gold['nms_dets'], thr, ge=True) == want


def test_nms_threshold_equality_conventions():
    # two 10x10 boxes (pixel-inclusive) sharing 50 of 150 union pixels: ovr = 1/3 exactly representable? use thresh = ovr
    d = np.array([[0, 0, 9, 9, 0.9], [5, 0, 14, 9, 0.8]], np.float32)
    ovr = np.float32(50.0) / np.float32(150.0)
    assert rp.cpu_nms(d, float(ovr), ge=True) == [0]            # cpu_nms.pyx:65 suppresses on >=
    assert rp.cpu_nms(d, float(ovr), ge=False) == [0, 1]        # py_cpu_nms.py:35 keeps <=
    assert rp.py_cpu_nms(d, float(ovr)) == [0, 1]


def test_faceboxes_chain(gold):
    h, w = gold['fb_image'].shape[:2]
    for tag in ('net', 'rnd'):
        d = rp.faceboxes_dets(gold['fb_loc'], gold[f'fb_{tag}_conf'], h, w)
        want = gold[f'fb_{tag}_dets_sorted']
        assert d.shape == want.shape
        if d.shape[0]:
            assert np.allclose(d, want, rtol=1e-6, atol=1e-5)
            assert rp.py_cpu_nms(d, 0.3) == gold[f'fb_{tag}_keep'].tolist()


# ---- the detector network ------------------------------------------------------------------------------------------------
def _max_rel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


@pytest.mark.parametrize('hw', [(250, 333, 0), (120, 96, 1)])
def test_detector_network_oracle(gold, hw):
    h, w, seed = hw
    sd = synthetic.make_faceboxes_state_dict(0)
    loc, conf = rp.faceboxes_forward(sd, synthetic.make_scene_u8(h, w, seed))
    assert loc.shape == gold[f'fbs_loc_{h}x{w}'].shape
    assert _max_rel(loc, gold[f'fbs_loc_{h}x{w}']) <= 2e-5 and _max_rel(conf, gold[f'fbs_conf_{h}x{w}']) <= 2e-5


def test_detector_end_to_end_oracle(gold):
    sd = synthetic.make_faceboxes_state_dict(0)
    got = np.array(rp.faceboxes_detect(sd, synthetic.make_scene_u8(120, 96, 1)), np.float32).reshape(-1, 5)
    want = gold['fbs_final_120x96']
    assert got.shape == want.shape and np.allclose(got, want, rtol=1e-5, atol=1e-4)


def test_detector_key_schema():
    from synergynet_b200 import faceboxes
    keys = faceboxes.state_dict_keys()
    assert len(keys) == 27 * 6 + 6 * 2 and keys[0] == 'conv1.conv.weight' and keys[-1] == 'conf.2.bias'
    assert set(keys) == set(synthetic.make_faceboxes_state_dict(0).keys())
