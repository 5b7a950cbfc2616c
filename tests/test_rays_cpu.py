"""`-m "not gpu"`: ray batches on the CPU side -- the oracle's ray entry points against its per-pixel renderer and
the reference's stored ray outputs, and the C-ABI's ray calls without a device."""
import ctypes as C
import glob
import os

import numpy as np
import pytest

from conftest import ROOT


def _oracle():
    from oracle import binding as ob, ray_binding as rayb
    return ob, rayb


def _cam(ob, W, H, pose):
    from volrend_b200 import synth
    return ob.make_camera(W, H, synth.focal_for(W), synth.focal_for(W), synth.c2w_to_colmajor12(pose))


def _pose(name):
    from volrend_b200 import synth
    return synth.config1_pose() if name == "sh1_full4" else synth.nerf_synthetic_test_poses(8)[(len(name) * 3) % 8]


@pytest.mark.parametrize("name", ["sh1_full4", "sh16_d6", "sh9_d6", "sh4_d5", "sh25_d5", "rgba_d5", "sg9_d5",
                                  "asg4_d5", "sg7_d5"])
def test_camera_rays_reproduce_oracle_frame(built, small_trees, name):
    ob, rayb = _oracle()
    t = ob.OracleTree.from_synth(small_trees[name])
    cam = _cam(ob, 40, 32, _pose(name))
    f, _, c = ob.render(t, cam, ob.make_options())
    o, d = rayb.camera_rays(cam)
    g, cr = rayb.render_rays(t, ob.make_options(), o, d)
    assert np.array_equal(g, f.reshape(-1, 4)) and cr == c
    # a tile's rays are the tile's pixels, row-major
    o2, d2 = rayb.camera_rays(cam, (5, 3, 17, 11))
    assert np.array_equal(d2.reshape(11, 17, 3), d.reshape(32, 40, 3)[3:14, 5:22])


def test_camera_rays_ndc_and_depth_limit(built, small_trees):
    """NDC tree, and t_max = a composite depth map: both equal the per-pixel renderer (offscreen background)."""
    from golden_cases import build_case
    ob, rayb = _oracle()
    st, W, H, pose, _, ndc = build_case("lego_sh16_ndc")
    t = ob.OracleTree.from_synth(st, ndc=ndc)
    cam = _cam(ob, W, H, pose)
    f, _, c = ob.render(t, cam, ob.make_options())
    o, d = rayb.camera_rays(cam)
    g, cr = rayb.render_rays(t, ob.make_options(), o, d)
    assert np.array_equal(g, f.reshape(-1, 4)) and cr == c
    st = small_trees["sh9_d6"]
    t = ob.OracleTree.from_synth(st)
    cam = _cam(ob, 48, 40, _pose("sh9_d6"))
    depth = np.random.default_rng(5).uniform(2.0, 5.5, (40, 48)).astype(np.float32)
    white = np.full((40, 48, 4), 255, np.uint8)                   # composite over white == background 1.0
    fc, _, cc = ob.render(t, cam, ob.make_options(), rgba_in=white, depth_in=depth)
    o, d = rayb.camera_rays(cam)
    g, cr = rayb.render_rays(t, ob.make_options(), o, d, depth)
    assert np.abs(g - fc.reshape(-1, 4)).max() <= 1e-6 and cr == cc
    assert np.array_equal(g[:, 3], fc.reshape(-1, 4)[:, 3])


def test_degenerate_rays_are_background_misses(built, small_trees):
    ob, rayb = _oracle()
    t = ob.OracleTree.from_synth(small_trees["sh16_d6"])
    o = np.array([[0.5, 0.5, 3.0]] * 6, np.float32)
    d = np.array([[0, 0, -1], [0, 0, 0], [np.nan, 0, -1], [0, np.inf, -1], [1e-30, 0, 0], [0, 0, -1]], np.float32)
    o[5, 0] = np.inf
    for depth, alpha in ((0, 0.0), (1, 1.0)):
        g, c = rayb.render_rays(t, ob.make_options(background_brightness=0.25, render_depth=depth), o, d)
        assert c["rays_hit"] <= 1
        for row in g[1:]:
            assert row[3] == alpha and np.all(row[:3] == (0.0 if depth else 0.25))


def test_oracle_matches_reference_ray_goldens(built):
    """tests/golden/rays: the reference's trace_ray on the seeded rays vs the CPU oracle, <= 1e-4."""
    from golden_cases import build_case
    from ray_cases import RAY_CASES
    ob, rayb = _oracle()
    paths = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "rays", "*.npz")))
    assert len(paths) == len(RAY_CASES)
    for p in paths:
        z = np.load(p)
        st, W, H, pose, optkw, ndc = build_case(RAY_CASES[str(z["case"])])
        t = ob.OracleTree.from_synth(st, ndc=ndc)
        g, _ = rayb.render_rays(t, ob.make_options(**optkw), z["origins"], z["dirs"], z["t_max"])
        err = np.abs(g - z["ref_f32"]).max()
        assert err <= 1e-4, (p, err)


def test_ray_calls_without_a_device(built):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from volrend_b200 import _capi, lib
    l = lib()
    o = _capi.vr_options()
    l.vr_default_options(C.byref(o))
    fake = C.create_string_buffer(4096)          # never dereferenced without a device
    buf = C.create_string_buffer(64)
    assert l.vr_render_rays(fake, buf, buf, None, 4, C.byref(o), buf, None, None) == _capi.VR_ENODEVICE
    assert b"no CPU fallback" in l.vr_last_error()
    assert l.vr_render_rays(None, buf, buf, None, 4, C.byref(o), buf, None, None) == _capi.VR_EINVAL
    assert l.vr_render_rays(fake, buf, buf, None, -1, C.byref(o), buf, None, None) == _capi.VR_EINVAL
    assert l.vr_render_rays(fake, None, None, None, 0, C.byref(o), None, None, None) == _capi.VR_OK
    cam = _capi.vr_camera(8, 6, 10.0, 10.0)
    assert l.vr_camera_rays(C.byref(cam), None, buf, buf, None) == _capi.VR_ENODEVICE
    assert l.vr_camera_rays(C.byref(cam), C.byref(_capi.vr_rect(4, 0, 5, 6)), buf, buf, None) == _capi.VR_EINVAL
    assert l.vr_camera_rays(C.byref(cam), None, None, buf, None) == _capi.VR_EINVAL
