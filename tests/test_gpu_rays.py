"""`-m gpu`: ray batches (vr_render_rays / vr_camera_rays) on the product kernels.  A camera's own rays must
reproduce launch_renderer bit for bit (float output and counters); arbitrary rays match the reference's ray tap
(tests/golden/rays) bit for bit and the CPU oracle within the tolerances of the frame tests."""
import glob
import os

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
QUEUE, INLINE = 7, 3 + 16 * 193
NAMES = ["sh1_full4", "sh16_d6", "sh9_d6", "sh4_d5", "sh25_d5", "rgba_d5", "sg9_d5", "asg4_d5", "sg7_d5"]


def _torch():
    import torch
    return torch


def make_cam(W, H, pose, fx=None):
    from volrend_b200 import Camera, synth
    f = synth.focal_for(W) if fx is None else fx
    c = Camera(W, H, f, f)
    c.set_c2w(pose)
    return c


def frame(tree, cam, opt, variant=0):
    torch = _torch()
    from volrend_b200 import launch_renderer, lib
    lib().vr_set_variant(variant)
    img = torch.zeros((cam.height, cam.width, 4), dtype=torch.uint8, device="cuda")
    fo = torch.zeros((cam.height, cam.width, 4), dtype=torch.float32, device="cuda")
    cnt = torch.zeros(5, dtype=torch.int64, device="cuda")
    launch_renderer(tree, cam, opt, img, None, None, True, float_out=fo)
    launch_renderer(tree, cam, opt, img, None, None, True, counters=cnt)
    torch.cuda.synchronize()
    lib().vr_set_variant(0)
    return fo.cpu().numpy(), cnt.cpu().numpy().tolist()


def rays_render(tree, o, d, opt, t_max=None, variant=0):
    torch = _torch()
    from volrend_b200 import lib, render_rays
    lib().vr_set_variant(variant)
    out = torch.full(tuple(o.shape[:-1]) + (4,), -7.0, dtype=torch.float32, device="cuda")
    cnt = torch.zeros(5, dtype=torch.int64, device="cuda")
    render_rays(tree, o, d, opt, out, t_max=t_max)
    render_rays(tree, o, d, opt, out.clone(), t_max=t_max, counters=cnt)
    torch.cuda.synchronize()
    lib().vr_set_variant(0)
    return out.cpu().numpy(), cnt.cpu().numpy().tolist()


def cam_rays(cam, tile=None):
    torch = _torch()
    from volrend_b200 import camera_rays
    w, h = (cam.width, cam.height) if tile is None else tile[2:]
    o = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    d = torch.empty((h, w, 3), dtype=torch.float32, device="cuda")
    camera_rays(cam, o, d, tile=tile)
    return o, d


def variants(tree):
    from volrend_b200 import lib
    kb = tree.info()["kernel_basis"]
    return [v for v in (0, QUEUE, INLINE) if lib().vr_variant_supported(kb, v)]


@pytest.fixture(scope="module")
def dev_trees(small_trees):
    from volrend_b200 import N3Tree
    return {k: (st, N3Tree.from_synth(st)) for k, st in small_trees.items()}


def _pose(name):
    from volrend_b200 import synth
    return synth.config1_pose() if name == "sh1_full4" else synth.nerf_synthetic_test_poses(8)[(len(name) * 3) % 8]


@pytest.mark.parametrize("name", NAMES)
def test_camera_rays_reproduce_frame_bit_for_bit(built, dev_trees, name):
    from volrend_b200 import RenderOptions
    st, tree = dev_trees[name]
    cam = make_cam(72, 56, _pose(name))
    o, d = cam_rays(cam)
    for v in variants(tree):
        f, c = frame(tree, cam, RenderOptions(), v)
        g, cr = rays_render(tree, o, d, RenderOptions(), variant=v)
        assert np.array_equal(g, f), (name, v)
        assert cr == c, (name, v)


@pytest.mark.parametrize("optkw", [dict(step_size=1e-5), dict(step_size=1e-2), dict(stop_thresh=0.0),
                                   dict(stop_thresh=1e-1), dict(sigma_thresh=0.0), dict(sigma_thresh=1.0),
                                   dict(background_brightness=0.3), dict(render_bbox=[0.2, 0.1, 0, 0.9, 0.8, 0.7]),
                                   dict(basis_minmax=[2, 9]), dict(rot_dirs=[0.4, 0.1, -0.3]),
                                   dict(render_depth=True)])
def test_camera_rays_option_sweep(built, dev_trees, optkw):
    from volrend_b200 import RenderOptions, synth
    st, tree = dev_trees["sh16_d6"]
    cam = make_cam(64, 64, synth.nerf_synthetic_test_poses(8)[6])
    o, d = cam_rays(cam)
    for v in variants(tree):
        f, c = frame(tree, cam, RenderOptions(**optkw), v)
        g, cr = rays_render(tree, o, d, RenderOptions(**optkw), variant=v)
        assert np.array_equal(g, f) and cr == c, (optkw, v)


def test_camera_rays_tile_and_oracle(built, dev_trees):
    from oracle import binding as ob, ray_binding as rayb
    from volrend_b200 import synth
    st, tree = dev_trees["sh9_d6"]
    cam = make_cam(100, 76, _pose("sh9_d6"))
    o, d = cam_rays(cam)
    oc = ob.make_camera(100, 76, cam.fx, cam.fy, np.ascontiguousarray(cam.transform, np.float32).reshape(12))
    ro, rd = rayb.camera_rays(oc)
    assert np.array_equal(o.cpu().numpy().reshape(-1, 3), ro) and np.array_equal(d.cpu().numpy().reshape(-1, 3), rd)
    to, td = cam_rays(cam, (13, 7, 50, 33))
    assert np.array_equal(td.cpu().numpy(), d.cpu().numpy()[7:40, 13:63])


@pytest.mark.parametrize("name", ["config2_pose0", "config4_pose7"])
def test_camera_rays_at_benchmark_scale_hash_to_reference(built, name):
    from golden_cases import FRAMES_DIR, frame_case, frame_digest
    from volrend_b200 import N3Tree, RenderOptions
    st, W, H, fx, pose = frame_case(name)
    tree = N3Tree.from_synth(st)
    o, d = cam_rays(make_cam(W, H, pose, fx))
    z = np.load(os.path.join(FRAMES_DIR, name + ".npz"))
    for v in variants(tree):
        g, _ = rays_render(tree, o, d, RenderOptions(), variant=v)
        assert frame_digest(g.reshape(H, W, 4)) == str(z["f32_sha256"]), (name, v)
    tree.free_cuda()


def _golden_trees():
    from golden_cases import build_case
    from ray_cases import RAY_CASES
    from volrend_b200 import N3Tree
    out = []
    for p in sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "rays", "*.npz"))):
        z = np.load(p)
        st, W, H, pose, optkw, ndc = build_case(RAY_CASES[str(z["case"])])
        tree = N3Tree()
        npz = dict(child=st.child, data=st.data, offset=st.offset, invradius3=st.invradius3,
                   data_dim=np.int64(st.data_dim), data_format=np.array(st.data_format))
        if st.extra is not None:
            npz["extra_data"] = st.extra
        tree.load_npz(npz)
        if ndc is not None:
            tree.use_ndc = True
            tree.ndc_width, tree.ndc_height, tree.ndc_focal = ndc
        tree.load_cuda()
        kw = dict(optkw)
        if "render_depth" in kw:
            kw["render_depth"] = bool(kw["render_depth"])
        out.append((z, st, ndc, optkw, kw, tree))
    return out


def test_arbitrary_rays_match_reference_goldens_and_oracle(built):
    torch = _torch()
    from oracle import binding as ob, ray_binding as rayb
    from volrend_b200 import RenderOptions
    cases = _golden_trees()
    assert len(cases) >= 6
    for z, st, ndc, optkw, kw, tree in cases:
        o, d, t = (torch.from_numpy(z[k]).cuda() for k in ("origins", "dirs", "t_max"))
        go, co = rayb.render_rays(ob.OracleTree.from_synth(st, ndc=ndc), ob.make_options(**optkw), z["origins"],
                                  z["dirs"], z["t_max"])
        tol = 2e-5 if "rot_dirs" in optkw else 2e-6
        for v in variants(tree):
            g, c = rays_render(tree, o, d, RenderOptions(**kw), t, variant=v)
            assert np.array_equal(g, z["ref_f32"]), (str(z["case"]), v, float(np.abs(g - z["ref_f32"]).max()))
            assert np.abs(g - go).max() <= tol, (str(z["case"]), v)
            assert c[:4] == [co["samples"], co["child_loads"], co["shaded"], co["rays_hit"]], (str(z["case"]), v)
            # a permutation of the rays permutes the outputs: no per-lane state leaks from one ray to the next
            perm = torch.from_numpy(np.random.default_rng(1).permutation(o.shape[0])).cuda()
            gp, cp = rays_render(tree, o[perm], d[perm], RenderOptions(**kw), t[perm], variant=v)
            assert np.array_equal(gp, g[perm.cpu().numpy()]) and cp == c, (str(z["case"]), v)


def test_degenerate_rays_small_batches_and_stream_order(built, dev_trees):
    torch = _torch()
    from volrend_b200 import RenderOptions, render_rays
    st, tree = dev_trees["sh16_d6"]
    o = torch.tensor([[0.5, 0.5, 3.0]] * 6, device="cuda")
    d = torch.tensor([[0, 0, -1], [0, 0, 0], [float("nan"), 0, -1], [0, float("inf"), -1], [1e-30, 0, 0], [0, 0, -1]],
                     device="cuda")
    o[5, 0] = float("inf")
    for v in variants(tree):
        for depth, alpha in ((False, 0.0), (True, 1.0)):
            g, c = rays_render(tree, o, d, RenderOptions(background_brightness=0.25, render_depth=depth), variant=v)
            assert c[3] <= 1
            for row in g[1:]:
                assert row[3] == alpha and np.all(row[:3] == (0.0 if depth else 0.25)), (v, depth, row)
    cam = make_cam(40, 30, _pose("sh16_d6"))
    co, cd = cam_rays(cam)
    full, _ = rays_render(tree, co, cd, RenderOptions())
    fo, fd = co.reshape(-1, 3), cd.reshape(-1, 3)
    for v in variants(tree):
        for n in (0, 1, 31, 33, 1200):
            g, _ = rays_render(tree, fo[:n].contiguous(), fd[:n].contiguous(), RenderOptions(), variant=v)
            assert np.array_equal(g, full.reshape(-1, 4)[:n]), (v, n)
    # rays written by a torch op on the stream right before the call, no synchronisation in between
    torch.cuda.synchronize()
    src_o, src_d = fo.clone(), fd * 0.5
    for v in variants(tree):
        from volrend_b200 import lib
        lib().vr_set_variant(v)
        dst_o = torch.zeros_like(fo)
        dst_d = torch.zeros_like(fd)
        out = torch.zeros((fo.shape[0], 4), device="cuda")
        for _ in range(3):
            dst_o.zero_(); dst_d.zero_()
            dst_o.copy_(src_o); torch.mul(src_d, 2.0, out=dst_d)
            render_rays(tree, dst_o, dst_d, RenderOptions(), out)
        torch.cuda.synchronize()
        lib().vr_set_variant(0)
        assert np.array_equal(out.cpu().numpy(), full.reshape(-1, 4)), v


def test_python_validation(built, dev_trees):
    torch = _torch()
    from volrend_b200 import RenderOptions, camera_rays, render_rays
    st, tree = dev_trees["sh4_d5"]
    o = torch.zeros((10, 3), device="cuda")
    d = torch.ones((10, 3), device="cuda")
    out = torch.zeros((10, 4), device="cuda")
    opt = RenderOptions()
    bad = [(o.cpu(), d, out, None), (o.double(), d, out, None), (o, d, out[:, :3], None),
           (torch.zeros((3, 10), device="cuda").t(), d, out, None), (o, d[:9], out, None),
           (o, d, torch.zeros((10, 4), device="cuda")[::1, :].t().contiguous().t(), None), (o, d, out, torch.zeros(9, device="cuda")),
           (o, d, out, torch.zeros(10, device="cuda", dtype=torch.float16))]
    for oo, dd, oo4, tt in bad:
        with pytest.raises(ValueError):
            render_rays(tree, oo, dd, opt, oo4, t_max=tt)
    if torch.cuda.device_count() > 1:
        with pytest.raises(ValueError):
            render_rays(tree, o.to("cuda:1"), d, opt, out)
    from volrend_b200 import Camera
    cam = Camera(4, 3)
    with pytest.raises(ValueError):
        camera_rays(cam, torch.zeros((11, 3), device="cuda"), torch.zeros((11, 3), device="cuda"))
    with pytest.raises(ValueError):
        camera_rays(cam, torch.zeros((12, 3)), torch.zeros((12, 3)))
    render_rays(tree, o[:0], d[:0], opt, out[:0])      # zero rays: a no-op
