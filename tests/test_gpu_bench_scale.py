"""`-m gpu`: parity of the DEFAULT kernel at the sizes bench.py and BASELINE.json quote (VERDICT r1 item 3).

  config 2   depth-10 SH16 bench tree, 800x800      full frames vs the reference kernel, bit for bit
  config 4   depth-11 SH25 tree, 1920x1080           full frame vs the reference kernel; vr_render_bands for 2/4/8 parts
                                                     reassembles to exactly that frame

The reference kernel's frames are stored as whole-frame digests plus a pixel sample (tests/golden/frames).
The same frames are also checked against the CPU oracle on windows that include the image borders and the
silhouette (tolerance 1e-4 required, 2e-6 achieved).  These trees exercise what the small cases cannot:
6 levels of wide tables, table ids > 2^17, record offsets > 2^31 bytes."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
TOL = 1e-4


def _cam(W, H, fx, pose):
    from volrend_b200 import Camera
    c = Camera(W, H, fx, fx)
    c.set_c2w(pose)
    return c


def _render_default(tree, cam, want_counters=False):
    import torch
    from volrend_b200 import RenderOptions, launch_renderer, lib
    assert lib().vr_get_variant() == 0, "a previous test left a non-default kernel variant selected"
    H, W = cam.height, cam.width
    img = torch.zeros((H, W, 4), dtype=torch.uint8, device="cuda")
    fo = torch.zeros((H, W, 4), dtype=torch.float32, device="cuda")
    launch_renderer(tree, cam, RenderOptions(), img, None, None, True, float_out=fo)
    cnt = None
    if want_counters:
        c = torch.zeros(5, dtype=torch.int64, device="cuda")
        launch_renderer(tree, cam, RenderOptions(), img, None, None, True, counters=c)
        cnt = c.cpu().tolist()
    torch.cuda.synchronize()
    return fo.cpu().numpy(), img.cpu().numpy(), cnt


def _check_against_reference_and_oracle(st, tree, cams, names, windows):
    """Full frames vs the stored frames of the reference CUDA kernel, then the first frame vs oracle windows."""
    from golden_cases import check_reference_frame
    from oracle import binding as ob
    frames = [_render_default(tree, c, want_counters=(i == 0)) for i, c in enumerate(cams)]
    for (f, u, _), name in zip(frames, names):
        check_reference_frame(name, f, u, TOL)
    # the oracle windows also pin the work counters' building blocks
    ot = ob.OracleTree.from_synth(st)
    f, u, cnt = frames[0]
    cam = cams[0]
    oc = ob.make_camera(cam.width, cam.height, cam.fx, cam.fy, np.ascontiguousarray(cam.transform, np.float32).reshape(12))
    tot = dict(samples=0, shaded=0)
    for (x0, y0, w, h) in windows:
        fo, uo, co = ob.render(ot, oc, ob.make_options(), tile=(x0, y0, w, h))
        assert np.abs(f[y0:y0 + h, x0:x0 + w] - fo).max() <= 2e-6, (x0, y0)
        assert (u[y0:y0 + h, x0:x0 + w] != uo).any(-1).sum() <= 2
        tot["samples"] += co["samples"]
        tot["shaded"] += co["shaded"]
    assert tot["samples"] > 0 and tot["shaded"] > 0, "windows must cover the object"
    assert cnt[0] >= tot["samples"] and cnt[2] >= tot["shaded"]
    return frames


def test_config2_bench_tree_800x800_default_kernel(built):
    """BASELINE config 2 at full size: the tree bench.py times (depth 10, SH16, seed 0), 800x800."""
    from volrend_b200 import N3Tree, lib, synth
    st = synth.make_tree("lego", depth=10, basis_dim=16, seed=0)
    tree = N3Tree.from_synth(st)
    info = tree.info()
    assert info["max_depth"] == 10 and lib().vr_tree_variant(tree._handle) == 3 + 16 * 193   # the batch default
    # the frames below are single-view launches: they run the shading-queue kernel (the single-frame default),
    # the batch at the end of this test runs the inline kernel -- both are compared with the reference
    poses = synth.nerf_synthetic_test_poses(200)
    fx = synth.focal_for(800)
    cams = [_cam(800, 800, fx, poses[i]) for i in (0, 77)]
    windows = [(0, 0, 64, 48), (736, 752, 64, 48), (368, 376, 64, 48), (250, 300, 48, 64)]
    frames = _check_against_reference_and_oracle(st, tree, cams, ["config2_pose0", "config2_pose77"], windows)
    # the batch default (inline shading) and, explicitly, each product kernel on single frames: same bits
    import torch
    from volrend_b200 import RenderOptions, launch_renderer, render_batch
    fb = torch.zeros((2, 800, 800, 4), dtype=torch.float32, device="cuda")
    render_batch(tree, cams, RenderOptions(), None, float_out=fb)
    torch.cuda.synchronize()
    assert np.array_equal(fb[0].cpu().numpy(), frames[0][0]) and np.array_equal(fb[1].cpu().numpy(), frames[1][0])
    for v in (7, 3 + 16 * 193):
        lib().vr_set_variant(v)
        try:
            fo = torch.zeros((800, 800, 4), dtype=torch.float32, device="cuda")
            launch_renderer(tree, cams[1], RenderOptions(), None, None, None, True, float_out=fo)
            torch.cuda.synchronize()
            assert np.array_equal(fo.cpu().numpy(), frames[1][0]), v
        finally:
            lib().vr_set_variant(0)


def test_config4_sh25_depth11_1080p_and_bands(built):
    """BASELINE config 4: depth-11 SH25 tree at 1920x1080, full frame + ray-tile (band) sharding for 2/4/8 GPUs."""
    import torch
    from volrend_b200 import N3Tree, RenderOptions, render_bands, synth
    from volrend_b200 import dist as vd
    st = synth.make_tree("gyroid_small", depth=11, basis_dim=25, seed=0, band_cells=1.0)
    tree = N3Tree.from_synth(st)
    assert tree.info()["max_depth"] == 11 and tree.info()["kernel_basis"] == 25
    from volrend_b200 import lib
    assert lib().vr_tree_variant(tree._handle) == 3 + 16 * 193                     # SH25: inline shading is the default
    W, H, fx = 1920, 1080, 1500.0
    pose = synth.nerf_synthetic_test_poses(40, radius=1.6, elev_deg=25.0)[7]
    cam = _cam(W, H, fx, pose)
    windows = [(0, 0, 48, 32), (W - 48, H - 32, 48, 32), (900, 500, 64, 48), (600, 700, 48, 32)]
    frames = _check_against_reference_and_oracle(st, tree, [cam], ["config4_pose7"], windows)
    f_full, u_full, _ = frames[0]
    for world in (2, 4, 8):
        band_h = 8
        seen = np.zeros(H, int)
        for part in range(world):
            rows = vd.band_rows(H, band_h, world, part)
            img = torch.zeros((rows, W, 4), dtype=torch.uint8, device="cuda")
            fo = torch.zeros((rows, W, 4), dtype=torch.float32, device="cuda")
            assert render_bands(tree, cam, RenderOptions(), band_h, world, part, img, float_out=fo) == rows
            torch.cuda.synchronize()
            gi, gf = img.cpu().numpy(), fo.cpu().numpy()
            r0 = 0
            for (x0, y0, w, h) in vd.shard_bands(W, H, part, world, band_h):
                assert np.array_equal(gi[r0:r0 + h], u_full[y0:y0 + h]), (world, part, y0)
                assert np.array_equal(gf[r0:r0 + h], f_full[y0:y0 + h]), (world, part, y0)
                seen[y0:y0 + h] += 1
                r0 += h
        assert np.all(seen == 1)
