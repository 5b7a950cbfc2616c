"""`-m gpu`: the CUDA path through the C-ABI against (a) the CPU oracle, (b) the golden vectors of
the reference CUDA kernel, (c) stored frames of the reference loader + kernel on tree.npz files, and
through size-independent properties at the full benchmark size.

Tolerances: float RGBA <= 1e-4 abs per channel (BASELINE.json north_star).  In practice the sample
positions are bit-identical, so we also assert the exact work counters and that pixels are
bit-identical to the reference kernel."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu
TOL = 1e-4
QUEUE, INLINE, POOL = 7, 3 + 16 * 193, 8     # the product kernels (vr_kernels.h): shading queue, inline shading, queue + ray pool
# round-1 experiment kernels: present only in a -DVR_EXPERIMENTS build (make lib EXTRA=-DVR_EXPERIMENTS)
VARIANTS = [QUEUE, POOL, INLINE, 1, 2, 3, 4, 5, 6, 19, 3 + 16 * 64, 3 + 16 * 65]


def supported(tree, variant) -> bool:
    from volrend_b200 import lib
    return bool(lib().vr_variant_supported(tree.info()["kernel_basis"], variant))


def _torch():
    import torch
    return torch


def make_cam(W, H, pose):
    from volrend_b200 import Camera, synth
    c = Camera(W, H, synth.focal_for(W), synth.focal_for(W))
    c.set_c2w(pose)
    return c


def gpu_render(tree, cam, opt, variant=0, counters=False, tile=None, composite=None):
    torch = _torch()
    from volrend_b200 import launch_renderer, lib
    lib().vr_set_variant(variant)
    w, h = (cam.width, cam.height) if tile is None else (tile[2], tile[3])
    img = torch.zeros((h, w, 4), dtype=torch.uint8, device="cuda")
    fo = torch.zeros((h, w, 4), dtype=torch.float32, device="cuda")
    cnt = torch.zeros(5, dtype=torch.int64, device="cuda") if counters else None
    if composite is not None:
        rgba, depth = composite
        img.copy_(torch.from_numpy(rgba))
        d = torch.from_numpy(depth).cuda()
        launch_renderer(tree, cam, opt, img, d, None, False, float_out=fo, tile=tile)
    else:
        launch_renderer(tree, cam, opt, img, None, None, True, float_out=fo, counters=cnt, tile=tile)
    torch.cuda.synchronize()
    lib().vr_set_variant(0)
    return fo.cpu().numpy(), img.cpu().numpy(), (cnt.cpu().numpy().tolist() if counters else None)


def oracle_render(st, cam, optkw, ndc=None, **kw):
    from oracle import binding as ob
    t = ob.OracleTree.from_synth(st, ndc=ndc)
    c12 = np.ascontiguousarray(cam.transform, np.float32).reshape(12)
    oc = ob.make_camera(cam.width, cam.height, cam.fx, cam.fy, c12)
    return ob.render(t, oc, ob.make_options(**optkw), **kw)


@pytest.fixture(scope="module")
def dev_trees(small_trees):
    from volrend_b200 import N3Tree
    return {k: (st, N3Tree.from_synth(st)) for k, st in small_trees.items()}


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("name", ["sh1_full4", "sh16_d6", "sh9_d6", "sh4_d5", "sh25_d5", "rgba_d5", "sg9_d5",
                                  "asg4_d5", "sg7_d5"])
def test_matches_oracle_all_formats(built, dev_trees, name, variant):
    from volrend_b200 import RenderOptions, synth
    st, tree = dev_trees[name]
    if not supported(tree, variant):
        pytest.skip("variant not built for this basis size (experiments need -DVR_EXPERIMENTS)")
    pose = synth.config1_pose() if name == "sh1_full4" else synth.nerf_synthetic_test_poses(8)[(len(name) * 3) % 8]
    cam = make_cam(72, 56, pose)
    f, u, cnt = gpu_render(tree, cam, RenderOptions(), variant=variant, counters=(variant in (QUEUE, POOL, INLINE, 5, 6)))   # instrumented builds of the two product kernels
    fo, uo, co = oracle_render(st, cam, {})
    assert np.abs(f - fo).max() <= TOL
    assert np.abs(f - fo).max() <= 2e-6          # what we actually achieve (expf ulps only)
    assert (u != uo).any(-1).sum() <= 3
    if cnt is not None:                            # identical sample sequence => identical counters
        assert cnt[:4] == [co["samples"], co["child_loads"], co["shaded"], co["rays_hit"]]
        assert cnt[4] <= co["child_loads"]


@pytest.mark.parametrize("optkw", [dict(step_size=1e-5), dict(step_size=1e-2), dict(stop_thresh=0.0),
                                   dict(stop_thresh=1e-1), dict(sigma_thresh=0.0), dict(sigma_thresh=1.0),
                                   dict(background_brightness=0.3), dict(render_bbox=[0.2, 0.1, 0, 0.9, 0.8, 0.7]),
                                   dict(basis_minmax=[2, 9]), dict(rot_dirs=[0.4, 0.1, -0.3]),
                                   dict(render_depth=True)])
def test_option_sweep_vs_oracle(built, dev_trees, optkw):
    """BASELINE config 3: step-size / early-stop / sigma-threshold sweep (+ the other options)."""
    from volrend_b200 import RenderOptions, synth
    st, tree = dev_trees["sh16_d6"]
    cam = make_cam(64, 64, synth.nerf_synthetic_test_poses(8)[6])
    f, u, cnt = gpu_render(tree, cam, RenderOptions(**optkw), counters=True)
    okw = dict(optkw)
    if "render_depth" in okw:
        okw["render_depth"] = 1
    fo, uo, co = oracle_render(st, cam, okw)
    tol = 2e-5 if "rot_dirs" in optkw else 2e-6    # rodrigues: libdevice vs glibc cosf/sinf
    assert np.abs(f - fo).max() <= tol
    assert cnt[:4] == [co["samples"], co["child_loads"], co["shaded"], co["rays_hit"]]


def test_golden_vectors_of_reference_kernel(built):
    """Committed outputs of the reference CUDA kernel (tests/golden) vs our kernel: <= 1e-4,
    and bit-identical in practice."""
    import glob
    from golden_cases import build_case, composite_inputs
    from volrend_b200 import N3Tree, RenderOptions
    paths = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz")))
    assert len(paths) >= 4
    for p in paths:
        z = np.load(p)
        st, W, H, pose, optkw, ndc = build_case(str(z["case"]))
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
        cam = make_cam(W, H, pose)
        kw = dict(optkw)
        if "render_depth" in kw:
            kw["render_depth"] = bool(kw["render_depth"])
        f, u, _ = gpu_render(tree, cam, RenderOptions(**kw), composite=composite_inputs(str(z["case"]), W, H))
        d = np.abs(f - z["ref_f32"])
        assert d.max() <= TOL, (p, d.max())
        assert (d > 0).any(-1).mean() <= 0.01, (p, "expected (near) bit-exact floats")
        assert np.abs(u.astype(int) - z["ref_u8"].astype(int)).max() <= 1
        assert (u != z["ref_u8"]).any(-1).sum() <= 2


def test_reference_frames_through_our_loader(built, tmp_path):
    """The same tree.npz through our loader + kernel vs the stored frames of the reference loader +
    launch_renderer (tests/golden/frames): bit-identical."""
    from golden_cases import check_reference_frame, frame_case
    from volrend_b200 import N3Tree, RenderOptions
    for name in ("loader_sh16", "loader_sh25", "loader_rgba"):
        st, W, H, fx, pose = frame_case(name)
        path = str(tmp_path / f"{name}.npz")
        st.save_npz(path)
        tree = N3Tree(path)
        f, u, _ = gpu_render(tree, make_cam(W, H, pose), RenderOptions())
        check_reference_frame(name, f, u, TOL)


def test_tiles_batches_and_variants_are_bit_identical(built, dev_trees):
    """Tile-sharded render == full frame, batch == per-view, every variant == every other."""
    torch = _torch()
    from volrend_b200 import RenderOptions, lib, render_batch, synth
    st, tree = dev_trees["sh9_d6"]
    poses = synth.nerf_synthetic_test_poses(8)
    cams = [make_cam(100, 76, p) for p in poses[:5]]
    opt = RenderOptions()
    full = [gpu_render(tree, c, opt, variant=INLINE) for c in cams]
    for v in VARIANTS:
        if not supported(tree, v):
            continue
        f, u, _ = gpu_render(tree, cams[0], opt, variant=v)
        assert np.array_equal(f, full[0][0]) and np.array_equal(u, full[0][1]), v
    for tile in [(0, 0, 100, 76), (13, 7, 50, 33), (96, 70, 4, 6), (0, 38, 100, 38), (5, 5, 1, 1)]:
        ft, ut, _ = gpu_render(tree, cams[1], opt, tile=tile)
        x0, y0, w, h = tile
        assert np.array_equal(ft, full[1][0][y0:y0 + h, x0:x0 + w]), tile
        assert np.array_equal(ut, full[1][1][y0:y0 + h, x0:x0 + w]), tile
    for v in (QUEUE, POOL, INLINE, 1, 5):
        if not supported(tree, v):
            continue
        lib().vr_set_variant(v)
        imgs = torch.zeros((len(cams), 76, 100, 4), dtype=torch.uint8, device="cuda")
        fo = torch.zeros((len(cams), 76, 100, 4), dtype=torch.float32, device="cuda")
        render_batch(tree, cams, opt, imgs, float_out=fo)
        torch.cuda.synchronize()
        for i in range(len(cams)):
            assert np.array_equal(fo[i].cpu().numpy(), full[i][0]) and np.array_equal(imgs[i].cpu().numpy(), full[i][1])
    lib().vr_set_variant(0)


def test_composite_mode_vs_oracle(built, dev_trees):
    """launch_renderer(offscreen=false): existing colour + depth limit (volrend.cu:92-96,143-163)."""
    from volrend_b200 import RenderOptions, synth
    st, tree = dev_trees["sh4_d5"]
    cam = make_cam(48, 40, synth.nerf_synthetic_test_poses(8)[3])
    rng = np.random.default_rng(0)
    rgba = rng.integers(0, 256, (40, 48, 4)).astype(np.uint8)
    depth = rng.uniform(2.5, 5.0, (40, 48)).astype(np.float32)
    f, u, _ = gpu_render(tree, cam, RenderOptions(), composite=(rgba, depth))
    fo, uo, _ = oracle_render(st, cam, {}, rgba_in=rgba, depth_in=depth)
    assert np.abs(f - fo).max() <= 2e-6
    assert (u != uo).any(-1).sum() <= 2


def test_empty_and_degenerate_inputs(built, dev_trees):
    torch = _torch()
    from volrend_b200 import RenderOptions, VolrendError, launch_renderer, render_batch, synth
    st, tree = dev_trees["sh4_d5"]
    cam = make_cam(33, 17, synth.nerf_synthetic_test_poses(8)[0])
    # zero-sized tile and zero views are no-ops
    launch_renderer(tree, cam, RenderOptions(), None, None, None, True, tile=(3, 3, 0, 0))
    render_batch(tree, [], RenderOptions(), None)
    # tile outside the frame is rejected, never clipped silently
    img = torch.zeros((17, 33, 4), dtype=torch.uint8, device="cuda")
    with pytest.raises(VolrendError):
        launch_renderer(tree, cam, RenderOptions(), img, None, None, True, tile=(30, 0, 8, 8))
    # a camera looking away: pure background
    away = synth.look_at_c2w((0, -4, 0), target=(0, -8, 0))
    f, u, _ = gpu_render(tree, make_cam(33, 17, away), RenderOptions(background_brightness=0.5))
    assert np.all(f[..., :3] == 0.5) and np.all(f[..., 3] == 0) and np.all(u[..., :3] == 127)


def test_tree_validation_errors(built, small_trees):
    from volrend_b200 import N3Tree, VolrendError
    st = small_trees["sh4_d5"]
    bad = st.child.copy()
    bad[0, 0, 0, 0] = 10 ** 6                     # link outside the node array
    t = N3Tree()
    with pytest.raises(VolrendError, match="links outside"):
        t.open_arrays(child=bad, data=st.data, offset=st.offset, invradius3=st.invradius3,
                      data_dim=st.data_dim, data_format=st.data_format)
    t3 = N3Tree()
    with pytest.raises(VolrendError, match="N=2"):
        t3.open_arrays(child=np.zeros((1, 3, 3, 3), np.int32), data=np.zeros((1, 3, 3, 3, 4), np.float16),
                       offset=st.offset, invradius3=st.invradius3, data_dim=4, data_format="RGBA")


def test_probe_lumisphere(built, dev_trees):
    """retrieve_cursor_lumisphere_kernel (volrend.cu:175-191)."""
    torch = _torch()
    from volrend_b200 import lib
    from volrend_b200._capi import check
    st, tree = dev_trees["sh9_d6"]
    # world point -> tree coords -> leaf, by hand
    xyz = np.array([0.1, -0.2, 0.05], np.float32)
    p = st.offset + st.invradius3 * xyz
    node, leaf = 0, None
    for _ in range(32):
        p = p * 2
        k = np.floor(p).astype(int)
        p -= k
        skip = st.child[node, k[0], k[1], k[2]]
        if skip == 0:
            leaf = st.data[node, k[0], k[1], k[2]]
            break
        node += skip
    out = torch.zeros(st.data_dim - 1, dtype=torch.float32, device="cuda")
    arr = (C.c_float * 3)(*xyz.tolist())
    check(lib().vr_probe_lumisphere(tree._handle, arr, out.data_ptr(), None))
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), leaf[:-1].astype(np.float32))


def test_frames_host_and_launch_count(built, dev_trees):
    torch = _torch()
    from volrend_b200 import RenderOptions, lib, render_frames_host, synth
    st, tree = dev_trees["sh16_d6"]
    cams = [make_cam(64, 48, p) for p in synth.nerf_synthetic_test_poses(6)]
    host = torch.zeros((6, 48, 64, 4), dtype=torch.uint8).pin_memory()
    n0 = lib().vr_launch_count()
    render_frames_host(tree, cams, RenderOptions(), host)
    assert 1 <= lib().vr_launch_count() - n0 <= 6
    for i, c in enumerate(cams):
        _, u, _ = gpu_render(tree, c, RenderOptions())
        assert np.array_equal(host[i].numpy(), u)


def test_full_size_properties(built):
    """BASELINE config 2 size (800x800, depth-9 stand-in): properties that need no oracle."""
    torch = _torch()
    from volrend_b200 import N3Tree, RenderOptions, lib, render_batch, synth
    st = synth.make_tree("lego", depth=9, basis_dim=16, seed=0)
    tree = N3Tree.from_synth(st)
    poses = synth.nerf_synthetic_test_poses(200)[::25]
    cams = [make_cam(800, 800, p) for p in poses]
    opt = RenderOptions()
    outs = {}
    for v in (QUEUE, INLINE, POOL):
        if not supported(tree, v):
            continue
        lib().vr_set_variant(v)
        imgs = torch.zeros((len(cams), 800, 800, 4), dtype=torch.uint8, device="cuda")
        fo = torch.zeros((len(cams), 800, 800, 4), dtype=torch.float32, device="cuda")
        cnt = torch.zeros(5, dtype=torch.int64, device="cuda")
        render_batch(tree, cams, opt, imgs, float_out=fo)
        render_batch(tree, cams, opt, imgs, counters=cnt)
        torch.cuda.synchronize()
        outs[v] = (fo.cpu().numpy(), imgs.cpu().numpy(), cnt.cpu().tolist())
    lib().vr_set_variant(0)
    f, u, cnt = outs[QUEUE]
    assert np.array_equal(f, outs[INLINE][0]) and np.array_equal(u, outs[INLINE][1])     # variant-independent
    assert cnt == outs[INLINE][2]
    # the ray pool moves rays between warps, never changes what a ray computes
    if POOL in outs:
        assert np.array_equal(f, outs[POOL][0]) and np.array_equal(u, outs[POOL][1]) and cnt == outs[POOL][2]
    assert np.isfinite(f).all() and f[..., 3].min() >= 0 and f[..., 3].max() <= 1
    assert (f[..., :3] >= 0).all() and (f[..., :3] <= 1 + 1e-5).all()         # sigmoid colours, bg <= 1
    assert np.all(u[..., 3] == 255)
    q = np.floor(f[..., :3] * np.float32(255)).astype(np.uint8)
    assert np.array_equal(q, u[..., :3])                                        # volrend.cu:166
    # a band of tiles == the same rows of the full frame, at full size
    ft = torch.zeros((1, 200, 800, 4), dtype=torch.float32, device="cuda")
    render_batch(tree, cams[:1], opt, None, float_out=ft, tile=(0, 400, 800, 200))
    torch.cuda.synchronize()
    assert np.array_equal(ft[0].cpu().numpy(), f[0, 400:600])
    # oracle spot check on a 64x64 window of one full-size frame
    fo, uo, co = oracle_render(st, cams[3], {}, tile=(368, 368, 64, 64))
    assert np.abs(f[3, 368:432, 368:432] - fo).max() <= 2e-6
    S, D, SH, HIT, FETCH = cnt
    assert S > 0 and D >= S and SH <= S and HIT <= 800 * 800 * len(cams) and FETCH < D


def test_cxx_shim_and_headless_cli(built, small_trees, tmp_path):
    """The reference's unchanged C++ callers on our backend (build/shim_test, build/volrend_headless):
    launch_renderer into a cudaArray and VolumeRenderer::render()."""
    exe = os.path.join(ROOT, "build", "shim_test")
    cli = os.path.join(ROOT, "build", "volrend_headless")
    if not (os.path.exists(exe) and os.path.exists(cli)):
        pytest.skip("shim binaries not built (they need the reference headers at build time)")
    from volrend_b200 import N3Tree, RenderOptions, synth
    st = small_trees["sh16_d6"]
    path = str(tmp_path / "tree.npz")
    st.save_npz(path)
    poses = synth.nerf_synthetic_test_poses(8)
    ppaths = synth.write_pose_files(poses, str(tmp_path), synth.focal_for(80))
    o1, o2 = str(tmp_path / "a.rgba"), str(tmp_path / "b.rgba")
    r = subprocess.run([exe, path, ppaths[2], "80", "60", str(synth.focal_for(80)), o1, o2], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    assert "backend CUDA" in r.stdout
    tree = N3Tree(path)
    cam = make_cam(80, 60, poses[2])
    _, u, _ = gpu_render(tree, cam, RenderOptions())
    a = np.fromfile(o1, np.uint8).reshape(60, 80, 4)
    assert np.array_equal(a, u)                                     # launch_renderer drop-in: identical bytes
    b = np.fromfile(o2, np.uint8).reshape(60, 80, 4)
    assert np.abs(b.astype(int) - u.astype(int)).mean() < 0.5        # pose went through Camera::_update
    r = subprocess.run([cli, path, "-w", "80", "-h", "60", "--fx", str(synth.focal_for(80))] + ppaths,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ms per frame" in r.stdout and "fps" in r.stdout


def test_back_to_back_launches_keep_stream_order(built, dev_trees):
    """Per-frame launches overlap their predecessor's tail (programmatic dependent launch);
    stream order must still hold: same-buffer launches leave the LAST frame, separate buffers
    each hold their own frame, and a composite launch sees the image its predecessor wrote."""
    torch = _torch()
    from volrend_b200 import RenderOptions, launch_renderer, synth
    st, tree = dev_trees["sh16_d6"]
    cams = [make_cam(200, 160, p) for p in synth.nerf_synthetic_test_poses(12)]
    opt = RenderOptions()
    solo = [gpu_render(tree, c, opt)[1] for c in cams]
    same = torch.zeros((160, 200, 4), dtype=torch.uint8, device="cuda")
    sep = torch.zeros((len(cams), 160, 200, 4), dtype=torch.uint8, device="cuda")
    for rep in range(3):
        for i, c in enumerate(cams):
            launch_renderer(tree, c, opt, same, None, None, True)
        for i, c in enumerate(cams):
            launch_renderer(tree, c, opt, sep[i], None, None, True)
        torch.cuda.synchronize()
        assert np.array_equal(same.cpu().numpy(), solo[-1])
        for i in range(len(cams)):
            assert np.array_equal(sep[i].cpu().numpy(), solo[i]), i
    # offscreen render followed immediately by a composite pass over it (reads what was just written)
    img = torch.zeros((160, 200, 4), dtype=torch.uint8, device="cuda")
    depth = torch.full((160, 200), 1e9, dtype=torch.float32, device="cuda")
    launch_renderer(tree, cams[0], opt, img, None, None, True)
    launch_renderer(tree, cams[1], opt, img, depth, None, False)
    torch.cuda.synchronize()
    _, want, _ = oracle_render(st, cams[1], {}, rgba_in=solo[0], depth_in=np.full((160, 200), 1e9, np.float32))
    assert (img.cpu().numpy() != want).any(-1).sum() <= 2


def test_render_bands_matches_full_frame(built, dev_trees):
    """vr_render_bands: every part's compact buffer holds exactly its interleaved bands."""
    torch = _torch()
    from volrend_b200 import RenderOptions, render_bands, synth
    from volrend_b200 import dist as vd
    st, tree = dev_trees["sh9_d6"]
    cam = make_cam(120, 92, synth.nerf_synthetic_test_poses(8)[4])       # 92 rows: ragged last band
    f_full, u_full, _ = gpu_render(tree, cam, RenderOptions())
    for world, band_h in ((1, 8), (2, 8), (3, 4), (4, 16)):
        seen = np.zeros(92, int)
        for part in range(world):
            rows = vd.band_rows(92, band_h, world, part)
            img = torch.zeros((max(rows, 1), 120, 4), dtype=torch.uint8, device="cuda")
            fo = torch.zeros((max(rows, 1), 120, 4), dtype=torch.float32, device="cuda")
            got = render_bands(tree, cam, RenderOptions(), band_h, world, part, img, float_out=fo)
            torch.cuda.synchronize()
            assert got == rows
            r0 = 0
            for (x0, y0, w, h) in vd.shard_bands(120, 92, part, world, band_h):
                assert np.array_equal(img[r0:r0 + h].cpu().numpy(), u_full[y0:y0 + h])
                assert np.array_equal(fo[r0:r0 + h].cpu().numpy(), f_full[y0:y0 + h])
                seen[y0:y0 + h] += 1
                r0 += h
        assert np.all(seen == 1)


def test_gpu_decode_of_quantised_tree(built, tmp_path):
    """vr_tree_create_quantized (GPU decode of quant_colors/quant_map/sigma/data_retained) gives the
    same device tree as the reference's CPU decode (src/n3tree.cpp:279-340): identical renders,
    identical probed coefficients, and for SH the stored frames of the reference loader + kernel."""
    torch = _torch()
    from golden_cases import check_reference_frame
    from volrend_b200 import N3Tree, RenderOptions, lib, synth
    from volrend_b200._capi import check
    for basis, n_retain, fmt in ((16, 1, "SH"), (9, 0, "SH"), (7, 2, "SG")):
        st = synth.make_tree("lego", depth=6, basis_dim=basis, seed=basis, fmt=fmt)
        npz = synth.quantise_tree(st, n_retain=n_retain, seed=3)
        path = str(tmp_path / f"q{basis}.npz")
        np.savez(path, **npz)
        t_gpu, t_cpu = N3Tree(path, gpu_decode=True), N3Tree(path, gpu_decode=False)
        assert t_gpu._data is None                      # nothing was decoded on the host
        cam = make_cam(96, 80, synth.nerf_synthetic_test_poses(8)[3])
        fg, ug, _ = gpu_render(t_gpu, cam, RenderOptions())
        fc, uc, _ = gpu_render(t_cpu, cam, RenderOptions())
        assert np.array_equal(fg, fc) and np.array_equal(ug, uc)
        if basis in (1, 4, 9, 16, 25):
            out_g = torch.zeros(3 * basis, dtype=torch.float32, device="cuda")
            out_c = torch.zeros(3 * basis, dtype=torch.float32, device="cuda")
            arr = (C.c_float * 3)(0.05, -0.1, 0.02)
            check(lib().vr_probe_lumisphere(t_gpu._handle, arr, out_g.data_ptr(), None))
            check(lib().vr_probe_lumisphere(t_cpu._handle, arr, out_c.data_ptr(), None))
            torch.cuda.synchronize()
            assert torch.equal(out_g, out_c)
        if fmt == "SH":                                 # the reference loader decodes on the CPU
            check_reference_frame(f"quant_sh{basis}", fg, ug, TOL)


def test_png_egress_api_and_cli(built, dev_trees, small_trees, tmp_path):
    """SURVEY.md 8(f) rank 2: frames -> PNG files (vr_render_frames_png) and the reference CLI's
    `-o <dir>` on our backend; decoded pixels must equal the rendered bytes."""
    from PIL import Image
    from volrend_b200 import RenderOptions, render_frames_png, synth
    st, tree = dev_trees["sh16_d6"]
    poses = synth.nerf_synthetic_test_poses(40)
    cams = [make_cam(96, 64, p) for p in poses]
    paths = [str(tmp_path / f"v{i:03d}.png") for i in range(len(cams))]
    render_frames_png(tree, cams, RenderOptions(), paths, n_threads=4)
    for i in (0, 7, 33, 39):
        _, u, _ = gpu_render(tree, cams[i], RenderOptions())
        assert np.array_equal(np.asarray(Image.open(paths[i])), u), i
    cli = os.path.join(ROOT, "build", "volrend_headless")
    if not os.path.exists(cli):
        pytest.skip("shim binaries not built")
    npz = str(tmp_path / "tree.npz")
    small_trees["sh16_d6"].save_npz(npz)
    ppaths = synth.write_pose_files(poses[:3], str(tmp_path), synth.focal_for(96))
    outdir = str(tmp_path / "out")
    r = subprocess.run([cli, npz, "-w", "96", "-h", "64", "--fx", str(synth.focal_for(96)), "-o", outdir] + ppaths,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    for i in range(3):
        got = np.asarray(Image.open(os.path.join(outdir, f"{i:04d}.png")))
        _, u, _ = gpu_render(tree, cams[i], RenderOptions())
        assert np.array_equal(got, u)


def test_multi_gpu_renderer_matches_single_device(built, small_trees):
    """vr_mg_* (one process, N devices): view and ray-tile sharding reassemble to exactly the single-device
    frames.  On a 1-GPU box the device list repeats device 0, which still exercises the sharding, the per-device
    worker threads, the band scatter (2-D copies, ragged last band) and the double-buffered batches."""
    torch = _torch()
    from volrend_b200 import MultiGpuRenderer, N3Tree, RenderOptions, VR_MG_TILES, VR_MG_VIEWS, synth
    st = small_trees["sh16_d6"]
    tree = N3Tree.from_synth(st)
    cams = [make_cam(120, 92, p) for p in synth.nerf_synthetic_test_poses(7)]      # 92 rows: ragged last band of 8
    want = np.stack([gpu_render(tree, c, RenderOptions())[1] for c in cams])
    n_dev = torch.cuda.device_count()
    for devices in ([0], [0, 0, 0], list(range(n_dev)) if n_dev > 1 else [0, 0]):
        mg = MultiGpuRenderer(tree, devices)
        try:
            for mode, band_h, batch in ((VR_MG_VIEWS, 8, 0), (VR_MG_VIEWS, 8, 2), (VR_MG_TILES, 8, 0), (VR_MG_TILES, 4, 3),
                                        (VR_MG_TILES, 16, 1)):
                host = np.zeros_like(want)
                dev0 = torch.zeros(want.shape, dtype=torch.uint8, device="cuda:0")
                ms = mg.render(cams, RenderOptions(), mode=mode, band_h=band_h, batch=batch, out_dev0=dev0, out_host=host)
                assert ms > 0
                assert np.array_equal(host, want), (devices, mode, band_h, batch)
                assert np.array_equal(dev0.cpu().numpy(), want), (devices, mode, band_h, batch)
        finally:
            mg.close()


def test_headless_mg_cli(built, small_trees, tmp_path):
    """build/volrend_headless_mg: the reference's loader + option parser in front of vr_mg_*; --check compares
    with the single-GPU render inside the binary, and the PNGs must equal our own render of the same poses."""
    cli = os.path.join(ROOT, "build", "volrend_headless_mg")
    if not os.path.exists(cli):
        pytest.skip("shim binaries not built (they need the reference headers at build time)")
    from PIL import Image
    from volrend_b200 import N3Tree, RenderOptions, synth
    st = small_trees["sh9_d6"]
    npz = str(tmp_path / "tree.npz")
    st.save_npz(npz)
    poses = synth.nerf_synthetic_test_poses(5)
    ppaths = synth.write_pose_files(poses, str(tmp_path), synth.focal_for(96))
    tree = N3Tree(npz)
    for mode in ("views", "tiles"):
        outdir = str(tmp_path / f"out_{mode}")
        r = subprocess.run([cli, npz, "-w", "96", "-h", "68", "--fx", str(synth.focal_for(96)), "--mode", mode, "--batch", "2",
                            "--check", "-o", outdir] + ppaths, capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "ms per frame" in r.stdout and "(identical)" in r.stdout
        for i in (0, 4):
            got = np.asarray(Image.open(os.path.join(outdir, f"{i:04d}.png")))
            _, u, _ = gpu_render(tree, make_cam(96, 68, poses[i]), RenderOptions())
            assert np.array_equal(got, u)
