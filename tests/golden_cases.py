"""Deterministic inputs of the golden-vector cases (shared by tools/make_golden.py, which runs the
reference CUDA kernel on them on the B200, and by the CPU/GPU parity tests)."""
import hashlib
import os

import numpy as np

from volrend_b200 import synth

CASES = ["cfg1_sh1", "lego_sh16", "drums_sh9", "lego_sh25_bbox", "lego_sh4_stop0", "lego_rgba",
         "lego_sg9_rot", "lego_sh16_ndc", "lego_sh9_depth", "lego_asg4", "lego_sh9_composite"]

# Frames of the reference renderer on a tree.npz read by the reference's own loader, default options
# (tests/golden/frames/<name>.npz).  Full frames are too large to store, so each file holds digests of
# the whole frame plus a fixed sample of its pixels.
FRAME_CASES = ["loader_sh16", "loader_sh25", "loader_rgba", "quant_sh16", "quant_sh9",
               "config2_pose0", "config2_pose77", "config4_pose7"]
FRAMES_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "frames")
FRAME_SAMPLE = 1024


def frame_case(name: str):
    """-> (tree.npz arrays as a SynthTree or dict, W, H, fx, pose 4x4)"""
    poses = synth.nerf_synthetic_test_poses(8)
    kind, _, arg = name.partition("_")
    if kind == "loader":
        st = {"sh16": lambda: synth.make_tree("lego", depth=6, basis_dim=16, seed=1),
              "sh25": lambda: synth.make_tree("drums", depth=5, basis_dim=25, seed=4),
              "rgba": lambda: synth.make_tree("lego", depth=5, fmt="RGBA", seed=5)}[arg]()
        return st, 80, 60, synth.focal_for(80), poses[2]
    if kind == "quant":
        basis = int(arg[2:])
        st = synth.make_tree("lego", depth=6, basis_dim=basis, seed=basis)
        return synth.quantise_tree(st, n_retain={16: 1, 9: 0}[basis], seed=3), 96, 80, synth.focal_for(96), poses[3]
    if kind == "config2":          # the tree and orbit bench.py times
        st = synth.make_tree("lego", depth=10, basis_dim=16, seed=0)
        return st, 800, 800, synth.focal_for(800), synth.nerf_synthetic_test_poses(200)[int(arg[4:])]
    if kind == "config4":
        st = synth.make_tree("gyroid_small", depth=11, basis_dim=25, seed=0, band_cells=1.0)
        return st, 1920, 1080, 1500.0, synth.nerf_synthetic_test_poses(40, radius=1.6, elev_deg=25.0)[int(arg[4:])]
    raise KeyError(name)


def frame_digest(a: np.ndarray) -> str:
    """sha256 of a frame's bytes; -0.0 counts as 0.0, as np.array_equal does."""
    return hashlib.sha256(np.ascontiguousarray(a + a.dtype.type(0)).tobytes()).hexdigest()


def frame_record(f: np.ndarray, u: np.ndarray) -> dict:
    """What tests/golden/frames/<name>.npz stores of a float RGBA frame f and its RGBA8 bytes u."""
    n = f.shape[0] * f.shape[1]
    idx = np.sort(np.random.default_rng(0).choice(n, size=min(n, FRAME_SAMPLE), replace=False)).astype(np.int32)
    return dict(f32_sha256=np.array(frame_digest(f)), u8_sha256=np.array(frame_digest(u)), shape=np.array(f.shape),
                idx=idx, f32_sample=f.reshape(-1, 4)[idx], u8_sample=u.reshape(-1, 4)[idx])


def check_reference_frame(name: str, f: np.ndarray, u: np.ndarray, tol: float = 1e-4) -> None:
    """Our frame vs the stored reference frame: within tol on the sample, bit-identical as a whole."""
    z = np.load(os.path.join(FRAMES_DIR, name + ".npz"))
    assert tuple(f.shape) == tuple(z["shape"]) and tuple(u.shape) == tuple(z["shape"]), name
    fs, us = f.reshape(-1, 4)[z["idx"]], u.reshape(-1, 4)[z["idx"]]
    assert np.abs(fs - z["f32_sample"]).max() <= tol, (name, float(np.abs(fs - z["f32_sample"]).max()))
    assert np.array_equal(fs, z["f32_sample"]) and np.array_equal(us, z["u8_sample"]), \
        f"{name}: sampled pixels differ from the reference kernel (expected bit-identical)"
    assert frame_digest(f) == str(z["f32_sha256"]), f"{name}: float RGBA differs from the reference kernel"
    assert frame_digest(u) == str(z["u8_sha256"]), f"{name}: RGBA8 differs from the reference kernel"


def composite_inputs(name: str, W: int, H: int):
    """Existing colour + per-pixel depth limit of the launch_renderer(offscreen=false) cases
    (volrend.cu:92-96,143-163); None for offscreen cases."""
    if name != "lego_sh9_composite":
        return None
    rng = np.random.default_rng(21)
    rgba = rng.integers(0, 256, (H, W, 4)).astype(np.uint8)
    depth = rng.uniform(2.0, 5.5, (H, W)).astype(np.float32)     # world units; cuts some rays inside the object
    depth[: H // 4] = 1e9                                        # a band without a depth limit
    return rgba, depth


def build_case(name: str):
    """-> (SynthTree, W, H, pose 4x4, options dict, ndc tuple | None)"""
    poses = synth.nerf_synthetic_test_poses(8)
    if name == "cfg1_sh1":
        return synth.make_config1_tree(), 64, 64, synth.config1_pose(), {}, None
    if name == "lego_sh16":
        return synth.make_tree("lego", depth=6, basis_dim=16, seed=11), 96, 96, poses[3], {}, None
    if name == "drums_sh9":
        return synth.make_tree("drums", depth=6, basis_dim=9, seed=12), 80, 64, poses[5], {}, None
    if name == "lego_sh25_bbox":
        return (synth.make_tree("lego", depth=5, basis_dim=25, seed=13), 64, 64, poses[1],
                dict(render_bbox=[0.1, 0.05, 0.0, 0.8, 1.0, 0.9], background_brightness=0.5), None)
    if name == "lego_sh4_stop0":
        return (synth.make_tree("lego", depth=5, basis_dim=4, seed=14), 64, 48, poses[6],
                dict(stop_thresh=0.0, sigma_thresh=0.0, step_size=1e-3), None)
    if name == "lego_rgba":
        return synth.make_tree("lego", depth=5, fmt="RGBA", seed=15), 64, 48, poses[2], {}, None
    if name == "lego_sg9_rot":
        return (synth.make_tree("lego", depth=5, basis_dim=9, fmt="SG", seed=16), 64, 48, poses[7],
                dict(rot_dirs=[0.3, -0.2, 0.5], basis_minmax=[1, 7]), None)
    if name == "lego_sh16_ndc":
        # forward-facing camera in front of the NDC frustum (maybe_world2ndc, volrend.cu:34-54)
        pose = np.eye(4, dtype=np.float32)
        pose[:3, 3] = [0.05, -0.03, 0.2]
        st = synth.make_tree("lego", depth=5, basis_dim=16, seed=17, world_radius=1.0)
        return st, 64, 48, pose, {}, (64.0, 48.0, 60.0)
    if name == "lego_sh9_depth":
        return synth.make_tree("lego", depth=5, basis_dim=9, seed=18), 64, 48, poses[4], dict(render_depth=1), None
    if name == "lego_asg4":
        # anisotropic spherical gaussians (lumisphere.hpp:14-28), lobes in extra_data
        return synth.make_tree("lego", depth=5, basis_dim=4, fmt="ASG", seed=19), 64, 48, poses[0], {}, None
    if name == "lego_sh9_composite":
        return synth.make_tree("lego", depth=5, basis_dim=9, seed=20), 64, 48, poses[3], {}, None
    raise KeyError(name)
