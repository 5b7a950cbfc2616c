"""Seeded ray batches of the ray-golden cases (tests/golden/rays/<case>.npz, written by tools/make_golden.py with the
reference's ray tap; read by the CPU and GPU ray tests).  The trees are those of golden_cases.build_case."""
import numpy as np

from volrend_b200 import synth

# ray case -> golden_cases.build_case name (tree, pose, options, NDC)
RAY_CASES = {"rays_sh16": "lego_sh16", "rays_sh16_ndc": "lego_sh16_ndc", "rays_asg4": "lego_asg4",
             "rays_rgba": "lego_rgba", "rays_sh9_depth": "lego_sh9_depth", "rays_sg9_rot": "lego_sg9_rot"}
N_RAYS = 4096


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def make_rays(case: str, tree_case: tuple):
    """-> (origins [N,3], dirs [N,3], t_max [N]) float32, world space.  Mix: camera rays of the case's pose (64x32
    window, un-normalised as vr_camera_rays writes them), origins inside the tree's box, rays from a sphere aimed at
    random scene points, axis-aligned directions and directions with exact-zero components, lengths 1e-3 .. 1e3, and
    depth limits 1e9, (0, 3), 0 and -1."""
    st, W, H, pose, _, ndc = tree_case
    rng = np.random.default_rng(sum(map(ord, case)))
    n = N_RAYS
    off, sc = np.asarray(st.offset, np.float64), np.asarray(st.invradius3, np.float64)
    lo, hi = (0.0 - off) / sc, (1.0 - off) / sc            # the tree's unit cube in world space
    centre, radius = (lo + hi) / 2, np.linalg.norm(hi - lo) / 2
    o = np.zeros((n, 3)); d = np.zeros((n, 3))
    # 1) camera rays of the pose: pixels of a 64x32 window in the middle of the frame
    k = 2048
    c2w = np.asarray(pose, np.float64)[:3, :4]
    fx = synth.focal_for(W)
    ys, xs = np.divmod(np.arange(k), 64)
    px, py = xs + W // 2 - 32, ys + H // 2 - 16
    vx, vy = (px - W * 0.5) / fx, -(py - H * 0.5) / fx
    d[:k] = vx[:, None] * c2w[:, 0] + vy[:, None] * c2w[:, 1] - c2w[:, 2]
    o[:k] = c2w[:, 3]
    # 2) origins inside the box, random directions
    m = k + 768
    o[k:m] = lo + (hi - lo) * rng.uniform(0.05, 0.95, (m - k, 3))
    d[k:m] = rng.normal(size=(m - k, 3))
    # 3) from a sphere around the box, aimed at random scene points
    p = m + 768
    o[m:p] = centre + 1.5 * radius * _unit(rng.normal(size=(p - m, 3)))
    d[m:p] = lo + (hi - lo) * rng.uniform(0.2, 0.8, (p - m, 3)) - o[m:p]
    # 4) axis-aligned directions and exact-zero components
    axes = np.concatenate([np.eye(3), -np.eye(3)])
    d[p:] = axes[rng.integers(0, 6, n - p)]
    half = p + (n - p) // 2
    two = rng.normal(size=(n - half, 3))
    two[np.arange(n - half), rng.integers(0, 3, n - half)] = 0.0
    d[half:] = two
    o[p:] = lo + (hi - lo) * rng.uniform(-0.2, 1.2, (n - p, 3))
    if ndc is not None:     # forward-facing NDC scene: keep every ray in front of the camera plane, pointing into -z
        d[k:, 2] = -np.abs(d[k:, 2]) - 0.05
        o[k:] = c2w[:, 3] + 0.05 * rng.normal(size=(n - k, 3))
    # lengths 1e-3 .. 1e3 (camera rays keep theirs: they must reproduce the frame)
    d[k:] *= (10.0 ** rng.uniform(-3, 3, n - k))[:, None] / np.maximum(np.linalg.norm(d[k:], axis=1), 1e-30)[:, None]
    t = np.full(n, 1e9, np.float32)
    sel = rng.permutation(n)
    t[sel[: n // 8]] = rng.uniform(0.0, 3.0, n // 8)
    t[sel[n // 8: n // 8 + 64]] = 0.0
    t[sel[n // 8 + 64: n // 8 + 128]] = -1.0
    return o.astype(np.float32), d.astype(np.float32), t
