#!/usr/bin/env python
"""Generate tests/golden/*.npz: outputs of the UNMODIFIED reference CUDA renderer (oracle/_ref,
built from the reference sources by oracle/Makefile.ref) on the deterministic cases of
tests/golden_cases.py.  Needs a GPU and oracle/_ref.

  usage: make_golden.py [--out DIR] [case ...]     (default DIR: tests/golden; cases: all of CASES and FRAME_CASES)

  <case>.npz         ref_f32  float RGBA of the reference's per-pixel code (tap of out[4], see oracle/ref_harness.cu)
                     ref_u8   bytes written by volrend::launch_renderer (src/cuda/volrend.cu:166-172)
  frames/<case>.npz  digests + a pixel sample of the same two outputs (golden_cases.frame_record)
  rays/<case>.npz    origins, dirs, t_max of tests/ray_cases.py and ref_f32 [n,4] of the reference's ray tap
                     (oracle/ref_rays.cu); asserts on the way that the tap reproduces the reference's frame
                     for a camera's own rays
"""
import argparse
import os
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from golden_cases import CASES, FRAME_CASES, build_case, composite_inputs, frame_case, frame_record  # noqa: E402
from oracle import ref_binding as rb  # noqa: E402
from oracle import binding as ob, ray_binding as rayb  # noqa: E402
from ray_cases import RAY_CASES, make_rays  # noqa: E402
from volrend_b200 import synth  # noqa: E402


def write_case_files(name, st, ndc, tmpdir):
    path = os.path.join(tmpdir, name + ".npz")
    if isinstance(st, dict):
        np.savez(path, **st)
    else:
        st.save_npz(path)
    pb = path[:-4] + "_poses_bounds.npy"
    if ndc is not None:
        p = np.zeros((1, 17), np.float32)
        p[0, 0] = p[0, 6] = p[0, 12] = 1.0          # identity rotation
        p[0, 9], p[0, 4], p[0, 14] = ndc              # width, height, focal (n3tree.cpp:27-29)
        p[0, 15], p[0, 16] = 1.0, 10.0
        np.save(pb, p)
    return path


def render(path, W, H, fx, pose, optkw, comp=None):
    rt = rb.RefTree(path)
    info = rt.info()
    c12 = synth.c2w_to_colmajor12(pose)
    opt = rb.make_options(**optkw)
    rin, din = comp if comp is not None else (None, None)
    f = rt.render_f32(W, H, fx, fx, c12, opt, rgba_in=rin, depth_in=din)
    u = rt.render_u8(W, H, fx, fx, c12, opt, rgba_in=rin, depth_in=din)
    rt.close()
    return f, u, info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden"))
    ap.add_argument("cases", nargs="*")
    args = ap.parse_args()
    os.makedirs(os.path.join(args.out, "frames"), exist_ok=True)
    with tempfile.TemporaryDirectory() as tmp:
        for name in CASES:
            if args.cases and name not in args.cases:
                continue
            st, W, H, pose, optkw, ndc = build_case(name)
            f, u, info = render(write_case_files(name, st, ndc, tmp), W, H, synth.focal_for(W), pose, optkw,
                                composite_inputs(name, W, H))
            assert bool(info["use_ndc"]) == (ndc is not None)
            np.savez_compressed(os.path.join(args.out, name + ".npz"), case=np.array(name), ref_f32=f, ref_u8=u)
            print(name, info, "alpha mean %.3f" % f[..., 3].mean(), "rgb mean %.3f" % f[..., :3].mean(), flush=True)
        for name in FRAME_CASES:
            if args.cases and name not in args.cases:
                continue
            tree, W, H, fx, pose = frame_case(name)
            f, u, info = render(write_case_files(name, tree, None, tmp), W, H, fx, pose, {})
            np.savez_compressed(os.path.join(args.out, "frames", name + ".npz"), **frame_record(f, u))
            print(name, info, "alpha mean %.3f" % f[..., 3].mean(), "rgb mean %.3f" % f[..., :3].mean(), flush=True)

        os.makedirs(os.path.join(args.out, "rays"), exist_ok=True)
        for name, tree_case in RAY_CASES.items():
            if args.cases and name not in args.cases:
                continue
            bc = build_case(tree_case)
            st, W, H, pose, optkw, ndc = bc
            path = write_case_files(name, st, ndc, tmp)
            opt = rb.make_options(**optkw)
            # the contract on the reference side: its ray tap on a camera's rays == its per-pixel tap
            fx = synth.focal_for(W)
            c12 = synth.c2w_to_colmajor12(pose)
            co, cd = rayb.camera_rays(ob.make_camera(W, H, fx, fx, c12))
            frame, _, _ = render(path, W, H, fx, pose, optkw)
            assert np.array_equal(rayb.ref_render_rays(path, opt, co, cd), frame.reshape(-1, 4)), name
            o, d, t = make_rays(name, bc)
            f = rayb.ref_render_rays(path, opt, o, d, t)
            np.savez_compressed(os.path.join(args.out, "rays", name + ".npz"), case=np.array(name), origins=o, dirs=d,
                                t_max=t, ref_f32=f)
            print(name, "alpha mean %.3f" % f[:, 3].mean(), "hit %.3f" % (f[:, 3] > 0).mean(), flush=True)


if __name__ == "__main__":
    main()
