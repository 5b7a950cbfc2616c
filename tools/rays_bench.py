#!/usr/bin/env python
"""Throughput of caller-supplied ray batches vs camera batches on the config-2 tree (depth-10 SH16, 800x800,
200 orbit poses = 128 M rays), CUDA events after warm-up:
  (a) vr_render_batch of the 200 views (float output)
  (b) vr_render_rays over the same rays in camera (row-major) order, one launch
  (c) the same rays randomly permuted
Checks that (b)'s output equals (a)'s bit for bit; writes profiles/rays_bench.json (or --out).
  usage: rays_bench.py [--views 200] [--reps 5] [--out PATH]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from volrend_b200 import Camera, N3Tree, RenderOptions, camera_rays, render_batch, render_rays, synth  # noqa: E402


def timed(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        s.record(); fn(); e.record(); e.synchronize()
        ms.append(s.elapsed_time(e))
    return float(np.median(ms)), ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--views", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rays_bench.json"))
    a = ap.parse_args()
    W = H = 800
    tree = N3Tree.from_synth(synth.make_tree("lego", depth=10, basis_dim=16, seed=0))
    cams = []
    for p in synth.nerf_synthetic_test_poses(200)[: a.views]:
        c = Camera(W, H, synth.focal_for(W), synth.focal_for(W))
        c.set_c2w(p)
        cams.append(c)
    V, n = len(cams), len(cams) * W * H
    opt = RenderOptions()
    fa = torch.empty((V, H, W, 4), dtype=torch.float32, device="cuda")
    o = torch.empty((V, H, W, 3), dtype=torch.float32, device="cuda")
    d = torch.empty_like(o)
    for i, c in enumerate(cams):
        camera_rays(c, o[i], d[i])
    ta, ms_a = timed(lambda: render_batch(tree, cams, opt, None, float_out=fa), a.reps)
    fb = torch.empty_like(fa)
    tb, ms_b = timed(lambda: render_rays(tree, o, d, opt, fb), a.reps)
    torch.cuda.synchronize()
    bit_identical = bool(torch.equal(fa, fb))
    perm = torch.randperm(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))
    op, dp = o.reshape(-1, 3)[perm].contiguous(), d.reshape(-1, 3)[perm].contiguous()
    del o, d
    fc = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    tc, ms_c = timed(lambda: render_rays(tree, op, dp, opt, fc), a.reps)
    torch.cuda.synchronize()
    perm_ok = bool(torch.equal(fc, fb.reshape(-1, 4)[perm]))
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = dict(tree="config2 lego depth 10 SH16", width=W, height=H, views=V, rays=n, reps=a.reps,
               gpu=torch.cuda.get_device_name(0), nvidia_smi=q[0] if q else None, variant="default (inline shading)",
               ms=dict(batch=ta, rays_camera_order=tb, rays_permuted=tc),
               ms_all=dict(batch=ms_a, rays_camera_order=ms_b, rays_permuted=ms_c),
               grays_per_s=dict(batch=n / ta / 1e6, rays_camera_order=n / tb / 1e6, rays_permuted=n / tc / 1e6),
               ratio_b_over_a=ta / tb, ratio_c_over_a=ta / tc,
               rays_equal_batch_bit_for_bit=bit_identical, permuted_equal_permutation=perm_ok)
    print(json.dumps(res))
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    assert bit_identical and perm_ok


if __name__ == "__main__":
    main()
