#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 PlenOctree ray-marcher.

Metric (BASELINE.json): Mrays/s at 800x800 (FPS = Mrays/s / 0.64), plus the achieved
algorithmic GB/s against the measured HBM peak.  Workload = BASELINE config 2 ("lego tree.npz,
800x800, 200 test poses").  The real scene is an external download: when $VOLREND_DATA/lego/tree.npz
(+ pose/*.txt) exists it is used, otherwise the seeded lego-like stand-in of volrend_b200/synth.py;
`config.workload` says which.

  step      one sweep of the 200-pose NeRF-synthetic test orbit (main_headless.cpp:208-223),
            rendered by ONE batched launch of the fused march kernel (vr_render_batch)
  value     W*H*views / device time, frames stay in HBM (whole job, all ranks)
  e2e       same sweep through the host-buffer entry point (vr_render_frames_host): launches of 8
            poses each on two streams, cameras in via a 64-byte-per-pose H2D copy, every RGBA8 frame
            copied to pinned host memory inside the timed region
  cli       (N = 1, when build/volrend_headless exists) the reference's UNCHANGED main_headless.cpp,
            n3tree.cpp, camera.cpp, opts.cpp linked against this backend, timed by its own event
            pair (main_headless.cpp:203-228): the literal drop-in number
  N > 1     weak scaling: each rank renders its own 200 views of a 200*N-view orbit (tree
            replicated) and the finished RGBA8 frames are gathered on rank 0 -- by the copy engines
            over NVLink into a peer-mapped buffer (default; no SM-resident collective competes with
            the persistent march kernel) or by one NCCL gather (--gather nccl)
  --impl reference   the UNMODIFIED reference CUDA renderer (oracle/_ref/libvolrend_ref.so,
            built from /root/reference by oracle/Makefile.ref) on the same tree and poses, timed
            exactly like main_headless.cpp:203-228; falls back to the CPU oracle port when that
            library is absent.
  --workload config4   BASELINE config 4 instead: depth-11 SH25 tree, 1920x1080, 40 poses per step, STRONG scaling --
            every rank renders its interleaved 8-row bands of all frames with one launch and the copy
            engines scatter them into the frames on rank 0 (2-D peer copies); the reassembled frames are
            compared with a single-GPU render (`config.reassembly_identical_to_single_gpu`).
  --dump-outputs DIR   the RGBA8 frames of the last timed step (and of the last e2e step) as float32 .npy files, the
            same fixed sample of pixels on every run, so that two builds can be compared output for output.

Kernels: batches (the `value` / `e2e` legs) run the inline-shading kernel, single-view launches (the `cli` leg,
launch_renderer) the shading-queue kernel; `config.kernel_variant` names the batch kernel (DESIGN.md 4).
"""
from __future__ import annotations

import argparse
import ctypes
import datetime
import json
import math
import os
import re
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

W = H = 800
N_POSES = 200
WORKLOAD_SYNTH = ("synthetic lego-like SH16 N3Tree stand-in (depth 10, seed 0; real lego tree.npz is an external "
                  "download), 800x800, 200 NeRF-synthetic test-orbit poses, default RenderOptions")
DUMP_PIXELS = 1 << 20          # --dump-outputs: at most 1 Mi RGBA pixels (16 MB as float32) per array
_TMP = None


def tmp_dir() -> str:
    """This run's scratch directory (tree.npz and pose files for the CLI and reference legs), removed at exit."""
    global _TMP
    if _TMP is None:
        _TMP = tempfile.TemporaryDirectory(prefix="vr_bench_")
    return _TMP.name


def frame_sample(frames) -> np.ndarray:
    """float32 [n, 4] copy of an RGBA8 frame stack [V, H, W, 4] (CUDA or host tensor): every pixel when there are at
    most DUMP_PIXELS, else the same DUMP_PIXELS pixels on every run (seed 0, in index order)."""
    import torch
    px = frames.reshape(-1, 4)
    if px.shape[0] > DUMP_PIXELS:
        idx = np.sort(np.random.default_rng(0).choice(px.shape[0], DUMP_PIXELS, replace=False))
        px = px[torch.from_numpy(idx).to(px.device)]
    return px.float().cpu().numpy()


def dump_outputs(out_dir: str, arrays: dict) -> None:
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def usable_cores() -> int:
    """Host threads this process may really use: affinity mask, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, math.ceil(int(txt[0]) / int(txt[1]))))
            else:
                quota = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    n = min(n, max(1, math.ceil(quota / period)))
            break
        except Exception:  # noqa: BLE001
            continue
    return max(1, n)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md recipe).  Started BEFORE the warm-up so that
    its start-up time is not part of the window; samples are attributed to the timed region by their
    nvidia-smi timestamps."""

    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []
        self.t0 = self.t1 = None

    def start(self, wait_s: float = 4.0):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "50"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            t_end = time.time() + wait_s
            while not self.lines and time.time() < t_end:      # first sample has arrived: the sampler is live
                time.sleep(0.02)
        except Exception:  # noqa: BLE001
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    @staticmethod
    def _ts(s: str):
        try:
            return datetime.datetime.strptime(s.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except ValueError:
            return None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.12)
        self.proc.terminate()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        sm, mx, reasons, sm_all = [], [], set(), []
        for arrived, ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 10:
                continue
            try:
                clk, cmax = float(f[2]), float(f[3])
            except ValueError:
                continue
            ts = self._ts(f[0]) or arrived
            sm_all.append(clk)
            if self.t0 is not None and not (self.t0 - 0.05 <= ts <= (self.t1 or time.time()) + 0.05):
                continue
            sm.append(clk)
            mx.append(cmax)
            for n, v in zip(names, f[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "samples_total": len(sm_all),
                "window_s": None if self.t0 is None else round((self.t1 or time.time()) - self.t0, 3)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(p))["hbm_gbs"]), "of measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001
        return 6650.0, "of fallback (6.65 TB/s, B200_PROFILING.md)"


class Scene:
    """The benchmark tree + poses: real data from $VOLREND_DATA when supplied, else the synthetic stand-in."""

    def __init__(self, rank: int, world: int):
        from volrend_b200 import synth
        self.depth = env_int("VR_BENCH_DEPTH", 10)
        self.real_npz = None
        root = os.environ.get("VOLREND_DATA", "")
        cand = os.path.join(root, "lego", "tree.npz") if root else ""
        poses_all = None
        if cand and os.path.exists(cand):
            self.real_npz = cand
            pdir = os.path.join(root, "lego", "pose")
            files = sorted(f for f in os.listdir(pdir)) if os.path.isdir(pdir) else []
            mats = [np.loadtxt(os.path.join(pdir, f)).reshape(4, 4) for f in files if f.endswith(".txt")]
            if mats:
                poses_all = np.stack(mats).astype(np.float32)
        if poses_all is None or len(poses_all) < N_POSES * world:
            poses_all = synth.nerf_synthetic_test_poses(N_POSES * world)
        self.poses = poses_all[rank::world][:N_POSES]
        self.st = None if self.real_npz else synth.make_tree("lego", depth=self.depth, basis_dim=16, seed=0)
        self.workload = (f"{self.real_npz} (real scene from $VOLREND_DATA), 800x800, {N_POSES} poses, default RenderOptions"
                         if self.real_npz else WORKLOAD_SYNTH)

    def device_tree(self):
        from volrend_b200 import N3Tree
        return N3Tree(self.real_npz) if self.real_npz else N3Tree.from_synth(self.st)

    def oracle_tree(self):
        from oracle import binding as ob
        if self.real_npz:
            z = np.load(self.real_npz)
            fmt = str(z["data_format"]) if "data_format" in z else ("RGBA" if int(z["data_dim"]) == 4 else f"SH{(int(z['data_dim']) - 1) // 3}")
            scale = z["invradius3"] if "invradius3" in z else np.full(3, float(z["invradius"]), np.float32)
            return ob.OracleTree(z["child"], z["data"], z["offset"], scale, int(z["data_dim"]), fmt)
        return ob.OracleTree.from_synth(self.st)

    def npz_path(self) -> str:
        if self.real_npz:
            return self.real_npz
        path = os.path.join(tmp_dir(), "vr_bench_tree.npz")
        if not os.path.exists(path):
            self.st.save_npz(path)
        return path


def cpu_baseline(scene: Scene, budget_s: float = 12.0):
    """Oracle port on the host cores, bounded sample of the same workload (full 800x800 frames)."""
    from oracle import binding as ob
    from volrend_b200 import synth
    cores = usable_cores()
    ot = scene.oracle_tree()
    opt = ob.make_options()
    poses = scene.poses
    t0 = time.perf_counter()
    n = 0
    while True:
        pose = poses[(n * 37) % len(poses)]
        cam = ob.make_camera(W, H, synth.focal_for(W), synth.focal_for(W), synth.c2w_to_colmajor12(pose))
        ob.render(ot, cam, opt, want_float=False, want_u8=True, nthreads=cores)
        n += 1
        el = time.perf_counter() - t0
        if el > budget_s or n >= 400:
            break
    return {"value": W * H * n / el / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port",
            "sample": f"{n} full 800x800 frames of the workload, oracle/march_oracle.c with {cores} threads "
                      f"(affinity/cgroup-limited; os.cpu_count() = {os.cpu_count()}), {el:.1f} s"}


class StdoutToStderr:
    """The reference loader prints with printf and no newline (src/n3tree.cpp:264 'INFO: Scale ...'); keep
    everything foreign code writes to fd 1 away from the one JSON line this script prints."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        try:
            ctypes.CDLL(None).fflush(None)
        except Exception:  # noqa: BLE001
            pass
        os.dup2(self._saved, 1)
        os.close(self._saved)
        return False


def cli_leg(scene: Scene, exe: str, n_frames: int = N_POSES):
    """ms/frame printed by a volrend_headless binary (main_headless.cpp:203-231) on the bench tree."""
    from volrend_b200 import synth
    if not os.path.exists(exe):
        return None
    try:
        npz = scene.npz_path()
        pdir = os.path.join(tmp_dir(), "vr_bench_poses")
        ppaths = synth.write_pose_files(scene.poses[:n_frames], pdir, synth.focal_for(W))
        cmd = [exe, npz, "-w", str(W), "-h", str(H), "--fx", str(synth.focal_for(W))] + ppaths
        best = None
        for _ in range(2):   # first run pays the page cache / module load
            r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
            # the loader's "INFO: Scale %f %f %f" has no newline (src/n3tree.cpp:264), so the "ms per frame" line is
            # glued to it; the "fps" line (main_headless.cpp:231) stands alone: ms = 1000 / fps
            m = re.search(r"^\s*([0-9]+\.[0-9]+) fps\s*$", r.stdout, re.M)
            if r.returncode != 0 or not m:
                return {"error": (r.stderr or r.stdout)[-300:]}
            ms = 1000.0 / float(m.group(1))
            best = ms if best is None else min(best, ms)
        return {"ms_per_frame": best, "value": W * H / best / 1e3, "unit": "Mrays/s", "frames": n_frames,
                "binary": os.path.relpath(exe, ROOT),
                "timing": "the binary's own cudaEvent pair around its pose loop (main_headless.cpp:203-228), best of 2 runs"}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)[:300]}


def reference_arm(args, rank, world):
    """--impl reference: the reference's own CUDA renderer (or the CPU port when it is absent)."""
    if rank != 0:
        return
    with StdoutToStderr():
        line = reference_config4(args) if args.workload == "config4" else _reference_line(args)
    print(json.dumps(line), flush=True)


def _reference_line(args):
    from volrend_b200 import synth
    scene = Scene(0, 1)
    poses = scene.poses
    line = {"impl": "reference", "metric": "Mrays/s @ 800x800", "unit": "Mrays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic" if not scene.real_npz else "real",
            "config": {"workload": scene.workload, "tree_depth": scene.depth,
                       "l2": "inputs larger than L2 (1.1 GB tree, a different pose every frame)"}}
    from oracle import ref_binding as rb
    import torch
    if rb.available() and torch.cuda.is_available():
        rt = rb.RefTree(scene.npz_path())
        c12 = np.stack([synth.c2w_to_colmajor12(p) for p in poses])
        fx = synth.focal_for(W)
        opt = rb.make_options()
        host = torch.empty((N_POSES, H, W, 4), dtype=torch.uint8).pin_memory()
        cs = ClockSampler(0)
        cs.start()
        for _ in range(args.warmup):
            rt.time_frames(W, H, fx, fx, c12, opt)
        cs.begin()
        ms = [rt.time_frames(W, H, fx, fx, c12, opt) for _ in range(args.steps)]
        cs.end()
        clocks = cs.stop()
        for _ in range(min(args.warmup, 2)):
            rt.time_frames(W, H, fx, fx, c12, opt, with_d2h=True, host_out=host)
        ms_e = [rt.time_frames(W, H, fx, fx, c12, opt, with_d2h=True, host_out=host) for _ in range(args.steps)]
        rt.close()
        t, te = sum(ms) / len(ms), sum(ms_e) / len(ms_e)
        val = W * H * N_POSES / t / 1e3
        line.update({"value": val, "ms_per_step": t, "clocks": clocks, "gpu_launches": N_POSES * args.steps,
                     "reference": "volrend::launch_renderer from /root/reference/src/cuda/volrend.cu, built -arch=sm_100 "
                                  "by oracle/Makefile.ref, timed as main_headless.cpp:203-228 on the same B200",
                     "e2e": {"value": W * H * N_POSES / te / 1e3, "unit": "Mrays/s",
                             "h2d_bytes_per_step": 48 * N_POSES, "d2h_bytes_per_step": 4 * W * H * N_POSES}})
        if not args.no_cli:
            cli = cli_leg(scene, os.path.join(ROOT, "oracle", "_ref", "volrend_headless_ref"))
            if cli:
                line["cli"] = cli
        line["cpu_baseline"] = cpu_baseline(scene, budget_s=8.0)
    else:
        # no reference binary (or no GPU): the CPU oracle port with all usable host threads
        per_step = []
        cb = None
        for _ in range(max(1, min(args.steps, 3))):
            cb = cpu_baseline(scene, budget_s=8.0)
            per_step.append(cb["value"])
        val = float(np.mean(per_step))
        line.update({"value": val, "ms_per_step": W * H * N_POSES / val / 1e3, "gpu_launches": 0,
                     "cpu_baseline": {**cb, "value": val},
                     "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    return line


class PeerGather:
    """Frames of every rank land in ONE buffer on rank 0, written by the ranks' copy engines over NVLink
    (cudaMemcpyAsync into the IPC-mapped buffer): no kernel of the gather runs on any SM."""

    def __init__(self, dist, lib, rank, world, bytes_per_rank):
        self.lib, self.rank, self.world, self.n = lib, rank, world, bytes_per_rank
        self.base = ctypes.c_void_p()
        self.mapped = None
        handle = ctypes.create_string_buffer(64)
        if rank == 0:
            assert lib.vr_dev_alloc(bytes_per_rank * world, ctypes.byref(self.base)) == 0, lib.vr_last_error()
            assert lib.vr_ipc_export(self.base, handle) == 0, lib.vr_last_error()
        obj = [bytes(handle.raw) if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        if rank == 0:
            self.root = self.base.value           # start of rank 0's buffer as THIS process addresses it
        else:
            p = ctypes.c_void_p()
            assert lib.vr_ipc_open(obj[0], ctypes.byref(p)) == 0, lib.vr_last_error()
            self.mapped = p
            self.root = p.value
        self.dst = self.root + rank * bytes_per_rank

    def send(self, src_ptr: int, offset: int, nbytes: int, stream_ptr: int):
        assert self.lib.vr_copy_async(ctypes.c_void_p(self.dst + offset), ctypes.c_void_p(src_ptr), nbytes,
                                      ctypes.c_void_p(stream_ptr)) == 0, self.lib.vr_last_error()

    def send2d(self, root_offset: int, dpitch: int, src_ptr: int, spitch: int, width: int, rows: int, stream_ptr: int):
        """Strided (band) copy to byte `root_offset` of rank 0's buffer."""
        assert self.lib.vr_copy2d_async(ctypes.c_void_p(self.root + root_offset), dpitch, ctypes.c_void_p(src_ptr), spitch,
                                        width, rows, ctypes.c_void_p(stream_ptr)) == 0, self.lib.vr_last_error()

    def close(self):
        if self.mapped is not None:
            self.lib.vr_ipc_close(self.mapped)
        if self.rank == 0 and self.base:
            self.lib.vr_dev_free(self.base)


C4_W, C4_H, C4_FX, C4_POSES, C4_BAND = 1920, 1080, 1500.0, 40, 8
C4_WORKLOAD = ("BASELINE config 4: synthetic depth-11 SH25 octree (gyroid shell, seed 0), 1920x1080, 40 orbit poses per step, "
               "every frame ray-tile sharded over the GPUs (interleaved 8-row bands)")


def config4_scene():
    from volrend_b200 import synth
    st = synth.make_tree("gyroid_small", depth=11, basis_dim=25, seed=0, band_cells=1.0)
    poses = synth.nerf_synthetic_test_poses(C4_POSES, radius=1.6, elev_deg=25.0)
    return st, poses


def reference_config4(args):
    """--impl reference --workload config4: the reference kernel on the same tree and poses at 1080p."""
    from volrend_b200 import synth
    from oracle import ref_binding as rb
    import torch
    line = {"impl": "reference", "metric": "Mrays/s @ 1920x1080", "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": {"workload": C4_WORKLOAD}}
    if not (rb.available() and torch.cuda.is_available()):
        line["unavailable"] = "oracle/_ref not built or no GPU"
        return line
    st, poses = config4_scene()
    path = os.path.join(tmp_dir(), "vr_config4_tree.npz")
    st.save_npz(path)
    rt = rb.RefTree(path)
    c12 = np.stack([synth.c2w_to_colmajor12(p) for p in poses])
    opt = rb.make_options()
    for _ in range(args.warmup):
        rt.time_frames(C4_W, C4_H, C4_FX, C4_FX, c12, opt)
    ms = [rt.time_frames(C4_W, C4_H, C4_FX, C4_FX, c12, opt) for _ in range(args.steps)]
    host = torch.empty((C4_POSES, C4_H, C4_W, 4), dtype=torch.uint8).pin_memory()
    ms_e = [rt.time_frames(C4_W, C4_H, C4_FX, C4_FX, c12, opt, with_d2h=True, host_out=host) for _ in range(args.steps)]
    rt.close()
    t, te = float(np.mean(ms)), float(np.mean(ms_e))
    rays = C4_W * C4_H * C4_POSES
    line.update({"value": rays / t / 1e3, "ms_per_step": t, "gpu_launches": C4_POSES * args.steps,
                 "reference": "volrend::launch_renderer (oracle/_ref, -arch=sm_100), one GPU: the reference has no multi-GPU path",
                 "e2e": {"value": rays / te / 1e3, "unit": "Mrays/s", "h2d_bytes_per_step": 48 * C4_POSES,
                         "d2h_bytes_per_step": 4 * C4_W * C4_H * C4_POSES}})
    return line


def main_config4(args, rank, world, local_rank):
    """--workload config4: STRONG scaling of one fixed job (40 frames of 1920x1080 on the depth-11 SH25 tree).
    Every rank renders its bands of ALL frames with one launch (vr_render_bands_batch); the copy engines scatter
    the compact bands straight into the frames on rank 0 (2-D peer copies into an IPC-mapped buffer)."""
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from volrend_b200 import Camera, N3Tree, RenderOptions, lib, render_bands_batch, render_batch
    from volrend_b200 import dist as vd
    if lib().vr_set_variant(args.variant) != 0:
        raise SystemExit(f"kernel variant {args.variant} is not built into this library")
    st, poses = config4_scene()
    tree = N3Tree.from_synth(st)
    info = tree.info()
    cams = []
    for p in poses:
        c = Camera(C4_W, C4_H, C4_FX, C4_FX)
        c.set_c2w(p)
        cams.append(c)
    opt = RenderOptions()
    row, frame = 4 * C4_W, 4 * C4_W * C4_H
    rows = vd.band_rows(C4_H, C4_BAND, world, rank)
    plan = vd.band_scatter_plan(C4_W, C4_H, C4_BAND, world, rank)
    peer = PeerGather(dist, lib(), rank, world, frame * C4_POSES // world + 1) if world > 1 else None
    if world == 1:
        frames = torch.zeros((C4_POSES, C4_H, C4_W, 4), dtype=torch.uint8, device=dev)
    local = [torch.zeros((C4_POSES, max(rows, 1), C4_W, 4), dtype=torch.uint8, device=dev) for _ in range(2)] if world > 1 else None
    comm = torch.cuda.Stream(device=dev) if world > 1 else None
    sent = [None, None]

    # work counters of the whole job (rank 0, untimed) for the roofline
    S = D = SH = HIT = FETCH = 0
    if rank == 0:
        cnt = torch.zeros(5, dtype=torch.int64, device=dev)
        tmp = torch.zeros((C4_POSES, C4_H, C4_W, 4), dtype=torch.uint8, device=dev) if world > 1 else frames
        render_batch(tree, cams, opt, tmp, counters=cnt)
        torch.cuda.synchronize()
        S, D, SH, HIT, FETCH = [int(v) for v in cnt.cpu().tolist()]
        solo = tmp[::13].cpu().numpy()           # single-GPU frames 0, 13, 26, 39 for the reassembly check
        del tmp
    a_step = 4 * D + 2 * S + 6 * 25 * SH + 4 * C4_W * C4_H * C4_POSES
    c_step = 4 * FETCH + info["rec_bytes"] * SH + 4 * C4_W * C4_H * C4_POSES

    def step(i):
        cur = torch.cuda.current_stream()
        if world == 1:
            render_batch(tree, cams, opt, frames)
            return
        k = i & 1
        if sent[k] is not None:
            cur.wait_event(sent[k])
        render_bands_batch(tree, cams, opt, C4_BAND, world, rank, local[k])
        done = torch.cuda.Event()
        done.record(cur)
        comm.wait_event(done)
        base = local[k].data_ptr()
        for v in range(C4_POSES):
            for (do, dp, so, sp, wb, n) in plan:
                peer.send2d(v * frame + do, dp, base + v * rows * row + so, sp, wb, n, comm.cuda_stream)
        ev = torch.cuda.Event()
        ev.record(comm)
        sent[k] = ev

    def sync_all():
        if world > 1:
            torch.cuda.current_stream().wait_stream(comm)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    cs = ClockSampler(local_rank)
    if rank == 0:
        cs.start()
    for i in range(args.warmup):
        step(i)
    sync_all()
    launches0 = lib().vr_launch_count()
    kern = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cs.begin()
    e0.record()
    for i in range(args.steps):
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        step(i)
        k1.record()
        kern.append((k0, k1))
    if world > 1:
        torch.cuda.current_stream().wait_stream(comm)
    e1.record()
    sync_all()
    launches = lib().vr_launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    extra = 0
    while rank == 0 and world == 1 and time.time() - cs.t0 < 1.2:
        step(extra)
        torch.cuda.synchronize()
        extra += 1
    cs.end()
    clocks = cs.stop() if rank == 0 else None
    kms = float(np.mean([a.elapsed_time(b) for a, b in kern]))
    t = torch.tensor([ms_total, kms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step, kms_max = float(t[0].item()) / args.steps, float(t[1].item())

    # reassembly check + e2e (frames to pinned host memory on rank 0 inside the timed region)
    identical = None
    host = torch.empty((C4_POSES, C4_H, C4_W, 4), dtype=torch.uint8).pin_memory() if rank == 0 else None

    def e2e_step(i):
        step(i)
        sync_all()                                 # every rank's bands have landed on rank 0
        if rank == 0:
            src = frames.data_ptr() if world == 1 else peer.root
            lib().vr_copy_async(ctypes.c_void_p(host.data_ptr()), ctypes.c_void_p(src), frame * C4_POSES, None)
            torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    e2e_step(0)
    if rank == 0:
        identical = bool(np.array_equal(host[::13].numpy(), solo))
    t0 = time.perf_counter()
    n_e2e = args.steps
    for i in range(n_e2e):
        e2e_step(i)
    te = torch.tensor([(time.perf_counter() - t0) * 1e3 / n_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item())

    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"frames": frame_sample(host)})
        peak, peak_note = measured_peak()
        rays = C4_W * C4_H * C4_POSES
        line = {
            "metric": "Mrays/s @ 1920x1080", "value": rays / ms_step / 1e3, "unit": "Mrays/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "ms_per_frame": ms_step / C4_POSES, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "fps": C4_POSES / ms_step * 1e3,
            "config": {"workload": C4_WORKLOAD, "tree_depth": info["max_depth"], "nodes": info["capacity"],
                       "tree_bytes_device": info["kernel_bytes"], "views_per_step": C4_POSES,
                       "parallelism": f"ray tiles x{world}" + ("" if world == 1 else ", bands to rank 0 by 2-D peer copies (copy engines, NVLink)"),
                       "kernel_variant": lib().vr_tree_variant(tree._handle), "reassembly_identical_to_single_gpu": identical,
                       "l2": "inputs larger than L2 (1.6 GB of tables + records, a different pose every frame); no flush needed"},
            "roofline": {"bound": "hbm", "achieved": a_step / world / (kms_max * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": a_step / world / (kms_max * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_note,
                         "algorithmic_bytes_per_launch": a_step / world, "kernel_ms_per_launch": kms_max,
                         "compulsory": {"bytes_per_launch": c_step / world, "achieved": c_step / world / (kms_max * 1e-3) / 1e9,
                                        "frac": c_step / world / (kms_max * 1e-3) / 1e9 / peak},
                         "counters": {"samples": S, "child_loads": D, "shaded": SH, "rays_hit": HIT, "node_fetches": FETCH},
                         "note": "per GPU: 1/N of the job's algorithmic bytes (SURVEY 8d) over the slowest rank's launch time"},
            "e2e": {"value": rays / e2e_ms / 1e3, "unit": "Mrays/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": 64 * C4_POSES * world,
                    "d2h_bytes_per_step": frame * C4_POSES},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        peer.close()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="config2", choices=["config2", "config4"],
                    help="config2 (default, the headline): lego 800x800, 200 poses, weak scaling by views; "
                         "config4: depth-11 SH25 1920x1080, strong scaling by ray tiles")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--variant", type=int, default=0, help="kernel variant (0 = default)")
    ap.add_argument("--gather", default="p2p", choices=["p2p", "nccl"], help="N>1: how frames reach rank 0")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cli", action="store_true", help="skip the volrend_headless leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the RGBA8 frames of the last timed step to DIR/<name>.npy as float32 (rank 0; a fixed "
                         "sample of %d pixels when there are more): frames (batch), frames_e2e (host-buffer leg); "
                         "config4: frames (reassembled)" % DUMP_PIXELS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3)

    rank = env_int("RANK", 0)
    world = env_int("WORLD_SIZE", 1)
    local_rank = env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return
    if args.workload == "config4":
        main_config4(args, rank, world, local_rank)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: volrend_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    from volrend_b200 import Camera, RenderOptions, lib, render_batch, render_frames_host, synth
    if lib().vr_set_variant(args.variant) != 0:
        raise SystemExit(f"kernel variant {args.variant} is not built into this library")
    scene = Scene(rank, world)
    tree = scene.device_tree()
    info = tree.info()
    cams = []
    for p in scene.poses:
        c = Camera(W, H, synth.focal_for(W), synth.focal_for(W))
        c.set_c2w(p)
        cams.append(c)
    opt = RenderOptions()
    imgs = [torch.zeros((N_POSES, H, W, 4), dtype=torch.uint8, device=dev) for _ in range(2)]
    host = torch.empty((N_POSES, H, W, 4), dtype=torch.uint8).pin_memory()
    frame_bytes = 4 * W * H
    gathered = None
    peer = None
    if world > 1:
        if args.gather == "p2p":
            try:
                peer = PeerGather(dist, lib(), rank, world, frame_bytes * N_POSES)
            except AssertionError as e:   # no peer access on this box: fall back to the NCCL gather
                print(f"[bench] peer-mapped gather unavailable ({e}); using NCCL", file=sys.stderr)
                peer = None
        if peer is None and rank == 0:
            gathered = [torch.empty_like(imgs[0]) for _ in range(world)]

    # ---- work counters of this rank's sweep from the instrumented kernel (not timed)
    cnt = torch.zeros(5, dtype=torch.int64, device=dev)
    render_batch(tree, cams, opt, imgs[0], counters=cnt)
    torch.cuda.synchronize()
    S, D, SH, HIT, FETCH = [int(v) for v in cnt.cpu().tolist()]
    basis = max(info["kernel_basis"], 1)
    a_step = 4 * D + 2 * S + 6 * basis * SH + 4 * W * H * N_POSES                 # SURVEY 8d: the reference's touches
    c_step = 4 * FETCH + info["rec_bytes"] * SH + 4 * W * H * N_POSES             # compulsory bytes of THIS kernel

    comm = torch.cuda.Stream(device=dev) if world > 1 else None
    gathered_ev = [None, None]
    n_chunks = 1 if world == 1 else 4     # N > 1: chunk k travels while chunk k+1 renders

    def step(i):
        buf = imgs[i & 1]
        cur = torch.cuda.current_stream()
        if world > 1 and gathered_ev[i & 1] is not None:
            cur.wait_event(gathered_ev[i & 1])      # this buffer's previous transfer has finished
        if world == 1:
            render_batch(tree, cams, opt, buf)
            return
        per = (N_POSES + n_chunks - 1) // n_chunks
        ev = None
        for c0 in range(0, N_POSES, per):
            c1 = min(N_POSES, c0 + per)
            render_batch(tree, cams[c0:c1], opt, buf[c0:c1])
            done = torch.cuda.Event()
            done.record(cur)
            comm.wait_event(done)
            with torch.cuda.stream(comm):
                if peer is not None:
                    # copy engine -> rank 0's buffer (rank 0 moves its own frames too, so its result is complete)
                    peer.send(buf[c0:c1].data_ptr(), c0 * frame_bytes, (c1 - c0) * frame_bytes, comm.cuda_stream)
                else:
                    dist.gather(buf[c0:c1], [g[c0:c1] for g in gathered] if rank == 0 else None, dst=0)
                ev = torch.cuda.Event()
                ev.record(comm)
        gathered_ev[i & 1] = ev

    def sync_all():
        if world > 1:
            torch.cuda.current_stream().wait_stream(comm)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    cs = ClockSampler(local_rank)
    if rank == 0:
        cs.start()
    for i in range(args.warmup):
        step(i)
    sync_all()
    launches0 = lib().vr_launch_count()
    kern_ms = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    cs.begin()
    e0.record()
    for i in range(args.steps):
        k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        k0.record()
        step(i)
        k1.record()
        kern_ms.append((k0, k1))
    if world > 1:
        torch.cuda.current_stream().wait_stream(comm)
    e1.record()
    sync_all()
    launches = lib().vr_launch_count() - launches0
    ms_total = e0.elapsed_time(e1)
    outputs = {"frames": frame_sample(imgs[(args.steps - 1) & 1])} if args.dump_outputs and rank == 0 else None
    # keep the identical load running (untimed) until the clock sampler has covered >= 1.2 s of it
    extra = 0
    while rank == 0 and world == 1 and time.time() - cs.t0 < 1.2:
        step(extra)
        torch.cuda.synchronize()
        extra += 1
    cs.end()
    clocks = cs.stop() if rank == 0 else None
    if clocks is not None:
        clocks["note"] = (f"window = the {args.steps} timed steps + {extra} identical untimed steps right behind them "
                          "(nvidia-smi samples every 50 ms)")
    kms = float(np.mean([a.elapsed_time(b) for a, b in kern_ms]))
    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_step = ms_total / args.steps

    # ---- e2e: host-buffer entry point, D2H of every frame inside the timed region
    for _ in range(2):
        render_frames_host(tree, cams, opt, host)
    sync_all()
    t0 = time.perf_counter()
    e2e_steps = args.steps
    for _ in range(e2e_steps):
        render_frames_host(tree, cams, opt, host)
    torch.cuda.synchronize()
    te = torch.tensor([(time.perf_counter() - t0) * 1e3 / e2e_steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_ms = float(te.item())
    if outputs is not None:
        outputs["frames_e2e"] = frame_sample(host)

    if rank == 0:
        peak, peak_note = measured_peak()
        rays = W * H * N_POSES * world
        variant = lib().vr_tree_variant(tree._handle)
        traffic, traffic_src = None, None
        try:
            ns = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json")))
            want = "march_queue_kernel" if (variant & 15) == 7 else "march_persistent_kernel"
            if want in ns.get("kernel", ""):
                traffic = ns["dram_bytes_per_frame"] * N_POSES
                traffic_src = (f"profiles/ncu_summary.json: ncu --set full of {ns['kernel']} "
                               f"({ns.get('captured', 'capture commit not recorded')}), dram read+write per frame x {N_POSES}")
            else:
                traffic_src = f"profiles/ncu_summary.json is for {ns.get('kernel')}, not the kernel timed here: omitted"
        except Exception:  # noqa: BLE001
            pass
        line = {
            "metric": "Mrays/s @ 800x800", "value": rays / ms_step / 1e3, "unit": "Mrays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "real" if scene.real_npz else "synthetic",
            "fps": N_POSES * world / ms_step * 1e3,
            "config": {"workload": scene.workload, "tree_depth": info["max_depth"], "nodes": info["capacity"],
                       "tree_bytes_device": info["kernel_bytes"], "tree_bytes_resident": info["device_bytes"],
                       "views_per_step_per_gpu": N_POSES,
                       "parallelism": f"views x{world}" + ("" if world == 1 else
                                                            (", frames to rank 0 by copy engines over NVLink (peer-mapped buffer)"
                                                             if peer is not None else ", one NCCL gather per chunk")),
                       "kernel_variant": variant,
                       "l2": "inputs larger than L2 (1.4 GB of tables + records, a different pose every frame); no flush needed"},
            "roofline": {"bound": "hbm", "achieved": a_step / (kms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": a_step / (kms * 1e-3) / 1e9 / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": peak_note,
                         "algorithmic_bytes_per_launch": a_step, "kernel_ms_per_launch": kms,
                         "compulsory": {"bytes_per_launch": c_step, "achieved": c_step / (kms * 1e-3) / 1e9,
                                        "frac": c_step / (kms * 1e-3) / 1e9 / peak,
                                        "note": "bytes this kernel cannot avoid: 4 B per table word it fetches + one padded colour "
                                                "record per shaded sample + the RGBA8 output; the honest DRAM-side figure"},
                         "counters": {"samples": S, "child_loads": D, "shaded": SH, "rays_hit": HIT,
                                      "node_fetches": FETCH},
                         "note": "algorithmic bytes count the reference algorithm's touches (SURVEY 8d); "
                                 "this kernel skips most of the root-restart chain, see DESIGN.md"},
            "e2e": {"value": rays / e2e_ms / 1e3, "unit": "Mrays/s", "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": 64 * N_POSES * world, "d2h_bytes_per_step": 4 * W * H * N_POSES * world},
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
        if world == 1 and not args.no_cli:
            cli = cli_leg(scene, os.path.join(ROOT, "build", "volrend_headless"))
            if cli:
                line["cli"] = cli
        if not args.no_cpu_baseline and world == 1:
            with StdoutToStderr():
                line["cpu_baseline"] = cpu_baseline(scene)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        if peer is not None:
            torch.cuda.synchronize()
            peer.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
