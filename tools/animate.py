"""Frame loop over a resident scene: an orbiting camera and bobbing spheres, rendered three ways per frame.

  (a) update   rtb200_scene_update (camera + every sphere, refit on the device) + rtb200_render_device
  (b) upload   rtb200_scene_upload (host BVH build, one H2D copy of the arena) + rtb200_render_device + release
  (c) rgb8     rtb200_render_rgb8 (upload, render, device->host copy)

Every path is timed on the host clock around work that ends in a device synchronise. Each frame's RGB8 output of (a) must
equal (c)'s bit for bit; the run fails otherwise. The refit kernels are timed alone in a separate torch.profiler pass. Runs
the cover scene and a ~100 k-sphere scenes.rtiow_config(half=158) scene (low spp, so the update cost shows against the frame).

    python tools/animate.py [--frames 24] [--png-dir DIR] [--json OUT.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(REPO, "rust-raytracer_b200"))
import rtb200 as R  # noqa: E402
from rtb200 import scenes  # noqa: E402


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return name, q


class Loop:
    """A scene whose sphere array is edited in place (numpy view of the ctypes rt_sphere array) frame by frame."""

    def __init__(self, cfg):
        self.sc = R.Scene.from_config(cfg, scenes.SCENES_DIR)
        self.sp = np.ctypeslib.as_array(self.sc._spheres)[: self.sc.n_spheres]
        self.y0 = self.sp["center"]["y"].copy()
        self.small = np.nonzero(np.abs(self.sp["radius"]) < 0.5)[0]
        self.cam = dict(self.sc.camera_params)
        lf = self.cam["look_from"]
        self.orbit_r, self.a0 = math.hypot(lf["x"], lf["z"]), math.atan2(lf["z"], lf["x"])

    def frame(self, f, n):
        y = self.y0.copy()
        y[self.small] += 0.15 * np.sin(0.6 * f + 0.37 * self.small)
        self.sp["center"]["y"] = y
        a = self.a0 + 0.5 * math.pi * f / max(n, 1)
        lf = self.cam["look_from"]
        self.sc.set_camera(look_from={"x": self.orbit_r * math.cos(a), "y": lf["y"], "z": self.orbit_r * math.sin(a)})
        self.sc.seed = 1000 + f


def run(label, cfg, n_frames, warmup, png_dir, out):
    import torch
    from torch.profiler import ProfilerActivity, profile

    L = Loop(cfg)
    sc = L.sc
    w, h, n = sc.c.width, sc.c.height, sc.n_spheres
    d8 = torch.zeros(w * h * 3, dtype=torch.uint8, device="cuda")
    rs = R.ResidentScene(sc)
    ta, tb, tc, tu, tup, dev_a = [], [], [], [], [], []
    h2d_upload = 0
    for f in range(-warmup, n_frames):
        L.frame(max(f, 0), n_frames)
        # (a) update + render
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rs.update(spheres=sc, camera=sc.c.camera, seed=sc.seed)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        st = rs.render(d8.data_ptr())
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        img_a = d8.cpu().numpy().reshape(h, w, 3)
        # (b) upload + render + release
        t3 = time.perf_counter()
        rb = R.ResidentScene(sc)
        torch.cuda.synchronize()
        t4 = time.perf_counter()
        rb.render(d8.data_ptr())
        rb.release()
        torch.cuda.synchronize()
        t5 = time.perf_counter()
        # (c) host in, host out
        img_c, st_c = R.render_rgb8(sc)
        t6 = time.perf_counter()
        if not np.array_equal(img_a, img_c):
            raise SystemExit(f"{label} frame {f}: update+render differs from render_rgb8")
        if f < 0:
            continue
        ta.append((t2 - t0) * 1e3); tu.append((t1 - t0) * 1e3); tb.append((t5 - t3) * 1e3); tup.append((t4 - t3) * 1e3)
        tc.append((t6 - t5) * 1e3); dev_a.append(st["device_ms"]); h2d_upload = st_c["h2d_bytes"]
        if png_dir:
            R.write_png(os.path.join(png_dir, f"{label}_frame_{f:03d}.png"), img_c)

    # refit kernels alone (profiler in its own pass: tracing slows the host)
    reps = 20
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            rs.update(spheres=sc)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.key_averages():
        if "rt_refit" in e.key:
            t = getattr(e, "device_time_total", None)
            if t is None:
                t = e.cuda_time_total
            short = next(k for k in ("spheres", "nodes", "maps", "levels") if f"rt_refit_{k}" in e.key)
            kern[short] = {"calls": e.count, "us_total": t}
    refit_us = sum(v["us_total"] for k, v in kern.items() if k in ("spheres", "nodes")) / reps
    info = rs.kernel_info()
    rs.release()

    med = lambda v: float(np.median(v))
    res = {"scene": label, "width": w, "height": h, "spp": sc.c.samples_per_pixel, "max_depth": sc.c.max_depth, "spheres": n,
           "bvh_nodes": info["bvh_nodes"], "bvh_depth": info["bvh_depth"], "frames": n_frames,
           "a_update_render_ms": med(ta), "a_update_only_ms": med(tu), "a_render_device_ms": med(dev_a),
           "b_upload_render_release_ms": med(tb), "b_upload_only_ms": med(tup), "c_render_rgb8_ms": med(tc),
           "refit_kernels_us_per_update": refit_us, "refit_kernels": kern,
           "h2d_bytes_per_frame_a": 64 * n, "h2d_bytes_per_frame_b_c": int(h2d_upload), "frames_bit_identical_a_c": True}
    print(f"{label}: {w}x{h} {sc.c.samples_per_pixel} spp depth {sc.c.max_depth}, {n} spheres, {info['bvh_nodes']} nodes, "
          f"median of {n_frames} frames (host clock + device synchronise):", file=out)
    print(f"  (a) update + render   {med(ta):9.3f} ms   (update alone {med(tu):.3f} ms, refit kernels {refit_us:.1f} us, "
          f"frame device time {med(dev_a):.3f} ms)   H2D {64 * n} B", file=out)
    print(f"  (b) upload + render   {med(tb):9.3f} ms   (upload alone {med(tup):.3f} ms)   H2D {int(h2d_upload)} B", file=out)
    print(f"  (c) render_rgb8       {med(tc):9.3f} ms", file=out)
    print(f"  refit kernels over {reps} updates: {json.dumps(kern)}", file=out)
    print(f"  (a) == (c) bit for bit on all {n_frames + warmup} frames", file=out)
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--frames", type=int, default=24)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--png-dir", default=None, help="write (c)'s frames as <scene>_frame_%%03d.png here")
    ap.add_argument("--json", default=None, help="write the results here")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this tool measures on the GPU only")
    if a.png_dir:
        os.makedirs(a.png_dir, exist_ok=True)
    name, q = card()
    print(f"device: {name}; nvidia-smi name, power.limit, clocks.max.sm: {q}")
    cases = [("cover", scenes._variant(scenes.cover_config(), 640, 360, 4, 50), a.frames),
             ("rtiow100k", scenes._variant(scenes.rtiow_config(158), 640, 360, 1, 8), max(a.frames // 3, 4))]
    results = [run(label, cfg, nf, a.warmup, a.png_dir, sys.stdout) for label, cfg, nf in cases]
    if a.json:
        with open(a.json, "w") as f:
            json.dump({"device": name, "nvidia_smi": q, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
