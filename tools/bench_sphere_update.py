"""Moving spheres: rfx_update_spheres against reloading the scene, per animation step.

Scenes: scenes.synthetic_scene at 1024, 16 384 and 65 536 spheres (n_side 32, 128, 256: a sphere hierarchy, one light grid, the eye
grid).  Each is animated for --steps steps of scenes.sphere_bounce (height 1.5, radius pulse 0.2) with every sphere moving, and again
with every 16th sphere moving, and rendered at 1920x1080, depth 4, default camera, into a device-resident frame on a torch stream.
Prints one JSON line with, per scene and moving fraction (medians over the steps):
  * update_host_ms: host wall time of the rfx_update_spheres call, and update_host_no_grid_ms: the same call in a context with the
    light grids off (rfx_set_option "light_grids" 0), which does everything but the light-grid rebuild; grid_rebuild_ms is their
    difference;
  * update_device_ms: CUDA events on the caller's stream around the call (the list copy, k_sphere_scatter, k_sphere_refit, the grid
    uploads);
  * frame_ms: CUDA events around the frame that follows each update;
  * step_ms: host wall time of update + frame + stream synchronisation;
  * device_path_steps: how many updates returned 1;
  * refit quality: after the animation, the frame time of the refitted hierarchy against a fresh context loaded with the same final
    spheres (median of 8 frames each, CUDA events);
and per scene reload_step_ms: load_scene of the moved scene (every object through the C ABI again) + frame (which re-flattens on the
host) + synchronisation, with every sphere moving.  nvidia-smi's card name, power limit and max SM clock are read in the same run.
    python tools/bench_sphere_update.py [--steps 32] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from reflaxman_b200 import capi, scenes as S  # noqa: E402

W, H, DEPTH = 1920, 1080, 4
SIZES = [("1024", 32), ("16384", 128), ("65536", 256)]
HEIGHT, PULSE = 1.5, 0.2


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:   # reported, not fatal
        return "nvidia-smi failed: %s" % e


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert a.steps >= 1
    res = {"card": card(), "steps": a.steps, "size": "%dx%d" % (W, H), "depth": DEPTH, "height": HEIGHT, "pulse": PULSE, "scenes": {}}
    cam = [S.default_camera()]
    floor = S.synthetic_texture(256, 256, 3)
    sky = S.synthetic_texture(512, 384, 5)
    stream = torch.cuda.Stream()
    buf = torch.empty(W * H, dtype=torch.int32, device="cuda:0")
    med = lambda v: round(float(np.median(v)), 4)

    def frame(c):
        c.render_frames_device(cam, DEPTH, 1, buf.data_ptr(), stream.cuda_stream)

    def timed_frames(c, n=8):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        ev[0].record(stream)
        for k in range(n):
            frame(c)
            ev[k + 1].record(stream)
        stream.synchronize()
        return med([ev[k].elapsed_time(ev[k + 1]) for k in range(n)])

    def context(scene, grids=True):
        c = capi.Context(0)
        c.load_scene(scene)
        if not grids:
            c.set_option("light_grids", 0)
        c.set_seeds(12345, 12345); c.set_image_size(W, H)
        frame(c); frame(c); stream.synchronize()          # flatten, modules, eye grid, queue scratch
        obj, sp = S.sphere_bounce(scene, 0.0)
        c.update_spheres(obj, sp); frame(c); stream.synchronize()   # the update's own buffers
        return c

    for name, n_side in SIZES:
        scene = S.synthetic_scene(n_side, floor=floor, skybox=sky)
        steps = [S.sphere_bounce(scene, 2.0 * np.pi * k / a.steps, height=HEIGHT, pulse=PULSE) for k in range(1, a.steps + 1)]
        r = {"spheres": n_side * n_side}
        for frac, every in (("all", 1), ("1/16", 16)):
            moves = [(o[::every], s[::every]) for o, s in steps]
            q = {}
            c = context(scene)
            try:
                host, dev, fr, step, device_path = [], [], [], [], 0
                for obj, sp in moves:
                    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                    t0 = time.perf_counter()
                    e0.record(stream)
                    device_path += c.update_spheres(obj, sp)
                    t1 = time.perf_counter()
                    e1.record(stream)
                    frame(c)
                    e2.record(stream)
                    stream.synchronize()
                    t2 = time.perf_counter()
                    host.append(1e3 * (t1 - t0)); step.append(1e3 * (t2 - t0))
                    dev.append(e0.elapsed_time(e1)); fr.append(e1.elapsed_time(e2))
                st = c.stats()
                q.update(update_host_ms=med(host), update_device_ms=med(dev), frame_ms=med(fr), step_ms=med(step), device_path_steps=device_path,
                         bvh_spheres=st["bvh_spheres"], light_grids=st["light_grids"])
                q["refitted_frame_ms"] = timed_frames(c)
            finally:
                c.close()
            final = S.with_spheres(scene, *moves[-1])   # (every step moves the same spheres)
            c = capi.Context(0)
            try:
                c.load_scene(final)
                c.set_seeds(12345, 12345); c.set_image_size(W, H)
                frame(c); frame(c); stream.synchronize()
                q["fresh_frame_ms"] = timed_frames(c)
            finally:
                c.close()
            c = context(scene, grids=False)
            try:
                host = []
                for obj, sp in moves:
                    t0 = time.perf_counter()
                    c.update_spheres(obj, sp)
                    host.append(1e3 * (time.perf_counter() - t0))
                    frame(c)
                    stream.synchronize()
                q["update_host_no_grid_ms"] = med(host)
                q["grid_rebuild_ms"] = round(q["update_host_ms"] - q["update_host_no_grid_ms"], 4)
            finally:
                c.close()
            r[frac] = q
            print("done", name, frac, q, file=sys.stderr, flush=True)
        c = capi.Context(0)
        try:
            c.load_scene(scene)
            c.set_seeds(12345, 12345); c.set_image_size(W, H)
            frame(c); stream.synchronize()
            reload = []
            for moved in [S.with_spheres(scene, obj, sp) for obj, sp in steps]:
                t0 = time.perf_counter()
                c.load_scene(moved)
                frame(c)
                stream.synchronize()
                reload.append(1e3 * (time.perf_counter() - t0))
            r["reload_step_ms"] = med(reload)
        finally:
            c.close()
        res["scenes"][name] = r
        print("done", name, "reload", r["reload_step_ms"], file=sys.stderr, flush=True)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
