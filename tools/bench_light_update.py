"""Moving lights: rfx_update_lights against reloading the scene, per animation step.

Scenes: scenes.synthetic_scene at 1024, 16 384 and 65 536 spheres (n_side 32, 128, 256: a sphere hierarchy, one light grid, the eye
grid) with the textured floor, wall and sky.  The sun orbits for --steps steps of scenes.sun_orbit (t = 0.2 k), each step one
rfx_update_lights call (the sun's grid built on the GPU) and one 1920x1080 depth-4 frame with the default camera into a device-resident
buffer on a torch stream.  Prints one JSON line with, per scene (medians over the steps):
  * update_host_ms: host wall time of the rfx_update_lights call;
  * update_device_ms: CUDA events on the caller's stream around the call (the stream is idle while the host works: the call, the record
    copies and the six grid-builder kernels);
  * build_device_ms: the update's device work alone: the stream is held by a sleep kernel while the host enqueues the update, and the
    events bracket only what the update queued (the copies and the grid build);
  * frame_ms: CUDA events around the frame that follows each update;
  * step_ms: host wall time of update + frame + stream synchronisation;
  * device_path_steps: how many updates returned 1, and light_grids: rfx_stats.light_grids at the end;
  * reload_step_ms: load_scene of the scene with the moved sun (every object through the C ABI again) + frame (which re-flattens on the
    host, light grid included) + synchronisation: the only way to move a light before rfx_update_lights.
nvidia-smi's card name, power limit and max SM clock are read in the same run.
    python tools/bench_light_update.py [--steps 32] [--out FILE]
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
DT = 0.2
HOLD_CYCLES = 20_000_000   # ~10 ms at the B200's clock: longer than any host call measured here


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
    res = {"card": card(), "steps": a.steps, "size": "%dx%d" % (W, H), "depth": DEPTH, "dt": DT, "scenes": {}}
    cam = [S.default_camera()]
    floor = S.synthetic_texture(256, 256, 3)
    sky = S.synthetic_texture(512, 384, 5)
    stream = torch.cuda.Stream()
    buf = torch.empty(W * H, dtype=torch.int32, device="cuda:0")
    med = lambda v: round(float(np.median(v)), 4)

    def frame(c):
        c.render_frames_device(cam, DEPTH, 1, buf.data_ptr(), stream.cuda_stream)

    for name, n_side in SIZES:
        scene = S.synthetic_scene(n_side, floor=floor, skybox=sky)
        steps = [S.sun_orbit(scene, DT * k) for k in range(1, a.steps + 1)]
        r = {"spheres": n_side * n_side}
        c = capi.Context(0)
        try:
            c.load_scene(scene)
            c.set_seeds(12345, 12345); c.set_image_size(W, H)
            frame(c); frame(c); stream.synchronize()          # flatten, modules, eye grid, queue scratch
            c.update_lights(*S.sun_orbit(scene, 0.0)); frame(c); stream.synchronize()   # the builder's first launches
            host, dev, fr, step, device_path = [], [], [], [], 0
            for li, rec in steps:
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                t0 = time.perf_counter()
                e0.record(stream)
                device_path += c.update_lights(li, rec)
                t1 = time.perf_counter()
                e1.record(stream)
                frame(c)
                e2.record(stream)
                stream.synchronize()
                t2 = time.perf_counter()
                host.append(1e3 * (t1 - t0)); step.append(1e3 * (t2 - t0))
                dev.append(e0.elapsed_time(e1)); fr.append(e1.elapsed_time(e2))
            build = []
            for li, rec in steps:
                e0, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
                with torch.cuda.stream(stream):
                    torch.cuda._sleep(HOLD_CYCLES)
                e0.record(stream)
                c.update_lights(li, rec)
                e1.record(stream)
                stream.synchronize()
                build.append(e0.elapsed_time(e1))
            st = c.stats()
            r.update(update_host_ms=med(host), update_device_ms=med(dev), build_device_ms=med(build), frame_ms=med(fr), step_ms=med(step),
                     device_path_steps=device_path, light_grids=st["light_grids"], bvh_spheres=st["bvh_spheres"],
                     grids_differ=c.light_grids_selftest()[0])
        finally:
            c.close()
        c = capi.Context(0)
        try:
            c.load_scene(scene)
            c.set_seeds(12345, 12345); c.set_image_size(W, H)
            frame(c); stream.synchronize()
            reload = []
            for moved in [S.with_lights(scene, li, rec) for li, rec in steps]:
                t0 = time.perf_counter()
                c.load_scene(moved)
                frame(c)
                stream.synchronize()
                reload.append(1e3 * (time.perf_counter() - t0))
            r["reload_step_ms"] = med(reload)
        finally:
            c.close()
        res["scenes"][name] = r
        print("done", name, r, file=sys.stderr, flush=True)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
