"""Animated meshes: rfx_update_mesh against reloading the scene, per animation step.

Scenes: scenes.mesh_scene with 16 388, 65 540 and 262 148 triangles (the torus plus the floor and wall), and the 262 148-triangle scene with
synthetic_scene's 1024 spheres.  Each is animated for --steps steps of scenes.torus_wave (a travelling wave on the tube radius) and
rendered at 1920x1080, depth 4, default camera, into a device-resident frame on a torch stream.  Prints one JSON line with, per scene:
  * update_host_ms: host wall time of the rfx_update_mesh call (median over the steps) and how many steps took the device path;
  * update_device_ms: CUDA events on the caller's stream around the call (the vertex copy, k_mesh_setup, k_tri_refit), median;
  * frame_ms: CUDA events around the frame that follows each update, median;
  * step_ms: host wall time of update + frame + stream synchronisation, median;
  * reload_step_ms: the same step without rfx_update_mesh: load_scene of the deformed scene (every object through the C ABI again)
    + frame (which re-flattens on the host) + synchronisation, median;
  * refit quality: after the animation, the frame time of the refitted hierarchy against a fresh context loaded with the same final
    vertices (median of 8 frames each, CUDA events);
  * nvidia-smi's card name, power limit and max SM clock, read in the same run.
    python tools/bench_mesh_update.py [--steps 32] [--out FILE]
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
MESHES = [("16k", 128, 64, 0), ("64k", 256, 128, 0), ("256k", 512, 256, 0), ("256k+1024sph", 512, 256, 32)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:   # reported, not fatal
        return "nvidia-smi failed: %s" % e


def with_vertices(scene, xyz):
    return dict(scene, objects=[("mesh", xyz) + tuple(o[2:]) if o[0] == "mesh" else o for o in scene["objects"]])


def main():
    import torch
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert a.steps >= 1
    res = {"card": card(), "steps": a.steps, "size": "%dx%d" % (W, H), "depth": DEPTH, "scenes": {}}
    cam = [S.default_camera()]
    floor = S.synthetic_texture(256, 256, 3)
    sky = S.synthetic_texture(512, 384, 5)
    stream = torch.cuda.Stream()
    buf = torch.empty(W * H, dtype=torch.int32, device="cuda:0")
    med = lambda v: round(float(np.median(v)), 4)
    for name, nu, nv, sph in MESHES:
        scene = S.mesh_scene(nu, nv, spheres=sph, floor=floor, skybox=sky)
        frames = [S.torus_wave(nu, nv, phase=2.0 * np.pi * k / a.steps, amplitude=0.3) for k in range(1, a.steps + 1)]

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

        r = {}
        c = capi.Context(0)
        try:
            first = c.load_scene(scene)[0]
            c.set_seeds(12345, 12345); c.set_image_size(W, H)
            frame(c); frame(c); stream.synchronize()          # flatten, modules, eye grid, queue scratch
            c.update_mesh(first, S.torus_mesh(nu, nv)[0]); frame(c); stream.synchronize()   # the update's own buffers
            host, dev, fr, step, device_path = [], [], [], [], 0
            for xyz in frames:
                e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                t0 = time.perf_counter()
                e0.record(stream)
                device_path += c.update_mesh(first, xyz)
                t1 = time.perf_counter()
                e1.record(stream)
                frame(c)
                e2.record(stream)
                stream.synchronize()
                t2 = time.perf_counter()
                host.append(1e3 * (t1 - t0)); step.append(1e3 * (t2 - t0))
                dev.append(e0.elapsed_time(e1)); fr.append(e1.elapsed_time(e2))
            r.update(update_host_ms=med(host), update_device_ms=med(dev), frame_ms=med(fr), step_ms=med(step), device_path_steps=device_path,
                     bvh_triangles=c.stats()["bvh_triangles"])
            r["refitted_frame_ms"] = timed_frames(c)
        finally:
            c.close()
        c = capi.Context(0)
        try:
            c.load_scene(scene)
            c.set_seeds(12345, 12345); c.set_image_size(W, H)
            frame(c); stream.synchronize()
            reload = []
            for xyz in frames:
                t0 = time.perf_counter()
                c.load_scene(with_vertices(scene, xyz))
                frame(c)
                stream.synchronize()
                reload.append(1e3 * (time.perf_counter() - t0))
            r["reload_step_ms"] = med(reload)
            frame(c); stream.synchronize()
            r["fresh_frame_ms"] = timed_frames(c)
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
