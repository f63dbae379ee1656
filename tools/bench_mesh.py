"""Triangle-mesh workload: the hierarchy over the triangles against the list walk, and the host cost of building it.

Scenes: scenes.mesh_scene (a reflective metal torus over the textured floor and wall) with 16 384, 65 536 and 262 144 triangles, and the
262 144-triangle torus with synthetic_scene's 1024 spheres.  Prints one JSON line:
  * ms per frame with the hierarchy (rfx_set_bvh_mode 0): device-resident rfx_render_frames_device over an orbit path, one warm-up batch,
    then --frames frames timed between two device synchronisations, at 1920x1080 and 3840x2160, depth 1 / 4 / 8;
  * the list walk (mode 2) at 16 384 triangles, 1920x1080, depth 1 and 4, over --list-frames frames;
  * the host time of re-flattening the scene (uploadScene: boxes, hierarchy, blob upload), which a camera leaving the reach box pays:
    a one-ray rfx_trace_rays after rfx_set_bvh_mode marked the scene dirty, minus the same call on a clean scene (median of 5);
  * nvidia-smi's card name and power limit, read in the same run.
    python tools/bench_mesh.py [--frames 32] [--list-frames 2] [--out FILE]
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

SIZES = [(1920, 1080), (3840, 2160)]
DEPTHS = [1, 4, 8]
MESHES = [("16k", 128, 64, 0), ("64k", 256, 128, 0), ("256k", 512, 256, 0), ("256k+1024sph", 512, 256, 32)]


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:   # reported, not fatal
        return "nvidia-smi failed: %s" % e


def time_frames(c, buf, cams, depth, n):
    c.render_frames_device(cams[:min(4, n)], depth, 1, buf)     # warm-up: modules, queue scratch, eye grids
    c.synchronize()
    t0 = time.perf_counter()
    c.render_frames_device(cams[:n], depth, 1, buf)
    c.synchronize()
    return 1e3 * (time.perf_counter() - t0) / n


def upload_ms(c):
    o = np.zeros((1, 3), np.float32) + np.float32(S.DEFAULT_EYE)
    r = np.array([[0.0, -1.0, 0.0]], np.float32)

    def once(dirty):
        if dirty:
            c.set_bvh_mode(0)
        t0 = time.perf_counter()
        c.trace_rays(o, r, 1)
        return 1e3 * (time.perf_counter() - t0)
    once(False)
    clean = np.median([once(False) for _ in range(5)])
    dirty = np.median([once(True) for _ in range(5)])
    return float(dirty - clean)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=32)
    ap.add_argument("--list-frames", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert a.frames >= 1 and a.list_frames >= 1
    res = {"card": card(), "frames": a.frames, "list_frames": a.list_frames, "hierarchy_ms": {}, "list_walk_ms": {}, "upload_ms": {},
           "bvh_triangles": {}}
    cams = capi.pack_cameras(S.orbit_cameras(max(a.frames, 8) * 8)[::8][:max(a.frames, 4)])
    floor = S.synthetic_texture(256, 256, 3)
    sky = S.synthetic_texture(512, 384, 5)
    for name, nu, nv, sph in MESHES:
        scene = S.mesh_scene(nu, nv, spheres=sph, floor=floor, skybox=sky)
        c = capi.Context(0)
        try:
            c.load_scene(scene)
            c.set_seeds(12345, 12345)
            buf = c.buffer_alloc(max(a.frames, 4) * 3840 * 2160 * 4)
            for W, H in SIZES:
                c.set_image_size(W, H)
                for depth in DEPTHS:
                    res["hierarchy_ms"]["%s %dx%d d%d" % (name, W, H, depth)] = round(time_frames(c, buf, cams, depth, a.frames), 3)
            res["bvh_triangles"][name] = c.stats()["bvh_triangles"]
            res["upload_ms"][name] = round(upload_ms(c), 2)
            if name == "16k":
                c.set_bvh_mode(2)
                c.set_image_size(1920, 1080)
                for depth in (1, 4):
                    res["list_walk_ms"]["%s 1920x1080 d%d" % (name, depth)] = round(time_frames(c, buf, cams, depth, a.list_frames), 3)
                c.set_bvh_mode(0)
            c.buffer_free(buf)
        finally:
            c.close()
        print("done", name, file=sys.stderr, flush=True)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
