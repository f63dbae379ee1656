"""Plane-scene workload: hierarchies in scenes with an unbounded ground plane, against the list walk and against the same scene without the plane.

Scenes (each over a metal ground plane y = -0.05, reflectivity 0.6, just below the floor triangles: scenes.with_ground_plane):
mesh_scene(128, 64) (16 384 triangles), mesh_scene(512, 256) (262 144 triangles) and synthetic_scene(32) (1024 spheres).
Cameras: an orbit path, and one camera low over the plane looking at the horizon (most bounces then start far out on the plane).
Prints one JSON line:
  * ms per frame with the hierarchies (rfx_set_bvh_mode 0): device-resident rfx_render_frames_device, one warm-up batch, then --frames
    frames timed between two device synchronisations, at 1920x1080 and 3840x2160, depth 1 / 4 / 8, both camera sets;
  * the same scene without the plane (what the growth of the boxes and the plane's own bounces cost);
  * the list walk (mode 2) at 1920x1080 over --list-frames frames: depth 1 / 4 / 8 for the spheres, 1 / 4 for the 16 384-triangle
    torus, 1 for the 262 144-triangle one;
  * bvh_spheres / bvh_triangles of each scene, and nvidia-smi's card name and power limit, read in the same run.
    python tools/bench_plane.py [--frames 8] [--list-frames 1] [--out FILE]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench_mesh import card, time_frames  # noqa: E402
from reflaxman_b200 import capi, scenes as S  # noqa: E402

SIZES = [(1920, 1080), (3840, 2160)]
DEPTHS = [1, 4, 8]
HORIZON_CAM = S.camera_lookat((0.0, 0.4, 26.0), (0.0, 0.3, -200.0), 1.2)
# name, scene builder, list-walk depths at 1920x1080
SCENES = [("16k", lambda fl, sk: S.mesh_scene(128, 64, floor=fl, skybox=sk), (1, 4)),
          ("256k", lambda fl, sk: S.mesh_scene(512, 256, floor=fl, skybox=sk), (1,)),
          ("1024sph", lambda fl, sk: S.synthetic_scene(32, floor=fl, skybox=sk), (1, 4, 8))]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=8)
    ap.add_argument("--list-frames", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert a.frames >= 1 and a.list_frames >= 1
    res = {"card": card(), "frames": a.frames, "list_frames": a.list_frames, "plane_hierarchy_ms": {}, "no_plane_ms": {}, "plane_list_walk_ms": {},
           "bvh": {}}
    n = max(a.frames, 4)
    cam_sets = {"orbit": capi.pack_cameras(S.orbit_cameras(n * 8)[::8][:n]), "horizon": capi.pack_cameras([HORIZON_CAM] * n)}
    floor = S.synthetic_texture(256, 256, 3)
    sky = S.synthetic_texture(512, 384, 5)
    for name, build, list_depths in SCENES:
        base = build(floor, sky)
        for plane in (True, False):
            c = capi.Context(0)
            try:
                c.load_scene(S.with_ground_plane(base) if plane else base)
                c.set_seeds(12345, 12345)
                buf = c.buffer_alloc(n * 3840 * 2160 * 4)
                key = "plane_hierarchy_ms" if plane else "no_plane_ms"
                for W, H in SIZES:
                    c.set_image_size(W, H)
                    for depth in DEPTHS:
                        for cname, cams in cam_sets.items():
                            res[key]["%s %s %dx%d d%d" % (name, cname, W, H, depth)] = round(time_frames(c, buf, cams, depth, a.frames), 3)
                st = c.stats()
                res["bvh"]["%s%s" % (name, " plane" if plane else "")] = {"spheres": st["bvh_spheres"], "triangles": st["bvh_triangles"]}
                if plane:
                    c.set_bvh_mode(2)
                    c.set_image_size(1920, 1080)
                    for depth in list_depths:
                        for cname, cams in cam_sets.items():
                            res["plane_list_walk_ms"]["%s %s 1920x1080 d%d" % (name, cname, depth)] = round(time_frames(c, buf, cams, depth, a.list_frames), 3)
                    c.set_bvh_mode(0)
                c.buffer_free(buf)
            finally:
                c.close()
            print("done", name, "plane" if plane else "no plane", file=sys.stderr, flush=True)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
