"""Moving cameras over big scenes: the eye grid built on the GPU, binned on the host, or not used, per frame of a camera path.

Scenes: scenes.synthetic_scene at 1024, 16 384 and 65 536 spheres (n_side 32, 128, 256: a sphere hierarchy, one light grid, the eye
grid) with the textured floor, wall and sky.  The camera path is scenes.orbit_cameras(--cams): every frame has a new camera, so every
frame needs a new eye grid.  Each frame is one rfx_render_frames_device call, 1920x1080 at depth 4, into a device buffer on a torch
stream.  Arms: "device" (option eye_grid_device 1, the default), "host" (eye_grid_device 0: binned on the host and uploaded, as before
the builder) and "none" (eye_grid 0: every first query walks the hierarchy).  Prints one JSON line with, per scene and arm (medians
over the path):
  * frame_ms: CUDA events on the stream around the call (the eye grid, the random streams and the trace kernels, and whatever time the
    stream sits idle while the host works inside the call);
  * host_ms: host wall time of the call (it returns after enqueueing);
  * step_ms: host wall time of the call and the stream synchronisation after it;
  * build_ms: the eye grid's share of the frame on the device: the stream is held by a sleep kernel while the host enqueues, and the
    events bracket the frame of a new camera minus those of the same camera rendered again (cached grid);
  * selftest: rfx_selftest_eye_grid after the path (differences, items on the device, items on the host, builds dropped).
nvidia-smi's card name, power limit and max SM clock are read in the same run.
    python tools/bench_camera_path.py [--cams 32] [--out FILE]
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
ARMS = [("device", {"eye_grid": 1, "eye_grid_device": 1}), ("host", {"eye_grid": 1, "eye_grid_device": 0}), ("none", {"eye_grid": 0})]
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
    ap.add_argument("--cams", type=int, default=32)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert a.cams >= 2
    res = {"card": card(), "cams": a.cams, "size": "%dx%d" % (W, H), "depth": DEPTH, "scenes": {}}
    cams = S.orbit_cameras(a.cams)
    floor = S.synthetic_texture(256, 256, 3)
    sky = S.synthetic_texture(512, 384, 5)
    stream = torch.cuda.Stream()
    buf = torch.empty(W * H, dtype=torch.int32, device="cuda:0")
    med = lambda v: round(float(np.median(v)), 4)

    def frame(c, cam):
        c.render_frames_device([cam], DEPTH, 1, buf.data_ptr(), stream.cuda_stream)

    for name, n_side in SIZES:
        scene = S.synthetic_scene(n_side, floor=floor, skybox=sky)
        res["scenes"][name] = {"spheres": n_side * n_side}
        for arm, opts in ARMS:
            c = capi.Context(0)
            try:
                c.load_scene(scene)
                c.set_seeds(12345, 12345); c.set_image_size(W, H)
                for k, v in opts.items():
                    c.set_option(k, v)
                frame(c, cams[-1]); frame(c, cams[-2]); stream.synchronize()     # flatten, modules, grid regions, queue scratch
                c.synchronize()
                fr, host, step = [], [], []
                for cam in cams:
                    e0, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
                    t0 = time.perf_counter()
                    e0.record(stream)
                    frame(c, cam)
                    t1 = time.perf_counter()
                    e1.record(stream)
                    stream.synchronize()
                    t2 = time.perf_counter()
                    fr.append(e0.elapsed_time(e1)); host.append(1e3 * (t1 - t0)); step.append(1e3 * (t2 - t0))
                st = c.eye_grid_selftest()
                held = {True: [], False: []}
                for cam in cams:
                    for new in (True, False):
                        e0, e1 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
                        with torch.cuda.stream(stream):
                            torch.cuda._sleep(HOLD_CYCLES)
                        e0.record(stream)
                        frame(c, cam)
                        e1.record(stream)
                        stream.synchronize()
                        held[new].append(e0.elapsed_time(e1))
                r = {"frame_ms": med(fr), "host_ms": med(host), "step_ms": med(step),
                     "held_new_camera_ms": med(held[True]), "held_same_camera_ms": med(held[False]),
                     "build_ms": round(med(held[True]) - med(held[False]), 4), "selftest": list(st)}
            finally:
                c.close()
            res["scenes"][name][arm] = r
            print("done", name, arm, r, file=sys.stderr, flush=True)
    res["card_after"] = card()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
