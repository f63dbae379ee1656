"""What share of the fast kernel is the first segment of a path (primary ray, first query, first hit set-up, first-light
choice)?  The debug build (-DRFX_DEBUG_FIRST_SEGMENT) ends every path there; its kernel time against the normal build's,
on config 2 (the bench's 32 successive 1080p frames of one camera), bounds what computing that segment once per batch of
same-camera frames can save.

usage: first_segment_prize.py build            compile both libraries into build/first_segment/ (git-ignored)
       first_segment_prize.py run [ROUNDS]     time them alternately (one subprocess per arm and round), print JSON lines
"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "build", "first_segment")
ARMS = {"normal": (os.path.join(OUT, "normal.so"), []), "first_segment": (os.path.join(OUT, "first_segment.so"), ["RFX_DEBUG_FIRST_SEGMENT=1"])}
W, H, DEPTH, F, STEPS = 1920, 1080, 20, 32, 40


def time_arm(name):
    """one arm in this process: warm up, then STEPS steps of F frames; the kernel time comes from the per-launch events"""
    import torch
    from reflaxman_b200 import capi, scenes as S
    c = capi.Context(0)
    c.load_scene(S.default_scene()); c.set_seeds(12345, 12345); c.set_image_size(W, H)
    c.set_option("frame_batch", 0)            # one launch per frame: the debug build's cut applies to every path
    cams = capi.pack_cameras([S.default_camera()] * F)
    out = torch.empty((F, H, W), dtype=torch.int32, device="cuda")
    for _ in range(3):
        c.render_frames_device(cams, DEPTH, 1, out.data_ptr())
    c.synchronize()
    c.enable_profiling(True)
    c.stats_reset()
    for _ in range(STEPS):
        c.render_frames_device(cams, DEPTH, 1, out.data_ptr())
    c.synchronize()
    st = c.stats()
    c.close()
    return {"arm": name, "kernel_ms_per_frame": st["trace_kernel_ms"] / (STEPS * F), "launches": st["trace_kernels"],
            "device": torch.cuda.get_device_name(0)}


if __name__ == "__main__":
    if sys.argv[1] == "build":
        from reflaxman_b200 import build as B
        os.makedirs(OUT, exist_ok=True)
        for so, defs in ARMS.values():
            B.build(force=True, defines=defs, out=so)
    elif sys.argv[1] == "arm":
        print(json.dumps(time_arm(sys.argv[2])))
    else:
        rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 3
        for r in range(rounds):
            for name, (so, _) in ARMS.items():
                env = dict(os.environ, RFX_LIB=so)
                res = subprocess.run([sys.executable, os.path.abspath(__file__), "arm", name], env=env, capture_output=True, text=True, check=True)
                line = json.loads(res.stdout.strip().splitlines()[-1])
                line["round"] = r
                print(json.dumps(line), flush=True)
