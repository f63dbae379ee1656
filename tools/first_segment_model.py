"""CPU model of the frame batch: how much of config 2's work is the first segment of a path, and what other layouts would save.

It renders F successive config-2 frames (default scene, 1920x1080, depth 20, seed 12345; the random stream continues from frame
to frame, one camera) with a private copy of the C oracle whose pixel loop records, per pixel, the bounce-loop iterations, the
shadow rays and whether the primary ray went to the sky.  The copy is patched and compiled in a temporary directory; oracle/
stays as it is.  Prints one JSON object (profiles/first_segment/model.json).

usage: first_segment_model.py [FRAMES]
"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
W, H, DEPTH, SEED = 1920, 1080, 20, 12345

# the pixel loop's signature store becomes a record of the path: bounces | shadow rays << 8 | primary miss << 16
PATCHES = [
    ("        C3 fin = c3(0.0f, 0.0f, 0.0f);\n        uint32_t h = 2166136261u;\n",
     "        C3 fin = c3(0.0f, 0.0f, 0.0f);\n        uint32_t h = 2166136261u;\n"
     "        const uint64_t b0 = w->k.bounces, s0 = w->k.shadow_rays, k0 = w->k.sky;\n"),
    ("        if (j->sig) j->sig[(size_t)y * W + x] = h;\n      }\n  }\n  else",
     "        if (j->sig) j->sig[(size_t)y * W + x] = (uint32_t)((w->k.bounces - b0) | ((w->k.shadow_rays - s0) << 8) |\n"
     "                                                            ((w->k.bounces - b0 == 1 && w->k.sky - k0 == 1) ? 1u << 16 : 0u));\n"
     "      }\n  }\n  else"),
]


def build(tmp):
    src = open(os.path.join(ROOT, "oracle", "rfx_oracle.c")).read()
    for a, b in PATCHES:
        assert src.count(a) == 1, "oracle pixel loop changed: update PATCHES"
        src = src.replace(a, b)
    c = os.path.join(tmp, "rfx_oracle_events.c")
    open(c, "w").write(src)
    so = os.path.join(tmp, "librfx_oracle_events.so")
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-fno-fast-math", "-std=c11", "-fPIC", "-shared", "-pthread", "-o", so, c, "-lm"], check=True)
    return so


def warp_passes(q, tw, th):
    """sum over warps of the longest path (queries) of the warp's tw x th pixel tile: the trips the state machine runs"""
    t = q.reshape(H // th, th, W // tw, tw).swapaxes(1, 2).reshape(H // th, W // tw, tw * th)
    return float(t.max(axis=2).sum())


def main():
    from oracle import pyoracle as O
    from reflaxman_b200 import scenes as S
    F = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    with tempfile.TemporaryDirectory() as tmp:
        L = O.lib(build(tmp))
        o = O.OracleRender(S.default_scene(), W, H, seed=SEED, L=L)
        rec = np.stack([o.render(S.default_camera(), DEPTH, want_sig=True).sig.copy() for _ in range(F)])   # [F, H, W]
    b = (rec & 0xFF).astype(np.int64)
    s = ((rec >> 8) & 0xFF).astype(np.int64)
    miss = ((rec >> 16) & 1).astype(bool)
    q = b + s
    assert (miss == miss[0]).all(), "the primary miss is frame-invariant"
    tile = sum(warp_passes(q[f], 4, 8) for f in range(F))
    # lanes = frames: a warp holds one pixel in `g` frames (32 // g pixels of a row side by side)
    lanes_frames = {}
    for g in (8, 16):
        per = 32 // g
        n = F // g * g
        t = q[:n].reshape(n // g, g, H, W // per, per).transpose(0, 2, 3, 1, 4).reshape(n // g, H, W // per, 32)
        lanes_frames["frames_%d_per_warp" % g] = float(t.max(axis=3).sum()) * F / n
    print(json.dumps({
        "frames": F, "W": W, "H": H, "depth": DEPTH, "seed": SEED,
        "queries_per_pixel": float(q.mean()), "bounce_iterations_per_pixel": float(b.mean()), "shadow_rays_per_pixel": float(s.mean()),
        "first_query_share_of_queries": float(1.0 / q.mean()),
        "primary_miss_fraction": float(miss[0].mean()),
        "two_bounce_iterations_fraction": float((b == 2).mean()),
        "same_query_count_in_all_frames_fraction": float((q == q[0]).all(axis=0).mean()),
        "warp_passes_4x8_tiles": tile,
        "lanes_busy_per_trip_4x8_tiles": float(q.sum() / tile),
        **{"warp_passes_" + k: v for k, v in lanes_frames.items()},
        **{"saving_" + k: 1.0 - v / tile for k, v in lanes_frames.items()},
    }))


if __name__ == "__main__":
    main()
