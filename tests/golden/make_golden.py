"""Generates tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref/ref_render, built by oracle/Makefile
from the tree RFX_REFERENCE_SRC names).  Run in the build container only:  python tests/golden/make_golden.py

Each vector stores the inputs needed to replay it (scene name, camera floats, size, depth, samples, seed) and the
reference's outputs (ARGB, and the float image for the small cases), zlib-compressed by numpy.
"""
import hashlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import pyoracle as O            # noqa: E402
from reflaxman_b200 import scenes as S      # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def textured_default():
    sky = S.synthetic_texture(512, 384, 7)
    floor = S.synthetic_texture(256, 256, 11)
    return S.default_scene(skybox=sky, floor=floor)


def small_synth():
    return S.synthetic_scene(n_side=6, floor=S.synthetic_texture(128, 128, 3))


def config4_scene():
    return S.synthetic_scene(32, floor=S.synthetic_texture(1024, 1024, 11), skybox=S.synthetic_texture(2048, 1536, 7))


CASES = [
    # name, scene factory (None = the reference's own built-in scene), W, H, refl, samples, additive passes, frames, seed, keep float
    ("default_160x120_d20", None, 160, 120, 20, 1, 0, 1, 12345, True),
    ("default_160x120_d4_seed777", None, 160, 120, 4, 1, 0, 1, 777, True),
    ("default_96x64_ss3", None, 96, 64, 15, 3, 0, 1, 12345, True),
    ("default_96x64_block4", None, 96, 64, 4, -4, 0, 1, 12345, True),
    ("default_96x64_additive3", None, 96, 64, 15, 1, 3, 1, 12345, True),
    ("default_64x48_2frames", None, 64, 48, 20, 1, 0, 2, 12345, True),
    ("textured_160x120_d20", textured_default, 160, 120, 20, 1, 0, 1, 12345, True),
    ("synth36_128x72_d8", small_synth, 128, 72, 8, 1, 0, 1, 12345, True),
    # BASELINE.json configs[3] (1024 spheres + textured floor and sky) at a size the reference's list walk finishes in ~15 s
    ("synth1024_480x270_d8", config4_scene, 480, 270, 8, 1, 0, 1, 12345, False),
]


def main(only=None):
    """only: names of the cases to (re)generate (default: everything, ~3 minutes)"""
    O.build(ref=True)
    assert O.have_ref(), "oracle/_ref/ref_render missing: set RFX_REFERENCE_SRC to the reference's src/common"
    index = {}
    if not only or "plane_probe" in only:
        # Plane::trace is unreachable through Scene: the reference's own function probed directly (oracle/ref_plane_probe.cpp)
        inputs, outputs = O.run_plane_probe(4096, 777)
        np.savez_compressed(os.path.join(OUT, "plane_probe.npz"), inputs=inputs, outputs=outputs)
        print("plane_probe", hashlib.sha256(outputs.tobytes()).hexdigest()[:16], "hits %.3f" % outputs[:, 0].mean())
    if not only or "pulse_headless" in only:
        # the reference's UI controller driven headless (oracle/pulse_headless.cpp built with the reference's own Render):
        # the last repaint of a scripted interactive session and the hash of the screenshot BMP it saves
        import subprocess, tempfile
        with tempfile.TemporaryDirectory() as td:
            subprocess.run([os.path.join(O.REF_DIR, "ref_pulse_headless"), td + "/", "160", "120", "260", "2", "2"], check=True, stdout=subprocess.DEVNULL)
            inter = np.fromfile(os.path.join(td, "interactive.bin"), dtype=np.uint32).reshape(120, 160)
            hud = open(os.path.join(td, "hud.txt")).read()
            bmp = open(os.path.join(td, "scrnshoot_0000000100000002.bmp"), "rb").read()
        np.savez_compressed(os.path.join(OUT, "pulse_headless.npz"), interactive=inter, hud=np.array(hud), bmp_sha256=np.array(hashlib.sha256(bmp).hexdigest()),
                            bmp_bytes=np.array(len(bmp)))
        print("pulse_headless", hashlib.sha256(bmp).hexdigest()[:16], len(bmp))
    for name, factory, W, H, refl, samples, add, frames, seed, keepf in CASES:
        if only and name not in only:
            continue
        scene = factory() if factory else None
        info, imgs = O.run_reference(W, H, refl=refl, samples=samples, additive_passes=add, frames=frames, scene=scene, seed=seed)
        data = {"W": W, "H": H, "refl": refl, "samples": samples, "additive": add, "frames": frames, "seed": seed}
        for i, (rgbf, argb) in enumerate(imgs):
            data["argb%d" % i] = argb
            if keepf:
                data["rgbf%d" % i] = rgbf
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **data)
        index[name] = hashlib.sha256(imgs[-1][1].tobytes()).hexdigest()
        print(name, index[name][:16])
    # full-size hashes only (images are too big to commit): config 1 and config 2
    # configs 1, 2 and 3 (7680x4320, a reference screenshot preset, Pulse.cpp:20)
    if only and "full_size" not in only:
        return
    with open(os.path.join(OUT, "full_size_sha256.txt"), "w") as f:
        for W, H in ((1024, 768), (1920, 1080), (7680, 4320)):
            info, imgs = O.run_reference(W, H, refl=20, seed=12345)
            hs = hashlib.sha256(imgs[0][1].tobytes()).hexdigest()
            hf = hashlib.sha256(imgs[0][0].tobytes()).hexdigest()
            f.write("default_%dx%d_d20_seed12345 argb %s rgbf %s\n" % (W, H, hs, hf))
            print(W, H, hs[:16])


if __name__ == "__main__":
    main(sys.argv[1:])
