"""Shared replay helpers for the golden vectors (tests/golden/*.npz, generated from the unmodified reference by
tests/golden/make_golden.py)."""
import os

import numpy as np

from reflaxman_b200 import scenes as S

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def textured_default():
    return S.default_scene(skybox=S.synthetic_texture(512, 384, 7), floor=S.synthetic_texture(256, 256, 11))


def small_synth():
    return S.synthetic_scene(n_side=6, floor=S.synthetic_texture(128, 128, 3))


def config4_scene():
    """BASELINE.json configs[3]: 1024 spheres on a jittered 32x32 grid, textured floor and sky (the bench's scene)"""
    return S.synthetic_scene(32, floor=S.synthetic_texture(1024, 1024, 11), skybox=S.synthetic_texture(2048, 1536, 7))


SCENES = {
    "default": S.default_scene,
    "textured": textured_default,
    "synth36": small_synth,
    "synth1024": config4_scene,
}

GOLDEN = [
    "default_160x120_d20",
    "default_160x120_d4_seed777",
    "default_96x64_ss3",
    "default_96x64_block4",
    "default_96x64_additive3",
    "default_64x48_2frames",
    "textured_160x120_d20",
    "synth36_128x72_d8",
    "synth1024_480x270_d8",
]


def load_golden(name):
    z = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    g = {k: (z[k] if z[k].ndim else z[k].item()) for k in z.files}
    g["scene"] = SCENES[name.split("_")[0]]()
    return g


def full_size_hashes():
    """{case: (sha256 of the reference's ARGB image, sha256 of its float image)} for the frames too large to store"""
    want = {}
    with open(os.path.join(GOLDEN_DIR, "full_size_sha256.txt")) as f:
        for line in f:
            p = line.split()
            want[p[0]] = (p[2], p[4])
    return want


def replay(engine, g):
    """engine: object with set_image_size / render(cam, refl, samples, additive) / read_rgbf|resolve.
    Returns [(rgbf, argb)] per dumped frame, following oracle/ref_harness.cpp's frame loop."""
    cam = S.default_camera()
    out = []
    for f in range(g["frames"]):
        if g["additive"]:
            for _ in range(g["additive"]):
                engine.render(cam, g["refl"], g["samples"], True)
        else:
            engine.render(cam, g["refl"], g["samples"], False)
        out.append(engine.read())
    return out


class OracleEngine:
    def __init__(self, oracle, scene, W, H, seed, nthreads=4):
        self.r = oracle.OracleRender(scene, W, H, seed=seed, nthreads=nthreads)

    def render(self, cam, refl, samples, additive):
        self.r.render(cam, refl, samples, additive)

    def read(self):
        return self.r.resolve()


class GpuEngine:
    def __init__(self, capi, scene, W, H, seed, chunk=None):
        self.c = capi.Context(0)
        self.c.load_scene(scene)
        self.c.set_seeds(seed, seed)
        self.c.set_image_size(W, H)
        self.chunk = chunk

    def render(self, cam, refl, samples, additive):
        self.c.render(cam, refl, samples, additive, chunk=self.chunk)

    def read(self):
        return self.c.read_rgbf(), self.c.read_argb()

    def close(self):
        self.c.close()


def lsb_diff(a, b):
    """per-pixel max channel difference of two 0x00RRGGBB images"""
    d = np.zeros(a.shape, np.int32)
    for sh in (16, 8, 0):
        ca = ((a >> sh) & 0xFF).astype(np.int32)
        cb = ((b >> sh) & 0xFF).astype(np.int32)
        d = np.maximum(d, np.abs(ca - cb))
    return d


def assert_parity(argb, ref_argb, what=""):
    """BASELINE.json's bar: <= 1 LSB per channel on >= 99.9 % of pixels, no pixel off by more than 4 LSB."""
    d = lsb_diff(argb, ref_argb)
    frac1 = float((d <= 1).mean())
    assert d.max() <= 4, "%s: max channel difference %d LSB > 4 (at %s)" % (what, d.max(), np.argwhere(d == d.max())[:4].tolist())
    assert frac1 >= 0.999, "%s: only %.5f of pixels within 1 LSB" % (what, frac1)
    return {"max_lsb": int(d.max()), "frac_le1": frac1, "frac_exact": float((d == 0).mean())}
