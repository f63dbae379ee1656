"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

ctypes front end for the CPU oracle (oracle/librfx_oracle.so, our C restatement) and a subprocess front end for
the unmodified reference (oracle/_ref/ref_render*, built by oracle/Makefile from the tree $RFX_REFERENCE_SRC names).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / ``--impl reference`` legs may import this.
"""
from __future__ import annotations

import ctypes as C
import json
import os
import subprocess
import tempfile

import numpy as np

from reflaxman_b200.build import REFERENCE_SRC   # where the unmodified reference's src/common lies, if anywhere

HERE = os.path.dirname(os.path.abspath(__file__))
PORT_SO = os.path.join(HERE, "librfx_oracle.so")
POWCR_SO = os.path.join(HERE, "librfx_oracle_powcr.so")   # both power sites as the GPU computes them (RFXO_POW_CR)
REF_DIR = os.path.join(HERE, "_ref")

_fp = C.POINTER(C.c_float)
_u32p = C.POINTER(C.c_uint32)

COUNTER_FIELDS = ["rays", "bounces", "shadow_rays", "hits", "lit", "sky", "spec_pow", "fresnel_pow",
                  "sphere_tests", "tri_tests", "plane_tests", "tex_lookups", "samples",
                  "op_add", "op_mul", "op_div", "op_sqrt", "op_powf"]


class Counters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in COUNTER_FIELDS]

    def as_dict(self):
        return {n: int(getattr(self, n)) for n in COUNTER_FIELDS}


def build(ref=True, quiet=True):
    """Compile the port (always) and, when the reference tree is present, the reference binaries."""
    targets = ["port"]
    if ref and os.path.isdir(REFERENCE_SRC):
        targets.append("ref")
    subprocess.run(["make", "-C", HERE, *targets, "REF=" + REFERENCE_SRC], check=True,
                   stdout=subprocess.DEVNULL if quiet else None)


def have_ref(name="ref_render"):
    return os.access(os.path.join(REF_DIR, name), os.X_OK)


_lib = None


def lib(path=None):
    global _lib
    if _lib is not None and path is None:
        return _lib
    so = path or PORT_SO
    if not os.path.exists(so):
        build(ref=False)   # `make port` builds every port library, the default one and the variants
    L = C.CDLL(so)
    L.rfxo_scene_new.restype = C.c_void_p
    L.rfxo_scene_new.argtypes = [_fp, C.c_float]
    L.rfxo_scene_free.argtypes = [C.c_void_p]
    L.rfxo_add_light.argtypes = [C.c_void_p, _fp, C.c_float, _fp, C.c_float]
    L.rfxo_add_sphere.argtypes = [C.c_void_p, _fp, C.c_float, C.c_int, _fp, C.c_float, C.c_float]
    L.rfxo_add_texture.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, _u32p]
    L.rfxo_set_skybox.argtypes = [C.c_void_p, C.c_int]
    L.rfxo_add_triangle.argtypes = [C.c_void_p, _fp, C.c_int, _fp, C.c_float, C.c_float, C.c_int, _fp]
    L.rfxo_add_plane.argtypes = [C.c_void_p, _fp, _fp, C.c_int, _fp, C.c_float, C.c_float]
    L.rfxo_get_triangle.argtypes = [C.c_void_p, C.c_int, _fp, _fp, _fp]
    L.rfxo_get_env.argtypes = [C.c_void_p, _fp, _fp]
    L.rfxo_trace_one.argtypes = [C.c_void_p, _fp, _fp, C.c_int, _fp, _fp, _u32p]
    L.rfxo_trace_many.argtypes = [C.c_void_p, C.c_int, _fp, _fp, C.c_int, _fp, _fp, _u32p]
    L.rfxo_rand_dirs.argtypes = [_u32p, C.c_uint64, _fp]
    L.rfxo_plane_probe.argtypes = [_fp, C.c_int, _fp]
    L.rfxo_render_pass.restype = C.c_int
    L.rfxo_render_pass.argtypes = [C.c_void_p, _fp, _fp, C.c_float, C.c_uint32, C.c_uint32, C.c_int, C.c_int, C.c_int,
                                   C.c_int, _fp, _u32p, C.POINTER(Counters), _u32p, C.c_int]
    L.rfxo_resolve.argtypes = [_fp, C.c_uint32, C.c_uint32, C.c_int, _fp, _u32p]
    L.rfxo_camera_lookat.argtypes = [_fp, _fp, _fp]
    L.rfxo_census_enabled.restype = C.c_int
    if path is None:
        _lib = L
    return L


_lib_powcr = None


def lib_powcr():
    """The oracle built with -DRFXO_POW_CR (cached apart from :func:`lib`): the GPU's arithmetic, powers included."""
    global _lib_powcr
    if _lib_powcr is None:
        _lib_powcr = lib(POWCR_SO)
    return _lib_powcr


def _f(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(_fp)


class OracleScene:
    """Scene flattened into the C oracle from a :mod:`reflaxman_b200.scenes` dict."""

    def __init__(self, scene, L=None):
        self.L = L or lib()
        rgb, p = scene["ambient"]
        _, prgb = _f(rgb)
        self.h = C.c_void_p(self.L.rfxo_scene_new(prgb, C.c_float(p)))
        self._keep = []
        for t in scene["textures"]:
            self._add_tex(t)
        if scene.get("skybox") is not None:
            self.L.rfxo_set_skybox(self.h, self._add_tex(scene["skybox"]))
        for o, r, c, pw in scene["lights"]:
            self.L.rfxo_add_light(self.h, _f(o)[1], C.c_float(r), _f(c)[1], C.c_float(pw))
        for ob in scene["objects"]:
            if ob[0] == "sphere":
                _, c, r, mt, col, refl, tr = ob
                self.L.rfxo_add_sphere(self.h, _f(c)[1], C.c_float(r), mt, _f(col)[1], C.c_float(refl), C.c_float(tr))
            elif ob[0] == "tri":
                _, v, mt, col, refl, tr, tex, uv = ob
                self.L.rfxo_add_triangle(self.h, _f(v)[1], mt, _f(col)[1], C.c_float(refl), C.c_float(tr), tex, _f(uv)[1])
            elif ob[0] == "plane":
                _, pos, nrm, mt, col, refl, tr = ob
                self.L.rfxo_add_plane(self.h, _f(pos)[1], _f(nrm)[1], mt, _f(col)[1], C.c_float(refl), C.c_float(tr))
            else:
                raise ValueError(ob[0])

    def _add_tex(self, t):
        if t is None:
            return self.L.rfxo_add_texture(self.h, 0, 0, None)
        a = np.ascontiguousarray(t, dtype=np.uint32)
        return self.L.rfxo_add_texture(self.h, a.shape[1], a.shape[0], a.ctypes.data_as(_u32p))

    def triangle(self, idx):
        n = np.zeros(3, np.float32); ax = np.zeros(9, np.float32); tuv = np.zeros(9, np.float32)
        self.L.rfxo_get_triangle(self.h, idx, n.ctypes.data_as(_fp), ax.ctypes.data_as(_fp), tuv.ctypes.data_as(_fp))
        return n, ax, tuv

    def env(self):
        e = np.zeros(3, np.float32); ht = np.zeros(2, np.float32)
        self.L.rfxo_get_env(self.h, e.ctypes.data_as(_fp), ht.ctypes.data_as(_fp))
        return e, ht

    def close(self):
        if self.h:
            self.L.rfxo_scene_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class OracleRender:
    """Mirror of the reference's ``Render`` state machine on top of the C oracle (reference Render.cpp:57-134)."""

    def __init__(self, scene, width, height, seed=12345, nthreads=None, L=None):
        self.L = L or lib()
        self.scene = scene if isinstance(scene, OracleScene) else OracleScene(scene, self.L)
        self.seeds = np.array([seed, seed], dtype=np.uint32)   # [Vector3.cpp TU, Render.cpp TU]
        self.nthreads = nthreads or min(os.cpu_count() or 1, 64)
        self.set_image_size(width, height)
        self.counters = None
        self.sig = None

    def set_image_size(self, w, h):
        self.W, self.H = int(w), int(h)
        self.image = np.zeros((self.H, self.W, 3), np.float32)
        self.additive_counter = 0

    def render(self, cam, refl, samples=1, additive=False, want_sig=False):
        """renderBegin + renderNext to completion."""
        eye, view, fov = cam
        if additive:
            self.additive_counter += 1
        else:
            self.additive_counter = 0
        k = Counters()
        sig = np.zeros((self.H, self.W), np.uint32) if want_sig else None
        rc = self.L.rfxo_render_pass(self.scene.h, _f(eye)[1], _f(view)[1], C.c_float(fov), self.W, self.H, refl, samples,
                                     1 if additive else 0, 1 if self.additive_counter > 1 else 0,
                                     self.image.ctypes.data_as(_fp), self.seeds.ctypes.data_as(_u32p), C.byref(k),
                                     sig.ctypes.data_as(_u32p) if want_sig else None, self.nthreads)
        if rc != 0:
            raise RuntimeError("rfxo_render_pass failed: %d" % rc)
        self.counters = k.as_dict()
        self.sig = sig
        return self

    def resolve(self):
        rgbf = np.zeros((self.H, self.W, 3), np.float32)
        argb = np.zeros((self.H, self.W), np.uint32)
        self.L.rfxo_resolve(self.image.ctypes.data_as(_fp), self.W, self.H, self.additive_counter,
                            rgbf.ctypes.data_as(_fp), argb.ctypes.data_as(_u32p))
        return rgbf, argb


def rand_dirs(seed, n):
    s = np.array([seed], dtype=np.uint32)
    out = np.zeros((n, 3), np.float32)
    lib().rfxo_rand_dirs(s.ctypes.data_as(_u32p), n, out.ctypes.data_as(_fp))
    return out, int(s[0])


def trace_many(scene, origins, rays, refl, seed, L=None):
    """Scene::trace for a ray list, as rfx_trace_rays runs it: ray i takes the i-th direction of the stream that starts at
    ``seed``.  ``scene``: an :class:`OracleScene` or a scenes.py dict.  Returns (rgb [n, 3], signatures [n], stream end state)."""
    sc = scene if isinstance(scene, OracleScene) else OracleScene(scene, L)
    o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
    r = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 3)
    n = o.shape[0]
    dirs, end = rand_dirs(seed, n)
    rgb = np.zeros((n, 3), np.float32)
    sig = np.zeros(n, np.uint32)
    sc.L.rfxo_trace_many(sc.h, n, o.ctypes.data_as(_fp), r.ctypes.data_as(_fp), refl, dirs.ctypes.data_as(_fp),
                         rgb.ctypes.data_as(_fp), sig.ctypes.data_as(_u32p))
    return rgb, sig, end


def plane_probe(inputs):
    """Plane::trace restatement on [n, 12] float32 inputs (pos, norm, origin, ray) -> [n, 12] outputs (see rfxo_plane_probe)."""
    a = np.ascontiguousarray(inputs, dtype=np.float32).reshape(-1, 12)
    out = np.zeros((a.shape[0], 12), np.float32)
    lib().rfxo_plane_probe(a.ctypes.data_as(_fp), a.shape[0], out.ctypes.data_as(_fp))
    return out


def run_plane_probe(n, seed):
    """The reference's own Plane::trace on n seeded inputs (oracle/_ref/ref_plane_probe) -> ([n, 12] inputs, [n, 12] outputs)."""
    exe = os.path.join(REF_DIR, "ref_plane_probe")
    if not os.access(exe, os.X_OK):
        raise FileNotFoundError(exe)
    with tempfile.TemporaryDirectory() as td:
        outp = os.path.join(td, "planes.bin")
        subprocess.run([exe, str(n), str(seed), outp], check=True)
        raw = np.fromfile(outp, dtype=np.float32).reshape(n, 24)
    return raw[:, :12].copy(), raw[:, 12:].copy()


def camera_lookat(eye, at):
    v = np.zeros(9, np.float32)
    lib().rfxo_camera_lookat(_f(eye)[1], _f(at)[1], v.ctypes.data_as(_fp))
    return v


def run_reference(width, height, refl=20, samples=1, additive_passes=0, frames=1, cams=None, scene=None,
                  seed=12345, binary="ref_render", chunk=None, rows=None, dump=None, want_images=True, tmpdir=None,
                  timeout=3600):
    """Run the unmodified reference (oracle/_ref/<binary>) headless.

    ``scene``: a scenes.py dict (textures are written as TGAs) or None for the reference's own default scene.
    ``cams``: list of (eye, view, fov) or None for the reference's default camera.
    Returns (info_json, [(rgbf HxWx3, argb HxW), ...] for the dumped frames).
    """
    from reflaxman_b200 import scenes as S  # host-side description helpers only (no GPU)

    exe = os.path.join(REF_DIR, binary)
    if not os.access(exe, os.X_OK):
        raise FileNotFoundError(exe)
    with tempfile.TemporaryDirectory(dir=tmpdir) as td:
        args = [exe, "--size", str(width), str(height), "--refl", str(refl), "--samples", str(samples), "--frames", str(frames)]
        if additive_passes:
            args += ["--additive", str(additive_passes)]
        if chunk:
            args += ["--chunk", str(chunk)]
        if rows:
            args += ["--rows", str(rows[0]), str(rows[1])]
        if scene is not None:
            tex_paths = []
            for i, t in enumerate(scene["textures"]):
                p = os.path.join(td, "tex%d.tga" % i)
                if t is not None:
                    S.write_tga(p, t, 32)
                tex_paths.append(p)
            sky_path = os.path.join(td, "sky.tga")
            if scene.get("skybox") is not None:
                S.write_tga(sky_path, scene["skybox"], 32)
            sp = os.path.join(td, "scene.txt")
            with open(sp, "w") as f:
                f.write(S.scene_to_text(scene, tex_paths, sky_path))
            args += ["--scene", sp]
        if cams is not None:
            cp = os.path.join(td, "cams.txt")
            with open(cp, "w") as f:
                f.write(S.cameras_to_text(cams))
            args += ["--cams", cp]
        outp = os.path.join(td, "out.bin")
        if want_images:
            args += ["--out", outp]
            for d in (dump or []):
                args += ["--dump", str(d)]
        env = dict(os.environ, RFX_SEED=str(seed))
        res = subprocess.run(args, env=env, check=True, capture_output=True, text=True, timeout=timeout)
        info = json.loads(res.stdout)
        images = []
        if want_images:
            raw = np.fromfile(outp, dtype=np.uint8)
            per = width * height * 16
            for i in range(len(raw) // per):
                blk = raw[i * per:(i + 1) * per]
                rgbf = blk[:width * height * 12].view(np.float32).reshape(height, width, 3).copy()
                argb = blk[width * height * 12:].view(np.uint32).reshape(height, width).copy()
                images.append((rgbf, argb))
        return info, images
