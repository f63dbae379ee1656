"""Scene / camera-path descriptions shared by the bench driver and the tests.

A scene is a plain dict of float32 data (no classes), mirroring what the reference builds through
``Scene::addSphere/addTriangle/addLight/addTexture/setSkyboxTexture`` (reference Scene.h:29-39):

    {"ambient": (rgb[3], power),
     "skybox": None | HxW uint32 ARGB array,            # None = texture failed to load -> checker fallback
     "textures": [None | HxW uint32 ARGB array, ...],   # Scene::addTexture order
     "lights": [(origin[3], radius, rgb[3], power), ...],
     "objects": [("sphere", center[3], radius, mtype, rgb[3], refl, transp) |
                 ("tri", v[9], mtype, rgb[3], refl, transp, tex_index_or_-1, uv[6]) |
                 ("plane", pos[3], norm[3], mtype, rgb[3], refl, transp) |
                 ("mesh", xyz[N,3], idx[M,3], mtype, rgb[3], refl, transp), ...]}   # insertion order matters (ties)

A "mesh" is M triangles with one material, triangle k = vertices xyz[idx[k]] (rfx_add_mesh); :func:`expand_meshes` turns it into
the M "tri" objects it stands for, which is what the reference's Scene (it has no mesh call) and the oracle take.

Material types follow reference Material.h:8: 0 = mtMetal, 1 = mtDielectric.
Nothing here touches the GPU; :mod:`reflaxman_b200.capi` uploads a scene through the C ABI.
"""
from __future__ import annotations

import math
import struct

import numpy as np

MT_METAL = 0
MT_DIELECTRIC = 1

DEFAULT_EYE = (7.427, 3.494, -3.773)       # reference Render.cpp:30
DEFAULT_AT = (6.5981, 3.127, -3.352)
DEFAULT_FOV = 1.05
SCREENSHOT_REFLECTIONS = 20                # reference defaults.h:9
STATIC_REFLECTIONS = 15                    # reference defaults.h:7
MOTION_REFLECTIONS = 4                     # reference defaults.h:8


def f32(x):
    return np.asarray(x, dtype=np.float32)


def default_scene(skybox=None, floor=None):
    """The reference's built-in demo scene (reference Render.cpp:25-55).

    ``skybox`` / ``floor``: optional uint32 ARGB arrays standing in for textures/skybox.tga and
    textures/himiya.tga; ``None`` reproduces this checkout's behaviour (files missing -> checker fallback).
    """
    M, D = MT_METAL, MT_DIELECTRIC
    objs = [
        ("sphere", (-1.25, 1.5, -0.25), 1.5, M, (1.0, 1.0, 1.0), 1.0, 0.0),
        ("sphere", (0.15, 1.0, 1.75), 1.0, M, (1.0, 1.0, 1.0), 0.95, 0.0),
        ("sphere", (-3.0, 0.6, -3.0), 0.6, D, (1.0, 1.0, 1.0), 0.0, 0.0),
        ("sphere", (-0.5, 0.5, -2.5), 0.5, D, (0.5, 1.0, 0.15), 0.75, 0.0),
        ("sphere", (1.0, 0.4, -1.5), 0.4, D, (0.0, 0.5, 1.0), 1.0, 0.0),
        ("sphere", (1.8, 0.4, 0.1), 0.4, M, (1.0, 0.65, 0.45), 1.0, 0.0),
        ("sphere", (1.7, 0.5, 1.9), 0.5, M, (1.0, 0.90, 0.60), 0.75, 0.0),
        ("sphere", (0.6, 0.6, 4.2), 0.6, M, (0.9, 0.9, 0.9), 0.0, 0.0),
        ("tri", (-14.0, 0.0, -10.0, -14.0, 0.0, 10.0, 14.0, 0.0, -10.0), D, (1.0, 1.0, 1.0), 0.95, 0.0, 0,
         (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)),
        ("tri", (-14.0, 0.0, 10.0, 14.0, 0.0, 10.0, 14.0, 0.0, -10.0), D, (1.0, 1.0, 1.0), 0.95, 0.0, 0,
         (0.0, 1.0, 1.0, 1.0, 1.0, 0.0)),
    ]
    return {
        "ambient": ((0.95, 0.95, 1.0), 0.15),
        "skybox": skybox,
        "textures": [floor],
        "lights": [((11.8e9, 4.26e9, 3.08e9), 3.48e8, (1.0, 1.0, 0.95), 0.85)],
        "objects": objs,
    }


class _Lcg:
    """Generator fixed by SURVEY §8(d) config 4: s = s*1664525 + 1013904223, u = (s >> 8) / 2^24."""

    def __init__(self, seed=0x9E3779B9):
        self.s = seed & 0xFFFFFFFF

    def u(self):
        self.s = (self.s * 1664525 + 1013904223) & 0xFFFFFFFF
        return (self.s >> 8) / float(1 << 24)


def synthetic_scene(n_side=32, floor=None, skybox=None, seed=0x9E3779B9, back_wall=True):
    """Config 4: n_side^2 random reflective spheres on a jittered grid over the 28x20 textured floor.

    x in [-13,13], z in [-9,9], r in [0.1,0.3], y = r; alternating metal/dielectric; colour in [0.3,1]^3;
    reflectivity 1.0 w.p. 1/2 else U(0,1).  Floor (and optional back wall) are textured triangle pairs
    (the reference's Plane is untextured and unreachable through Scene).
    """
    g = _Lcg(seed)
    objs = []
    for iz in range(n_side):
        for ix in range(n_side):
            cellx, cellz = 26.0 / n_side, 18.0 / n_side
            r = 0.1 + 0.2 * g.u()
            r = min(r, 0.45 * min(cellx, cellz))
            x = -13.0 + (ix + 0.5) * cellx + (g.u() - 0.5) * (cellx - 2 * r)
            z = -9.0 + (iz + 0.5) * cellz + (g.u() - 0.5) * (cellz - 2 * r)
            col = (0.3 + 0.7 * g.u(), 0.3 + 0.7 * g.u(), 0.3 + 0.7 * g.u())
            refl = 1.0 if g.u() < 0.5 else g.u()
            mt = MT_METAL if (ix + iz) % 2 == 0 else MT_DIELECTRIC
            objs.append(("sphere", (x, r, z), r, mt, col, refl, 0.0))
    D = MT_DIELECTRIC
    objs.append(("tri", (-14.0, 0.0, -10.0, -14.0, 0.0, 10.0, 14.0, 0.0, -10.0), D, (1.0, 1.0, 1.0), 0.95, 0.0, 0,
                 (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
    objs.append(("tri", (-14.0, 0.0, 10.0, 14.0, 0.0, 10.0, 14.0, 0.0, -10.0), D, (1.0, 1.0, 1.0), 0.95, 0.0, 0,
                 (0.0, 1.0, 1.0, 1.0, 1.0, 0.0)))
    if back_wall:
        # wall at x = -14 facing +x (normal = (v1-v0) x (v2-v0))
        objs.append(("tri", (-14.0, 0.0, -10.0, -14.0, 8.0, -10.0, -14.0, 0.0, 10.0), D, (1.0, 1.0, 1.0), 0.5, 0.0, 0,
                     (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
        objs.append(("tri", (-14.0, 8.0, -10.0, -14.0, 8.0, 10.0, -14.0, 0.0, 10.0), D, (1.0, 1.0, 1.0), 0.5, 0.0, 0,
                     (0.0, 1.0, 1.0, 1.0, 1.0, 0.0)))
    return {
        "ambient": ((0.95, 0.95, 1.0), 0.15),
        "skybox": skybox,
        "textures": [floor],
        "lights": [((11.8e9, 4.26e9, 3.08e9), 3.48e8, (1.0, 1.0, 0.95), 0.85)],
        "objects": objs,
    }


def _torus_vertices(n_u, n_v, major, minor, center, tilt):
    """vertices of :func:`torus_mesh`; ``minor``: the tube radius, a scalar or one per (u, v) vertex [n_u, n_v]"""
    u = 2.0 * np.pi * np.arange(n_u) / n_u
    v = 2.0 * np.pi * np.arange(n_v) / n_v
    uu, vv = np.meshgrid(u, v, indexing="ij")
    ring = major + minor * np.cos(vv)
    x, y, z = ring * np.cos(uu), minor * np.sin(vv), ring * np.sin(uu)
    c, s = math.cos(tilt), math.sin(tilt)
    y, z = c * y - s * z, s * y + c * z
    return np.stack([x + center[0], y + center[1], z + center[2]], axis=-1).reshape(-1, 3).astype(np.float32)


def torus_mesh(n_u, n_v, major=2.2, minor=0.6, center=(0.0, 2.6, 0.0), tilt=1.0):
    """An indexed torus of 2 * n_u * n_v triangles: n_u segments around the ring, n_v around the tube, the ring's axis tilted by
    ``tilt`` radians about x.  Returns (xyz float32 [n_u * n_v, 3], idx uint32 [2 * n_u * n_v, 3]); the triangles face outwards."""
    xyz = _torus_vertices(n_u, n_v, major, minor, center, tilt)
    i, j = np.meshgrid(np.arange(n_u), np.arange(n_v), indexing="ij")
    a = i * n_v + j
    b = ((i + 1) % n_u) * n_v + j
    cc = ((i + 1) % n_u) * n_v + (j + 1) % n_v
    d = i * n_v + (j + 1) % n_v
    idx = np.stack([np.stack([a, cc, b], axis=-1), np.stack([a, d, cc], axis=-1)], axis=2).reshape(-1, 3).astype(np.uint32)
    return xyz, idx


def torus_wave(n_u, n_v, phase, amplitude=0.25, waves=3, major=2.2, minor=0.6, center=(0.0, 2.6, 0.0), tilt=1.0):
    """The vertices of :func:`torus_mesh` (same count and order: its index list applies) with a wave travelling around the ring on
    the tube radius: minor * (1 + amplitude * sin(waves * u - phase)) at ring angle u.  Stepping ``phase`` animates the torus."""
    u = 2.0 * np.pi * np.arange(n_u) / n_u
    r = minor * (1.0 + amplitude * np.sin(waves * u - phase))
    return _torus_vertices(n_u, n_v, major, np.repeat(r[:, None], n_v, axis=1), center, tilt)


def mesh_scene(n_u, n_v, spheres=0, floor=None, skybox=None):
    """A reflective metal torus of 2 * n_u * n_v triangles (:func:`torus_mesh`) in view of the default camera, over the textured floor
    and back wall of :func:`synthetic_scene`; ``spheres`` = n_side > 0 keeps that scene's n_side^2 spheres too."""
    base = synthetic_scene(max(spheres, 1), floor=floor, skybox=skybox)
    objs = [ob for ob in base["objects"] if spheres or ob[0] != "sphere"]
    xyz, idx = torus_mesh(n_u, n_v)
    objs.append(("mesh", xyz, idx, MT_METAL, (0.95, 0.8, 0.55), 0.85, 0.0))
    base["objects"] = objs
    return base


def with_ground_plane(scene, y=-0.05, refl=0.6, mtype=MT_METAL):
    """The same scene over an unbounded ground plane y = ``y`` facing up (a little below the floor triangles of :func:`synthetic_scene`):
    a reflective plane sends bounces from points far outside the objects' box back into the scene."""
    objs = list(scene["objects"]) + [("plane", (0.0, float(y), 0.0), (0.0, 1.0, 0.0), mtype, (0.55, 0.6, 0.65), float(refl), 0.0)]
    return dict(scene, objects=objs)


def object_indices(scene):
    """The object index the C ABI gives the first object of each entry of ``scene["objects"]`` (a "mesh" entry counts all its
    triangles), as :meth:`capi.Context.load_scene` issues them."""
    out, k = [], 0
    for ob in scene["objects"]:
        out.append(k)
        k += len(np.asarray(ob[2]).reshape(-1, 3)) if ob[0] == "mesh" else 1
    return out


def sphere_bounce(scene, t, height=1.5, pulse=0.0):
    """Every "sphere" entry of ``scene`` bouncing at time ``t``: returns (objects int32 [n], spheres float32 [n, 4] rows of
    (cx, cy, cz, r)) for :meth:`capi.Context.update_spheres`.  Sphere k rises by height * |sin(t + phase_k)| above its loaded centre
    (phase_k = 2.399963 k, the golden angle) and, with ``pulse``, its radius scales by 1 + pulse * sin(2 t + phase_k); a sphere that
    grows rises by as much, so its lowest point never sinks below the loaded one (a sphere resting on the floor stays on it).  At t = 0
    with pulse = 0 the rows are the loaded values bit for bit.  (For :func:`synthetic_scene`, height <= 4 with pulse <= 0.3 keeps every
    sphere above the floor and below the back wall's top, y = 8: inside the box the hierarchies and the light grid were built for.)"""
    objects, rows = [], []
    for k, (ob, i) in enumerate((ob, i) for ob, i in zip(scene["objects"], object_indices(scene)) if ob[0] == "sphere"):
        _, c, r, *_ = ob
        objects.append(i)
        rows.append((float(np.float32(c[0])), float(np.float32(c[1])), float(np.float32(c[2])), float(np.float32(r))))
    if not rows:
        return np.zeros(0, np.int32), np.zeros((0, 4), np.float32)
    base = np.asarray(rows, np.float64)
    phase = 2.399963 * np.arange(len(rows))
    out = base.copy()
    if pulse != 0.0:
        out[:, 3] = base[:, 3] * (1.0 + pulse * np.sin(2.0 * t + phase))
        out[:, 1] += np.maximum(out[:, 3] - base[:, 3], 0.0)
    if t != 0.0:
        out[:, 1] += height * np.abs(np.sin(t + phase))
    return np.asarray(objects, np.int32), out.astype(np.float32)


def with_spheres(scene, objects, spheres):
    """The same scene with the "sphere" entries whose object index (:func:`object_indices`) is in ``objects`` moved to the matching
    rows (cx, cy, cz, r) of ``spheres`` (a repeated index takes its last row): what rfx_update_spheres(objects, spheres) describes."""
    new = {int(i): tuple(float(x) for x in np.asarray(row, np.float32)) for i, row in zip(np.asarray(objects).reshape(-1), np.asarray(spheres, np.float32).reshape(-1, 4))}
    objs = []
    for ob, i in zip(scene["objects"], object_indices(scene)):
        if i in new:
            if ob[0] != "sphere":
                raise ValueError("object %d is not a sphere" % i)
            cx, cy, cz, r = new[i]
            ob = ("sphere", (cx, cy, cz), r) + tuple(ob[3:])
        objs.append(ob)
    return dict(scene, objects=objs)


def with_lights(scene, lights, records):
    """The same scene with the lights whose index is in ``lights`` replaced by the matching rows (origin[3], radius, rgb[3], power) of
    ``records`` (a repeated index takes its last row): what rfx_update_lights(lights, records) describes."""
    new = {int(i): tuple(float(x) for x in np.asarray(row, np.float32))
           for i, row in zip(np.asarray(lights).reshape(-1), np.asarray(records, np.float32).reshape(-1, 8))}
    out = list(scene["lights"])
    for i, r in new.items():
        if not 0 <= i < len(out):
            raise ValueError("light %d is not a light of the scene" % i)
        out[i] = ((r[0], r[1], r[2]), r[3], (r[4], r[5], r[6]), r[7])
    return dict(scene, lights=out)


def sun_orbit(scene, t, speed=1.0, swing=0.5):
    """The scene's first light as a sun crossing the sky at time ``t``: returns (lights int32 [1], records float32 [1, 8]) for
    :meth:`capi.Context.update_lights`.  The light keeps its distance from the origin, radius, colour and power; its azimuth about the
    vertical axis turns by speed * t and its elevation swings by ``swing`` * sin(t / 2) around the loaded one (kept between 0.1 and 1.4
    radians), so a light that is far from the scene stays far.  At t = 0 the record is the loaded light bit for bit."""
    (o, r, c, p) = scene["lights"][0]
    o64 = np.asarray(o, np.float32).astype(np.float64)
    if t != 0.0:
        dist = float(np.linalg.norm(o64))
        el = math.asin(max(-1.0, min(1.0, o64[1] / dist)))
        az = math.atan2(o64[2], o64[0])
        el = min(1.4, max(0.1, el + swing * math.sin(0.5 * t)))
        az += speed * t
        o64 = np.array([dist * math.cos(el) * math.cos(az), dist * math.sin(el), dist * math.cos(el) * math.sin(az)])
    rec = np.concatenate([o64, [r], np.asarray(c, np.float64), [p]]).astype(np.float32)
    return np.zeros(1, np.int32), rec.reshape(1, 8)


def expand_meshes(scene):
    """The same scene with every "mesh" object replaced by its triangles, in order (untextured "tri" objects)."""
    objs = []
    for ob in scene["objects"]:
        if ob[0] != "mesh":
            objs.append(ob)
            continue
        _, xyz, idx, mt, col, refl, tr = ob
        v = np.asarray(xyz, np.float32)[np.asarray(idx, np.int64)].reshape(-1, 9)
        objs.extend(("tri", tuple(float(x) for x in row), mt, col, refl, tr, -1, (0.0, 0.0, 0.0, 0.0, 0.0, 0.0)) for row in v)
    return dict(scene, objects=objs)


def synthetic_texture(w, h, seed, alpha=True):
    """Seeded synthetic ARGB texture (smooth gradients + hashed detail) — stands in for the missing TGA blobs."""
    ys, xs = np.mgrid[0:h, 0:w].astype(np.uint32)
    v = (xs * np.uint32(2654435761) ^ (ys * np.uint32(40503) + np.uint32(seed))) * np.uint32(2246822519)
    v ^= v >> np.uint32(13)
    r = ((xs * 255 // max(w - 1, 1)) + (v & np.uint32(31))) & np.uint32(255)
    g = ((ys * 255 // max(h - 1, 1)) + ((v >> np.uint32(8)) & np.uint32(31))) & np.uint32(255)
    b = (((xs // 16 + ys // 16) % 2) * 128 + ((v >> np.uint32(16)) & np.uint32(127))) & np.uint32(255)
    a = np.uint32(0xFF000000) if alpha else np.uint32(0)
    return (a | (r << np.uint32(16)) | (g << np.uint32(8)) | b).astype(np.uint32)


def write_tga(path, argb, bpp=32):
    """Type-2 uncompressed TGA as the reference loader expects (reference Texture.cpp:34-108, image_headers.h:4-18).

    Row 0 of the file is row 0 of the texture (the loader ignores the origin flag)."""
    h, w = argb.shape
    header = struct.pack("<bbbhhbhhhhbb", 0, 0, 2, 0, 0, 0, 0, 0, w, h, bpp, 0)
    a = np.ascontiguousarray(argb, dtype="<u4").view(np.uint8).reshape(h, w, 4)  # B, G, R, A in memory
    body = a.tobytes() if bpp == 32 else np.ascontiguousarray(a[:, :, :3]).tobytes()
    with open(path, "wb") as f:
        f.write(header)
        f.write(body)


def loaded_texture(argb, bpp=32):
    """What the reference holds in memory after loading ``write_tga(argb, bpp)``: 24-bpp files get alpha 0xFF."""
    if bpp == 24:
        return (argb | np.uint32(0xFF000000)).astype(np.uint32)
    return argb.astype(np.uint32)


def camera_lookat(eye, at, fov=DEFAULT_FOV):
    """``Camera(eye, at, fov)`` (reference Camera.cpp:24-36) in float32, op for op: returns (eye[3], view[9] row-major, fov).

    view columns are ox, oy, oz.  All arithmetic is float32 numpy scalars (IEEE RN, no contraction) so the result is
    bit-identical to the reference's constructor compiled without -ffast-math.
    """
    f = np.float32
    eye = [f(v) for v in eye]
    at = [f(v) for v in at]

    def sub(a, b):
        return [a[0] - b[0], a[1] - b[1], a[2] - b[2]]

    def cross(a, b):
        return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]

    def norm(a):
        ln = np.sqrt((a[0] * a[0] + a[1] * a[1]) + a[2] * a[2], dtype=np.float32)
        if ln > f(2.0 ** -63):
            return [a[0] / ln, a[1] / ln, a[2] / ln]
        return a

    up = [f(0.0), f(1.0), f(0.0)]
    oz = norm(sub(at, eye))
    ox = norm(cross(up, oz))
    oy = norm(cross(oz, ox))
    view = [ox[0], oy[0], oz[0], ox[1], oy[1], oz[1], ox[2], oy[2], oz[2]]
    return f32(eye), f32(view), np.float32(fov)


def default_camera():
    return camera_lookat(DEFAULT_EYE, DEFAULT_AT, DEFAULT_FOV)


def orbit_cameras(n_frames=240, fov=DEFAULT_FOV):
    """Config 5: frame k = default eye and at rotated about the world y axis by 2*pi*k/n (frame 0 == default camera)."""
    cams = []
    for k in range(n_frames):
        if k == 0:
            cams.append(default_camera())
            continue
        a = 2.0 * math.pi * k / n_frames
        c, s = math.cos(a), math.sin(a)

        def rot(p):
            return (np.float32(c * p[0] + s * p[2]), np.float32(p[1]), np.float32(-s * p[0] + c * p[2]))

        cams.append(camera_lookat(rot(DEFAULT_EYE), rot(DEFAULT_AT), fov))
    return cams


def _fmt(x):
    return "%.9g" % float(np.float32(x))


def scene_to_text(scene, tex_paths=None, sky_path=None):
    """Serialise for oracle/ref_harness.cpp (test infrastructure).  ``tex_paths[i]`` / ``sky_path``: TGA file
    paths for textures that are present; missing ones are written as '-' (load fails -> checker fallback)."""
    out = []
    rgb, p = scene["ambient"]
    out.append("ambient " + " ".join(_fmt(v) for v in rgb) + " " + _fmt(p))
    out.append("skybox " + (sky_path if (scene.get("skybox") is not None and sky_path) else "-"))
    for o, r, c, p in scene["lights"]:
        out.append("light " + " ".join(_fmt(v) for v in (*o, r, *c, p)))
    for i, t in enumerate(scene["textures"]):
        out.append("texture " + (tex_paths[i] if (t is not None and tex_paths) else "-"))
    for ob in scene["objects"]:
        if ob[0] == "sphere":
            _, c, r, mt, col, refl, tr = ob
            out.append("sphere " + " ".join(_fmt(v) for v in (*c, r)) + " %d " % mt + " ".join(_fmt(v) for v in (*col, refl, tr)))
        elif ob[0] == "tri":
            _, v, mt, col, refl, tr, tex, uv = ob
            out.append("tri " + " ".join(_fmt(x) for x in v) + " %d " % mt + " ".join(_fmt(x) for x in (*col, refl, tr)) +
                       " %d " % tex + " ".join(_fmt(x) for x in uv))
        else:
            raise ValueError("the reference Scene cannot hold a %s (no addPlane)" % ob[0])
    return "\n".join(out) + "\n"


def cameras_to_text(cams):
    lines = []
    for eye, view, fov in cams:
        lines.append("view " + " ".join(_fmt(v) for v in (*eye, *view, fov)))
    return "\n".join(lines) + "\n"
