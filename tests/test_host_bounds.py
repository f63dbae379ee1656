"""CPU tests of the two host-side bound computations the kernels' skipping rests on (pure host functions of the C-ABI library: no
GPU, no context), each against the kernels' float32 expressions evaluated op for op in numpy:
  * primary-ray screen bounds (rfx_trace_small.cu makePrimaryCull): no pixel outside an object's rectangle passes its accept test;
  * shadow-ray candidate grids of far lights (rfx_scene.cpp buildLightGrid): every sphere a jittered shadow ray passes the gate of is
    listed in the grid cell of the ray's origin."""
import math
import os
import sys

import numpy as np
import pytest

from reflaxman_b200 import scenes as S

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import primary_cull_proto as P  # noqa: E402

F = np.float32


@pytest.fixture(scope="module")
def capi(rfx_lib):
    from reflaxman_b200 import capi
    return capi


def _mixed_like_scene():
    """nine spheres of very different sizes, a floor and a wall (the constant-bank limits are 16 spheres / 8 triangles)"""
    objs = [("sphere", (float(x), float(r), float(z)), float(r), i % 2, (1.0, 1.0, 1.0), 0.5, 0.0)
            for i, (x, z, r) in enumerate([(-3, -2, 0.05), (-1, 1, 0.3), (0.5, -1.5, 0.8), (2, 2, 1.5), (4, -3, 0.1), (-5, 3, 2.5), (6, 0, 0.6), (0, 5, 0.02), (1, 0, 0.4)])]
    objs.append(("tri", (-14.0, 0.0, -10.0, -14.0, 0.0, 10.0, 14.0, 0.0, -10.0), 1, (1.0, 1.0, 1.0), 0.9, 0.0, -1, (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
    objs.append(("tri", (-14.0, 0.0, 10.0, 14.0, 0.0, 10.0, 14.0, 0.0, -10.0), 1, (1.0, 1.0, 1.0), 0.9, 0.0, -1, (0.0, 1.0, 1.0, 1.0, 1.0, 0.0)))
    objs.append(("tri", (-14.0, 0.0, -10.0, -14.0, 8.0, -10.0, -14.0, 0.0, 10.0), 1, (1.0, 1.0, 1.0), 0.5, 0.0, -1, (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
    return {"objects": objs}


@pytest.mark.parametrize("which", ["default", "sizes"])
def test_primary_bounds_host_are_conservative(capi, which):
    """213 cameras per scene — orbit, inside spheres, under the floor, looking away, fov 0.3..2.6 — at 256x144: the accept expressions of
    Sphere.cpp:49-57 / Triangle.cpp:56-68 in float32 on every pixel, and on the far corner of its SSAA / jitter footprint, never accept
    outside the rectangle the library derives; and the rectangles do exclude most of the image on average."""
    scene = S.default_scene() if which == "default" else _mixed_like_scene()
    sph, tris = P.scene_arrays(scene)
    W, H = 256, 144
    inside = total = 0
    for cam in P.random_cameras(200, 3 if which == "default" else 4, sph):
        srect, trect = capi.primary_bounds_host(cam, W, H, sph, tris)
        P.assert_inside(cam[0], cam[1], cam[2], W, H, sph, tris, srect, trect)
        for r in list(srect) + list(trect):
            inside += max(0, min(int(r[1]), W - 1) - max(int(r[0]), 0) + 1) * max(0, min(int(r[3]), H - 1) - max(int(r[2]), 0) + 1)
            total += W * H
    assert inside < 0.5 * total, (inside, total)


def test_primary_bounds_host_of_a_skewed_camera_are_the_whole_image(capi):
    sph, tris = P.scene_arrays(S.default_scene())
    eye, view, fov = S.default_camera()
    view = np.array(view, np.float32); view[0] *= np.float32(1.01)
    srect, trect = capi.primary_bounds_host((eye, view, fov), 320, 200, sph, tris)
    for r in list(srect) + list(trect):
        assert r[0] <= 0 and r[1] >= 319 and r[2] <= 0 and r[3] >= 199


def _shadow_gate_hits(P0, rd, light, spheres):
    """float32, op for op: qd = (L - P) + randDir * radius (Scene.cpp:129), then the gate of Sphere.cpp:49-53 against every sphere"""
    L = [F(light[0]), F(light[1]), F(light[2])]
    rad = F(light[3])
    d = [(L[k] - P0[:, k]) + rd[:, k] * rad for k in range(3)]
    a = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
    a4 = F(4) * a
    hits = np.zeros((len(P0), len(spheres)), bool)
    for i, s in enumerate(spheres):
        vx, vy, vz = P0[:, 0] - F(s[0]), P0[:, 1] - F(s[1]), P0[:, 2] - F(s[2])
        b = ((d[0] * F(2)) * vx + (d[1] * F(2)) * vy) + (d[2] * F(2)) * vz
        c = ((vx * vx + vy * vy) + vz * vz) - F(s[3]) * F(s[3])
        with np.errstate(all="ignore"):
            disc = b * b - a4 * c
        hits[:, i] = (disc >= 0) & (b < 0)
    return hits


@pytest.mark.parametrize("seed", range(6))
def test_light_grid_host_lists_every_sphere_a_shadow_ray_can_hit(capi, seed):
    rng = np.random.default_rng(500 + seed)
    n = int(rng.integers(60, 400))
    r = (10 ** rng.uniform(-1.6, 0.2, n)).astype(F)
    c = rng.uniform([-13, 0, -9], [13, 4, 9], (n, 3)).astype(F)
    c[:, 1] += r
    spheres = np.concatenate([c, r[:, None]], axis=1).astype(F)
    lo = np.minimum((c - r[:, None]).min(0), [-14, 0, -10]).astype(float)
    hi = np.maximum((c + r[:, None]).max(0), [14, 8 if seed % 2 else 0, 10]).astype(float)
    diag = float(np.linalg.norm(hi - lo))
    pad = 1e-3 * diag + 1e-5 * (np.abs(lo).sum() + np.abs(hi).sum())           # as uploadScene pads the box of the drop points
    box = np.concatenate([lo - pad, hi + pad])
    reach = 1.2 * diag + 20.0
    checked = 0
    for k in range(4):
        dvec = rng.normal(size=3)
        if k == 1:
            dvec = np.array([0.0, 1.0, 0.0])
        if k == 2:
            dvec = np.array([1.0, 0.03, -0.4])
        dvec /= np.linalg.norm(dvec)
        dist = float(10 ** rng.uniform(3.0, 10.0))
        light = np.array([*(dvec * dist), dist * float(rng.uniform(0.0005, 0.04))], F)
        g = capi.light_grid_host(light, spheres, box, reach)
        assert g is not None
        uv, nx, ny, cells, items = g
        member = np.zeros((nx * ny + 1, n), bool)                              # last row: origins outside the grid (no candidates)
        for cell in range(nx * ny):
            member[cell, items[cells[cell]:cells[cell + 1]]] = True
        # origins: points of sphere surfaces, of the floor, and anywhere in the box; jitter anywhere in the unit ball
        m = 30000
        pick = rng.integers(0, n, m)
        u3 = rng.normal(size=(m, 3)); u3 /= np.linalg.norm(u3, axis=1)[:, None]
        on_sph = (c[pick].astype(float) + u3 * r[pick, None].astype(float))
        floor = np.stack([rng.uniform(-14, 14, m), np.zeros(m), rng.uniform(-10, 10, m)], axis=1)
        anywhere = rng.uniform(lo, hi, (m, 3))
        P0 = np.concatenate([on_sph, floor, anywhere]).astype(F)
        P0 = np.clip(P0, (lo).astype(F), (hi).astype(F))
        rd = rng.normal(size=(len(P0), 3)); rd /= np.linalg.norm(rd, axis=1)[:, None]
        rd = (rd * rng.uniform(0, 1, (len(P0), 1)) ** (1 / 3)).astype(F)
        hits = _shadow_gate_hits(P0, rd, light, spheres)
        # the device's cell: floor(fma(u0, x, fma(u1, y, fma(u2, z, u3)))) in float32
        def coord(row):
            t = (np.float64(row[2]) * P0[:, 2].astype(np.float64) + np.float64(row[3])).astype(F)
            t = (np.float64(row[1]) * P0[:, 1].astype(np.float64) + t.astype(np.float64)).astype(F)
            t = (np.float64(row[0]) * P0[:, 0].astype(np.float64) + t.astype(np.float64)).astype(F)
            return np.floor(t).astype(np.int64)
        cu, cv = coord(uv[0]), coord(uv[1])
        inside = (cu >= 0) & (cu < nx) & (cv >= 0) & (cv < ny)
        cell = np.where(inside, cv * nx + cu, nx * ny)
        missing = hits & ~member[cell]
        assert not missing.any(), (seed, k, int(missing.sum()), np.argwhere(missing)[:3])
        checked += int(hits.sum())
        assert len(items) < 40 * n                                            # the lists stay short: the grid does select
    assert checked > 1000                                                     # the rays did hit spheres


def test_light_grid_host_declines_a_near_light(capi):
    spheres = np.array([[0, 1, 0, 1], [3, 0.5, 1, 0.5]], F)
    assert capi.light_grid_host((2.0, 6.0, -1.0, 0.5), spheres, (-5, 0, -5, 5, 3, 5), 30.0) is None


@pytest.mark.parametrize("which", ["grid16", "cloud"])
def test_eye_grid_host_lists_every_sphere_a_primary_ray_can_hit(capi, which):
    """The screen grid of a path's first query (blob scenes): for 113 cameras per scene — orbit, inside spheres, under the floor, looking
    away — every sphere whose float32 accept expression (Sphere.cpp:49-57) a pixel's primary ray passes, or the ray through the far
    corner of the pixel's SSAA / jitter footprint, is listed in the pixel's 32x32 cell; and the lists are short."""
    if which == "grid16":
        scene = S.synthetic_scene(16)
    else:
        rng = np.random.default_rng(78)
        objs = []
        for i in range(180):
            r = float(10 ** rng.uniform(-1.5, 0.3))
            c = rng.uniform([-8, 0, -6], [8, 5, 6])
            objs.append(("sphere", (float(c[0]), float(c[1]) + r, float(c[2])), r, i % 2, (1.0, 1.0, 1.0), 0.5, 0.0))
        scene = {"objects": objs}
    sph, _ = P.scene_arrays(scene)
    n = len(sph)
    W, H = 200, 120
    listed = cells_total = 0
    for eye, view, fov in P.random_cameras(100, 9, sph):
        g = capi.eye_grid_host((eye, view, fov), W, H, sph)
        assert g is not None
        nx, ny, shift, cells, items = g
        assert (nx, ny, shift) == ((W + 31) // 32, (H + 31) // 32, 5)
        member = np.zeros((nx * ny, n), bool)
        for cell in range(nx * ny):
            member[cell, items[cells[cell]:cells[cell + 1]]] = True
        cell_of = ((np.arange(H)[:, None] >> shift) * nx + (np.arange(W)[None, :] >> shift))
        rz = F(F(W) / F(2) / F(math.tan(F(fov) / F(2))))
        for offx, offy in ((0.0, 0.0), (1.99, 1.99)):
            d = P.primary_rays(eye, view, rz, F(W) / F(2), F(H) / F(2), W, H, offx, offy)
            for i, s in enumerate(sph):
                acc = P.sphere_accept(eye, d, s)
                assert not (acc & ~member[cell_of, i]).any(), (which, i)
        listed += len(items); cells_total += nx * ny
    assert listed < 0.35 * n * cells_total, (listed, cells_total)
