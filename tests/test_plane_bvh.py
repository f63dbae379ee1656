"""Hierarchies in scenes with a plane: a bounce or shadow ray can start anywhere on the plane, so queries from outside the reach box grow
every box they test by grow * (L1 distance of the origin from the box) (rfx_selftest_far_bounds_host; rfx_scene.cpp has the derivation).

CPU: for origins 0.1 ... 1e5 reach diagonals outside the box, every point at which the float32 tests of Sphere.cpp:49-57 and
Triangle.cpp:56-68 (evaluated op for op in numpy) accept a ray lies in its box grown by that amount — with the slab test's share of the
margin left over — for grazing sphere silhouettes, rays aimed at the corners and edges of effective triangles, and shadow-ray-like
directions; tiny spheres, zero-area triangles and slivers included.  Without the growth the check fails.
GPU (-m gpu, tests/test_gpu_plane_bvh.py): the hierarchies in plane scenes give the list walk's frames bit for bit."""
import numpy as np
import pytest

from test_meshes import _accept, _construct, _effective

F = np.float32
VSN = F(2.0 ** -63)
DELTA = F(1e-4)


@pytest.fixture(scope="module")
def capi(rfx_lib):
    from reflaxman_b200 import capi
    return capi


def _sphere_accept(o, d, sph):
    """Sphere.cpp:49-62 in float32 for rays (o, d) [r][3] against spheres (cx, cy, cz, r) [s]: (accepted [r][s], t_f [r][s])"""
    c, sq = sph[None, :, :3], (sph[:, 3] * sph[:, 3])[None]          # sqRadius = radius * radius, Sphere.cpp:13
    o, d = o[:, None, :], d[:, None, :]
    with np.errstate(all="ignore"):
        a = (d[..., 0] * d[..., 0] + d[..., 1] * d[..., 1]) + d[..., 2] * d[..., 2]
        r2 = d * F(2)
        v = o - c
        b = (r2[..., 0] * v[..., 0] + r2[..., 1] * v[..., 1]) + r2[..., 2] * v[..., 2]
        cc = ((v[..., 0] * v[..., 0] + v[..., 1] * v[..., 1]) + v[..., 2] * v[..., 2]) - sq
        a4 = np.where(a > VSN, F(4) * a, F(np.nan))
        disc = b * b - a4 * cc
        t = (-b - np.sqrt(np.maximum(disc, F(0)))) / (F(2) * a)
        f = d * t[..., None]
        dist = np.sqrt((f[..., 0] * f[..., 0] + f[..., 1] * f[..., 1]) + f[..., 2] * f[..., 2])
        acc = (disc >= F(0)) & (b < F(0)) & (t > VSN) & (dist > DELTA)
    return acc, t


def _far_origins(rng, reach, n):
    """origins 0.1 ... 1e5 reach diagonals outside the reach box, in every direction"""
    lo, hi = reach[:3].astype(np.float64), reach[3:].astype(np.float64)
    R = float(np.linalg.norm(hi - lo))
    u = rng.normal(size=(n, 3))
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    D = R * 10.0 ** rng.uniform(-1, 5, (n, 1))
    return (0.5 * (lo + hi) + u * (0.5 * R + D)).astype(F)


def _distance(o, reach):
    """sum of the per-axis distances of o outside the box (binary64)"""
    o = o.astype(np.float64)
    lo, hi = reach[:3].astype(np.float64), reach[3:].astype(np.float64)
    return np.sum(np.maximum(np.maximum(lo - o, o - hi), 0.0), axis=1)


def _shadow_like(rng, o):
    """(L - P) + radius * randDir with |L| up to 1e10, in float32 as Scene.cpp:129"""
    n = len(o)
    L = rng.normal(size=(n, 3))
    L *= 10.0 ** rng.uniform(1, 10, (n, 1)) / np.linalg.norm(L, axis=1, keepdims=True)
    rd = rng.uniform(-1, 1, (n, 3))
    rad = 10.0 ** rng.uniform(-2, 8, (n, 1))
    return ((L.astype(F) - o) + rad.astype(F) * rd.astype(F)).astype(F)


def _outside(X, boxes, grow, shrink):
    """rows of X (binary64) outside their box grown by `grow` (per row) and shrunk by `shrink`"""
    g = (grow - shrink)[:, None]
    return np.any((X < boxes[:, :3] - g) | (X > boxes[:, 3:] + g), axis=1)


def _check(accept, o, d, objs, boxes, reach, K, R):
    """accepted (ray, object) pairs whose exact point o + t_f d lies outside the object's box grown by K * distance, with the slab
    test's share (1e-6 of the reach diagonal and of the distance) left over; (bad, accepted)"""
    bad = acc_n = 0
    dist = _distance(o, reach)
    for s in range(0, len(o), 256):
        acc, t = accept(o[s:s + 256], d[s:s + 256], objs)
        r, c = np.nonzero(acc)
        acc_n += len(r)
        X = o[s:s + 256][r].astype(np.float64) + t[r, c].astype(np.float64)[:, None] * d[s:s + 256][r].astype(np.float64)
        dd = dist[s:s + 256][r]
        keep = np.isfinite(boxes[c, 0])              # (-inf, +inf): tested by every query, nothing to check
        bad += int(np.sum(_outside(X, boxes[c].astype(np.float64), K * dd, 1e-6 * (R + dd)) & keep))
    return bad, acc_n


def _sphere_rays(rng, sph, reach, n):
    """far origins; directions grazing a sphere's silhouette (offsets from the radius up to 1e-2.5 of the distance), aimed at its
    centre, and shadow-ray-like"""
    o = _far_origins(rng, reach, n)
    k = rng.randint(0, len(sph), n)
    c, r = sph[k, :3].astype(np.float64), np.abs(sph[k, 3].astype(np.float64))
    v = c - o.astype(np.float64)
    perp = np.cross(v, rng.normal(size=(n, 3)))
    perp /= np.linalg.norm(perp, axis=1, keepdims=True)
    off = r + np.linalg.norm(v, axis=1) * 10.0 ** rng.uniform(-9, -2.5, n)
    graze = (c + perp * off[:, None] - o).astype(F)
    return np.concatenate([o, o, o]), np.concatenate([graze, v.astype(F), _shadow_like(rng, o)])


def _tri_rays(rng, v0, ax, reach, n):
    """far origins; directions aimed at the corners and edges of the effective triangles (binary64 targets), and shadow-ray-like"""
    E = _effective(v0, ax)
    fin = np.all(np.isfinite(E.reshape(len(E), -1)), 1)
    E = E[fin]
    o = _far_origins(rng, reach, n)
    j = rng.randint(0, len(E), n)
    w = rng.choice([0.0, 0.5, 1.0], (n, 2))
    w[:, 1] = np.minimum(w[:, 1], 1.0 - w[:, 0])
    target = E[j, 0] + w[:, :1] * (E[j, 1] - E[j, 0]) + w[:, 1:] * (E[j, 2] - E[j, 0])
    target += rng.normal(size=(n, 3)) * 10.0 ** rng.uniform(-9, -3, (n, 1)) * np.linalg.norm(target - o, axis=1, keepdims=True)
    return np.concatenate([o, o]), np.concatenate([(target - o.astype(np.float64)).astype(F), _shadow_like(rng, o)])


def _scene(rng):
    """spheres (unit-ish, tiny r 1e-4 ... 1e-2, large) and triangles (a torus mesh, random, zero-area, slivers kappa 1e3 ... 1e7) in
    one scene, with the reach box a scene of them would have (the eye at the origin)"""
    from reflaxman_b200 import scenes as S
    sph = [np.concatenate([rng.uniform(-6, 6, 3), [r]]) for r in rng.uniform(0.2, 1.5, 12)]
    sph += [np.concatenate([rng.uniform(-6, 6, 3), [r]]) for r in 10.0 ** rng.uniform(-4, -2, 16)]
    sph += [np.array([0.0, -40.0, 0.0, 38.0])]
    xyz, idx = S.torus_mesh(12, 6)
    tris = list(xyz[idx].reshape(-1, 9)) + list(rng.uniform(-5, 5, (20, 9)))
    for k in range(12):
        p0, e = rng.uniform(-3, 3, 3), rng.normal(size=3) * rng.choice([0.0, 0.01, 0.3])
        tris.append(np.concatenate([p0, p0 + e, p0 + 2.0 * e]) if k % 3 else np.concatenate([p0, p0, p0]))
    for kappa in np.logspace(3, 7, 16):
        p0, e, f = rng.uniform(-4, 4, 3), rng.normal(size=3), rng.normal(size=3)
        e *= 3.0 / np.linalg.norm(e)
        f -= e * (f @ e) / (e @ e)
        f *= 3.0 / np.linalg.norm(f) / kappa
        tris.append(np.concatenate([p0, p0 + e, p0 + 0.5 * e + f]))
    sph, tris = np.array(sph, F), np.array(tris, F)
    pts = np.concatenate([tris.reshape(-1, 3), sph[:, :3] - np.abs(sph[:, 3:]), sph[:, :3] + np.abs(sph[:, 3:])]).astype(np.float64)
    lo, hi = np.minimum(pts.min(0), 0.0), np.maximum(pts.max(0), 0.0)
    pad = 0.1 * (hi - lo)
    return sph, tris, np.concatenate([lo - pad, hi + pad]).astype(F)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_far_bounds_hold_every_accepted_point(capi, seed):
    """every sphere and triangle hit the float32 tests accept from 0.1 ... 1e5 reach diagonals outside the reach box lies in its box
    grown by grow * distance; with grow = 0 the same check fails for both kinds"""
    rng = np.random.RandomState(seed)
    sph, v, reach = _scene(rng)
    v0, ax = _construct(v)
    tris = np.concatenate([v0, ax], 1)
    sbox, tbox, s_reach, t_reach, (gs, gt) = capi.far_bounds_host(sph, tris, reach)
    assert np.array_equal(s_reach, reach)
    assert np.all(t_reach[:3] <= reach[:3]) and np.all(t_reach[3:] >= reach[3:])
    assert gs > 4 * 7.7e-4 and 1e-6 < gt <= 2.0 + 1e-6
    R_s = float(np.linalg.norm(reach[3:].astype(np.float64) - reach[:3]))
    R_t = float(np.linalg.norm(t_reach[3:].astype(np.float64) - t_reach[:3]))

    o, d = _sphere_rays(rng, sph, reach, 1500)
    bad, n_acc = _check(_sphere_accept, o, d, sph, sbox, s_reach, gs, R_s)
    assert n_acc > 200 and bad == 0, (bad, n_acc)
    teeth_s, _ = _check(_sphere_accept, o, d, sph, sbox, s_reach, 0.0, R_s)

    o, d = _tri_rays(rng, v0, ax, t_reach, 1500)
    acc_tri = lambda oo, dd, _: _accept(oo, dd, v0, ax)
    bad, n_acc = _check(acc_tri, o, d, None, tbox, t_reach, gt, R_t)
    assert n_acc > 200 and bad == 0, (bad, n_acc)
    teeth_t, _ = _check(acc_tri, o, d, None, tbox, t_reach, 0.0, R_t)
    assert teeth_s > 0 and teeth_t > 0, (teeth_s, teeth_t)


def test_far_bounds_slivers_are_tested_by_every_query(capi):
    """slivers (16u kappa > 1/2) and non-finite triangles get (-inf, +inf) under the plane-scene rule, where the in-box rule gives them
    the whole reach box; the other triangles' boxes are the in-box rule's, and the triangle growth follows the largest kappa of those"""
    rng = np.random.RandomState(11)
    sph, v, reach = _scene(rng)
    v0, ax = _construct(v)
    tris = np.concatenate([v0, ax], 1)
    _, tbox, _, _, (_, gt) = capi.far_bounds_host(sph, tris, reach)
    inbox = capi.tri_bounds_host(tris, reach)
    always = np.isinf(tbox[:, 0])
    assert always.sum() >= 4 and np.all(np.isneginf(tbox[always, :3])) and np.all(np.isposinf(tbox[always, 3:]))
    assert np.array_equal(tbox[~always], inbox[~always])
    A = np.linalg.inv(ax[~always].astype(np.float64).reshape(-1, 3, 3))
    M = ax[~always].astype(np.float64).reshape(-1, 3, 3)
    kappa = sum(np.linalg.norm(A[:, :, k], axis=1) * np.linalg.norm(M[:, k, :], axis=1) for k in range(3))
    assert gt >= 64 * 2.0 ** -24 * kappa.max() + 1e-6
    # a scene without triangles grows its triangle boxes by the slab share alone
    _, tb0, _, _, (_, gt0) = capi.far_bounds_host(sph, np.zeros((0, 12), F), reach)
    assert tb0.shape == (0, 6) and 1e-6 <= gt0 < 1.001e-6


def test_far_bounds_host_rejects_bad_arguments(capi):
    L = capi.load()
    reach = np.zeros(6, F)
    out = np.zeros(12, F)
    assert L.rfx_selftest_far_bounds_host(-1, None, 0, None, reach.ctypes.data_as(capi._fp), None, None, out.ctypes.data_as(capi._fp),
                                          out.ctypes.data_as(capi._fp)) == -1
    assert L.rfx_selftest_far_bounds_host(2, None, 0, None, reach.ctypes.data_as(capi._fp), None, None, out.ctypes.data_as(capi._fp),
                                          out.ctypes.data_as(capi._fp)) == -1
    assert L.rfx_selftest_far_bounds_host(0, None, 0, None, None, None, None, out.ctypes.data_as(capi._fp), out.ctypes.data_as(capi._fp)) == -1
    assert L.rfx_selftest_far_bounds_host(0, None, 0, None, reach.ctypes.data_as(capi._fp), None, None, out.ctypes.data_as(capi._fp),
                                          out.ctypes.data_as(capi._fp)) == 0
