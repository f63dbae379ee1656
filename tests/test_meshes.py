"""Triangle meshes in blob scenes: the hierarchy over the triangles (rfx_set_bvh_mode), indexed-mesh upload (rfx_add_mesh) and scenes
larger than the old 200 KB blob cap.

CPU: the boxes of the triangle hierarchy (rfx_selftest_tri_bounds_host) hold every point at which the float32 test of
Triangle.cpp:56-68, evaluated op for op in numpy, accepts a ray — for mesh, random, sliver, zero-area, tiny-and-far and huge triangles,
rays from anywhere in the reach box and from drop points on other triangles, aimed at the corners and edges of what the test accepts.
GPU (-m gpu): every frame, signature, ray count and stream position under the hierarchy is identical to the list walk."""
import numpy as np
import pytest

from reflaxman_b200 import scenes as S
from reflaxman_b200 import sharding as P

F = np.float32
VSN = F(2.0 ** -63)


@pytest.fixture(scope="module")
def capi(rfx_lib):
    from reflaxman_b200 import capi
    return capi


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------

def _construct(v):
    """rfx_add_triangle's float32 constructor (Triangle.cpp:11-21, Matrix33.cpp:49-79) over arrays of triangles v [n][9]:
    (v0 [n][3], axTrans [n][9])."""
    v = np.asarray(v, F).reshape(-1, 9)
    v0, v1, v2 = v[:, 0:3], v[:, 3:6], v[:, 6:9]
    e1, e2 = v1 - v0, v2 - v0
    n = np.stack([e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1], e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2], e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]], 1)
    ln = np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])
    with np.errstate(all="ignore"):
        n = np.where((ln > VSN)[:, None], n / ln[:, None], n)
    u, w, m = e2, e1, -n                                     # columns v2-v0 | v1-v0 | -n
    _11, _12, _13, _21, _22, _23, _31, _32, _33 = u[:, 0], w[:, 0], m[:, 0], u[:, 1], w[:, 1], m[:, 1], u[:, 2], w[:, 2], m[:, 2]
    d = (_11 * (_22 * _33 - _32 * _23) + _21 * (_32 * _13 - _12 * _33)) + _31 * (_12 * _23 - _13 * _22)
    with np.errstate(all="ignore"):
        ax = np.stack([(_22 * _33 - _23 * _32) / d, (_13 * _32 - _12 * _33) / d, (_12 * _23 - _13 * _22) / d,
                       (_23 * _31 - _21 * _33) / d, (_11 * _33 - _13 * _31) / d, (_13 * _21 - _11 * _23) / d,
                       (_21 * _32 - _22 * _31) / d, (_12 * _31 - _11 * _32) / d, (_11 * _22 - _12 * _21) / d], 1)
    ax = np.where((np.abs(d) > VSN)[:, None], ax, np.eye(3, dtype=F).reshape(1, 9))
    return v0.astype(F), ax.astype(F)


def _effective(v0, ax):
    """binary64 corners v0, v0 + a, v0 + b of the triangle the test accepts ([a | b | c] = axTrans^-1)"""
    A = np.linalg.inv(ax.astype(np.float64).reshape(-1, 3, 3))
    p0 = v0.astype(np.float64)
    return np.stack([p0, p0 + A[:, :, 0], p0 + A[:, :, 1]], 1)


def _accept(o, d, v0, ax):
    """Triangle.cpp:56-68 in float32 for rays (o, d) [r][3] against triangles [t]: (accepted [r][t], t_f [r][t])"""
    o, d = o[:, None, :], d[:, None, :]
    p = o - v0[None]

    def row(k, vec):
        return (vec[..., 0] * ax[None, :, 3 * k] + vec[..., 1] * ax[None, :, 3 * k + 1]) + vec[..., 2] * ax[None, :, 3 * k + 2]
    with np.errstate(all="ignore"):
        oz, rz = row(2, p), row(2, d)
        gate = (np.signbit(oz) != np.signbit(rz)) & (np.abs(rz) > VSN) & (np.abs(oz) > F(0))
        t = -oz / rz
        u = row(0, p) + t * row(0, d)
        v = row(1, p) + t * row(1, d)
        acc = gate & (t > VSN) & (u >= F(0)) & (v >= F(0)) & (u + v < F(1))
    return acc, t


def _tri_groups(rng):
    """name -> (vertices [n][9], reach lo/hi [6]) — each group with the reach box a scene of it would have"""
    g = {}
    xyz, idx = S.torus_mesh(24, 12)
    g["torus"] = xyz[idx].reshape(-1, 9)
    g["random"] = rng.uniform(-5, 5, (150, 9))
    sl = []
    for kappa in np.logspace(3, 7, 40):
        p0, e, f = rng.uniform(-4, 4, 3), rng.normal(size=3), rng.normal(size=3)
        e *= 3.0 / np.linalg.norm(e)
        f -= e * (f @ e) / (e @ e)
        f *= 3.0 / np.linalg.norm(f) / kappa
        sl.append(np.concatenate([p0, p0 + e, p0 + 0.5 * e + f]))
    g["slivers"] = np.array(sl)
    za = []
    for k in range(30):
        p0, e = rng.uniform(-0.6, 0.6, 3), rng.normal(size=3) * rng.choice([0.0, 0.01, 0.3])
        za.append(np.concatenate([p0, p0 + e, p0 + 2.0 * e]) if k % 3 else np.concatenate([p0, p0, p0]))
    g["zero_area"] = np.array(za)
    far = []
    for k in range(30):
        c = np.array([1000.0, 0.0, 0.0]) + rng.uniform(-20, 20, 3)
        far.append(np.concatenate([c, c + rng.normal(size=3) * 1e-4, c + rng.normal(size=3) * 1e-4]))
    g["tiny_far"] = np.array(far)
    g["huge"] = rng.uniform(-1e4, 1e4, (20, 9))
    out = {}
    for name, v in g.items():
        v = np.asarray(v, F)
        pts = v.reshape(-1, 3).astype(np.float64)
        lo, hi = np.minimum(pts.min(0), 0.0), np.maximum(pts.max(0), 0.0)   # the eye at the origin
        pad = 0.1 * (hi - lo)
        out[name] = (v, np.concatenate([lo - pad, hi + pad]).astype(F))
    return out


def _rays(rng, v0, ax, reach, n):
    """origins: uniform in reach, and drop points on the triangles; directions: aimed at the corners and edges of the effective
    triangles (where the box is tight), unit, non-unit, and shadow-ray-like (L - P) + r randDir with |L| = 1e10"""
    lo, hi = reach[:3].astype(np.float64), reach[3:].astype(np.float64)
    E = _effective(v0, ax)
    fin = np.all(np.isfinite(E.reshape(len(E), -1)), 1)
    E = E[fin]
    o_box = rng.uniform(lo, hi, (n, 3))
    k = rng.randint(0, len(E), n)
    bu, bv = rng.uniform(0, 1, n), rng.uniform(0, 1, n)
    sw = bu + bv > 1
    bu[sw], bv[sw] = 1 - bu[sw], 1 - bv[sw]
    o_drop = E[k, 0] + bu[:, None] * (E[k, 1] - E[k, 0]) + bv[:, None] * (E[k, 2] - E[k, 0])
    origins = np.concatenate([o_box, o_drop]).astype(F)
    m = len(origins)
    j = rng.randint(0, len(E), m)
    w = rng.choice([0.0, 0.5, 1.0], (m, 2))
    w[:, 1] = np.minimum(w[:, 1], 1.0 - w[:, 0])
    target = E[j, 0] + w[:, :1] * (E[j, 1] - E[j, 0]) + w[:, 1:] * (E[j, 2] - E[j, 0])
    aimed = (target - origins.astype(np.float64))
    unit = rng.normal(size=(m, 3))
    unit /= np.linalg.norm(unit, axis=1, keepdims=True)
    scaled = unit * np.exp(rng.uniform(-7, 7, (m, 1)))
    L = rng.normal(size=(m, 3))
    L *= 1e10 / np.linalg.norm(L, axis=1, keepdims=True)
    rd = rng.uniform(-1, 1, (m, 3))
    shadow = ((L.astype(F) - origins) + F(3.48e8) * rd.astype(F)).astype(F)
    o = np.concatenate([origins] * 4)
    d = np.concatenate([aimed.astype(F), unit.astype(F), scaled.astype(F), shadow])
    return o, d


def _check(o, d, v0, ax, boxes, shrink):
    """accepted pairs whose exact point o + t_f d (binary64) lies outside the box shrunk by `shrink`"""
    bad = 0
    for s in range(0, len(o), 256):
        acc, t = _accept(o[s:s + 256], d[s:s + 256], v0, ax)
        r, c = np.nonzero(acc)
        X = o[s:s + 256][r].astype(np.float64) + t[r, c].astype(np.float64)[:, None] * d[s:s + 256][r].astype(np.float64)
        b = boxes[c].astype(np.float64)
        bad += int(np.sum(np.any((X < b[:, :3] + shrink) | (X > b[:, 3:] - shrink), axis=1)))
    return bad


def _reach_diagonal(v0, ax, reach):
    E = _effective(v0, ax)
    E = E[np.all(np.isfinite(E.reshape(len(E), -1)), 1)].reshape(-1, 3)
    lo = np.minimum(reach[:3].astype(np.float64), E.min(0))
    hi = np.maximum(reach[3:].astype(np.float64), E.max(0))
    return float(np.linalg.norm(hi - lo))


def test_tri_bounds_host_hold_every_accepted_point(capi):
    """for every (ray, triangle) pair the float32 test accepts, the exact point o + t_f d lies inside the triangle's box shrunk by 1e-6 R;
    and the check has teeth: boxes of the effective triangles without margin fail it, and boxes of the given vertices fail it for the
    zero-area triangles (their test accepts a unit triangle at v0)"""
    rng = np.random.RandomState(7)
    teeth_e = teeth_v = 0
    for name, (v, reach) in _tri_groups(rng).items():
        v0, ax = _construct(v)
        tris = np.concatenate([v0, ax], 1)
        boxes = capi.tri_bounds_host(tris, reach)
        assert boxes.shape == (len(v), 6) and np.all(boxes[:, :3] <= boxes[:, 3:]), name
        R = _reach_diagonal(v0, ax, reach)
        o, d = _rays(rng, v0, ax, reach, 400)
        acc_pairs = sum(int(_accept(o[s:s + 256], d[s:s + 256], v0, ax)[0].sum()) for s in range(0, len(o), 256))
        assert acc_pairs > 50, (name, acc_pairs)
        assert _check(o, d, v0, ax, boxes, 1e-6 * R) == 0, name
        E = _effective(v0, ax)
        ok = np.all(np.isfinite(E.reshape(len(E), -1)), 1)
        ebox = np.concatenate([E.min(1), E.max(1)], 1).astype(np.float64)
        ebox[~ok] = boxes[~ok]
        teeth_e += _check(o, d, v0, ax, ebox, 1e-6 * R)
        if name == "zero_area":
            vv = v.reshape(-1, 3, 3).astype(np.float64)
            teeth_v += _check(o, d, v0, ax, np.concatenate([vv.min(1), vv.max(1)], 1), 1e-6 * R)
    assert teeth_e > 0 and teeth_v > 0, (teeth_e, teeth_v)


def test_tri_bounds_host_rejects_bad_arguments(capi):
    L = capi.load()
    reach = np.zeros(6, F)
    assert L.rfx_selftest_tri_bounds_host(-1, None, reach.ctypes.data_as(capi._fp), None) == -1
    assert L.rfx_selftest_tri_bounds_host(3, None, reach.ctypes.data_as(capi._fp), None) == -1
    assert L.rfx_selftest_tri_bounds_host(0, None, reach.ctypes.data_as(capi._fp), None) == 0


def test_mesh_scene_expands_to_its_triangles():
    """2 n_u n_v triangles; expand_meshes keeps every other object and the triangle order of the index array"""
    xyz, idx = S.torus_mesh(16, 8)
    assert idx.shape == (2 * 16 * 8, 3) and xyz.shape == (16 * 8, 3) and int(idx.max()) < len(xyz)
    sc = S.mesh_scene(16, 8)
    ex = S.expand_meshes(sc)
    assert [o[0] for o in ex["objects"]] == ["tri"] * (4 + 256)
    assert ex["objects"][4 + 5][1] == tuple(float(x) for x in xyz[idx[5]].reshape(9))
    assert len(S.expand_meshes(S.mesh_scene(16, 8, spheres=4))["objects"]) == 16 + 4 + 256
    S.scene_to_text(ex)


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------

def _adversarial(rng, xyz, idx, n):
    """triangles the exact test treats unusually, placed on and around the torus: zero-area (collinear and coincident vertices: identity
    basis), slivers, exact copies of mesh triangles and of their edge-sharing neighbours (coplanar ties resolved by insertion order)"""
    objs = []
    col = (0.6, 0.9, 0.7)
    for k in range(n):
        t = xyz[idx[rng.randint(len(idx))]].astype(np.float64)
        kind = k % 4
        if kind == 0:
            e = rng.normal(size=3) * 0.2
            v = np.concatenate([t[0], t[0] + e, t[0] + 2 * e])
        elif kind == 1:
            v = np.concatenate([t[0], t[0], t[0]])
        elif kind == 2:
            v = np.concatenate([t[0], t[1], t[0] + 0.5 * (t[1] - t[0]) + 1e-5 * (t[2] - t[0])])
        else:
            v = t.reshape(9)
        objs.append(("tri", tuple(float(x) for x in v.astype(F)), k % 2, col, 0.7, 0.0, -1, (0.0,) * 6))
    return objs


def _mesh_case(n_u, n_v, spheres=0, adversarial=64):
    scene = S.mesh_scene(n_u, n_v, spheres=spheres, floor=S.synthetic_texture(64, 64, 3), skybox=S.synthetic_texture(128, 96, 5))
    xyz, idx = S.torus_mesh(n_u, n_v)
    scene["objects"] += _adversarial(np.random.RandomState(n_u * 7 + n_v), xyz, idx, adversarial)
    return scene


def _n_tris(scene):
    return sum(len(o[2]) if o[0] == "mesh" else o[0] == "tri" for o in scene["objects"])


FAR_CAM = S.camera_lookat((38.0, 17.0, -30.0), (0.0, 2.0, 0.0), 0.6)


def _run_modes(capi, scene, fn, modes=(2, 0, 1)):
    out = {}
    for mode in modes:
        c = capi.Context(0)
        try:
            c.load_scene(scene)
            c.set_bvh_mode(mode)
            out[mode] = fn(c)
        finally:
            c.close()
    return out


def _assert_same(out, what):
    ref = out[2]
    for mode, got in out.items():
        assert len(got) == len(ref), (what, mode)
        for k, (a, b) in enumerate(zip(got, ref)):
            if isinstance(a, np.ndarray):
                assert a.dtype == b.dtype and np.array_equal(a.view(np.uint32) if a.dtype == np.float32 else a, b.view(np.uint32) if b.dtype == np.float32 else b), (what, mode, k)
            else:
                assert a == b, (what, mode, k, a, b)


@pytest.mark.gpu
@pytest.mark.parametrize("n_u,n_v", [(32, 32), (128, 64)], ids=["2048", "16384"])
def test_tri_bvh_equals_list_walk(capi, n_u, n_v):
    """batch frames (wavefront pair and single tile kernel) and the general kernel with hit-path signatures: float image, ARGB,
    signatures, ray and bounce counts and the stream position identical to the list walk, for the default camera and one orbiting far
    outside the mesh; bvh_triangles = every triangle under modes 0 and 1, 0 under mode 2"""
    scene = _mesh_case(n_u, n_v)
    n = _n_tris(scene)
    W, H, depth = 160, 90, 8
    cams = [S.default_camera(), FAR_CAM]

    def run(c):
        res = []
        c.set_seeds(77, 77); c.set_image_size(W, H)
        for path, wave in ((2, 2), (2, 0)):
            c.force_path(path); c.set_option("blob_wavefront", wave); c.stats_reset()
            res += [c.render_frames(cams, depth).copy(), c.stats()["rays"], c.stats()["bounces"], c.get_seeds()]
        c.force_path(3); c.enable_signatures(True); c.stats_reset()
        for cam in cams:
            c.render(cam, depth)
            res += [c.read_rgbf().copy(), c.read_argb().copy(), c.read_signatures().copy()]
        st = c.stats()
        res += [st["rays"], st["bounces"], c.get_seeds(), st["bvh_triangles"]]
        return res
    out = _run_modes(capi, scene, run)
    assert out[2][-1] == 0 and out[0][-1] == n and out[1][-1] == n, (out[2][-1], out[0][-1], out[1][-1], n)
    for m in out:
        out[m] = out[m][:-1]
    _assert_same(out, "mesh %d" % n)


@pytest.mark.gpu
def test_tri_bvh_every_render_mode_equals_list_walk(capi):
    """2x2 SSAA, 3 additive passes, ragged render_next slices, block preview, rfx_trace_rays from origins outside the reach box
    (re-flatten), a 2-way render_strips split, and an eye inside the torus's box then far away (re-flatten): identical to the list walk"""
    scene = _mesh_case(32, 32)
    W, H, depth = 96, 60, 6
    cam = S.orbit_cameras(9)[2]
    inside = S.camera_lookat((0.3, 2.6, 0.2), (3.0, 2.0, 1.0), 1.3)

    def run(c):
        res = []
        c.set_seeds(5, 9); c.set_image_size(W, H); c.force_path(2)
        c.render(cam, depth, samples=2)
        res += [c.read_rgbf().copy(), c.read_argb().copy()]
        for _ in range(3):
            c.render(cam, depth, additive=True)
        res.append(c.read_rgbf().copy())
        c.render(cam, depth, chunk=1013)
        res.append(c.read_rgbf().copy())
        c.render(cam, depth, samples=-3)
        res.append(c.read_argb().copy())
        rng = np.random.RandomState(3)
        o = rng.uniform(-60, 60, (500, 3)).astype(F)
        r = (np.array([0.0, 2.6, 0.0], F) + rng.uniform(-3, 3, (500, 3)).astype(F) - o).astype(F)
        res.append(c.trace_rays(o, r, depth).copy())
        gather = c.buffer_alloc(W * H * 4)
        for rank in range(2):
            P.split_frame(c, cam, depth, 1, 2, rank, gather, strip_rows=8)
            c.synchronize()
        res.append(c.buffer_read(gather, np.zeros((H, W), np.uint32)).copy())
        c.buffer_free(gather)
        for eye_cam in (inside, FAR_CAM):
            c.render(eye_cam, depth)
            res.append(c.read_rgbf().copy())
        st = c.stats()
        res += [st["rays"], st["bounces"], c.get_seeds()]
        return res
    _assert_same(_run_modes(capi, scene, run), "render modes")


@pytest.mark.gpu
def test_mesh_scene_matches_oracle(capi, oracle):
    """2 048 mesh triangles (plus adversarial ones) at 128x72, depth 8: the hierarchy's hit-path signatures equal the oracle's on every
    pixel (the oracle takes the expanded triangles), and the frame meets the parity bar"""
    import cases
    scene = _mesh_case(32, 32, adversarial=16)
    W, H, depth = 128, 72, 8
    cam = S.default_camera()
    c = capi.Context(0)
    try:
        c.load_scene(scene); c.set_seeds(321, 321); c.set_image_size(W, H); c.enable_signatures(True); c.stats_reset()
        c.render(cam, depth)
        argb, sig, st = c.read_argb(), c.read_signatures(), c.stats()
        assert st["bvh_triangles"] == _n_tris(scene)
    finally:
        c.close()
    o = oracle.OracleRender(S.expand_meshes(scene), W, H, seed=321).render(cam, depth, want_sig=True)
    assert np.array_equal(sig, o.sig), "hit-path signatures differ on %d pixels" % int((sig != o.sig).sum())
    assert st["rays"] == o.counters["rays"]
    cases.assert_parity(argb, o.resolve()[1], "mesh scene")


@pytest.mark.gpu
def test_mixed_spheres_and_mesh_equal_list_walk(capi):
    """synthetic_scene(32)'s 1024 spheres and floor plus a 16 384-triangle torus: sphere hierarchy, light grid, eye grid and triangle
    hierarchy all on under mode 0; identical to the list walk"""
    scene = _mesh_case(128, 64, spheres=32, adversarial=16)
    W, H, depth = 192, 108, 8
    cams = [S.default_camera(), S.orbit_cameras(7)[3]]

    def run(c):
        c.set_seeds(11, 11); c.set_image_size(W, H); c.force_path(2); c.stats_reset()
        frames = c.render_frames(cams, depth).copy()
        c.render(cams[1], depth)
        st = c.stats()
        return [frames, c.read_rgbf().copy(), st["rays"], st["bounces"], c.get_seeds(), st["light_grids"] > 0, st["bvh_triangles"] > 0]
    out = _run_modes(capi, scene, run, modes=(2, 0))
    assert out[0][-2:] == [True, True] and out[2][-2:] == [False, False]
    for m in out:
        out[m] = out[m][:-2]
    _assert_same(out, "mixed")


@pytest.mark.gpu
def test_add_mesh_equals_per_triangle_adds(capi):
    """rfx_add_mesh gives the object indices and the frames of the same triangles added one by one; a bad vertex index or a NULL array is
    RFX_ERR_ARG and adds nothing; mesh triangles take a texture like any triangle"""
    xyz, idx = S.torus_mesh(12, 6)
    base = S.mesh_scene(12, 6)
    base["objects"] = [o for o in base["objects"] if o[0] != "mesh"]
    W, H, depth = 96, 54, 6
    frames = []
    for use_mesh in (True, False):
        c = capi.Context(0)
        try:
            c.load_scene(base)
            first = 4
            if use_mesh:
                assert c.add_mesh(xyz, idx, S.MT_METAL, (0.9, 0.8, 0.5), 0.8, 0.0) == first
            else:
                for k, t in enumerate(idx):
                    assert c._ck(c.L.rfx_add_triangle(c.h, xyz[t].reshape(9).ctypes.data_as(capi._fp), S.MT_METAL,
                                                      np.array([0.9, 0.8, 0.5], F).ctypes.data_as(capi._fp), F(0.8), F(0.0)), "add") == first + k
            c._ck(c.L.rfx_set_triangle_texture(c.h, first + 3, 0, np.array([0, 0, 1, 0, 0, 1], F).ctypes.data_as(capi._fp)), "texture")
            bad = idx.copy(); bad[5, 1] = len(xyz)
            with pytest.raises(capi.RfxError):
                c.add_mesh(xyz, bad, S.MT_METAL, (1.0, 1.0, 1.0), 0.5, 0.0)
            assert c.L.rfx_add_mesh(c.h, len(xyz), None, len(idx), idx.ctypes.data_as(capi._u32p), 0, np.ones(3, F).ctypes.data_as(capi._fp), F(0), F(0)) == -1
            nxt = c._ck(c.L.rfx_add_triangle(c.h, np.array([0, 9, 0, 1, 9, 0, 0, 9, 1], F).ctypes.data_as(capi._fp), 0,
                                             np.ones(3, F).ctypes.data_as(capi._fp), F(0.5), F(0.0)), "add")
            assert nxt == first + len(idx)                      # the failed calls added nothing
            c.set_seeds(4, 4); c.set_image_size(W, H); c.set_bvh_mode(1)
            frames.append(c.render_frames([S.default_camera(), FAR_CAM], depth).copy())
        finally:
            c.close()
    assert np.array_equal(frames[0], frames[1])


@pytest.mark.gpu
def test_scene_over_200kb_loads_and_renders(capi):
    """4 096 mesh triangles make a scene blob of about 470 KB (the blob was once capped at 200 KB): it loads and renders, the
    torus is in the frame, and the list walk gives the same frame"""
    scene = S.mesh_scene(64, 32)
    W, H = 128, 72

    def run(c):
        c.set_seeds(1, 1); c.set_image_size(W, H); c.enable_signatures(True)
        c.render(S.default_camera(), 4)
        return [c.read_argb().copy(), c.read_signatures().copy()]
    out = _run_modes(capi, scene, run, modes=(2, 0))
    _assert_same(out, "over 200 KB")
    assert len(np.unique(out[0][1])) > 10


@pytest.mark.gpu
def test_tri_bvh_65536_equals_list_walk(capi):
    """65 536 mesh triangles at 960x540, depth 4 (batch path): the hierarchy's frames, ray counts and stream position equal the list walk's"""
    scene = S.mesh_scene(256, 128, floor=S.synthetic_texture(64, 64, 3))
    W, H = 960, 540

    def run(c):
        c.set_seeds(21, 21); c.set_image_size(W, H); c.stats_reset()
        f = c.render_frames([S.default_camera()], 4).copy()
        st = c.stats()
        return [f, st["rays"], st["bounces"], c.get_seeds()]
    _assert_same(_run_modes(capi, scene, run, modes=(2, 0)), "65536")
