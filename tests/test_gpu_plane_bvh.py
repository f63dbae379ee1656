"""Hierarchies in scenes with a plane (GPU): a bounce or shadow ray that starts on the plane far outside the reach box grows the boxes it
tests (the kernels instantiated with FAR; tests/test_plane_bvh.py checks the bound on the CPU).  Under rfx_set_bvh_mode 0 and 1 every
frame, float image, hit-path signature, ray and bounce count and stream position equals the list walk's (mode 2), and bvh_spheres /
bvh_triangles show that the hierarchies are in use."""
import numpy as np
import pytest

from reflaxman_b200 import scenes as S
from reflaxman_b200 import sharding as P
from test_meshes import _adversarial, _assert_same, _n_tris, _run_modes

F = np.float32

# a camera low over the plane looking at the horizon: most of its bounces start far out on the plane
HORIZON_CAM = S.camera_lookat((0.0, 0.4, 26.0), (0.0, 0.3, -200.0), 1.2)
# under the plane, looking up through it (the plane's back face)
UNDER_CAM = S.camera_lookat((3.0, -6.0, 14.0), (0.0, 2.0, 0.0), 1.0)


@pytest.fixture(scope="module")
def capi(rfx_lib):
    from reflaxman_b200 import capi
    return capi


def _bench_scene(name):
    """the scenes of tools/bench_plane.py: mesh_scene(128, 64), mesh_scene(512, 256), synthetic_scene(32), each over a metal ground
    plane just below the floor triangles"""
    floor = S.synthetic_texture(64, 64, 3)
    if name == "mesh16k":
        return S.with_ground_plane(S.mesh_scene(128, 64, floor=floor))
    if name == "mesh256k":
        return S.with_ground_plane(S.mesh_scene(512, 256, floor=floor))
    return S.with_ground_plane(S.synthetic_scene(32, floor=floor))


def _n_spheres(scene):
    return sum(o[0] == "sphere" for o in scene["objects"])


def _tiny_and_slivers_scene():
    """36 spheres, 40 tiny ones (r 1e-4 ... 1e-2) and a 2 048-triangle torus with zero-area triangles and slivers (kappa 1e3 ... 1e7)
    over a mirror plane (reflectivity 1)"""
    rng = np.random.RandomState(5)
    scene = S.mesh_scene(32, 32, spheres=6, floor=S.synthetic_texture(64, 64, 3))
    xyz, idx = S.torus_mesh(32, 32)
    scene["objects"] += _adversarial(rng, xyz, idx, 32)
    for k, kappa in enumerate(np.logspace(3, 7, 12)):
        p0, e, f = rng.uniform(-4, 4, 3) + np.array([0.0, 4.0, 0.0]), rng.normal(size=3), rng.normal(size=3)
        e *= 3.0 / np.linalg.norm(e)
        f -= e * (f @ e) / (e @ e)
        f *= 3.0 / np.linalg.norm(f) / kappa
        v = np.concatenate([p0, p0 + e, p0 + 0.5 * e + f]).astype(F)
        scene["objects"].append(("tri", tuple(float(x) for x in v), k % 2, (0.9, 0.7, 0.6), 0.8, 0.0, -1, (0.0,) * 6))
    for k in range(40):
        c = rng.uniform([-8.0, 0.0, -6.0], [8.0, 5.0, 6.0])
        scene["objects"].append(("sphere", tuple(float(x) for x in c), float(10.0 ** rng.uniform(-4, -2)), k % 2, (0.8, 0.8, 0.9), 0.9, 0.0))
    return S.with_ground_plane(scene, refl=1.0)


def _frames_and_signatures(c, cams, depth, W, H):
    """batch frames through the wavefront pair and the single tile kernel, then the general kernel with signatures, per camera"""
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
    res += [st["rays"], st["bounces"], c.get_seeds()]
    return res


def _check_modes(out, scene, what):
    """bvh_spheres / bvh_triangles (the last two entries) > 0 under modes 0 and 1 where the scene has more than 32 of them (any under
    mode 1), 0 under mode 2; everything else identical to the list walk"""
    ns, nt = _n_spheres(scene), _n_tris(scene)
    assert out[2][-2:] == [0, 0], (what, out[2][-2:])
    assert out[1][-2:] == [ns, nt], (what, out[1][-2:], ns, nt)
    assert out[0][-2:] == [ns if ns > 32 else 0, nt if nt > 32 else 0], (what, out[0][-2:])
    assert out[0][-2] + out[0][-1] > 0
    for m in out:
        out[m] = out[m][:-2]
    _assert_same(out, what)


def _stats_tail(c):
    st = c.stats()
    return [st["bvh_spheres"], st["bvh_triangles"]]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["mesh16k", "mesh256k", "synth1024"])
def test_plane_scene_hierarchy_equals_list_walk(capi, name):
    """the benchmark scenes with a plane at 128x72, depth 8, for an orbit camera and one low over the plane looking at the horizon"""
    scene = _bench_scene(name)
    cams = [S.orbit_cameras(9)[2], HORIZON_CAM]
    out = _run_modes(capi, scene, lambda c: _frames_and_signatures(c, cams, 8, 128, 72) + _stats_tail(c))
    _check_modes(out, scene, name)


@pytest.mark.gpu
def test_plane_tiny_spheres_and_slivers_equal_list_walk(capi):
    """tiny spheres, zero-area triangles and slivers (tested after the walk in plane scenes) under a mirror plane"""
    scene = _tiny_and_slivers_scene()
    cams = [S.default_camera(), HORIZON_CAM]
    out = _run_modes(capi, scene, lambda c: _frames_and_signatures(c, cams, 8, 120, 68) + _stats_tail(c))
    _check_modes(out, scene, "tiny and slivers")


@pytest.mark.gpu
def test_plane_every_render_mode_equals_list_walk(capi):
    """2x2 SSAA, 3 additive passes, ragged render_next slices, block preview, a 2-way render_strips split, rfx_trace_rays from origins
    on the plane 1e2 ... 1e5 units out (re-flatten) and a camera under the plane looking up: identical to the list walk"""
    scene = _tiny_and_slivers_scene()
    W, H, depth = 96, 60, 6
    cam = S.orbit_cameras(9)[5]

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
        gather = c.buffer_alloc(W * H * 4)
        for rank in range(2):
            P.split_frame(c, cam, depth, 1, 2, rank, gather, strip_rows=8)
            c.synchronize()
        res.append(c.buffer_read(gather, np.zeros((H, W), np.uint32)).copy())
        c.buffer_free(gather)
        c.render(UNDER_CAM, depth)
        res.append(c.read_rgbf().copy())
        rng = np.random.RandomState(3)
        n = 600
        u = rng.normal(size=(n, 2))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        dist = 10.0 ** rng.uniform(2, 5, n)
        o = np.stack([u[:, 0] * dist, np.full(n, -0.05), u[:, 1] * dist], 1).astype(F)
        target = rng.uniform([-10.0, 0.0, -8.0], [10.0, 6.0, 8.0], (n, 3))
        r = (target - o).astype(F)
        r[::3, 1] = np.abs(r[::3, 1]) * F(1e-3)                 # grazing along the plane
        res.append(c.trace_rays(o, r, depth).copy())
        st = c.stats()
        res += [st["rays"], st["bounces"], c.get_seeds()] + _stats_tail(c)
        return res
    _check_modes(_run_modes(capi, scene, run), scene, "render modes")


@pytest.mark.gpu
def test_plane_scene_matches_oracle(capi, oracle):
    """a plane scene with 36 spheres and 2 048 + 16 triangles (both hierarchies and the FAR kernels under mode 0) at 128x72, depth 8:
    hit-path signatures equal the oracle's on every pixel, and the frame meets the parity bar"""
    import cases
    scene = S.mesh_scene(32, 32, spheres=6, floor=S.synthetic_texture(64, 64, 3))
    xyz, idx = S.torus_mesh(32, 32)
    scene["objects"] += _adversarial(np.random.RandomState(9), xyz, idx, 16)
    scene = S.with_ground_plane(scene, refl=0.8)
    W, H, depth = 128, 72, 8
    cam = HORIZON_CAM
    c = capi.Context(0)
    try:
        c.load_scene(scene); c.set_seeds(321, 321); c.set_image_size(W, H); c.enable_signatures(True); c.stats_reset()
        c.render(cam, depth)
        argb, sig, st = c.read_argb(), c.read_signatures(), c.stats()
        assert st["bvh_spheres"] == _n_spheres(scene) > 32 and st["bvh_triangles"] == _n_tris(scene) > 32, st
    finally:
        c.close()
    o = oracle.OracleRender(S.expand_meshes(scene), W, H, seed=321).render(cam, depth, want_sig=True)
    assert np.array_equal(sig, o.sig), "hit-path signatures differ on %d pixels" % int((sig != o.sig).sum())
    assert st["rays"] == o.counters["rays"]
    cases.assert_parity(argb, o.resolve()[1], "plane scene")
