"""rfx_update_mesh: a mesh's vertices replaced in place.

Every case animates one context through rfx_update_mesh and renders the same frames, in the same order and from the same seeds, in a
reference context that loads the scene anew with the deformed vertices (rfx_add_mesh(new xyz), a host flatten) before each frame.
Everything must agree bit for bit: float images as uint32, ARGB, signatures, ray and bounce counts and the stream position after.
Each update's return value states which path served it (1: set up and refitted on the device, 0: host re-flatten at the next render),
and each case checks it is the path it means to test.

CPU: the deformation of scenes.py keeps the torus's vertex count and index list."""
import numpy as np
import pytest

from reflaxman_b200 import scenes as S
from reflaxman_b200 import sharding as P

F = np.float32


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------

def test_torus_wave_keeps_the_mesh_topology():
    """torus_wave gives the vertex count and order of torus_mesh (its index list applies), moves the vertices when the amplitude is
    nonzero, and is torus_mesh bit for bit at amplitude 0"""
    xyz, idx = S.torus_mesh(32, 16)
    w = S.torus_wave(32, 16, phase=0.7, amplitude=0.3)
    assert w.shape == xyz.shape and w.dtype == np.float32 and int(idx.max()) < len(w)
    assert not np.array_equal(w, xyz)
    assert np.array_equal(S.torus_wave(32, 16, phase=0.7, amplitude=0.0).view(np.uint32), xyz.view(np.uint32))


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu(rfx_lib):
    import torch
    from reflaxman_b200 import capi
    return capi, torch


def _case(n_u, n_v, xyz, spheres=0, plane=False, adversarial=64):
    """mesh_scene(n_u, n_v) with the torus's vertices replaced by xyz, plus the adversarial triangles of test_meshes (zero-area,
    slivers, exact copies) around the undeformed torus"""
    import test_meshes as T
    scene = S.mesh_scene(n_u, n_v, spheres=spheres, floor=S.synthetic_texture(64, 64, 3), skybox=S.synthetic_texture(128, 96, 5))
    scene["objects"] = [("mesh", np.asarray(xyz, F)) + tuple(o[2:]) if o[0] == "mesh" else o for o in scene["objects"]]
    x0, idx = S.torus_mesh(n_u, n_v)
    scene["objects"] += T._adversarial(np.random.RandomState(n_u * 7 + n_v), x0, idx, adversarial)
    return S.with_ground_plane(scene) if plane else scene


def _frame(torch, c, cam, depth, stream):
    """one rfx_render_frames_device frame into a torch buffer on ``stream``; ARGB [H, W]"""
    buf = torch.empty(c.H * c.W, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    c.render_frames_device([cam], depth, 1, buf.data_ptr(), stream.cuda_stream)
    torch.cuda.synchronize()
    return buf.cpu().numpy().view(np.uint32).reshape(c.H, c.W).copy()


class _Pair:
    """the animated context and its reference, set up alike, each with one depth-1 frame rendered (the first flatten: a device update
    needs a flattened scene)"""

    def __init__(self, capi, scene, mode, W, H, seeds=(77, 77), setup=None):
        self.capi, self.setup = capi, setup
        self.anim, self.ref = capi.Context(0), capi.Context(0)
        self.first = None
        for c in (self.anim, self.ref):
            firsts = c.load_scene(scene)
            self.first = firsts[0]
            c.set_bvh_mode(mode); c.set_seeds(*seeds); c.set_image_size(W, H)
            if setup:
                setup(c, self.first)
            c.render(S.default_camera(), 1)

    def update(self, scene_of_xyz, xyz):
        """update the animated context, reload the reference; returns the update's path"""
        r = self.anim.update_mesh(self.first, xyz)
        assert self.ref.load_scene(scene_of_xyz(xyz)) == [self.first]
        if self.setup:
            self.setup(self.ref, self.first)
        return r

    def both(self, fn):
        return fn(self.anim), fn(self.ref)

    def tail(self):
        out = []
        for c in (self.anim, self.ref):
            st = c.stats()
            out.append([st["rays"], st["bounces"], c.get_seeds()])
        return out

    def close(self):
        self.anim.close(); self.ref.close()


def _same(a, b, what):
    assert len(a) == len(b), what
    for k, (x, y) in enumerate(zip(a, b)):
        if isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and np.array_equal(x.view(np.uint32) if x.dtype == np.float32 else x,
                                                         y.view(np.uint32) if y.dtype == np.float32 else y), (what, k)
        else:
            assert x == y, (what, k, x, y)


ORBIT = S.orbit_cameras(9)[2]


@pytest.mark.gpu
@pytest.mark.parametrize("n_u,n_v", [(32, 32), (128, 64)], ids=["2048", "16384"])
def test_animation_on_the_device_equals_fresh_scenes(gpu, n_u, n_v):
    """8 wave steps, each update_mesh (device path) then frames on a torch stream: the wavefront pair, the single tile kernel and the
    general kernel with signatures, under bvh modes 0, 1 and 2, equal the reference's (which reloads the deformed scene) every step"""
    capi, torch = gpu
    W, H, depth = 160, 90, 8
    stream = torch.cuda.Stream()
    scene_of = lambda xyz: _case(n_u, n_v, xyz)
    for mode in (0, 1, 2):
        pr = _Pair(capi, scene_of(S.torus_mesh(n_u, n_v)[0]), mode, W, H)
        try:
            pr.anim.enable_signatures(True); pr.ref.enable_signatures(True)
            for step in range(8):
                xyz = S.torus_wave(n_u, n_v, phase=0.8 * step, amplitude=0.3)
                assert pr.update(scene_of, xyz), (mode, step)
                for path, wave in ((2, 2), (2, 0)):
                    a, b = pr.both(lambda c: (c.force_path(path), c.set_option("blob_wavefront", wave), _frame(torch, c, ORBIT if step % 2 else S.default_camera(), depth, stream))[2])
                    _same([a], [b], (mode, step, wave))
                a, b = pr.both(lambda c: (c.force_path(3), c.render(S.default_camera(), depth), [c.read_rgbf().copy(), c.read_argb().copy(), c.read_signatures().copy()])[2])
                _same(a, b, (mode, step, "general"))
            a, b = pr.tail()
            _same(a, b, (mode, "counts"))
            assert (pr.anim.stats()["bvh_triangles"] > 0) == (mode != 2)
        finally:
            pr.close()


@pytest.mark.gpu
def test_every_refitted_triangle_is_reachable(gpu):
    """after a large deformation on the device, rays from inside the reach box aimed at every mesh triangle's centroid (depth 1 and 4)
    give the reference's colours under the list walk: every refitted leaf, seen by the camera or not"""
    capi, torch = gpu
    n_u, n_v = 32, 32
    _, idx = S.torus_mesh(n_u, n_v)
    scene_of = lambda xyz: _case(n_u, n_v, xyz)
    anim = capi.Context(0)
    ref = capi.Context(0)
    try:
        rng = np.random.RandomState(5)
        o = rng.uniform([-6, 0.5, -6], [6, 6, 6], (2 * n_u * n_v, 3)).astype(F)
        first = anim.load_scene(scene_of(S.torus_mesh(n_u, n_v)[0]))[0]
        ref.load_scene(scene_of(S.torus_mesh(n_u, n_v)[0]))
        anim.set_bvh_mode(1); anim.set_seeds(3, 3)
        ref.set_bvh_mode(2); ref.set_seeds(3, 3)
        d0 = (F([0.0, 2.6, 0.0]) - o).astype(F)
        _same([anim.trace_rays(o, d0, 2)], [ref.trace_rays(o, d0, 2)], "before")   # (also the first flatten)
        xyz = S.torus_wave(n_u, n_v, phase=1.3, amplitude=0.7, waves=5)
        assert anim.update_mesh(first, xyz)
        ref.load_scene(scene_of(xyz))
        cen = xyz.astype(np.float64)[idx.astype(np.int64)].mean(1)
        d = (cen - o).astype(F)
        for depth in (1, 4):
            _same([anim.trace_rays(o, d, depth)], [ref.trace_rays(o, d, depth)], depth)
        assert anim.stats()["bvh_triangles"] > 0
        assert anim.get_seeds() == ref.get_seeds()
    finally:
        anim.close(); ref.close()


@pytest.mark.gpu
def test_spheres_and_mesh_then_leaving_the_grid_and_reach_boxes(gpu):
    """1024 spheres (sphere hierarchy, light grid, eye grid) and a torus: wave updates take the device path and leave the sphere
    structures valid; a torus lifted out of the light grid's box, then out of the reach box, takes the host path; every frame equals
    the reference's"""
    capi, torch = gpu
    n_u, n_v = 32, 32
    W, H, depth = 192, 108, 6
    stream = torch.cuda.Stream()
    scene_of = lambda xyz: _case(n_u, n_v, xyz, spheres=32, adversarial=16)
    x0 = S.torus_mesh(n_u, n_v)[0]
    pr = _Pair(capi, scene_of(x0), 0, W, H, seeds=(11, 11))
    try:
        steps = [(S.torus_wave(n_u, n_v, phase=0.9 * k, amplitude=0.25), True) for k in range(3)]
        steps += [(x0 + F([0, 3.0, 0]), False), (x0 + F([0, 5.0, 0]), False), (x0, True)]
        for k, (xyz, device) in enumerate(steps):
            assert pr.update(scene_of, xyz) == device, k
            a, b = pr.both(lambda c: [_frame(torch, c, cam, depth, stream) for cam in (S.default_camera(), ORBIT)])
            _same(a, b, k)
        a, b = pr.tail()
        _same(a, b, "counts")
        st = pr.anim.stats()
        assert st["light_grids"] > 0 and st["bvh_spheres"] > 0 and st["bvh_triangles"] > 0
    finally:
        pr.close()


@pytest.mark.gpu
def test_plane_scene_slivers_leave_and_rejoin(gpu):
    """over a ground plane (boxes grow for far origins): a deformation that collapses part of the torus into slivers and zero-area
    triangles takes the device path (slivers join the triangles tested after the walk), then the undeformed torus again; frames equal
    the reference's under the hierarchy and under the list walk"""
    capi, torch = gpu
    n_u, n_v = 32, 32
    W, H, depth = 160, 90, 8
    stream = torch.cuda.Stream()
    x0, idx = S.torus_mesh(n_u, n_v)
    scene_of = lambda xyz: _case(n_u, n_v, xyz, plane=True, adversarial=16)
    bad = x0.copy().reshape(n_u, n_v, 3)
    a0, b0 = bad[4, 0].astype(np.float64), bad[12, n_v // 2].astype(np.float64)
    nrm = np.cross(b0 - a0, [0.0, 1.0, 0.0]); nrm /= np.linalg.norm(nrm)
    for i in range(5, 12):        # rows 5..11 onto one segment, a hair apart: slivers, some exactly degenerate
        for j in range(n_v):
            bad[i, j] = a0 + (b0 - a0) * (j / n_v) + 1e-7 * (i - 5) * nrm
    bad[13] = bad[13, 0]          # one row collapsed to a point: zero-area triangles
    bad = bad.reshape(-1, 3).astype(F)
    # the deformation does make triangles that no box holds from far origins
    import test_meshes as T
    v0, ax = T._construct(bad[idx.astype(np.int64)].reshape(-1, 9))
    _, tb, _, _, _ = capi.far_bounds_host(np.zeros((0, 4), F), np.concatenate([v0, ax], 1), np.array([-20, -1, -20, 20, 10, 20], F))
    assert np.isinf(tb[:, 0]).sum() > 10
    pr = _Pair(capi, scene_of(x0), 1, W, H, seeds=(9, 9))
    walk = capi.Context(0)
    try:
        walk.load_scene(scene_of(x0)); walk.set_bvh_mode(2); walk.set_seeds(9, 9); walk.set_image_size(W, H)
        walk.render(S.default_camera(), 1)
        for k, xyz in enumerate((bad, x0, bad)):
            assert pr.update(scene_of, xyz), k
            walk.load_scene(scene_of(xyz))
            cams = (S.default_camera(), ORBIT)
            a, b = pr.both(lambda c: [_frame(torch, c, cam, depth, stream) for cam in cams])
            _same(a, b, k)
            _same(a, [_frame(torch, walk, cam, depth, stream) for cam in cams], (k, "walk"))
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close(); walk.close()


@pytest.mark.gpu
def test_textures_of_mesh_triangles_survive_updates(gpu):
    """mesh triangles with rfx_set_triangle_texture keep their textures through device updates"""
    capi, torch = gpu
    n_u, n_v = 32, 32
    W, H, depth = 160, 90, 6
    stream = torch.cuda.Stream()
    scene_of = lambda xyz: _case(n_u, n_v, xyz, adversarial=0)
    uv = np.array([0, 0, 1, 0, 0, 1], F)

    def texture(c, first):
        for k in range(0, 2 * n_u * n_v, 7):
            c._ck(c.L.rfx_set_triangle_texture(c.h, first + k, 0, uv.ctypes.data_as(capi._fp)), "texture")
    pr = _Pair(capi, scene_of(S.torus_mesh(n_u, n_v)[0]), 0, W, H, setup=texture)
    try:
        for step in range(3):
            assert pr.update(scene_of, S.torus_wave(n_u, n_v, phase=1.1 * step, amplitude=0.2)), step
            a, b = pr.both(lambda c: _frame(torch, c, S.default_camera(), depth, stream))
            _same([a], [b], step)
    finally:
        pr.close()


@pytest.mark.gpu
def test_host_reflatten_after_device_updates_sees_the_new_vertices(gpu):
    """device updates, then a camera outside the reach box: the host re-flattens from its own records, which must hold the updated
    vertices; a device update after that re-flatten is served on the device again"""
    capi, torch = gpu
    n_u, n_v = 32, 32
    W, H, depth = 160, 90, 6
    stream = torch.cuda.Stream()
    far = S.camera_lookat((38.0, 17.0, -30.0), (0.0, 2.0, 0.0), 0.6)
    scene_of = lambda xyz: _case(n_u, n_v, xyz)
    pr = _Pair(capi, scene_of(S.torus_mesh(n_u, n_v)[0]), 0, W, H)
    try:
        for step, cam in enumerate((S.default_camera(), S.default_camera(), far, far)):
            assert pr.update(scene_of, S.torus_wave(n_u, n_v, phase=0.6 * step, amplitude=0.3)), step
            if step < 2:
                continue
            a, b = pr.both(lambda c: _frame(torch, c, cam, depth, stream))
            _same([a], [b], step)
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()


@pytest.mark.gpu
def test_render_api_modes_after_a_device_update(gpu):
    """after a device update: 2x2 SSAA, 3 additive passes, ragged render_next slices, block preview and a 2-way render_strips split
    equal the reference's"""
    capi, torch = gpu
    n_u, n_v = 32, 32
    W, H, depth = 96, 60, 6
    scene_of = lambda xyz: _case(n_u, n_v, xyz)
    pr = _Pair(capi, scene_of(S.torus_mesh(n_u, n_v)[0]), 0, W, H, seeds=(5, 9))
    try:
        assert pr.update(scene_of, S.torus_wave(n_u, n_v, phase=2.0, amplitude=0.35))

        def run(c):
            res = []
            c.force_path(2)
            c.render(ORBIT, depth, samples=2)
            res += [c.read_rgbf().copy(), c.read_argb().copy()]
            for _ in range(3):
                c.render(ORBIT, depth, additive=True)
            res.append(c.read_rgbf().copy())
            c.render(ORBIT, depth, chunk=1013)
            res.append(c.read_rgbf().copy())
            c.render(ORBIT, depth, samples=-3)
            res.append(c.read_argb().copy())
            gather = c.buffer_alloc(W * H * 4)
            for rank in range(2):
                P.split_frame(c, ORBIT, depth, 1, 2, rank, gather, strip_rows=8)
                c.synchronize()
            res.append(c.buffer_read(gather, np.zeros((H, W), np.uint32)).copy())
            c.buffer_free(gather)
            st = c.stats()
            return res + [st["rays"], st["bounces"], c.get_seeds()]
        a, b = pr.both(run)
        _same(a, b, "render modes")
    finally:
        pr.close()


def _small_scene(xyz):
    """the demo scene's spheres and light with an 8-triangle mesh instead of the floor: it fits the constant bank"""
    base = S.default_scene()
    _, idx = S.torus_mesh(2, 2)
    objs = [o for o in base["objects"] if o[0] == "sphere"] + [("mesh", np.asarray(xyz, F), idx, S.MT_METAL, (0.9, 0.8, 0.5), 0.8, 0.0)]
    return dict(base, objects=objs)


@pytest.mark.gpu
def test_constant_bank_scene_takes_the_host_path(gpu):
    """an 8-triangle mesh in a scene that fits the constant bank: updates return 0 and the frames are the reference's"""
    capi, torch = gpu
    W, H, depth = 128, 72, 8
    stream = torch.cuda.Stream()
    pr = _Pair(capi, _small_scene(S.torus_mesh(2, 2)[0]), 0, W, H)
    try:
        for step in range(3):
            assert pr.update(_small_scene, S.torus_wave(2, 2, phase=0.7 * step, amplitude=0.4)) is False, step
            a, b = pr.both(lambda c: _frame(torch, c, S.default_camera(), depth, stream))
            _same([a], [b], step)
        assert pr.anim.stats()["launches_small_fast"] + pr.anim.stats()["launches_small_any"] > 0
    finally:
        pr.close()


@pytest.mark.gpu
def test_bad_updates_are_rejected_and_change_nothing(gpu):
    """NULL xyz, a first that does not start a mesh, and a mesh index from before rfx_scene_reset are RFX_ERR_ARG; the frames around
    them are those of a context that never made the calls"""
    capi, torch = gpu
    n_u, n_v = 16, 16
    W, H, depth = 96, 54, 6
    stream = torch.cuda.Stream()
    x0 = S.torus_mesh(n_u, n_v)[0]
    scene = _case(n_u, n_v, x0, adversarial=0)
    anim, ref = capi.Context(0), capi.Context(0)
    try:
        frames = []
        for c, bad in ((anim, True), (ref, False)):
            first = c.load_scene(scene)[0]
            c.set_seeds(2, 2); c.set_image_size(W, H)
            out = [_frame(torch, c, S.default_camera(), depth, stream)]
            if bad:
                assert c.L.rfx_update_mesh(c.h, first, None) == -1
                assert c.L.rfx_update_mesh(c.h, first + 1, x0.ctypes.data_as(capi._fp)) == -1
                with pytest.raises(capi.RfxError):
                    c.update_mesh(first + 3, x0)
            out.append(_frame(torch, c, S.default_camera(), depth, stream))
            c.load_scene(S.default_scene())   # rfx_scene_reset: the mesh is gone, object `first` is now a sphere
            if bad:
                assert c.L.rfx_update_mesh(c.h, first, x0.ctypes.data_as(capi._fp)) == -1
            out.append(_frame(torch, c, S.default_camera(), depth, stream))
            st = c.stats()
            frames.append(out + [st["rays"], c.get_seeds()])
        _same(frames[0], frames[1], "errors")
    finally:
        anim.close(); ref.close()
