"""rfx_update_spheres: spheres moved and resized in place.

Every case animates one context through rfx_update_spheres and renders the same frames, in the same order and from the same seeds, in a
reference context that loads the scene anew with the moved spheres (rfx_add_sphere(new centre, new radius), a host flatten) before each
frame.  Everything must agree bit for bit: float images as uint32, ARGB, signatures, ray and bounce counts and the stream position after.
Each update's return value states which path served it (1: records written and the sphere hierarchy refitted on the device, 0: host
re-flatten at the next render), and each case checks it is the path it means to test.

CPU: object_indices, sphere_bounce and with_spheres of scenes.py."""
import numpy as np
import pytest

from reflaxman_b200 import scenes as S
from reflaxman_b200 import sharding as P

F = np.float32


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------

def test_object_indices_count_mesh_triangles():
    sc = S.mesh_scene(4, 4, spheres=2)
    # 4 spheres, the floor and wall (4 triangles), then the torus (32 triangles) as one entry
    assert S.object_indices(sc) == list(range(9))
    sc["objects"].append(("sphere", (0.0, 1.0, 0.0), 0.5, 0, (1.0, 1.0, 1.0), 0.5, 0.0))
    assert S.object_indices(sc)[-1] == 8 + 32
    assert S.object_indices(S.synthetic_scene(6))[:3] == [0, 1, 2]


def test_sphere_bounce_is_the_loaded_scene_at_rest_and_stays_in_the_boxes():
    sc = S.synthetic_scene(16)
    obj, sp = S.sphere_bounce(sc, 0.0)
    assert obj.dtype == np.int32 and sp.dtype == np.float32 and sp.shape == (256, 4)
    assert list(obj) == list(range(256))
    loaded = np.array([list(o[1]) + [o[2]] for o in sc["objects"] if o[0] == "sphere"], F)
    assert np.array_equal(sp.view(np.uint32), loaded.view(np.uint32))
    lo_y = loaded[:, 1]
    for t in (0.3, 1.1, 2.9):
        _, m = S.sphere_bounce(sc, t, height=4.0, pulse=0.3)
        assert not np.array_equal(m, sp)
        assert np.array_equal(m[:, [0, 2]], sp[:, [0, 2]])
        assert np.all(m[:, 1] >= lo_y) and np.all(m[:, 1] + m[:, 3] < 8.0)          # under the back wall's top
        assert np.all(m[:, 1] - m[:, 3] >= lo_y - sp[:, 3] - 1e-6)                   # ... and not below the floor
        assert np.all(m[:, 3] > 0) and np.all(np.abs(m[:, 3] / sp[:, 3] - 1) <= 0.3 + 1e-6)
    # each sphere has its own phase
    _, m = S.sphere_bounce(sc, 0.5)
    assert len(np.unique(m[:, 1] - lo_y)) > 200


def test_with_spheres_replaces_exactly_the_given_spheres():
    sc = S.mesh_scene(4, 4, spheres=2)
    obj = np.array([1, 3, 1], np.int32)
    sp = np.array([[1, 2, 3, 0.5], [4, 5, 6, 0.25], [7, 8, 9, 0.75]], F)
    new = S.with_spheres(sc, obj, sp)
    assert new["objects"][1][:3] == ("sphere", (7.0, 8.0, 9.0), 0.75)      # the later row wins
    assert new["objects"][3][:3] == ("sphere", (4.0, 5.0, 6.0), 0.25)
    assert new["objects"][1][3:] == sc["objects"][1][3:]
    for k in (0, 2, 4, 5, 6, 7, 8):
        assert new["objects"][k] is sc["objects"][k]
    with pytest.raises(ValueError):
        S.with_spheres(sc, [4], sp[:1])
    # at rest, sphere_bounce describes the loaded scene
    o, s0 = S.sphere_bounce(sc, 0.0)
    assert S.with_spheres(sc, o, s0)["objects"] == [tuple(x) if x[0] != "sphere" else
                                                    ("sphere", tuple(float(F(v)) for v in x[1]), float(F(x[2]))) + tuple(x[3:])
                                                    for x in sc["objects"]]


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu(rfx_lib):
    import torch
    from reflaxman_b200 import capi
    return capi, torch


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

    def __init__(self, capi, scene, mode, W, H, seeds=(77, 77)):
        self.scene = scene
        self.anim, self.ref = capi.Context(0), capi.Context(0)
        for c in (self.anim, self.ref):
            c.load_scene(scene)
            c.set_bvh_mode(mode); c.set_seeds(*seeds); c.set_image_size(W, H)
            c.render(S.default_camera(), 1)

    def update(self, objects, spheres):
        """update the animated context, reload the reference with the moved spheres; returns the update's path"""
        r = self.anim.update_spheres(objects, spheres)
        self.scene = S.with_spheres(self.scene, objects, spheres)
        self.ref.load_scene(self.scene)
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


def _frames(torch, pr, stream, depth, cams=(None, ORBIT)):
    a, b = pr.both(lambda c: [_frame(torch, c, cam or S.default_camera(), depth, stream) for cam in cams])
    return a, b


@pytest.mark.gpu
@pytest.mark.parametrize("n_side", [6, 16])
def test_bounces_on_the_device_equal_fresh_scenes(gpu, n_side):
    """8 bounce steps, each update_spheres (device path) then frames on a torch stream: the wavefront pair, the single tile kernel and
    the general kernel with signatures, on the default and an orbit camera, under bvh modes 0, 1 and 2, equal the reference's"""
    capi, torch = gpu
    W, H, depth = 160, 90, 8
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(n_side, floor=S.synthetic_texture(64, 64, 3), skybox=S.synthetic_texture(128, 96, 5))
    for mode in (0, 1, 2):
        pr = _Pair(capi, scene, mode, W, H)
        try:
            pr.anim.enable_signatures(True); pr.ref.enable_signatures(True)
            for step in range(8):
                assert pr.update(*S.sphere_bounce(scene, 0.45 * (step + 1), height=2.0, pulse=0.2 if step % 2 else 0.0)), (mode, step)
                for cam in (S.default_camera(), ORBIT):
                    for path, wave in ((2, 2), (2, 0)):
                        a, b = pr.both(lambda c: (c.force_path(path), c.set_option("blob_wavefront", wave), _frame(torch, c, cam, depth, stream))[2])
                        _same([a], [b], (mode, step, wave))
                    a, b = pr.both(lambda c: (c.force_path(3), c.render(cam, depth), [c.read_rgbf().copy(), c.read_argb().copy(), c.read_signatures().copy()])[2])
                    _same(a, b, (mode, step, "general"))
            a, b = pr.tail()
            _same(a, b, (mode, "counts"))
            st = pr.anim.stats()
            assert (st["bvh_spheres"] > 0) == (mode != 2)
            assert (st["light_grids"] > 0) == (mode != 2)
        finally:
            pr.close()


@pytest.mark.gpu
def test_radius_changes_overlaps_and_duplicates_keep_the_tie_break(gpu):
    """spheres grow, shrink and pass through each other; some become exact copies of another sphere: the closest-hit ties still go to
    the earlier object, as in the reference"""
    capi, torch = gpu
    W, H, depth = 160, 90, 8
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(8)
    pr = _Pair(capi, scene, 0, W, H, seeds=(3, 5))
    try:
        obj, sp = S.sphere_bounce(scene, 0.0)
        for step in range(5):
            new = sp.copy()
            new[:, 3] *= F(1.0 + 0.8 * np.sin(0.9 * step + np.arange(len(sp))))            # grow and shrink
            new[:, 1] = new[:, 3] + F(0.05 * step)                                           # (above the floor)
            new[1::2, 0] = sp[0::2, 0] + F(0.1 * step)                                       # odd spheres slide into their neighbours
            new[10:20] = new[40:50]                                                          # exact duplicates of later spheres
            new[50:55] = new[5:10]                                                           # ... and of earlier ones
            assert pr.update(obj, new), step
            a, b = _frames(torch, pr, stream, depth)
            _same(a, b, step)
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()


@pytest.mark.gpu
def test_every_refitted_sphere_is_reachable(gpu):
    """after a large move on the device, rays from random origins inside the reach box aimed at every sphere centre (depth 1 and 4)
    give the colours of a reference under the list walk: every refitted leaf, seen by the camera or not"""
    capi, torch = gpu
    scene = S.synthetic_scene(16)
    anim, ref = capi.Context(0), capi.Context(0)
    try:
        anim.load_scene(scene); anim.set_bvh_mode(1); anim.set_seeds(3, 3)
        ref.load_scene(scene); ref.set_bvh_mode(2); ref.set_seeds(3, 3)
        rng = np.random.RandomState(5)
        obj, sp = S.sphere_bounce(scene, 0.0)
        o = rng.uniform([-12, 0.5, -8], [12, 6, 8], (len(sp), 3)).astype(F)
        d0 = (sp[:, :3] - o).astype(F)
        _same([anim.trace_rays(o, d0, 2)], [ref.trace_rays(o, d0, 2)], "before")   # (also the first flatten)
        new = sp.copy()
        perm = rng.permutation(len(sp))
        new[:, 0] = sp[perm, 0]; new[:, 2] = sp[perm, 2]                           # every sphere somewhere else
        new[:, 3] = sp[:, 3] * rng.uniform(0.5, 1.5, len(sp)).astype(F)
        new[:, 1] = new[:, 3] + F(3.0) * rng.uniform(0, 1, len(sp)).astype(F)      # (above the floor: inside the light grid's box)
        assert anim.update_spheres(obj, new)
        ref.load_scene(S.with_spheres(scene, obj, new))
        d = (new[:, :3] - o).astype(F)
        for depth in (1, 4):
            _same([anim.trace_rays(o, d, depth)], [ref.trace_rays(o, d, depth)], depth)
        assert anim.stats()["bvh_spheres"] > 0 and ref.stats()["bvh_spheres"] == 0
        assert anim.get_seeds() == ref.get_seeds()
    finally:
        anim.close(); ref.close()


@pytest.mark.gpu
def test_crowding_into_one_light_grid_cell_and_back(gpu):
    """every sphere clustered into one spot (one light-grid cell's shadow: the item arrays grow past their allocation), then spread out
    again: the light grids are rebuilt on each update and the frames equal the reference's"""
    capi, torch = gpu
    W, H, depth = 160, 90, 6
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(16)
    pr = _Pair(capi, scene, 0, W, H, seeds=(21, 8))
    try:
        obj, sp = S.sphere_bounce(scene, 0.0)
        rng = np.random.RandomState(1)
        crowd = sp.copy()
        crowd[:, :3] = (F([1.0, 4.0, 0.5]) + rng.uniform(-0.4, 0.4, (len(sp), 3))).astype(F)
        crowd[:, 3] = F(0.05)
        crowd[::16, 3] = F(3.5)              # big spheres among many small ones: small cells, each big one in hundreds of them
        # the crowd's grid has many more items than the spread scene's: the device arrays (1/8 headroom) grow
        light = scene["lights"][0]
        items = lambda s: len(capi.light_grid_host(tuple(light[0]) + (light[1],), s, [-14, 0, -10, 14, 8, 10], 40.0)[4])
        assert items(crowd) > 1.5 * items(sp)
        for k, s in enumerate((crowd, sp, crowd, S.sphere_bounce(scene, 1.0, height=3.0)[1])):
            assert pr.update(obj, s), k
            a, b = _frames(torch, pr, stream, depth)
            _same(a, b, k)
        a, b = pr.tail()
        _same(a, b, "counts")
        assert pr.anim.stats()["light_grids"] > 0
    finally:
        pr.close()


@pytest.mark.gpu
def test_host_path_cases(gpu):
    """a sphere lifted out of the light grid's box, then one moved out of the reach box, return 0 (host re-flatten); the next update
    after the re-flatten returns 1 again; an update before the first render and one in a constant-bank scene return 0; every frame
    equals the reference's"""
    capi, torch = gpu
    W, H, depth = 160, 90, 6
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(16)
    pr = _Pair(capi, scene, 0, W, H, seeds=(4, 4))
    try:
        obj, sp = S.sphere_bounce(scene, 0.0)
        one = np.array([7], np.int32)
        r = sp[7, 3]
        top = sp[7:8].copy(); top[0, 1] = F(8.4) - r     # its top at y = 8.4: above the wall (the light grid's box ends near 8.03), inside
                                                          # the reach box (padded by a tenth of its height: up to 8.8)
        steps = [(sp[7:8] + F([0, 1.0, 0, 0]), 1),
                 (top, 0),
                 (sp[7:8] + F([0, 2.0, 0, 0]), 1),       # after the re-flatten
                 (sp[7:8] + F([0, 60.0, 0, 0]), 0),      # out of the reach box
                 (sp[7:8], 1)]
        for k, (s, device) in enumerate(steps):
            assert pr.update(one, s) == device, k
            a, b = _frames(torch, pr, stream, depth)
            _same(a, b, k)
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()
    # before the first render: a re-flatten is pending anyway
    c = capi.Context(0)
    try:
        c.load_scene(scene)
        assert c.update_spheres(obj[:3], sp[:3] + F([0, 0.5, 0, 0])) is False
    finally:
        c.close()
    # the constant bank
    small = S.default_scene()
    pr = _Pair(capi, small, 0, W, H)
    try:
        for step in range(2):
            o, s = S.sphere_bounce(small, 0.7 * (step + 1), height=0.5, pulse=0.2)
            assert pr.update(o, s) is False, step
            a, b = _frames(torch, pr, stream, depth)
            _same(a, b, ("small", step))
        assert pr.anim.stats()["launches_small_fast"] + pr.anim.stats()["launches_small_any"] > 0
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [1, 2])
def test_plane_scene(gpu, mode):
    """over a ground plane (FAR kernels: boxes grow for far origins, no light grid, the eye grid under a hierarchy): bounces on the
    device equal the reference's"""
    capi, torch = gpu
    W, H, depth = 160, 90, 8
    stream = torch.cuda.Stream()
    scene = S.with_ground_plane(S.synthetic_scene(16))
    pr = _Pair(capi, scene, mode, W, H, seeds=(9, 9))
    try:
        for step in range(4):
            assert pr.update(*S.sphere_bounce(scene, 0.6 * (step + 1), height=2.5, pulse=0.25)), step
            a, b = _frames(torch, pr, stream, depth)
            _same(a, b, step)
        a, b = pr.tail()
        _same(a, b, "counts")
        st = pr.anim.stats()
        assert (st["bvh_spheres"] > 0) == (mode == 1) and st["light_grids"] == 0
    finally:
        pr.close()


@pytest.mark.gpu
def test_render_api_modes_after_a_device_update(gpu):
    """after a device update: 2x2 SSAA, 3 additive passes, ragged render_next slices, block preview, a 2-way render_strips split and
    rfx_render_frames to host memory equal the reference's"""
    capi, torch = gpu
    W, H, depth = 96, 60, 6
    scene = S.synthetic_scene(16)
    pr = _Pair(capi, scene, 0, W, H, seeds=(5, 9))
    try:
        assert pr.update(*S.sphere_bounce(scene, 1.7, height=2.0, pulse=0.3))

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
            res.append(np.asarray(c.render_frames([S.default_camera(), ORBIT], depth)).copy())
            st = c.stats()
            return res + [st["rays"], st["bounces"], c.get_seeds()]
        a, b = pr.both(run)
        _same(a, b, "render modes")
    finally:
        pr.close()


@pytest.mark.gpu
def test_spheres_and_mesh_updates_alternate(gpu):
    """mesh_scene(32, 32, spheres=8): rfx_update_spheres and rfx_update_mesh alternate, each on the device; every frame equals the
    reference's"""
    capi, torch = gpu
    n_u, n_v = 32, 32
    W, H, depth = 160, 90, 6
    stream = torch.cuda.Stream()
    scene = S.mesh_scene(n_u, n_v, spheres=8)
    pr = _Pair(capi, scene, 0, W, H, seeds=(13, 2))
    first = S.object_indices(scene)[[o[0] for o in scene["objects"]].index("mesh")]
    try:
        for step in range(6):
            if step % 2 == 0:
                assert pr.update(*S.sphere_bounce(scene, 0.5 * (step + 1), height=1.5, pulse=0.2)), step
            else:
                xyz = S.torus_wave(n_u, n_v, phase=0.7 * step, amplitude=0.2)
                assert pr.anim.update_mesh(first, xyz), step
                pr.scene = dict(pr.scene, objects=[("mesh", xyz) + tuple(o[2:]) if o[0] == "mesh" else o for o in pr.scene["objects"]])
                pr.ref.load_scene(pr.scene)
            a, b = _frames(torch, pr, stream, depth)
            _same(a, b, step)
        a, b = pr.tail()
        _same(a, b, "counts")
        st = pr.anim.stats()
        assert st["bvh_spheres"] > 0 and st["bvh_triangles"] > 0 and st["light_grids"] > 0
    finally:
        pr.close()


@pytest.mark.gpu
def test_bad_updates_are_rejected_and_change_nothing(gpu):
    """NULL pointers, n = 0, a triangle's index, an out-of-range index, a valid entry followed by an invalid one and an index from before
    rfx_scene_reset are RFX_ERR_ARG; the frames around them are those of a context that never made the calls"""
    capi, torch = gpu
    import ctypes as C
    W, H, depth = 96, 54, 6
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(8)
    tri = S.object_indices(scene)[[o[0] for o in scene["objects"]].index("tri")]
    i32 = lambda a: np.ascontiguousarray(a, np.int32)
    anim, ref = capi.Context(0), capi.Context(0)
    try:
        frames = []
        for c, bad in ((anim, True), (ref, False)):
            c.load_scene(scene)
            c.set_seeds(2, 2); c.set_image_size(W, H)
            out = [_frame(torch, c, S.default_camera(), depth, stream)]
            if bad:
                sp = np.array([[1, 2, 3, 0.5], [4, 5, 6, 0.5]], F)
                ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
                fp = sp.ctypes.data_as(capi._fp)
                ok = i32([3, 4])
                assert c.L.rfx_update_spheres(c.h, 2, None, fp) == -1
                assert c.L.rfx_update_spheres(c.h, 2, ip(ok), None) == -1
                assert c.L.rfx_update_spheres(c.h, 0, ip(ok), fp) == -1
                for objs in ([tri, 3], [3, tri], [3, 10 ** 6], [3, -1]):
                    o = i32(objs)
                    assert c.L.rfx_update_spheres(c.h, 2, ip(o), fp) == -1, objs
                with pytest.raises(capi.RfxError):
                    c.update_spheres([3, tri], sp)
                with pytest.raises(ValueError):
                    c.update_spheres([3], sp)
            out.append(_frame(torch, c, S.default_camera(), depth, stream))
            c.load_scene(S.default_scene())   # rfx_scene_reset: objects 20 and up are gone
            if bad:
                o = i32([20]); s1 = np.array([[0, 1, 0, 0.5]], F)
                assert c.L.rfx_update_spheres(c.h, 1, ip(o), s1.ctypes.data_as(capi._fp)) == -1
            out.append(_frame(torch, c, S.default_camera(), depth, stream))
            st = c.stats()
            frames.append(out + [st["rays"], c.get_seeds()])
        _same(frames[0], frames[1], "errors")
    finally:
        anim.close(); ref.close()


@pytest.mark.gpu
def test_identity_update_and_duplicates(gpu):
    """an identity update is served on the device and leaves every frame as it was; with a repeated index the last entry wins"""
    capi, torch = gpu
    W, H, depth = 160, 90, 8
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(16)
    still = capi.Context(0)
    pr = _Pair(capi, scene, 0, W, H, seeds=(6, 6))
    try:
        still.load_scene(scene); still.set_seeds(6, 6); still.set_image_size(W, H); still.render(S.default_camera(), 1)
        obj, sp = S.sphere_bounce(scene, 0.0)
        assert pr.anim.update_spheres(obj, sp)
        a = [_frame(torch, pr.anim, cam, depth, stream) for cam in (S.default_camera(), ORBIT)]
        b = [_frame(torch, still, cam, depth, stream) for cam in (S.default_camera(), ORBIT)]
        _same(a, b, "identity")
        _, moved = S.sphere_bounce(scene, 0.8, height=2.0, pulse=0.2)
        dup_obj = np.concatenate([obj[:50], obj[:50], obj[20:30]])
        dup_sp = np.concatenate([moved[:50] + F([0, 1.0, 0, 0]), moved[:50], moved[20:30] * F([1, 1, 1, 0.5])])
        pr.ref.set_seeds(6, 6); pr.anim.set_seeds(6, 6)
        assert pr.update(dup_obj, dup_sp)
        final = S.with_spheres(scene, dup_obj, dup_sp)["objects"]
        assert final[25][2] == float(moved[25, 3] * F(0.5)) and final[5][1] == tuple(float(x) for x in moved[5, :3])
        a, b = _frames(torch, pr, stream, depth)
        _same(a, b, "duplicates")
    finally:
        pr.close(); still.close()
