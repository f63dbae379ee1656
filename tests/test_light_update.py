"""rfx_update_lights: lights moved, resized and recoloured in place, their candidate grids built on the GPU.

Every GPU case animates one context through rfx_update_lights (and, in one case, rfx_update_spheres / rfx_update_mesh) and renders the
same frames, in the same order and from the same seeds, in a reference context that loads the scene anew with the moved lights
(rfx_add_light(new values), a host flatten) before each frame.  Everything must agree bit for bit: ARGB, float images as uint32,
signatures, ray, bounce and shadow counts and the stream position after.  Each update's return value states which path served it (1: on
the device, 0: host re-flatten at the next render), and rfx_selftest_light_grids compares every grid the device built with the host's
rebuild of it, byte for byte.

CPU: with_lights and sun_orbit of scenes.py."""
import math

import numpy as np
import pytest

from reflaxman_b200 import scenes as S

F = np.float32


# ---- CPU ---------------------------------------------------------------------------------------------------------------------------

def test_with_lights_replaces_exactly_the_given_lights():
    sc = S.synthetic_scene(4)
    sc["lights"] = sc["lights"] + [((1.0, 9.0, 2.0), 0.5, (0.2, 0.3, 0.4), 0.5), ((3.0, 9.0, 2.0), 0.25, (1.0, 0.0, 0.0), 1.0)]
    rec = np.array([[1, 2, 3, 0.5, 0.1, 0.2, 0.3, 1.5], [4, 5, 6, 0.25, 1, 1, 1, -0.5], [7, 8, 9, 0.75, 0.5, 0.5, 0.5, 0.25]], F)
    new = S.with_lights(sc, [2, 0, 2], rec)
    assert new["lights"][2] == ((7.0, 8.0, 9.0), 0.75, (0.5, 0.5, 0.5), 0.25)       # the later row wins
    assert new["lights"][0] == ((4.0, 5.0, 6.0), 0.25, (1.0, 1.0, 1.0), -0.5)
    assert new["lights"][1] is sc["lights"][1]
    assert new["objects"] is sc["objects"] and sc["lights"][0][0] == (11.8e9, 4.26e9, 3.08e9)
    with pytest.raises(ValueError):
        S.with_lights(sc, [3], rec[:1])


def test_sun_orbit_is_the_loaded_light_at_rest_and_stays_far():
    sc = S.synthetic_scene(8)
    li, rec = S.sun_orbit(sc, 0.0)
    assert li.dtype == np.int32 and list(li) == [0] and rec.dtype == F and rec.shape == (1, 8)
    o, r, c, p = sc["lights"][0]
    assert np.array_equal(rec[0].view(np.uint32), np.array(list(o) + [r] + list(c) + [p], F).view(np.uint32))
    assert S.with_lights(sc, li, rec)["lights"][0] == tuple((tuple(float(F(v)) for v in o), float(F(r)), tuple(float(F(v)) for v in c), float(F(p))))
    dist = float(np.linalg.norm(rec[0, :3].astype(np.float64)))
    seen = set()
    for t in np.linspace(0.3, 12.0, 40):
        _, m = S.sun_orbit(sc, float(t))
        assert np.array_equal(m[0, 3:], rec[0, 3:])                                # radius, colour and power stay
        d = float(np.linalg.norm(m[0, :3].astype(np.float64)))
        assert abs(d / dist - 1.0) < 1e-5
        el = math.asin(m[0, 1] / d)
        assert 0.1 - 1e-4 <= el <= 1.4 + 1e-4                                      # above the horizon
        # far from the scene: the grid's test (distance > 8 * (half the scene's diagonal + radius)) holds with a margin
        assert d > 4.0 * 8.0 * (0.5 * math.sqrt(28 ** 2 + 8 ** 2 + 20 ** 2) + float(m[0, 3]))
        seen.add(round(math.atan2(m[0, 2], m[0, 0]), 2))
    assert len(seen) > 30


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu(rfx_lib):
    import torch
    from reflaxman_b200 import capi
    return capi, torch


def _frame(torch, c, cam, depth, stream, samples=1):
    """one rfx_render_frames_device frame into a torch buffer on ``stream``; ARGB [H, W]"""
    buf = torch.empty(c.H * c.W, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    c.render_frames_device([cam], depth, samples, buf.data_ptr(), stream.cuda_stream)
    torch.cuda.synchronize()
    return buf.cpu().numpy().view(np.uint32).reshape(c.H, c.W).copy()


class _Pair:
    """the animated context and its reference, set up alike, each with one depth-1 frame rendered (the first flatten: a device update
    needs a flattened scene)"""

    def __init__(self, capi, scene, mode, W, H, seeds=(77, 77)):
        self.scene = scene
        self.anim, self.ref = capi.Context(0), capi.Context(0)
        self.meshes = None
        for c in (self.anim, self.ref):
            self.meshes = c.load_scene(scene)
            c.set_bvh_mode(mode); c.set_seeds(*seeds); c.set_image_size(W, H)
            c.render(S.default_camera(), 1)

    def update(self, lights, records):
        """update the animated context, reload the reference with the moved lights; returns the update's path"""
        r = self.anim.update_lights(lights, records)
        self.scene = S.with_lights(self.scene, lights, records)
        self.ref.load_scene(self.scene)
        return r

    def both(self, fn):
        return fn(self.anim), fn(self.ref)

    def tail(self):
        out = []
        for c in (self.anim, self.ref):
            st = c.stats()
            out.append([st["rays"], st["bounces"], st["shadow_rays"], c.get_seeds()])
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
    return pr.both(lambda c: [_frame(torch, c, cam or S.default_camera(), depth, stream) for cam in cams])


def _grids(c):
    return c.stats()["light_grids"]


@pytest.mark.gpu
def test_sun_orbit_over_the_synthetic_scene(gpu):
    """12 orbit steps of the sun over synthetic_scene(32) with its floor, wall and sky: the tile kernel, the wavefront pair at depths
    4 and 8, the general kernel (ragged render_next slices, block preview), 2x2 SSAA, additive passes and rfx_trace_rays equal the
    reference's; after every update the device's grid is the host's, byte for byte"""
    capi, torch = gpu
    W, H = 160, 90
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(32, floor=S.synthetic_texture(64, 64, 3), skybox=S.synthetic_texture(128, 96, 5))
    pr = _Pair(capi, scene, 0, W, H)
    rng = np.random.RandomState(4)
    try:
        pr.anim.enable_signatures(True); pr.ref.enable_signatures(True)
        for step in range(12):
            assert pr.update(*S.sun_orbit(scene, 0.55 * (step + 1))), step
            assert pr.anim.light_grids_selftest() == (0, 1, 1), step
            kind = step % 4
            if kind == 0:
                for path, wave, depth in ((2, 0, 4), (2, 2, 4), (2, 2, 8)):
                    a, b = pr.both(lambda c: (c.force_path(path), c.set_option("blob_wavefront", wave), _frame(torch, c, ORBIT, depth, stream))[2])
                    _same([a], [b], (step, wave, depth))
            elif kind == 1:
                a, b = pr.both(lambda c: (c.force_path(3), c.render(S.default_camera(), 6, chunk=997),
                                          [c.read_rgbf().copy(), c.read_argb().copy(), c.read_signatures().copy()])[2])
                _same(a, b, (step, "ragged"))
                a, b = pr.both(lambda c: (c.force_path(3), c.render(ORBIT, 4, samples=-3), [c.read_rgbf().copy(), c.read_argb().copy()])[2])
                _same(a, b, (step, "block preview"))
            elif kind == 2:
                a, b = pr.both(lambda c: (c.force_path(0), _frame(torch, c, ORBIT, 4, stream, samples=2))[1])
                _same([a], [b], (step, "ssaa"))
                a, b = pr.both(lambda c: (c.force_path(0), c.render(S.default_camera(), 4, additive=True), c.render(S.default_camera(), 4, additive=True),
                                          c.read_image(divide=False))[3])
                _same(list(a), list(b), (step, "additive"))
            else:
                o = rng.uniform([-12, 0.5, -8], [12, 6, 8], (500, 3)).astype(F)
                d = rng.normal(size=(500, 3)).astype(F)
                a, b = pr.both(lambda c: c.trace_rays(o, d, 4))
                _same([a], [b], (step, "rays"))
        a, b = pr.tail()
        _same(a, b, "counts")
        assert _grids(pr.anim) == _grids(pr.ref) == 1
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_bvh_modes(gpu, mode):
    """bvh modes 0, 1 and 2 (no hierarchy, no grid: still updated on the device)"""
    capi, torch = gpu
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(8)
    pr = _Pair(capi, scene, mode, 160, 90, seeds=(5, 9))
    try:
        for step in range(4):
            assert pr.update(*S.sun_orbit(scene, 1.3 * (step + 1))), (mode, step)
            a, b = _frames(torch, pr, stream, 6)
            _same(a, b, (mode, step))
            assert pr.anim.light_grids_selftest() == ((0, 1, 1) if mode != 2 else (0, 0, 0))
        a, b = pr.tail()
        _same(a, b, "counts")
        assert _grids(pr.anim) == _grids(pr.ref) == (1 if mode != 2 else 0)
    finally:
        pr.close()


@pytest.mark.gpu
def test_grid_transitions(gpu):
    """the only far light moves into the scene (it loses its grid: the kernels without grids run), back out (it regains it), and a
    scene whose flatten built no grid gets a far light (host re-flatten)"""
    capi, torch = gpu
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(8)
    pr = _Pair(capi, scene, 0, 160, 90, seeds=(11, 3))
    try:
        _, sun = S.sun_orbit(scene, 0.0)
        near = sun.copy(); near[0, :4] = (2.0, 9.0, 1.0, 0.5)
        for k, rec in enumerate((near, S.sun_orbit(scene, 2.0)[1], near, sun)):
            assert pr.update([0], rec), k
            assert pr.anim.light_grids_selftest() == (0, k % 2, k % 2), k
            a, b = _frames(torch, pr, stream, 6)
            _same(a, b, k)
            assert _grids(pr.anim) == _grids(pr.ref) == k % 2, k      # (the reference's after its flatten)
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()
    lamp = dict(scene, lights=[((2.0, 9.0, 1.0), 0.5, (1.0, 1.0, 0.95), 0.85)])
    pr = _Pair(capi, lamp, 0, 160, 90)
    try:
        assert _grids(pr.anim) == 0
        assert not pr.update([0], S.sun_orbit(scene, 1.0)[1])
        a, b = _frames(torch, pr, stream, 6)
        _same(a, b, "reflattened")
        assert _grids(pr.anim) == _grids(pr.ref) == 1
        assert pr.update([0], S.sun_orbit(scene, 2.0)[1])           # ... and now it has a grid to build on the device
        a, b = _frames(torch, pr, stream, 6)
        _same(a, b, "after")
        assert pr.anim.light_grids_selftest() == (0, 1, 1)
    finally:
        pr.close()


@pytest.mark.gpu
@pytest.mark.parametrize("sky", [False, True])
def test_colour_power_and_radius(gpu, sky):
    """power above 1 and below 0 (the record clamps it, the ambient term adds it as given), radius <= VSN, colour changes"""
    capi, torch = gpu
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(8, skybox=S.synthetic_texture(128, 96, 5) if sky else None)
    pr = _Pair(capi, scene, 0, 160, 90, seeds=(2, 2))
    try:
        _, rec = S.sun_orbit(scene, 0.7)
        for k, (power, radius, rgb) in enumerate(((1.7, 3.48e8, (1.0, 0.6, 0.3)), (-0.3, 3.48e8, (0.2, 0.9, 1.0)), (0.5, 0.0, (1.0, 1.0, 1.0)),
                                                  (0.85, -5.0, (0.7, 0.7, 0.2)), (2.5, 1e-30, (0.3, 0.3, 0.3)))):
            r = rec.copy(); r[0, 3] = radius; r[0, 4:7] = rgb; r[0, 7] = power
            assert pr.update([0], r), k
            a, b = _frames(torch, pr, stream, 4)
            _same(a, b, k)
            a, b = pr.both(lambda c: (c.force_path(3), c.render(S.default_camera(), 3), c.read_rgbf().copy())[2])
            _same([a], [b], (k, "rgbf"))
            assert pr.anim.light_grids_selftest()[0] == 0
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()


@pytest.mark.gpu
def test_three_lights_subsets_duplicates_and_identity(gpu):
    """two far lights and a near lamp: subsets, a duplicated index (the later row wins) and an identity update, which rebuilds the
    grids byte-equal to the flatten's"""
    capi, torch = gpu
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(12)
    sun2 = ((-6.0e9, 9.0e9, 2.0e9), 2.0e8, (0.6, 0.7, 1.0), 0.4)
    lamp = ((1.0, 7.0, -2.0), 0.3, (1.0, 0.8, 0.6), 0.6)
    scene = dict(scene, lights=scene["lights"] + [sun2, lamp])
    pr = _Pair(capi, scene, 0, 160, 90, seeds=(8, 1))
    rows = lambda sc: np.array([list(o) + [r] + list(c) + [p] for o, r, c, p in sc["lights"]], F)
    try:
        assert pr.anim.light_grids_selftest() == (0, 2, 2) and _grids(pr.anim) == 2
        ident = rows(scene)
        assert pr.update([0, 1, 2], ident)
        assert pr.anim.light_grids_selftest() == (0, 2, 2)
        a, b = _frames(torch, pr, stream, 5)
        _same(a, b, "identity")
        for step in range(4):
            cur = rows(pr.scene)
            s1 = S.sun_orbit(pr.scene, 0.8 * (step + 1))[1][0]
            lamp_row = cur[2].copy(); lamp_row[0] += F(0.5 * step); lamp_row[7] = F(0.2 * step)
            sun2_row = cur[1].copy(); sun2_row[:3] *= F(1.0 + 0.1 * step); sun2_row[4] = F(0.3)
            if step % 2 == 0:
                li, rec = [2, 1, 2], np.stack([cur[2], sun2_row, lamp_row])      # the lamp twice: its last row wins
            else:
                li, rec = [0, 2], np.stack([s1, lamp_row])
            assert pr.update(li, rec), step
            assert pr.anim.light_grids_selftest() == (0, 2, 2), step
            a, b = _frames(torch, pr, stream, 5)
            _same(a, b, step)
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()


@pytest.mark.gpu
def test_plane_scene_and_constant_bank_scene(gpu):
    """a scene with a plane has no light grids (updated on the device); the constant-bank default scene re-flattens"""
    capi, torch = gpu
    stream = torch.cuda.Stream()
    scene = S.with_ground_plane(S.synthetic_scene(8))
    pr = _Pair(capi, scene, 0, 160, 90)
    try:
        for step in range(3):
            assert pr.update(*S.sun_orbit(scene, 1.1 * (step + 1))), step
            a, b = _frames(torch, pr, stream, 6)
            _same(a, b, step)
        assert _grids(pr.anim) == 0 and pr.anim.light_grids_selftest() == (0, 0, 0)
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()
    scene = S.default_scene()
    pr = _Pair(capi, scene, 0, 160, 90)
    try:
        for step in range(2):
            assert not pr.update(*S.sun_orbit(scene, 1.1 * (step + 1))), step
            a, b = _frames(torch, pr, stream, 6)
            _same(a, b, step)
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()


@pytest.mark.gpu
def test_alternating_with_sphere_and_mesh_updates(gpu):
    """light updates between sphere updates (all spheres, 1/16 of them, a crowd in a few cells of the grid) and mesh updates: after
    each update the device's grid is the host's"""
    capi, torch = gpu
    stream = torch.cuda.Stream()
    scene = S.mesh_scene(16, 8, spheres=16)
    pr = _Pair(capi, scene, 0, 160, 90, seeds=(6, 4))
    try:
        first = pr.meshes[0]
        obj, sp = S.sphere_bounce(scene, 0.0)
        rng = np.random.RandomState(2)
        crowd = sp.copy()
        crowd[:, :3] = (F([1.0, 4.0, 0.5]) + rng.uniform(-0.4, 0.4, (len(sp), 3))).astype(F)
        crowd[:, 3] = F(0.05)
        crowd[::16, 3] = F(1.5)
        for step in range(6):
            assert pr.update(*S.sun_orbit(scene, 0.9 * (step + 1))), step
            assert pr.anim.light_grids_selftest() == (0, 1, 1)
            if step % 3 == 0:
                o, s = S.sphere_bounce(scene, 0.4 * (step + 1), height=2.0)
            elif step % 3 == 1:
                o, s = obj[::16], S.sphere_bounce(scene, 0.4 * (step + 1), height=2.0)[1][::16]
            else:
                o, s = obj, crowd
            assert pr.anim.update_spheres(o, s), step
            pr.scene = S.with_spheres(pr.scene, o, s)
            assert pr.anim.light_grids_selftest() == (0, 1, 1), step
            xyz = S.torus_wave(16, 8, 0.7 * (step + 1))
            assert pr.anim.update_mesh(first, xyz), step
            pr.scene = dict(pr.scene, objects=[ob if ob[0] != "mesh" else ob[:1] + (xyz,) + ob[2:] for ob in pr.scene["objects"]])
            pr.ref.load_scene(pr.scene)
            a, b = _frames(torch, pr, stream, 6)
            _same(a, b, step)
        a, b = pr.tail()
        _same(a, b, "counts")
        assert _grids(pr.anim) == 1
    finally:
        pr.close()


@pytest.mark.gpu
def test_updates_and_frames_queued_on_a_caller_stream(gpu):
    """(update, frame) pairs queued on a caller's torch stream with no synchronisation in between, then one synchronisation"""
    capi, torch = gpu
    scene = S.synthetic_scene(16)
    W, H, n = 160, 90, 8
    anim, ref = capi.Context(0), capi.Context(0)
    try:
        for c in (anim, ref):
            c.load_scene(scene); c.set_seeds(13, 13); c.set_image_size(W, H); c.render(S.default_camera(), 1)
        stream = torch.cuda.Stream()
        bufs = torch.zeros((n, H * W), dtype=torch.int32, device="cuda:0")
        cams = [S.default_camera(), ORBIT]
        torch.cuda.synchronize()
        for k in range(n):
            assert anim.update_lights(*S.sun_orbit(scene, 0.4 * (k + 1)))
            anim.render_frames_device([cams[k % 2]], 6, 1, bufs[k].data_ptr(), stream.cuda_stream)
        torch.cuda.synchronize()
        got = bufs.cpu().numpy().view(np.uint32)
        for k in range(n):
            ref.load_scene(S.with_lights(scene, *S.sun_orbit(scene, 0.4 * (k + 1))))
            exp = _frame(torch, ref, cams[k % 2], 6, stream)
            assert np.array_equal(got[k].reshape(H, W), exp), k
        sa, sr = anim.stats(), ref.stats()
        assert [sa["rays"], sa["bounces"], sa["shadow_rays"], anim.get_seeds()] == [sr["rays"], sr["bounces"], sr["shadow_rays"], ref.get_seeds()]
    finally:
        anim.close(); ref.close()


@pytest.mark.gpu
def test_a_grid_that_does_not_fit_is_dropped_and_restored(gpu):
    """under a tiny item capacity a grid built on the device is dropped (the frames still equal; light_grids counts it out), and a later
    build with room restores it"""
    capi, torch = gpu
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(16)
    pr = _Pair(capi, scene, 0, 160, 90, seeds=(1, 7))
    try:
        pr.anim.set_option("light_grid_items", 1)
        assert pr.update(*S.sun_orbit(scene, 1.0))
        a, b = _frames(torch, pr, stream, 6)
        _same(a, b, "dropped")
        assert _grids(pr.anim) == 0 and _grids(pr.ref) == 1
        assert pr.anim.light_grids_selftest() == (0, 0, 1)
        pr.anim.set_option("light_grid_items", 0)
        assert pr.update(*S.sun_orbit(scene, 2.0))
        a, b = _frames(torch, pr, stream, 6)
        _same(a, b, "restored")
        assert _grids(pr.anim) == 1 and pr.anim.light_grids_selftest() == (0, 1, 1)
        a, b = pr.tail()
        _same(a, b, "counts")
    finally:
        pr.close()


@pytest.mark.gpu
def test_bad_updates_are_rejected_and_change_nothing(gpu):
    """NULL pointers, n = 0, index -1 and index = number of lights are RFX_ERR_ARG; the frame after them and the stream position are
    those of a context that never made the calls"""
    capi, torch = gpu
    import ctypes as C
    stream = torch.cuda.Stream()
    scene = S.synthetic_scene(8)
    pr = _Pair(capi, scene, 0, 160, 90, seeds=(3, 3))
    try:
        c = pr.anim
        _, rec = S.sun_orbit(scene, 1.0)
        fp = rec.ctypes.data_as(capi._fp)
        ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int32))
        ok = np.zeros(1, np.int32)
        assert c.L.rfx_update_lights(c.h, 1, None, fp) == -1
        assert c.L.rfx_update_lights(c.h, 1, ip(ok), None) == -1
        assert c.L.rfx_update_lights(c.h, 0, ip(ok), fp) == -1
        assert c.L.rfx_update_lights(None, 1, ip(ok), fp) == -1
        for bad in (-1, 1):
            li = np.array([0, bad], np.int32)
            two = np.concatenate([rec, rec])
            assert c.L.rfx_update_lights(c.h, 2, ip(li), two.ctypes.data_as(capi._fp)) == -1, bad
        a, b = _frames(torch, pr, stream, 6)
        _same(a, b, "after")
        a, b = pr.tail()
        _same(a, b, "counts")
        assert c.light_grids_selftest() == (0, 1, 1)
    finally:
        pr.close()
