"""The eye grid built on the GPU: the screen grid of a path's first query in blob scenes (EyeGrid), built on the device for every new
camera, image size and sphere update (rfx_eye_grid.cu) instead of binned on the host.

rfx_selftest_eye_grid compares the grid the last blob render used with the host's binning (rfx_scene.cpp binEyeGrid) for that render's
camera and the current spheres: dims, every cell offset, every item's sphere index and record.  Frames must not depend on where the grid
was built, nor on whether there is one: ARGB, float images, ray counts, stream positions and hit-path signatures are compared bit for bit
under "eye_grid_device" 1 and 0 and "eye_grid" 0."""
import os
import sys

import numpy as np
import pytest

from reflaxman_b200 import scenes as S
from reflaxman_b200 import sharding as P

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
import primary_cull_proto as PC  # noqa: E402

F = np.float32
ORBIT = S.orbit_cameras(9)[2]
SETTINGS = ({"eye_grid": 1, "eye_grid_device": 1}, {"eye_grid": 1, "eye_grid_device": 0}, {"eye_grid": 0})


@pytest.fixture(scope="module")
def gpu(rfx_lib):
    import torch
    from reflaxman_b200 import capi
    return capi, torch


def _cloud(n=150, seed=77):
    """spheres of radii 0.03 .. 2 over a dielectric floor (test_gpu_parity.py::test_eye_grid_equals_hierarchy_walk)"""
    rng = np.random.default_rng(seed)
    objs = []
    for i in range(n):
        r = float(10 ** rng.uniform(-1.5, 0.3))
        c = rng.uniform([-8, 0, -6], [8, 5, 6])
        objs.append(("sphere", (float(c[0]), float(c[1]) + r, float(c[2])), r, int(i % 2), tuple(float(v) for v in rng.uniform(0.3, 1.0, 3)),
                     float(rng.uniform(0.0, 1.0)), 0.0))
    objs.append(("tri", (-14.0, 0.0, -10.0, -14.0, 0.0, 10.0, 14.0, 0.0, -10.0), S.MT_DIELECTRIC, (1.0, 1.0, 1.0), 0.9, 0.0, -1, (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
    objs.append(("tri", (-14.0, 0.0, 10.0, 14.0, 0.0, 10.0, 14.0, 0.0, -10.0), S.MT_DIELECTRIC, (1.0, 1.0, 1.0), 0.9, 0.0, -1, (0.0, 1.0, 1.0, 1.0, 1.0, 0.0)))
    return {"ambient": ((0.9, 0.9, 1.0), 0.2), "skybox": None, "textures": [], "lights": S.default_scene()["lights"], "objects": objs}


def _skewed(cam):
    eye, view, fov = cam
    view = np.array(view, np.float32)
    view[0] *= np.float32(1.01)
    return eye, view, fov


def _context(capi, scene, W, H, seeds=(3, 3), **options):
    c = capi.Context(0)
    c.load_scene(scene); c.set_seeds(*seeds); c.set_image_size(W, H)
    c.set_bvh_mode(1)
    for k, v in options.items():
        c.set_option(k, v)
    return c


def _clean(c, what):
    diff, dev, host, dropped = c.eye_grid_selftest()
    assert diff == 0 and dev == host and dropped == 0, (what, diff, dev, host, dropped)
    return host


def _same(a, b, what):
    assert len(a) == len(b), what
    for k, (x, y) in enumerate(zip(a, b)):
        if isinstance(x, np.ndarray):
            assert x.dtype == y.dtype and np.array_equal(x.view(np.uint32) if x.dtype == np.float32 else x,
                                                         y.view(np.uint32) if y.dtype == np.float32 else y), (what, k)
        else:
            assert x == y, (what, k, x, y)


# ---- device grid == host binning -------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("which", ["grid16", "grid32", "grid64", "cloud"])
def test_device_grid_equals_host_binning(gpu, which):
    """cameras all over the place — orbit, inside spheres, under the floor, looking away, fov 0.3 .. 2.6 — at 1x1, ragged sizes and
    up to 7680x4320: the grid built on the device is the host's, cell for cell and item for item.  The item region is sized at the first
    build (here 8x8 pixels): a bigger grid is dropped, and after rfx_synchronize the same camera's grid fits.  A skewed (non-orthonormal)
    camera gets a grid on neither side."""
    capi, _ = gpu
    scene = _cloud() if which == "cloud" else S.synthetic_scene(int(which[4:]))
    sph, _ = PC.scene_arrays(scene)
    cams = PC.random_cameras(12, 5, sph)
    c = _context(capi, scene, 8, 8)
    try:
        listed = drops = 0
        for W, H, n in ((1, 1, 4), (333, 77, 12), (200, 120, 12), (1000, 563, 6), (7680, 4320, 2)):
            c.set_image_size(W, H)
            for cam in cams[:n]:
                c.render(cam, 1)
                diff, dev, host, dropped = c.eye_grid_selftest()
                if dev == 0 and host > 0:
                    assert diff == 0 and dropped == drops + 1, (which, W, H, diff, dropped)
                    drops = dropped
                    c.synchronize()
                    c.render(cam, 1)
                    diff, dev, host, dropped = c.eye_grid_selftest()
                assert diff == 0 and dev == host and dropped == drops, (which, W, H, diff, dev, host, dropped)
                listed += host
        assert listed > 0
        c.set_image_size(200, 120)
        c.render(_skewed(S.orbit_cameras(9)[4]), 1)
        assert c.eye_grid_selftest() == (0, 0, 0, drops)
    finally:
        c.close()


# ---- frames identical -----------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("plane", [False, True])
def test_frames_do_not_depend_on_where_the_grid_is_built(gpu, plane):
    """a camera path through rfx_render_frames (depths 1, 2, 6: tile kernel and wavefront pair) and through rfx_render_frames_device on a
    torch stream; the Render API with 2x2 SSAA, additive passes, block preview and ragged renderNext slices on the general kernel with
    signatures; a 2-way rfx_render_strips split: identical under eye_grid_device 1 / 0 and eye_grid 0, with and without a ground plane"""
    capi, torch = gpu
    scene = S.synthetic_scene(16, floor=S.synthetic_texture(64, 64, 3))
    if plane:
        scene = S.with_ground_plane(scene)
    sph, _ = PC.scene_arrays(scene)
    cams = PC.random_cameras(12, 7, sph)
    W, H = 200, 120
    stream = torch.cuda.Stream()
    res = []
    for opt in SETTINGS:
        c = _context(capi, scene, W, H, **opt)
        try:
            out = [c.render_frames(cams, d) for d in (1, 2, 6)]
            buf = torch.empty(len(cams) * W * H, dtype=torch.int32, device="cuda:0")
            torch.cuda.synchronize()
            c.render_frames_device(cams, 4, 1, buf.data_ptr(), stream.cuda_stream)
            c.synchronize()
            torch.cuda.synchronize()
            out.append(buf.cpu().numpy().view(np.uint32).copy())
            if opt.get("eye_grid"):
                _clean(c, opt)
            for cam in cams[::5]:
                c.render(cam, 4, samples=2)
                out += [c.read_rgbf().copy(), c.read_argb().copy()]
            for _ in range(3):
                c.render(ORBIT, 4, additive=True)
            out.append(c.read_rgbf().copy())
            c.render(ORBIT, 4, samples=-3)
            out.append(c.read_argb().copy())
            gather = c.buffer_alloc(W * H * 4)
            for rank in range(2):
                P.split_frame(c, cams[3], 6, 1, 2, rank, gather, strip_rows=8)
                c.synchronize()
            out.append(c.buffer_read(gather, np.zeros((H, W), np.uint32)).copy())
            c.buffer_free(gather)
            c.force_path(3)
            c.enable_signatures(True)
            for cam in cams[1::4]:
                c.render(cam, 5, chunk=W * 7 + 13)
                out += [c.read_argb().copy(), c.read_signatures().copy()]
            st = c.stats()
            assert st["launches_blob_any"] > 0 and st["launches_blob_fast"] > 0
            res.append(out + [st["rays"], st["bounces"], c.get_seeds()])
        finally:
            c.close()
    _same(res[0], res[1], "device / host")
    _same(res[0], res[2], "device / none")


# ---- sphere animation ---------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_bouncing_spheres_under_a_moving_camera(gpu):
    """16 steps of sphere_bounce, a new camera each step, frames into a torch stream: the grid is clean after every step, and the last
    frame equals a fresh context loaded with the moved spheres"""
    capi, torch = gpu
    scene = S.synthetic_scene(16)
    W, H, depth = 160, 90, 6
    cams = S.orbit_cameras(16)
    stream = torch.cuda.Stream()
    buf = torch.empty(W * H, dtype=torch.int32, device="cuda:0")
    c = _context(capi, scene, W, H, seeds=(7, 7))
    try:
        c.render(S.default_camera(), 1)
        for step in range(16):
            obj, sp = S.sphere_bounce(scene, 0.37 * (step + 1), height=2.0, pulse=0.2 if step % 2 else 0.0)
            assert c.update_spheres(obj, sp), step
            c.render_frames_device([cams[step]], depth, 1, buf.data_ptr(), stream.cuda_stream)
            _clean(c, step)
        c.synchronize()
        torch.cuda.synchronize()
        last = buf.cpu().numpy().view(np.uint32).copy()
        seeds = c.get_seeds()
    finally:
        c.close()
    # a fresh context loaded with the moved spheres renders the same sequence (the stream advances alike): its last frame is the same
    r = _context(capi, S.with_spheres(scene, obj, sp), W, H, seeds=(7, 7))
    try:
        r.render(S.default_camera(), 1)
        for step in range(16):
            r.render_frames_device([cams[step]], depth, 1, buf.data_ptr(), stream.cuda_stream)
        r.synchronize()
        torch.cuda.synchronize()
        assert np.array_equal(buf.cpu().numpy().view(np.uint32), last)
        assert r.get_seeds() == seeds
    finally:
        r.close()


@pytest.mark.gpu
def test_light_and_mesh_updates_do_not_rebuild_the_grid(gpu):
    """rfx_update_lights and rfx_update_mesh between frames of one camera leave the eye grid alone: the render after them launches as many
    kernels as a render after no update, the grid stays clean and its item count unchanged; a sphere update then rebuilds it"""
    capi, _ = gpu
    n_u, n_v = 16, 16
    scene = S.mesh_scene(n_u, n_v, spheres=8)
    first = [i for ob, i in zip(scene["objects"], S.object_indices(scene)) if ob[0] == "mesh"][0]
    W, H, depth = 160, 90, 4
    c = _context(capi, scene, W, H)
    try:
        c.render(ORBIT, depth)
        items = _clean(c, "first")
        assert items > 0

        def launches():
            return c.stats()["kernel_launches"]
        k0 = launches(); c.render(ORBIT, depth); plain = launches() - k0
        for step in range(4):
            if step % 2:
                assert c.update_mesh(first, S.torus_wave(n_u, n_v, phase=0.7 * step, amplitude=0.2)), step
            else:
                assert c.update_lights(*S.sun_orbit(scene, 0.5 * (step + 1))), step
            k0 = launches(); c.render(ORBIT, depth)
            assert launches() - k0 == plain, step
            assert _clean(c, step) == items
        assert c.update_spheres(*S.sphere_bounce(scene, 1.3, height=2.0))
        k0 = launches(); c.render(ORBIT, depth)
        assert launches() - k0 > plain
        _clean(c, "spheres")
    finally:
        c.close()


# ---- capacity ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_a_dropped_build_walks_the_hierarchy_and_the_next_one_fits(gpu):
    """with "eye_grid_items" small the device build is dropped: the frame equals the frame without a grid, the selftest counts the drop
    and reports no items on the device; after rfx_synchronize (and the cap lifted) the next render's grid is clean"""
    capi, _ = gpu
    scene = S.synthetic_scene(16)
    W, H, depth = 200, 120, 6
    cams = S.orbit_cameras(9)[1:4]
    c = _context(capi, scene, W, H, eye_grid_items=16)
    r = _context(capi, scene, W, H, eye_grid=0)
    try:
        a, b = c.render_frames(cams, depth), r.render_frames(cams, depth)
        assert np.array_equal(a, b)
        diff, dev, host, dropped = c.eye_grid_selftest()
        assert diff == 0 and dev == 0 and host > 16 and dropped >= 1, (diff, dev, host, dropped)
        c.set_option("eye_grid_items", 0)
        c.synchronize()
        a, b = c.render_frames(cams, depth), r.render_frames(cams, depth)
        assert np.array_equal(a, b)
        diff, dev, host, dropped2 = c.eye_grid_selftest()
        assert diff == 0 and dev == host > 0 and dropped2 == dropped
        assert c.get_seeds() == r.get_seeds()
    finally:
        c.close(); r.close()


@pytest.mark.gpu
def test_the_item_region_grows_after_a_build_that_did_not_fit(gpu):
    """40 spheres around the eye, each covering the whole 7680x4320 screen: more items than the first region holds.  The first frame's build
    is dropped (and the frame is the no-grid frame); rfx_get_stats grows the region, and the next render's grid fits and is clean"""
    capi, _ = gpu
    objs = [("sphere", (0.0, 1.0, 0.0), 1.0 + 0.5 * k, 0, (0.9, 0.8, 0.7), 0.3, 0.0) for k in range(40)]
    scene = {"ambient": ((0.9, 0.9, 1.0), 0.2), "skybox": None, "textures": [], "lights": S.default_scene()["lights"], "objects": objs}
    cam = S.camera_lookat((0.0, 1.0, 0.0), (0.0, 1.0, 5.0))
    W, H = 7680, 4320
    c = _context(capi, scene, W, H)
    r = _context(capi, scene, W, H, eye_grid=0)
    try:
        a = c.render(cam, 2).read_argb().copy()
        b = r.render(cam, 2).read_argb().copy()
        assert np.array_equal(a, b)
        diff, dev, host, dropped = c.eye_grid_selftest()
        assert diff == 0 and dev == 0 and host == 40 * 240 * 135 and dropped == 1, (diff, dev, host, dropped)
        c.stats()
        a = c.render(cam, 2).read_argb().copy()
        b = r.render(cam, 2).read_argb().copy()
        assert np.array_equal(a, b)
        assert c.eye_grid_selftest() == (0, host, host, 1)
    finally:
        c.close(); r.close()


# ---- scenes without a grid, bad calls -----------------------------------------------------------------------------------------------

@pytest.mark.gpu
def test_constant_bank_scenes_build_no_eye_grid(gpu):
    """the default scene renders on the constant-bank kernels: no blob frame, so the selftest has nothing to compare (RFX_ERR_ARG); a
    blob scene's selftest before its first render, and after a scene change, is refused too"""
    capi, _ = gpu
    c = capi.Context(0)
    try:
        c.load_scene(S.default_scene()); c.set_image_size(96, 60)
        c.render(S.default_camera(), 4)
        assert c.stats()["launches_blob_fast"] == 0 and c.stats()["launches_blob_any"] == 0
        with pytest.raises(capi.RfxError):
            c.eye_grid_selftest()
        c.load_scene(S.synthetic_scene(8)); c.set_bvh_mode(1)
        with pytest.raises(capi.RfxError):
            c.eye_grid_selftest()
        c.render(S.default_camera(), 1)
        _clean(c, "blob")
        c.load_scene(S.synthetic_scene(9))
        with pytest.raises(capi.RfxError):
            c.eye_grid_selftest()
        for name, bad in (("eye_grid_device", 2), ("eye_grid_items", -1)):
            with pytest.raises(capi.RfxError):
                c.set_option(name, bad)
    finally:
        c.close()
