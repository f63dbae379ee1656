"""GPU parity at the REAL sizes of BASELINE.json's configs 3 and 4, the chunked SSAA path, and regression tests for the
round-1 advisor findings.  Everything goes through the C ABI (ctypes).

  * config 3 (7680x4320, depth 20): whole frame == the same frame rendered in chunks == the 2- and 3-way interleaved-strip
    split == the oracle (and the unmodified reference binary / its committed hash): exercises q < 2^32 pixel indexing, tile
    edges, K1 block ownership under strips and the 540-row tile grid at full size;
  * config 4 (1024 spheres, 3840x2160, depth 8): wavefront kernel pair == tile kernel == brute-force list walk == round-1 general kernel, and the
    multithreaded oracle at 960x540;
  * renderRange's chunk loop (huge SSAA factors): driven at small sizes by lowering "max_calls_per_launch".
"""
import hashlib

import numpy as np
import pytest

import cases
from reflaxman_b200 import scenes as S, sharding as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi(rfx_lib):
    from reflaxman_b200 import capi
    return capi


def _ctx(capi, scene, W, H, seed):
    c = capi.Context(0)
    c.load_scene(scene); c.set_seeds(seed, seed); c.set_image_size(W, H)
    return c


def test_config3_full_size_whole_chunked_split_oracle_reference(capi, oracle):
    W, H, refl, seed = 7680, 4320, 20, 12345
    cam = S.default_camera()
    scene = S.default_scene()

    c = _ctx(capi, scene, W, H, seed)
    try:
        c.stats_reset()
        whole = c.render_frames([cam], refl)[0]
        st = c.stats()
        seeds_after = c.get_seeds()
        assert st["launches_small_fast"] == 1 and st["launches_small_any"] == 0, st      # one launch of the fast kernel
        # the same frame with the launch cap below the frame's 33.2 M calls: four chunks of whole rows, each its own K1 pass
        c.set_seeds(seed, seed)
        c.set_option("max_calls_per_launch", 10_000_000)
        c.stats_reset()
        chunked = c.render_frames([cam], refl)[0]
        st2 = c.stats()
        assert st2["launches_small_fast"] == 4 and st2["launches_small_any"] == 0, st2
        assert np.array_equal(chunked, whole) and st2["rays"] == st["rays"] and c.get_seeds() == seeds_after
        # Render API (float image, renderNext in Pulse-sized slices that are not whole rows) at full size
        c.set_option("max_calls_per_launch", 1 << 25)
        c.set_seeds(seed, seed)
        c.render(cam, refl, chunk=W * 1000 + 777)
        assert np.array_equal(c.read_argb(), whole) and c.get_seeds() == seeds_after

        # interleaved 16-row strips dealt to 2 and to 3 "ranks" (contexts), stored straight into one gather buffer
        for world in (2, 3):
            gather = c.buffer_alloc(W * H * 4)        # zero-filled
            for rank in range(world):
                d = _ctx(capi, scene, W, H, seed)
                try:
                    d.stats_reset()
                    P.split_frame(d, cam, refl, 1, world, rank, gather, strip_rows=16)
                    d.synchronize()
                    assert d.get_seeds() == seeds_after, (world, rank)
                    assert d.stats()["launches_small_fast"] == 1
                finally:
                    d.close()
            got = c.buffer_read(gather, np.zeros((H, W), np.uint32))
            assert np.array_equal(got, whole), "split over %d ranks differs from the whole frame" % world
            c.buffer_free(gather)
    finally:
        c.close()

    # the oracle (pinned to the reference at this size by tests/test_oracle.py::test_oracle_config3_hash)
    o = oracle.OracleRender(scene, W, H, seed=seed).render(cam, refl)
    _, oargb = o.resolve()
    stp = cases.assert_parity(whole, oargb, "config 3 vs oracle")
    assert st["rays"] == o.counters["rays"] and seeds_after[0] == int(o.seeds[0])
    ref_hash = cases.full_size_hashes()["default_7680x4320_d20_seed12345"][0]
    exact = hashlib.sha256(whole.tobytes()).hexdigest() == ref_hash
    print("config 3 parity:", stp, "sha256 equals the reference's:", exact)
    assert hashlib.sha256(oargb.tobytes()).hexdigest() == ref_hash
    if oracle.have_ref():
        _, imgs = oracle.run_reference(W, H, refl=refl, seed=seed)
        cases.assert_parity(whole, imgs[0][1], "config 3 vs the reference binary")


def test_config4_full_size_bvh_equals_list_walk_equals_general_kernel(capi, oracle):
    W, H, refl, seed = 3840, 2160, 8, 12345
    cam = S.default_camera()
    scene = cases.config4_scene()
    out = {}
    # wave > 0: wavefront pair — the tile kernel for `wave` segments + the queue-driven kernel (hierarchy in shared memory, or, "L1",
    # read in place); wave 0: the single tile kernel; path 3: the round-1 general kernel
    for name, path, bvh, wave in (("batch+bvh", 2, 0, 2), ("wave1+bvh", 2, 0, 1), ("wave3+bvh", 2, 0, 3), ("batch+bvh+L1", 2, 0, 2), ("tile+bvh", 2, 0, 0),
                                  ("general+bvh", 3, 0, 0), ("batch+list", 2, 2, 2)):
        c = _ctx(capi, scene, W, H, seed)
        try:
            c.force_path(path); c.set_bvh_mode(bvh); c.stats_reset()
            c.set_option("blob_wavefront", wave); c.set_option("blob_smem_bvh", 0 if name.endswith("L1") else 1)
            img = c.render_frames([cam], refl)[0].copy()
            st = c.stats()
            want = 2 if wave > 0 else 1
            assert (st["launches_blob_fast"], st["launches_blob_any"]) == ((want, 0) if path == 2 else (0, 1)), (name, st)
            out[name] = (img, st["rays"], st["bounces"], c.get_seeds())
        finally:
            c.close()
    base = out["batch+bvh"]
    for name, got in out.items():
        assert np.array_equal(got[0], base[0]), name
        assert got[1:] == base[1:], name
    # the oracle at a quarter of the linear size (its list walk costs ~100 us per pixel per core)
    w, h = 960, 540
    o = oracle.OracleRender(scene, w, h, seed=seed).render(cam, refl, want_sig=True)
    c = _ctx(capi, scene, w, h, seed)
    try:
        c.stats_reset()
        small = c.render_frames([cam], refl)[0]
        st = c.stats()
        assert st["launches_blob_fast"] == 2
        assert st["rays"] == o.counters["rays"] and st["bounces"] == o.counters["bounces"]
        print("config 4 at 960x540 vs oracle:", cases.assert_parity(small, o.resolve()[1], "config 4 vs oracle"))
        c.set_seeds(seed, seed)
        c.enable_signatures(True)
        c.render(cam, refl)
        assert np.array_equal(c.read_signatures(), o.sig), "hit paths differ"
        assert np.array_equal(c.read_argb(), small)
    finally:
        c.close()


@pytest.mark.parametrize("path", [1, 2], ids=["constbank", "blob"])
@pytest.mark.parametrize("name,cap", [("default_96x64_ss3", 20000), ("default_96x64_ss3", 500), ("default_96x64_ss3", 9 * 96 * 7 + 5),
                                      ("default_96x64_additive3", 2000), ("default_96x64_additive3", 333)])
def test_chunked_launches_match_golden(capi, name, cap, path):
    """renderRange's chunk loop (rfx_capi.cu): with the cap below the frame's call count a frame takes >= 3 launches — whole-row
    chunks on the tiled kernels when the cap holds at least a row, ragged pixel chunks on the general kernels otherwise — each
    with its own K1 pass; the golden vectors (reference output) must still come out, and the streams must end where they do
    without chunking."""
    g = cases.load_golden(name)
    plain = cases.GpuEngine(capi, g["scene"], g["W"], g["H"], g["seed"])
    eng = cases.GpuEngine(capi, g["scene"], g["W"], g["H"], g["seed"])
    eng.c.force_path(path); plain.c.force_path(path)
    eng.c.set_option("max_calls_per_launch", cap)
    try:
        eng.c.stats_reset()
        frames = cases.replay(eng, g)
        st = eng.c.stats()
        per_pass = g["W"] * g["H"] * g["samples"] ** 2
        passes = max(g["additive"], 1) * g["frames"]
        launches = st["launches_small_fast"] + st["launches_small_any"] + st["launches_blob_fast"] + st["launches_blob_any"]
        assert launches >= passes * max(3, per_pass // cap), (launches, st)
        want = cases.replay(plain, g)
        for i, (rgbf, argb) in enumerate(frames):
            assert np.array_equal(rgbf.view(np.uint32), want[i][0].view(np.uint32)), "chunking changed the float image"
            cases.assert_parity(argb, g["argb%d" % i], "%s frame %d, cap %d" % (name, i, cap))
            assert np.max(np.abs(rgbf - g["rgbf%d" % i])) < 2e-5
        assert eng.c.get_seeds() == plain.c.get_seeds()
    finally:
        eng.close(); plain.close()


def test_ssaa16_matches_oracle(capi, oracle):
    """16x16 grid SSAA (256 Scene::trace calls per pixel; the reference's menu goes to 256x256, Pulse.cpp:22-34) at 160x120 against
    the oracle; and the same frame with a cap that splits it into 5 launches."""
    W, H, refl, s, seed = 160, 120, 12, 16, 31
    cam = S.default_camera()
    o = oracle.OracleRender(S.default_scene(), W, H, seed=seed).render(cam, refl, s)
    orgbf, oargb = o.resolve()
    c = _ctx(capi, S.default_scene(), W, H, seed)
    try:
        c.stats_reset()
        c.render(cam, refl, s)
        rgbf, argb = c.read_rgbf(), c.read_argb()
        st = c.stats()
        assert st["rays"] == o.counters["rays"] and st["samples"] == W * H * s * s
        assert c.get_seeds()[0] == int(o.seeds[0])
        print("16x16 SSAA:", cases.assert_parity(argb, oargb, "ssaa16"))
        assert np.max(np.abs(rgbf - orgbf)) < 2e-5
        c.set_seeds(seed, seed)
        c.set_option("max_calls_per_launch", 1_000_000)      # 3 rows of 160 pixels x 256 calls per launch... whole rows: 24 rows
        c.stats_reset()
        c.render(cam, refl, s)
        assert c.stats()["launches_small_fast"] >= 5
        assert np.array_equal(c.read_rgbf().view(np.uint32), rgbf.view(np.uint32))
    finally:
        c.close()


@pytest.mark.parametrize("path", [1, 2], ids=["constbank", "blob"])
@pytest.mark.parametrize("s,size", [(128, (16, 12)), (256, (8, 6))])
def test_showcase_ssaa_factors_match_oracle(capi, oracle, s, size, path):
    """The reference README's showcase is a 128x128-SSAA screenshot and Pulse's menu goes to 256x256 (Pulse.cpp:22-34): 16 384 and
    65 536 Scene::trace calls per pixel, summed in the reference's ssx-outer / ssy-inner order.  A tiny image keeps the oracle in
    seconds; with the launch cap at 2^20 calls the 8x6 frame at s = 256 is three chunks of rows."""
    W, H = size
    refl, seed = 10, 77
    cam = S.default_camera()
    o = oracle.OracleRender(S.default_scene(), W, H, seed=seed).render(cam, refl, s)
    orgbf, oargb = o.resolve()
    c = _ctx(capi, S.default_scene(), W, H, seed)
    try:
        c.force_path(path)
        c.set_option("max_calls_per_launch", 1 << 20)
        c.stats_reset()
        c.render(cam, refl, s)
        st = c.stats()
        assert st["samples"] == W * H * s * s and st["rays"] == o.counters["rays"]
        assert c.get_seeds()[0] == int(o.seeds[0])
        cases.assert_parity(c.read_argb(), oargb, "ssaa %d" % s)
        assert np.max(np.abs(c.read_rgbf() - orgbf)) < 2e-5
    finally:
        c.close()


# ---------------------------------------------------------------------------------------------- advisor findings (round 1)
def test_resize_then_read_then_batch_does_not_overrun_frame_slots(capi):
    """ADVICE r1 (medium): render_frames at size A, set_image_size(B > A), read_argb, render_frames at B used to leave two of
    the three staging slots at size A.  Now the read path has its own buffer; the frames must equal a fresh context's."""
    cams = S.orbit_cameras(7)[:5]
    c = _ctx(capi, S.default_scene(), 64, 48, 9)
    fresh = _ctx(capi, S.default_scene(), 200, 120, 9)
    try:
        a = c.render_frames(cams, 6)
        c.set_image_size(200, 120)
        c.render(cams[0], 6)
        c.read_argb()
        c.set_seeds(9, 9)
        got = c.render_frames(cams, 6)
        want = fresh.render_frames(cams, 6)
        assert np.array_equal(got, want)
        assert a.shape == (5, 48, 64)
    finally:
        c.close(); fresh.close()


@pytest.mark.parametrize("path", [1, 2], ids=["constbank", "blob"])
def test_unaligned_device_framebuffer(capi, path):
    """ADVICE r1 (low): a caller's ARGB pointer that is 4-byte but not 16-byte aligned must not reach the 128-bit stores."""
    W, H, refl = 64, 40, 6
    cam = S.default_camera()
    scene = S.default_scene() if path == 1 else cases.small_synth()
    c = _ctx(capi, scene, W, H, 3)
    try:
        c.force_path(path)
        want = c.render_frames([cam], refl)[0].copy()
        buf = c.buffer_alloc((W * H + 4) * 4)
        c.set_seeds(3, 3)
        c.stats_reset()
        c.render_frames_device(capi.pack_cameras([cam]), refl, 1, buf + 4)
        c.synchronize()
        st = c.stats()
        # (the blob scenes' wavefront pair stores 4-byte words and takes any frame; its single tile kernel, like the constant-bank
        # fast kernel, stores 128-bit words and hands a misaligned frame to the general kernel)
        assert st["launches_small_fast"] == 0 and (st["launches_blob_fast"] == 0 if path == 1 else st["launches_blob_fast"] > 1), st
        if path == 2:
            c.set_option("blob_wavefront", 0)
            c.set_seeds(3, 3)
            c.stats_reset()
            c.render_frames_device(capi.pack_cameras([cam]), refl, 1, buf + 4)
            c.synchronize()
            st = c.stats()
            assert st["launches_blob_fast"] == 0 and st["launches_blob_any"] == 1, st
        got = c.buffer_read(buf, np.zeros(W * H + 4, np.uint32))
        assert got[0] == 0 and np.array_equal(got[1:1 + W * H].reshape(H, W), want)
        c.buffer_free(buf)
    finally:
        c.close()


def test_bvh_far_camera_tiny_spheres(capi, oracle):
    """ADVICE r1 (low): the BVH boxes must cover the rounding noise of the exact sphere test, which grows with the distance
    between ray origin and sphere and with 1/radius.  Tiny spheres seen from a camera 300 units away through a narrow field of
    view: hierarchy == list walk (image, hit paths, ray counts), both == oracle."""
    rng = np.random.RandomState(5)
    scene = {"ambient": ((0.95, 0.95, 1.0), 0.15), "skybox": None, "textures": [None],
             "lights": [((11.8e9, 4.26e9, 3.08e9), 3.48e8, (1.0, 1.0, 0.95), 0.85)], "objects": []}
    for k in range(48):
        r = float(10 ** rng.uniform(-3.0, -1.0))
        scene["objects"].append(("sphere", (float(rng.uniform(-1.5, 1.5)), r + float(rng.uniform(0, 0.5)), float(rng.uniform(-1.5, 1.5))), r,
                                 S.MT_METAL if k % 2 else S.MT_DIELECTRIC, (0.9, 0.5 + 0.01 * k, 0.3), float(rng.uniform(0, 1)), 0.0))
    scene["objects"].append(("tri", (-3.0, 0.0, -3.0, -3.0, 0.0, 3.0, 3.0, 0.0, -3.0), S.MT_DIELECTRIC, (1.0, 1.0, 1.0), 0.5, 0.0, 0, (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
    scene["objects"].append(("tri", (3.0, 0.0, 3.0, 3.0, 0.0, -3.0, -3.0, 0.0, 3.0), S.MT_DIELECTRIC, (1.0, 1.0, 1.0), 0.5, 0.0, 0, (1.0, 1.0, 1.0, 0.0, 0.0, 1.0)))
    W, H, refl = 192, 128, 8
    cams = [S.camera_lookat((240.0, 150.0, -100.0), (0.0, 0.2, 0.0), 0.014), S.camera_lookat((3.0, 1.0, -2.0), (0.0, 0.1, 0.0), 0.9)]
    res = {}
    for mode in (1, 2):
        c = _ctx(capi, scene, W, H, 11)
        try:
            c.force_path(2); c.set_bvh_mode(mode); c.enable_signatures(True); c.stats_reset()
            frames = []
            for cam in cams:
                c.render(cam, refl)
                frames.append((c.read_rgbf().view(np.uint32).copy(), c.read_signatures().copy()))
            res[mode] = (frames, c.stats()["rays"])
            c.enable_signatures(False)
            c.set_seeds(11, 11)
            batch = c.render_frames(cams, refl)      # the pair-node walk of the batch kernel
            res[(mode, "batch")] = batch.copy()
        finally:
            c.close()
    assert res[1][1] == res[2][1]
    for (f1, s1), (f2, s2) in zip(res[1][0], res[2][0]):
        assert np.array_equal(f1, f2) and np.array_equal(s1, s2)
    assert np.array_equal(res[(1, "batch")], res[(2, "batch")])
    o = oracle.OracleRender(scene, W, H, seed=11)
    for k, cam in enumerate(cams):
        o.render(cam, refl, want_sig=True)
        assert np.array_equal(res[1][0][k][1], o.sig)
        cases.assert_parity(res[(1, "batch")][k], o.resolve()[1], "far camera frame %d" % k)
