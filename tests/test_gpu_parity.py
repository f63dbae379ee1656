"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against
  (1) the golden vectors generated from the unmodified reference (committed fixtures),
  (2) the CPU oracle on the same seeded inputs at sizes it finishes in seconds,
  (3) the unmodified reference's config-2 frame, identified by its stored hash.
Bar (BASELINE.json): <= 1 LSB/channel on >= 99.9 % of pixels, none > 4 LSB.  The only arithmetic that may differ is
powf (CUDA vs glibc); everything else is expected to be identical, so we also require identical hit-path signatures
and report the exact-match fraction."""
import hashlib

import numpy as np
import pytest

import cases
from reflaxman_b200 import scenes as S

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi(rfx_lib):
    from reflaxman_b200 import capi
    return capi


@pytest.mark.parametrize("path", [1, 2], ids=["constbank", "blob"])
@pytest.mark.parametrize("name", cases.GOLDEN)
def test_gpu_matches_golden(capi, name, path):
    """both K2 variants: 1 = constant-bank kernel (small scenes), 2 = general blob kernel (any scene)"""
    g = cases.load_golden(name)
    eng = cases.GpuEngine(capi, g["scene"], g["W"], g["H"], g["seed"])
    eng.c.force_path(path)
    try:
        frames = cases.replay(eng, g)
        for i, (rgbf, argb) in enumerate(frames):
            st = cases.assert_parity(argb, g["argb%d" % i], "%s frame %d" % (name, i))
            # float image: identical up to powf rounding (<= a few ulp of a colour contribution)
            if "rgbf%d" % i in g:
                assert np.max(np.abs(rgbf - g["rgbf%d" % i])) < 2e-5, name
            assert st["frac_exact"] > 0.995, (name, st)
    finally:
        eng.close()


@pytest.mark.parametrize("chunk", [1, 777, 4096])
def test_render_next_slicing_is_invisible(capi, chunk):
    """renderNext(pixels) in arbitrary slices == one full-frame call (reference Render.cpp:198-211 cursor)."""
    scene = S.default_scene()
    cam = S.default_camera()
    a = cases.GpuEngine(capi, scene, 80, 60, 99)
    b = cases.GpuEngine(capi, scene, 80, 60, 99, chunk=chunk)
    try:
        for samples in (1, 2, -3):
            a.render(cam, 8, samples, False)
            b.render(cam, 8, samples, False)
            assert np.array_equal(a.read()[0].view(np.uint32), b.read()[0].view(np.uint32)), samples
        assert a.c.get_seeds() == b.c.get_seeds()
    finally:
        a.close(); b.close()


@pytest.mark.parametrize("path", [1, 2], ids=["constbank", "blob"])
def test_signatures_and_rays_match_oracle_config1(capi, oracle, path):
    """config 1 (1024x768, depth 20): identical hit paths on 100 % of pixels, identical ray count, parity bar met."""
    W, H = 1024, 768
    cam = S.default_camera()
    o = oracle.OracleRender(S.default_scene(), W, H, seed=12345).render(cam, 20, want_sig=True)
    _, oargb = o.resolve()
    c = capi.Context(0)
    try:
        c.load_scene(S.default_scene()); c.set_seeds(12345, 12345); c.set_image_size(W, H)
        c.force_path(path)
        c.enable_signatures(True)
        c.stats_reset()
        c.render(cam, 20)
        argb = c.read_argb()
        sig = c.read_signatures()
        st = c.stats()
        assert np.array_equal(sig, o.sig), "hit-path signatures differ on %d pixels" % int((sig != o.sig).sum())
        assert st["rays"] == o.counters["rays"] and st["bounces"] == o.counters["bounces"]
        cases.assert_parity(argb, oargb, "config 1")
        assert c.get_seeds()[0] == int(o.seeds[0])
    finally:
        c.close()


def test_gpu_vs_reference_binary_config2(capi, oracle):
    """config 2 (1920x1080, depth 20, seed 12345) against the unmodified reference's frame: the oracle's frame hashes to the
    reference's (tests/golden/full_size_sha256.txt), so it is that frame, bit for bit."""
    W, H = 1920, 1080
    ref_hash = cases.full_size_hashes()["default_%dx%d_d20_seed12345" % (W, H)][0]
    _, ref_argb = oracle.OracleRender(S.default_scene(), W, H, seed=12345).render(S.default_camera(), 20).resolve()
    assert hashlib.sha256(ref_argb.tobytes()).hexdigest() == ref_hash
    c = capi.Context(0)
    try:
        c.load_scene(S.default_scene()); c.set_seeds(12345, 12345); c.set_image_size(W, H)
        c.render(S.default_camera(), 20)
        st = cases.assert_parity(c.read_argb(), ref_argb, "config 2 vs reference")
        print("config 2 parity:", st)
    finally:
        c.close()


def test_batch_frames_continue_the_stream(capi, oracle):
    """rfx_render_frames over a camera path == the oracle rendering the same frames in one process (stream
    continues from frame to frame); and a context that skips ahead reproduces a later frame (frame sharding)."""
    W, H, refl = 96, 54, 20
    cams = S.orbit_cameras(12)[:5]
    o = oracle.OracleRender(S.default_scene(), W, H, seed=2024)
    want = [o.render(cam, refl).resolve()[1] for cam in cams]
    c = capi.Context(0)
    d = capi.Context(0)
    try:
        for ctx in (c, d):
            ctx.load_scene(S.default_scene()); ctx.set_seeds(2024, 2024); ctx.set_image_size(W, H)
        got = c.render_frames(cams, refl)
        for i in range(len(cams)):
            cases.assert_parity(got[i], want[i], "batch frame %d" % i)
        d.skip_samples(3 * W * H)
        late = d.render_frames(cams[3:], refl)
        assert np.array_equal(late[0], got[3]) and np.array_equal(late[1], got[4])
    finally:
        c.close(); d.close()


def test_error_behaviour(capi):
    c = capi.Context(0)
    try:
        with pytest.raises(capi.RfxError):
            c.render_begin(20)                 # no image size yet
        c.set_image_size(8, 8)
        with pytest.raises(capi.RfxError):
            c.render_begin(0)                  # reflectNum must be > 0 (reference asserts, Render.cpp:118)
        with pytest.raises(capi.RfxError):
            c.render_begin(5, 0)               # sampleNum != 0 (Render.cpp:119)
        assert c.render_next(10) is False      # not in progress -> false (Render.cpp:143-144)
        c.load_scene(S.default_scene())
        c.set_camera(S.default_camera())
        c.render_begin(3)
        assert c.render_next(10) is True and abs(c.progress() - 100.0 * 10 / 64) < 1e-4
        assert c.render_next(1000) is False and c.progress() == 100.0 and not c.in_progress()
        assert np.array_equal(c.read_pixel(-1, 0), np.zeros(3, np.float32))   # Render.cpp:112-113
    finally:
        c.close()


@pytest.mark.parametrize("n_side,size,depth", [(6, (128, 72), 8), (12, (160, 90), 6), (32, (96, 54), 4)])
def test_bvh_equals_brute_force(capi, oracle, n_side, size, depth):
    """SURVEY f-3: the bounding-volume hierarchy of the general blob kernel only selects which spheres get the exact test;
    the float image, the hit-path signatures and the ray counts must be IDENTICAL to the brute-force list walk, and both
    must meet the parity bar against the oracle."""
    W, H = size
    scene = S.synthetic_scene(n_side, floor=S.synthetic_texture(64, 64, 3), skybox=S.synthetic_texture(128, 96, 5))
    cams = [S.default_camera(), S.orbit_cameras(7)[3]]
    out = {}
    for mode in (2, 1):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(321, 321); c.set_image_size(W, H)
            c.force_path(2); c.set_bvh_mode(mode); c.enable_signatures(True); c.stats_reset()
            frames = []
            for cam in cams:
                c.render(cam, depth)
                frames.append((c.read_rgbf(), c.read_argb(), c.read_signatures()))
            out[mode] = (frames, c.stats()["rays"], c.get_seeds())
        finally:
            c.close()
    assert out[1][1] == out[2][1] and out[1][2] == out[2][2]
    for (f1, a1, s1), (f2, a2, s2) in zip(out[1][0], out[2][0]):
        assert np.array_equal(f1.view(np.uint32), f2.view(np.uint32))
        assert np.array_equal(s1, s2)
    o = oracle.OracleRender(scene, W, H, seed=321)
    for k, cam in enumerate(cams):
        o.render(cam, depth, want_sig=True)
        assert np.array_equal(out[1][0][k][2], o.sig)
        cases.assert_parity(out[1][0][k][1], o.resolve()[1], "bvh frame %d" % k)


@pytest.mark.parametrize("which,size,depth,bvh", [("grid6", (128, 72), 8, 1), ("grid12", (161, 90), 6, 0), ("grid12", (160, 91), 6, 2),
                                                   ("mixed", (250, 131), 12, 0), ("mixed", (64, 40), 12, 1), ("grid2", (64, 40), 6, 1)])
def test_blob_batch_kernel_equals_general_blob_kernel(capi, oracle, which, size, depth, bvh):
    """rfx_trace_blob.cu (state machine, shared-memory traversal stack; row-aligned one-sample ARGB slices of blob scenes: as the
    wavefront kernel pair and as the single tile kernel) against
    k_trace: identical frames, ray counts and stream position, with and without the hierarchy, widths that are not a multiple of
    the tile width, heights that are not a multiple of the tile height, a hierarchy whose root is a leaf (4 spheres); and both meet the
    parity bar against the oracle."""
    W, H = size
    scene = _mixed_scene() if which == "mixed" else S.synthetic_scene(int(which[4:]), floor=S.synthetic_texture(64, 64, 3), skybox=S.synthetic_texture(128, 96, 5))
    cams = [S.default_camera(), S.orbit_cameras(7)[3]]
    out = {}
    for path, wave in ((2, 2), (2, 0), (3, 0)):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(99, 99); c.set_image_size(W, H)
            c.force_path(path); c.set_bvh_mode(bvh); c.set_option("blob_wavefront", wave); c.stats_reset()
            frames = c.render_frames(cams, depth)
            st = c.stats()
            # the wavefront (two segments in tiles, the rest in the queue-driven kernel) is two launches per frame, the tile kernel one
            assert st["launches_blob_fast"] == (0 if path == 3 else len(cams) * (2 if wave else 1)), st
            out[(path, wave)] = (frames.copy(), st["rays"], st["bounces"], c.get_seeds())
        finally:
            c.close()
    for key in ((2, 0), (3, 0)):
        assert np.array_equal(out[(2, 2)][0], out[key][0]), key
        assert out[(2, 2)][1:] == out[key][1:], key
    out = {2: out[(2, 2)], 3: out[(3, 0)]}
    o = oracle.OracleRender(scene, W, H, seed=99)
    rays = 0
    for k, cam in enumerate(cams):
        o.render(cam, depth)
        rays += o.counters["rays"]
        cases.assert_parity(out[2][0][k], o.resolve()[1], "blob batch kernel frame %d" % k)
    assert out[2][1] == rays


@pytest.mark.parametrize("case", range(6))
def test_wavefront_pair_randomized_against_tile_and_general_kernels(capi, case):
    """The wavefront pair (k_blob_wave_first + k_blob_wave_rest) on seeded random scenes, sizes and depths — odd sizes, scenes in which
    every path ends in its first segments (empty queue), a scene without a hierarchy (list walk), a sky-less box of mirrors in which no
    path ends early (every pixel queued), depth exactly at the wavefront's threshold — for every number of tile segments: frames, ray
    counts and stream positions identical to the single tile kernel and to the general kernel."""
    rng = np.random.RandomState(100 + case)
    W, H = int(rng.randint(33, 200)), int(rng.randint(9, 120))
    depth = [4, 5, 7, 12, 20, 4][case]
    if case == 1:      # nothing to hit: every path ends at the sky in its first segment
        scene = {"ambient": ((0.9, 0.9, 1.0), 0.2), "skybox": S.synthetic_texture(64, 48, 2), "textures": [], "lights": [((5.0e9, 4.0e9, 3.0e9), 1.0e8, (1.0, 1.0, 1.0), 0.8)],
                 "objects": [("sphere", (100.0 + k, 0.0, 0.0), 0.5, S.MT_METAL, (1.0, 1.0, 1.0), 1.0, 0.0) for k in range(40)]}
    elif case == 3:    # closed box of perfect mirrors around the camera: no path ends before the depth limit
        scene = {"ambient": ((1.0, 1.0, 1.0), 0.1), "skybox": None, "textures": [], "lights": [((0.0, 0.5, 0.0), 0.05, (1.0, 0.9, 0.8), 1.0)], "objects": []}
        c = [(-9.0, -9.0, -9.0), (9.0, -9.0, -9.0), (9.0, 9.0, -9.0), (-9.0, 9.0, -9.0), (-9.0, -9.0, 9.0), (9.0, -9.0, 9.0), (9.0, 9.0, 9.0), (-9.0, 9.0, 9.0)]
        for q in ((0, 1, 2, 3), (5, 4, 7, 6), (4, 0, 3, 7), (1, 5, 6, 2), (3, 2, 6, 7), (4, 5, 1, 0)):
            for t in ((q[0], q[1], q[2]), (q[0], q[2], q[3]), (q[0], q[2], q[1]), (q[0], q[3], q[2])):     # both windings: one of them faces inward
                scene["objects"].append(("tri", c[t[0]] + c[t[1]] + c[t[2]], S.MT_METAL, (1.0, 1.0, 1.0), 1.0, 0.0, -1, (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
        for k in range(40):
            scene["objects"].append(("sphere", tuple(float(v) for v in rng.uniform(-6, 6, 3)), float(rng.uniform(0.3, 1.2)), S.MT_METAL, (1.0, 1.0, 1.0), 1.0, 0.0))
    else:
        scene = S.synthetic_scene(int(rng.randint(6, 14)), floor=S.synthetic_texture(64, 64, 3 + case), skybox=S.synthetic_texture(128, 96, 5))
    cams = [S.default_camera(), S.orbit_cameras(11)[int(rng.randint(1, 10))]] if case != 3 else [S.camera_lookat((0.5, 0.2, -0.3), (3.0, 1.0, 2.0), 1.2)] * 2
    out = {}
    for key, path, wave, bvh in (("wave1", 2, 1, 1), ("wave2", 2, 2, 1), ("wave3", 2, 3, 1), ("wave2+L1", 2, 2, 1), ("wave2+list", 2, 2, 2), ("tile", 2, 0, 1), ("general", 3, 0, 1)):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(1000 + case, 7); c.set_image_size(W, H)
            c.force_path(path); c.set_bvh_mode(bvh); c.set_option("blob_wavefront", wave); c.set_option("blob_smem_bvh", 0 if key.endswith("L1") else 1)
            c.stats_reset()
            frames = c.render_frames(cams, depth)
            st = c.stats()
            if key.startswith("wave"):
                assert st["launches_blob_fast"] == (2 * len(cams) if depth > wave else len(cams)), (key, st)
            out[key] = (frames.copy(), st["rays"], st["bounces"], c.get_seeds())
        finally:
            c.close()
    for key, got in out.items():
        assert np.array_equal(got[0], out["general"][0]), (case, key)
        assert got[1:] == out["general"][1:], (case, key)


def test_blob_batch_kernel_float_image_equals_general_blob_kernel(capi):
    """Render API (float image) on a blob scene: whole frames and row-aligned chunks go to rfx_trace_blob.cu, ragged chunks to k_trace;
    the float images are bit-identical to k_trace rendering everything."""
    W, H, depth = 136, 75, 6
    scene = S.synthetic_scene(8, floor=S.synthetic_texture(64, 64, 3), skybox=S.synthetic_texture(128, 96, 5))
    cam = S.orbit_cameras(5)[1]
    out = {}
    for path, chunk in ((3, None), (2, None), (2, W * 16), (2, 1000)):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(5, 5); c.set_image_size(W, H)
            c.force_path(path); c.set_bvh_mode(1); c.stats_reset()
            c.render(cam, depth, chunk=chunk)
            out[(path, chunk)] = (c.read_rgbf().view(np.uint32).copy(), c.read_argb().copy(), c.stats()["rays"], c.get_seeds())
        finally:
            c.close()
    ref = out[(3, None)]
    for key, got in out.items():
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]) and got[2:] == ref[2:], key


def _edge_case(case):
    if case == "empty":          # nothing to hit, nothing to light: every ray goes to the skybox
        scene = {"ambient": ((0.95, 0.95, 1.0), 0.15), "skybox": S.synthetic_texture(128, 96, 5), "textures": [], "lights": [], "objects": []}
        return scene, 37, 5, 3, 1
    if case in ("constbank_full", "constbank_plus_one"):
        # every array of the constant-bank scene at its capacity (16 spheres, 8 triangles, 2 planes, 4 lights) / one sphere more
        # (the scene no longer fits and goes to the blob kernels, list walk)
        scene = _mixed_scene()
        for k in range(7 if case == "constbank_full" else 8):
            scene["objects"].append(("sphere", (-4.0 + 1.1 * k, 0.35, -4.5 + 0.3 * k), 0.35, S.MT_METAL if k % 2 else S.MT_DIELECTRIC,
                                     (0.4 + 0.07 * k, 0.9 - 0.05 * k, 0.6), 0.1 * k, 0.0))
        for k in range(5):
            scene["objects"].append(("tri", (-5.0 + 2.0 * k, 0.0, 4.0, -5.0 + 2.0 * k, 1.5, 4.0, -4.0 + 2.0 * k, 0.0, 4.0), S.MT_DIELECTRIC,
                                     (0.9, 0.8 - 0.1 * k, 0.3), 0.5, 0.0, -1, (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
        scene["objects"].append(("plane", (0.0, 12.0, 0.0), (0.0, -1.0, 0.0), S.MT_METAL, (0.5, 0.5, 0.6), 0.2, 0.0))
        return scene, 96, 54, 10, 1
    scene = S.default_scene()
    scene["lights"] = []         # ambient only: no shadow rays at all
    return (scene, 1, 1, 20, 1) if case == "nolight_1x1" else (scene, 1, 67, 20, 2)


@pytest.mark.parametrize("case", ["empty", "nolight_1x1", "nolight_1x67_ss2", "constbank_full", "constbank_plus_one"])
def test_edge_cases_match_oracle(capi, oracle, case):
    """Empty scene, no lights, a single pixel, an image one pixel wide with 2x2 SSAA (tiles hang over three edges), the constant-bank scene at
    capacity and one sphere past it: every kernel
    (constant-bank general and fast, blob batch, blob general) against the oracle, with identical ray counts and stream position."""
    scene, W, H, depth, samples = _edge_case(case)
    cam = S.default_camera()
    o = oracle.OracleRender(scene, W, H, seed=7).render(cam, depth, samples)
    _, oargb = o.resolve()
    for path in (1, 2, 3):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(7, 7); c.set_image_size(W, H)
            c.force_path(path); c.stats_reset()
            c.render(cam, depth, samples)
            argb = c.read_argb()
            st = c.stats()
            assert st["rays"] == o.counters["rays"] and st["bounces"] == o.counters["bounces"], (case, path)
            assert c.get_seeds()[0] == int(o.seeds[0]), (case, path)
            cases.assert_parity(argb, oargb, "%s, kernel %d" % (case, path))
            c.set_seeds(7, 7)
            batch = c.render_frames([cam], depth, samples)[0]      # ARGB-only batch path (fast kernels)
            assert np.array_equal(batch, argb), (case, path)
        finally:
            c.close()


def _mixed_scene():
    """Everything the state machine has to get right at once: three lights (one near the scene, one behind most surfaces,
    one with zero power), nine spheres (an odd count: the pairwise sphere loop has a remainder), a vertical wall, a plane
    (unreachable through the reference's Scene but part of the C ABI), textured floor and skybox."""
    s = S.default_scene(skybox=S.synthetic_texture(256, 192, 5), floor=S.synthetic_texture(64, 64, 9))
    s["objects"].insert(3, ("sphere", (3.0, 0.8, 2.5), 0.8, S.MT_DIELECTRIC, (0.9, 0.3, 0.3), 0.6, 0.0))
    s["objects"].append(("tri", (-6.0, 0.0, 5.0, -6.0, 4.0, 5.0, 6.0, 0.0, 5.0), S.MT_METAL, (0.8, 0.8, 1.0), 0.7, 0.0, -1,
                         (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
    s["objects"].append(("plane", (0.0, 0.0, 9.0), (0.0, 0.0, -1.0), S.MT_DIELECTRIC, (0.4, 0.5, 0.4), 0.3, 0.0))
    s["lights"].append(((2.0, 6.0, -4.0), 0.5, (1.0, 0.6, 0.4), 0.4))            # inside the scene's bounding box
    s["lights"].append(((-5.0e9, -3.0e9, 1.0e9), 2.0e8, (0.3, 0.3, 1.0), 0.3))   # below the floor: faces almost nothing
    s["lights"].append(((0.0, 9.0e9, 0.0), 1.0e8, (1.0, 1.0, 1.0), 0.0))         # zero power: shadow rays are still cast
    return s


def test_mixed_scene_all_kernels_match_oracle(capi, oracle):
    """fast kernel (ARGB batch path), general constant-bank kernel and blob kernel on a scene with several lights
    and every object kind: identical hit paths and ray counts to the oracle, identical images to each other."""
    W, H, refl, seed = 250, 131, 12, 4242
    cam = S.orbit_cameras(7)[2]
    scene = _mixed_scene()
    o = oracle.OracleRender(scene, W, H, seed=seed).render(cam, refl, want_sig=True)
    _, oargb = o.resolve()
    images = {}
    for path in (1, 2):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(seed, seed); c.set_image_size(W, H)
            c.force_path(path)
            c.enable_signatures(True)
            c.stats_reset()
            c.render(cam, refl)
            images[path] = c.read_argb()
            assert np.array_equal(c.read_signatures(), o.sig), "kernel %d: hit paths differ" % path
            st = c.stats()
            assert st["rays"] == o.counters["rays"] and st["bounces"] == o.counters["bounces"], path
            cases.assert_parity(images[path], oargb, "mixed scene, kernel %d" % path)
        finally:
            c.close()
    assert np.array_equal(images[1], images[2])
    c = capi.Context(0)
    try:
        c.load_scene(scene); c.set_seeds(seed, seed); c.set_image_size(W, H)
        c.stats_reset()
        fast = c.render_frames([cam], refl)[0]          # ARGB-only batch path -> k_trace_small (2-D grid fast kernel)
        assert np.array_equal(fast, images[1])
        assert c.stats()["rays"] == o.counters["rays"]
    finally:
        c.close()


def test_fast_kernel_equals_general_kernel_full_size(capi):
    """config 2 size: the division-free fast kernel and the general kernel produce the same 1920x1080 frame bit for bit."""
    W, H = 1920, 1080
    cam = S.default_camera()
    a = capi.Context(0)
    b = capi.Context(0)
    try:
        for c in (a, b):
            c.load_scene(S.default_scene()); c.set_seeds(12345, 12345); c.set_image_size(W, H)
        a.render(cam, 20)
        got = b.render_frames([cam], 20)[0]
        assert np.array_equal(a.read_argb(), got)
        assert a.stats()["rays"] == b.stats()["rays"]
    finally:
        a.close(); b.close()


def test_tile_ordering_does_not_change_results(capi):
    """Cost-ordered tile scheduling only permutes which CTA renders which tile group: frames rendered with the history of the
    previous launch (recorded on every launch, on every 2nd, on every 8th — the launches in between replay the last recording),
    without it, and across an image-size change (history dropped) are bit-identical."""
    cams = S.orbit_cameras(9)[:6]
    frames = {}
    for key, on, period in (("every", True, 1), ("every2nd", True, 2), ("default", True, None), ("off", False, None)):
        c = capi.Context(0)
        try:
            c.load_scene(S.default_scene()); c.set_seeds(77, 77)
            c.set_tile_ordering(on)
            if period:
                c.set_option("tile_order_period", period)
            c.set_image_size(200, 120)
            a = c.render_frames(cams, 20)            # frame 0 in index order, the others in a recorded order
            c.set_image_size(136, 96)                # different grid: the history must not be reused
            b = c.render_frames(cams[:2], 20)
            c.set_image_size(200, 120)
            d = c.render_frames(cams[:1], 20)
            frames[key] = (a, b, d, c.stats()["rays"])
        finally:
            c.close()
    for key in ("every", "every2nd", "default"):
        for x, y in zip(frames[key][:3], frames["off"][:3]):
            assert np.array_equal(x, y), key
        assert frames[key][3] == frames["off"][3], key


def _lcg_state_at(position):
    """state of the reference's LCG (trace_math.h:36-39) `position` steps after state 0"""
    a, c, s, n = 214013, 2531011, 0, position
    while n:
        if n & 1:
            s = (a * s + c) & 0xFFFFFFFF
        c = (c * (a + 1)) & 0xFFFFFFFF
        a = (a * a) & 0xFFFFFFFF
        n >>= 1
    return s


@pytest.mark.parametrize("back", [3001, 3002, 3003])
def test_random_stream_across_the_lcg_cycle_wrap(capi, oracle, back):
    """K1 ranks the stream from a table over the LCG's 2^32-state cycle; a stream that starts just before the end of the cycle
    changes residue class when the position wraps.  Two frames from such a seed (all three classes), and a context that skips
    the first frame, against the oracle's serial LCG."""
    W, H, refl = 64, 48, 6
    seed = _lcg_state_at((1 << 32) - back)
    cams = S.orbit_cameras(5)[:2]
    o = oracle.OracleRender(S.default_scene(), W, H, seed=seed)
    want = [o.render(cam, refl).resolve()[1] for cam in cams]
    c = capi.Context(0)
    d = capi.Context(0)
    try:
        for ctx in (c, d):
            ctx.load_scene(S.default_scene()); ctx.set_seeds(seed, seed); ctx.set_image_size(W, H)
        got = c.render_frames(cams, refl)
        for i in range(2):
            cases.assert_parity(got[i], want[i], "wrap frame %d" % i)
        assert c.get_seeds()[0] == int(o.seeds[0])
        d.skip_samples(W * H)
        late = d.render_frames(cams[1:], refl)
        assert np.array_equal(late[0], got[1])
        assert d.get_seeds()[0] == c.get_seeds()[0]
    finally:
        c.close(); d.close()


def test_k1_accept_test_equals_reference_expression_on_the_whole_lcg_cycle(capi):
    """K1 decides acceptance of a draw-triple with an integer test and evaluates the reference's float expression only inside a guard
    band around the unit sphere's surface; rfx_selftest_rng runs both on all 4.29e9 triples of the LCG's cycle: no disagreement."""
    c = capi.Context(0)
    try:
        differ, band = c.selftest_rng()
        assert differ == 0, "%d triples decided differently from the reference's float expression" % differ
        assert 1000 < band < 1_000_000, band         # the band exists and is thin (~3e-6 of the triples)
    finally:
        c.close()


def test_stream_skip_matches_serial_stream(capi, oracle):
    """rfx_skip_samples finds the end of the skipped stretch in the table of the LCG cycle (one small kernel whatever n is):
    the resulting stream state equals the oracle's serial walk, skips compose, and a skip longer than a whole residue class
    of the cycle (chunked by the host) equals the same distance in pieces."""
    seed = 20260101
    n = 3_000_000
    _, end_state = oracle.rand_dirs(seed, n)
    c = capi.Context(0)
    d = capi.Context(0)
    try:
        c.set_seeds(seed, 1); d.set_seeds(seed, 1)
        c.skip_samples(n)
        assert c.get_seeds()[0] == end_state
        for part in (1, 999_999, 2_000_000):
            d.skip_samples(part)
        assert d.get_seeds()[0] == end_state
        big = 1_700_000_000                       # > 0.75e9 accepted triples of one residue class: crosses the cycle wrap at least twice
        c.skip_samples(big)
        for _ in range(17):
            d.skip_samples(100_000_000)
        assert c.get_seeds()[0] == d.get_seeds()[0]
    finally:
        c.close(); d.close()


def _primary_proto():
    import os
    import sys
    tools = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools")
    if tools not in sys.path:
        sys.path.insert(0, tools)
    import primary_cull_proto
    return primary_cull_proto


@pytest.mark.parametrize("which", ["default", "mixed"])
def test_primary_bounds_are_conservative(capi, which):
    """The fast kernel lets a warp's first pass over the objects skip what its 4x8 tile cannot see: per launch the library bounds, for
    every sphere and triangle, the pixels whose primary ray can pass that object's test.  For cameras all over the place (orbit, inside
    spheres, under the floor, looking away, fov 0.3..2.6) the accept expressions of Sphere.cpp:49-57 / Triangle.cpp:56-68, evaluated in
    float32 op for op on every pixel (and on the far corner of its SSAA / jitter footprint), never accept outside the rectangle."""
    P = _primary_proto()
    scene = S.default_scene() if which == "default" else _mixed_scene()
    sph, tris = P.scene_arrays(scene)
    W, H = 320, 180
    c = capi.Context(0)
    try:
        c.load_scene(scene); c.set_image_size(W, H)
        culled = 0
        for eye, view, fov in P.random_cameras(60, 11 if which == "default" else 12, sph):
            c.set_camera((eye, view, fov))
            srect, trect = c.selftest_primary_bounds()
            assert len(srect) == len(sph) and len(trect) == len(tris)
            P.assert_inside(eye, view, fov, W, H, sph, tris, srect, trect)
            culled += sum(1 for r in list(srect) + list(trect) if r[0] > 0 or r[1] < W - 1 or r[2] > 0 or r[3] < H - 1)
        assert culled > 100, culled          # the bounds do exclude something (they are not all "whole image")
    finally:
        c.close()


@pytest.mark.parametrize("which", ["default", "mixed"])
def test_primary_cull_leaves_every_frame_identical(capi, which):
    """Frames of the fast kernel (tiles skip the objects outside their primary bounds) against the general kernel (signature run:
    every query sees every object) for the same cameras: identical ARGB, identical ray counts; the same with 2x2 SSAA through the
    Render API (the MULTI instantiation shares the tile's answer between the sub-samples)."""
    P = _primary_proto()
    scene = S.default_scene() if which == "default" else _mixed_scene()
    sph, _ = P.scene_arrays(scene)
    W, H = 200, 120
    cams = P.random_cameras(28, 21, sph)
    a = capi.Context(0)
    b = capi.Context(0)
    try:
        for c in (a, b):
            c.load_scene(scene); c.set_seeds(5, 5); c.set_image_size(W, H)
        b.enable_signatures(True)
        fast = a.render_frames(cams, 12)
        st = a.stats()
        assert st["launches_small_fast"] == len(cams) and st["launches_small_any"] == 0, st
        for k, cam in enumerate(cams):
            b.render(cam, 12)
            assert np.array_equal(b.read_argb(), fast[k]), "camera %d" % k
        assert a.stats()["rays"] == b.stats()["rays"]
        b.enable_signatures(False)
        for cam in cams[::5]:
            a.render(cam, 6, samples=2)
            b.enable_signatures(True)
            b.render(cam, 6, samples=2)
            b.enable_signatures(False)
            assert np.array_equal(a.read_argb(), b.read_argb())
    finally:
        a.close(); b.close()


def _with_lights(scene, lights):
    out = dict(scene)
    out["lights"] = lights
    return out


@pytest.mark.parametrize("case", ["far", "overhead", "grazing", "far+near", "near", "two_far"])
def test_light_grid_equals_hierarchy_walk(capi, case):
    """Scenes with a sphere hierarchy answer the shadow queries of far lights from a grid of candidate spheres across the light's
    direction (rfx_capi.cu buildLightGrid) instead of walking the hierarchy.  The query is an any-hit query (Scene.cpp:131-143), so
    a complete candidate list gives the same answer: frames, ray counts and the stream position are identical with the grids
    on and off — far light (config 4's), straight overhead, grazing (long shadows), a far and a near light together (the near
    one keeps the hierarchy), near light only (no grid), two far lights; tile kernel, wavefront pair and general kernel."""
    far = ((11.8e9, 4.26e9, 3.08e9), 3.48e8, (1.0, 1.0, 0.95), 0.85)
    lights = {
        "far": [far],
        "overhead": [((0.0, 5.0e6, 0.0), 2.0e5, (1.0, 0.9, 0.8), 0.9)],
        "grazing": [((-4.0e5, 1.5e4, 2.0e5), 6.0e3, (0.9, 1.0, 1.0), 0.8)],
        "far+near": [far, ((2.0, 6.0, -1.0), 0.5, (1.0, 0.6, 0.4), 0.6)],
        "near": [((2.0, 6.0, -1.0), 0.5, (1.0, 0.6, 0.4), 0.6)],
        "two_far": [far, ((-3.0e4, 2.0e4, -1.0e4), 9.0e2, (0.5, 0.6, 1.0), 0.5)],
    }[case]
    expect = {"far": 1, "overhead": 1, "grazing": 1, "far+near": 1, "near": 0, "two_far": 2}[case]
    scene = _with_lights(S.synthetic_scene(16, floor=S.synthetic_texture(64, 64, 3)), lights)
    W, H = 192, 108
    cams = [S.default_camera(), S.camera_lookat((3.0, 0.8, 2.0), (-2.0, 0.2, -1.0), 1.3)]
    results = {}
    for on in (1, 0):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(31, 31); c.set_image_size(W, H)
            c.set_option("light_grids", on)
            frames = [c.render_frames(cams, d) for d in (2, 8)]          # tile kernel (depth < 3) and wavefront pair
            st = c.stats()
            assert st["light_grids"] == (expect if on else 0), st
            c.enable_signatures(True)                                      # general kernel
            c.render(cams[1], 5)
            results[on] = (frames, st["rays"], c.read_argb(), c.read_signatures(), c.get_seeds())
        finally:
            c.close()
    for a, b in zip(results[1][0], results[0][0]):
        assert np.array_equal(a, b)
    assert results[1][1] == results[0][1]
    assert np.array_equal(results[1][2], results[0][2]) and np.array_equal(results[1][3], results[0][3])
    assert results[1][4] == results[0][4]


@pytest.mark.parametrize("seed", range(8))
def test_light_grid_random_scenes(capi, seed):
    """Random sphere clouds (stacked, radii over two orders of magnitude, some overlapping) under one to three far lights from random
    directions — from below, along an axis, nearly horizontal — plus a floor: grids on and off give identical frames and ray counts."""
    rng = np.random.default_rng(1000 + seed)
    n = int(rng.integers(40, 200))
    objs = []
    for i in range(n):
        r = float(10 ** rng.uniform(-1.7, 0.2))
        c = rng.uniform([-8, 0, -6], [8, 5, 6])
        objs.append(("sphere", (float(c[0]), float(c[1]) + r, float(c[2])), r, int(i % 2), tuple(float(v) for v in rng.uniform(0.3, 1.0, 3)),
                     float(rng.uniform(0.0, 1.0)), 0.0))
    objs.append(("tri", (-14.0, 0.0, -10.0, -14.0, 0.0, 10.0, 14.0, 0.0, -10.0), S.MT_DIELECTRIC, (1.0, 1.0, 1.0), 0.9, 0.0, -1, (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
    objs.append(("tri", (-14.0, 0.0, 10.0, 14.0, 0.0, 10.0, 14.0, 0.0, -10.0), S.MT_DIELECTRIC, (1.0, 1.0, 1.0), 0.9, 0.0, -1, (0.0, 1.0, 1.0, 1.0, 1.0, 0.0)))
    lights = []
    for k in range(int(rng.integers(1, 4))):
        d = rng.normal(size=3)
        if seed % 4 == 1 and k == 0:
            d = np.array([0.0, 1.0, 0.0])                       # along an axis
        if seed % 4 == 2 and k == 0:
            d = np.array([1.0, 0.02, 0.3])                      # nearly horizontal
        d = d / np.linalg.norm(d)
        dist = float(10 ** rng.uniform(3.0, 9.0))
        lights.append((tuple(float(v) for v in d * dist), dist * float(rng.uniform(0.001, 0.04)), (1.0, 0.9, 0.8), float(rng.uniform(0.3, 0.9))))
    scene = {"ambient": ((0.9, 0.9, 1.0), 0.2), "skybox": None, "textures": [], "lights": lights, "objects": objs}
    cams = [S.default_camera(), S.camera_lookat(tuple(rng.uniform([-10, 0.5, -8], [10, 6, 8])), tuple(rng.uniform([-3, 0, -3], [3, 3, 3])), 1.2)]
    res = {}
    for on in (1, 0):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(9, 9); c.set_image_size(128, 72)
            c.set_bvh_mode(1)
            c.set_option("light_grids", on)
            res[on] = (c.render_frames(cams, 2), c.render_frames(cams, 6), c.stats())
        finally:
            c.close()
    assert res[1][2]["light_grids"] == len(lights) and res[0][2]["light_grids"] == 0
    assert np.array_equal(res[1][0], res[0][0]) and np.array_equal(res[1][1], res[0][1])
    assert res[1][2]["rays"] == res[0][2]["rays"]


@pytest.mark.parametrize("which", ["grid16", "cloud"])
def test_eye_grid_equals_hierarchy_walk(capi, which):
    """Scenes with a sphere hierarchy take the candidates of a path's FIRST query (origin = eye) from a screen grid the host bins per
    camera out of the spheres' primary-ray bounds (rfx_capi.cu buildEyeGrid) instead of walking the hierarchy.  Cameras all over the
    place — orbit, inside spheres, under the floor, looking away, fov 0.3..2.6: frames, ray counts and stream positions are identical
    with the grid on and off; tile kernel (depth 1 and 2), wavefront pair (depth 6), 2x2 SSAA through the Render API, and the general
    kernel on ragged renderNext slices with identical hit-path signatures."""
    P = _primary_proto()
    if which == "grid16":
        scene = S.synthetic_scene(16, floor=S.synthetic_texture(64, 64, 3))
    else:
        rng = np.random.default_rng(77)
        objs = []
        for i in range(150):
            r = float(10 ** rng.uniform(-1.5, 0.3))
            c = rng.uniform([-8, 0, -6], [8, 5, 6])
            objs.append(("sphere", (float(c[0]), float(c[1]) + r, float(c[2])), r, int(i % 2), tuple(float(v) for v in rng.uniform(0.3, 1.0, 3)),
                         float(rng.uniform(0.0, 1.0)), 0.0))
        objs.append(("tri", (-14.0, 0.0, -10.0, -14.0, 0.0, 10.0, 14.0, 0.0, -10.0), S.MT_DIELECTRIC, (1.0, 1.0, 1.0), 0.9, 0.0, -1, (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
        objs.append(("tri", (-14.0, 0.0, 10.0, 14.0, 0.0, 10.0, 14.0, 0.0, -10.0), S.MT_DIELECTRIC, (1.0, 1.0, 1.0), 0.9, 0.0, -1, (0.0, 1.0, 1.0, 1.0, 1.0, 0.0)))
        scene = {"ambient": ((0.9, 0.9, 1.0), 0.2), "skybox": None, "textures": [], "lights": S.default_scene()["lights"], "objects": objs}
    sph, _ = P.scene_arrays(scene)
    cams = P.random_cameras(30, 5, sph)
    W, H = 200, 120
    res = {}
    for on in (1, 0):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(3, 3); c.set_image_size(W, H)
            c.set_bvh_mode(1)
            c.set_option("eye_grid", on)
            frames = [c.render_frames(cams, d) for d in (1, 2, 6)]
            st = c.stats()
            assert st["launches_blob_fast"] == len(cams) * 4 and st["launches_blob_any"] == 0, st
            ss = []
            for cam in cams[::6]:
                c.render(cam, 4, samples=2)
                ss.append(c.read_argb())
            c.enable_signatures(True)                                      # general kernel (every renderNext mode), hit paths recorded
            gen = []
            for cam in cams[1::7]:
                c.render(cam, 5, chunk=W * 7 + 13)                           # ragged renderNext slices
                gen.append((c.read_argb(), c.read_signatures()))
            assert c.stats()["launches_blob_any"] > 0
            res[on] = (frames, st["rays"], ss, c.get_seeds(), gen)
        finally:
            c.close()
    for a, b in zip(res[1][0], res[0][0]):
        assert np.array_equal(a, b)
    assert res[1][1] == res[0][1] and res[1][3] == res[0][3]
    for a, b in zip(res[1][2], res[0][2]):
        assert np.array_equal(a, b)
    for (a, sa), (b, sb) in zip(res[1][4], res[0][4]):
        assert np.array_equal(a, b) and np.array_equal(sa, sb)
