"""Bit for bit: the GPU against the oracle built with the GPU's power targets (oracle/librfx_oracle_powcr.so, RFXO_POW_CR).

DESIGN.md §2: every float operation on the GPU is the reference's, in the reference's order; the two powers are computed as the
correctly rounded value (rfx_device.cuh).  The powcr oracle computes exactly that, so the float results must be IDENTICAL — no
tolerance — for explicit ray lists (rfx_trace_rays, the shim's Scene::trace), for every kernel family and render mode, and for
cameras at the edges of the arithmetic.  A powLikePowf miss (tests/test_device_math.py) would be the one legitimate exception; none
occurs in these cases.

The CPU tests below check the powcr oracle itself: it meets the parity bar against every golden vector and differs from the plain
oracle only where the powers do."""
import ctypes as C
import ctypes.util
import math

import numpy as np
import pytest

import cases
from reflaxman_b200 import scenes as S
from test_gpu_parity import _edge_case, _mixed_scene

f32 = np.float32


@pytest.fixture(scope="module")
def capi(rfx_lib):
    from reflaxman_b200 import capi
    return capi


@pytest.fixture(scope="module")
def powcr(oracle):
    return oracle.lib_powcr()


def same_bits(a, b):
    """float arrays identical bit for bit, except that a NaN matches any NaN (and only a NaN)"""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def first_diff(a, b):
    a, b = np.asarray(a, np.float32).reshape(len(a), -1), np.asarray(b, np.float32).reshape(len(b), -1)
    bad = np.nonzero(~((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all(axis=1))[0]
    return len(bad), [(int(i), a[i].tolist(), b[i].tolist()) for i in bad[:4]]


# ---------------------------------------------------------------------------------------------------------------- CPU: the powcr oracle
@pytest.mark.parametrize("name", cases.GOLDEN)
def test_powcr_oracle_meets_the_parity_bar_on_every_golden_vector(oracle, powcr, name):
    g = cases.load_golden(name)
    eng = cases.OracleEngine(oracle, g["scene"], g["W"], g["H"], g["seed"])
    eng.r = oracle.OracleRender(g["scene"], g["W"], g["H"], seed=g["seed"], nthreads=4, L=powcr)
    for i, (rgbf, argb) in enumerate(cases.replay(eng, g)):
        cases.assert_parity(argb, g["argb%d" % i], "%s frame %d" % (name, i))


def test_powcr_oracle_differs_from_the_plain_oracle_only_at_the_powers(oracle, powcr):
    """default_160x120_d20: the float images agree on all but 4 of 19 200 pixels (99.979 %; DESIGN.md measures 99.989 % at full
    size), by at most 6e-8: the two builds differ only in the last bits of the powers."""
    g = cases.load_golden("default_160x120_d20")
    cam = S.default_camera()
    a = oracle.OracleRender(g["scene"], g["W"], g["H"], seed=g["seed"]).render(cam, g["refl"]).resolve()[0]
    b = oracle.OracleRender(g["scene"], g["W"], g["H"], seed=g["seed"], L=powcr).render(cam, g["refl"]).resolve()[0]
    assert np.array_equal(a.view(np.uint32), g["rgbf0"].view(np.uint32))
    same = (a.view(np.uint32) == b.view(np.uint32)).all(axis=-1).mean()
    assert same >= 0.9997, same
    assert np.abs(a - b).max() < 1e-7


# ---------------------------------------------------------------------------------------------------------------- scenes
def _material(k):
    return ((1.0, 0.2, 0.2), (0.2, 1.0, 0.2), (0.2, 0.2, 1.0))[k]


def tie_scene(order, spheres_bvh=False, tris_bvh=False):
    """A sphere at the origin (r = 1), an axis-aligned triangle in z = -1 with power-of-two edges and the plane z = -1: the ray
    (0, 0, -5) -> (0, 0, 1) meets all three at distance 4.0 exactly.  ``order``: insertion order of the three (the first inserted
    wins the tie, Scene.cpp:98).  spheres_bvh: 40 far-off spheres as well (a sphere hierarchy); tris_bvh: 40 far-off triangles and
    no plane (a triangle hierarchy)."""
    objs = {
        0: ("sphere", (0.0, 0.0, 0.0), 1.0, S.MT_METAL, _material(0), 0.5, 0.0),
        1: ("tri", (-1.0, -1.0, -1.0, -1.0, 3.0, -1.0, 3.0, -1.0, -1.0), S.MT_DIELECTRIC, _material(1), 0.25, 0.0, -1, (0.0,) * 6),
        2: ("plane", (0.0, 0.0, -1.0), (0.0, 0.0, -1.0), S.MT_METAL, _material(2), 0.75, 0.0),
    }
    out = [objs[k] for k in order if not (tris_bvh and k == 2)]
    if spheres_bvh:
        out += [("sphere", (60.0 + 3.0 * i, 0.5 * (i % 5), 40.0), 1.0, i % 2, (0.5, 0.6, 0.7), 0.3, 0.0) for i in range(40)]
    if tris_bvh:
        out += [("tri", (70.0 + 2.0 * i, 0.0, -30.0, 70.0 + 2.0 * i, 1.0, -30.0, 71.0 + 2.0 * i, 0.0, -30.0), S.MT_METAL, (0.9, 0.9, 0.9), 0.4, 0.0, -1,
                 (0.0,) * 6) for i in range(40)]
    return {"ambient": ((0.9, 0.9, 1.0), 0.2), "skybox": S.synthetic_texture(64, 48, 3), "textures": [],
            "lights": [((3.0, 8.0, -9.0), 0.5, (1.0, 1.0, 0.9), 0.8)], "objects": out}


def overflow_scene():
    """More than 32 triangles and no plane (a triangle hierarchy): a cluster of small triangles at z = 0 and, behind it along +z, a
    cluster of large slanted triangles whose boxes begin nearer (z = -9) than the small ones'.  A ray from (x, y, -10) along +z meets a
    large triangle's box first but a small triangle first.  With |d| > 1.8e19 (|d|^2 overflows to inf) the pruning distance of the
    triangle walk must not collapse to 0 after the first (farther) hit."""
    objs = []
    for i in range(6):
        for j in range(6):
            x, y = -3.0 + i, -3.0 + j
            objs.append(("tri", (x, y, 0.0, x, y + 0.9, 0.0, x + 0.9, y, 0.0), S.MT_METAL, (0.3, 0.9, 0.3), 0.5, 0.0, -1, (0.0,) * 6))
    for i in range(6):
        for j in range(6):
            x, y = -3.0 + i, -3.0 + j
            objs.append(("tri", (x - 0.5, y - 0.5, -9.0, x - 0.5, y + 1.5, 9.0, x + 1.5, y - 0.5, 9.0), S.MT_METAL, (0.9, 0.3, 0.3), 0.5, 0.0, -1,
                         (0.0,) * 6))
    return {"ambient": ((0.9, 0.9, 1.0), 0.2), "skybox": None, "textures": [],
            "lights": [((0.0, 5.0, -20.0), 0.5, (1.0, 1.0, 1.0), 0.8)], "objects": objs}


def _geometry(scene):
    sph = [(np.array(o[1], f32), f32(o[2])) for o in scene["objects"] if o[0] == "sphere"]
    tri = [np.array(o[1], f32).reshape(3, 3) for o in scene["objects"] if o[0] == "tri"]
    for o in scene["objects"]:
        if o[0] == "mesh":
            tri += list(np.asarray(o[1], f32)[np.asarray(o[2], np.int64)])
    return sph, tri


def _unit(rng, n):
    v = rng.normal(size=(n, 3))
    return (v / np.linalg.norm(v, axis=1, keepdims=True)).astype(f32)


def ray_catalogue(scene, seed, n_random=600):
    """Seeded rays aimed at the edges of the arithmetic (origins, rays as float32 [n, 3])."""
    rng = np.random.default_rng(seed)
    sph, tri = _geometry(scene)
    O, R = [], []

    def add(o, r):
        o, r = np.asarray(o, f32).reshape(-1, 3), np.asarray(r, f32).reshape(-1, 3)
        n = max(len(o), len(r))
        O.append(np.broadcast_to(o, (n, 3))); R.append(np.broadcast_to(r, (n, 3)))

    eye = np.array(S.DEFAULT_EYE, f32)
    add(eye + rng.uniform(-1, 1, (n_random, 3)).astype(f32), _unit(rng, n_random))                     # ordinary rays
    for c, r in sph[:12]:
        u = _unit(rng, 24)
        surf = (c + r * u).astype(f32)                                                                   # float points c + r u
        add(surf, _unit(rng, 24))
        add(surf, u)                                                                                      # leaving along the normal
        add((c + f32(0.5) * r * u[:8]).astype(f32), _unit(rng, 8))                                        # inside
        add(c, _unit(rng, 4))                                                                             # at the centre
        t = np.cross(u[:8], _unit(rng, 8)).astype(f32)                                                   # grazing tangents
        add((c + r * u[:8] - f32(5) * t).astype(f32), t)
    pick = rng.choice(len(tri), min(len(tri), 24), replace=False) if tri else []
    for k in pick:
        v0, v1, v2 = tri[k]
        e1, e2 = (v1 - v0).astype(f32), (v2 - v0).astype(f32)
        nrm = np.cross(e1, e2)
        nrm = (nrm / max(np.linalg.norm(nrm), 1e-30)).astype(f32)
        bary = [(0, 0), (1, 0), (0, 1), (0.5, 0), (0, 0.5), (0.5, 0.5), (0.25, 0.75), (0.3, 0.2), (1 - 2 ** -20, 0), (0, 1 - 2 ** -20)]
        pts = np.array([v0 + f32(a) * e1 + f32(b) * e2 for a, b in bary], f32)                          # vertices, edges, u + v = 1
        add(pts, _unit(rng, len(pts)))                                                                    # origins on the surface
        add((pts + f32(3) * nrm).astype(f32), -nrm)                                                       # aimed at the boundaries
        add((pts - f32(3) * nrm).astype(f32), nrm)
        for s in (1e-4, 1e-4 * (1 + 2 ** -20), 1e-4 * (1 - 2 ** -20)):                                  # the DELTA boundary
            add((pts[:4] + f32(s) * nrm).astype(f32), -nrm)
        c = ((v0 + v1 + v2) / f32(3)).astype(f32)
        for h in (0.0, 1e-3, 2.0 ** -63, -2.0 ** -63, 2.0 ** -60):                                       # parallel, |rz| around 2^-63
            add((c + f32(0.25) * nrm - f32(4) * e1).astype(f32), (e1 + f32(h) * nrm).astype(f32))
            add((c + f32(1e-3) * nrm).astype(f32), (e2 + f32(h) * nrm).astype(f32))
    # the floor's checker cells (empty texture: u * 50 on integers) and texture coordinates 0, 1, 1 - eps, outside [0, 1]
    for q in (0.0, 0.02, 0.04, 0.5, 1 - 2 ** -24, 1.0, 1.02, -0.02):
        x = f32(-14.0 + 28.0 * q)
        add((x, 4.0, 0.3), (0.0, -1.0, 0.0))
        add((1.7, 4.0, f32(-10.0 + 20.0 * q)), (0.0, -1.0, 0.0))
    # towards the sky: axes and the cube-map seams |x| = |y|, |x| = |z|, |x| = |y| = |z|, with +-0 components
    dirs = []
    for a in (1.0, -1.0):
        for b in (1.0, -1.0, 0.0, -0.0):
            dirs += [(a, b, 0.0), (a, 0.0, b), (0.0, a, b), (a, -0.0, 0.0), (-0.0, a, -0.0), (0.0, 0.0, a), (a, b, b), (a, a, b)]
    add((0.0, 60.0, 0.0), dirs)
    add(eye, dirs)
    # direction magnitudes: 0, 2^-70, 2^-30, 2^30, 2^65 (|d|^2 overflows) and denormal components
    base = _unit(rng, 40)
    for m in (0.0, 2.0 ** -70, 2.0 ** -30, 2.0 ** 30, 2.0 ** 65):
        add(eye + rng.uniform(-1, 1, (40, 3)).astype(f32), (base * f32(m)).astype(f32))
    add(eye, [(1e-40, -1.0, 1e-42), (-1e-45, 0.3, 1.0), (1e-40, 1e-41, 1e-42), (1e-38, -1e-38, 2e-38)])
    # origins outside the reach box of the hierarchies (the scene is re-flattened)
    add(np.array([(1e6, 3.0, 0.0), (-1e6, 1e6, 2.0), (0.5, 0.5, -1e6)], f32), [(-1.0, 0.0, 0.0), (1.0, -1.0, 0.0), (0.0, 0.0, 1.0)])
    return np.concatenate(O).astype(f32), np.concatenate(R).astype(f32)


def _mesh(n_u=32, n_v=32):
    return S.mesh_scene(n_u, n_v)


# (scene factory, bvh mode, extra rays) per ray-list case
RAY_SCENES = {
    "default": (S.default_scene, 0),
    "mixed": (_mixed_scene, 0),
    "synth16_bvh0": (lambda: S.synthetic_scene(16), 0),
    "synth16_bvh1": (lambda: S.synthetic_scene(16), 1),
    "synth16_list": (lambda: S.synthetic_scene(16), 2),
    "mesh_bvh": (_mesh, 1),
    "mesh_list": (_mesh, 2),
    "overflow_bvh": (overflow_scene, 0),
    "overflow_list": (overflow_scene, 2),
}
TIE_ORDERS = [(0, 1, 2), (0, 2, 1), (1, 0, 2), (1, 2, 0), (2, 0, 1), (2, 1, 0)]
for _o in TIE_ORDERS:
    _k = "".join(map(str, _o))
    RAY_SCENES["tie" + _k] = (lambda o=_o: tie_scene(o), 0)
    RAY_SCENES["tie" + _k + "_spheres"] = (lambda o=_o: tie_scene(o, spheres_bvh=True), 0)
    RAY_SCENES["tie" + _k + "_tris"] = (lambda o=_o: tie_scene(o, tris_bvh=True), 0)


def _extra_rays(name):
    if name.startswith("tie"):
        o = [(0.0, 0.0, -5.0)] * 3 + [(0.0, 0.0, 5.0)] * 3
        return np.array(o, f32), np.array([(0, 0, 1), (0, 0, 2), (0, 0, 0.5), (0, 0, -1), (0, 0, -2), (0, 0, -0.5)], f32)
    if name.startswith("overflow"):
        g = np.array([(-2.7 + i + 0.1 * k, -2.7 + j + 0.1 * k, -10.0) for i in range(6) for j in range(6) for k in range(3)], f32)
        d = np.array([(0.0, 0.0, m) for m in (1.0, 2.0 ** 65, 2.0 ** 100)], f32)
        return np.repeat(g, 3, axis=0), np.tile(d, (len(g), 1))
    return np.zeros((0, 3), f32), np.zeros((0, 3), f32)


def _gpu_trace(capi, scene, bvh, seed, batches, depth):
    c = capi.Context(0)
    try:
        c.load_scene(scene); c.set_bvh_mode(bvh); c.set_seeds(seed, seed)
        outs = [c.trace_rays(o, r, depth) for o, r in batches]
        return outs, c.get_seeds()[0], c.stats()
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(RAY_SCENES))
def test_trace_rays_bit_exact_against_powcr_oracle(capi, oracle, powcr, name):
    """rfx_trace_rays == rfxo_trace_many on a catalogue of edge rays, depths 1, 2, 8 and 20: every float of every ray identical, the
    random stream's end state identical; two consecutive calls == one call over the concatenated rays; 1, 31, 32, 33 rays."""
    make, bvh = RAY_SCENES[name]
    scene = make()
    oscene = oracle.OracleScene(S.expand_meshes(scene), powcr)
    O, R = ray_catalogue(scene, seed=len(name) * 7919 + sum(map(ord, name)))
    eo, er = _extra_rays(name)
    O, R = np.concatenate([eo, O]), np.concatenate([er, R])
    for depth, seed in ((1, 11), (2, 22), (8, 88), (20, 2020)):
        want, _, end = oracle.trace_many(oscene, O, R, depth, seed)
        (got,), gend, st = _gpu_trace(capi, scene, bvh, seed, [(O, R)], depth)
        n, where = first_diff(got, want)
        assert n == 0, "%s depth %d: %d of %d rays differ, e.g. %s (origins %s, rays %s)" % (
            name, depth, n, len(O), where, O[[w[0] for w in where]].tolist(), R[[w[0] for w in where]].tolist())
        assert gend == end, (name, depth)
    # split calls continue the stream; launch edges
    want, _, end = oracle.trace_many(oscene, O, R, 8, 5)
    (a, b), gend, _ = _gpu_trace(capi, scene, bvh, 5, [(O[:33], R[:33]), (O[33:], R[33:])], 8)
    assert same_bits(np.concatenate([a, b]), want) and gend == end, name
    for n in (1, 31, 32, 33):
        w, _, e = oracle.trace_many(oscene, O[-n:], R[-n:], 20, 77)
        (g,), ge, _ = _gpu_trace(capi, scene, bvh, 77, [(O[-n:], R[-n:])], 20)
        assert same_bits(g, w) and ge == e, (name, n)


@pytest.mark.gpu
@pytest.mark.parametrize("bvh", [0, 2], ids=["hierarchy", "list"])
def test_overflowing_directions_keep_the_nearest_triangle(capi, oracle, powcr, bvh):
    """Rays of |d| = 2^65 and 2^100 (|d|^2 overflows binary32) through the overflow scene, origins inside the hierarchy's reach box, one
    call: the triangle walk must find the small triangle in front of the large one it meets first, as the list walk and the oracle do.
    (With 1/sqrtf(inf) = 0 as the walk's pruning scale, every box after the first hit was pruned.)"""
    scene = overflow_scene()
    O, R = _extra_rays("overflow")
    want, sig, end = oracle.trace_many(oracle.OracleScene(scene, powcr), O, R, 1, 17)
    (got,), gend, _ = _gpu_trace(capi, scene, bvh, 17, [(O, R)], 1)
    n, where = first_diff(got, want)
    assert n == 0, "%d of %d rays differ, e.g. %s (origins %s, rays %s)" % (n, len(O), where, O[[w[0] for w in where]].tolist(),
                                                                          R[[w[0] for w in where]].tolist())
    assert gend == end


@pytest.mark.gpu
def test_tie_scenes_pick_the_first_inserted_object(capi, oracle, powcr):
    """The exact ties (distance 4.0 to a sphere, a triangle and a plane) resolve to the object inserted first, on the GPU as in the
    oracle: the colour of the first bounce differs per winner, and the three directions of one tie give the same first hit."""
    colours = set()
    for order in TIE_ORDERS:
        scene = tie_scene(order)
        O = np.array([(0.0, 0.0, -5.0)] * 3, f32)
        R = np.array([(0, 0, 1), (0, 0, 2), (0, 0, 0.5)], f32)
        want, sig, _ = oracle.trace_many(oracle.OracleScene(scene, powcr), O, R, 1, 3)
        (got,), _, _ = _gpu_trace(capi, scene, 0, 3, [(O, R)], 1)
        assert same_bits(got, want), order
        assert len(set(sig.tolist())) == 1, order               # the same object wins for all three directions
        colours.add(tuple(want[0].tolist()))
    assert len(colours) == 3, colours                            # three different winners over the six orders


# ---------------------------------------------------------------------------------------------------------------- kernel families
def _oracle_frames(oracle, powcr, scene, W, H, seed, jobs):
    """jobs: [(cam, depth, samples, additive)] -> [(rgbf, argb, sig, rays, bounces, seed0)] of the powcr oracle, one Render"""
    o = oracle.OracleRender(scene, W, H, seed=seed, L=powcr)
    out = []
    for cam, depth, samples, additive in jobs:
        o.render(cam, depth, samples, additive, want_sig=True)
        rgbf, argb = o.resolve()
        out.append((rgbf, argb, o.sig.copy(), o.counters["rays"], o.counters["bounces"], int(o.seeds[0])))
    return out


def _golden_jobs(name):
    g = cases.load_golden(name)
    jobs = []
    for _ in range(g["frames"]):
        for _ in range(max(g["additive"], 1)):
            jobs.append((S.default_camera(), g["refl"], g["samples"], bool(g["additive"])))
    return g["scene"], g["W"], g["H"], g["seed"], jobs


FAMILY_CASES = [n for n in cases.GOLDEN if not n.startswith("synth1024")] + ["synth1024_160x90_d8", "mixed", "mixed_ss2", "mixed_block3",
                                                                            "empty", "nolight_1x1", "nolight_1x67_ss2", "constbank_full",
                                                                            "constbank_plus_one"]


def _family_case(name):
    if name == "synth1024_160x90_d8":
        return cases.config4_scene(), 160, 90, 1234, [(S.default_camera(), 8, 1, False), (S.orbit_cameras(7)[3], 8, 1, False)]
    if name.startswith("mixed"):
        samples = {"mixed": 1, "mixed_ss2": 2, "mixed_block3": -3}[name]
        return _mixed_scene(), 125, 66, 4242, [(S.orbit_cameras(7)[2], 12, samples, False), (S.default_camera(), 5, samples, False)]
    if name in ("empty", "nolight_1x1", "nolight_1x67_ss2", "constbank_full", "constbank_plus_one"):
        scene, W, H, depth, samples = _edge_case(name)
        return scene, W, H, 7, [(S.default_camera(), depth, samples, False)]
    return _golden_jobs(name)


def _gpu_configs(scene):
    """(label, force_path, bvh mode, options, chunk)"""
    cfg = [("const", 1, 0, {}, None), ("blob", 2, 0, {}, None), ("general", 3, 0, {}, None), ("ragged", 2, 0, {}, 997)]
    for bvh in (1, 2):
        cfg.append(("blob_bvh%d" % bvh, 2, bvh, {}, None))
        cfg.append(("general_bvh%d" % bvh, 3, bvh, {}, None))
    cfg += [("grids_off", 2, 1, {"light_grids": 0, "eye_grid": 0}, None), ("grids_on", 2, 1, {"light_grids": 1, "eye_grid": 1}, None)]
    return cfg


@pytest.mark.gpu
@pytest.mark.parametrize("name", FAMILY_CASES)
def test_every_kernel_family_bit_exact_against_powcr_oracle(capi, oracle, powcr, name):
    """Render API (constant-bank, blob tile, general kernels; bvh modes 0/1/2; light and eye grids on and off; SSAA, additive passes,
    block preview, ragged renderNext slices): float image, ARGB, hit-path signatures (signature runs), rays, bounces and stream
    position identical to the powcr oracle.  Batch path (fast kernels, blob_wavefront 1/2/3): ARGB, rays and stream identical."""
    scene, W, H, seed, jobs = _family_case(name)
    want = _oracle_frames(oracle, powcr, scene, W, H, seed, jobs)
    for label, path, bvh, opts, chunk in _gpu_configs(scene):
        for sig in (False, True):
            c = capi.Context(0)
            try:
                c.load_scene(scene); c.set_seeds(seed, seed); c.set_image_size(W, H)
                c.force_path(path); c.set_bvh_mode(bvh)
                for k, v in opts.items():
                    c.set_option(k, v)
                c.enable_signatures(sig)
                for j, (cam, depth, samples, additive) in enumerate(jobs):
                    c.stats_reset()
                    c.render(cam, depth, samples, additive, chunk=chunk)
                    st = c.stats()
                    rgbf, argb, osig, rays, bounces, s0 = want[j]
                    what = "%s %s sig=%d job %d" % (name, label, sig, j)
                    n, where = first_diff(c.read_rgbf().reshape(-1, 3), rgbf.reshape(-1, 3))
                    assert n == 0, "%s: %d pixels differ, e.g. %s" % (what, n, where)
                    assert np.array_equal(c.read_argb(), argb), what
                    assert st["rays"] == rays and st["bounces"] == bounces and c.get_seeds()[0] == s0, what
                    if sig:
                        assert np.array_equal(c.read_signatures(), osig), what
            finally:
                c.close()
    # batch path: one-sample ARGB frames (fast kernels; blob scenes: tile kernel or wavefront pair)
    batch = [(j, job) for j, job in enumerate(jobs) if job[2] == 1 and not job[3]]
    if not batch:
        return
    for label, path, wave in (("fast", 0, None), ("blob_wave1", 2, 1), ("blob_wave2", 2, 2), ("blob_wave3", 2, 3), ("blob_tile", 2, 0)):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_image_size(W, H); c.force_path(path)
            if wave is not None:
                c.set_option("blob_wavefront", wave)
            for j, (cam, depth, samples, additive) in batch:
                if any(jb[2] != 1 or jb[3] for jb in jobs[:j]):
                    continue                                           # start the stream where the oracle's job j started
                c.set_seeds(seed, seed)
                if j:
                    c.skip_samples(W * H * j)
                c.stats_reset()
                got = c.render_frames([cam], depth)[0]
                assert np.array_equal(got, want[j][1]), (name, label, j)
                assert c.stats()["rays"] == want[j][3] and c.get_seeds()[0] == want[j][5], (name, label, j)
        finally:
            c.close()


# ---------------------------------------------------------------------------------------------------------------- edge cameras
def _host_tanf():
    libm = C.CDLL(ctypes.util.find_library("m"))
    libm.tanf.restype = C.c_float
    libm.tanf.argtypes = [C.c_float]
    return libm.tanf


def seam_fov(W):
    """A float fov for which the host computes rz = (W / 2) / tanf(fov / 2) == W / 2 exactly (Render.cpp:148), so that pixel column
    0 of an identity view has |x| == rz: its rays run exactly along the seam of two sky-cube faces."""
    tanf = _host_tanf()
    lo = hi = f32(math.pi / 2)
    for _ in range(256):                       # outwards from pi/2, one float at a time
        for fov in (lo, hi):
            if f32(f32(W) / f32(2)) / f32(tanf(f32(fov / f32(2)))) == f32(W) / f32(2):
                return fov
        lo, hi = np.nextafter(lo, f32(0)), np.nextafter(hi, f32(4))
    raise AssertionError("no fov near pi/2 gives tanf(fov/2) == 1")


def _edge_cameras():
    ident = np.array([1, 0, 0, 0, 1, 0, 0, 0, 1], f32)
    sph = S.default_scene()["objects"][1]                    # sphere (0.15, 1.0, 1.75), r = 1
    c, r = np.array(sph[1], f32), f32(sph[2])
    u = np.array([0.6, 0.0, -0.8], f32)
    on_surface = (c + r * u).astype(f32)
    return {
        "eye_on_sphere": (S.default_scene(), S.camera_lookat(tuple(on_surface), (6.0, 2.0, -5.0), 1.05)),
        "eye_on_floor": (S.default_scene(), S.camera_lookat((3.0, 0.0, -2.0), (-1.0, 1.0, 1.0), 1.05)),
        "eye_in_sphere": (S.default_scene(), S.camera_lookat((-1.0, 1.4, -0.2), (3.0, 1.0, 2.0), 1.2)),
        "fov_tiny_default": (S.default_scene(), S.camera_lookat(S.DEFAULT_EYE, S.DEFAULT_AT, 1e-20)),
        "fov_tiny_mesh": (_mesh(), S.camera_lookat((6.0, 3.5, -5.0), (0.0, 2.6, 0.0), 1e-20)),
        "fov_near_pi": (S.default_scene(), S.camera_lookat(S.DEFAULT_EYE, S.DEFAULT_AT, float(np.nextafter(f32(math.pi), f32(0))))),
        "sky_seam": (S.default_scene(skybox=S.synthetic_texture(128, 96, 5)), (np.array((0.0, 50.0, 0.0), f32), ident, seam_fov(96))),
    }


def test_seam_fov_gives_an_exact_seam_column():
    """CPU: the fov search finds a float fov whose rz equals W / 2, so column 0's ray (-W/2, y - H/2, rz) has |x| == |z| in float32."""
    W = 96
    fov = seam_fov(W)
    rz = f32(f32(W) / f32(2)) / f32(_host_tanf()(f32(fov / f32(2))))
    assert rz == f32(48.0) and abs(f32(0) - f32(W) / f32(2)) == rz


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["eye_on_sphere", "eye_on_floor", "eye_in_sphere", "fov_tiny_default", "fov_tiny_mesh", "fov_near_pi", "sky_seam"])
def test_edge_cameras_bit_exact_against_powcr_oracle(capi, oracle, powcr, name):
    """Small images at cameras the arithmetic finds hard, on both machines (traceSmall where the scene fits the constant bank, and
    traceBlob): float image, ARGB, signatures, rays and stream identical to the powcr oracle."""
    scene, cam = _edge_cameras()[name]
    W, H, depth, seed = 96, 64, 8, 99
    o = oracle.OracleRender(S.expand_meshes(scene), W, H, seed=seed, L=powcr).render(cam, depth, want_sig=True)
    rgbf, argb = o.resolve()
    for path, bvh in ((1, 0), (2, 0), (3, 0), (2, 1), (2, 2)):
        c = capi.Context(0)
        try:
            c.load_scene(scene); c.set_seeds(seed, seed); c.set_image_size(W, H)
            c.force_path(path); c.set_bvh_mode(bvh); c.enable_signatures(True); c.stats_reset()
            c.render(cam, depth)
            n, where = first_diff(c.read_rgbf().reshape(-1, 3), rgbf.reshape(-1, 3))
            assert n == 0, "%s path %d bvh %d: %d pixels differ, e.g. %s" % (name, path, bvh, n, where)
            assert np.array_equal(c.read_argb(), argb) and np.array_equal(c.read_signatures(), o.sig), (name, path, bvh)
            assert c.stats()["rays"] == o.counters["rays"] and c.get_seeds()[0] == int(o.seeds[0]), (name, path, bvh)
            c.enable_signatures(False); c.set_seeds(seed, seed)
            assert np.array_equal(c.render_frames([cam], depth)[0], argb), (name, path, bvh, "batch")
        finally:
            c.close()
