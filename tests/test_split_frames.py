"""Split frames rank by rank against the correctly-rounded-pow oracle (oracle/librfx_oracle_powcr.so, as in test_gpu_bitexact.py).

rfx_render_strips and rfx_render_range render part of a frame: a rank's interleaved strips, or any increasing list of pixel ranges.
Each rank here has its own context and its own device buffer, filled with a sentinel whose alpha byte packArgb never writes.  The
pixels a rank owns (`written`) must equal the oracle's whole frame bit for bit, and every other pixel must still hold the sentinel.
After the frame both random streams stand where the oracle's stand; the ranks' rays, bounces and shadow rays add up to the oracle's,
each rank's `samples` counts the Scene::trace calls of its own pixels, and the launch-family counters name the kernel that ran.

CPU: the write-set model against a brute-force restatement of Render::renderNext's pixel and block loop and against
sharding.strip_ranges; the oracle reference frames against the stream positions and call counts the GPU tests rely on."""
import numpy as np
import pytest

import cases
from reflaxman_b200 import scenes as S, sharding as P
from test_gpu_parity import _mixed_scene

SENTINEL = 0x5A0000A5          # alpha 0x5A: packArgb writes alpha 0
RFX_ERR_ARG = -1
FAMILIES = ("launches_small_fast", "launches_small_any", "launches_blob_fast", "launches_blob_any")
BLOB_WAVEFRONT = 2             # rfx_set_option "blob_wavefront" default: segments the tile kernel renders before it queues a path


# ---------------------------------------------------------------------------------------------------------------- write-set model
def _origins(W, H, a):
    """linear pixel indices of the block-preview origins (x % a == 0 and y % a == 0), scan order"""
    ys, xs = np.mgrid[0:H:a, 0:W:a]
    return (ys * W + xs).ravel()


def written(W, H, samples, ranges):
    """bool [H, W]: the pixels render_range over ``ranges`` stores.  Grid modes: the pixels of the ranges.  Block preview (samples =
    -a): every a x a block whose origin pixel index lies in a range, clipped to the image."""
    if samples > 0:
        m = np.zeros(W * H, bool)
        for p0, p1 in ranges:
            m[p0:p1] = True
        return m.reshape(H, W)
    a = -samples
    idx = _origins(W, H, a)
    inside = np.zeros(len(idx), bool)
    for p0, p1 in ranges:
        inside |= (idx >= p0) & (idx < p1)
    owned = np.zeros(((H + a - 1) // a, (W + a - 1) // a), bool)
    owned.ravel()[inside] = True
    return np.kron(owned, np.ones((a, a), bool))[:H, :W].astype(bool)


def calls_in(W, H, samples, ranges):
    """Scene::trace calls the reference makes for the pixels of ``ranges``"""
    if samples > 0:
        return sum(p1 - p0 for p0, p1 in ranges) * samples * samples
    idx = _origins(W, H, -samples)
    return int(sum(((idx >= p0) & (idx < p1)).sum() for p0, p1 in ranges))


def render_next_model(W, H, samples, ranges):
    """Brute force: Render::renderNext's loop (Render.cpp:158-196) over the pixels of each range in scan order.  Grid modes store the
    pixel; block preview traces only at an origin and fills its block, clipped to the image.  Returns (stored mask, calls)."""
    m = np.zeros((H, W), bool)
    calls = 0
    for p0, p1 in ranges:
        for p in range(p0, p1):
            y, x = divmod(p, W)
            if samples > 0:
                m[y, x] = True
                calls += samples * samples
                continue
            a = -samples
            if x % a or y % a:
                continue
            calls += 1
            for qy in range(y, min(y + a, H)):
                for qx in range(x, min(x + a, W)):
                    m[qy, qx] = True
    return m, calls


def gapped_ranges(W, H, samples, seed):
    """A seeded increasing partition with gaps: it starts after pixel 0 and ends before the last, cuts rows in the middle, holds an
    empty range, two adjacent ranges and one range of whole rows.  In block preview some boundaries lie in rows that hold origins
    and some in rows that hold none."""
    rng = np.random.default_rng(seed)
    total = W * H
    for _ in range(1000):
        c = np.sort(rng.choice(np.arange(1, total), 10, replace=False)).tolist()
        # R: a range c[i] .. c[i+1], G: a gap, E: an empty range at c[i]
        out, i = [], 0
        for k in "RGRERRGRGR":
            if k == "E":
                out.append((c[i], c[i]))
                continue
            if k == "R":
                out.append((c[i], c[i + 1]))
            i += 1
        lo, hi = -(-out[6][0] // W) * W, out[6][1] // W * W      # the 7th range snapped inwards to whole rows
        if lo >= hi:
            continue
        out[6] = (lo, hi)
        bounds = [p for r in out for p in r]
        if not any(p % W for p in bounds):
            continue
        if samples < 0:
            a = -samples
            rows = {(p // W) % a == 0 for p in bounds}
            if rows != {True, False}:
                continue
        return [(int(p0), int(p1)) for p0, p1 in out]
    raise AssertionError("no partition found")


def test_written_equals_the_render_next_loop():
    """written() and calls_in() against the brute-force renderNext loop: strips, gapped partitions, a range of one pixel, ragged
    images, block sizes 2 to 5 (blocks cut by the right and bottom edges) and grid sampling 1 to 3"""
    for W, H in ((16, 64), (40, 20), (70, 45), (84, 61), (13, 7)):
        for samples in (1, 2, 3, -2, -3, -4, -5):
            parts = [[(0, W * H)], [(W * H - 1, W * H)], [(5, 6)], gapped_ranges(W, H, samples, W * 1000 + H)]
            parts += [P.strip_ranges(W, H, world, rank, rows) for (world, rows) in ((3, 5), (2, 8), (8, 1), (3, 16)) for rank in range(world)]
            for ranges in parts:
                m, calls = render_next_model(W, H, samples, ranges)
                assert np.array_equal(written(W, H, samples, ranges), m), (W, H, samples, ranges)
                assert calls_in(W, H, samples, ranges) == calls, (W, H, samples, ranges)


def test_strip_write_sets_partition_the_frame():
    """Over the ranks of a strip split every pixel is stored by exactly one rank and the ranks' calls add up to a whole frame's.  In
    grid modes a rank stores exactly its strips; in block preview a block belongs to the rank that owns its origin, even where it
    reaches into the next strip."""
    for W, H, rows, world in ((64, 52, 8, 3), (84, 61, 16, 5), (40, 20, 16, 3), (70, 45, 5, 3), (16, 64, 8, 8), (84, 61, 1, 3)):
        for samples in (1, 2, -3, -4):
            count = np.zeros((H, W), int)
            calls = 0
            for rank in range(world):
                ranges = P.strip_ranges(W, H, world, rank, rows)
                m = written(W, H, samples, ranges)
                count += m
                calls += calls_in(W, H, samples, ranges)
                if samples > 0:
                    strips = np.zeros((H, W), bool)
                    for s in range(rank, -(-H // rows), world):
                        strips[s * rows:(s + 1) * rows] = True
                    assert np.array_equal(m, strips), (W, H, rows, world, rank)
            assert (count == 1).all(), (W, H, rows, world, samples)
            assert calls == P.calls_per_frame(W, H, samples), (W, H, rows, world, samples)
    assert not written(40, 20, 1, P.strip_ranges(40, 20, 3, 2, 16)).any()        # more ranks than strips: rank 2 owns nothing


def test_gapped_ranges_have_the_promised_shape():
    for W, H in ((84, 61), (70, 45), (64, 52)):
        for samples in (1, 2, -3, -4):
            r = gapped_ranges(W, H, samples, 7)
            assert r[0][0] > 0 and r[-1][1] < W * H
            assert all(p0 <= p1 for p0, p1 in r) and all(a[1] <= b[0] for a, b in zip(r, r[1:]))
            assert any(p0 == p1 for p0, p1 in r) and any(a[1] == b[0] and b[0] < b[1] for a, b in zip(r, r[1:]))
            assert any(a[1] < b[0] for a, b in zip(r, r[1:]))                                   # gaps
            assert any(p0 < p1 and p0 % W == 0 and p1 % W == 0 for p0, p1 in r)                # a band of whole rows


# ---------------------------------------------------------------------------------------------------------------- oracle frames
def _plane_scene():
    """the plane-hierarchy scene of test_gpu_plane_bvh.py::test_plane_scene_matches_oracle without its adversarial triangles: 36 spheres
    and a 2 048-triangle torus (both hierarchies) over a ground plane, so the blob kernels take their FAR instantiations"""
    return S.with_ground_plane(S.mesh_scene(32, 32, spheres=6, floor=S.synthetic_texture(64, 64, 3)), refl=0.8)


SCENES = {
    "default": S.default_scene,
    "mixed": _mixed_scene,
    "synth": cases.small_synth,
    "mesh": lambda: S.mesh_scene(32, 32),
    "plane": _plane_scene,
}
SMALL = {"default", "mixed"}      # the scenes that fit the constant bank


def _camera(name):
    if name == "default":
        return S.default_camera()
    return S.orbit_cameras(12)[int(name[5:])]     # "orbitK"


_ORACLE = {}


def oracle_frames(oracle, scene, W, H, seed, jobs):
    """jobs: ((camera name, depth, samples, additive), ...) rendered in order by one powcr OracleRender.  Returns per job a dict:
    argb, rgbf (resolved), raw (the float image after the pass), add (what the pass added to each pixel: for an accumulating pass
    raw = previous raw + add, one float addition), sig, rays, bounces, shadow_rays, samples and seeds (both streams after the pass).
    Cached: many rank and world combinations share one frame."""
    key = (scene, W, H, seed, tuple(jobs))
    if key not in _ORACLE:
        o = oracle.OracleRender(S.expand_meshes(SCENES[scene]()), W, H, seed=seed, L=oracle.lib_powcr())
        out = []
        for cam, depth, samples, additive in jobs:
            accumulate = additive and o.additive_counter >= 1
            before = o.image.copy()
            if accumulate:
                o.image[:] = 0                      # the pass adds its colours to zeros: exactly what it adds
            o.render(_camera(cam), depth, samples, additive, want_sig=True)
            add = o.image.copy()
            if accumulate:
                o.image[:] = before + add
            rgbf, argb = o.resolve()
            k = o.counters
            out.append({"argb": argb, "rgbf": rgbf, "raw": o.image.copy(), "add": add, "sig": o.sig.copy(), "rays": k["rays"],
                        "bounces": k["bounces"], "shadow_rays": k["shadow_rays"], "samples": k["samples"],
                        "seeds": (int(o.seeds[0]), int(o.seeds[1]))})
        _ORACLE[key] = out
    return _ORACLE[key]


def _lcg_jump(s, n):
    for _ in range(n):
        s = (214013 * s + 2531011) & 0xFFFFFFFF
    return s


def test_oracle_frames_are_the_plain_pass_sequence(oracle):
    """The reference frames the GPU tests compare with: split additive passes (zeroed image, then one float addition) give the plain
    oracle's raw images bit for bit; each pass makes calls_per_frame Scene::trace calls, consumes exactly that many randDir draws
    (rand_dirs), and draws two jitter values per pixel from the Render.cpp stream when additive, none otherwise."""
    W, H, seed = 40, 20, 31
    jobs = (("default", 4, 1, True), ("default", 4, 2, True), ("orbit3", 4, 1, True), ("default", 4, -3, False), ("orbit5", 4, 2, False))
    got = oracle_frames(oracle, "mixed", W, H, seed, jobs)
    plain = oracle.OracleRender(SCENES["mixed"](), W, H, seed=seed, L=oracle.lib_powcr())
    s0, s1 = seed, seed
    for j, (cam, depth, samples, additive) in enumerate(jobs):
        plain.render(_camera(cam), depth, samples, additive)
        assert np.array_equal(got[j]["raw"].view(np.uint32), plain.image.view(np.uint32)), j
        n = P.calls_per_frame(W, H, samples)
        s0 = oracle.rand_dirs(s0, n)[1]
        if additive and samples > 0:
            s1 = _lcg_jump(s1, 2 * W * H)
        assert got[j]["seeds"] == (int(plain.seeds[0]), int(plain.seeds[1])) == (s0, s1), j
        assert got[j]["samples"] == n and got[j]["rays"] == got[j]["bounces"] + got[j]["shadow_rays"] > 0, j


# ---------------------------------------------------------------------------------------------------------------- GPU helpers
@pytest.fixture(scope="module")
def gpu(rfx_lib, oracle):
    import torch
    from reflaxman_b200 import capi
    return capi, torch


def launches(scene, W, H, samples, ranges, depth, path=0, argb=True, aligned=True, sig=False, jitter=False):
    """the launch-family counters rfx_render_range over ``ranges`` must show: the host's kernel choice per range that makes calls"""
    out = dict.fromkeys(FAMILIES, 0)
    for p0, p1 in ranges:
        if calls_in(W, H, samples, [(p0, p1)]) == 0:
            continue                                                             # no call: nothing is launched
        rows = samples > 0 and not sig and p0 % W == 0 and p1 % W == 0
        vec = not argb or W % 4 != 0 or aligned                                  # 128-bit stores need a 16-byte aligned frame
        if scene in SMALL and path < 2:
            out["launches_small_fast" if rows and vec else "launches_small_any"] += 1
        elif path != 3 and rows and samples == 1 and not jitter and argb and depth > BLOB_WAVEFRONT:
            out["launches_blob_fast"] += 2                                       # the wavefront pair
        elif path != 3 and rows and vec:
            out["launches_blob_fast"] += 1
        else:
            out["launches_blob_any"] += 1
    return out


class Frame:
    """a full-frame device buffer of int32 (torch, device 0) filled with the sentinel; ``offset`` bytes into the allocation"""

    def __init__(self, torch, W, H, offset=0):
        self.torch, self.W, self.H, self.off = torch, W, H, offset // 4
        self.t = torch.empty(W * H + 4, dtype=torch.int32, device="cuda:0")
        self.reset()
        self.ptr = self.t.data_ptr() + offset

    def reset(self):
        self.t.fill_(SENTINEL)
        self.torch.cuda.synchronize()          # the library's streams do not wait for torch's

    def read(self):
        self.torch.cuda.synchronize()
        a = self.t.cpu().numpy().view(np.uint32)
        outside = np.concatenate([a[:self.off], a[self.off + self.W * self.H:]])
        assert (outside == SENTINEL).all(), "a store outside the frame"
        return a[self.off:self.off + self.W * self.H].reshape(self.H, self.W)


def check_pixels(got, want, mask, what):
    bad = mask & (got != want)
    assert not bad.any(), "%s: %d of %d written pixels differ from the oracle, e.g. at (y, x) %s" % (what, bad.sum(), mask.sum(), np.argwhere(bad)[:4].tolist())
    stray = ~mask & (got != SENTINEL)
    assert not stray.any(), "%s: %d pixels outside the write set were stored, e.g. at (y, x) %s" % (what, stray.sum(), np.argwhere(stray)[:4].tolist())


def check_family(st, want, what):
    assert {k: st[k] for k in FAMILIES} == want, (what, {k: st[k] for k in FAMILIES}, want)


def context(capi, scene, W, H, seed, path=0, bvh=0, sig=False):
    c = capi.Context(0)
    c.load_scene(SCENES[scene]()); c.set_seeds(seed, seed); c.set_image_size(W, H)
    c.force_path(path); c.set_bvh_mode(bvh); c.enable_signatures(sig); c.stats_reset()
    return c


# ---------------------------------------------------------------------------------------------------------------- 1. render_strips
# (id, scene, W, H, depth, samples, strip_rows, worlds, {path, bvh, sig, offset})
STRIP_CASES = [
    ("default_64x52_s8", "default", 64, 52, 8, 1, 8, (1, 2, 3), {}),               # every tile group staged, short last strip
    ("default_84x61_s16", "default", 84, 61, 8, 1, 16, (2, 3, 5), {}),             # W % 16 = 4: an unstaged right-edge group
    ("default_70x45_s24", "default", 70, 45, 8, 1, 24, (2, 3), {}),                # W % 4 != 0: scalar stores
    ("default_40x20_s16", "default", 40, 20, 8, 1, 16, (3, 8), {}),                # rank 1: a short strip, rank 2: nothing
    ("default_84x61_ss2_s8", "default", 84, 61, 6, 2, 8, (2, 3), {}),              # MULTI + STRIPS
    ("mixed_70x45_ss3_s8", "mixed", 70, 45, 6, 3, 8, (3,), {}),                    # F_ALL, MULTI + STRIPS
    ("mixed_84x61_s16", "mixed", 84, 61, 8, 1, 16, (2, 8), {}),                    # F_ALL, staged
    ("default_84x61_s5", "default", 84, 61, 8, 1, 5, (3,), {}),                    # general path: one range per strip
    ("default_40x20_s1", "default", 40, 20, 8, 1, 1, (3,), {}),                    # strips of one row
    ("mixed_70x45_ss2_s12", "mixed", 70, 45, 6, 2, 12, (2,), {}),
    ("default_70x45_block3_s5", "default", 70, 45, 8, -3, 5, (3,), {}),            # blocks reach into the next rank's strip
    ("mixed_84x61_block4_s8", "mixed", 84, 61, 8, -4, 8, (2,), {}),
    ("default_64x52_sig_s8", "default", 64, 52, 8, 1, 8, (3,), {"sig": True}),
    ("mixed_84x61_ss2_sig_s16", "mixed", 84, 61, 6, 2, 16, (2,), {"sig": True}),
    ("default_64x52_s8_off4", "default", 64, 52, 8, 1, 8, (3,), {"offset": 4}),    # 4-byte aligned: the strip remap of renderAny
    ("mixed_84x61_ss2_s8_off4", "mixed", 84, 61, 6, 2, 8, (2, 3), {"offset": 4}),
    ("default_70x45_s8_off4", "default", 70, 45, 8, 1, 8, (3,), {"offset": 4}),    # W % 4 != 0: the fast kernel all the same
    ("default_16x64_s8_k1", "default", 16, 64, 6, 1, 8, (8,), {}),                # a strip of 128 calls, a ranking block of ~1072
    ("default_200x64_ss3_s16_k1", "default", 200, 64, 5, 3, 16, (2, 3), {}),      # a strip of 28 800 calls
    ("synth_64x52_bvh0_s8", "synth", 64, 52, 6, 1, 8, (3,), {"path": 2, "bvh": 0}),
    ("synth_70x45_list_s8", "synth", 70, 45, 6, 1, 8, (2,), {"path": 2, "bvh": 2}),
    ("synth_84x61_ss2_s16", "synth", 84, 61, 4, 2, 16, (3,), {"path": 2, "bvh": 0, "offset": 4}),
    ("synth_64x52_general_block3_s8", "synth", 64, 52, 6, -3, 8, (2,), {"path": 3, "bvh": 0}),
    ("mesh_84x61_s16", "mesh", 84, 61, 4, 1, 16, (2,), {"path": 0}),
    ("plane_70x45_s8", "plane", 70, 45, 4, 1, 8, (3,), {"path": 0}),
]


def _strip_launches(scene, W, H, depth, samples, strip_rows, world, rank, path, sig, aligned):
    ranges = P.strip_ranges(W, H, world, rank, strip_rows)
    if scene in SMALL and path < 2 and samples > 0 and not sig and strip_rows % 8 == 0:
        out = dict.fromkeys(FAMILIES, 0)                # one launch over the rank's strips (none when it owns no row)
        if ranges:
            out["launches_small_fast" if aligned or W % 4 else "launches_small_any"] = 1
        return out
    return launches(scene, W, H, samples, ranges, depth, path, aligned=aligned, sig=sig)


@pytest.mark.gpu
@pytest.mark.parametrize("case", STRIP_CASES, ids=[c[0] for c in STRIP_CASES])
def test_render_strips_rank_by_rank(gpu, oracle, case):
    capi, torch = gpu
    name, scene, W, H, depth, samples, rows, worlds, opt = case
    path, bvh, sig, offset = opt.get("path", 0), opt.get("bvh", 0), opt.get("sig", False), opt.get("offset", 0)
    seed = 4000 + W + H
    want = oracle_frames(oracle, scene, W, H, seed, (("orbit2", depth, samples, False),))[0]
    for world in worlds:
        total = dict.fromkeys(("rays", "bounces", "shadow_rays"), 0)
        for rank in range(world):
            what = "%s world %d rank %d" % (name, world, rank)
            ranges = P.strip_ranges(W, H, world, rank, rows)
            mask = written(W, H, samples, ranges)
            buf = Frame(torch, W, H, offset)
            c = context(capi, scene, W, H, seed, path, bvh, sig)
            try:
                P.split_frame(c, _camera("orbit2"), depth, samples, world, rank, buf.ptr, strip_rows=rows)
                c.synchronize()                                          # raises on RFX_ERR_RNG
                check_pixels(buf.read(), want["argb"], mask, what)
                if sig:
                    assert np.array_equal(c.read_signatures()[mask], want["sig"][mask]), what
                assert c.get_seeds() == want["seeds"], what
                st = c.stats()
                assert st["samples"] == calls_in(W, H, samples, ranges), (what, st["samples"], calls_in(W, H, samples, ranges))
                check_family(st, _strip_launches(scene, W, H, depth, samples, rows, world, rank, path, sig, offset == 0), what)
                for k in total:
                    total[k] += st[k]
            finally:
                c.close()
        assert total == {k: want[k] for k in total}, (name, world, total)


# ---------------------------------------------------------------------------------------------------------------- 2. repeated frames
@pytest.mark.gpu
@pytest.mark.parametrize("ordering", ["off", "period1", "period8"])
@pytest.mark.parametrize("scene", ["default", "mixed"])
def test_repeated_split_frames_on_one_context(gpu, oracle, scene, ordering):
    """Config 3's loop (tools/bench_extra.py) on a 12-frame orbit: each rank context renders its strips of every frame on a caller's
    stream, with the tile order recorded and replayed across frames, and one whole frame through render_frames after frame 5 (a launch
    over another grid: the tile history starts again).  Every frame's written pixels, seeds and launch family match the oracle's."""
    capi, torch = gpu
    W, H, depth, rows, world, seed = 84, 61, 8, 8, 3, 99
    jobs = [("orbit%d" % f, depth, 1, False) for f in range(6)] + [("orbit6", depth, 1, False)] + \
           [("orbit%d" % f, depth, 1, False) for f in range(6, 12)]
    want = oracle_frames(oracle, scene, W, H, seed, tuple(jobs))
    stream = torch.cuda.Stream()
    for rank in range(world):
        ranges = P.strip_ranges(W, H, world, rank, rows)
        mask = written(W, H, 1, ranges)
        buf = Frame(torch, W, H)
        c = context(capi, scene, W, H, seed)
        try:
            c.set_tile_ordering(ordering != "off")
            if ordering == "period1":
                c.set_option("tile_order_period", 1)
            for j, (cam, _, _, _) in enumerate(jobs):
                what = "%s %s rank %d job %d" % (scene, ordering, rank, j)
                c.stats_reset()
                if j == 6:
                    got = c.render_frames([_camera(cam)], depth)[0]
                    assert np.array_equal(got, want[j]["argb"]), what
                    check_family(c.stats(), dict(dict.fromkeys(FAMILIES, 0), launches_small_fast=1), what)
                else:
                    buf.reset()
                    P.split_frame(c, _camera(cam), depth, 1, world, rank, buf.ptr, strip_rows=rows, stream=stream.cuda_stream)
                    c.synchronize()
                    stream.synchronize()
                    check_pixels(buf.read(), want[j]["argb"], mask, what)
                    st = c.stats()
                    assert st["samples"] == calls_in(W, H, 1, ranges), what
                    check_family(st, dict(dict.fromkeys(FAMILIES, 0), launches_small_fast=1), what)
                assert c.get_seeds() == want[j]["seeds"], what
        finally:
            c.close()


# ---------------------------------------------------------------------------------------------------------------- 3. render_range
RANGE_MODES = [(s, path) for s in (1, 2, -3, -4) for path in (0, 2, 3)]


def _render_ranges(c, cam, depth, samples, ranges, ptr=0, additive=False):
    c.set_camera(_camera(cam))
    c.render_begin(depth, samples, additive)
    for p0, p1 in ranges:
        c.render_range(p0, p1, ptr)
    c.render_finish()
    c.synchronize()


@pytest.mark.gpu
@pytest.mark.parametrize("samples,path", RANGE_MODES, ids=["s%d_path%d" % m for m in RANGE_MODES])
def test_render_range_gapped_into_a_buffer(gpu, oracle, samples, path):
    """seeded gapped partitions of one frame into a sentinel buffer, one context: written pixels, stream ends, the calls of the ranges
    and the kernel of every range"""
    capi, torch = gpu
    W, H, depth, seed = 84, 61, 6, 17
    want = oracle_frames(oracle, "default", W, H, seed, (("orbit4", depth, samples, False),))[0]
    ranges = gapped_ranges(W, H, samples, 100 + samples)
    buf = Frame(torch, W, H)
    c = context(capi, "default", W, H, seed, path)
    try:
        _render_ranges(c, "orbit4", depth, samples, ranges, buf.ptr)
        check_pixels(buf.read(), want["argb"], written(W, H, samples, ranges), "ranges")
        assert c.get_seeds() == want["seeds"]
        st = c.stats()
        assert st["samples"] == calls_in(W, H, samples, ranges)
        check_family(st, launches("default", W, H, samples, ranges, depth, path), "ranges")
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("scene,path", [("default", 2), ("synth", 2), ("default", 1)])
def test_render_range_row_band_at_an_offset(gpu, oracle, scene, path):
    """one band of whole rows that starts after row 0: blob scenes at depth 5 take the wavefront pair, which addresses the frame from
    the band's first pixel (argbOut + p0); the constant-bank fast kernel takes the band as its slice"""
    capi, torch = gpu
    W, H, depth, seed = 84, 61, 5, 23
    want = oracle_frames(oracle, scene, W, H, seed, (("orbit7", depth, 1, False),))[0]
    ranges = [(7 * W, 30 * W)]
    buf = Frame(torch, W, H)
    c = context(capi, scene, W, H, seed, path)
    try:
        _render_ranges(c, "orbit7", depth, 1, ranges, buf.ptr)
        check_pixels(buf.read(), want["argb"], written(W, H, 1, ranges), "band")
        assert c.get_seeds() == want["seeds"]
        st = c.stats()
        assert st["samples"] == 23 * W
        family = "launches_small_fast" if path == 1 else "launches_blob_fast"
        check_family(st, dict(dict.fromkeys(FAMILIES, 0), **{family: 1 if path == 1 else 2}), "band")
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("samples,path", RANGE_MODES, ids=["s%d_path%d" % m for m in RANGE_MODES])
def test_render_range_gapped_into_the_float_image(gpu, oracle, samples, path):
    """argb_device NULL: the ranges land in the context's float image bit for bit; gap pixels keep what they held (0 after
    set_image_size, the first frame's value in the second frame)"""
    capi, _ = gpu
    W, H, depth, seed = 70, 45, 6, 29
    want = oracle_frames(oracle, "default", W, H, seed, (("orbit1", depth, samples, False), ("orbit8", depth, samples, False)))
    c = context(capi, "default", W, H, seed, path)
    try:
        prev = np.zeros((H, W, 3), np.float32)
        for j, cam in enumerate(("orbit1", "orbit8")):
            ranges = gapped_ranges(W, H, samples, 200 + 10 * j + samples)
            c.stats_reset()
            _render_ranges(c, cam, depth, samples, ranges)
            mask = written(W, H, samples, ranges)
            exp = np.where(mask[..., None], want[j]["raw"], prev)
            got = c.read_rgbf()
            assert np.array_equal(got.view(np.uint32), exp.view(np.uint32)), ("frame", j, int((got.view(np.uint32) != exp.view(np.uint32)).any(-1).sum()))
            assert c.get_seeds() == want[j]["seeds"], j
            st = c.stats()
            assert st["samples"] == calls_in(W, H, samples, ranges), j
            check_family(st, launches("default", W, H, samples, ranges, depth, path, argb=False), ("frame", j))
            prev = got
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("samples,path", [(1, 0), (2, 0), (1, 2), (2, 3)], ids=["s1_path0", "s2_path0", "s1_path2", "s2_path3"])
def test_additive_passes_through_gapped_ranges(gpu, oracle, samples, path):
    """three additive passes: the first over the whole frame, the next two over gapped ranges.  The raw image (rfx_read_image with
    divide = 0) adds each pass's colours on the pixels of its ranges and keeps the others; the jitter stream (seed_render) ends
    where the oracle's does after render_finish."""
    capi, _ = gpu
    W, H, depth, seed = 84, 61, 5, 41
    jobs = (("orbit9", depth, samples, True),) * 3
    want = oracle_frames(oracle, "mixed", W, H, seed, jobs)
    c = context(capi, "mixed", W, H, seed, path)
    try:
        prev = None
        for k in range(3):
            ranges = [(0, W * H)] if k == 0 else gapped_ranges(W, H, samples, 300 + k)
            c.stats_reset()
            _render_ranges(c, "orbit9", depth, samples, ranges, additive=True)
            mask = written(W, H, samples, ranges)
            exp = want[0]["raw"] if k == 0 else np.where(mask[..., None], prev + want[k]["add"], prev)
            got, _ = c.read_image(divide=False)
            assert np.array_equal(got.view(np.uint32), exp.view(np.uint32)), ("pass", k, int((got.view(np.uint32) != exp.view(np.uint32)).any(-1).sum()))
            assert c.get_seeds() == want[k]["seeds"], k
            st = c.stats()
            assert st["samples"] == calls_in(W, H, samples, ranges), k
            check_family(st, launches("mixed", W, H, samples, ranges, depth, path, argb=False, jitter=True), ("pass", k))
            prev = got
    finally:
        c.close()


# ---------------------------------------------------------------------------------------------------------------- 4. argument checks
@pytest.mark.gpu
def test_split_frame_argument_checks(gpu, oracle):
    """decreasing ranges, ranges past the frame or behind the cursor, render_range with no frame begun, render_strips with rank >=
    world, strip_rows 0, a NULL buffer or after a range: RFX_ERR_ARG, and the frame then splits correctly all the same"""
    capi, torch = gpu
    W, H, depth, seed, world = 64, 52, 6, 53, 3
    total = W * H
    jobs = (("orbit2", depth, 1, False), ("orbit3", depth, 1, False), ("orbit4", depth, 1, False))
    want = oracle_frames(oracle, "default", W, H, seed, jobs)
    import ctypes as C
    for rank in range(world):
        c = context(capi, "default", W, H, seed)
        L, h = c.L, c.h
        buf = Frame(torch, W, H)
        rng_ = lambda p0, p1, ptr=buf.ptr: L.rfx_render_range(h, p0, p1, C.c_void_p(ptr), None)
        strips = lambda rows, wd, rk, ptr=buf.ptr: L.rfx_render_strips(h, rows, wd, rk, C.c_void_p(ptr) if ptr else None, None)
        try:
            assert rng_(0, W) == RFX_ERR_ARG                                   # no frame begun
            # frame 0: bad render_strips calls change nothing
            c.set_camera(_camera("orbit2")); c.render_begin(depth, 1, False)
            assert strips(8, world, world) == RFX_ERR_ARG
            assert strips(0, world, rank) == RFX_ERR_ARG
            assert strips(8, world, rank, 0) == RFX_ERR_ARG
            assert strips(8, 0, 0) == RFX_ERR_ARG
            c.render_strips(8, world, rank, buf.ptr)
            c.synchronize()
            check_pixels(buf.read(), want[0]["argb"], written(W, H, 1, P.strip_ranges(W, H, world, rank, 8)), "strips after bad calls")
            assert c.get_seeds() == want[0]["seeds"]
            assert rng_(0, W) == RFX_ERR_ARG                                   # the frame is complete
            # frame 1: render_strips after a range; the frame continues by ranges
            buf.reset()
            c.set_camera(_camera("orbit3")); c.render_begin(depth, 1, False)
            mine = P.strip_ranges(W, H, world, rank, 8)
            c.render_range(mine[0][0], mine[0][1], buf.ptr)
            assert strips(8, world, rank) == RFX_ERR_ARG
            for p0, p1 in mine[1:]:
                c.render_range(p0, p1, buf.ptr)
            c.render_finish(); c.synchronize()
            check_pixels(buf.read(), want[1]["argb"], written(W, H, 1, mine), "ranges after a refused render_strips")
            assert c.get_seeds() == want[1]["seeds"]
            # frame 2: decreasing, past the end, behind the cursor
            buf.reset()
            c.set_camera(_camera("orbit4")); c.render_begin(depth, 1, False)
            assert rng_(100, 99) == RFX_ERR_ARG
            assert rng_(0, total + 1) == RFX_ERR_ARG
            assert rng_(total + 1, total + 1) == RFX_ERR_ARG
            ranges = [(37 + rank, 600), (1000, 1000 + 13 * rank + 7)]
            c.render_range(*ranges[0], buf.ptr)
            assert rng_(500, 700) == RFX_ERR_ARG                               # starts behind the cursor
            c.render_range(*ranges[1], buf.ptr)
            c.render_finish(); c.synchronize()
            check_pixels(buf.read(), want[2]["argb"], written(W, H, 1, ranges), "ranges after refused ones")
            assert c.get_seeds() == want[2]["seeds"]
        finally:
            c.close()
