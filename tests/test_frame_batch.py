"""GPU tests (-m gpu): rfx_render_frames_device renders runs of frames of one camera in batched launches of the fast kernel
(first segment of each path once per batch, option "frame_batch").  With the option on and off the call must produce the same
ARGB frames bit for bit, the same ray, bounce and shadow-ray counts, and leave the random stream at the same position."""
import numpy as np
import pytest

import cases
from reflaxman_b200 import scenes as S

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi(rfx_lib):
    from reflaxman_b200 import capi
    return capi


def _mixed_scene():
    """textured floor and skybox, a plane, three lights: the F_ALL instantiation"""
    s = S.default_scene(skybox=S.synthetic_texture(256, 192, 5), floor=S.synthetic_texture(64, 64, 9))
    s["objects"].insert(3, ("sphere", (3.0, 0.8, 2.5), 0.8, S.MT_DIELECTRIC, (0.9, 0.3, 0.3), 0.6, 0.0))
    s["objects"].append(("tri", (-6.0, 0.0, 5.0, -6.0, 4.0, 5.0, 6.0, 0.0, 5.0), S.MT_METAL, (0.8, 0.8, 1.0), 0.7, 0.0, -1,
                         (0.0, 0.0, 0.0, 1.0, 1.0, 0.0)))
    s["objects"].append(("plane", (0.0, 0.0, 9.0), (0.0, 0.0, -1.0), S.MT_DIELECTRIC, (0.4, 0.5, 0.4), 0.3, 0.0))
    s["lights"].append(((2.0, 6.0, -4.0), 0.5, (1.0, 0.6, 0.4), 0.4))
    s["lights"].append(((-5.0e9, -3.0e9, 1.0e9), 2.0e8, (0.3, 0.3, 1.0), 0.3))
    s["lights"].append(((0.0, 9.0e9, 0.0), 1.0e8, (1.0, 1.0, 1.0), 0.0))
    return s


def _render(capi, scene, W, H, cams, depth, batch, max_calls=None, offset_words=0):
    """frames of one call (+ the first frame of the next call: the stream position), stats, seeds after the call"""
    import torch
    c = capi.Context(0)
    try:
        c.load_scene(scene); c.set_seeds(99, 99); c.set_image_size(W, H)
        c.set_option("frame_batch", batch)
        if max_calls:
            c.set_option("max_calls_per_launch", max_calls)
        n = len(cams)
        buf = torch.zeros(n * W * H + offset_words + 4, dtype=torch.int32, device="cuda")
        c.stats_reset()
        c.render_frames_device(capi.pack_cameras(cams), depth, 1, buf.data_ptr() + 4 * offset_words)
        c.synchronize()
        st = c.stats()
        seeds = c.get_seeds()
        nxt = torch.zeros(W * H, dtype=torch.int32, device="cuda")
        c.render_frames_device(capi.pack_cameras(cams[:1]), depth, 1, nxt.data_ptr())
        c.synchronize()
        frames = buf[offset_words:offset_words + n * W * H].cpu().numpy().reshape(n, H, W)
        return frames, (st["rays"], st["bounces"], st["shadow_rays"], st["samples"]), seeds, nxt.cpu().numpy(), st
    finally:
        c.close()


def _same(capi, scene, W, H, cams, depth=20, **kw):
    a = _render(capi, scene, W, H, cams, depth, 1, **kw)
    b = _render(capi, scene, W, H, cams, depth, 0, **kw)
    assert np.array_equal(a[0], b[0]), "frames differ"
    assert a[1] == b[1], (a[1], b[1])
    assert a[2] == b[2] and np.array_equal(a[3], b[3]), "stream position differs"
    return a


ORBIT = S.orbit_cameras(12)


@pytest.mark.parametrize("n", [1, 2, 7, 8, 9, 16, 17, 33])
def test_runs_of_one_camera(capi, n):
    """batch lengths around the batch size and across the 16-frame ranking group of 1080p"""
    W, H = 1920, 1080
    frames, _, _, _, st = _same(capi, S.default_scene(), W, H, [S.default_camera()] * n, depth=4)
    if n > 1:
        assert st["launches_small_fast"] < n, st            # the batched kernel did run


@pytest.mark.parametrize("pos", range(9))
def test_camera_change_inside_a_batch(capi, pos):
    """one frame of another camera at every position of a 9-frame run"""
    cams = [S.default_camera()] * 9
    cams[pos] = ORBIT[3]
    _same(capi, S.default_scene(), 160, 96, cams)


def test_eye_leaves_the_reach_box(capi):
    """a camera far outside the scene's reach box in the middle of a run"""
    far = S.camera_lookat((0.0, 40.0, -400.0), (0.0, 1.0, 0.0))
    cams = [S.default_camera()] * 4 + [far] * 4 + [S.default_camera()] * 4
    _same(capi, S.default_scene(), 160, 96, cams)
    _same(capi, _mixed_scene(), 160, 96, cams)


@pytest.mark.parametrize("size", [(157, 93), (161, 100), (3, 5)])
def test_ragged_frame_sizes(capi, size):
    """W not a multiple of 4, H not a multiple of 8"""
    _same(capi, S.default_scene(), size[0], size[1], [S.default_camera()] * 9)


def test_unaligned_caller_buffer(capi):
    _same(capi, S.default_scene(), 160, 96, [S.default_camera()] * 9, offset_words=1)


def test_small_ranking_groups(capi):
    """max_calls_per_launch lowered so that a ranking group holds 3 frames"""
    W, H = 160, 96
    _same(capi, S.default_scene(), W, H, [S.default_camera()] * 10, max_calls=3 * W * H)
    _same(capi, S.default_scene(), W, H, [S.default_camera()] * 4, max_calls=W * H - 1)


@pytest.mark.parametrize("which", ["default", "mixed"])
@pytest.mark.parametrize("where", ["inside_sphere", "under_floor", "orbit"])
def test_cameras_and_scenes(capi, which, where):
    scene = S.default_scene() if which == "default" else _mixed_scene()
    if where == "inside_sphere":
        o = scene["objects"][0]
        cam = S.camera_lookat(tuple(o[1]), (0.0, 1.0, 5.0))
    elif where == "under_floor":
        cam = S.camera_lookat((0.5, -1.5, -6.0), (0.0, 1.0, 0.0))
    else:
        cam = ORBIT[7]
    _same(capi, scene, 192, 120, [cam] * 10)


def test_batched_frames_match_oracle(capi, oracle):
    """8 frames of one camera at 320x240 against the oracle rendering them in one process"""
    W, H, refl = 320, 240, 20
    cam = S.default_camera()
    o = oracle.OracleRender(S.default_scene(), W, H, seed=99)
    want = [o.render(cam, refl).resolve()[1] for _ in range(8)]
    frames, counts, _, _, _ = _same(capi, S.default_scene(), W, H, [cam] * 8, depth=refl)
    for i in range(8):
        cases.assert_parity(frames[i].view(np.uint32), want[i], "batched frame %d" % i)
