"""CPU tests: pin the oracle (our C restatement) against the golden vectors generated from the unmodified
reference, and — where the reference binary is present — against the reference itself at config-1 size."""
import hashlib
import os

import numpy as np
import pytest

import cases
from reflaxman_b200 import scenes as S


@pytest.mark.parametrize("name", cases.GOLDEN)
def test_oracle_matches_golden_bit_exact(oracle, name):
    g = cases.load_golden(name)
    eng = cases.OracleEngine(oracle, g["scene"], g["W"], g["H"], g["seed"])
    frames = cases.replay(eng, g)
    for i, (rgbf, argb) in enumerate(frames):
        assert np.array_equal(argb, g["argb%d" % i]), "%s frame %d: ARGB differs from the reference" % (name, i)
        if "rgbf%d" % i in g:   # the large vectors keep the 8-bit image only
            assert np.array_equal(rgbf.view(np.uint32), g["rgbf%d" % i].view(np.uint32)), "%s frame %d: float image differs" % (name, i)


def test_oracle_plane_trace_matches_reference_plane_trace(oracle):
    """Plane::trace (Plane.cpp:36-73) is unreachable through the reference's Scene, so no render pins it: the golden vector
    holds 4096 direct calls of the reference's own function (oracle/ref_plane_probe.cpp: parallel rays, origins on the plane,
    2^-63 thresholds, the DELTA boundary, zero and unnormalised normals, shadow-ray magnitudes) — hit flag, drop, norm,
    reflected ray and distance, and the NULL-output shadow call.  The oracle's plane_trace must agree bit for bit; where the
    probe binary is present it is also re-run live on a different seed."""
    z = np.load(os.path.join(cases.GOLDEN_DIR, "plane_probe.npz"))
    got = oracle.plane_probe(z["inputs"])
    assert 0.2 < z["outputs"][:, 0].mean() < 0.5            # the probe exercises both outcomes
    assert np.array_equal(got.view(np.uint32), z["outputs"].view(np.uint32))
    if os.access(os.path.join(oracle.REF_DIR, "ref_plane_probe"), os.X_OK):
        inputs, outputs = oracle.run_plane_probe(2048, 20261018)
        assert np.array_equal(oracle.plane_probe(inputs).view(np.uint32), outputs.view(np.uint32))


def test_oracle_thread_count_invariance(oracle):
    cam = S.default_camera()
    a = oracle.OracleRender(S.default_scene(), 96, 64, nthreads=1).render(cam, 20).resolve()[1]
    b = oracle.OracleRender(S.default_scene(), 96, 64, nthreads=7).render(cam, 20).resolve()[1]
    assert np.array_equal(a, b)


def test_oracle_config1_hash(oracle):
    """config 1 (1024x768, depth 20, seed 12345): the port's images hash to what the reference produced."""
    want = cases.full_size_hashes()
    r = oracle.OracleRender(S.default_scene(), 1024, 768, seed=12345).render(S.default_camera(), 20)
    rgbf, argb = r.resolve()
    assert hashlib.sha256(argb.tobytes()).hexdigest() == want["default_1024x768_d20_seed12345"][0]
    assert hashlib.sha256(rgbf.tobytes()).hexdigest() == want["default_1024x768_d20_seed12345"][1]
    # SURVEY §8(d): 3.2111 rays per pixel at config 1
    assert abs(r.counters["rays"] / (1024 * 768) - 3.2111) < 1e-3


def test_oracle_config3_hash(oracle):
    """config 3's frame (7680x4320, depth 20, seed 12345, a reference screenshot preset): the port's 8-bit image hashes to what
    the unmodified reference produced — the GPU tests at that size compare against the port."""
    want = cases.full_size_hashes()
    r = oracle.OracleRender(S.default_scene(), 7680, 4320, seed=12345).render(S.default_camera(), 20)
    rgbf, argb = r.resolve()
    assert hashlib.sha256(argb.tobytes()).hexdigest() == want["default_7680x4320_d20_seed12345"][0]
    assert hashlib.sha256(rgbf.tobytes()).hexdigest() == want["default_7680x4320_d20_seed12345"][1]


def test_oracle_vs_reference_binary(oracle):
    """Where oracle/_ref/ref_render exists (build container and, via the gpurun snapshot, the GPU box): a scene and a
    camera the golden set does not contain, chunked renderNext, bit-exact."""
    if not oracle.have_ref():
        pytest.skip("oracle/_ref/ref_render not built here")
    scene = cases.small_synth()
    cams = S.orbit_cameras(8)[3:5]
    info, imgs = oracle.run_reference(120, 80, refl=6, frames=2, cams=cams, scene=scene, seed=4242, chunk=997)
    r = oracle.OracleRender(scene, 120, 80, seed=4242)
    for i, cam in enumerate(cams):
        rgbf, argb = r.render(cam, 6).resolve()
        assert np.array_equal(argb, imgs[i][1])
        assert np.array_equal(rgbf.view(np.uint32), imgs[i][0].view(np.uint32))


def test_camera_lookat_matches_reference_ctor(oracle):
    """scenes.camera_lookat (numpy float32) == the oracle's restatement of Camera(eye, at, fov), bit for bit."""
    import math
    for k in range(16):
        a = 2.0 * math.pi * k / 16
        c, s = math.cos(a), math.sin(a)
        rot = lambda p: (np.float32(c * p[0] + s * p[2]), np.float32(p[1]), np.float32(-s * p[0] + c * p[2]))
        eye, at = (S.DEFAULT_EYE, S.DEFAULT_AT) if k == 0 else (rot(S.DEFAULT_EYE), rot(S.DEFAULT_AT))
        v_np = S.camera_lookat(eye, at)[1]
        v_c = oracle.camera_lookat(eye, at)
        assert np.array_equal(v_np.view(np.uint32), v_c.view(np.uint32)), k


def test_rand_dirs_parallel_model(oracle):
    """The parallel formulation K1 implements (jump-ahead + accept flag + rank) reproduces the serial stream."""
    seed, n = 12345, 5000
    dirs, end_state = oracle.rand_dirs(seed, n)
    A, C = 214013, 2531011
    m = 3 * (2 * n + 4096)
    st = np.empty(m + 1, np.uint32)
    s = seed
    st[0] = s
    for i in range(m):
        s = (A * s + C) & 0xFFFFFFFF
        st[i + 1] = s
    r = ((st[1:] >> 16) & 0x7FFF).astype(np.float32)
    v = (r / np.float32(16383.5) - np.float32(1.0)).reshape(-1, 3)
    sq = (v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2]
    acc = np.nonzero(~(sq > np.float32(1.0)))[0]
    assert len(acc) >= n
    assert np.array_equal(v[acc[:n]].view(np.uint32), dirs.view(np.uint32))
    assert int(st[3 * (acc[n - 1] + 1)]) == end_state
    assert abs(len(acc) / (m // 3) - 0.5236) < 0.01


def test_constant_division_is_exact():
    """rfx_device.cuh::divExact — q0 = RN(r*c), rem = fma(-q0, D, r), q = fma(rem, c, q0) with c = RN(1/D) — equals the
    correctly rounded r / D on the whole input domain of each call site (exact rational arithmetic, exhaustive)."""
    from fractions import Fraction
    import math

    def rn32(x):
        if x == 0:
            return Fraction(0)
        sgn = -1 if x < 0 else 1
        x = abs(x)
        e = math.floor(math.log2(x))
        while Fraction(2) ** e > x:
            e -= 1
        while Fraction(2) ** (e + 1) <= x:
            e += 1
        ulp = Fraction(2) ** (e - 23)
        q = x / ulp
        n = q.numerator // q.denominator
        r = q - n
        if r > Fraction(1, 2) or (r == Fraction(1, 2) and (n & 1)):
            n += 1
        return sgn * n * ulp

    for D, hi, c_src in ((Fraction(32767, 2), 32768, 6.103701889514923e-05), (Fraction(32767), 32768, 3.0518509447574615e-05),
                         (Fraction(255), 256, 0.003921568859368563)):
        c = rn32(1 / D)
        assert float(c) == float(np.float32(c_src))          # the literal in rfx_device.cuh is RN(1/D)
        for r in range(hi):
            rf = Fraction(r)
            q0 = rn32(rf * c)
            rem = rn32(rf - q0 * D)
            assert rn32(q0 + rem * c) == rn32(rf / D), (D, r)


def test_rand_dirs_cycle_table_model(oracle):
    """The formulation K1 implements on the GPU (rfx_kernels.cu): the accept flag of a triple depends only on its start position
    on the LCG's 2^32-state cycle, the position of a seed follows from a bitwise discrete logarithm, and the stream visits
    positions p0, p0+3, ... in residue class p0 mod 3 until it wraps into the next class (0 -> 2 -> 1 -> 0).  Checked against
    the oracle's serial stream for a seed just before the wrap (all three classes) and an ordinary one."""
    A, C, M = 214013, 2531011, 1 << 32

    def jump(s, n):
        a, c = A, C
        while n:
            if n & 1:
                s = (a * s + c) % M
            c = (c * (a + 1)) % M
            a = (a * a) % M
            n >>= 1
        return s

    pow2 = []
    for k in range(32):
        c = jump(0, 1 << k)
        pow2.append(((jump(1, 1 << k) - c) % M, c))

    def position(s):                       # k_rng_locate's discrete logarithm
        pos, t = 0, 0
        for k in range(32):
            if ((t ^ s) >> k) & 1:
                a, c = pow2[k]
                t = (a * t + c) % M
                pos |= 1 << k
        assert t == s
        return pos

    def accept_at(p):                      # accept flag and states of the triple that starts at cycle position p
        s0 = jump(0, p % M)
        st = [s0]
        for _ in range(3):
            st.append((A * st[-1] + C) % M)
        r = ((np.array(st[1:], np.uint32) >> 16) & 0x7FFF).astype(np.float32)
        v = r / np.float32(16383.5) - np.float32(1.0)
        sq = (v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]
        return (not sq > np.float32(1.0)), s0, st[3], v

    for p0 in (M - 601, M - 602, M - 603, 123456789):
        seed = jump(0, p0)
        assert position(seed) == p0
        n = 300
        dirs, end_state = oracle.rand_dirs(seed, n)
        cls_seq = []
        got, end, p = [], None, p0
        while len(got) < n:
            acc, _, after, v = accept_at(p)
            cls_seq.append(p % 3)
            if acc:
                got.append(v)
                end = after
            p += 3
            if p >= M:
                p -= M                     # the wrapped position lands in the next residue class
        assert np.array_equal(np.array(got, np.float32).view(np.uint32), dirs.view(np.uint32)), p0
        assert end == end_state
        changes = [i for i in range(1, len(cls_seq)) if cls_seq[i] != cls_seq[i - 1]]
        if p0 > M - 1000:
            r0 = p0 % 3
            assert len(changes) == 1 and cls_seq[-1] == (2 if r0 == 0 else r0 - 1)
        else:
            assert not changes
