"""Prototype + brute-force check of the primary-ray screen bounds (the host side of RFX_PRIMARY_CULL in rfx_trace_small.cu).

For every sphere / triangle of a constant-bank scene and one camera: a pixel rectangle outside of which no primary ray can pass
the kernel's hit test.  The check evaluates the kernel's own float32 expressions on every pixel (numpy, op for op) and asserts
that every accepting pixel lies inside the rectangle.  usage: primary_cull_proto.py [n_random_cameras]"""
import math
import sys

import numpy as np

F = np.float32
INT_LO, INT_HI = -(1 << 30), (1 << 30)
PIX_MARGIN = 3.0          # pixels: SSAA sub-samples and additive jitter reach up to 2 pixels to the right/top of the pixel origin


def sphere_rect(eye, cols, rz, w_half, h_half, centre, r2):
    """(x0, x1, y0, y1) inclusive pixel bounds, x0 > x1 = empty."""
    c0, c1, c2 = cols
    w = np.asarray(centre, float) - np.asarray(eye, float)
    wl = float(np.linalg.norm(w))
    r = math.sqrt(max(float(r2), 0.0))
    if not (math.isfinite(wl) and math.isfinite(r)):
        return (INT_LO, INT_HI, INT_LO, INT_HI)
    r_eff = r * 1.001 + 1e-3 * wl + 1e-30
    wx, wy, wz = float(c0 @ w), float(c1 @ w), float(c2 @ w)

    def axis(a, z, half):
        d2 = math.hypot(a, z)
        if d2 <= r_eff:
            return (INT_LO, INT_HI)
        th = math.atan2(a, z)
        al = math.asin(r_eff / d2)
        lo, hi = th - al, th + al
        lim = math.pi / 2 - 1e-4
        if hi <= -lim or lo >= lim:
            return None                       # entirely behind the eye in this projection
        p0 = INT_LO if lo <= -lim else rz * math.tan(lo) + half - PIX_MARGIN
        p1 = INT_HI if hi >= lim else rz * math.tan(hi) + half + PIX_MARGIN
        return (max(INT_LO, math.floor(p0)) if p0 != INT_LO else INT_LO, min(INT_HI, math.ceil(p1)) if p1 != INT_HI else INT_HI)

    xr = axis(wx, wz, w_half)
    yr = axis(wy, wz, h_half)
    if xr is None or yr is None:
        return (1, 0, 1, 0)
    return (int(xr[0]), int(xr[1]), int(yr[0]), int(yr[1]))


def tri_rect(eye, cols, rz, w_half, h_half, W, H, v0, ax):
    c0, c1, c2 = cols
    A = np.asarray(ax, float).reshape(3, 3)
    full = (INT_LO, INT_HI, INT_LO, INT_HI)
    if not np.all(np.isfinite(A)):
        return full
    det = np.linalg.det(A)
    if not math.isfinite(det) or abs(det) < 1e-30:
        return full
    B = np.linalg.inv(A)
    ea, eb, nn = B[:, 0], B[:, 1], B[:, 2]
    if not np.all(np.isfinite(B)):
        return full
    v0 = np.asarray(v0, float)
    E = np.asarray(eye, float)
    nl = float(np.linalg.norm(nn))
    emin = min(float(np.linalg.norm(ea)), float(np.linalg.norm(eb)))
    if nl <= 0 or emin <= 0:
        return full
    dist = abs(float(nn @ (E - v0))) / nl          # lower bound of the distance from the eye to any point of the triangle
    reach = float(np.linalg.norm(E - v0)) + float(np.linalg.norm(ea)) + float(np.linalg.norm(eb))
    if dist <= 1e-6 * reach:
        return full
    mu = 1e-3 + 1e-5 * reach / emin
    P = [v0 + u * ea + v * eb for (u, v) in ((-mu, -mu), (1 + 2 * mu, -mu), (-mu, 1 + 2 * mu))]
    D = math.hypot(max(w_half, W - w_half), max(h_half, H - h_half)) + 8.0
    znear = 0.5 * dist / math.sqrt(1.0 + (2.0 * D / rz) ** 2)
    cam = [np.array([c0 @ (p - E), c1 @ (p - E), c2 @ (p - E)]) for p in P]
    poly = []
    for i in range(3):
        a, b = cam[i], cam[(i + 1) % 3]
        ina, inb = a[2] >= znear, b[2] >= znear
        if ina:
            poly.append(a)
        if ina != inb:
            t = (znear - a[2]) / (b[2] - a[2])
            poly.append(a + t * (b - a))
    if not poly:
        return (1, 0, 1, 0)
    xs = [rz * p[0] / p[2] + w_half for p in poly]
    ys = [rz * p[1] / p[2] + h_half for p in poly]

    def clampi(v, fn):
        if not math.isfinite(v):
            return INT_LO if v < 0 else INT_HI
        return int(max(INT_LO, min(INT_HI, fn(v))))
    return (clampi(min(xs) - PIX_MARGIN, math.floor), clampi(max(xs) + PIX_MARGIN, math.ceil),
            clampi(min(ys) - PIX_MARGIN, math.floor), clampi(max(ys) + PIX_MARGIN, math.ceil))


def camera_ok(view):
    M = np.asarray(view, float).reshape(3, 3)
    return bool(np.all(np.abs(M.T @ M - np.eye(3)) < 1e-4))


def primary_rects(eye, view, rz, w_half, h_half, W, H, spheres, tris):
    """spheres: [(cx,cy,cz,r2)], tris: [(v0[3], ax[9])]"""
    M = np.asarray(view, float).reshape(3, 3)
    if not camera_ok(view) or not (math.isfinite(rz) and rz > 0):
        full = (INT_LO, INT_HI, INT_LO, INT_HI)
        return [full] * len(spheres), [full] * len(tris)
    cols = (M[:, 0], M[:, 1], M[:, 2])
    return ([sphere_rect(eye, cols, rz, w_half, h_half, s[:3], s[3]) for s in spheres],
            [tri_rect(eye, cols, rz, w_half, h_half, W, H, t[0], t[1]) for t in tris])


# ---- brute force: the kernel's float32 expressions on every pixel ------------------------------------------------------
def primary_rays(eye, view, rz, w_half, h_half, W, H, offx=0.0, offy=0.0):
    v = [F(x) for x in view]
    x = np.arange(W, dtype=F)[None, :]
    y = np.arange(H, dtype=F)[:, None]
    rx = (x - F(w_half)) + F(offx)
    ry = (y - F(h_half)) + F(offy)
    rzf = F(rz)
    d = [(rx * v[3 * i] + ry * v[3 * i + 1]) + rzf * v[3 * i + 2] for i in range(3)]
    return [np.broadcast_to(c, (H, W)).astype(F) for c in d]


def sphere_accept(eye, d, s):
    o = [F(e) for e in eye]
    a = (d[0] * d[0] + d[1] * d[1]) + d[2] * d[2]
    vx, vy, vz = o[0] - F(s[0]), o[1] - F(s[1]), o[2] - F(s[2])
    b = ((d[0] * F(2)) * vx + (d[1] * F(2)) * vy) + (d[2] * F(2)) * vz
    c = ((vx * vx + vy * vy) + vz * vz) - F(s[3])
    disc = b * b - (F(4) * a) * c
    return (disc >= 0) & (b < 0)


def tri_accept(eye, d, v0, ax):
    o = [F(e) for e in eye]
    ax = [F(x) for x in ax]
    p = [o[i] - F(v0[i]) for i in range(3)]

    def row(r, vec):
        return (vec[0] * ax[3 * r] + vec[1] * ax[3 * r + 1]) + vec[2] * ax[3 * r + 2]
    oz, rzz = row(2, p), row(2, d)
    with np.errstate(all="ignore"):
        t = -oz / rzz
        u = row(0, p) + t * row(0, d)
        v = row(1, p) + t * row(1, d)
        return (t > F(2.0 ** -63)) & (u >= 0) & (v >= 0) & (u + v < F(1)) & np.isfinite(t)


def check(eye, view, fov, W, H, spheres, tris, offsets=((0.0, 0.0),)):
    rz = F(F(W) / F(2) / F(math.tan(F(fov) / F(2))))
    w_half, h_half = F(W) / F(2), F(H) / F(2)
    srect, trect = primary_rects(eye, view, float(rz), float(w_half), float(h_half), W, H, spheres, tris)
    stats = []
    for offx, offy in offsets:
        d = primary_rays(eye, view, rz, w_half, h_half, W, H, offx, offy)
        for objs, rects, fn in ((spheres, srect, lambda s: sphere_accept(eye, d, s)), (tris, trect, lambda t: tri_accept(eye, d, t[0], t[1]))):
            for ob, r in zip(objs, rects):
                acc = fn(ob)
                ys, xs = np.nonzero(acc)
                if len(xs):
                    assert r[0] <= xs.min() and xs.max() <= r[1] and r[2] <= ys.min() and ys.max() <= r[3], (r, xs.min(), xs.max(), ys.min(), ys.max(), ob)
                    box = (xs.max() - xs.min() + 1) * (ys.max() - ys.min() + 1)
                else:
                    box = 0
                cx0, cx1, cy0, cy1 = max(r[0], 0), min(r[1], W - 1), max(r[2], 0), min(r[3], H - 1)
                stats.append((box, max(0, cx1 - cx0 + 1) * max(0, cy1 - cy0 + 1)))
    return stats


def scene_arrays(scene):
    """spheres and triangles of a scenes.py dict as the kernel sees them (float32 flattening of rfx_scene.cpp restated in numpy)."""
    sph, tris = [], []
    for ob in scene["objects"]:
        if ob[0] == "sphere":
            c, r = ob[1], F(ob[2])
            sph.append((F(c[0]), F(c[1]), F(c[2]), F(r * r)))
        elif ob[0] == "tri":
            v = [F(x) for x in ob[1]]
            v0, v1, v2 = np.array(v[0:3], F), np.array(v[3:6], F), np.array(v[6:9], F)
            e1, e2 = (v1 - v0).astype(float), (v2 - v0).astype(float)
            n = np.cross(e1, e2)
            n = n / np.linalg.norm(n)
            Bm = np.stack([e2, e1, -n], axis=1)            # columns v2-v0 | v1-v0 | -n
            tris.append((v0, np.linalg.inv(Bm).astype(F).reshape(9)))
    return sph, tris


def random_cameras(n, seed, sph):
    """default + orbit cameras, then random ones: around the scene, close to / inside a sphere, under the floor, looking away"""
    from reflaxman_b200 import scenes as S
    rng = np.random.default_rng(seed)
    cams = [S.default_camera()] + S.orbit_cameras(12)
    for _ in range(n):
        kind = rng.integers(0, 4)
        if kind == 0:
            eye = rng.uniform([-20, 0.05, -15], [20, 12, 15]); at = rng.uniform([-5, 0, -5], [5, 3, 5])
        elif kind == 1:
            s = sph[rng.integers(0, len(sph))]
            eye = np.array(s[:3], float) + rng.normal(size=3) * math.sqrt(float(s[3])) * rng.uniform(0.2, 1.5); at = rng.uniform([-5, 0, -5], [5, 3, 5])
        elif kind == 2:
            eye = rng.uniform([-10, -3, -8], [10, 0.0, 8]); at = rng.uniform([-5, -1, -5], [5, 3, 5])
        else:
            eye = rng.uniform([-10, 0.5, -8], [10, 6, 8]); at = eye + (eye - rng.uniform([-3, 0, -3], [3, 2, 3]))
        cams.append(S.camera_lookat(tuple(eye), tuple(at), float(rng.uniform(0.3, 2.6))))
    return cams


def assert_inside(eye, view, fov, W, H, spheres, tris, srect, trect, offsets=((0.0, 0.0), (1.99, 1.99))):
    """every pixel whose primary ray (or a sub-sample / jittered ray of it) passes an object's accept test lies inside that object's rectangle"""
    rz = F(F(W) / F(2) / F(math.tan(F(fov) / F(2))))
    w_half, h_half = F(W) / F(2), F(H) / F(2)
    for offx, offy in offsets:
        d = primary_rays(eye, view, rz, w_half, h_half, W, H, offx, offy)
        for objs, rects, fn in ((spheres, srect, lambda s: sphere_accept(eye, d, s)), (tris, trect, lambda t: tri_accept(eye, d, t[0], t[1]))):
            for ob, r in zip(objs, rects):
                ys, xs = np.nonzero(fn(ob))
                if len(xs):
                    assert r[0] <= xs.min() and xs.max() <= r[1] and r[2] <= ys.min() and ys.max() <= r[3], (tuple(r), xs.min(), xs.max(), ys.min(), ys.max(), ob)


if __name__ == "__main__":
    sys.path.insert(0, __file__.rsplit("/tools/", 1)[0])
    from reflaxman_b200 import scenes as S
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 20
    W, H = 480, 270
    sph, tris = scene_arrays(S.default_scene())
    cams = random_cameras(n, 7, sph)
    tot_box = tot_rect = 0
    for eye, view, fov in cams:
        st = check(eye, view, fov, W, H, sph, tris, offsets=((0.0, 0.0), (1.99, 1.99)))
        tot_box += sum(s[0] for s in st); tot_rect += sum(s[1] for s in st)
    print("ok: %d cameras, every accepting pixel inside its rectangle; rect area / tight box area = %.3f" % (len(cams), tot_rect / max(tot_box, 1)))
