"""ctypes binding of the C ABI (include/reflax_c.h) — what the tests and bench.py call.

This is deliberately thin: every method is one C call.  The library is the in-tree
``reflaxman_b200/libreflax_b200.so`` (sm_100a only).  There is no CPU fallback: if the library is missing or no B200
is visible, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RFX_LIB") or os.path.join(HERE, "libreflax_b200.so")   # RFX_LIB: experimental variant (tools/variants.py)

_fp = C.POINTER(C.c_float)
_u32p = C.POINTER(C.c_uint32)


class RfxStats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("rays", "bounces", "shadow_rays", "samples", "kernel_launches",
                                          "h2d_bytes", "d2h_bytes", "trace_kernels")] + [("trace_kernel_ms", C.c_double)] + \
               [(n, C.c_uint64) for n in ("launches_small_fast", "launches_small_any", "launches_blob_fast", "launches_blob_any", "light_grids",
                                          "bvh_triangles", "bvh_spheres")]

    def as_dict(self):
        return {n: (float if n == "trace_kernel_ms" else int)(getattr(self, n)) for n, _ in self._fields_}


class RfxDeviceInfo(C.Structure):
    _fields_ = [("device", C.c_int), ("sm_count", C.c_int), ("cc_major", C.c_int), ("cc_minor", C.c_int),
                ("clock_khz", C.c_int), ("total_mem", C.c_uint64), ("name", C.c_char * 128)]


# every symbol include/reflax_c.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("rfx_create", C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    ("rfx_destroy", None, [C.c_void_p]),
    ("rfx_last_error", C.c_char_p, [C.c_void_p]),
    ("rfx_get_device_info", C.c_int, [C.c_void_p, C.POINTER(RfxDeviceInfo)]),
    ("rfx_version", C.c_char_p, []),
    ("rfx_scene_reset", C.c_int, [C.c_void_p, _fp, C.c_float]),
    ("rfx_add_light", C.c_int, [C.c_void_p, _fp, C.c_float, _fp, C.c_float]),
    ("rfx_add_sphere", C.c_int, [C.c_void_p, _fp, C.c_float, C.c_int, _fp, C.c_float, C.c_float]),
    ("rfx_add_triangle", C.c_int, [C.c_void_p, _fp, C.c_int, _fp, C.c_float, C.c_float]),
    ("rfx_add_mesh", C.c_int, [C.c_void_p, C.c_uint32, _fp, C.c_uint32, _u32p, C.c_int, _fp, C.c_float, C.c_float]),
    ("rfx_update_mesh", C.c_int, [C.c_void_p, C.c_int, _fp]),
    ("rfx_update_spheres", C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_int32), _fp]),
    ("rfx_update_lights", C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(C.c_int32), _fp]),
    ("rfx_set_triangle_texture", C.c_int, [C.c_void_p, C.c_int, C.c_int, _fp]),
    ("rfx_add_plane", C.c_int, [C.c_void_p, _fp, _fp, C.c_int, _fp, C.c_float, C.c_float]),
    ("rfx_add_texture_argb", C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, _u32p]),
    ("rfx_set_skybox", C.c_int, [C.c_void_p, C.c_int]),
    ("rfx_set_camera", C.c_int, [C.c_void_p, _fp, _fp, C.c_float]),
    ("rfx_set_seeds", C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    ("rfx_get_seeds", C.c_int, [C.c_void_p, _u32p]),
    ("rfx_skip_samples", C.c_int, [C.c_void_p, C.c_uint64]),
    ("rfx_selftest_rng", C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    ("rfx_selftest_light_grids", C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    ("rfx_selftest_eye_grid", C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    ("rfx_selftest_primary_bounds", C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("rfx_selftest_primary_bounds_host", C.c_int, [_fp, C.c_uint32, C.c_uint32, C.c_int, _fp, C.c_int, _fp, C.POINTER(C.c_int32)]),
    ("rfx_selftest_light_grid_host", C.c_int, [_fp, C.c_int, _fp, _fp, C.c_float, _fp, C.POINTER(C.c_int32), _u32p, C.c_uint64,
                                              C.POINTER(C.c_int32), C.c_uint64, C.POINTER(C.c_uint64)]),
    ("rfx_selftest_tri_bounds_host", C.c_int, [C.c_int, _fp, _fp, _fp]),
    ("rfx_selftest_far_bounds_host", C.c_int, [C.c_int, _fp, C.c_int, _fp, _fp, _fp, _fp, _fp, _fp]),
    ("rfx_selftest_eye_grid_host", C.c_int, [_fp, C.c_uint32, C.c_uint32, C.c_int, _fp, C.POINTER(C.c_int32), _u32p, C.c_uint64,
                                            C.POINTER(C.c_int32), C.c_uint64, C.POINTER(C.c_uint64)]),
    ("rfx_set_image_size", C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32]),
    ("rfx_render_begin", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    ("rfx_render_next", C.c_int, [C.c_void_p, C.c_uint32]),
    ("rfx_progress", C.c_float, [C.c_void_p]),
    ("rfx_additive_counter", C.c_int, [C.c_void_p]),
    ("rfx_in_progress", C.c_int, [C.c_void_p]),
    ("rfx_read_argb", C.c_int, [C.c_void_p, _u32p]),
    ("rfx_read_rgbf", C.c_int, [C.c_void_p, _fp]),
    ("rfx_read_image", C.c_int, [C.c_void_p, _fp, _u32p, C.c_int]),
    ("rfx_read_pixel", C.c_int, [C.c_void_p, C.c_int, C.c_int, _fp]),
    ("rfx_trace_rays", C.c_int, [C.c_void_p, C.c_int, _fp, _fp, C.c_int, _fp]),
    ("rfx_render_range", C.c_int, [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p, C.c_void_p]),
    ("rfx_render_finish", C.c_int, [C.c_void_p]),
    ("rfx_render_strips", C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]),
    ("rfx_buffer_alloc", C.c_int, [C.c_void_p, C.c_uint64, C.POINTER(C.c_void_p)]),
    ("rfx_buffer_free", C.c_int, [C.c_void_p, C.c_void_p]),
    ("rfx_buffer_read", C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64]),
    ("rfx_ipc_export", C.c_int, [C.c_void_p, C.c_void_p, C.c_char_p]),
    ("rfx_ipc_import", C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_void_p)]),
    ("rfx_ipc_close", C.c_int, [C.c_void_p, C.c_void_p]),
    ("rfx_read_signatures", C.c_int, [C.c_void_p, _u32p]),
    ("rfx_enable_signatures", C.c_int, [C.c_void_p, C.c_int]),
    ("rfx_render_frames", C.c_int, [C.c_void_p, C.c_int, _fp, C.c_int, C.c_int, C.c_void_p]),
    ("rfx_render_frames_device", C.c_int, [C.c_void_p, C.c_int, _fp, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    ("rfx_synchronize", C.c_int, [C.c_void_p]),
    ("rfx_get_stats", C.c_int, [C.c_void_p, C.POINTER(RfxStats)]),
    ("rfx_stats_reset", C.c_int, [C.c_void_p]),
    ("rfx_enable_profiling", C.c_int, [C.c_void_p, C.c_int]),
    ("rfx_set_option", C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    ("rfx_force_path", C.c_int, [C.c_void_p, C.c_int]),
    ("rfx_set_bvh_mode", C.c_int, [C.c_void_p, C.c_int]),
    ("rfx_set_tile_ordering", C.c_int, [C.c_void_p, C.c_int]),
]

_lib = None


def load():
    """dlopen the in-tree extension; fails loudly when it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("reflaxman_b200: %s is missing — run `python -m reflaxman_b200.build` "
                               "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(L, name)   # AttributeError if the library does not export what the header declares
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class RfxError(RuntimeError):
    pass


def _f(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a, a.ctypes.data_as(_fp)


def primary_bounds_host(cam, width, height, spheres, tris):
    """Pure host function (no GPU): the primary-ray screen bounds of ``spheres`` [(cx, cy, cz, r^2)] and ``tris`` [(v0[3], axTrans[9])]
    for ``cam`` = (eye, view, fov): (sphere rectangles [nS][4], triangle rectangles [nT][4]) as x0, x1, y0, y1 inclusive."""
    L = load()
    eye, view, fov = cam
    c = np.concatenate([np.asarray(eye, np.float32), np.asarray(view, np.float32), [np.float32(fov)]]).astype(np.float32)
    sp = np.ascontiguousarray(np.asarray(spheres, np.float32).reshape(-1, 4)) if len(spheres) else np.zeros((0, 4), np.float32)
    tr = np.ascontiguousarray(np.asarray([np.concatenate([np.asarray(t[0], np.float32), np.asarray(t[1], np.float32)]) for t in tris], np.float32).reshape(-1, 12)) \
        if len(tris) else np.zeros((0, 12), np.float32)
    out = (C.c_int32 * 96)()
    rc = L.rfx_selftest_primary_bounds_host(c.ctypes.data_as(_fp), width, height, len(sp), sp.ctypes.data_as(_fp), len(tr), tr.ctypes.data_as(_fp), out)
    if rc != 0:
        raise RfxError("rfx_selftest_primary_bounds_host failed (%d)" % rc)
    a = np.ctypeslib.as_array(out).reshape(24, 4).copy()
    return a[:len(sp)], a[16:16 + len(tr)]


def light_grid_host(light, spheres, box, reach_diagonal):
    """Pure host function (no GPU): the shadow-ray candidate grid of one far light.  light = (ox, oy, oz, radius), spheres [n][4] =
    (cx, cy, cz, r), box = (lo[3], hi[3]).  Returns None when the light is too close, else (uv[2][4], nx, ny, cell_start, items)."""
    L = load()
    lt = np.asarray(light, np.float32)
    sp = np.ascontiguousarray(np.asarray(spheres, np.float32).reshape(-1, 4))
    bx = np.asarray(box, np.float32).reshape(6)
    uv = np.zeros(8, np.float32)
    dims = (C.c_int32 * 2)()
    counts = (C.c_uint64 * 2)()
    args = (lt.ctypes.data_as(_fp), len(sp), sp.ctypes.data_as(_fp), bx.ctypes.data_as(_fp), C.c_float(reach_diagonal), uv.ctypes.data_as(_fp), dims)
    rc = L.rfx_selftest_light_grid_host(*args, None, 0, None, 0, counts)
    if rc != 0:
        raise RfxError("rfx_selftest_light_grid_host failed (%d)" % rc)
    if dims[0] == 0:
        return None
    cells = np.zeros(int(counts[0]), np.uint32)
    items = np.zeros(max(int(counts[1]), 1), np.int32)
    rc = L.rfx_selftest_light_grid_host(*args, cells.ctypes.data_as(_u32p), len(cells), items.ctypes.data_as(C.POINTER(C.c_int32)), len(items), counts)
    if rc != 0:
        raise RfxError("rfx_selftest_light_grid_host failed (%d)" % rc)
    return uv.reshape(2, 4), int(dims[0]), int(dims[1]), cells, items[:int(counts[1])]


def tri_bounds_host(tris, reach):
    """Pure host function (no GPU): the boxes of the triangle hierarchy.  tris [n][12] = (v0[3], axTrans[9] row-major), reach = (lo[3], hi[3])
    of every ray origin.  Returns boxes [n][6] = (lo[3], hi[3])."""
    L = load()
    tr = np.ascontiguousarray(np.asarray(tris, np.float32).reshape(-1, 12))
    rc_ = np.ascontiguousarray(np.asarray(reach, np.float32).reshape(6))
    out = np.zeros((len(tr), 6), np.float32)
    if L.rfx_selftest_tri_bounds_host(len(tr), tr.ctypes.data_as(_fp), rc_.ctypes.data_as(_fp), out.ctypes.data_as(_fp)) != 0:
        raise RfxError("rfx_selftest_tri_bounds_host failed")
    return out


def far_bounds_host(spheres, tris, reach):
    """Pure host function (no GPU): the hierarchies' boxes in a scene with a plane.  spheres [n][4] = (cx, cy, cz, r), tris [m][12] =
    (v0[3], axTrans[9] row-major), reach = (lo[3], hi[3]) of the box the margins are sized for.  Returns (sphere_boxes [n][6],
    tri_boxes [m][6] (slivers and non-finite triangles: (-inf, +inf), tested after the walk), sphere_reach [6], tri_reach [6],
    (grow_spheres, grow_triangles)): a query from origin o grows every box by grow * (sum of o's per-axis distances outside the
    reach box of its kind)."""
    L = load()
    sp = np.ascontiguousarray(np.asarray(spheres, np.float32).reshape(-1, 4))
    tr = np.ascontiguousarray(np.asarray(tris, np.float32).reshape(-1, 12))
    rc_ = np.ascontiguousarray(np.asarray(reach, np.float32).reshape(6))
    sb = np.zeros((max(len(sp), 1), 6), np.float32)
    tb = np.zeros((max(len(tr), 1), 6), np.float32)
    reaches = np.zeros(12, np.float32)
    grow = np.zeros(2, np.float32)
    if L.rfx_selftest_far_bounds_host(len(sp), sp.ctypes.data_as(_fp), len(tr), tr.ctypes.data_as(_fp), rc_.ctypes.data_as(_fp), sb.ctypes.data_as(_fp),
                                      tb.ctypes.data_as(_fp), reaches.ctypes.data_as(_fp), grow.ctypes.data_as(_fp)) != 0:
        raise RfxError("rfx_selftest_far_bounds_host failed")
    return sb[:len(sp)], tb[:len(tr)], reaches[:6], reaches[6:], (float(grow[0]), float(grow[1]))


def eye_grid_host(cam, width, height, spheres):
    """Pure host function (no GPU): the screen grid of the first query for ``cam`` and spheres [n][4] = (cx, cy, cz, r^2).
    Returns None when the camera gets no grid, else (nx, ny, shift, cell_start, items)."""
    L = load()
    eye, view, fov = cam
    c = np.concatenate([np.asarray(eye, np.float32), np.asarray(view, np.float32), [np.float32(fov)]]).astype(np.float32)
    sp = np.ascontiguousarray(np.asarray(spheres, np.float32).reshape(-1, 4))
    dims = (C.c_int32 * 3)()
    counts = (C.c_uint64 * 2)()
    args = (c.ctypes.data_as(_fp), width, height, len(sp), sp.ctypes.data_as(_fp), dims)
    if L.rfx_selftest_eye_grid_host(*args, None, 0, None, 0, counts) != 0:
        raise RfxError("rfx_selftest_eye_grid_host failed")
    if dims[0] == 0:
        return None
    cells = np.zeros(int(counts[0]), np.uint32)
    items = np.zeros(max(int(counts[1]), 1), np.int32)
    if L.rfx_selftest_eye_grid_host(*args, cells.ctypes.data_as(_u32p), len(cells), items.ctypes.data_as(C.POINTER(C.c_int32)), len(items), counts) != 0:
        raise RfxError("rfx_selftest_eye_grid_host failed")
    return int(dims[0]), int(dims[1]), int(dims[2]), cells, items[:int(counts[1])]


def pack_cameras(cams):
    """[(eye[3], view[9], fov), ...] -> contiguous float32 [n, 13] as rfx_render_frames expects."""
    out = np.zeros((len(cams), 13), np.float32)
    for i, (eye, view, fov) in enumerate(cams):
        out[i, 0:3] = eye
        out[i, 3:12] = view
        out[i, 12] = fov
    return out


class Context:
    """One rfx_ctx: one GPU, one host thread (the reference's Render is single-threaded and non-reentrant)."""

    def __init__(self, device=0):
        self.L = load()
        h = C.c_void_p()
        rc = self.L.rfx_create(C.byref(h), device)
        if rc != 0:
            raise RfxError("rfx_create failed (%d): %s" % (rc, self.L.rfx_last_error(None).decode()))
        self.h = h
        self.W = self.H = 0
        self._mesh_vertices = {}   # first object index of each mesh -> its vertex count

    def close(self):
        if getattr(self, "h", None):
            self.L.rfx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc, what):
        if rc < 0:
            raise RfxError("%s failed (%d): %s" % (what, rc, self.L.rfx_last_error(self.h).decode()))
        return rc

    # ---- scene -----------------------------------------------------------------------------------------------
    def load_scene(self, scene):
        """Issue a scenes.py dict through the scene-building calls, in the reference's order (Render.cpp:32-54).  Returns the first
        object index of each "mesh" entry, in order (what :meth:`update_mesh` takes)."""
        rgb, p = scene["ambient"]
        self._ck(self.L.rfx_scene_reset(self.h, _f(rgb)[1], C.c_float(p)), "rfx_scene_reset")
        self._mesh_vertices = {}
        meshes = []
        tex_ids = []
        for t in scene["textures"]:
            tex_ids.append(self.add_texture(t))
        if scene.get("skybox") is not None:
            self._ck(self.L.rfx_set_skybox(self.h, self.add_texture(scene["skybox"])), "rfx_set_skybox")
        for o, r, c, pw in scene["lights"]:
            self._ck(self.L.rfx_add_light(self.h, _f(o)[1], C.c_float(r), _f(c)[1], C.c_float(pw)), "rfx_add_light")
        for ob in scene["objects"]:
            if ob[0] == "sphere":
                _, c, r, mt, col, refl, tr = ob
                self._ck(self.L.rfx_add_sphere(self.h, _f(c)[1], C.c_float(r), mt, _f(col)[1], C.c_float(refl), C.c_float(tr)), "rfx_add_sphere")
            elif ob[0] == "tri":
                _, v, mt, col, refl, tr, tex, uv = ob
                idx = self._ck(self.L.rfx_add_triangle(self.h, _f(v)[1], mt, _f(col)[1], C.c_float(refl), C.c_float(tr)), "rfx_add_triangle")
                if tex >= 0:
                    self._ck(self.L.rfx_set_triangle_texture(self.h, idx, tex_ids[tex], _f(uv)[1]), "rfx_set_triangle_texture")
            elif ob[0] == "mesh":
                _, xyz, idx, mt, col, refl, tr = ob
                meshes.append(self.add_mesh(xyz, idx, mt, col, refl, tr))
            elif ob[0] == "plane":
                _, pos, nrm, mt, col, refl, tr = ob
                self._ck(self.L.rfx_add_plane(self.h, _f(pos)[1], _f(nrm)[1], mt, _f(col)[1], C.c_float(refl), C.c_float(tr)), "rfx_add_plane")
            else:
                raise ValueError(ob[0])
        return meshes

    def add_mesh(self, xyz, idx, mtype, rgb, refl, transp):
        """rfx_add_mesh: xyz [N][3] vertices, idx [M][3] vertex indices; returns the object index of the first of the M triangles."""
        v = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        ix = np.ascontiguousarray(idx, dtype=np.uint32).reshape(-1, 3)
        first = self._ck(self.L.rfx_add_mesh(self.h, v.shape[0], v.ctypes.data_as(_fp), ix.shape[0], ix.ctypes.data_as(_u32p), mtype,
                                             _f(rgb)[1], C.c_float(refl), C.c_float(transp)), "rfx_add_mesh")
        self._mesh_vertices[first] = v.shape[0]
        return first

    def update_mesh(self, first, xyz):
        """rfx_update_mesh: new vertices xyz [N][3] for the mesh whose first triangle is object ``first`` (N as given to add_mesh).
        True: the device scene was updated in place; False: the scene is re-flattened on the host at the next render."""
        v = np.ascontiguousarray(xyz, dtype=np.float32).reshape(-1, 3)
        n = self._mesh_vertices.get(first)
        if n is not None and v.shape[0] != n:
            raise ValueError("update_mesh: %d vertices given, the mesh has %d" % (v.shape[0], n))
        return self._ck(self.L.rfx_update_mesh(self.h, first, v.ctypes.data_as(_fp)), "rfx_update_mesh") == 1

    def update_spheres(self, objects, spheres):
        """rfx_update_spheres: objects [n] sphere object indices, spheres [n][4] rows of their new (cx, cy, cz, r); a repeated object
        takes its last row.  True: the device scene was updated in place; False: the scene is re-flattened on the host at the next
        render."""
        ob = np.ascontiguousarray(objects, dtype=np.int32).reshape(-1)
        sp = np.ascontiguousarray(spheres, dtype=np.float32)
        if sp.ndim != 2 or sp.shape[1] != 4 or sp.shape[0] != ob.shape[0]:
            raise ValueError("update_spheres: %d objects need [%d, 4] spheres, got %s" % (ob.shape[0], ob.shape[0], sp.shape))
        return self._ck(self.L.rfx_update_spheres(self.h, ob.shape[0], ob.ctypes.data_as(C.POINTER(C.c_int32)), sp.ctypes.data_as(_fp)),
                        "rfx_update_spheres") == 1

    def update_lights(self, lights, records):
        """rfx_update_lights: lights [n] light indices, records [n][8] rows of their new (origin[3], radius, rgb[3], power), as
        rfx_add_light takes them; a repeated light takes its last row.  True: the device scene was updated in place (the grids of far
        lights built on the GPU); False: the scene is re-flattened on the host at the next render."""
        li = np.ascontiguousarray(lights, dtype=np.int32).reshape(-1)
        rec = np.ascontiguousarray(records, dtype=np.float32)
        if rec.ndim != 2 or rec.shape[1] != 8 or rec.shape[0] != li.shape[0]:
            raise ValueError("update_lights: %d lights need [%d, 8] records, got %s" % (li.shape[0], li.shape[0], rec.shape))
        return self._ck(self.L.rfx_update_lights(self.h, li.shape[0], li.ctypes.data_as(C.POINTER(C.c_int32)), rec.ctypes.data_as(_fp)),
                        "rfx_update_lights") == 1

    def light_grids_selftest(self):
        """rfx_selftest_light_grids: (lights whose device grid differs from the host's rebuild, lights with a grid on the device, lights
        with a grid on the host)"""
        out = (C.c_uint64 * 3)()
        self._ck(self.L.rfx_selftest_light_grids(self.h, out), "rfx_selftest_light_grids")
        return int(out[0]), int(out[1]), int(out[2])

    def eye_grid_selftest(self):
        """rfx_selftest_eye_grid: (differences between the eye grid the last blob render used and the host's binning, items on the
        device (0: no grid or dropped), items on the host, device builds dropped since creation)"""
        out = (C.c_uint64 * 4)()
        self._ck(self.L.rfx_selftest_eye_grid(self.h, out), "rfx_selftest_eye_grid")
        return int(out[0]), int(out[1]), int(out[2]), int(out[3])

    def add_texture(self, argb):
        if argb is None:
            return self._ck(self.L.rfx_add_texture_argb(self.h, 0, 0, None), "rfx_add_texture_argb")
        a = np.ascontiguousarray(argb, dtype=np.uint32)
        return self._ck(self.L.rfx_add_texture_argb(self.h, a.shape[1], a.shape[0], a.ctypes.data_as(_u32p)), "rfx_add_texture_argb")

    # ---- camera / seeds ----------------------------------------------------------------------------------------
    def set_camera(self, cam):
        eye, view, fov = cam
        self._ck(self.L.rfx_set_camera(self.h, _f(eye)[1], _f(view)[1], C.c_float(fov)), "rfx_set_camera")

    def set_seeds(self, seed_vector3=12345, seed_render=12345):
        self._ck(self.L.rfx_set_seeds(self.h, seed_vector3 & 0xFFFFFFFF, seed_render & 0xFFFFFFFF), "rfx_set_seeds")

    def get_seeds(self):
        out = (C.c_uint32 * 2)()
        self._ck(self.L.rfx_get_seeds(self.h, out), "rfx_get_seeds")
        return int(out[0]), int(out[1])

    def selftest_rng(self):
        """(triples of the whole LCG cycle on which K1's integer accept test and the reference's float expression disagree,
        triples inside the guard band)"""
        out = (C.c_uint64 * 2)()
        self._ck(self.L.rfx_selftest_rng(self.h, out), "rfx_selftest_rng")
        return int(out[0]), int(out[1])

    def selftest_primary_bounds(self):
        """Screen bounds of the scene's objects for the primary rays of the current camera and image size:
        (sphere rectangles [nS][4], triangle rectangles [nT][4]) as x0, x1, y0, y1 inclusive (x0 > x1: no pixel)."""
        out = (C.c_int32 * 96)()
        cnt = (C.c_int32 * 2)()
        self._ck(self.L.rfx_selftest_primary_bounds(self.h, out, cnt), "rfx_selftest_primary_bounds")
        a = np.ctypeslib.as_array(out).reshape(24, 4).copy()
        return a[:cnt[0]], a[16:16 + cnt[1]]

    def skip_samples(self, n):
        self._ck(self.L.rfx_skip_samples(self.h, n), "rfx_skip_samples")

    # ---- Render ------------------------------------------------------------------------------------------------
    def set_image_size(self, w, h):
        self._ck(self.L.rfx_set_image_size(self.h, w, h), "rfx_set_image_size")
        self.W, self.H = int(w), int(h)

    def render_begin(self, refl, samples=1, additive=False):
        self._ck(self.L.rfx_render_begin(self.h, refl, samples, 1 if additive else 0), "rfx_render_begin")

    def render_next(self, pixels):
        return self._ck(self.L.rfx_render_next(self.h, pixels), "rfx_render_next") == 1

    def render(self, cam, refl, samples=1, additive=False, chunk=None):
        """renderBegin + renderNext(chunk) until done, as Pulse does (reference Pulse.cpp:124-131,176-186)."""
        self.set_camera(cam)
        self.render_begin(refl, samples, additive)
        chunk = chunk or self.W * self.H
        while self.render_next(chunk):
            pass
        return self

    def progress(self):
        return float(self.L.rfx_progress(self.h))

    def additive_counter(self):
        return int(self.L.rfx_additive_counter(self.h))

    def in_progress(self):
        return bool(self.L.rfx_in_progress(self.h))

    def read_argb(self):
        out = np.empty((self.H, self.W), np.uint32)
        self._ck(self.L.rfx_read_argb(self.h, out.ctypes.data_as(_u32p)), "rfx_read_argb")
        return out

    def read_rgbf(self):
        out = np.empty((self.H, self.W, 3), np.float32)
        self._ck(self.L.rfx_read_rgbf(self.h, out.ctypes.data_as(_fp)), "rfx_read_rgbf")
        return out

    def read_image(self, divide=True):
        """rfx_read_image: (float image [H, W, 3], ARGB [H, W]).  divide=False reads the raw sums of the additive passes, as
        Render::copyImage packs them; divide=True divides by the additive counter as imagePixel does."""
        rgbf = np.empty((self.H, self.W, 3), np.float32)
        argb = np.empty((self.H, self.W), np.uint32)
        self._ck(self.L.rfx_read_image(self.h, rgbf.ctypes.data_as(_fp), argb.ctypes.data_as(_u32p), 1 if divide else 0), "rfx_read_image")
        return rgbf, argb

    def read_pixel(self, x, y):
        out = (C.c_float * 3)()
        self._ck(self.L.rfx_read_pixel(self.h, x, y, out), "rfx_read_pixel")
        return np.array(out[:], np.float32)

    # ---- frame splitting / shared buffers ---------------------------------------------------------------------
    def render_range(self, p0, p1, argb_device_ptr=0, stream=0):
        self._ck(self.L.rfx_render_range(self.h, p0, p1, C.c_void_p(int(argb_device_ptr) or None), C.c_void_p(int(stream) or None)), "rfx_render_range")

    def render_strips(self, strip_rows, world, rank, argb_device_ptr, stream=0):
        self._ck(self.L.rfx_render_strips(self.h, strip_rows, world, rank, C.c_void_p(int(argb_device_ptr)), C.c_void_p(int(stream) or None)), "rfx_render_strips")

    def render_finish(self):
        self._ck(self.L.rfx_render_finish(self.h), "rfx_render_finish")

    def buffer_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self.L.rfx_buffer_alloc(self.h, nbytes, C.byref(p)), "rfx_buffer_alloc")
        return p.value

    def buffer_free(self, ptr):
        self._ck(self.L.rfx_buffer_free(self.h, C.c_void_p(ptr)), "rfx_buffer_free")

    def buffer_read(self, ptr, out):
        self._ck(self.L.rfx_buffer_read(self.h, C.c_void_p(ptr), C.c_void_p(out.ctypes.data), out.nbytes), "rfx_buffer_read")
        return out

    def ipc_export(self, ptr):
        buf = C.create_string_buffer(64)
        self._ck(self.L.rfx_ipc_export(self.h, C.c_void_p(ptr), buf), "rfx_ipc_export")
        return buf.raw

    def ipc_import(self, handle):
        p = C.c_void_p()
        self._ck(self.L.rfx_ipc_import(self.h, handle, C.byref(p)), "rfx_ipc_import")
        return p.value

    def ipc_close(self, ptr):
        self._ck(self.L.rfx_ipc_close(self.h, C.c_void_p(ptr)), "rfx_ipc_close")

    def trace_rays(self, origins, rays, refl):
        o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
        r = np.ascontiguousarray(rays, dtype=np.float32).reshape(-1, 3)
        out = np.empty_like(o)
        self._ck(self.L.rfx_trace_rays(self.h, o.shape[0], o.ctypes.data_as(_fp), r.ctypes.data_as(_fp), refl, out.ctypes.data_as(_fp)), "rfx_trace_rays")
        return out

    def enable_signatures(self, on=True):
        self._ck(self.L.rfx_enable_signatures(self.h, 1 if on else 0), "rfx_enable_signatures")

    def read_signatures(self):
        out = np.empty((self.H, self.W), np.uint32)
        self._ck(self.L.rfx_read_signatures(self.h, out.ctypes.data_as(_u32p)), "rfx_read_signatures")
        return out

    # ---- batch -------------------------------------------------------------------------------------------------
    def render_frames(self, cams, refl, samples=1, out=None):
        """Host-buffer batch render; ``out``: uint32 array [n, H, W] (pinned for full copy/compute overlap)."""
        packed = cams if isinstance(cams, np.ndarray) else pack_cameras(cams)
        n = packed.shape[0]
        if out is None:
            out = np.empty((n, self.H, self.W), np.uint32)
        ptr = out.ctypes.data if isinstance(out, np.ndarray) else int(out)
        self._ck(self.L.rfx_render_frames(self.h, n, packed.ctypes.data_as(_fp), refl, samples, C.c_void_p(ptr)), "rfx_render_frames")
        return out

    def render_frames_device(self, cams, refl, samples, argb_device_ptr, stream=0):
        packed = cams if isinstance(cams, np.ndarray) else pack_cameras(cams)
        self._ck(self.L.rfx_render_frames_device(self.h, packed.shape[0], packed.ctypes.data_as(_fp), refl, samples,
                                                 C.c_void_p(int(argb_device_ptr)), C.c_void_p(int(stream))), "rfx_render_frames_device")

    def synchronize(self):
        self._ck(self.L.rfx_synchronize(self.h), "rfx_synchronize")

    def stats(self):
        s = RfxStats()
        self._ck(self.L.rfx_get_stats(self.h, C.byref(s)), "rfx_get_stats")
        return s.as_dict()

    def stats_reset(self):
        self._ck(self.L.rfx_stats_reset(self.h), "rfx_stats_reset")

    def enable_profiling(self, on=True):
        self._ck(self.L.rfx_enable_profiling(self.h, 1 if on else 0), "rfx_enable_profiling")

    def set_option(self, name, value):
        """tuning / test hook (include/reflax_c.h): "max_calls_per_launch", "copy_streams", "light_grid_items", ...; results never
        depend on it"""
        self._ck(self.L.rfx_set_option(self.h, name.encode(), int(value)), "rfx_set_option")

    def force_path(self, path):
        """0 automatic, 1 constant-bank kernels when the scene fits, 2 blob kernels, 3 general blob kernel only (tests)."""
        self._ck(self.L.rfx_force_path(self.h, path), "rfx_force_path")

    def set_bvh_mode(self, mode):
        """0 automatic (hierarchies over the spheres / the triangles when there are more than 32 of them), 1 always (whenever there
        are any), 2 never (list walk).  In scenes with a plane, queries from outside the box the margins are sized for grow the boxes
        they test (far_bounds_host)."""
        self._ck(self.L.rfx_set_bvh_mode(self.h, mode), "rfx_set_bvh_mode")

    def set_tile_ordering(self, on=True):
        self._ck(self.L.rfx_set_tile_ordering(self.h, 1 if on else 0), "rfx_set_tile_ordering")

    def device_info(self):
        d = RfxDeviceInfo()
        self._ck(self.L.rfx_get_device_info(self.h, C.byref(d)), "rfx_get_device_info")
        return {"device": d.device, "sm_count": d.sm_count, "cc": (d.cc_major, d.cc_minor), "clock_khz": d.clock_khz,
                "total_mem": int(d.total_mem), "name": d.name.decode()}
