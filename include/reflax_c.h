/* reflax_c.h — the drop-in boundary: a plain C ABI over the B200 (sm_100a) trace-and-shade path.
 *
 * ReflaxMan has no plugin/FFI layer; its hot path sits behind the public surface of the C++ classes Render, Scene
 * and Camera (reference src/common/Render.h:22-41, Scene.h:29-39, Camera.h:50-52) whose only client is Pulse
 * (reference Pulse.cpp:38,96,108-131,174-207,273-278,448-457).  Each entry point below names the reference member
 * it stands in for.  The C++ shim in reflaxman_b200/shim/ (classes Render/Scene/Camera/... with the reference's
 * names and members) forwards to these calls, so src/linux/main.cpp and src/windows/Main.cpp build against it
 * unchanged; INTEGRATION.md shows the binding.
 *
 * Conventions: plain pointers and sizes only; the caller owns every input buffer (copied before return); the
 * context owns all device memory; every call returns RFX_OK (0) or a negative error code and never throws
 * (reference convention: no exceptions, bool/silent fallbacks — Render.cpp:143-144, Texture.cpp:34,175);
 * rfx_last_error() gives the text.  One context drives one GPU from one host thread (the reference is
 * single-threaded and non-reentrant, SURVEY §8b).  There is no CPU fallback: without a usable sm_100 device
 * rfx_create() fails.
 *
 * Framebuffer convention (reference Render.cpp:154-156, Color.cpp:114-117): row 0 is the BOTTOM scanline,
 * ARGB is 0x00RRGGBB with alpha 0, channel = (unsigned char)(c * 255.999f).
 */
#ifndef REFLAX_C_H
#define REFLAX_C_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RFX_API __attribute__((visibility("default")))

typedef struct rfx_ctx rfx_ctx;

enum
{
  RFX_OK = 0,
  RFX_ERR_ARG = -1,     /* bad argument / bad state (the reference would assert, then fall back silently) */
  RFX_ERR_CUDA = -2,    /* CUDA runtime error (text in rfx_last_error) */
  RFX_ERR_NODEV = -3,   /* no usable sm_100 device: there is no CPU fallback */
  RFX_ERR_RNG = -4      /* random-stream ranking ran out of its over-provisioned draws (> 7 sigma event; fatal) */
};

enum { RFX_MT_METAL = 0, RFX_MT_DIELECTRIC = 1 };   /* reference Material.h:8 */

typedef struct rfx_stats
{
  uint64_t rays;            /* bounce-loop iterations + shadow rays cast since rfx_stats_reset (SURVEY §8d "ray") */
  uint64_t bounces;         /* reference Scene.cpp:80 iterations */
  uint64_t shadow_rays;     /* reference Scene.cpp:125-143 */
  uint64_t samples;         /* Scene::trace calls */
  uint64_t kernel_launches; /* kernels of ours launched */
  uint64_t h2d_bytes;       /* host->device bytes copied by the library */
  uint64_t d2h_bytes;       /* device->host bytes copied by the library */
  uint64_t trace_kernels;   /* K2 launches timed while profiling was enabled */
  double trace_kernel_ms;   /* their summed device time (CUDA events on the launching stream); 0 unless rfx_enable_profiling */
  /* K2 launches by kernel family: constant-bank fast kernel (k_trace_small<FEAT, MULTI>), constant-bank general kernel
   * (k_trace_small_any), blob batch kernel (k_trace_blob<MULTI>), blob general kernel (k_trace) */
  uint64_t launches_small_fast, launches_small_any, launches_blob_fast, launches_blob_any;
  uint64_t light_grids;     /* lights of the uploaded scene whose shadow queries use a candidate grid (not a counter: survives rfx_stats_reset) */
  uint64_t bvh_triangles;   /* triangles of the uploaded scene under a bounding-volume hierarchy, 0 = they are walked one by one (not a counter) */
} rfx_stats;

typedef struct rfx_device_info
{
  int device;
  int sm_count;
  int cc_major, cc_minor;
  int clock_khz;            /* cudaDevAttrClockRate */
  uint64_t total_mem;
  char name[128];
} rfx_device_info;

/* ---- lifetime ------------------------------------------------------------------------------------------- */
/* Render::Render / ~Render (reference Render.cpp:5-23).  device = CUDA ordinal.  The context starts EMPTY (no
 * default scene): the shim's Render::loadScene issues the reference's scene through the calls below.
 * Creation builds the accept-count table of the random stream's LCG cycle on the device (about 5 ms, 8.4 MB). */
RFX_API int rfx_create(rfx_ctx ** out, int device);
RFX_API void rfx_destroy(rfx_ctx * ctx);
RFX_API const char * rfx_last_error(const rfx_ctx * ctx);       /* ctx may be NULL: last rfx_create failure */
RFX_API int rfx_get_device_info(const rfx_ctx * ctx, rfx_device_info * out);
RFX_API const char * rfx_version(void);

/* ---- scene (reference Scene.h:29-39; use at Render.cpp:32-54).  Objects keep insertion order: closest-hit
 * ties go to the earlier object (reference Scene.cpp:98, strict <).  Upload happens lazily at rfx_render_begin,
 * because the reference mutates triangles after insertion (Triangle::setTexture, Render.cpp:52-54). ---------- */
RFX_API int rfx_scene_reset(rfx_ctx * ctx, const float ambient_rgb[3], float ambient_power);   /* Scene::Scene(Color,float), Scene.cpp:10-15 */
RFX_API int rfx_add_light(rfx_ctx * ctx, const float origin[3], float radius, const float rgb[3], float power); /* Scene::addLight, Scene.cpp:47-58 -> light index */
RFX_API int rfx_add_sphere(rfx_ctx * ctx, const float center[3], float radius, int mtype, const float rgb[3],
                           float reflectivity, float transparency);                             /* Scene::addSphere, Scene.cpp:29-39 -> object index */
RFX_API int rfx_add_triangle(rfx_ctx * ctx, const float v[9], int mtype, const float rgb[3], float reflectivity,
                             float transparency);                                               /* Scene::addTriangle, Scene.cpp:41-46 -> object index */
/* an indexed triangle mesh: triangle k = rfx_add_triangle(xyz[idx[3k]], xyz[idx[3k+1]], xyz[idx[3k+2]]), added in order with one
 * material (xyz = n_vertices x 3 floats, idx = n_tris x 3 vertex indices).  Returns the object index of the first triangle; the others
 * follow it.  An index >= n_vertices, a NULL pointer or n_tris = 0 adds nothing and returns RFX_ERR_ARG.  Mesh triangles are ordinary
 * objects (rfx_set_triangle_texture applies to each). */
RFX_API int rfx_add_mesh(rfx_ctx * ctx, uint32_t n_vertices, const float * xyz, uint32_t n_tris, const uint32_t * idx, int mtype,
                         const float rgb[3], float reflectivity, float transparency);
RFX_API int rfx_set_triangle_texture(rfx_ctx * ctx, int object, int texture, const float uv[6]); /* Triangle::setTexture, Triangle.cpp:110-120 (u1,v1,u2,v2,u3,v3) */
RFX_API int rfx_add_plane(rfx_ctx * ctx, const float pos[3], const float norm[3], int mtype, const float rgb[3],
                          float reflectivity, float transparency);                              /* Plane::Plane, Plane.cpp:9-14 (no Scene::addPlane exists upstream) */
/* Scene::addTexture (Scene.cpp:60-65) with the pixels already decoded (0xAARRGGBB, row 0 = v 0, Texture.cpp:34-108).
 * argb == NULL or w*h == 0 is a texture whose file failed to load: sampling it gives the reference's grey
 * checker (Texture.cpp:242-243).  Returns the texture id. */
RFX_API int rfx_add_texture_argb(rfx_ctx * ctx, uint32_t w, uint32_t h, const uint32_t * argb);
RFX_API int rfx_set_skybox(rfx_ctx * ctx, int texture);   /* Scene::setSkyboxTexture / Skybox::loadTexture, Skybox.cpp:21-37; -1 or an empty texture = none */

/* ---- camera (reference Camera.h:50-52; snapshot taken by renderBegin, Render.cpp:125-126) ------------------ */
RFX_API int rfx_set_camera(rfx_ctx * ctx, const float eye[3], const float view[9] /* row-major _11.._33 */, float fov);

/* ---- random streams (reference trace_math.h:34-39).  seed_vector3 drives Vector3::randomInsideSphere
 * (one randDir per Scene::trace call, Scene.cpp:75); seed_render drives the additive-mode pixel jitter
 * (Render.cpp:177-178).  Both streams continue across frames exactly as in one reference process. ----------- */
RFX_API int rfx_set_seeds(rfx_ctx * ctx, uint32_t seed_vector3, uint32_t seed_render);
RFX_API int rfx_get_seeds(rfx_ctx * ctx, uint32_t out[2]);            /* current LCG states (synchronises) */
/* advance the randDir stream as if n Scene::trace calls had run (frame sharding).  The stream's accept pattern is tabulated
 * over the LCG's whole 2^32-state cycle at rfx_create, so the cost does not depend on n: one small kernel. */
RFX_API int rfx_skip_samples(rfx_ctx * ctx, uint64_t n_trace_calls);
/* diagnostic: the library decides whether a draw-triple of Vector3::randomInsideSphere is accepted (Vector3.cpp:185) with an integer
 * test and falls back to the reference's float expression inside a guard band; this runs both on every triple of the LCG's whole
 * 2^32-state cycle.  out[0] = triples on which they disagree (0 = the decisions are the reference's, by exhaustion),
 * out[1] = triples inside the guard band.  About 20 ms. */
RFX_API int rfx_selftest_rng(rfx_ctx * ctx, uint64_t out[2]);
/* diagnostic: every path of a frame starts at the eye (Render.cpp:154-156), so the fast kernel lets a warp's first pass over the
 * objects skip those whose screen bounds miss its 4x8 pixel tile.  This returns the bounds the library derives for the current
 * scene (constant-bank scenes only), camera and image size: out[4*i .. 4*i+3] = x0, x1, y0, y1 (inclusive; x0 > x1 = no pixel) of
 * sphere i (i < 16) or triangle i - 16 (16 <= i < 24), objects in insertion order within their kind; counts = {spheres, triangles}.
 * A test evaluates Sphere::trace's / Triangle::trace's accept expressions on every pixel against them. */
RFX_API int rfx_selftest_primary_bounds(rfx_ctx * ctx, int32_t out[96], int32_t counts[2]);
/* The same bounds as a pure host function (no device, no context), for tests that run without a GPU: cam = eye[3], view[9] (row-major),
 * fov; spheres = n_spheres x (cx, cy, cz, r^2); tris = n_tris x (v0[3], axTrans[9] row-major: what Triangle::trace reads, Triangle.cpp:56-57). */
RFX_API int rfx_selftest_primary_bounds_host(const float cam[13], uint32_t width, uint32_t height, int n_spheres, const float * spheres,
                                             int n_tris, const float * tris, int32_t out[96]);
/* diagnostic, pure host function: the candidate grid the library builds for the shadow queries of one far light (option "light_grids").
 * light = origin[3], radius; spheres = n_spheres x (cx, cy, cz, r); box = lo[3], hi[3] of every point a shadow ray can start from;
 * reach_diagonal = diagonal of the box of ALL ray origins (sizes the rounding-noise margin of the exact sphere test).  Returns
 * uv = the two cell-coordinate rows (column = floor(uv[0..2] . p + uv[3]), row = floor(uv[4..6] . p + uv[7])), dims = {nx, ny}
 * ({0, 0}: the light is too close for a grid), counts = {nx*ny + 1, items}; cell_start / items (sphere indices, cell after cell) are
 * filled when their capacities suffice.  A test casts random jittered shadow rays and checks that every sphere the float32 test of
 * Sphere.cpp:49-57 reports is listed in the cell of the ray's origin. */
RFX_API int rfx_selftest_light_grid_host(const float light[4], int n_spheres, const float * spheres, const float box[6], float reach_diagonal,
                                         float uv[8], int32_t dims[2], uint32_t * cell_start, uint64_t cell_cap, int32_t * items, uint64_t item_cap,
                                         uint64_t counts[2]);
/* diagnostic, pure host function: the boxes of the triangle hierarchy (rfx_set_bvh_mode).  tris = n x (v0[3], axTrans[9] row-major: what
 * Triangle::trace reads); reach = lo[3], hi[3] of every ray origin.  boxes out = n x (lo[3], hi[3]): each holds every point at which the
 * float32 test of Triangle.cpp:56-68 can accept a ray from inside reach (a zero-area triangle's test accepts the unit triangle its
 * identity basis describes, not its vertices), inflated by that test's rounding noise and by 1e-6 of the reach diagonal. */
RFX_API int rfx_selftest_tri_bounds_host(int n, const float * tris, const float reach[6], float * boxes);
/* diagnostic, pure host function: the screen grid of a path's first query (option "eye_grid") for cam = eye[3], view[9], fov and
 * spheres = n_spheres x (cx, cy, cz, r^2): dims = {nx, ny, shift} (cells of 2^shift pixels; {0, 0, 0}: no grid for this camera),
 * counts = {nx*ny + 1, items}, cell_start / items (sphere indices, cell after cell) filled when their capacities suffice. */
RFX_API int rfx_selftest_eye_grid_host(const float cam[13], uint32_t width, uint32_t height, int n_spheres, const float * spheres, int32_t dims[3],
                                       uint32_t * cell_start, uint64_t cell_cap, int32_t * items, uint64_t item_cap, uint64_t counts[2]);

/* ---- Render (reference Render.h:30-41) ----------------------------------------------------------------- */
RFX_API int rfx_set_image_size(rfx_ctx * ctx, uint32_t width, uint32_t height);   /* Render::setImageSize, Render.cpp:57-80 */
RFX_API int rfx_render_begin(rfx_ctx * ctx, int reflect_num, int sample_num, int additive); /* Render::renderBegin, Render.cpp:116-134 */
RFX_API int rfx_render_next(rfx_ctx * ctx, uint32_t pixels);   /* Render::renderNext, Render.cpp:136-215: 1 = more to do, 0 = frame complete, <0 error */
RFX_API float rfx_progress(const rfx_ctx * ctx);               /* Render::getRenderProgress, Render.cpp:223-226 (percent) */
RFX_API int rfx_additive_counter(const rfx_ctx * ctx);         /* Render::additiveCounter */
RFX_API int rfx_in_progress(const rfx_ctx * ctx);              /* Render::inProgress */
RFX_API int rfx_read_argb(rfx_ctx * ctx, uint32_t * dst);      /* imagePixel(x,y).argb() for the whole image (Pulse.cpp:455-458 / Render::copyImage, Render.cpp:82-101) */
RFX_API int rfx_read_rgbf(rfx_ctx * ctx, float * dst);         /* imagePixel(x,y) for the whole image, 3 floats per pixel (Render.cpp:103-114) */
RFX_API int rfx_read_image(rfx_ctx * ctx, float * rgbf, uint32_t * argb, int divide); /* both outputs optional; divide = 0 packs the RAW image as Render::copyImage does (Render.cpp:82-101), 1 = imagePixel semantics */
RFX_API int rfx_read_pixel(rfx_ctx * ctx, int x, int y, float rgb[3]);            /* Render::imagePixel(x,y) */
RFX_API int rfx_read_signatures(rfx_ctx * ctx, uint32_t * dst); /* per-pixel hit-path signature of the last pass (parity localiser; enabled by rfx_enable_signatures) */
RFX_API int rfx_enable_signatures(rfx_ctx * ctx, int on);

/* ---- frame splitting (one frame shared by several GPUs, SURVEY §8e): render only pixels [p0, p1) of the frame latched by
 * rfx_render_begin.  Ranges must be issued in increasing order; the random streams are advanced over the pixels in between,
 * so every range consumes exactly the draws it would get in a full-frame render, and rfx_render_finish advances them to the
 * end of the frame.  argb_device (optional) is a FULL-FRAME ARGB buffer; it may live on another GPU (peer mapping over
 * NVLink, see rfx_ipc_*): the kernel then stores its pixels straight into the gathering GPU's framebuffer.  Any 4-byte aligned
 * frame is accepted (16-byte aligned frames of a width that is a multiple of 4 take the kernels with 128-bit stores). */
RFX_API int rfx_render_range(rfx_ctx * ctx, uint64_t p0, uint64_t p1, uint32_t * argb_device, void * stream);
RFX_API int rfx_render_finish(rfx_ctx * ctx);
/* the same for the usual partition — interleaved strips of strip_rows rows, strip s owned by rank s % world — in ONE random-stream
 * pass over the frame and ONE trace launch covering only this rank's rows; completes the frame (no rfx_render_finish needed) */
RFX_API int rfx_render_strips(rfx_ctx * ctx, uint32_t strip_rows, uint32_t world, uint32_t rank, uint32_t * argb_device, void * stream);
/* device buffers that can be shared between the per-GPU processes of one node (cudaIpc) */
RFX_API int rfx_buffer_alloc(rfx_ctx * ctx, uint64_t bytes, void ** device_ptr);
RFX_API int rfx_buffer_free(rfx_ctx * ctx, void * device_ptr);
RFX_API int rfx_buffer_read(rfx_ctx * ctx, const void * device_ptr, void * host_dst, uint64_t bytes);   /* synchronises */
RFX_API int rfx_ipc_export(rfx_ctx * ctx, void * device_ptr, unsigned char handle[64]);
RFX_API int rfx_ipc_import(rfx_ctx * ctx, const unsigned char handle[64], void ** device_ptr);       /* peer mapping of another process's buffer */
RFX_API int rfx_ipc_close(rfx_ctx * ctx, void * device_ptr);

/* ---- Scene::trace (reference Scene.h:39, Scene.cpp:73-236) for n arbitrary rays: ray i consumes the i-th next randDir of the
 * stream, exactly as n successive Scene::trace calls would.  origins/rays: 3n floats; rgb out: 3n floats.  Synchronous. */
RFX_API int rfx_trace_rays(rfx_ctx * ctx, int n, const float * origins, const float * rays, int reflect_num, float * rgb);

/* ---- headless batch path (the bench driver; models Pulse's screenshot flow, Pulse.cpp:174-208, for a camera
 * path).  cams = n_frames x 13 floats (eye[3], view[9], fov).  Each frame is setImageSize-sized, rendered with
 * renderBegin(reflect_num, sample_num, false) + renderNext to completion, and packed with imagePixel().argb().
 * The randDir stream continues from frame to frame. ------------------------------------------------------- */
/* output to HOST memory (n_frames * W * H uint32); device->host copies are overlapped with the next frame */
RFX_API int rfx_render_frames(rfx_ctx * ctx, int n_frames, const float * cams, int reflect_num, int sample_num, uint32_t * argb_host);
/* output to DEVICE memory the caller owns, on the caller's stream (cudaStream_t as void*; NULL = context stream);
 * asynchronous: returns after enqueueing */
RFX_API int rfx_render_frames_device(rfx_ctx * ctx, int n_frames, const float * cams, int reflect_num, int sample_num,
                                     uint32_t * argb_device, void * stream);
RFX_API int rfx_synchronize(rfx_ctx * ctx);

/* ---- bookkeeping --------------------------------------------------------------------------------------- */
RFX_API int rfx_get_stats(rfx_ctx * ctx, rfx_stats * out);     /* synchronises */
RFX_API int rfx_stats_reset(rfx_ctx * ctx);
RFX_API int rfx_enable_profiling(rfx_ctx * ctx, int on);
/* tuning / test hook; results never depend on an option.  "max_calls_per_launch": Scene::trace calls one random-stream pass and
 * one trace launch may cover (default 2^25 = 128 MB of ranked states; large SSAA factors and 8K frames are rendered in chunks of
 * this many calls — tests lower it to drive the chunk loop at small sizes).  "copy_streams": device->host streams
 * rfx_render_frames alternates between (1 or 2, default 1).  "blob_wavefront": scenes that do not fit the constant bank render
 * their one-sample ARGB frames of reflection depth >= 4 with a two-kernel wavefront — the first k segments of every path in pixel
 * tiles, the rest from a path queue (k = the value, default 2; 0 = the single tile kernel).  "blob_smem_bvh": the queue-driven
 * kernel keeps a small sphere hierarchy in shared memory (default 1).  "tile_order_period": the cost-ordered tile scheduling of the
 * constant-bank fast kernel records the tiles' cost classes on every k-th launch over the same grid and replays the last recording
 * in between (default 8).  "light_grids": scenes with a sphere hierarchy answer the shadow queries of far lights from a 2-D grid of
 * candidate spheres across the light's direction instead of walking the hierarchy (default 1).  "eye_grid": the same scenes take the
 * candidates of a path's first query (origin = eye) from a screen grid binned per camera out of the spheres' primary-ray bounds
 * (default 1).  Both grids list spheres only: triangles are tested after them, through their own hierarchy when the scene has one
 * (rfx_set_bvh_mode).  Frames are bit-identical under every setting. */
RFX_API int rfx_set_option(rfx_ctx * ctx, const char * name, int64_t value);
/* kernel selection: 0 = automatic (constant-bank kernels when the scene fits, the blob kernels otherwise),
 * 1 = constant-bank kernel if it fits, 2 = always the blob kernels (tile / wavefront kernels for row-aligned slices, the general
 * one otherwise), 3 = always the general blob kernel.  Results are identical; tests use it. */
RFX_API int rfx_force_path(rfx_ctx * ctx, int path);
/* acceleration structures of the blob kernels: 0 = automatic (a bounding-volume hierarchy over the spheres when there are more than
 * 32 and the scene holds no unbounded plane; one over the triangles, walked after the spheres, when there are more than 32 triangles
 * and no plane), 1 = always (whenever there are any spheres / triangles and no plane), 2 = never (the
 * reference's brute-force list walk).  Results are identical; tests compare them. */
RFX_API int rfx_set_bvh_mode(rfx_ctx * ctx, int mode);
/* cost-ordered tile scheduling of the constant-bank fast kernel: launches record which tiles held long paths (every
 * "tile_order_period"-th launch over a grid) and the following launches over the same grid start those first (1 = on, the
 * default; 0 = off: middle rows of the slice first, outwards).  Results are identical. */
RFX_API int rfx_set_tile_ordering(rfx_ctx * ctx, int on);

#ifdef __cplusplus
}
#endif
#endif /* REFLAX_C_H */
