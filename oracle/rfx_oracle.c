/* TEST INFRASTRUCTURE — NOT PRODUCT CODE.
 *
 * rfx_oracle.c — plain-C CPU restatement of ReflaxMan's per-pixel trace-and-shade path, used ONLY as the parity
 * checker (tests/, __graft_entry__.smoke(), bench.py's cpu_baseline leg).  The product (reflaxman_b200/csrc) never
 * links, imports or calls this file; it has no CPU fallback.
 *
 * Parity status: PINNED.  tests/test_oracle_vs_reference.py checks this restatement bit-for-bit (float image and
 * ARGB) against the unmodified reference compiled from /root/reference by oracle/Makefile (oracle/_ref/ref_render),
 * and against golden vectors generated from that binary (tests/golden/, made by tests/golden/make_golden.py).
 *
 * Every float operation goes through ADD/SUB/MUL/DIV/SQRT so that (a) the evaluation order of the reference's
 * overloaded C++ operators is spelled out, and (b) a -DRFXO_CENSUS build can count algorithmic flops exactly the
 * way SURVEY.md §8(d) defines them (add/sub/mul/div/sqrt = 1; powf, floor, compares, conversions = 0).
 * Build with: gcc -O2 -ffp-contract=off (see oracle/Makefile).  Never -ffast-math.
 *
 * Reference map (path:line relative to /root/reference/src/common):
 *   rng_next / rand_in_sphere        trace_math.h:34-39, Vector3.cpp:176-188
 *   v_* helpers                      Vector3.cpp:36-64,104-151; trace_math.cpp:3-23 (normalize, reflect)
 *   sphere_trace                     Sphere.cpp:44-85
 *   tri_setup / tri_trace            Triangle.cpp:11-21,110-120 / Triangle.cpp:53-108; Matrix33.cpp:10-15,49-79,230-235
 *   plane_trace                      Plane.cpp:36-73
 *   tex_fetch / tex_sample           Texture.cpp:216-229 / 231-269; Color.cpp:9-14
 *   sky_sample                       Skybox.cpp:21-37 (half tile), 39-106
 *   scene_trace                      Scene.cpp:73-236
 *   rfxo_render_pass                 Render.cpp:116-134 (renderBegin), 136-215 (renderNext)
 *   rfxo_resolve                     Render.cpp:103-114 (imagePixel), Color.cpp:114-117 (argb)
 *   rfxo_camera_lookat               Camera.cpp:24-36
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <float.h>
#include <pthread.h>

/* ------------------------------------------------------------------------------------------------ op layer */
#ifdef RFXO_CENSUS
static __thread uint64_t g_ops[5]; /* add(sub), mul, div, sqrt, powf */
#define CNT(i) (g_ops[i]++)
#else
#define CNT(i) ((void)0)
#endif
static inline float ADD(float a, float b) { CNT(0); return a + b; }
static inline float SUB(float a, float b) { CNT(0); return a - b; }
static inline float MUL(float a, float b) { CNT(1); return a * b; }
static inline float DIV(float a, float b) { CNT(2); return a / b; }
static inline float SQRT(float a) { CNT(3); return sqrtf(a); }
static inline float POWF(float a, float b) { CNT(4); return powf(a, b); }
#ifdef RFXO_POW_CR
/* -DRFXO_POW_CR: each power site computes what the GPU computes there (rfx_device.cuh): the specular power as the correctly
 * rounded x^y, the Fresnel cube as the binary64 cube rounded once.  Per site, not by exponent: the specular exponent can be 3. */
static inline float POW_SPEC(float a, float b) { CNT(4); return (float)pow((double)a, (double)b); }
static inline float POW_CUBE(float a) { CNT(4); const double d = (double)a; return (float)((d * d) * d); }
#else
static inline float POW_SPEC(float a, float b) { return POWF(a, b); }
static inline float POW_CUBE(float a) { return POWF(a, 3.0f); }
#endif

#define VSN 1.08420217248550443e-19f /* sqrtf(FLT_MIN) = 2^-63 exactly, trace_math.h:17 */
#define DELTA 0.0001f                /* trace_math.h:18 */

typedef struct { float x, y, z; } V3;
typedef struct { float r, g, b; } C3;
typedef struct { float m[9]; } M33; /* row-major _11.._33, Matrix33.h:16-20 */

static inline float clampf(float v, float lo, float hi) { return v < lo ? lo : v > hi ? hi : v; } /* trace_math.h:24 */

static inline V3 v3(float x, float y, float z) { V3 v = { x, y, z }; return v; }
static inline V3 v_add(V3 a, V3 b) { return v3(ADD(a.x, b.x), ADD(a.y, b.y), ADD(a.z, b.z)); }
static inline V3 v_sub(V3 a, V3 b) { return v3(SUB(a.x, b.x), SUB(a.y, b.y), SUB(a.z, b.z)); }
static inline V3 v_scale(V3 a, float f) { return v3(MUL(a.x, f), MUL(a.y, f), MUL(a.z, f)); }
static inline V3 v_neg(V3 a) { return v3(-a.x, -a.y, -a.z); }
static inline float v_dot(V3 a, V3 b) { return ADD(ADD(MUL(a.x, b.x), MUL(a.y, b.y)), MUL(a.z, b.z)); } /* Vector3.cpp:124-127 */
static inline float v_sqlen(V3 a) { return ADD(ADD(MUL(a.x, a.x), MUL(a.y, a.y)), MUL(a.z, a.z)); }     /* Vector3.cpp:41-44 */
static inline float v_len(V3 a) { return SQRT(v_sqlen(a)); }                                            /* Vector3.cpp:36-39 */
static inline V3 v_cross(V3 a, V3 b)                                                                    /* Vector3.cpp:136-141 */
{
  return v3(SUB(MUL(a.y, b.z), MUL(a.z, b.y)), SUB(MUL(a.z, b.x), MUL(a.x, b.z)), SUB(MUL(a.x, b.y), MUL(a.y, b.x)));
}
static inline V3 v_div(V3 a, float f) /* Vector3.cpp:143-151: three true divides, guarded */
{
  if (fabsf(f) > VSN) return v3(DIV(a.x, f), DIV(a.y, f), DIV(a.z, f));
  return a;
}
static inline V3 v_normalized(V3 a) /* Vector3.cpp:55-64 and trace_math.cpp:3-12 (same arithmetic) */
{
  const float l = v_len(a);
  if (l > VSN) return v_div(a, l);
  return a;
}
static inline V3 v_reflect(V3 v, V3 n) /* trace_math.cpp:14-23 */
{
  const float dn = v_dot(n, n);
  if (dn > VSN)
  {
    const float s = DIV(v_dot(v, n), dn);
    const V3 n2 = v_scale(n, 2.0f);
    return v_sub(v, v_scale(n2, s));
  }
  return v;
}
static inline V3 m_mulv(const M33 * m, V3 v) /* Matrix33.cpp:230-235 */
{
  const float * a = m->m;
  return v3(ADD(ADD(MUL(v.x, a[0]), MUL(v.y, a[1])), MUL(v.z, a[2])),
            ADD(ADD(MUL(v.x, a[3]), MUL(v.y, a[4])), MUL(v.z, a[5])),
            ADD(ADD(MUL(v.x, a[6]), MUL(v.y, a[7])), MUL(v.z, a[8])));
}
static M33 m_cols(V3 u, V3 v, V3 n) /* Matrix33.cpp:10-15: columns u, v, n */
{
  M33 r = { { u.x, v.x, n.x, u.y, v.y, n.y, u.z, v.z, n.z } };
  return r;
}
static M33 m_inverted(const M33 * s) /* Matrix33.cpp:49-79 */
{
  const float _11 = s->m[0], _12 = s->m[1], _13 = s->m[2], _21 = s->m[3], _22 = s->m[4], _23 = s->m[5], _31 = s->m[6], _32 = s->m[7], _33 = s->m[8];
  const float d = ADD(ADD(MUL(_11, SUB(MUL(_22, _33), MUL(_32, _23))), MUL(_21, SUB(MUL(_32, _13), MUL(_12, _33)))), MUL(_31, SUB(MUL(_12, _23), MUL(_13, _22))));
  M33 r;
  if (fabsf(d) > VSN)
  {
    r.m[0] = DIV(SUB(MUL(_22, _33), MUL(_23, _32)), d);
    r.m[1] = DIV(SUB(MUL(_13, _32), MUL(_12, _33)), d);
    r.m[2] = DIV(SUB(MUL(_12, _23), MUL(_13, _22)), d);
    r.m[3] = DIV(SUB(MUL(_23, _31), MUL(_21, _33)), d);
    r.m[4] = DIV(SUB(MUL(_11, _33), MUL(_13, _31)), d);
    r.m[5] = DIV(SUB(MUL(_13, _21), MUL(_11, _23)), d);
    r.m[6] = DIV(SUB(MUL(_21, _32), MUL(_22, _31)), d);
    r.m[7] = DIV(SUB(MUL(_12, _31), MUL(_11, _32)), d);
    r.m[8] = DIV(SUB(MUL(_11, _22), MUL(_12, _21)), d);
  }
  else
  {
    const M33 id = { { 1, 0, 0, 0, 1, 0, 0, 0, 1 } };
    r = id;
  }
  return r;
}

static inline C3 c3(float r, float g, float b) { C3 c = { r, g, b }; return c; }
static inline C3 c_add(C3 a, C3 b) { return c3(ADD(a.r, b.r), ADD(a.g, b.g), ADD(a.b, b.b)); }
static inline C3 c_mul(C3 a, C3 b) { return c3(MUL(a.r, b.r), MUL(a.g, b.g), MUL(a.b, b.b)); }
static inline C3 c_scale(C3 a, float f) { return c3(MUL(a.r, f), MUL(a.g, f), MUL(a.b, f)); }
static inline C3 c_clamp(C3 a) { return c3(clampf(a.r, 0.0f, 1.0f), clampf(a.g, 0.0f, 1.0f), clampf(a.b, 0.0f, 1.0f)); }
static inline C3 c_div(C3 a, float f) /* Color.cpp:50-61, 99-107 */
{
  if (fabsf(f) > VSN) return c3(DIV(a.r, f), DIV(a.g, f), DIV(a.b, f));
  return a;
}

/* ------------------------------------------------------------------------------------------------ RNG */
static inline int rng_next(uint32_t * s) /* trace_math.h:36-39 (signed overflow wraps in practice) */
{
  *s = 214013u * *s + 2531011u;
  return (int)((*s >> 16) & 0x7FFF);
}
static V3 rand_in_sphere(uint32_t * s) /* Vector3.cpp:176-188 with radius 1.0f (v * 1.0f is exact) */
{
  V3 v;
  const float half = 16383.5f; /* float(FAST_RAND_MAX) / 2, a compile-time constant */
  do
  {
    v.x = SUB(DIV((float)rng_next(s), half), 1.f);
    v.y = SUB(DIV((float)rng_next(s), half), 1.f);
    v.z = SUB(DIV((float)rng_next(s), half), 1.f);
  } while (v_sqlen(v) > 1.f);
  return v_scale(v, 1.0f);
}

/* ------------------------------------------------------------------------------------------------ scene */
enum { MT_METAL = 0, MT_DIELECTRIC = 1 };           /* Material.h:8 */
enum { OBJ_SPHERE = 0, OBJ_TRIANGLE = 1, OBJ_PLANE = 2 };

typedef struct { int type; C3 color; float reflectivity, transparency; } Mat;
typedef struct { uint32_t w, h; uint32_t * px; } Tex; /* px == NULL: empty texture -> checker fallback */
typedef struct
{
  int kind;
  Mat mat;
  V3 center; float radius, sqRadius;                 /* sphere */
  V3 v0, norm; M33 axTrans, tuvTrans; float tu0, tv0; int tex; /* triangle (tex < 0: untextured) */
  V3 pos;                                            /* plane (uses norm) */
} Obj;
typedef struct { V3 origin; float radius; C3 color; float power; } Light;

typedef struct rfxo_scene
{
  C3 diffLightColor, envColor; float diffLightPower;
  Obj * objs; int nobjs, capobjs;
  Light * lights; int nlights, caplights;
  Tex * tex; int ntex, captex;
  int skyTex; float halfTileW, halfTileH;
} rfxo_scene;

typedef struct
{
  uint64_t rays;         /* bounce-loop iterations + shadow rays cast (SURVEY §8d "ray") */
  uint64_t bounces, shadow_rays, hits, lit, sky, spec_pow, fresnel_pow;
  uint64_t sphere_tests, tri_tests, plane_tests, tex_lookups, samples;
  uint64_t ops[5];       /* census build only: add/sub, mul, div, sqrt, powf */
} rfxo_counters;

static Mat mk_mat(int type, const float rgb[3], float refl, float transp) /* Material.cpp:8-14 */
{
  Mat m;
  m.type = type ? MT_DIELECTRIC : MT_METAL;
  m.color = c3(rgb[0], rgb[1], rgb[2]);
  m.reflectivity = clampf(refl, 0.0f, 1.0f);
  m.transparency = clampf(transp, 0.0f, 1.0f);
  return m;
}

rfxo_scene * rfxo_scene_new(const float ambient_rgb[3], float ambient_power) /* Scene.cpp:10-15 */
{
  rfxo_scene * s = (rfxo_scene *)calloc(1, sizeof(rfxo_scene));
  s->diffLightColor = c3(ambient_rgb[0], ambient_rgb[1], ambient_rgb[2]);
  s->envColor = c_scale(s->diffLightColor, ambient_power);
  s->diffLightPower = ambient_power;
  s->skyTex = -1;
  s->halfTileW = SUB(DIV(1.0f, 8.0f), FLT_EPSILON); /* Skybox.cpp:6-7 */
  s->halfTileH = SUB(DIV(1.0f, 6.0f), FLT_EPSILON);
  return s;
}

void rfxo_scene_free(rfxo_scene * s)
{
  if (!s) return;
  for (int i = 0; i < s->ntex; i++) free(s->tex[i].px);
  free(s->tex); free(s->objs); free(s->lights); free(s);
}

static Obj * new_obj(rfxo_scene * s)
{
  if (s->nobjs == s->capobjs)
  {
    s->capobjs = s->capobjs ? s->capobjs * 2 : 16;
    s->objs = (Obj *)realloc(s->objs, sizeof(Obj) * (size_t)s->capobjs);
  }
  Obj * o = &s->objs[s->nobjs++];
  memset(o, 0, sizeof(*o));
  o->tex = -1;
  return o;
}

int rfxo_add_light(rfxo_scene * s, const float o[3], float radius, const float rgb[3], float power) /* Scene.cpp:47-58, OmniLight.cpp:8-14 */
{
  if (radius <= VSN) radius = VSN;
  if (s->nlights == s->caplights)
  {
    s->caplights = s->caplights ? s->caplights * 2 : 4;
    s->lights = (Light *)realloc(s->lights, sizeof(Light) * (size_t)s->caplights);
  }
  const C3 col = c3(rgb[0], rgb[1], rgb[2]);
  s->envColor = c_add(s->envColor, c_scale(col, power)); /* un-clamped power, as the reference */
  Light * l = &s->lights[s->nlights++];
  l->origin = v3(o[0], o[1], o[2]);
  l->radius = radius;
  l->color = col;
  l->power = clampf(power, 0.0f, 1.0f);
  return s->nlights - 1;
}

int rfxo_add_sphere(rfxo_scene * s, const float c[3], float radius, int type, const float rgb[3], float refl, float transp) /* Scene.cpp:29-39, Sphere.cpp:9-20 */
{
  if (radius <= VSN) radius = VSN;
  Obj * o = new_obj(s);
  o->kind = OBJ_SPHERE;
  o->mat = mk_mat(type, rgb, refl, transp);
  o->center = v3(c[0], c[1], c[2]);
  o->radius = radius;
  o->sqRadius = MUL(radius, radius);
  return s->nobjs - 1;
}

int rfxo_add_texture(rfxo_scene * s, uint32_t w, uint32_t h, const uint32_t * argb) /* Scene.cpp:60-65; NULL/0x0 = failed load */
{
  if (s->ntex == s->captex)
  {
    s->captex = s->captex ? s->captex * 2 : 4;
    s->tex = (Tex *)realloc(s->tex, sizeof(Tex) * (size_t)s->captex);
  }
  Tex * t = &s->tex[s->ntex++];
  if (argb && w && h)
  {
    t->w = w; t->h = h;
    t->px = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)w * h);
    memcpy(t->px, argb, sizeof(uint32_t) * (size_t)w * h);
  }
  else { t->w = 0; t->h = 0; t->px = NULL; }
  return s->ntex - 1;
}

int rfxo_set_skybox(rfxo_scene * s, int tex) /* Skybox.cpp:21-37 */
{
  if (tex >= 0 && tex < s->ntex && s->tex[tex].px)
  {
    s->skyTex = tex;
    s->halfTileW = SUB(SUB(DIV(1.0f, 8.0f), DIV(1.0f, (float)s->tex[tex].w)), FLT_EPSILON);
    s->halfTileH = SUB(SUB(DIV(1.0f, 6.0f), DIV(1.0f, (float)s->tex[tex].h)), FLT_EPSILON);
    return 1;
  }
  s->skyTex = -1;
  s->halfTileW = SUB(DIV(1.0f, 8.0f), FLT_EPSILON);
  s->halfTileH = SUB(DIV(1.0f, 6.0f), FLT_EPSILON);
  return 0;
}

/* v = 9 floats (v0,v1,v2); tex < 0 = untextured; uv = u1,v1,u2,v2,u3,v3 (Triangle.cpp:11-21, 110-120) */
int rfxo_add_triangle(rfxo_scene * s, const float v[9], int type, const float rgb[3], float refl, float transp, int tex, const float uv[6])
{
  Obj * o = new_obj(s);
  const V3 v0 = v3(v[0], v[1], v[2]), v1 = v3(v[3], v[4], v[5]), v2 = v3(v[6], v[7], v[8]);
  o->kind = OBJ_TRIANGLE;
  o->mat = mk_mat(type, rgb, refl, transp);
  o->v0 = v0;
  o->norm = v_normalized(v_cross(v_sub(v1, v0), v_sub(v2, v0)));
  const M33 basis = m_cols(v_sub(v2, v0), v_sub(v1, v0), v_neg(o->norm));
  o->axTrans = m_inverted(&basis);
  if (tex >= 0 && uv)
  {
    const V3 t1 = v3(uv[0], uv[1], 0), t2 = v3(uv[2], uv[3], 0), t3 = v3(uv[4], uv[5], 0);
    o->tex = tex;
    o->tu0 = uv[0]; o->tv0 = uv[1];
    o->tuvTrans = m_cols(v_sub(t3, t1), v_sub(t2, t1), v3(0, 0, -1));
  }
  return s->nobjs - 1;
}

int rfxo_add_plane(rfxo_scene * s, const float pos[3], const float norm[3], int type, const float rgb[3], float refl, float transp) /* Plane.cpp:9-14 */
{
  Obj * o = new_obj(s);
  o->kind = OBJ_PLANE;
  o->mat = mk_mat(type, rgb, refl, transp);
  o->pos = v3(pos[0], pos[1], pos[2]);
  o->norm = v3(norm[0], norm[1], norm[2]);
  return s->nobjs - 1;
}

/* read back what setup derived, so tests can compare the product's host-side flattening bit for bit */
void rfxo_get_triangle(const rfxo_scene * s, int idx, float norm[3], float axTrans[9], float tuvTrans[9])
{
  const Obj * o = &s->objs[idx];
  norm[0] = o->norm.x; norm[1] = o->norm.y; norm[2] = o->norm.z;
  memcpy(axTrans, o->axTrans.m, sizeof(float) * 9);
  memcpy(tuvTrans, o->tuvTrans.m, sizeof(float) * 9);
}
void rfxo_get_env(const rfxo_scene * s, float env[3], float halfTile[2])
{
  env[0] = s->envColor.r; env[1] = s->envColor.g; env[2] = s->envColor.b;
  halfTile[0] = s->halfTileW; halfTile[1] = s->halfTileH;
}

/* ------------------------------------------------------------------------------------------------ textures */
static C3 tex_fetch(const Tex * t, uint32_t x, uint32_t y) /* Texture.cpp:216-229 (non-empty case) + Color.cpp:9-14 */
{
  if (x >= t->w || y >= t->h) return c3(0, 0, 0);
  const uint32_t c = t->px[x + t->w * y];
  return c3(DIV((float)((c >> 16) & 0xFF), 255.0f), DIV((float)((c >> 8) & 0xFF), 255.0f), DIV((float)(c & 0xFF), 255.0f));
}

static C3 tex_sample(const Tex * t, float u, float v, rfxo_counters * k) /* Texture.cpp:231-269; t == NULL or empty -> checker */
{
  k->tex_lookups++;
  if (u < 0.0f || u > 1.0f || v < 0.0f || v > 1.0f) return c3(0.0f, 0.0f, 0.0f);
  if (!t || !t->px)
    return (((int)MUL(u, 50) % 2) ^ ((int)MUL(v, 50) % 2)) ? c3(0.5f, 0.5f, 0.5f) : c3(0.75f, 0.75f, 0.75f);

  const float fx = MUL(clampf(u, 0.0f, SUB(1.0f, FLT_EPSILON)), (float)t->w);
  const float fy = MUL(clampf(v, 0.0f, SUB(1.0f, FLT_EPSILON)), (float)t->h);
  const uint32_t x = (uint32_t)fx, y = (uint32_t)fy;
  if (x < t->w - 1 && y < t->h - 1)
  {
    const C3 c00 = tex_fetch(t, x, y), c01 = tex_fetch(t, x, y + 1), c10 = tex_fetch(t, x + 1, y), c11 = tex_fetch(t, x + 1, y + 1);
    const float uf = SUB(fx, floorf(fx)), vf = SUB(fy, floorf(fy));
    const float uo = SUB(1, uf), vo = SUB(1, vf);
    return c_add(c_scale(c_add(c_scale(c00, uo), c_scale(c10, uf)), vo), c_scale(c_add(c_scale(c01, uo), c_scale(c11, uf)), vf));
  }
  return tex_fetch(t, x, y);
}

static C3 sky_sample(const rfxo_scene * s, V3 ray, rfxo_counters * k) /* Skybox.cpp:39-106 */
{
  const float uLeft = DIV(1.0f, 8.0f), vLeft = DIV(3.0f, 6.0f), uFront = DIV(3.0f, 8.0f), vFront = DIV(3.0f, 6.0f);
  const float uRight = DIV(5.0f, 8.0f), vRight = DIV(3.0f, 6.0f), uBack = DIV(7.0f, 8.0f), vBack = DIV(3.0f, 6.0f);
  const float uTop = DIV(3.0f, 8.0f), vTop = DIV(5.0f, 6.0f), uBottom = DIV(3.0f, 8.0f), vBottom = DIV(1.0f, 6.0f);
#ifdef RFXO_CENSUS
  g_ops[2] -= 12; /* compile-time constants in the reference */
#endif
  const V3 n = v_normalized(ray);
  const float x = n.x, y = n.y, z = n.z;
  const float ax = ADD(fabsf(x), VSN), ay = ADD(fabsf(y), VSN), az = ADD(fabsf(z), VSN);
  const float hw = s->halfTileW, hh = s->halfTileH;
  float u, v;
  if (az >= ax && az >= ay)
  {
    if (z > 0) { u = ADD(uFront, MUL(DIV(x, az), hw)); v = ADD(vFront, MUL(DIV(y, az), hh)); }
    else       { u = SUB(uBack, MUL(DIV(x, az), hw));  v = ADD(vBack, MUL(DIV(y, az), hh)); }
  }
  else if (ax >= ay && ax >= az)
  {
    if (x > 0) { u = SUB(uRight, MUL(DIV(z, ax), hw)); v = ADD(vRight, MUL(DIV(y, ax), hh)); }
    else       { u = ADD(uLeft, MUL(DIV(z, ax), hw));  v = ADD(vLeft, MUL(DIV(y, ax), hh)); }
  }
  else
  {
    if (y > 0) { u = ADD(uTop, MUL(DIV(x, ay), hw));    v = SUB(vTop, MUL(DIV(z, ay), hh)); }
    else       { u = ADD(uBottom, MUL(DIV(x, ay), hw)); v = ADD(vBottom, MUL(DIV(z, ay), hh)); }
  }
  return tex_sample(s->skyTex >= 0 ? &s->tex[s->skyTex] : NULL, u, v, k);
}

/* ------------------------------------------------------------------------------------------------ intersectors */
typedef struct { V3 drop, norm, reflect; float dist; Mat mat; } Hit;

static int sphere_trace(const rfxo_scene * s, const Obj * o, V3 origin, V3 ray, Hit * out, rfxo_counters * k) /* Sphere.cpp:44-85 */
{
  (void)s;
  k->sphere_tests++;
  const V3 vco = v_sub(origin, o->center);
  const float a = v_sqlen(ray);
  const float b = v_dot(v_scale(ray, 2.0f), vco);
  const float c = SUB(v_sqlen(vco), o->sqRadius);
  const float d = SUB(MUL(b, b), MUL(MUL(4.0f, a), c));
  if (d >= 0.0f && a > VSN)
  {
    const float t = DIV(SUB(-b, SQRT(d)), MUL(2.0f, a));
    if (t > VSN)
    {
      const V3 fullRay = v_scale(ray, t);
      const float distance = v_len(fullRay);
      if (distance > DELTA)
      {
        const V3 drop = v_add(origin, fullRay);
        const V3 norm = v_sub(drop, o->center);
        if (out)
        {
          out->dist = distance;
          out->drop = drop;
          out->norm = norm;
          out->reflect = v_reflect(fullRay, norm);
          out->mat = o->mat;
        }
        return 1;
      }
    }
  }
  return 0;
}

static int tri_trace(const rfxo_scene * s, const Obj * o, V3 origin, V3 ray, Hit * out, rfxo_counters * k) /* Triangle.cpp:53-108 */
{
  k->tri_tests++;
  const V3 axO = m_mulv(&o->axTrans, v_sub(origin, o->v0));
  const V3 axR = m_mulv(&o->axTrans, ray);
  if (fabsf(axR.z) > VSN)
  {
    const float t = DIV(-axO.z, axR.z);
    if (t > VSN)
    {
      const float u = ADD(axO.x, MUL(t, axR.x));
      const float v = ADD(axO.y, MUL(t, axR.y));
      if (u >= 0.0f && v >= 0.0f && ADD(u, v) < 1.0f)
      {
        const V3 fullRay = v_scale(ray, t);
        const float sqd = v_sqlen(fullRay);
        if (sqd > MUL(DELTA, DELTA))
        {
#ifdef RFXO_CENSUS
          g_ops[1]--; /* DELTA*DELTA is a compile-time constant in the reference */
#endif
          if (out)
          {
            out->drop = v_add(origin, fullRay);
            out->norm = o->norm;
            out->reflect = v_reflect(fullRay, o->norm);
            out->dist = SQRT(sqd);
            out->mat = o->mat;
            if (o->tex >= 0)
            {
              const V3 tv = m_mulv(&o->tuvTrans, v3(u, v, 0));
              out->mat.color = tex_sample(&s->tex[o->tex], ADD(o->tu0, tv.x), ADD(o->tv0, tv.y), k);
            }
          }
          return 1;
        }
      }
    }
  }
  return 0;
}

static int plane_trace(const rfxo_scene * s, const Obj * o, V3 origin, V3 ray, Hit * out, rfxo_counters * k) /* Plane.cpp:36-73 */
{
  (void)s;
  k->plane_tests++;
  const V3 vop = v_sub(o->pos, origin);
  const float a = v_dot(o->norm, ray);
  if (fabsf(a) > VSN)
  {
    const float t = DIV(v_dot(o->norm, vop), a);
    if (t > VSN)
    {
      const V3 fullRay = v_scale(ray, t);
      const float sqd = v_sqlen(fullRay);
      if (sqd > MUL(DELTA, DELTA))
      {
#ifdef RFXO_CENSUS
        g_ops[1]--;
#endif
        if (out)
        {
          out->drop = v_add(origin, fullRay);
          out->norm = o->norm;
          out->reflect = v_reflect(fullRay, o->norm);
          out->dist = SQRT(sqd);
          out->mat = o->mat;
        }
        return 1;
      }
    }
  }
  return 0;
}

static inline int obj_trace(const rfxo_scene * s, const Obj * o, V3 origin, V3 ray, Hit * out, rfxo_counters * k)
{
  switch (o->kind)
  {
  case OBJ_SPHERE: return sphere_trace(s, o, origin, ray, out, k);
  case OBJ_TRIANGLE: return tri_trace(s, o, origin, ray, out, k);
  default: return plane_trace(s, o, origin, ray, out, k);
  }
}

/* ------------------------------------------------------------------------------------------------ Scene::trace */
#define SIG_STEP(h, ev) ((h) = ((h) ^ (uint32_t)(ev)) * 16777619u)

/* sig: running hit-path signature (object index / miss, facing and shadow flags per bounce) — parity localiser */
static C3 scene_trace(const rfxo_scene * s, V3 origin, V3 ray, int reflNumber, V3 randDir, rfxo_counters * k, uint32_t * sig)
{
  C3 mulColor = c3(1.0f, 1.0f, 1.0f);
  C3 pixelColor = c3(0.0f, 0.0f, 0.0f);
  k->samples++;

  for (int refl = 0; refl < reflNumber; ++refl)
  {
    float minDistance = FLT_MAX;
    int hitObject = -1;
    Hit hit;
    memset(&hit, 0, sizeof(hit));
    k->bounces++; k->rays++;

    for (int i = 0; i < s->nobjs; i++)
    {
      Hit cur;
      if (obj_trace(s, &s->objs[i], origin, ray, &cur, k) && cur.dist < minDistance)
      {
        minDistance = cur.dist;
        hit = cur;
        hitObject = i;
      }
    }

    if (hitObject >= 0)
    {
      k->hits++;
      SIG_STEP(*sig, hitObject + 1);
      const float rayLen = v_len(ray);
      const float normLen = v_len(hit.norm);
      const float reflectLen = v_len(hit.reflect);
      C3 sumLightColor = c3(0.0f, 0.0f, 0.0f);
      C3 sumSpecColor = c3(0.0f, 0.0f, 0.0f);

      for (int li = 0; li < s->nlights; li++)
      {
        const Light * light = &s->lights[li];
        const V3 dropToLight = v_sub(light->origin, hit.drop);
        if (v_dot(dropToLight, hit.norm) > VSN)
        {
          const float lightRadius = light->radius;
          const V3 shadowRay = v_add(dropToLight, v_scale(randDir, lightRadius));
          int inShadow = 0;
          k->shadow_rays++; k->rays++;
          for (int i = 0; i < s->nobjs; i++)
            if (i != hitObject && obj_trace(s, &s->objs[i], hit.drop, shadowRay, NULL, k))
            {
              inShadow = 1;
              break;
            }
          SIG_STEP(*sig, 0x100 + 2 * li + inShadow);

          if (!inShadow)
          {
            k->lit++;
            const float dropToLightLen = v_len(dropToLight);
            const C3 lightColor = light->color;
            const float lightPower = light->power;
            float a = MUL(dropToLightLen, normLen);
            const float lightDropCos = (a > VSN) ? DIV(v_dot(dropToLight, hit.norm), a) : 0.0f;

            if (lightPower > VSN)
              sumLightColor = c_add(sumLightColor, c_scale(c_scale(lightColor, lightDropCos), lightPower));

            a = v_sqlen(dropToLight);
            const float larsc = (a > VSN) ? SUB(1.0f, DIV(MUL(lightRadius, lightRadius), a)) : 0.0f;

            if (larsc > 0)
            {
              const V3 dtlRand = v_add(v_normalized(dropToLight), v_scale(randDir, SUB(1.0f, hit.mat.reflectivity)));
              a = MUL(v_len(dtlRand), reflectLen);
              float rsc = (a > VSN) ? DIV(v_dot(dtlRand, hit.reflect), a) : 0.0f;
              rsc = clampf(ADD(rsc, SUB(1.0f, SQRT(larsc))), 0.0f, 1.0f);

              if (rsc > VSN)
              {
                float specPower = rsc;
                if (lightRadius > VSN)
                {
                  k->spec_pow++;
                  specPower = MUL(POW_SPEC(specPower, ADD(1, DIV(MUL(MUL(3, hit.mat.reflectivity), dropToLightLen), lightRadius))), hit.mat.reflectivity);
                  sumSpecColor = c_add(sumSpecColor, c_scale(lightColor, specPower));
                }
              }
            }
          }
        }
      }

      const float reflectivity = hit.mat.reflectivity;
      const C3 color = hit.mat.color;
      sumLightColor = c_add(c_scale(s->diffLightColor, s->diffLightPower), sumLightColor);

      C3 finColor;
      if (hit.mat.type == MT_DIELECTRIC)
      {
        const float a = MUL(rayLen, normLen);
        const float dropAngleCos = (a > VSN) ? clampf(DIV(v_dot(ray, v_neg(hit.norm)), a), 0.0f, 1.0f) : 0.0f;
        k->fresnel_pow++;
        const float rf = ADD(0.2f, MUL(0.8f, POW_CUBE(SUB(1.0f, dropAngleCos))));
        finColor = c_add(c_mul(c_scale(color, SUB(1.0f, rf)), sumLightColor), sumSpecColor);
        finColor = c_mul(finColor, mulColor);
        mulColor = c_scale(mulColor, rf);
      }
      else
      {
        const float rf = 0.8f;
        finColor = c_add(c_mul(c_scale(color, SUB(1.0f, rf)), sumLightColor), sumSpecColor);
        finColor = c_mul(finColor, mulColor);
        mulColor = c_mul(mulColor, c_scale(color, rf));
      }

      pixelColor = c_clamp(c_add(pixelColor, finColor));

      if (mulColor.r < 0.01f && mulColor.g < 0.01f && mulColor.b < 0.01f)
        break;

      origin = hit.drop;
      ray = v_add(v_normalized(hit.reflect), v_scale(randDir, SUB(1.0f, reflectivity)));
    }
    else
    {
      k->sky++;
      SIG_STEP(*sig, 0xFFFF);
      pixelColor = c_clamp(c_add(pixelColor, c_mul(c_mul(mulColor, sky_sample(s, ray, k)), s->envColor)));
      break;
    }
  }
  return pixelColor;
}

/* single Scene::trace call for unit tests: dir = pre-drawn randDir */
void rfxo_trace_one(const rfxo_scene * s, const float origin[3], const float ray[3], int refl, const float randDir[3], float rgb[3], uint32_t * sig)
{
  rfxo_counters k;
  uint32_t h = 2166136261u;
  memset(&k, 0, sizeof(k));
  const C3 c = scene_trace(s, v3(origin[0], origin[1], origin[2]), v3(ray[0], ray[1], ray[2]), refl, v3(randDir[0], randDir[1], randDir[2]), &k, &h);
  rgb[0] = c.r; rgb[1] = c.g; rgb[2] = c.b;
  if (sig) *sig = h;
}

/* n independent Scene::trace calls (rfx_trace_rays' operation): ray i from origins[3i] along rays[3i] with randDirs[3i];
 * rgb and sig (may be NULL) receive 3 floats / one signature per ray */
void rfxo_trace_many(const rfxo_scene * s, int n, const float * origins, const float * rays, int refl, const float * randDirs,
                     float * rgb, uint32_t * sig)
{
  for (int i = 0; i < n; i++)
    rfxo_trace_one(s, origins + 3 * (size_t)i, rays + 3 * (size_t)i, refl, randDirs + 3 * (size_t)i, rgb + 3 * (size_t)i,
                   sig ? sig + i : NULL);
}

/* Plane::trace (Plane.cpp:36-73) on n independent (pos, norm, origin, ray) inputs of 12 floats each, for the pin against the
 * reference's own Plane::trace (oracle/ref_plane_probe.cpp).  out: 12 floats per input = hit, drop[3], norm[3], reflected[3],
 * distance, shadowHit (the NULL-output call of Scene.cpp:135); outputs of a miss stay 0 as in the probe. */
void rfxo_plane_probe(const float * in, int n, float * out)
{
  rfxo_counters k;
  memset(&k, 0, sizeof(k));
  for (int i = 0; i < n; i++)
  {
    const float * p = in + 12 * i;
    float * o = out + 12 * i;
    Obj pl;
    memset(&pl, 0, sizeof(pl));
    pl.kind = OBJ_PLANE;
    pl.pos = v3(p[0], p[1], p[2]);
    pl.norm = v3(p[3], p[4], p[5]);
    Hit h;
    memset(&h, 0, sizeof(h));
    memset(o, 0, 12 * sizeof(float));
    const int hit = plane_trace(NULL, &pl, v3(p[6], p[7], p[8]), v3(p[9], p[10], p[11]), &h, &k);
    o[0] = (float)hit;
    if (hit)
    {
      o[1] = h.drop.x; o[2] = h.drop.y; o[3] = h.drop.z;
      o[4] = h.norm.x; o[5] = h.norm.y; o[6] = h.norm.z;
      o[7] = h.reflect.x; o[8] = h.reflect.y; o[9] = h.reflect.z;
      o[10] = h.dist;
    }
    o[11] = (float)plane_trace(NULL, &pl, v3(p[6], p[7], p[8]), v3(p[9], p[10], p[11]), NULL, &k);
  }
}

/* n successive Vector3::randomInsideSphere(1.0f) draws starting from *seed; seed is advanced */
void rfxo_rand_dirs(uint32_t * seed, uint64_t n, float * out_xyz)
{
  for (uint64_t i = 0; i < n; i++)
  {
    const V3 v = rand_in_sphere(seed);
    out_xyz[3 * i] = v.x; out_xyz[3 * i + 1] = v.y; out_xyz[3 * i + 2] = v.z;
  }
}

/* ------------------------------------------------------------------------------------------------ Render */
typedef struct
{
  const rfxo_scene * s;
  V3 eye; M33 view; float rz, wh, hh;
  uint32_t W, H; int refl, samples; int accumulate;
  float * image; uint32_t * sig;
  /* per chunk */
  uint32_t y0, y1; size_t p0, p1; const V3 * dirs; const float * jit; /* jit: rndx, rndy per pixel (samples > 0) */
  int nthreads;
} Job;

typedef struct { const Job * j; int tid; rfxo_counters k; } Worker;

static void * worker_main(void * arg)
{
  Worker * w = (Worker *)arg;
  const Job * j = w->j;
  const uint32_t W = j->W, H = j->H;
#ifdef RFXO_CENSUS
  memset(g_ops, 0, sizeof(g_ops));
#endif
  if (j->samples > 0)
  {
    const int sn = j->samples;
    const float sq = (float)(sn * sn);
    for (size_t p = j->p0 + (size_t)w->tid; p < j->p1; p += (size_t)j->nthreads)
      {
        const uint32_t y = (uint32_t)(p / W), x = (uint32_t)(p % W);
        const size_t local = p - j->p0;
        const float rx = SUB((float)x, j->wh), ry = SUB((float)y, j->hh);
        const float rndx = j->jit ? j->jit[2 * local] : 0, rndy = j->jit ? j->jit[2 * local + 1] : 0;
        C3 fin = c3(0.0f, 0.0f, 0.0f);
        uint32_t h = 2166136261u;
        const V3 * d = j->dirs + local * (size_t)(sn * sn);
        for (int ssx = 0; ssx < sn; ssx++)
          for (int ssy = 0; ssy < sn; ssy++)
          {
            V3 ray = v3(ADD(ADD(rx, DIV((float)ssx, (float)sn)), rndx), ADD(ADD(ry, DIV((float)ssy, (float)sn)), rndy), j->rz);
            ray = m_mulv(&j->view, ray);
            fin = c_add(fin, scene_trace(j->s, j->eye, ray, j->refl, *d++, &w->k, &h));
          }
        fin = c_div(fin, sq);
        float * px = j->image + ((size_t)y * W + x) * 3;
        if (j->accumulate) { px[0] = ADD(px[0], fin.r); px[1] = ADD(px[1], fin.g); px[2] = ADD(px[2], fin.b); }
        else { px[0] = fin.r; px[1] = fin.g; px[2] = fin.b; }
        if (j->sig) j->sig[(size_t)y * W + x] = h;
      }
  }
  else
  {
    /* block preview (Render.cpp:158-173): only block-origin pixels trace; the block is splatted */
    const uint32_t a = (uint32_t)(-j->samples);
    const uint32_t bw = (W + a - 1) / a;
    for (uint32_t y = j->y0 + (uint32_t)w->tid * a; y < j->y1; y += (uint32_t)j->nthreads * a)
      for (uint32_t x = 0; x < W; x += a)
      {
        const size_t local = (size_t)((y - j->y0) / a) * bw + x / a;
        V3 ray = v3(SUB((float)x, j->wh), SUB((float)y, j->hh), j->rz);
        ray = m_mulv(&j->view, ray);
        uint32_t h = 2166136261u;
        const C3 c = scene_trace(j->s, j->eye, ray, j->refl, j->dirs[local], &w->k, &h);
        const uint32_t ex = x + a < W ? x + a : W, ey = y + a < H ? y + a : H;
        for (uint32_t qx = x; qx < ex; qx++)
          for (uint32_t qy = y; qy < ey; qy++)
          {
            float * px = j->image + ((size_t)qy * W + qx) * 3;
            px[0] = c.r; px[1] = c.g; px[2] = c.b;
            if (j->sig) j->sig[(size_t)qy * W + qx] = h;
          }
      }
  }
#ifdef RFXO_CENSUS
  memcpy(w->k.ops, g_ops, sizeof(g_ops));
#endif
  return NULL;
}

static void add_counters(rfxo_counters * a, const rfxo_counters * b)
{
  uint64_t * pa = (uint64_t *)a; const uint64_t * pb = (const uint64_t *)b;
  for (size_t i = 0; i < sizeof(rfxo_counters) / sizeof(uint64_t); i++) pa[i] += pb[i];
}

/* One renderBegin(refl, samples, additive) + renderNext(...) to completion (Render.cpp:116-215).
 *   image            W*H*3 floats, in/out (row 0 = bottom scanline); accumulated into when accumulate != 0
 *                    (the reference's `additiveCounter > 1`, Render.cpp:191-194)
 *   jitter           != 0: draw rndx,rndy per pixel from the Render.cpp TU stream (the reference's `renderAdditive`)
 *   seeds[0]         Vector3.cpp TU LCG state (randDir stream); seeds[1] Render.cpp TU LCG state; both advanced
 *   nthreads         row-interleaved workers; the RNG streams are drawn serially in reference call order first,
 *                    so the result is independent of nthreads
 */
int rfxo_render_pass(const rfxo_scene * s, const float eye[3], const float view[9], float fov, uint32_t W, uint32_t H,
                     int refl, int samples, int jitter, int accumulate, float * image, uint32_t * seeds,
                     rfxo_counters * counters, uint32_t * sig, int nthreads)
{
  if (!s || !W || !H || refl <= 0 || samples == 0) return -1;
  if (nthreads < 1) nthreads = 1;
  if (nthreads > 256) nthreads = 256;

  Job j;
  memset(&j, 0, sizeof(j));
  j.s = s;
  j.eye = v3(eye[0], eye[1], eye[2]);
  memcpy(j.view.m, view, sizeof(float) * 9);
  j.rz = DIV(DIV((float)W, 2.0f), tanf(DIV(fov, 2.0f))); /* Render.cpp:148 */
  j.wh = DIV((float)W, 2.0f);
  j.hh = DIV((float)H, 2.0f);
  j.W = W; j.H = H; j.refl = refl; j.samples = samples; j.accumulate = accumulate;
  j.image = image; j.sig = sig; j.nthreads = nthreads;

  const uint32_t a = samples < 0 ? (uint32_t)(-samples) : 1u;
  const size_t perPixel = samples > 0 ? (size_t)samples * samples : 1;
  /* chunking bounds the pre-drawn direction buffer to ~2M samples: linear pixel ranges when samples > 0,
     block-aligned row ranges in block-preview mode */
  size_t rows = (size_t)(2u << 20) / W + 1;
  rows = ((rows + a - 1) / a) * a;
  if (rows > H) rows = H;
  size_t pixPerChunk = (size_t)(2u << 20) / perPixel;
  if (pixPerChunk < 1) pixPerChunk = 1;
  const size_t npix = (size_t)W * H;
  if (pixPerChunk > npix) pixPerChunk = npix;

  V3 * dirs = (V3 *)malloc(sizeof(V3) * (samples > 0 ? pixPerChunk * perPixel : rows * W));
  float * jit = (jitter && samples > 0) ? (float *)malloc(sizeof(float) * 2 * pixPerChunk) : NULL;
  pthread_t th[256];
  Worker wk[256];
  rfxo_counters total;
  memset(&total, 0, sizeof(total));

  /* both streams are drawn serially in the reference's call order: per pixel rndx, rndy (Render.cpp:177-178) and one
     randDir per Scene::trace call (Scene.cpp:75); the two are independent LCGs so only per-stream order matters */
  const size_t nchunks = samples > 0 ? (npix + pixPerChunk - 1) / pixPerChunk : (H + rows - 1) / rows;
  for (size_t c = 0; c < nchunks; c++)
  {
    size_t n = 0;
    if (samples > 0)
    {
      j.p0 = c * pixPerChunk;
      j.p1 = j.p0 + pixPerChunk < npix ? j.p0 + pixPerChunk : npix;
      for (size_t p = j.p0; p < j.p1; p++)
      {
        if (jit)
        {
          jit[2 * (p - j.p0)] = DIV((float)rng_next(&seeds[1]), (float)0x7FFF);
          jit[2 * (p - j.p0) + 1] = DIV((float)rng_next(&seeds[1]), (float)0x7FFF);
        }
        for (size_t k2 = 0; k2 < perPixel; k2++) dirs[n++] = rand_in_sphere(&seeds[0]);
      }
    }
    else
    {
      j.y0 = (uint32_t)(c * rows);
      j.y1 = (j.y0 + rows < H) ? (uint32_t)(j.y0 + rows) : H;
      for (uint32_t y = j.y0; y < j.y1; y++)
        for (uint32_t x = 0; x < W; x++)
          if (!(x % a || y % a)) dirs[n++] = rand_in_sphere(&seeds[0]);
    }

    j.dirs = dirs; j.jit = jit;
    for (int t = 0; t < nthreads; t++)
    {
      wk[t].j = &j; wk[t].tid = t;
      memset(&wk[t].k, 0, sizeof(rfxo_counters));
      if (nthreads > 1) pthread_create(&th[t], NULL, worker_main, &wk[t]);
      else worker_main(&wk[t]);
    }
    for (int t = 0; t < nthreads; t++)
    {
      if (nthreads > 1) pthread_join(th[t], NULL);
      add_counters(&total, &wk[t].k);
    }
  }
  free(dirs); free(jit);
  if (counters) *counters = total;
  return 0;
}

/* imagePixel(x,y) (Render.cpp:103-114) and imagePixel(x,y).argb() (Color.cpp:114-117; MAKEARGB Color.h:11-15) */
void rfxo_resolve(const float * image, uint32_t W, uint32_t H, int additiveCounter, float * rgbf, uint32_t * argb)
{
  for (size_t p = 0; p < (size_t)W * H; p++)
  {
    C3 c = c3(image[3 * p], image[3 * p + 1], image[3 * p + 2]);
    if (additiveCounter > 1) c = c_div(c, (float)additiveCounter);
    if (rgbf) { rgbf[3 * p] = c.r; rgbf[3 * p + 1] = c.g; rgbf[3 * p + 2] = c.b; }
    if (argb)
      argb[p] = ((uint32_t)(unsigned char)MUL(c.r, 255.999f) << 16) | ((uint32_t)(unsigned char)MUL(c.g, 255.999f) << 8) |
                (uint32_t)(unsigned char)MUL(c.b, 255.999f);
  }
}

/* Camera(eye, at, fov) (Camera.cpp:24-36): view columns = ox, oy, oz */
void rfxo_camera_lookat(const float eye[3], const float at[3], float view[9])
{
  const V3 up = v3(0.0f, 1.0f, 0.0f);
  const V3 oz = v_normalized(v_sub(v3(at[0], at[1], at[2]), v3(eye[0], eye[1], eye[2])));
  const V3 ox = v_normalized(v_cross(up, oz));
  const V3 oy = v_normalized(v_cross(oz, ox));
  const M33 m = m_cols(ox, oy, oz);
  memcpy(view, m.m, sizeof(float) * 9);
}

int rfxo_census_enabled(void)
{
#ifdef RFXO_CENSUS
  return 1;
#else
  return 0;
#endif
}
