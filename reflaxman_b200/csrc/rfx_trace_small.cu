// rfx_trace_small.cu — K2 for scenes that fit the kernel-parameter constant bank (the reference's demo scene and
// anything up to 16 spheres / 8 triangles / 2 planes / 4 lights / 8 textures).
//
// Design (B200, FP32 CUDA cores; this path has no dense contraction, so no tensor cores):
//   * The whole scene travels as a __grid_constant__ kernel parameter: every sphere/triangle coefficient is a
//     constant-bank operand — no global or shared loads in the test loops.
//   * ONE intersection call site.  Scene::trace is a state machine per lane: the query in flight is either the bounce
//     segment (closest hit) or the shadow ray of light `li` (any hit); lanes in either state share the same pass over
//     the objects.  That halves the code of the kernel (it fits the 32 KB L1.5 instruction cache) and keeps lanes of a
//     warp that sit in different phases busy in the same loops.
//   * The pass over the objects: four spheres per trip — the reference's discriminant expression, 17 un-fused FP32 ops
//     per sphere, the FP32 pipe is the limit there — behind ONE divergent gate region for their sqrt/divide tails; then
//     the triangles (plane-side test on sign bits, tail with the divide); planes last.
//   * Warps own 4x8 pixel tiles of a 2-D grid (no integer division per thread); tiles are started in the cost order the
//     previous launch recorded (TileOrder: long paths first), which removes the ~45 us drain behind the mirror-sphere tiles.
//   * 128-thread CTAs, 63 registers, 8 CTAs per SM; the frame is written with one 128-bit store per tile row (split frames that
//     store into another GPU's framebuffer: 64-byte row segments staged through shared memory).
//   * The same kernel (MULTI instantiation) serves row-aligned SSAA / additive / float-image slices of the Render API;
//     k_trace_small_any keeps the arbitrary pixel slices, block preview and signature runs.
//   * The bounce recursion is the reference's own bounded iterative loop carrying throughput (mulColor).
// Every step above was measured; profiles/README.md has the numbers, including the experiments that were not kept.
//
// ARITHMETIC CONTRACT: compiled with --fmad=false, no fast-math: every + - * / sqrtf is the IEEE binary32 RN
// operation, in the reference's evaluation order (SURVEY.md Appendix A).  Hoisting a per-ray invariant (|ray|^2,
// 2*ray, 4a, 2a) or skipping work whose result is provably unused does not change any produced bit.
//
// Reference map (path:line under /root/reference/src/common): Sphere.cpp:44-85, Triangle.cpp:53-108, Plane.cpp:36-73,
// Scene.cpp:73-236, Render.cpp:136-215, trace_math.cpp:3-23, Texture.cpp:216-269, Skybox.cpp:39-106, Color.cpp:114-117.
#include "rfx_kernels.h"
#include "rfx_device.cuh"

namespace rfx
{

#ifndef RFX_TILE_W
#define RFX_TILE_W 4u      // pixel tile of one warp: RFX_TILE_W x RFX_TILE_H = 32 (4x8 measured best, profiles/variants_d_r1.jsonl)
#endif
#define RFX_TILE_H (32u / RFX_TILE_W)
#ifndef RFX_TILE_BOUNDS
// cost classes of the tile scheduler: class c holds the tile groups whose longest path has >= bound[c] segments (last class: the rest)
#define RFX_TILE_BOUNDS { 8u, 4u, 2u }
#endif
#ifndef RFX_ANY_MINBLOCKS
#define RFX_ANY_MINBLOCKS 6        // general kernel (signatures, float image, every mode)
#endif
#ifndef RFX_SMALL_THREADS
#define RFX_SMALL_THREADS 128
#endif
#ifndef RFX_ALIGN_PHASES
#define RFX_ALIGN_PHASES 1         // single-light scenes: lanes whose hit faces no light idle through the shadow trip (keeps the tile's lanes in one phase)
#endif
#ifndef RFX_STRIP_STAGING
#define RFX_STRIP_STAGING 1        // split frames: 64-byte row-segment stores staged through shared memory (0: the A/B arm, direct 16-byte stores)
#endif
#ifndef RFX_PRIMARY_CULL
#define RFX_PRIMARY_CULL 1         // the first query of a path (origin = eye) skips the object-loop trips whose screen bounds miss the warp's tile
#endif
#ifndef RFX_SMALL_MINBLOCKS
#define RFX_SMALL_MINBLOCKS 8      // fast kernel: 64 registers, no spills, 32 warps per SM
#endif

// Scene features a kernel instantiation supports.  The lean instantiation (FEAT = 0: no planes, no texels, one light) is
// what the reference's demo scene needs; leaving the other paths out keeps its code inside the 32 KB instruction cache.
constexpr int F_PLANES = 1, F_TEXELS = 2, F_LIGHTS = 4, F_ALL = 7;

constexpr int SM_TRI_BIT = SMALL_MAX_SPHERES;                       // object slots: spheres | triangles | planes
constexpr int SM_PLANE_BIT = SMALL_MAX_SPHERES + SMALL_MAX_TRIS;

struct Best
{
  float dist;
  int slot;          // slot of the winning object, -1 = none
  int order;         // insertion index (closest-hit tie-break, reference Scene.cpp:98 walks the list in order)
  float t;
  float u, v;        // triangle barycentrics
};

__device__ __forceinline__ void considerHit(Best & best, float dist, int slot, int order, float t, float u, float v)
{
  if (dist < best.dist || (dist == best.dist && order < best.order))
  {
    best.dist = dist; best.slot = slot; best.order = order; best.t = t; best.u = u; best.v = v;
  }
}

// All objects against one ray.  `skip` is the slot the query ignores (the shadow loop's `*obj != hitObject`,
// Scene.cpp:135; -1 = none).  anyHit: the caller only asks whether something is hit (shadow query), so a lane that has
// found an occluder stops entering the sqrt/divide tails.
// The object loops run over [range.s0, range.s1) of the sphere quads and [range.t0, range.t1) of the triangles (byte offsets):
// everything for every query but the first of a path, whose tile may see only part of the scene (PrimaryCull below).
struct ObjRange { int s0, s1, t0, t1; };

template <int FEAT, bool RANGED>
__device__ __forceinline__ void intersectSmall(const SmallScene & sc, V3 o, V3 d, int skip, bool anyHit, Best & best, const ObjRange range)
{
  const float a = vsqlen(d);                                          // Sphere.cpp:50
  const float r2x = d.x * 2.0f, r2y = d.y * 2.0f, r2z = d.z * 2.0f;   // 2.0f * ray, Sphere.cpp:51
  const float a2 = 2.0f * a;                                          // Sphere.cpp:57
  // A lane that must not take any (more) sphere hit — a <= 2^-63 (Sphere.cpp:55), or an any-hit query that has found its
  // occluder — gets a NaN in place of 4a: its discriminant becomes NaN and fails `disc >= 0` without an extra predicate
  float a4 = (a > RFX_VSN) ? 4.0f * a : __int_as_float(0x7FC00000);  // Sphere.cpp:53

  // ---- spheres: discriminant of Sphere.cpp:49-53 with the per-ray invariants hoisted.  t = (-b - sqrt(disc)) / 2a can
  // only exceed 2^-63 when b < 0 (sqrt >= 0, 2a > 0), so lanes with b >= 0 never enter the tail — same decisions, fewer sqrt.
  const char * sphBase = reinterpret_cast<const char *>(sc.sph);
  const char * ordBase = reinterpret_cast<const char *>(&sc.mat[0].order);
  const int skipOff = skip << 4;
  // One induction variable: the byte offset of sphere i inside sc.sph (16 B each; Material is 32 B).
#define RFX_SPHERE_REJECT(OFF, S, B, DISC)                                                   \
    const float4 S = *reinterpret_cast<const float4 *>(sphBase + (OFF));                     \
    float B, DISC;                                                                           \
    {                                                                                        \
      const float vx = o.x - S.x, vy = o.y - S.y, vz = o.z - S.z;                            \
      B = (r2x * vx + r2y * vy) + r2z * vz;                                                  \
      const float c = ((vx * vx + vy * vy) + vz * vz) - S.w;                                 \
      DISC = B * B - a4 * c;                                                                 \
    }
#define RFX_SPHERE_GATE(B, DISC) ((DISC) >= 0.0f && (B) < 0.0f)
#define RFX_SPHERE_TAIL(OFF, B, DISC)                                                        \
    {                                                                                        \
      const float t = (-B - sqrtf(DISC)) / a2;                        /* Sphere.cpp:57 */    \
      if (t > RFX_VSN)                                                                       \
      {                                                                                      \
        const float fx = d.x * t, fy = d.y * t, fz = d.z * t;                                \
        const float dist = sqrtf((fx * fx + fy * fy) + fz * fz);      /* fullRay.length(), Sphere.cpp:62 */ \
        if (dist > RFX_DELTA && (OFF) != skipOff)   /* the skipped sphere is the one the ray leaves (b > 0): it rarely gets here */ \
        {                                                                                    \
          considerHit(best, dist, (OFF) >> 4, *reinterpret_cast<const int *>(ordBase + 2 * (OFF)), t, 0.0f, 0.0f); \
          if (anyHit) a4 = __int_as_float(0x7FC00000);                                       \
        }                                                                                    \
      }                                                                                      \
    }
  // Four spheres per trip: their reject chains are independent (ILP for a scheduler that holds ~7 warps), they share the
  // loop bookkeeping, and ONE divergent region gates all their tails (the common case — no lane passes any gate — costs one
  // branch).  The discriminants of a trip are evaluated before its tails, so an any-hit lane that closes in an earlier tail
  // (a4 becomes NaN) must not enter a later one.  The host pads the sphere array to whole quads with NaN records, whose
  // discriminant is NaN and whose gate stays shut: no remainder loops — 350 SASS instructions (three more copies of the tail) that
  // the demo scene never executed and that still cost 3 % of the kernel (202.0 -> 195.9 us: the instruction cache is that tight).
  // (ONE copy of the tail, walked per lane over its open gates, is 184 instructions less again but 2 % slower: profiles/r2_prim.)
  const int endQuad = RANGED ? range.s1 : (sc.nS << 4);
  int off = RANGED ? range.s0 : 0;
#pragma unroll 1
  for (; off != endQuad; off += 64)
  {
    asm volatile("" : "+r"(off));   // keeps `off` the only induction variable (ptxas otherwise strength-reduces it into five)
    RFX_SPHERE_REJECT(off, s0, b0, disc0)
    RFX_SPHERE_REJECT(off + 16, s1, b1, disc1)
    RFX_SPHERE_REJECT(off + 32, s2, b2, disc2)
    RFX_SPHERE_REJECT(off + 48, s3, b3, disc3)
    const bool g0 = RFX_SPHERE_GATE(b0, disc0), g1 = RFX_SPHERE_GATE(b1, disc1), g2 = RFX_SPHERE_GATE(b2, disc2), g3 = RFX_SPHERE_GATE(b3, disc3);
    if (g0 || g1 || g2 || g3)
    {
      if (g0) RFX_SPHERE_TAIL(off, b0, disc0)
      if (g1 && a4 == a4) RFX_SPHERE_TAIL(off + 16, b1, disc1)
      if (g2 && a4 == a4) RFX_SPHERE_TAIL(off + 32, b2, disc2)
      if (g3 && a4 == a4) RFX_SPHERE_TAIL(off + 48, b3, disc3)
    }
  }
#undef RFX_SPHERE_GATE
#undef RFX_SPHERE_REJECT
#undef RFX_SPHERE_TAIL

  // ---- triangles: third row of axTrans*(origin - v0) and axTrans*ray (Triangle.cpp:56-57, Matrix33.cpp:232-234);
  // t = -oz/rz > 2^-63 needs |rz| > 2^-63 and oz, rz nonzero of opposite sign (the sign of an IEEE quotient is exact), so
  // everything else is skipped without dividing.  A closed lane (any-hit query
  // that has its occluder) carries +inf as the |rz| threshold.
  float rzMin = (anyHit && best.slot >= 0) ? __int_as_float(0x7F800000) : RFX_VSN;
  const char * triBase = reinterpret_cast<const char *>(sc.triPk);
  const char * triOrd = reinterpret_cast<const char *>(&sc.mat[SM_TRI_BIT].order);
  const int skipTri = (skip - SM_TRI_BIT) * 48;
  const int endTri = RANGED ? range.t1 : sc.nT * 48;
  // (a zero oz — a ray that starts exactly on the plane, common for rays leaving a floor triangle towards its coplanar
  // neighbour — would give t = 0 and fail in the tail, but 0 / rz takes div.rn's 30-instruction slow path: the gate rejects it)
#define RFX_TRI_REJECT(OFF, A, B, PX, PY, PZ, OZ, RZ)                                         \
    const float4 A = *reinterpret_cast<const float4 *>(triBase + (OFF));                      \
    const float4 B = *reinterpret_cast<const float4 *>(triBase + (OFF) + 16);                 \
    const float PX = o.x - A.x, PY = o.y - A.y, PZ = o.z - A.z;                               \
    const float OZ = (PX * A.w + PY * B.x) + PZ * B.y;                                        \
    const float RZ = (d.x * A.w + d.y * B.x) + d.z * B.y;
#define RFX_TRI_GATE(OFF, OZ, RZ) ((__float_as_int(OZ) ^ __float_as_int(RZ)) < 0 && fabsf(RZ) > rzMin && fabsf(OZ) > 0.0f && (OFF) != skipTri)
#define RFX_TRI_TAIL(OFF, B, PX, PY, PZ, OZ, RZ)                                              \
    {                                                                                         \
      const float t = -OZ / RZ;                                       /* Triangle.cpp:61 */   \
      if (t > RFX_VSN)                                                                        \
      {                                                                                       \
        const float4 C = *reinterpret_cast<const float4 *>(triBase + (OFF) + 32);             \
        const float ox = (PX * B.z + PY * B.w) + PZ * C.x;                                    \
        const float rx = (d.x * B.z + d.y * B.w) + d.z * C.x;                                 \
        const float oy = (PX * C.y + PY * C.z) + PZ * C.w;                                    \
        const float ry = (d.x * C.y + d.y * C.z) + d.z * C.w;                                 \
        const float u = ox + t * rx;                                  /* Triangle.cpp:65-66 */ \
        const float v = oy + t * ry;                                                          \
        if (u >= 0.0f && v >= 0.0f && u + v < 1.0f)                                           \
        {                                                                                     \
          const float fx = d.x * t, fy = d.y * t, fz = d.z * t;                               \
          const float sq = (fx * fx + fy * fy) + fz * fz;                                     \
          if (sq > RFX_DELTA * RFX_DELTA)                                                     \
          {                                                                                   \
            const int k = (OFF) / 48;                                                         \
            considerHit(best, sqrtf(sq), SM_TRI_BIT + k, *reinterpret_cast<const int *>(triOrd + k * 32), t, u, v); \
            if (anyHit) rzMin = __int_as_float(0x7F800000);                                   \
          }                                                                                   \
        }                                                                                     \
      }                                                                                       \
    }
  int toff = RANGED ? range.t0 : 0;
#pragma unroll 1
  for (; toff != endTri; toff += 48)
  {
    asm volatile("" : "+r"(toff));
    RFX_TRI_REJECT(toff, A0, B0, px0, py0, pz0, oz0, rz0)
    if (RFX_TRI_GATE(toff, oz0, rz0)) RFX_TRI_TAIL(toff, B0, px0, py0, pz0, oz0, rz0)
  }
#undef RFX_TRI_REJECT
#undef RFX_TRI_GATE
#undef RFX_TRI_TAIL

  // ---- planes (unreachable through the reference's Scene, kept for API completeness): Plane.cpp:36-73
  const int nP = (FEAT & F_PLANES) ? sc.nP : 0;
#pragma unroll 1
  for (int k = 0; k < nP; k++)
  {
    if ((SM_PLANE_BIT + k) == skip) continue;
    const Plane & pl = sc.pl[k];
    const V3 n = mk(pl.n[0], pl.n[1], pl.n[2]);
    const V3 vop = mk(pl.pos[0] - o.x, pl.pos[1] - o.y, pl.pos[2] - o.z);
    const float den = vdot(n, d);
    if (fabsf(den) > RFX_VSN)
    {
      const float t = vdot(n, vop) / den;
      if (t > RFX_VSN)
      {
        const float fx = d.x * t, fy = d.y * t, fz = d.z * t;
        const float sq = (fx * fx + fy * fy) + fz * fz;
        if (sq > RFX_DELTA * RFX_DELTA) considerHit(best, sqrtf(sq), SM_PLANE_BIT + k, sc.mat[SM_PLANE_BIT + k].order, t, 0.0f, 0.0f);
      }
    }
  }
}

// ---- Scene::trace (reference Scene.cpp:73-236) ------------------------------------------------------------------------
// `events` counts bounce-loop iterations in its low half and shadow rays in its high half (one register instead of two).
// RANGED: `first` is the object range of the path's first query (the tile's PrimaryCull answer); every later query sees everything.
//
// BATCH (frames of one camera, see k_trace_small): everything a path computes before it first reads randDir — the first query
// and the hit set-up — is the same in every frame.  SEG_FIRST runs that first segment only and leaves its state in `cache`
// (PATH_WORDS words at a stride of SMALL_THREADS, shared memory); SEG_RESUME starts from that state at the choice of the first
// light, with this frame's randDir.  A primary miss stores its finished colour (hslot = -1).  Same operations, same operands.
constexpr int SEG_WHOLE = 0, SEG_FIRST = 1, SEG_RESUME = 2;
constexpr int PATH_WORDS = 17;
constexpr int SMALL_THREADS = RFX_SMALL_THREADS;

template <bool SIG, int FEAT, bool RANGED = false, bool BATCH = false>
__device__ __forceinline__ V3 traceSmall(const SmallScene & sc, V3 origin, V3 ray, int reflNumber, V3 randDir, uint32_t & events, uint32_t & sig,
                                         const ObjRange first = ObjRange(), int mode = SEG_WHOLE, float * cache = nullptr)
{
  V3 mul = mk(1.0f, 1.0f, 1.0f);
  V3 pix = mk(0.0f, 0.0f, 0.0f);
  if (reflNumber <= 0) return pix;

  // The query in flight is (qo, qd).  Bounce state: qo = origin, qd = ray of the reference's loop.  Shadow state
  // (hslot >= 0 and shadowQuery): qo = drop, qd = the jittered ray towards light li, the hit object is ignored.
  V3 qo = origin, qd = ray;
  bool shadowQuery = false;
  int li = 0, hslot = -1;   // (the segment index of the reference's loop is the low half of `events` minus one)
  // what survives of the hit while its lights are being answered
  V3 norm = ray, reflect = ray, color = mul;
  // light sums of the hit: loop-carried only when a hit can have a second shadow query (F_LIGHTS); with one light they are
  // born in the shadow answer and die in the finish of the same trip, which frees six registers across the object loops
  V3 carryLight = pix, carrySpec = pix;
  float normLen = 0.0f, reflectLen = 0.0f, mrefl = 0.0f;
  float rfs = 0.0f;         // weight of the reflected continuation (Scene.cpp:196 / :207), negated for metals (one register
                            // for the weight and the material type; the weight is in [0.2, 1], never zero)
  ObjRange range = first;
  constexpr int S = SMALL_THREADS;
  bool resume = false;
  if (BATCH && mode == SEG_RESUME)
  {
    events++;                                                            // the first bounce-loop iteration, run once per batch
    color = mk(cache[9 * S], cache[10 * S], cache[11 * S]);
    hslot = __float_as_int(cache[16 * S]);
    if (hslot < 0) return color;                                         // primary miss: the finished colour
    qo = mk(cache[0], cache[S], cache[2 * S]);
    norm = mk(cache[3 * S], cache[4 * S], cache[5 * S]);
    reflect = mk(cache[6 * S], cache[7 * S], cache[8 * S]);
    normLen = cache[12 * S]; reflectLen = cache[13 * S]; mrefl = cache[14 * S]; rfs = cache[15 * S];
    resume = true;
  }

  for (;;)
  {
    V3 sumLight = (FEAT & F_LIGHTS) ? carryLight : mk(0.0f, 0.0f, 0.0f);
    V3 sumSpec = (FEAT & F_LIGHTS) ? carrySpec : mk(0.0f, 0.0f, 0.0f);
    if (BATCH && resume) { resume = false; goto chooseLight; }   // (a forward jump inside the loop body: one intersection call site)
    Best hit;
    hit.dist = FLT_MAX; hit.slot = -1; hit.order = 0x7FFFFFFF; hit.t = 0; hit.u = 0; hit.v = 0;
    intersectSmall<FEAT, RANGED>(sc, qo, qd, shadowQuery ? hslot : -1, shadowQuery, hit, range);
    if (RANGED) { range.s0 = 0; range.s1 = sc.nS << 4; range.t0 = 0; range.t1 = sc.nT * 48; }   // rematerialised from the constant bank

    if (!shadowQuery)
    {
      // ---- closest hit of the bounce segment (origin = qo, ray = qd), Scene.cpp:80-112
      events++;
      if (hit.slot < 0)
      {
        if (SIG) RFX_SIG(sig, 0xFFFF);
        float u, v;
        skyDirToUv(qd, vlen(qd), sc.halfTileW, sc.halfTileH, u, v);
        const V3 sky = texSampleRef((FEAT & F_TEXELS) && sc.skyTex >= 0 ? &sc.tex[sc.skyTex] : nullptr, sc.byteLut, u, v);
        pix = mk(clamp01(pix.x + (mul.x * sky.x) * sc.env[0]), clamp01(pix.y + (mul.y * sky.y) * sc.env[1]),
                 clamp01(pix.z + (mul.z * sky.z) * sc.env[2]));            // Scene.cpp:230-231
        if (BATCH && mode == SEG_FIRST) { cache[9 * S] = pix.x; cache[10 * S] = pix.y; cache[11 * S] = pix.z; cache[16 * S] = __int_as_float(-1); }
        break;
      }
      if (SIG) RFX_SIG(sig, hit.order + 1);
      const V3 full = vscale(qd, hit.t);
      qo = vadd(qo, full);                                                 // drop point: origin of everything that follows
      const Material & m = sc.mat[hit.slot];
      color = mk(m.r, m.g, m.b);
      mrefl = m.reflectivity;
      const bool dielectric = m.type == 1;
      hslot = hit.slot;
      if (hit.slot < SM_TRI_BIT)
      {
        const float4 s = sc.sph[hit.slot];
        norm = mk(qo.x - s.x, qo.y - s.y, qo.z - s.z);                     // Sphere.cpp:67
      }
      else if (hit.slot < SM_PLANE_BIT)
      {
        const Triangle & tr = sc.tri[hit.slot - SM_TRI_BIT];
        norm = mk(tr.n[0], tr.n[1], tr.n[2]);
        const int tex = m.tex;
        if (tex >= 0)
        {
          // tuvTrans * Vector3(u, v, 0): (u*_11 + v*_12) + 0*_13 with _13 == 0, Triangle.cpp:91
          const float tx = (hit.u * tr.tuv[0] + hit.v * tr.tuv[1]) + 0.0f;
          const float ty = (hit.u * tr.tuv[2] + hit.v * tr.tuv[3]) + 0.0f;
          color = texSampleRef((FEAT & F_TEXELS) ? &sc.tex[tex] : nullptr, sc.byteLut, tr.tu0 + tx, tr.tv0 + ty);
        }
      }
      else if (FEAT & F_PLANES)
      {
        const Plane & pl = sc.pl[hit.slot - SM_PLANE_BIT];
        norm = mk(pl.n[0], pl.n[1], pl.n[2]);
      }
      reflect = reflectVec(full, norm);
      normLen = vlen(norm);
      reflectLen = vlen(reflect);
      // the continuation weight only depends on ray and norm: evaluate it while the ray is still in registers
      rfs = -0.8f;                                                         // metal, Scene.cpp:207
      if (dielectric)                                                      // Scene.cpp:192-196
      {
        const float a = vlen(qd) * normLen;
        const float cosA = (a > RFX_VSN) ? clamp01(((qd.x * -norm.x + qd.y * -norm.y) + qd.z * -norm.z) / a) : 0.0f;
        rfs = 0.2f + 0.8f * cubeLikePowf(1.0f - cosA);
      }
      sumLight = mk(0.0f, 0.0f, 0.0f);
      sumSpec = mk(0.0f, 0.0f, 0.0f);
      li = 0;
      if (BATCH && mode == SEG_FIRST)
      {
        cache[0] = qo.x; cache[S] = qo.y; cache[2 * S] = qo.z;
        cache[3 * S] = norm.x; cache[4 * S] = norm.y; cache[5 * S] = norm.z;
        cache[6 * S] = reflect.x; cache[7 * S] = reflect.y; cache[8 * S] = reflect.z;
        cache[9 * S] = color.x; cache[10 * S] = color.y; cache[11 * S] = color.z;
        cache[12 * S] = normLen; cache[13 * S] = reflectLen; cache[14 * S] = mrefl; cache[15 * S] = rfs;
        cache[16 * S] = __int_as_float(hslot);
        return pix;
      }
    }
    else
    {
      // ---- answer of the shadow query for light li, Scene.cpp:125-186
      const Light & L = sc.light[(FEAT & F_LIGHTS) ? li : 0];
      // (li < 0: the "query" was the idle trip of a hit that faces no light — see below — and has no answer to take)
      const bool inShadow = hit.slot >= 0 || (RFX_ALIGN_PHASES && !SIG && !(FEAT & F_LIGHTS) && li < 0);
      if (SIG) RFX_SIG(sig, 0x100 + 2 * li + (inShadow ? 1 : 0));
      if (!inShadow)
      {
        const V3 toLight = mk(L.ox - qo.x, L.oy - qo.y, L.oz - qo.z);     // the same subtractions as before the query
        const float facing = vdot(toLight, norm);
        const float toLightLen = vlen(toLight);
        float a = toLightLen * normLen;
        const float lightDropCos = (a > RFX_VSN) ? facing / a : 0.0f;
        if (L.power > RFX_VSN)
        {
          sumLight.x = sumLight.x + (L.r * lightDropCos) * L.power;       // Scene.cpp:156
          sumLight.y = sumLight.y + (L.g * lightDropCos) * L.power;
          sumLight.z = sumLight.z + (L.b * lightDropCos) * L.power;
        }
        a = vsqlen(toLight);
        const float larsc = (a > RFX_VSN) ? 1.0f - L.radius * L.radius / a : 0.0f;   // Scene.cpp:160
        if (larsc > 0)
        {
          // dropToLight.normalized(): same length value as toLightLen (same operations), Vector3.cpp:55-64
          const V3 nl = (toLightLen > RFX_VSN) ? mk(toLight.x / toLightLen, toLight.y / toLightLen, toLight.z / toLightLen) : toLight;
          const V3 dtl = vadd(nl, vscale(randDir, 1.0f - mrefl));
          a = vlen(dtl) * reflectLen;
          float rsc = (a > RFX_VSN) ? vdot(dtl, reflect) / a : 0.0f;
          rsc = clamp01(rsc + (1.0f - sqrtf(larsc)));
          if (rsc > RFX_VSN && L.radius > RFX_VSN)
          {
            const float sp = powLikePowf(rsc, 1 + 3 * mrefl * toLightLen / L.radius) * mrefl;   // Scene.cpp:175
            sumSpec.x = sumSpec.x + L.r * sp;
            sumSpec.y = sumSpec.y + L.g * sp;
            sumSpec.z = sumSpec.z + L.b * sp;
          }
        }
      }
      li++;
    }

    // ---- next light that faces the surface gets a shadow query, Scene.cpp:118-129
  chooseLight:
    bool cast = false;
    const int nL = (FEAT & F_LIGHTS) ? sc.nL : ((sc.nL > 0 && !shadowQuery) ? 1 : 0);   // one light: an answered query is the last
    for (; li < nL; li++)
    {
      const Light & L = sc.light[li];
      const V3 toLight = mk(L.ox - qo.x, L.oy - qo.y, L.oz - qo.z);
      if (vdot(toLight, norm) > RFX_VSN)
      {
        qd = vadd(toLight, vscale(randDir, L.radius));                    // Scene.cpp:129
        cast = true;
        break;
      }
    }
#ifdef RFX_DEBUG_FIRST_SEGMENT
    // debug build (tools/first_segment_prize.py): the path ends after its first hit set-up and first-light choice; the colour
    // folds in everything that set-up produced so that none of it is dead code
    if (!shadowQuery)
      return mk(color.x * rfs + qd.x + norm.x + reflect.x, color.y * mrefl + qd.y + normLen + reflect.y,
                color.z + qd.z + reflectLen + (float)(li + hslot) + norm.z + reflect.z + qo.x);
#endif
    if (cast)
    {
      if (FEAT & F_LIGHTS) { carryLight = sumLight; carrySpec = sumSpec; }
      shadowQuery = true;
      events += 0x10000u;
      continue;
    }
    if (RFX_ALIGN_PHASES && !SIG && !(FEAT & F_LIGHTS) && !shadowQuery)
    {
      // Single-light scenes: a hit that faces no light would finish now and start its next bounce while its neighbours run their
      // shadow queries — from then on the lanes of the warp are in both phases of the machine on every trip, and every trip executes
      // the hit set-up AND the shadow answer with part of the lanes.  It sits out one trip instead (a null query: a zero ray fails
      // every gate; the warp runs the object loops for its neighbours anyway), so that bounce and shadow trips keep alternating
      // for the whole tile.  Nothing it computes changes.
      qd = mk(0.0f, 0.0f, 0.0f);
      shadowQuery = true;
      li = -1;
      continue;
    }

    // ---- all lights answered: finish the hit, Scene.cpp:189-226
    sumLight = mk(sc.ambient[0] * sc.ambientPower + sumLight.x, sc.ambient[1] * sc.ambientPower + sumLight.y,
                  sc.ambient[2] * sc.ambientPower + sumLight.z);         // Scene.cpp:189
    const bool dielectric = rfs > 0.0f;
    const float rf = fabsf(rfs);
    const float k = 1.0f - rf;
    const V3 fin = mk(((color.x * k) * sumLight.x + sumSpec.x) * mul.x, ((color.y * k) * sumLight.y + sumSpec.y) * mul.y,
                      ((color.z * k) * sumLight.z + sumSpec.z) * mul.z); // Scene.cpp:198-199 / 209-210
    if (dielectric) mul = vscale(mul, rf);                               // Scene.cpp:202
    else mul = mk(mul.x * (color.x * rf), mul.y * (color.y * rf), mul.z * (color.z * rf));   // Scene.cpp:213

    pix = mk(clamp01(pix.x + fin.x), clamp01(pix.y + fin.y), clamp01(pix.z + fin.z));

    if (mul.x < 0.01f && mul.y < 0.01f && mul.z < 0.01f) break;
    if ((int)(events & 0xFFFFu) >= reflNumber) break;                    // ++refl < reflNumber, Scene.cpp:80

    // reflect.normalized(): its length is the reflectLen of the hit set-up (same operands, same operations), Vector3.cpp:55-64
    const V3 rn = (reflectLen > RFX_VSN) ? mk(reflect.x / reflectLen, reflect.y / reflectLen, reflect.z / reflectLen) : reflect;
    qd = vadd(rn, vscale(randDir, 1.0f - mrefl));                        // Scene.cpp:226
    shadowQuery = false;
  }
  return pix;
}

// ---- screen bounds of the objects for the primary rays ---------------------------------------------------------------
// Every path of a launch starts at the eye, and a warp owns a 4x8 pixel tile: most tiles see none of the spheres and a part
// of the triangles.  Per launch the host bounds, for each sphere and triangle of the scene, the pixels whose primary ray can pass
// that object's hit test (a rectangle, conservative: float noise of the test, SSAA sub-samples and additive jitter are inside
// the margins).  A warp compares its tile with the rectangles (one object per lane, one ballot) and its FIRST pass over the
// objects runs only the sphere quads / triangles from the first to the last candidate.  A trip that is skipped could not have
// produced a hit, so nothing a path computes changes; later queries of the path (shadow rays, bounces) see every object.
// tests/test_oracle.py::test_primary_bounds_are_conservative evaluates the kernel's float expressions on every pixel for
// random cameras (inside spheres, under the floor, looking away) against rfx_selftest_primary_bounds.
// (struct PrimaryCull: rfx_kernels.h; the sphere rectangles, cullSphere, and the helpers: rfx_eye_grid.h, which the screen grid of the
// blob scenes' first query shares)

// A triangle: the edges come back out of axTrans (its inverse holds v2-v0 | v1-v0 | -n), the triangle is widened in barycentric
// space by the noise of u = ox + t*rx (Triangle.cpp:65-66), clipped against a near plane so close to the eye that what it cuts
// off projects outside the image, and projected.
static int4 cullTriangle(const double * c0, const double * c1, const double * c2, const double * eye, double rz, double wHalf, double hHalf,
                         double W, double H, const Triangle & tr)
{
  double A[9];
  for (int i = 0; i < 9; i++) { A[i] = (double)tr.ax[i]; if (!(fabs(A[i]) < 1e300)) return cullFull(); }
  const double det = A[0] * (A[4] * A[8] - A[5] * A[7]) - A[1] * (A[3] * A[8] - A[5] * A[6]) + A[2] * (A[3] * A[7] - A[4] * A[6]);
  if (!(fabs(det) > 1e-30) || !(fabs(det) < 1e300)) return cullFull();
  // columns of the inverse
  const double ea[3] = { (A[4] * A[8] - A[5] * A[7]) / det, -(A[3] * A[8] - A[5] * A[6]) / det, (A[3] * A[7] - A[4] * A[6]) / det };
  const double eb[3] = { -(A[1] * A[8] - A[2] * A[7]) / det, (A[0] * A[8] - A[2] * A[6]) / det, -(A[0] * A[7] - A[1] * A[6]) / det };
  const double nn[3] = { (A[1] * A[5] - A[2] * A[4]) / det, -(A[0] * A[5] - A[2] * A[3]) / det, (A[0] * A[4] - A[1] * A[3]) / det };
  const double v0[3] = { (double)tr.v0[0], (double)tr.v0[1], (double)tr.v0[2] };
  const double ev[3] = { eye[0] - v0[0], eye[1] - v0[1], eye[2] - v0[2] };
  const double la = sqrt(ea[0] * ea[0] + ea[1] * ea[1] + ea[2] * ea[2]), lb = sqrt(eb[0] * eb[0] + eb[1] * eb[1] + eb[2] * eb[2]);
  const double nl = sqrt(nn[0] * nn[0] + nn[1] * nn[1] + nn[2] * nn[2]);
  const double emin = la < lb ? la : lb;
  if (!(nl > 0.0) || !(emin > 0.0) || !(la < 1e300) || !(lb < 1e300) || !(nl < 1e300)) return cullFull();
  const double dist = fabs(nn[0] * ev[0] + nn[1] * ev[1] + nn[2] * ev[2]) / nl;     // lower bound of the distance from the eye to the triangle
  const double reach = sqrt(ev[0] * ev[0] + ev[1] * ev[1] + ev[2] * ev[2]) + la + lb;
  if (!(dist > 1e-6 * reach) || !(reach < 1e300)) return cullFull();
  const double mu = 1e-3 + 1e-5 * reach / emin;
  const double dx = (wHalf > W - wHalf ? wHalf : W - wHalf), dy = (hHalf > H - hHalf ? hHalf : H - hHalf);
  const double D = sqrt(dx * dx + dy * dy) + 8.0;
  const double znear = 0.5 * dist / sqrt(1.0 + (2.0 * D / rz) * (2.0 * D / rz));
  const double uv[3][2] = { { -mu, -mu }, { 1.0 + 2.0 * mu, -mu }, { -mu, 1.0 + 2.0 * mu } };
  double cam[3][3];
  for (int i = 0; i < 3; i++)
  {
    double p[3];
    for (int k = 0; k < 3; k++) p[k] = uv[i][0] * ea[k] + uv[i][1] * eb[k] - ev[k];     // point - eye
    cam[i][0] = c0[0] * p[0] + c0[1] * p[1] + c0[2] * p[2];
    cam[i][1] = c1[0] * p[0] + c1[1] * p[1] + c1[2] * p[2];
    cam[i][2] = c2[0] * p[0] + c2[1] * p[1] + c2[2] * p[2];
  }
  double x0 = 1e300, x1 = -1e300, y0 = 1e300, y1 = -1e300;
  int n = 0;
  auto take = [&](double px, double py, double pz)
  {
    const double sx = rz * px / pz + wHalf, sy = rz * py / pz + hHalf;
    x0 = sx < x0 ? sx : x0; x1 = sx > x1 ? sx : x1; y0 = sy < y0 ? sy : y0; y1 = sy > y1 ? sy : y1;
    n++;
  };
  for (int i = 0; i < 3; i++)
  {
    const double * a = cam[i], * b = cam[(i + 1) % 3];
    const bool ina = a[2] >= znear, inb = b[2] >= znear;
    if (ina) take(a[0], a[1], a[2]);
    if (ina != inb)
    {
      const double t = (znear - a[2]) / (b[2] - a[2]);
      take(a[0] + t * (b[0] - a[0]), a[1] + t * (b[1] - a[1]), znear);
    }
  }
  if (!n) return cullNone();
  if (!(x0 == x0) || !(x1 == x1) || !(y0 == y0) || !(y1 == y1)) return cullFull();
  return make_int4(cullClamp(floor(x0 - CULL_PIX_MARGIN)), cullClamp(ceil(x1 + CULL_PIX_MARGIN)), cullClamp(floor(y0 - CULL_PIX_MARGIN)), cullClamp(ceil(y1 + CULL_PIX_MARGIN)));
}

PrimaryCull makePrimaryCull(const SmallScene & sc, const FrameParams & fp)
{
  PrimaryCull pc;
  for (int i = 0; i < SMALL_MAX_SPHERES + SMALL_MAX_TRIS; i++) pc.rect[i] = cullFull();
  const PrimaryCamera cam = makePrimaryCamera(fp);
  if (!cam.ok) return pc;
  for (int i = 0; i < sc.nS && i < SMALL_MAX_SPHERES; i++) pc.rect[i] = sc.sph[i].x == sc.sph[i].x ? primarySphereBounds(cam, sc.sph[i]) : cullNone();   // NaN: padding
  for (int k = 0; k < sc.nT && k < SMALL_MAX_TRIS; k++)
    pc.rect[SMALL_MAX_SPHERES + k] = cullTriangle(cam.c[0], cam.c[1], cam.c[2], cam.eye, cam.rz, cam.wHalf, cam.hHalf, cam.W, cam.H, sc.tri[k]);
  return pc;
}

// ---- K2 ----------------------------------------------------------------------------------------------------------------

#ifdef RFX_CTA_TIMES
// debug build (tools/cta_times.py): start/end time and SM of every CTA of the last fast-kernel launch
__device__ unsigned long long g_ctaTimes[1 << 16][3];
extern "C" __attribute__((visibility("default"))) int rfx_debug_cta_times(unsigned long long * out, int n)
{
  return (int)cudaMemcpyFromSymbol(out, g_ctaTimes, sizeof(unsigned long long) * 3 * n);
}
__device__ __forceinline__ unsigned long long globalTimer() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
__device__ __forceinline__ unsigned smId() { unsigned s; asm volatile("mov.u32 %0, %smid;" : "=r"(s)); return s; }
#endif

// Fast kernel: a row-aligned slice (whole frame, band of rows, or this GPU's strips of a split frame).  2-D grid:
// blockIdx.y = tile row, blockIdx.x * warps + warp = tile column.  MULTI = false: one sample per pixel, no jitter, ARGB
// output only (the bench path).  MULTI = true: the same tiling and scheduling for grid SSAA (Render.cpp:174-196), additive
// jitter and accumulation, and the float image of the Render API.
//
// BATCH: nFrames frames of one camera (whole frames, one sample, ARGB).  Each lane runs its pixel's first segment once (SEG_FIRST,
// state in shared memory), then every frame from there with that frame's random state; frame f reads its states and writes its
// ARGB one frame further on (sampleStates / argbOut + f * W * rows).  The frames run one after the other for the whole warp, so
// that the bounce and shadow trips of a tile stay aligned; the tile's cost class is its longest path over all frames.
template <int FEAT, bool MULTI, bool STRIPS, bool BATCH = false>
__global__ void __launch_bounds__(SMALL_THREADS, MULTI ? 7 : RFX_SMALL_MINBLOCKS) k_trace_small(const __grid_constant__ SmallScene sc, const __grid_constant__ FrameParams fp,
                                                               const uint32_t * __restrict__ sampleStates, uint32_t * __restrict__ argbOut,
                                                               unsigned long long * __restrict__ counters, uint32_t y0, uint32_t y1,
                                                               const TileOrder ord, float * __restrict__ image, const __grid_constant__ PrimaryCull pc,
                                                               uint32_t nFrames)
{
  static_assert(!BATCH || (!MULTI && !STRIPS), "frame batches are whole one-sample frames");
  // which tile group does this CTA render: index order, or the previous launch's cost order (expensive classes first)
  uint32_t bx = blockIdx.x, by = blockIdx.y;
  if (ord.zeroCounts && (blockIdx.x | blockIdx.y) == 0u && threadIdx.x < TILE_CLASSES) ord.zeroCounts[threadIdx.x] = 0u;   // for the next launch
  if (!ord.inLists)
  {
    // no recording to replay (first launch over this grid): start the tile rows of the middle of the slice first and work outwards.
    // The subject of a picture tends to sit near its centre and the long paths with it; in plain index order they would start
    // in the middle of the launch and the last rows of sky would run against a long tail.
    const uint32_t mid = gridDim.y >> 1, b = blockIdx.y;
    by = (b & 1u) ? mid - 1u - (b >> 1) : mid + (b >> 1);      // even indices walk up from the middle row, odd ones down: a permutation
  }
  else
  {
    uint32_t total = 0;
#pragma unroll
    for (int c = 0; c < TILE_CLASSES; c++) total += ord.inCounts[c];
    if (total == gridDim.x * gridDim.y)      // the lists are a permutation of this grid (always, unless the recording launch failed)
    {
      uint32_t b = blockIdx.y * gridDim.x + blockIdx.x;
      int c = 0;
#pragma unroll
      for (; c < TILE_CLASSES - 1; c++)
      {
        const uint32_t n = ord.inCounts[c];
        if (b < n) break;
        b -= n;
      }
      const uint32_t packed = ord.inLists[(uint32_t)c * ord.capacity + b];
      bx = packed & 0xFFFFu; by = packed >> 16;
    }
  }
#ifdef RFX_CTA_TIMES
  const unsigned long long tStart = globalTimer();
#endif
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t xCta = bx * (SMALL_THREADS / 32) * RFX_TILE_W;          // the CTA's tile group: its warps' tiles side by side
  const uint32_t x = xCta + warp * RFX_TILE_W + (lane % RFX_TILE_W);
  uint32_t yTop = y0 + by * RFX_TILE_H;                                  // frame row of the group's first row
  if (STRIPS)
  {
    // split frame: the launch enumerates only this GPU's rows; compact row -> (own strip k, row in strip) -> frame row.  Strips
    // are multiples of the tile height, so the rows of a tile group lie in one strip
    const uint32_t k = yTop / fp.stripRows;
    yTop = (k * fp.stripWorld + fp.stripRank) * fp.stripRows + (yTop % fp.stripRows);
  }
  const uint32_t y = yTop + (lane / RFX_TILE_W);
  const bool valid = x < fp.W && y < y1;
  // which objects can the primary rays of this warp's tile hit: lane i asks for object i (spheres 0..15, triangles 16..23)
  ObjRange first;
  first.s0 = 0; first.s1 = 0; first.t0 = 0; first.t1 = 0;
  if (RFX_PRIMARY_CULL)
  {
    const int tx0 = (int)(xCta + warp * RFX_TILE_W), ty0 = (int)yTop;
    const int4 r = pc.rect[lane < SMALL_MAX_SPHERES + SMALL_MAX_TRIS ? lane : 0];
    const bool seen = lane < SMALL_MAX_SPHERES + SMALL_MAX_TRIS && tx0 + (int)RFX_TILE_W - 1 >= r.x && tx0 <= r.y && ty0 + (int)RFX_TILE_H - 1 >= r.z && ty0 <= r.w;
    const uint32_t m = __ballot_sync(0xffffffffu, seen);
    const uint32_t ms = m & ((1u << sc.nS) - 1u);
    const uint32_t mq = (ms | (ms >> 1) | (ms >> 2) | (ms >> 3)) & 0x1111u;   // bit 4q: quad q has a candidate
    if (mq) { first.s0 = (__ffs(mq) - 1) << 4; first.s1 = ((31 - __clz(mq)) << 4) + 64; }
    const uint32_t mt = (m >> SMALL_MAX_SPHERES) & ((1u << sc.nT) - 1u);
    if (mt) { first.t0 = (__ffs(mt) - 1) * 48; first.t1 = (32 - __clz(mt)) * 48; }
  }
  uint32_t events = 0;                                                   // of the longest call / frame in the low half (cost class)
  uint32_t nBounces = 0, nShadow = 0;                                    // totals over the calls / frames
  constexpr uint32_t GROUP_W = (SMALL_THREADS / 32) * RFX_TILE_W, STAGE_STRIDE = GROUP_W + 4;   // +4 words: conflict-free column writes
  __shared__ uint32_t sStage[(MULTI || !STRIPS) ? 1 : RFX_TILE_H * STAGE_STRIDE];
  __shared__ float sPath[BATCH ? PATH_WORDS * SMALL_THREADS : 1];
  const bool staged = RFX_STRIP_STAGING && !MULTI && STRIPS && xCta + GROUP_W <= fp.W && yTop + RFX_TILE_H <= y1;   // uniform over the CTA
  if (!MULTI)
  {
    const uint32_t q = y * fp.W + x;                                     // < 2^32 for every frame size the API accepts
    const size_t frameStride = (size_t)(y1 - y0) * fp.W;
#pragma unroll 1
    for (int f = BATCH ? -1 : 0; f < (BATCH ? (int)nFrames : 1); f++)   // BATCH: f = -1 is the first segment
    {
      ObjRange range = first;                                          // BATCH: every query of a frame sees every object
      if (BATCH && f >= 0) { range.s0 = 0; range.s1 = sc.nS << 4; range.t0 = 0; range.t1 = sc.nT * 48; }
      uint32_t packed = 0;
      if (valid)
      {
        V3 rd = mk(0.0f, 0.0f, 0.0f);                                    // (the first segment reads no randDir)
        if (f >= 0)
        {
          uint32_t s = __ldg(sampleStates + (size_t)f * frameStride + (q - y0 * fp.W));
          rngTriple(s, rd.x, rd.y, rd.z);
        }
        const float rx = float(x) - fp.wHalf;                            // Render.cpp:154-155
        const float ry = float(y) - fp.hHalf;
        const V3 ray = primaryRay(fp, rx, ry);
        uint32_t ev = 0, sig = 0;
        const V3 c = traceSmall<false, FEAT, RFX_PRIMARY_CULL != 0, BATCH>(sc, mk(fp.eye[0], fp.eye[1], fp.eye[2]), ray, fp.reflNum, rd, ev, sig,
                                                                         range,
                                                                         !BATCH ? SEG_WHOLE : f < 0 ? SEG_FIRST : SEG_RESUME, sPath + threadIdx.x);
#ifdef RFX_DEBUG_DEPTH
        packed = ev;               // debug build (tools/depth_stats.py): bounce-loop iterations | shadow rays << 16 instead of the colour
#else
        packed = packArgb(c.x, c.y, c.z);
#endif
        if (f >= 0)
        {
          nBounces += ev & 0xFFFFu; nShadow += ev >> 16;
          events = max(events, ev & 0xFFFFu);
        }
      }
      if (BATCH && f < 0) { __syncwarp(); continue; }                    // every lane of the tile starts frame 0 together
      // Framebuffer store of the one-sample path.
      //  * Frame in local HBM: one 128-bit store per tile row (storeTileRow).
      //  * Split frame (rfx_render_strips): argbOut may be ANOTHER GPU's framebuffer (peer mapping), and then every store
      //    instruction leaves this GPU as NVLink write packets.  Eight 16-byte pieces per instruction (one per tile row) throttled
      //    the 7-to-1 gather of an 8K frame to 0.70 ms against 0.48 ms with local stores (profiles/r2_s2), so a tile group that lies
      //    inside the image is staged in shared memory and written by whole row segments — warp w stores rows 2w and 2w+1, 16
      //    consecutive pixels (64 contiguous bytes) per half warp — after the CTA barrier the tile scheduler needs anyway.
      //    (For local frames the staging costs 0.8 % — measured — so they keep the direct stores: STRIPS is a template parameter and
      //    the whole-frame instantiations carry none of this.)
      if (staged) sStage[(lane / RFX_TILE_W) * STAGE_STRIDE + warp * RFX_TILE_W + (lane % RFX_TILE_W)] = packed;
      else storeTileRow(argbOut + (BATCH ? (size_t)f * frameStride : 0) + (valid ? q : 0u), packed, valid, fp.W, RFX_TILE_W);
    }
  }
  if (valid && MULTI)
  {
    const uint32_t q = y * fp.W + x;
    const uint32_t rel = q - y0 * fp.W;                                  // pixel index inside the slice
    const int sn = fp.sampleNum;
    float rndx = 0, rndy = 0;
    if (fp.jitter) pixelJitter(fp, rel, rndx, rndy);
    const V3 fin = samplePixel(fp, float(x) - fp.wHalf, float(y) - fp.hHalf, rndx, rndy, sn, false, sampleStates + (uint64_t)rel * (uint64_t)(sn * sn), true,
                               nBounces, nShadow, events, [&](V3 ray, V3 rd, uint32_t & ev) {
      uint32_t sig = 0;
      return traceSmall<false, FEAT, RFX_PRIMARY_CULL != 0>(sc, mk(fp.eye[0], fp.eye[1], fp.eye[2]), ray, fp.reflNum, rd, ev, sig, first);
    });
    if (image)
    {
      float * px = image + (uint64_t)q * 3;
      if (fp.accumulate) { px[0] = px[0] + fin.x; px[1] = px[1] + fin.y; px[2] = px[2] + fin.z; }
      else { px[0] = fin.x; px[1] = fin.y; px[2] = fin.z; }
    }
    if (argbOut) argbOut[q] = packArgb(fin.x, fin.y, fin.z);
  }
  // file this tile group under its cost class for the next launch: the longest path (bounce-loop iterations) of its pixels
  __shared__ uint32_t sLongest[SMALL_THREADS / 32];
  if (ord.outLists)
  {
    const uint32_t longest = __reduce_max_sync(0xffffffffu, events & 0xFFFFu);
    if (lane == 0) sLongest[warp] = longest;
  }
  if (staged || ord.outLists) __syncthreads();   // (the barrier and the atomic below cost 2.2 % of the kernel — measured — which is why the host
                                                 // only asks for a recording on every 8th launch over a grid)
  if (staged)
  {
    constexpr uint32_t ROWS_PER_WARP = RFX_TILE_H / (SMALL_THREADS / 32), LANES_PER_ROW = 32 / ROWS_PER_WARP;
    static_assert(MULTI || (RFX_TILE_H % (SMALL_THREADS / 32) == 0 && LANES_PER_ROW == GROUP_W), "staged store: one lane per pixel of the warp's rows");
    const uint32_t row = warp * ROWS_PER_WARP + lane / LANES_PER_ROW, col = lane % LANES_PER_ROW;
    argbOut[(yTop + row) * fp.W + xCta + col] = sStage[row * STAGE_STRIDE + col];
  }
  if (ord.outLists && threadIdx.x == 0)
  {
    uint32_t m = 0;
#pragma unroll
    for (int w = 0; w < SMALL_THREADS / 32; w++) m = max(m, sLongest[w]);
    const uint32_t bounds[TILE_CLASSES - 1] = RFX_TILE_BOUNDS;
    uint32_t cls = 0;
#pragma unroll
    for (int c = 0; c < TILE_CLASSES - 1; c++) cls += m < bounds[c] ? 1u : 0u;   // bounds descend: the count of bounds above m is the class
    const uint32_t idx = atomicAdd(&ord.outCounts[cls], 1u);
    if (idx < ord.capacity) ord.outLists[cls * ord.capacity + idx] = (by << 16) | bx;
  }
#ifdef RFX_CTA_TIMES
  __syncthreads();
  if (threadIdx.x == 0)
  {
    const unsigned id = by * gridDim.x + bx;
    if (id < (1u << 16)) { g_ctaTimes[id][0] = tStart; g_ctaTimes[id][1] = globalTimer(); g_ctaTimes[id][2] = smId(); }
  }
#endif
  flushCounters(counters, nBounces, nShadow, (blockIdx.y * gridDim.x + blockIdx.x) * (SMALL_THREADS / 32) + warp);
}

// General kernel: every mode of Render::renderNext (grid SSAA, block preview, additive jitter, arbitrary pixel slices,
// float image, signatures).
__global__ void __launch_bounds__(SMALL_THREADS, RFX_ANY_MINBLOCKS) k_trace_small_any(const __grid_constant__ SmallScene sc, const __grid_constant__ FrameParams fp,
                                                               const uint32_t * __restrict__ sampleStates, float * __restrict__ image,
                                                               uint32_t * __restrict__ argbOut, uint32_t * __restrict__ sigOut,
                                                               unsigned long long * __restrict__ counters, int tiled)
{
  const V3 eye = mk(fp.eye[0], fp.eye[1], fp.eye[2]);
  renderAny(fp, sampleStates, image, argbOut, sigOut, counters, tiled, RFX_TILE_W, SMALL_THREADS, [&](uint32_t, uint32_t) {
    return [&](V3 ray, V3 rd, uint32_t & events, uint32_t & sig) { return traceSmall<true, F_ALL>(sc, eye, ray, fp.reflNum, rd, events, sig); };
  });
}

// rows the fast kernel enumerates for this work (0 = does not qualify): whole rows, grid sampling (not block preview), no signatures
static uint64_t fastRows(const TraceWork & w)
{
  const FrameParams & fp = w.fp;
  if (fp.sampleNum < 1 || w.sigOut || (!w.argbOut && !w.image) || fp.W == 0) return 0;
  if ((uint64_t)fp.sampleNum * fp.sampleNum * (fp.p1 - fp.p0) >= (1ull << 32)) return 0;
  if (fp.p0 % fp.W != 0 || fp.p1 % fp.W != 0 || (uint64_t)fp.W * fp.H >= (1ull << 32)) return 0;
  // the 128-bit framebuffer stores need a 16-byte aligned frame (rows of a W % 4 == 0 image then stay aligned); a caller's
  // offset sub-buffer that is only 4-byte aligned takes the general kernel's scalar stores
  if (w.argbOut && (fp.W & 3u) == 0u && (reinterpret_cast<uintptr_t>(w.argbOut) & 15u) != 0u) return 0;
  const uint64_t rows = ownedRows(fp, (fp.p1 - fp.p0) / fp.W);
  if ((rows + RFX_TILE_H - 1) / RFX_TILE_H > 65535u) return 0;
  return rows;
}

static dim3 fastGrid3(const TraceWork & w, uint64_t rows)
{
  const uint32_t tilesX = (w.fp.W + RFX_TILE_W - 1) / RFX_TILE_W, warps = SMALL_THREADS / 32;
  return dim3((tilesX + warps - 1) / warps, (uint32_t)((rows + RFX_TILE_H - 1) / RFX_TILE_H));
}

uint32_t fastGridSize(const TraceWork & w)
{
  const uint64_t rows = fastRows(w);
  if (!rows) return 0;
  const dim3 g = fastGrid3(w, rows);
  return g.x <= 65535u ? g.x * g.y : 0;
}

bool fastBatchOk(const TraceWork & w)
{
  const FrameParams & fp = w.fp;
  return fastGridSize(w) && fp.sampleNum == 1 && !fp.jitter && !w.image && w.argbOut && !fp.stripWorld && fp.p0 == 0 && fp.p1 == (uint64_t)fp.W * fp.H;
}

int launchTraceSmall(const SmallScene & sc, const TraceWork & w, cudaStream_t st, uint32_t * fastGrid)
{
  if (fastGrid) *fastGrid = 0;
  const FrameParams & fp = w.fp;
  if (fastGridSize(w))
  {
    const dim3 grid = fastGrid3(w, fastRows(w));
    if (fastGrid) *fastGrid = grid.x * grid.y;
    // scene features decide the instantiation: texel-free, plane-free, single-light scenes run the lean one
    bool texels = false;
    for (int i = 0; i < SMALL_MAX_TEX; i++) texels = texels || sc.tex[i].px != nullptr;
    const bool lean = !texels && sc.nP == 0 && sc.nL <= 1;
    const bool multi = fp.sampleNum != 1 || fp.jitter || w.image != nullptr;
    const uint32_t y0 = (uint32_t)(fp.p0 / fp.W), y1 = (uint32_t)(fp.p1 / fp.W);
    const PrimaryCull pc = RFX_PRIMARY_CULL ? makePrimaryCull(sc, fp) : PrimaryCull();
    if (w.frames > 1)   // the caller checked fastBatchOk
      withFlag(lean, [&](auto L) {
        k_trace_small<decltype(L)::value ? 0 : F_ALL, false, false, true><<<grid, SMALL_THREADS, 0, st>>>(sc, fp, w.sampleStates, w.argbOut, w.counters, y0, y1, w.order, nullptr, pc, w.frames);
      });
    else
      withFlag(lean, [&](auto L) { withFlag(multi, [&](auto M) { withFlag(fp.stripWorld != 0, [&](auto S) {
        k_trace_small<decltype(L)::value ? 0 : F_ALL, decltype(M)::value, decltype(S)::value><<<grid, SMALL_THREADS, 0, st>>>(sc, fp, w.sampleStates, w.argbOut, w.counters, y0, y1,
                                                                                                    w.order, decltype(M)::value ? w.image : nullptr, pc, 1u);
      }); }); });
    return 1;
  }
  int tiled;
  const uint64_t nThreads = anyThreads(fp, RFX_TILE_W, tiled);
  if (nThreads == 0) return 0;
  const uint32_t blocks = (uint32_t)((nThreads + SMALL_THREADS - 1) / SMALL_THREADS);
  k_trace_small_any<<<blocks, SMALL_THREADS, 0, st>>>(sc, fp, w.sampleStates, w.image, w.argbOut, w.sigOut, w.counters, tiled);
  return 1;
}

} // namespace rfx
