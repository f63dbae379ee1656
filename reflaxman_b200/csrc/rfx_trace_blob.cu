// rfx_trace_blob.cu — K2 for scenes that do not fit the constant bank (config 4: 1024 spheres), every mode of Render::renderNext:
//   k_trace_blob<MULTI, GRIDS>             row-aligned slices, ARGB and/or float image; one sample per pixel or grid SSAA / additive jitter
//   k_blob_wave_first<GRIDS> + k_blob_wave_rest   one-sample ARGB frames of reflection depth >= 3 as a two-kernel wavefront (below)
//   k_trace_blob_any                       arbitrary pixel slices, block preview, signature runs
//   k_trace_blob_rays                      Scene::trace for an explicit ray list (rfx_trace_rays)
// All of them run ONE restatement of Scene::trace, traceBlob<SIG, MODE> (round 1 kept a second one, k_trace in rfx_kernels.cu, with two
// inlined traversals; it is gone).
//
// It is the structure of the constant-bank kernel (rfx_trace_small.cu) applied to the scene blob in global memory:
//   * Scene::trace as a per-lane state machine with ONE traversal site: the query in flight is the bounce segment (closest
//     hit) or the shadow ray of light li (any hit).
//   * The BVH over the spheres (built by rfx_scene.cpp, every box inflated beyond the rounding noise of the exact test) only
//     selects which spheres get the reference's exact test.  It is walked over PAIR NODES (both children's boxes in the parent,
//     four 16-byte loads per trip): the walk continues into the nearer hit child in a register and defers the other one to a
//     stack in shared memory (one column per thread); "while-while" order — every lane walks to its next leaf, then the warp
//     tests its leaves together.  A leaf is four contiguous sphere records (NaN-padded) tested behind one gate, like a quad of
//     the constant-bank kernel.  The slab test is the one piece of arithmetic here that is not the reference's, so it is fused.
//   * Shadow queries towards a FAR light do not walk the hierarchy: their rays are nearly parallel, so the host bins the spheres'
//     (inflated) shadows on a plane across the light's direction and the query tests the candidate list of its origin's cell with
//     the exact arithmetic (LightGrid, rfx_scene.cpp buildLightGrid) — an any-hit query only asks whether something is hit.
//   * Neither does the FIRST query of a path: every path starts at the eye, so the host bins the spheres' primary-ray screen bounds
//     into 32x32-pixel cells per camera (EyeGrid, buildEyeGrid) and the 32 lanes of a tile walk the same short list.
//     (Both lists go through the same branch of intersectBlob; the queue-driven kernel is compiled without it: traceBlob.)
//   * 4x8 pixel tiles per warp on a 2-D grid, 128-bit framebuffer stores, 64 registers / 8 CTAs per SM.
// Each step was measured (profiles/README.md: 6.66 -> 3.63 ms for a 3840x2160 frame of the 1024-sphere scene at depth 8, 1.19 -> 0.57 at depth 1).
//
// ARITHMETIC CONTRACT: as in rfx_trace_small.cu — --fmad=false, every + - * / sqrtf of the reference's arithmetic is the IEEE
// binary32 RN operation in the reference's evaluation order; the expressions below are the ones of rfx_trace_small.cu.
// Reference map (path:line under /root/reference/src/common): Sphere.cpp:44-85, Triangle.cpp:53-108, Plane.cpp:36-73,
// Scene.cpp:73-236, Render.cpp:136-215.
#include "rfx_kernels.h"
#include "rfx_device.cuh"

namespace rfx
{

namespace
{

#ifndef RFX_QUEUE_RESERVE
#define RFX_QUEUE_RESERVE 1  // queue-driven kernel: consecutive records a lane reserves per atomic (1 measured best: the lanes of a warp
#endif                       // then hold neighbouring paths; 4: +7 %, 8: +14 %; handing records out from a per-warp shared-memory
                             // buffer behind a __syncwarp per query: +11 % — profiles/r2_s6)
#ifndef RFX_BLOB_MINBLOCKS
#define RFX_BLOB_MINBLOCKS 8
#endif

#ifndef RFX_BLOB_TILE_W
#define RFX_BLOB_TILE_W 4     // pixel tile of a warp: 4 x 8 (a multiple of 4: one 128-bit framebuffer store per 4 lanes)
#endif

constexpr int BLOB_THREADS = 128;
constexpr uint32_t BLOB_TILE_W = RFX_BLOB_TILE_W, BLOB_TILE_H = 32 / RFX_BLOB_TILE_W;
constexpr int BLOB_STACK = 24;          // entries per thread; the host only routes BVHs of depth <= BLOB_STACK - 2 here

struct BlobView
{
  const SceneHeader * h;
  const Light * lights;
  const float4 * spheres;
  const Triangle * tris;
  const Plane * planes;
  const Material * mats;
  const TexRef * tex;
  const float4 * bvhLeaves;   // leaf sphere records (4 per leaf) and pair nodes (4 float4 per inner node): the global arrays of the
  const float4 * bvhPairs;    // header, or the CTA's shared-memory copy (kernels instantiated with SMEM); NULL: no hierarchy
};

__device__ __forceinline__ BlobView blobView(const unsigned char * base)
{
  BlobView v;
  v.h = reinterpret_cast<const SceneHeader *>(base);
  v.lights = reinterpret_cast<const Light *>(base + v.h->offLights);
  v.spheres = reinterpret_cast<const float4 *>(base + v.h->offSpheres);
  v.tris = reinterpret_cast<const Triangle *>(base + v.h->offTris);
  v.planes = reinterpret_cast<const Plane *>(base + v.h->offPlanes);
  v.mats = reinterpret_cast<const Material *>(base + v.h->offMats);
  v.tex = reinterpret_cast<const TexRef *>(base + v.h->offTex);
  v.bvhLeaves = v.h->bvhLeafSph;
  v.bvhPairs = v.h->bvhPairs;
  return v;
}

struct Hit
{
  float dist;
  int idx;           // position in the sorted object arrays (spheres, triangles, planes), -1 = none
  int order;         // insertion index (closest-hit tie-break, reference Scene.cpp:98)
  float t;
  float u, v;
};

__device__ __forceinline__ void consider(Hit & best, float dist, int idx, int order, float t, float u, float v)
{
  if (dist < best.dist || (dist == best.dist && order < best.order))
  {
    best.dist = dist; best.idx = idx; best.order = order; best.t = t; best.u = u; best.v = v;
  }
}

// The pair-node walk of a hierarchy (the spheres' and the triangles'), in the scope of intersectBlob: the slab-test terms ix, iy, iz,
// oxi, oyi, ozi, the pruning distance reachT (refreshed from best.dist after every leaf), invLen, the per-thread stack and STRIDE.
// SMEM_: the nodes are in shared memory; PAIRS / ROOT: nodes and root ref; LEAF(slot): the exact test of a leaf's slots;
// OPEN: false once an any-hit query has its occluder (the walk ends).
#define RFX_BLOB_WALK(SMEM_, PAIRS, ROOT, LEAF, OPEN)                                                                          \
  {                                                                                                                          \
    constexpr int DONE = (int)0x80000000;                                                                                    \
    const float4 * __restrict__ pn = (PAIRS);                                                                                \
    int cur = (ROOT);                                                                                                        \
    int sp = 1;                                                                                                              \
    stack[0] = DONE;                                                                                                         \
    _Pragma("unroll 1")                                                                                                      \
    while (cur != DONE)                                                                                                      \
    {                                                                                                                        \
      _Pragma("unroll 1")                                                                                                    \
      while (cur >= 0)                                                                                                       \
      {                                                                                                                      \
        const float4 * q = pn + 4 * cur;                                                                                     \
        const float4 n0 = SMEM_ ? q[0] : __ldg(q), n1 = SMEM_ ? q[1] : __ldg(q + 1), n2 = SMEM_ ? q[2] : __ldg(q + 2), n3 = SMEM_ ? q[3] : __ldg(q + 3); \
        const float ax1 = __fmaf_rn(n0.x, ix, oxi), ax2 = __fmaf_rn(n1.x, ix, oxi);                                          \
        const float ay1 = __fmaf_rn(n0.y, iy, oyi), ay2 = __fmaf_rn(n1.y, iy, oyi);                                          \
        const float az1 = __fmaf_rn(n0.z, iz, ozi), az2 = __fmaf_rn(n1.z, iz, ozi);                                          \
        const float bx1 = __fmaf_rn(n2.x, ix, oxi), bx2 = __fmaf_rn(n3.x, ix, oxi);                                          \
        const float by1 = __fmaf_rn(n2.y, iy, oyi), by2 = __fmaf_rn(n3.y, iy, oyi);                                          \
        const float bz1 = __fmaf_rn(n2.z, iz, ozi), bz2 = __fmaf_rn(n3.z, iz, ozi);                                          \
        const float tminA = fmaxf(fmaxf(fminf(ax1, ax2), fminf(ay1, ay2)), fmaxf(fminf(az1, az2), 0.0f));                    \
        const float tmaxA = fminf(fminf(fmaxf(ax1, ax2), fmaxf(ay1, ay2)), fmaxf(az1, az2));                                 \
        const float tminB = fmaxf(fmaxf(fminf(bx1, bx2), fminf(by1, by2)), fmaxf(fminf(bz1, bz2), 0.0f));                    \
        const float tmaxB = fminf(fminf(fmaxf(bx1, bx2), fmaxf(by1, by2)), fmaxf(bz1, bz2));                                 \
        const bool hitA = tminA <= tmaxA && !(tminA > reachT);                                                               \
        const bool hitB = tminB <= tmaxB && !(tminB > reachT);                                                               \
        int ra = __float_as_int(n0.w), rb = __float_as_int(n1.w);                                                            \
        if (hitA && hitB)                                                                                                    \
        {                                                                                                                    \
          if (tminB < tminA) { const int t = ra; ra = rb; rb = t; }                                                          \
          stack[sp * STRIDE] = rb; sp++;                                                                                     \
          cur = ra;                                                                                                          \
        }                                                                                                                    \
        else if (hitA) cur = ra;                                                                                             \
        else if (hitB) cur = rb;                                                                                             \
        else cur = stack[(--sp) * STRIDE];                                                                                   \
      }                                                                                                                      \
      if (cur == DONE) break;                                                                                                \
      LEAF(~cur)                                                                                                             \
      reachT = (best.dist * 1.001f + 1e-2f) * invLen;                                                                        \
      cur = (OPEN) ? stack[(--sp) * STRIDE] : DONE;                                                                          \
    }                                                                                                                        \
  }

// All objects against one ray; `skip` = object the query ignores (-1 none); anyHit = shadow query (stop at the first hit).
// STRIDE: threads of the CTA (the traversal stack is one column per thread).  SMEM: bvh points at the CTA's shared-memory copy of
// the hierarchy (leaf sphere records, then pair nodes), else at the global arrays (read-only path).
// grid: the candidate grid of the light this (shadow) query runs towards, NULL for bounce queries and for lights that have none.
// GRIDS = false compiles the candidate-list branch out (the queue-driven kernel, see traceBlob).
// TRIS: the scene has a hierarchy over its triangles (h.triPairs) and the triangles are walked through it instead of one by one;
// the host picks the instantiation by scene, so the kernels of scenes without one are compiled as before.
template <int STRIDE, bool SMEM, bool GRIDS, bool TRIS = false>
__device__ __forceinline__ void intersectBlob(const BlobView & sc, int * __restrict__ stack, V3 o, V3 d, int skip, bool anyHit, Hit & best,
                                              const uint32_t * __restrict__ cellStart, const float4 * __restrict__ itemSphere,
                                              const int * __restrict__ itemIndex, int cell)
{
  const SceneHeader & h = *sc.h;
  const float a = vsqlen(d);                                          // Sphere.cpp:50
  const float r2x = d.x * 2.0f, r2y = d.y * 2.0f, r2z = d.z * 2.0f;   // 2.0f * ray, Sphere.cpp:51
  const float a2 = 2.0f * a;                                          // Sphere.cpp:57
  // a lane that must not take any (more) sphere hit carries NaN instead of 4a (see rfx_trace_small.cu)
  float a4 = (a > RFX_VSN) ? 4.0f * a : __int_as_float(0x7FC00000);  // Sphere.cpp:53,55
  bool open = true;                                                   // false: an any-hit query that has its occluder

  // exact sphere test (Sphere.cpp:44-85) in two halves: REJECT computes b and the discriminant, TAIL (behind the gate
  // disc >= 0 && b < 0; b < 0 is implied by t > 2^-63) the root, the distance and the bookkeeping
#define RFX_BLOB_REJECT(S, B, DISC)                                                          \
  float B, DISC;                                                                             \
  {                                                                                          \
    const float vx = o.x - S.x, vy = o.y - S.y, vz = o.z - S.z;                              \
    B = (r2x * vx + r2y * vy) + r2z * vz;                                                    \
    const float c = ((vx * vx + vy * vy) + vz * vz) - S.w;                                   \
    DISC = B * B - a4 * c;                                                                   \
  }
#define RFX_BLOB_GATE(B, DISC) ((DISC) >= 0.0f && (B) < 0.0f)
#define RFX_BLOB_TAIL(IDX, B, DISC)                                                          \
  {                                                                                          \
    const float t = (-B - sqrtf(DISC)) / a2;                          /* Sphere.cpp:57 */    \
    if (t > RFX_VSN)                                                                         \
    {                                                                                        \
      const float fx = d.x * t, fy = d.y * t, fz = d.z * t;                                  \
      const float dist = sqrtf((fx * fx + fy * fy) + fz * fz);        /* Sphere.cpp:62 */    \
      if (dist > RFX_DELTA)                                                                  \
      {                                                                                      \
        const int si = (IDX);                                                                \
        if (si != skip)                                                                      \
        {                                                                                    \
          consider(best, dist, si, sc.mats[si].order, t, 0.0f, 0.0f);                        \
          if (anyHit) { a4 = __int_as_float(0x7FC00000); open = false; }                     \
        }                                                                                    \
      }                                                                                      \
    }                                                                                        \
  }
  // one leaf = 4 contiguous sphere records (NaN in unused slots: the gate stays shut), tested behind one gate region
#define RFX_BLOB_LEAF(CA)                                                                    \
  {                                                                                          \
    const float4 * ls = sc.bvhLeaves + (CA);                                                  \
    const float4 s0 = SMEM ? ls[0] : __ldg(ls), s1 = SMEM ? ls[1] : __ldg(ls + 1), s2 = SMEM ? ls[2] : __ldg(ls + 2), s3 = SMEM ? ls[3] : __ldg(ls + 3); \
    RFX_BLOB_REJECT(s0, b0, disc0)                                                           \
    RFX_BLOB_REJECT(s1, b1, disc1)                                                           \
    RFX_BLOB_REJECT(s2, b2, disc2)                                                           \
    RFX_BLOB_REJECT(s3, b3, disc3)                                                           \
    const bool g0 = RFX_BLOB_GATE(b0, disc0), g1 = RFX_BLOB_GATE(b1, disc1), g2 = RFX_BLOB_GATE(b2, disc2), g3 = RFX_BLOB_GATE(b3, disc3); \
    if (g0 | g1 | g2 | g3)                                                                   \
    {                                                                                        \
      if (g0) RFX_BLOB_TAIL(__ldg(&h.bvhPrims[(CA)]), b0, disc0)                             \
      if (g1 && a4 == a4) RFX_BLOB_TAIL(__ldg(&h.bvhPrims[(CA) + 1]), b1, disc1)             \
      if (g2 && a4 == a4) RFX_BLOB_TAIL(__ldg(&h.bvhPrims[(CA) + 2]), b2, disc2)             \
      if (g3 && a4 == a4) RFX_BLOB_TAIL(__ldg(&h.bvhPrims[(CA) + 3]), b3, disc3)             \
    }                                                                                        \
  }

  if (sc.bvhPairs == nullptr)
  {
#pragma unroll 1
    for (int i = 0; i < h.nSpheres; i++)
    {
      const float4 s = __ldg(&sc.spheres[i]);
      RFX_BLOB_REJECT(s, b, disc)
      if (RFX_BLOB_GATE(b, disc)) RFX_BLOB_TAIL(i, b, disc)
    }
  }
  else if (GRIDS && cellStart != nullptr)
  {
    // The query comes with a candidate list — cell `cell` of a grid the host built (traceBlob says which) — that holds every
    // sphere this ray can hit: the exact test over that list gives the hierarchy walk's answer.  cell < 0: no sphere can be hit.
    if (cell >= 0)
    {
      uint32_t k = __ldg(cellStart + cell);
      const uint32_t e = __ldg(cellStart + cell + 1);
#pragma unroll 1
      for (; k < e && open; k++)
      {
        const float4 s = __ldg(itemSphere + k);
        RFX_BLOB_REJECT(s, b, disc)
        if (RFX_BLOB_GATE(b, disc)) RFX_BLOB_TAIL(__ldg(itemIndex + k), b, disc)
      }
    }
  }
  else
  {
    // Slab test.  The hierarchy only selects candidates for the exact test and its boxes carry margins (rfx_scene.cpp), so — unlike
    // everything the reference computes — this arithmetic may be fused: t = box * (1/d) - origin * (1/d) is one FFMA per plane
    // instead of a subtraction and a multiplication.  Its error moves a box plane by at most 2^-22 |origin| along the axis, which
    // the margins' 1e-6 * R term covers.  The reciprocals are clamped to +-1e30 so that an axis-parallel ray (1/0 = inf) gives
    // large finite distances of the right sign instead of inf - inf.
    const float ix = fminf(fmaxf(1.0f / d.x, -1e30f), 1e30f), iy = fminf(fmaxf(1.0f / d.y, -1e30f), 1e30f), iz = fminf(fmaxf(1.0f / d.z, -1e30f), 1e30f);
    const float oxi = -(o.x * ix), oyi = -(o.y * iy), ozi = -(o.z * iz);
    // a box whose entry lies beyond the closest hit so far cannot improve it: compared in ray-parameter space, with generous slack
    // (0.1 % + 0.01 length units; +inf while there is no hit and in any-hit queries); refreshed after every leaf.  |d|^2 overflows
    // for |d| > ~1.8e19: 1/sqrtf(inf) = 0 would make reachT 0 after the first hit and prune every box ahead, so such rays prune nothing
    const float invLen = (a < FLT_MAX) ? 1.0f / sqrtf(a) : __int_as_float(0x7F800000);
    float reachT = (best.dist * 1.001f + 1e-2f) * invLen;
    // pair nodes: one trip tests both children of an inner node; the walk continues into a hit child in a register (the nearer
    // one) and only defers the other to the stack; "while-while": every lane walks to its next leaf, then the warp tests its
    // leaves together.  The bottom stack entry is the end marker.  (Single-box nodes, if-if order and far-child-first were
    // measured slower: profiles/README.md.)
    RFX_BLOB_WALK(SMEM, sc.bvhPairs, h.bvhRoot, RFX_BLOB_LEAF, open)
  }
#undef RFX_BLOB_LEAF
#undef RFX_BLOB_TAIL
#undef RFX_BLOB_GATE
#undef RFX_BLOB_REJECT

  // ---- triangles (Triangle.cpp:53-108): third matrix row first; t = -oz/rz > 2^-63 needs oz, rz nonzero of opposite sign
  const float rzMin = open ? RFX_VSN : __int_as_float(0x7F800000);
  bool openT = open;
  // the exact test of the list walk below (same operations in the same order) for one leaf slot of the hierarchy; the slot's
  // position K in the sorted triangle array is read behind the gate, so the skip test comes after it
#define RFX_BLOB_TRI(K, V0X, V0Y, V0Z, A0, A1, A2, A3, A4, A5, A6, A7, A8)                                     \
  {                                                                                                            \
    const float px = o.x - (V0X), py = o.y - (V0Y), pz = o.z - (V0Z);                                          \
    const float oz = (px * (A6) + py * (A7)) + pz * (A8);                                                      \
    const float rz = (d.x * (A6) + d.y * (A7)) + d.z * (A8);                                                   \
    if ((__float_as_int(oz) ^ __float_as_int(rz)) < 0 && fabsf(rz) > rzMin && fabsf(oz) > 0.0f && openT)      \
    {                                                                                                          \
      const int ti = h.nSpheres + (K);                                                                         \
      const float t = -oz / rz;                                       /* Triangle.cpp:61 */                    \
      if (t > RFX_VSN && ti != skip)                                                                           \
      {                                                                                                        \
        const float ox = (px * (A0) + py * (A1)) + pz * (A2);                                                  \
        const float rx = (d.x * (A0) + d.y * (A1)) + d.z * (A2);                                               \
        const float oy = (px * (A3) + py * (A4)) + pz * (A5);                                                  \
        const float ry = (d.x * (A3) + d.y * (A4)) + d.z * (A5);                                               \
        const float u = ox + t * rx;                                  /* Triangle.cpp:65-66 */                 \
        const float v = oy + t * ry;                                                                           \
        if (u >= 0.0f && v >= 0.0f && u + v < 1.0f)                                                           \
        {                                                                                                      \
          const float fx = d.x * t, fy = d.y * t, fz = d.z * t;                                                \
          const float sq = (fx * fx + fy * fy) + fz * fz;                                                      \
          if (sq > RFX_DELTA * RFX_DELTA)                                                                      \
          {                                                                                                    \
            consider(best, sqrtf(sq), ti, sc.mats[ti].order, t, u, v);                                         \
            if (anyHit) openT = false;                                                                         \
          }                                                                                                    \
        }                                                                                                      \
      }                                                                                                        \
    }                                                                                                          \
  }
  if (TRIS && h.triPairs != nullptr)
  {
    // The hierarchy over the triangles (rfx_scene.cpp buildTriBoxes: every box holds every point the exact test below can accept,
    // with margin) selects which triangles get that test, as the sphere hierarchy does.  A leaf is 4 slots of 3 float4 (unused
    // slots have a zero third row: the gate stays shut); the slot's position in the sorted triangle array is read only behind the
    // gate.  The stack is free again (the sphere walk has ended); a sphere hit already prunes the boxes behind it.
    if (openT)
    {
      const float ix = fminf(fmaxf(1.0f / d.x, -1e30f), 1e30f), iy = fminf(fmaxf(1.0f / d.y, -1e30f), 1e30f), iz = fminf(fmaxf(1.0f / d.z, -1e30f), 1e30f);
      const float oxi = -(o.x * ix), oyi = -(o.y * iy), ozi = -(o.z * iz);
      const float invLen = (a < FLT_MAX) ? 1.0f / sqrtf(a) : __int_as_float(0x7F800000);   // as in the sphere walk
      float reachT = (best.dist * 1.001f + 1e-2f) * invLen;
#define RFX_TRI_LEAF(CA)                                                                                       \
      {                                                                                                        \
        _Pragma("unroll 1")                                                                                    \
        for (int j = (CA); j < (CA) + 4; j++)                                                                  \
        {                                                                                                      \
          const float4 * lt = h.triLeaf + 3 * j;                                                               \
          const float4 q0 = __ldg(lt), q1 = __ldg(lt + 1), q2 = __ldg(lt + 2);                                 \
          RFX_BLOB_TRI(__ldg(h.triPrims + j), q0.x, q0.y, q0.z, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w, q0.w, q1.x, q1.y) \
        }                                                                                                      \
      }
      RFX_BLOB_WALK(false, h.triPairs, h.triRoot, RFX_TRI_LEAF, openT)
#undef RFX_TRI_LEAF
    }
  }
  else
  {
#pragma unroll 1
    for (int k = 0; k < h.nTris; k++)
    {
      const int ti = h.nSpheres + k;
      const Triangle & tr = sc.tris[k];
      const float px = o.x - tr.v0[0], py = o.y - tr.v0[1], pz = o.z - tr.v0[2];
      const float oz = (px * tr.ax[6] + py * tr.ax[7]) + pz * tr.ax[8];
      const float rz = (d.x * tr.ax[6] + d.y * tr.ax[7]) + d.z * tr.ax[8];
      if ((__float_as_int(oz) ^ __float_as_int(rz)) < 0 && fabsf(rz) > rzMin && fabsf(oz) > 0.0f && ti != skip && openT)
      {
        const float t = -oz / rz;                                       // Triangle.cpp:61
        if (t > RFX_VSN)
        {
          const float ox = (px * tr.ax[0] + py * tr.ax[1]) + pz * tr.ax[2];
          const float rx = (d.x * tr.ax[0] + d.y * tr.ax[1]) + d.z * tr.ax[2];
          const float oy = (px * tr.ax[3] + py * tr.ax[4]) + pz * tr.ax[5];
          const float ry = (d.x * tr.ax[3] + d.y * tr.ax[4]) + d.z * tr.ax[5];
          const float u = ox + t * rx;                                  // Triangle.cpp:65-66
          const float v = oy + t * ry;
          if (u >= 0.0f && v >= 0.0f && u + v < 1.0f)
          {
            const float fx = d.x * t, fy = d.y * t, fz = d.z * t;
            const float sq = (fx * fx + fy * fy) + fz * fz;
            if (sq > RFX_DELTA * RFX_DELTA)
            {
              consider(best, sqrtf(sq), ti, sc.mats[ti].order, t, u, v);
              if (anyHit) openT = false;
            }
          }
        }
      }
    }
  }
#undef RFX_BLOB_TRI

  // ---- planes (Plane.cpp:36-73)
#pragma unroll 1
  for (int k = 0; k < h.nPlanes; k++)
  {
    const int pi = h.nSpheres + h.nTris + k;
    if (pi == skip || !openT) continue;
    const Plane & pl = sc.planes[k];
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
        if (sq > RFX_DELTA * RFX_DELTA) consider(best, sqrtf(sq), pi, sc.mats[pi].order, t, 0.0f, 0.0f);
      }
    }
  }
}

// ---- the path queue of the wavefront kernels (see k_blob_wave_first / k_blob_wave_rest) -----------------------------------
// One record per path that survives its first segment: 64 bytes = four 16-byte words, written and read with 128-bit accesses.
//   [0] origin.xyz, ray.x   [1] ray.yz, mulColor.xy   [2] mulColor.z, pixelColor.xyz   [3] pixel index in the slice, events, random state, -
// (randDir is regenerated from the path's ranked random state: 3 LCG steps instead of 8 more bytes)
struct PathQueue
{
  uint4 * records;                  // [capacity]
  uint32_t * count;                 // records pushed by the first-segment kernel
  uint32_t * cursor;                // next record the second kernel hands out
};

// What feeds a lane of the queue-driven machine (MODE_QUEUE) and receives its finished paths
struct QueueFeed
{
  const uint4 * records;
  const uint32_t * count;
  uint32_t * cursor;
  uint32_t * argbOut;               // first pixel of the slice
  uint32_t bufNext, bufCount;       // records this lane has reserved: [bufNext, bufCount)
  uint32_t doneBounces, doneShadow; // event totals of the paths this lane finished
};

constexpr int MODE_PATH = 0;        // one path from its first segment to its end (Scene::trace)
constexpr int MODE_FIRST = 1;       // the first `firstSegments` segments only (closest hit, its shadow queries, shading): returns false when the path goes on
constexpr int MODE_QUEUE = 2;       // paths come from the queue; a lane whose path ends takes the next record at once

// Scene::trace (Scene.cpp:73-236) as a per-lane state machine with ONE intersection site: the query in flight is the bounce
// segment (closest hit) or the shadow ray of light li (any hit); see traceSmall in rfx_trace_small.cu, whose expressions these are.
// (qo, qd) in: origin and ray of the path's next segment; mul, pix, events: Scene::trace's mulColor, pixelColor and the event
// counter (bounce-loop iterations in the low half, shadow rays in the high half).  Returns true when the path has ended (pix is
// final); MODE_FIRST returns false with (qo, qd, mul, pix, events) ready for the next segment.
// Candidate grids (GRIDS): the tile kernels' lanes alternate bounce and shadow queries together, so a shadow trip is a short list
// walk for the whole warp (-12..16 % on the first two segments of config 4).  The queue-driven kernel's lanes are in both kinds of
// query on every trip: a shadow lane rides along in the hierarchy walk of its warp's bounce lanes for free, and the list walk
// would be added to the trip (+6 % measured; making the warp run its shadow lanes first and its bounce lanes together recovers
// only part of it) — that kernel keeps walking the hierarchy for every query.  profiles/r2_grid has the measurements.
// Kernels that serve the batch path are instantiated both ways and the host picks by scene, because the grid branch costs a scene
// without far lights 4-5 % although it is never taken (registers across the walk).
template <bool SIG, int MODE, int STRIDE = BLOB_THREADS, bool SMEM = false, bool GRIDS = (MODE != MODE_QUEUE), bool TRIS = false>
__device__ __forceinline__ bool traceBlob(const BlobView & sc, int * __restrict__ stack, V3 & qo, V3 & qd, int reflNumber, V3 randDir,
                                          V3 & mul, V3 & pix, uint32_t & events, uint32_t & sig, QueueFeed * feed = nullptr, int firstSegments = 1,
                                          const EyeGrid * eyeGrid = nullptr, int eyeCell = -1)   // candidates of the first query (origin = eye), or NULL
{
  const SceneHeader & h = *sc.h;
  if (reflNumber <= 0) return true;

  bool shadowQuery = false;
  int li = 0, hidx = -1;
  V3 norm = qd, reflect = qd, color = mul, sumLight = pix, sumSpec = pix;
  float normLen = 0.0f, reflectLen = 0.0f, mrefl = 0.0f;
  float rfs = 0.0f;          // continuation weight (Scene.cpp:196 / :207), negated for metals
  uint32_t rel = 0;          // MODE_QUEUE: pixel of the path in flight
  bool idle = MODE == MODE_QUEUE;

  for (;;)
  {
    if (MODE == MODE_QUEUE && idle)
    {
      // This lane's path has ended: take the next record.  A lane reserves RFX_QUEUE_RESERVE consecutive records at a time, and the
      // idle lanes that arrive here together share one atomic.  Nothing forces the warp to reconverge here: lanes in short
      // queries may loop ahead of lanes deep in a traversal (forcing them together with a __syncwarp per trip cost 19 %).
      const uint32_t lane = threadIdx.x & 31u;
      if (feed->bufNext == feed->bufCount)
      {
        const uint32_t act = __activemask();
        const uint32_t need = __ballot_sync(act, true);
        const int leader = __ffs(need) - 1;
        uint32_t base = 0;
        if ((int)lane == leader) base = atomicAdd(feed->cursor, (uint32_t)__popc(need) * RFX_QUEUE_RESERVE);
        base = __shfl_sync(need, base, leader);
        feed->bufNext = base + (uint32_t)__popc(need & ((1u << lane) - 1u)) * RFX_QUEUE_RESERVE;
        feed->bufCount = feed->bufNext + RFX_QUEUE_RESERVE;
      }
      const uint32_t idx = feed->bufNext++;
      if (idx >= *feed->count) break;                                      // queue exhausted: this lane retires
      const uint4 * r = feed->records + 4 * (size_t)idx;
      const uint4 r0 = r[0], r1 = r[1], r2 = r[2], r3 = r[3];
      if (RFX_QUEUE_RESERVE > 1 && feed->bufNext != feed->bufCount) asm volatile("prefetch.global.L2 [%0];" :: "l"(r + 4));
      qo = mk(__uint_as_float(r0.x), __uint_as_float(r0.y), __uint_as_float(r0.z));
      qd = mk(__uint_as_float(r0.w), __uint_as_float(r1.x), __uint_as_float(r1.y));
      mul = mk(__uint_as_float(r1.z), __uint_as_float(r1.w), __uint_as_float(r2.x));
      pix = mk(__uint_as_float(r2.y), __uint_as_float(r2.z), __uint_as_float(r2.w));
      rel = r3.x; events = r3.y;
      uint32_t st = r3.z;
      rngTriple(st, randDir.x, randDir.y, randDir.z);
      shadowQuery = false;
      idle = false;
    }
    Hit hit;
    hit.dist = FLT_MAX; hit.idx = -1; hit.order = 0x7FFFFFFF; hit.t = 0; hit.u = 0; hit.v = 0;
    // Candidate lists.  A shadow query towards a far light: the cell of its origin in the light's grid (rfx_scene.cpp, buildLightGrid;
    // an origin outside the grid lies outside every sphere's inflated shadow).  The first query of a path: the screen cell of its
    // pixel in the camera's grid (buildEyeGrid).  Everything else walks the hierarchy.
    const uint32_t * cellStart = nullptr;
    const float4 * itemSphere = nullptr;
    const int * itemIndex = nullptr;
    int cell = -1;
    if (GRIDS && shadowQuery)
    {
      if (h.lightGrids != nullptr)
      {
        const LightGrid * grid = h.lightGrids + li;
        if (grid->cellStart != nullptr)
        {
          const float fu = __fmaf_rn(grid->u[0], qo.x, __fmaf_rn(grid->u[1], qo.y, __fmaf_rn(grid->u[2], qo.z, grid->u[3])));
          const float fv = __fmaf_rn(grid->v[0], qo.x, __fmaf_rn(grid->v[1], qo.y, __fmaf_rn(grid->v[2], qo.z, grid->v[3])));
          const int cu = __float2int_rd(fu), cv = __float2int_rd(fv);
          const int nx = grid->nx;
          cellStart = grid->cellStart; itemSphere = grid->itemSphere; itemIndex = grid->itemIndex;
          if ((unsigned)cu < (unsigned)nx && (unsigned)cv < (unsigned)grid->ny) cell = cv * nx + cu;
        }
      }
    }
    else if (GRIDS && MODE != MODE_QUEUE && eyeGrid != nullptr && events == 0u)
    {
      cellStart = eyeGrid->cellStart; itemSphere = eyeGrid->itemSphere; itemIndex = eyeGrid->itemIndex;
      cell = eyeCell;
    }
    intersectBlob<STRIDE, SMEM, GRIDS, TRIS>(sc, stack, qo, qd, shadowQuery ? hidx : -1, shadowQuery, hit, cellStart, itemSphere, itemIndex, cell);

    bool ended = false;
    if (!shadowQuery)
    {
      // ---- closest hit of the bounce segment, Scene.cpp:80-112
      events++;
      if (hit.idx < 0)
      {
        if (SIG) RFX_SIG(sig, 0xFFFF);
        float u, v;
        skyDirToUv(qd, vlen(qd), h.halfTileW, h.halfTileH, u, v);
        const V3 sky = texSampleRef(h.skyTex >= 0 ? &sc.tex[h.skyTex] : nullptr, h.byteLut, u, v);
        pix = mk(clamp01(pix.x + (mul.x * sky.x) * h.env[0]), clamp01(pix.y + (mul.y * sky.y) * h.env[1]),
                 clamp01(pix.z + (mul.z * sky.z) * h.env[2]));            // Scene.cpp:230-231
        ended = true;
      }
      else
      {
        if (SIG) RFX_SIG(sig, hit.order + 1);
        const V3 full = vscale(qd, hit.t);
        qo = vadd(qo, full);                                               // drop point
        const Material m = sc.mats[hit.idx];
        color = mk(m.r, m.g, m.b);
        mrefl = m.reflectivity;
        const bool dielectric = m.type == 1;
        hidx = hit.idx;
        if (hit.idx < h.nSpheres)
        {
          const float4 s = __ldg(&sc.spheres[hit.idx]);
          norm = mk(qo.x - s.x, qo.y - s.y, qo.z - s.z);                   // Sphere.cpp:67
        }
        else if (hit.idx < h.nSpheres + h.nTris)
        {
          const Triangle & tr = sc.tris[hit.idx - h.nSpheres];
          norm = mk(tr.n[0], tr.n[1], tr.n[2]);
          if (m.tex >= 0)
          {
            // tuvTrans * Vector3(u, v, 0): (u*_11 + v*_12) + 0*_13 with _13 == 0, Triangle.cpp:91
            const float tx = (hit.u * tr.tuv[0] + hit.v * tr.tuv[1]) + 0.0f;
            const float ty = (hit.u * tr.tuv[2] + hit.v * tr.tuv[3]) + 0.0f;
            color = texSampleRef(&sc.tex[m.tex], h.byteLut, tr.tu0 + tx, tr.tv0 + ty);
          }
        }
        else
        {
          const Plane & pl = sc.planes[hit.idx - h.nSpheres - h.nTris];
          norm = mk(pl.n[0], pl.n[1], pl.n[2]);
        }
        reflect = reflectVec(full, norm);
        normLen = vlen(norm);
        reflectLen = vlen(reflect);
        rfs = -0.8f;                                                       // metal, Scene.cpp:207
        if (dielectric)                                                    // Scene.cpp:192-196
        {
          const float a = vlen(qd) * normLen;
          const float cosA = (a > RFX_VSN) ? clamp01(((qd.x * -norm.x + qd.y * -norm.y) + qd.z * -norm.z) / a) : 0.0f;
          rfs = 0.2f + 0.8f * cubeLikePowf(1.0f - cosA);
        }
        sumLight = mk(0.0f, 0.0f, 0.0f);
        sumSpec = mk(0.0f, 0.0f, 0.0f);
        li = 0;
      }
    }
    else
    {
      // ---- answer of the shadow query for light li, Scene.cpp:125-186
      const Light L = sc.lights[li];
      if (SIG) RFX_SIG(sig, 0x100 + 2 * li + (hit.idx >= 0 ? 1 : 0));
      if (hit.idx < 0)
      {
        const V3 toLight = mk(L.ox - qo.x, L.oy - qo.y, L.oz - qo.z);
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

    if (!ended)
    {
      // ---- next light that faces the surface gets a shadow query, Scene.cpp:118-129
      bool cast = false;
      for (; li < h.nLights; li++)
      {
        const Light L = sc.lights[li];
        const V3 toLight = mk(L.ox - qo.x, L.oy - qo.y, L.oz - qo.z);
        if (vdot(toLight, norm) > RFX_VSN)
        {
          qd = vadd(toLight, vscale(randDir, L.radius));                  // Scene.cpp:129
          cast = true;
          break;
        }
      }
      if (cast)
      {
        shadowQuery = true;
        events += 0x10000u;
        continue;
      }

      // ---- all lights answered: finish the hit, Scene.cpp:189-226
      sumLight = mk(h.ambient[0] * h.ambientPower + sumLight.x, h.ambient[1] * h.ambientPower + sumLight.y,
                    h.ambient[2] * h.ambientPower + sumLight.z);         // Scene.cpp:189
      const bool dielectric = rfs > 0.0f;
      const float rf = fabsf(rfs);
      const float k = 1.0f - rf;
      const V3 fin = mk(((color.x * k) * sumLight.x + sumSpec.x) * mul.x, ((color.y * k) * sumLight.y + sumSpec.y) * mul.y,
                        ((color.z * k) * sumLight.z + sumSpec.z) * mul.z); // Scene.cpp:198-199 / 209-210
      if (dielectric) mul = vscale(mul, rf);                             // Scene.cpp:202
      else mul = mk(mul.x * (color.x * rf), mul.y * (color.y * rf), mul.z * (color.z * rf));   // Scene.cpp:213

      pix = mk(clamp01(pix.x + fin.x), clamp01(pix.y + fin.y), clamp01(pix.z + fin.z));

      ended = (mul.x < 0.01f && mul.y < 0.01f && mul.z < 0.01f) ||
              (int)(events & 0xFFFFu) >= reflNumber;                     // ++refl < reflNumber, Scene.cpp:80
      if (!ended)
      {
        const V3 rn = (reflectLen > RFX_VSN) ? mk(reflect.x / reflectLen, reflect.y / reflectLen, reflect.z / reflectLen) : reflect;
        qd = vadd(rn, vscale(randDir, 1.0f - mrefl));                    // Scene.cpp:226
        shadowQuery = false;
        if (MODE == MODE_FIRST && (int)(events & 0xFFFFu) >= firstSegments) return false;
        continue;
      }
    }

    // ---- the path has ended
    if (MODE != MODE_QUEUE) return true;
    feed->argbOut[rel] = packArgb(pix.x, pix.y, pix.z);
    feed->doneBounces += events & 0xFFFFu;
    feed->doneShadow += events >> 16;
    idle = true;
  }
  return true;
}

// one whole Scene::trace call
template <bool SIG, bool GRIDS = true, bool TRIS = false>
__device__ __forceinline__ V3 tracePath(const BlobView & sc, int * __restrict__ stack, V3 origin, V3 ray, int reflNumber, V3 randDir, uint32_t & events, uint32_t & sig,
                                        const EyeGrid * eyeGrid = nullptr, int eyeCell = -1)
{
  V3 qo = origin, qd = ray, mul = mk(1.0f, 1.0f, 1.0f), pix = mk(0.0f, 0.0f, 0.0f);
  events = 0;
  traceBlob<SIG, MODE_PATH, BLOB_THREADS, false, GRIDS, TRIS>(sc, stack, qo, qd, reflNumber, randDir, mul, pix, events, sig, nullptr, 1, eyeGrid, eyeCell);
  return pix;
}

__device__ __forceinline__ void flushBlobCounters(unsigned long long * __restrict__ counters, uint32_t nBounces, uint32_t nShadow, uint32_t warpId)
{
  if (!counters) return;   // uniform
  __syncwarp();
  const uint32_t wb = __reduce_add_sync(0xffffffffu, nBounces);
  const uint32_t ws = __reduce_add_sync(0xffffffffu, nShadow);
  if ((threadIdx.x & 31u) == 0u)
  {
    const uint32_t slot = warpId & 31u;
    atomicAdd(&counters[slot * 2], (unsigned long long)wb);
    atomicAdd(&counters[slot * 2 + 1], (unsigned long long)ws);
  }
}

// K2 for row-aligned slices of blob scenes.  MULTI = false: one sample per pixel, no jitter (the batch path of the bench).
// MULTI = true: the same tiling for grid SSAA (Render.cpp:174-196: the thread walks its s*s samples in the reference's ssx, ssy
// order so the sum is formed in the same order) and additive jitter / accumulation (Render.cpp:177-178, :196-207).
template <bool MULTI, bool GRIDS, bool TRIS = false>
__global__ void __launch_bounds__(BLOB_THREADS, RFX_BLOB_MINBLOCKS) k_trace_blob(const unsigned char * __restrict__ sceneBlob, const __grid_constant__ FrameParams fp,
                                                                const uint32_t * __restrict__ sampleStates, uint32_t * __restrict__ argbOut,
                                                                unsigned long long * __restrict__ counters, uint32_t y0, uint32_t y1,
                                                                float * __restrict__ image, const __grid_constant__ EyeGrid eyeGrid)
{
  __shared__ int stackMem[BLOB_STACK * BLOB_THREADS];
  const BlobView sc = blobView(sceneBlob);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t x = (blockIdx.x * (BLOB_THREADS / 32) + warp) * BLOB_TILE_W + (lane % BLOB_TILE_W);
  const uint32_t y = y0 + blockIdx.y * BLOB_TILE_H + (lane / BLOB_TILE_W);
  const bool valid = x < fp.W && y < y1;
  uint32_t nBounces = 0, nShadow = 0, packed = 0, qOut = 0;
  const EyeGrid * eg = (GRIDS && eyeGrid.cellStart != nullptr) ? &eyeGrid : nullptr;
  const int eyeCell = eg ? (int)((y >> eyeGrid.shift) * (uint32_t)eyeGrid.nx + (x >> eyeGrid.shift)) : -1;
  if (valid)
  {
    const uint32_t q = y * fp.W + x;
    const float rx = float(x) - fp.wHalf;                                // Render.cpp:154-155
    const float ry = float(y) - fp.hHalf;
    const V3 eye = mk(fp.eye[0], fp.eye[1], fp.eye[2]);
    V3 c;
    if (!MULTI)
    {
      uint32_t s = __ldg(sampleStates + (q - y0 * fp.W));
      const V3 ray = mk((rx * fp.view[0] + ry * fp.view[1]) + fp.rz * fp.view[2],
                        (rx * fp.view[3] + ry * fp.view[4]) + fp.rz * fp.view[5],
                        (rx * fp.view[6] + ry * fp.view[7]) + fp.rz * fp.view[8]);
      V3 rd;
      rngTriple(s, rd.x, rd.y, rd.z);
      uint32_t events = 0, sig = 0;
      c = tracePath<false, GRIDS, TRIS>(sc, stackMem + threadIdx.x, eye, ray, fp.reflNum, rd, events, sig, eg, eyeCell);   // one sample: colour / 1 == colour
      nBounces = events & 0xFFFFu; nShadow = events >> 16;
    }
    else
    {
      const int sn = fp.sampleNum;
      const uint32_t rel = q - y0 * fp.W;                                // pixel index inside the slice
      float rndx = 0, rndy = 0;
      if (fp.jitter)
      {
        uint32_t s = lcgJump(fp.seedRender, 2u * rel);                   // two draws per pixel, Render.cpp:177-178
        s = 214013u * s + 2531011u; rndx = divExact(float((int)((s >> 16) & 0x7FFFu)), 32767.0f, RFX_RCP_32767);
        s = 214013u * s + 2531011u; rndy = divExact(float((int)((s >> 16) & 0x7FFFu)), 32767.0f, RFX_RCP_32767);
      }
      c = mk(0.0f, 0.0f, 0.0f);
      const uint32_t * st = sampleStates + (size_t)rel * (size_t)(sn * sn);
#pragma unroll 1
      for (int k = 0; k < sn * sn; k++)
      {
        const int ssx = k / sn, ssy = k - ssx * sn;
        uint32_t s = __ldg(st + k);
        V3 rd;
        rngTriple(s, rd.x, rd.y, rd.z);
        const float px = (rx + float(ssx) / float(sn)) + rndx;           // Render.cpp:184
        const float py = (ry + float(ssy) / float(sn)) + rndy;
        const V3 ray = mk((px * fp.view[0] + py * fp.view[1]) + fp.rz * fp.view[2],
                          (px * fp.view[3] + py * fp.view[4]) + fp.rz * fp.view[5],
                          (px * fp.view[6] + py * fp.view[7]) + fp.rz * fp.view[8]);
        uint32_t events = 0, sig = 0;
        const V3 one = tracePath<false, GRIDS, TRIS>(sc, stackMem + threadIdx.x, eye, ray, fp.reflNum, rd, events, sig, eg, eyeCell);
        nBounces += events & 0xFFFFu; nShadow += events >> 16;
        c = vadd(c, one);
      }
      const float sq = float(sn * sn);
      if (fabsf(sq) > RFX_VSN) c = mk(c.x / sq, c.y / sq, c.z / sq);     // Color::operator/=, Color.cpp:50-61
    }
    packed = packArgb(c.x, c.y, c.z);
    qOut = q;
    if (image)                                                           // Render.cpp:196-207
    {
      float * px = image + (size_t)q * 3;
      if (fp.accumulate) { px[0] = px[0] + c.x; px[1] = px[1] + c.y; px[2] = px[2] + c.z; }
      else { px[0] = c.x; px[1] = c.y; px[2] = c.z; }
    }
  }
  if (argbOut)
  {
    // framebuffer: one 128-bit store per tile row (see k_trace_small)
    const uint32_t p1 = __shfl_down_sync(0xffffffffu, packed, 1), p2 = __shfl_down_sync(0xffffffffu, packed, 2), p3 = __shfl_down_sync(0xffffffffu, packed, 3);
    const uint32_t validMask = __ballot_sync(0xffffffffu, valid);
    if ((fp.W & 3u) == 0u && ((validMask >> (lane & ~3u)) & 0xFu) == 0xFu)
    {
      if ((lane & 3u) == 0u) *reinterpret_cast<uint4 *>(argbOut + qOut) = make_uint4(packed, p1, p2, p3);
    }
    else if (valid) argbOut[qOut] = packed;
  }

  flushBlobCounters(counters, nBounces, nShadow, (blockIdx.y * gridDim.x + blockIdx.x) * (BLOB_THREADS / 32) + warp);
}

// ---- wavefront pair for one-sample ARGB frames (the batch path of the bench) -------------------------------------------------
// Paths of this kind of scene end after 1 to reflNum segments, and the deeper a segment the fewer lanes of a tile still hold a
// path: k_trace_blob runs config 4 at 15 of 32 lanes, and the rays of bounces 5-8 at a tenth of the first bounce's rate
// (profiles/README.md).  So a frame whose reflection depth is at least BLOB_WAVE_MIN_DEPTH is rendered by two kernels:
//   k_blob_wave_first  the tile kernel, but every path stops after its first TWO segments (primary rays, their shadow rays and the
//                      first reflection are the coherent part: neighbouring pixels walk the same nodes; queueing after one segment
//                      measured 9 % slower, after three 2 % slower); finished pixels are stored, the others are pushed to a queue
//                      in global memory, 64 bytes per path, the survivors of a warp side by side (one atomic per warp);
//   k_blob_wave_rest   a persistent grid that runs the queued paths to their ends with the same state machine in MODE_QUEUE: a
//                      lane whose path ends takes the next record at its next trip through the loop.  Its CTAs keep the
//                      hierarchy in shared memory.
// Which thread carries a path does not change any value it computes: frames are bit-identical to k_trace_blob's.
// Measured (config 4, 3840x2160, profiles/r2_s6*): depth 8 4.71 -> 3.86 ms, depth 4 3.59 -> 3.42 ms; depth 3 would lose 2 %.
// One stage kernel per remaining segment (survivors re-queued side by side after every segment) measured 4 % slower than the
// queue-driven kernel, and what bounds both is SIMT divergence inside the traversal — the queue-driven kernel issues at
// 11.5 of 32 lanes although every lane holds a path (ncu, profiles/r2_s7) — not idle lanes and not the L1 pipeline (the
// shared-memory copy of the hierarchy is worth 1.5 %).
template <bool GRIDS, bool TRIS = false>
__global__ void __launch_bounds__(BLOB_THREADS, RFX_BLOB_MINBLOCKS) k_blob_wave_first(const unsigned char * __restrict__ sceneBlob, const __grid_constant__ FrameParams fp,
                                                                     const uint32_t * __restrict__ sampleStates, uint32_t * __restrict__ argbOut,
                                                                     unsigned long long * __restrict__ counters, uint32_t y0, uint32_t y1, PathQueue queue,
                                                                     int firstSegments, const __grid_constant__ EyeGrid eyeGrid)
{
  __shared__ int stackMem[BLOB_STACK * BLOB_THREADS];
  const BlobView sc = blobView(sceneBlob);
  const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const uint32_t x = (blockIdx.x * (BLOB_THREADS / 32) + warp) * BLOB_TILE_W + (lane % BLOB_TILE_W);
  const uint32_t y = y0 + blockIdx.y * BLOB_TILE_H + (lane / BLOB_TILE_W);
  const bool valid = x < fp.W && y < y1;
  uint32_t nBounces = 0, nShadow = 0, events = 0, rel = 0, state0 = 0;
  V3 qo = mk(fp.eye[0], fp.eye[1], fp.eye[2]), qd = qo, mul = mk(1.0f, 1.0f, 1.0f), pix = mk(0.0f, 0.0f, 0.0f);
  bool alive = false;
  const EyeGrid * eg = (GRIDS && eyeGrid.cellStart != nullptr) ? &eyeGrid : nullptr;
  const int eyeCell = eg ? (int)((y >> eyeGrid.shift) * (uint32_t)eyeGrid.nx + (x >> eyeGrid.shift)) : -1;
  if (valid)
  {
    const uint32_t q = y * fp.W + x;
    rel = q - y0 * fp.W;
    uint32_t s = __ldg(sampleStates + rel);
    state0 = s;
    const float rx = float(x) - fp.wHalf;                                // Render.cpp:154-155
    const float ry = float(y) - fp.hHalf;
    qd = mk((rx * fp.view[0] + ry * fp.view[1]) + fp.rz * fp.view[2],
            (rx * fp.view[3] + ry * fp.view[4]) + fp.rz * fp.view[5],
            (rx * fp.view[6] + ry * fp.view[7]) + fp.rz * fp.view[8]);
    V3 rd;
    rngTriple(s, rd.x, rd.y, rd.z);
    uint32_t sig = 0;
    alive = !traceBlob<false, MODE_FIRST, BLOB_THREADS, false, GRIDS, TRIS>(sc, stackMem + threadIdx.x, qo, qd, fp.reflNum, rd, mul, pix, events, sig, nullptr, firstSegments, eg, eyeCell);
    if (!alive)
    {
      argbOut[q] = packArgb(pix.x, pix.y, pix.z);
      nBounces = events & 0xFFFFu; nShadow = events >> 16;
    }
  }
  // push the surviving paths of the warp side by side
  const uint32_t m = __ballot_sync(0xffffffffu, alive);
  if (m)
  {
    uint32_t base = 0;
    if (lane == 0) base = atomicAdd(queue.count, (uint32_t)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (alive)
    {
      uint4 * r = queue.records + 4 * (size_t)(base + (uint32_t)__popc(m & ((1u << lane) - 1u)));
      r[0] = make_uint4(__float_as_uint(qo.x), __float_as_uint(qo.y), __float_as_uint(qo.z), __float_as_uint(qd.x));
      r[1] = make_uint4(__float_as_uint(qd.y), __float_as_uint(qd.z), __float_as_uint(mul.x), __float_as_uint(mul.y));
      r[2] = make_uint4(__float_as_uint(mul.z), __float_as_uint(pix.x), __float_as_uint(pix.y), __float_as_uint(pix.z));
      r[3] = make_uint4(rel, events, state0, 0u);
    }
  }
  flushBlobCounters(counters, nBounces, nShadow, (blockIdx.y * gridDim.x + blockIdx.x) * (BLOB_THREADS / 32) + warp);
}

template <int THREADS, bool SMEM, bool TRIS = false>
__global__ void __launch_bounds__(THREADS, SMEM ? 2 : RFX_BLOB_MINBLOCKS) k_blob_wave_rest(const unsigned char * __restrict__ sceneBlob, int reflNum,
                                                                    uint32_t * __restrict__ argbSlice,
                                                                    unsigned long long * __restrict__ counters, PathQueue queue)
{
  // [traversal stacks: BLOB_STACK entries x THREADS][SMEM: the hierarchy — leaf sphere records and pair nodes]
  extern __shared__ int4 waveSmem[];
  int * stackMem = reinterpret_cast<int *>(waveSmem);
  BlobView sc = blobView(sceneBlob);
  if (SMEM)
  {
    // The queued paths are incoherent: every lane of a warp wants its own 64-byte node, and a 128-bit load whose lanes touch 32
    // different lines occupies the SM's one L1 pipeline for 32 wavefronts — four such loads per node visit.  That pipeline, not
    // instruction issue, bounded these rays (full warps were no faster than 40 %-full ones).  Shared memory serves 128 bytes per
    // clock whatever the addresses, so each CTA (persistent: it copies once) keeps its own copy of the hierarchy.
    float4 * copy = reinterpret_cast<float4 *>(stackMem + BLOB_STACK * THREADS);
    const float4 * src = sc.h->bvhLeafSph;
    for (uint32_t i = threadIdx.x; i < sc.h->bvhFloat4; i += THREADS) copy[i] = __ldg(src + i);
    __syncthreads();
    sc.bvhLeaves = copy;
    sc.bvhPairs = copy + (sc.h->bvhPairs - sc.h->bvhLeafSph);
  }
  QueueFeed feed;
  feed.records = queue.records; feed.count = queue.count; feed.cursor = queue.cursor;
  feed.argbOut = argbSlice;
  feed.bufNext = 0; feed.bufCount = 0;
  feed.doneBounces = 0; feed.doneShadow = 0;
  V3 qo = mk(0.0f, 0.0f, 0.0f), qd = qo, mul = qo, pix = qo;
  uint32_t events = 0, sig = 0;
  traceBlob<false, MODE_QUEUE, THREADS, SMEM, false, TRIS>(sc, stackMem + threadIdx.x, qo, qd, reflNum, qo, mul, pix, events, sig, &feed);
  flushBlobCounters(counters, feed.doneBounces, feed.doneShadow, blockIdx.x * (THREADS / 32) + (threadIdx.x >> 5));
}

// ---- general kernel: every mode of Render::renderNext for blob scenes (arbitrary pixel slices, block preview, signatures; grid SSAA,
// additive jitter, float image) — the blob counterpart of k_trace_small_any.  One thread per pixel (or per block origin).
template <bool TRIS = false>
__global__ void __launch_bounds__(BLOB_THREADS, RFX_BLOB_MINBLOCKS) k_trace_blob_any(const unsigned char * __restrict__ sceneBlob, const __grid_constant__ FrameParams fp,
                                                                    const uint32_t * __restrict__ sampleStates, float * __restrict__ image,
                                                                    uint32_t * __restrict__ argbOut, uint32_t * __restrict__ sigOut,
                                                                    unsigned long long * __restrict__ counters, int tiled,
                                                                    const __grid_constant__ EyeGrid eyeGrid)
{
  __shared__ int stackMem[BLOB_STACK * BLOB_THREADS];
  const BlobView sc = blobView(sceneBlob);
  uint32_t nBounces = 0, nShadow = 0;
  const V3 eye = mk(fp.eye[0], fp.eye[1], fp.eye[2]);
  const uint64_t gid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const EyeGrid * eg = eyeGrid.cellStart != nullptr ? &eyeGrid : nullptr;

  // ---- which pixel does this lane own, and how many Scene::trace calls does it make
  const bool blockMode = fp.sampleNum < 0;                 // block preview, Render.cpp:158-173
  const uint32_t blk = blockMode ? (uint32_t)(-fp.sampleNum) : 1u;
  const int sn = blockMode ? 1 : fp.sampleNum;             // grid SSAA factor, Render.cpp:174-196
  uint32_t x, y;
  bool valid;
  uint64_t firstState;                                     // index of this lane's first ranked random state
  if (blockMode)
  {
    // gid enumerates block origins in scan order starting at rank fp.firstRank
    const uint32_t bw = (fp.W + blk - 1) / blk;
    const uint64_t k = fp.firstRank + gid;
    y = (uint32_t)(k / bw) * blk; x = (uint32_t)(k % bw) * blk;
    valid = y < fp.H && ((uint64_t)y * fp.W + x) < fp.p1;
    firstState = gid;
  }
  else if (tiled)
  {
    // row-aligned slice (a whole frame or a band of rows): one pixel tile per warp
    const uint32_t tilesX = (fp.W + (BLOB_TILE_W - 1u)) / BLOB_TILE_W;
    const uint32_t y0 = (uint32_t)(fp.p0 / fp.W), y1 = (uint32_t)(fp.p1 / fp.W);
    const uint32_t warp = (uint32_t)(gid >> 5), lane = threadIdx.x & 31u;
    x = (warp % tilesX) * BLOB_TILE_W + (lane % BLOB_TILE_W);
    y = y0 + (warp / tilesX) * BLOB_TILE_H + (lane / BLOB_TILE_W);
    valid = x < fp.W && y < y1;
    firstState = (((uint64_t)y * fp.W + x) - fp.p0) * (uint64_t)(sn * sn);
  }
  else
  {
    const uint64_t p = fp.p0 + gid;
    valid = p < fp.p1;
    y = (uint32_t)(p / fp.W); x = (uint32_t)(p % fp.W);
    firstState = gid * (uint64_t)(sn * sn);
  }

  if (valid)
  {
    const uint64_t p = (uint64_t)y * fp.W + x;
    const float rx = float(x) - fp.wHalf;
    const float ry = float(y) - fp.hHalf;
    float rndx = 0, rndy = 0;
    if (fp.jitter && !blockMode)
    {
      uint32_t s = lcgJump(fp.seedRender, (uint32_t)(2 * (p - fp.p0)));      // two draws per pixel, Render.cpp:177-178
      s = 214013u * s + 2531011u; rndx = divExact(float((int)((s >> 16) & 0x7FFFu)), 32767.0f, RFX_RCP_32767);
      s = 214013u * s + 2531011u; rndy = divExact(float((int)((s >> 16) & 0x7FFFu)), 32767.0f, RFX_RCP_32767);
    }
    V3 fin = mk(0.0f, 0.0f, 0.0f);
    uint32_t sig = 2166136261u;
    const int eyeCell = eg ? (int)((y >> eyeGrid.shift) * (uint32_t)eyeGrid.nx + (x >> eyeGrid.shift)) : -1;
    const uint32_t * st = sampleStates + firstState;
    const int nCalls = sn * sn;
    int ssx = 0, ssy = 0;
#pragma unroll 1
    for (int call = 0; call < nCalls; call++)
    {
      uint32_t s = st[call];
      V3 rd;
      rngTriple(s, rd.x, rd.y, rd.z);
      float px = rx, py = ry;
      if (!blockMode)
      {
        // (rx + float(ssx)/s) + rndx, Render.cpp:184
        px = (rx + float(ssx) / float(sn)) + rndx;
        py = (ry + float(ssy) / float(sn)) + rndy;
      }
      const V3 ray = mk((px * fp.view[0] + py * fp.view[1]) + fp.rz * fp.view[2],
                        (px * fp.view[3] + py * fp.view[4]) + fp.rz * fp.view[5],
                        (px * fp.view[6] + py * fp.view[7]) + fp.rz * fp.view[8]);
      uint32_t events = 0;
      const V3 c = tracePath<true, true, TRIS>(sc, stackMem + threadIdx.x, eye, ray, fp.reflNum, rd, events, sig, eg, eyeCell);
      nBounces += events & 0xFFFFu; nShadow += events >> 16;
      fin = blockMode ? c : vadd(fin, c);
      if (++ssy == sn) { ssy = 0; ssx++; }                  // ssx outer, ssy inner: the reference's summation order
    }
    if (!blockMode)
    {
      const float sq = float(sn * sn);
      if (fabsf(sq) > RFX_VSN) fin = mk(fin.x / sq, fin.y / sq, fin.z / sq);   // Color::operator/=, Color.cpp:50-61
    }
    const uint32_t ex = min(x + blk, fp.W), ey = min(y + blk, fp.H);
    const uint32_t packed = packArgb(fin.x, fin.y, fin.z);
#pragma unroll 1
    for (uint32_t qy = y; qy < ey; qy++)
#pragma unroll 1
      for (uint32_t qx = x; qx < ex; qx++)
      {
        const uint64_t q = (uint64_t)qy * fp.W + qx;
        if (image)
        {
          float * px = image + q * 3;
          if (fp.accumulate && !blockMode) { px[0] = px[0] + fin.x; px[1] = px[1] + fin.y; px[2] = px[2] + fin.z; }
          else { px[0] = fin.x; px[1] = fin.y; px[2] = fin.z; }
        }
        if (argbOut) argbOut[q] = packed;
        if (sigOut) sigOut[q] = sig;
      }
  }
  flushBlobCounters(counters, nBounces, nShadow, blockIdx.x * (BLOB_THREADS / 32) + (threadIdx.x >> 5));
}

// ---- Scene::trace for an explicit ray list (rfx_trace_rays): ray i uses sampleStates[i]
template <bool TRIS = false>
__global__ void __launch_bounds__(BLOB_THREADS, RFX_BLOB_MINBLOCKS) k_trace_blob_rays(const unsigned char * __restrict__ sceneBlob, int n,
                                                                     const float * __restrict__ origins, const float * __restrict__ rays, int reflNum,
                                                                     const uint32_t * __restrict__ sampleStates, float * __restrict__ rgbOut,
                                                                     unsigned long long * __restrict__ counters)
{
  __shared__ int stackMem[BLOB_STACK * BLOB_THREADS];
  const BlobView sc = blobView(sceneBlob);
  uint32_t events = 0;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
  {
    uint32_t s = sampleStates[i], sig = 0;
    V3 rd;
    rngTriple(s, rd.x, rd.y, rd.z);
    const V3 c = tracePath<false, true, TRIS>(sc, stackMem + threadIdx.x, mk(origins[3 * i], origins[3 * i + 1], origins[3 * i + 2]),
                                  mk(rays[3 * i], rays[3 * i + 1], rays[3 * i + 2]), reflNum, rd, events, sig);
    rgbOut[3 * i] = c.x; rgbOut[3 * i + 1] = c.y; rgbOut[3 * i + 2] = c.z;
  }
  flushBlobCounters(counters, events & 0xFFFFu, events >> 16, blockIdx.x * (BLOB_THREADS / 32) + (threadIdx.x >> 5));
}

} // namespace

// pixels of the slice when it qualifies for the wavefront pair (one sample per pixel, no jitter, ARGB only, whole rows), else 0
uint64_t blobWavePixels(const TraceWork & w)
{
  const FrameParams & fp = w.fp;
  if (fp.sampleNum != 1 || fp.jitter || w.sigOut || !w.argbOut || w.image || fp.W == 0 || fp.stripWorld || fp.reflNum < BLOB_WAVE_MIN_DEPTH) return 0;
  if (fp.p0 % fp.W != 0 || fp.p1 % fp.W != 0 || fp.p1 - fp.p0 >= (1ull << 32) / 4) return 0;
  return fp.p1 - fp.p0;
}

// kernels launched (0 when the work does not qualify: the caller uses launchTraceBlobAny).  queue (optional): scratch for the
// wavefront pair, at least blobWavePixels(w) records of 64 bytes + two counters; persistentCtas: grid of the queue-driven kernel
int launchTraceBlobFast(const TraceWork & w, cudaStream_t st, void * queueRecords, uint32_t * queueCounters, uint32_t persistentCtas, int firstSegments,
                        uint32_t bvhFloat4)
{
  const FrameParams & fp = w.fp;
  if (fp.sampleNum < 1 || fp.sampleNum > 64 || w.sigOut || (!w.argbOut && !w.image) || fp.W == 0 || fp.stripWorld) return 0;
  if (fp.p0 % fp.W != 0 || fp.p1 % fp.W != 0 || (uint64_t)fp.W * fp.H >= (1ull << 32)) return 0;
  const uint64_t rows = (fp.p1 - fp.p0) / fp.W;
  if (rows == 0 || (rows + BLOB_TILE_H - 1) / BLOB_TILE_H > 65535u) return 0;
  const uint32_t tilesX = (fp.W + BLOB_TILE_W - 1) / BLOB_TILE_W, warps = BLOB_THREADS / 32;
  const dim3 grid((tilesX + warps - 1) / warps, (uint32_t)((rows + BLOB_TILE_H - 1) / BLOB_TILE_H));
  const unsigned char * blob = reinterpret_cast<const unsigned char *>(w.sceneBlob);
  const uint32_t y0 = (uint32_t)(fp.p0 / fp.W), y1 = (uint32_t)(fp.p1 / fp.W);
  if (queueRecords && queueCounters && persistentCtas && blobWavePixels(w) && fp.reflNum > firstSegments && firstSegments > 0)
  {
    if (cudaMemsetAsync(queueCounters, 0, 2 * sizeof(uint32_t), st) != cudaSuccess) return 0;
    PathQueue q;
    q.records = reinterpret_cast<uint4 *>(queueRecords); q.count = queueCounters; q.cursor = queueCounters + 1;
#define RFX_LAUNCH_FIRST(G, T) k_blob_wave_first<G, T><<<grid, BLOB_THREADS, 0, st>>>(blob, fp, w.sampleStates, w.argbOut, w.counters, y0, y1, q, firstSegments, w.eyeGrid)
    const bool gridsFirst = w.lightGrids || w.eyeGrid.cellStart != nullptr;
    if (w.triBvh) { if (gridsFirst) RFX_LAUNCH_FIRST(true, true); else RFX_LAUNCH_FIRST(false, true); }
    else if (gridsFirst) RFX_LAUNCH_FIRST(true, false);
    else RFX_LAUNCH_FIRST(false, false);
#undef RFX_LAUNCH_FIRST
    // the hierarchy in shared memory when it fits next to the stacks of two 512-thread CTAs per SM
    const size_t stackBytes512 = (size_t)BLOB_STACK * 512 * sizeof(int), bvhBytes = (size_t)bvhFloat4 * sizeof(float4);
    if (bvhFloat4 && stackBytes512 + bvhBytes <= 100 * 1024)
    {
      // (the triangle hierarchy, if any, stays in global memory and L1)
      const auto kRest = w.triBvh ? k_blob_wave_rest<512, true, true> : k_blob_wave_rest<512, true, false>;
      if (cudaFuncSetAttribute(kRest, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(stackBytes512 + bvhBytes)) != cudaSuccess) return 0;
      kRest<<<persistentCtas / 4, 512, stackBytes512 + bvhBytes, st>>>(blob, fp.reflNum, w.argbOut + fp.p0, w.counters, q);
    }
    else
    {
      const auto kRest = w.triBvh ? k_blob_wave_rest<BLOB_THREADS, false, true> : k_blob_wave_rest<BLOB_THREADS, false, false>;
      kRest<<<persistentCtas, BLOB_THREADS, (size_t)BLOB_STACK * BLOB_THREADS * sizeof(int), st>>>(blob, fp.reflNum, w.argbOut + fp.p0, w.counters, q);
    }
    return 2;
  }
  // 128-bit framebuffer stores need a 16-byte aligned frame: a caller's offset sub-buffer goes to the general kernel
  if (w.argbOut && (fp.W & 3u) == 0u && (reinterpret_cast<uintptr_t>(w.argbOut) & 15u) != 0u) return 0;
  const bool multi = !(fp.sampleNum == 1 && !fp.jitter);
#define RFX_LAUNCH_BLOB(M, G, T) k_trace_blob<M, G, T><<<grid, BLOB_THREADS, 0, st>>>(blob, fp, w.sampleStates, w.argbOut, w.counters, y0, y1, w.image, w.eyeGrid)
  const bool grids = w.lightGrids || w.eyeGrid.cellStart != nullptr;
  if (w.triBvh)
  {
    if (!multi && grids) RFX_LAUNCH_BLOB(false, true, true);
    else if (!multi) RFX_LAUNCH_BLOB(false, false, true);
    else if (grids) RFX_LAUNCH_BLOB(true, true, true);
    else RFX_LAUNCH_BLOB(true, false, true);
  }
  else if (!multi && grids) RFX_LAUNCH_BLOB(false, true, false);
  else if (!multi) RFX_LAUNCH_BLOB(false, false, false);
  else if (grids) RFX_LAUNCH_BLOB(true, true, false);
  else RFX_LAUNCH_BLOB(true, false, false);
#undef RFX_LAUNCH_BLOB
  return 1;
}

// every mode of Render::renderNext for blob scenes (the general kernel); returns kernels launched
int launchTraceBlobAny(const TraceWork & w, cudaStream_t st)
{
  const FrameParams & fp = w.fp;
  uint64_t nThreads;
  int tiled = 0;
  if (fp.sampleNum > 0)
  {
    nThreads = fp.p1 - fp.p0;
    if (fp.p0 % fp.W == 0 && fp.p1 % fp.W == 0)
    {
      tiled = 1;
      const uint64_t rows = (fp.p1 - fp.p0) / fp.W;
      nThreads = (uint64_t)((fp.W + BLOB_TILE_W - 1) / BLOB_TILE_W) * ((rows + BLOB_TILE_H - 1) / BLOB_TILE_H) * 32u;
    }
  }
  else
  {
    const uint32_t a = (uint32_t)(-fp.sampleNum);
    const uint32_t bw = (fp.W + a - 1) / a, bh = (fp.H + a - 1) / a;
    nThreads = (uint64_t)bw * bh - fp.firstRank;   // upper bound; threads past p1 exit
  }
  if (nThreads == 0) return 0;
  const uint32_t blocks = (uint32_t)((nThreads + BLOB_THREADS - 1) / BLOB_THREADS);
  const auto kAny = w.triBvh ? k_trace_blob_any<true> : k_trace_blob_any<false>;
  kAny<<<blocks, BLOB_THREADS, 0, st>>>(reinterpret_cast<const unsigned char *>(w.sceneBlob), fp, w.sampleStates, w.image, w.argbOut, w.sigOut,
                                        w.counters, tiled, w.eyeGrid);
  return 1;
}

int launchTraceBlobRays(const void * sceneBlob, int n, const float * origins, const float * rays, int reflNum,
                        const uint32_t * sampleStates, float * rgbOut, unsigned long long * counters, cudaStream_t st, bool triBvh)
{
  if (n <= 0) return 0;
  const auto kRays = triBvh ? k_trace_blob_rays<true> : k_trace_blob_rays<false>;
  kRays<<<(n + BLOB_THREADS - 1) / BLOB_THREADS, BLOB_THREADS, 0, st>>>(reinterpret_cast<const unsigned char *>(sceneBlob), n, origins, rays, reflNum,
                                                                                    sampleStates, rgbOut, counters);
  return 1;
}

} // namespace rfx
