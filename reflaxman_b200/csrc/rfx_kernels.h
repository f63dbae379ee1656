// rfx_kernels.h — launch interface between the C-ABI host layer (rfx_capi.cu, rfx_scene.cpp) and the sm_100a kernels (rfx_kernels.cu: K1 and K3;
// rfx_trace_small.cu, rfx_trace_blob.cu: K2).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>
#include "rfx_types.h"
#include "rfx_light_grid.h"
#include "rfx_eye_grid.h"

namespace rfx
{

// ---- K1: randDir stream ranking -------------------------------------------------------------------------------
// The reference draws one Vector3::randomInsideSphere per Scene::trace call from a single serial LCG with rejection
// sampling (reference Vector3.cpp:176-188, trace_math.h:34-39).  Trace call #p therefore owns the p-th ACCEPTED
// draw-triple of the stream.  K1 reproduces that in parallel from a table of the accept counts of the LCG's whole
// 2^32-state cycle (see the K1 header comment in rfx_kernels.cu).
constexpr int RNG_THREADS = 256;
constexpr int RNG_TRIPLES_PER_THREAD = 8;
constexpr int RNG_TRIPLES_PER_BLOCK = RNG_THREADS * RNG_TRIPLES_PER_THREAD;
constexpr uint32_t RNG_CLASS_BLOCKS = 699051;   // ceil(1431655766 / 2048): blocks of 2048 triples per residue class of start positions

struct RngLocate                // written by k_rng_locate, read by k_rng_rank: where on the cycle this pass starts
{
  uint32_t r0, j0;              // residue class of the start position and the block of that class holding it
  uint32_t r1, nb1;             // class after the wrap; virtual blocks [0, nb1) are blocks j0.. of class r0, the rest blocks 0.. of r1
  unsigned long long off1;      // accepted triples of class r0 before the stream's first triple
  unsigned long long seg1;      // accepted triples from the stream's first triple to the wrap
  uint32_t ownCount;            // split frames: number of virtual blocks in the list of blocks that hold ranks this GPU owns
};

struct RngWork
{
  const uint32_t * stateIn;     // device: LCG state before the first triple
  uint32_t * stateOut;          // device: LCG state after the triple that holds rank n-1
  const uint32_t * prefix;      // device [3][RNG_CLASS_BLOCKS + 1]: exclusive prefix sums of the per-block accept counts of the cycle
  RngLocate * locate;           // device scratch
  uint32_t * sampleStates;      // device out [n] (NULL: skip-only — one small CTA whatever n is)
  int * status;                 // device: set to 1 when the provisioned blocks do not hold n accepted triples
  uint64_t n;                   // accepted triples wanted
  uint32_t nBlocks;
  // optional scatter filter (split frames): only ranks r with (r / ownPeriod) % ownWorld == ownRank are stored (ownWorld = 0: all)
  uint64_t ownPeriod = 0;
  uint32_t ownWorld = 0, ownRank = 0;
  uint32_t * ownList = nullptr; // device scratch [ownListCap]: with ownWorld, k_rng_locate lists the virtual blocks that hold ranks this GPU owns and
  uint32_t ownListCap = 0;      // k_rng_rank is launched over that list only (an 8-GPU split 8K frame: 4 100 CTAs instead of 32 400, 74 -> 12 us)
};
// upper bound of the blocks that hold ranks of one GPU's strips (what ownListCap must be at least)
uint32_t rngOwnBlocksBound(uint64_t n, uint64_t ownPeriod, uint32_t ownWorld, uint32_t nBlocks);
// uploads K1's jump-ahead tables to the current device (once per context); 0 = ok
int initRngTables();
// fills the cycle's accept-count table: counts [3][RNG_CLASS_BLOCKS] scratch, prefix [3][RNG_CLASS_BLOCKS + 1]; returns kernels launched
int launchRngTable(uint32_t * counts, uint32_t * prefix, cudaStream_t st);
// K1 self-test over the LCG's whole cycle: out[0] = triples on which the integer accept test and the reference's float expression
// disagree (must be 0), out[1] = triples inside the guard band (decided by the float expression); out must be zeroed
int launchRngSelftest(unsigned long long * out, cudaStream_t st);
// number of blocks that over-provisions n accepted triples (acceptance pi/6 = 0.5236)
uint32_t rngBlocksFor(uint64_t n);
// enqueue locate (+ rank); returns the number of kernels launched
int launchRngRank(const RngWork & w, cudaStream_t st);

// ---- K2: trace + shade ----------------------------------------------------------------------------------------
// Cost-ordered tile scheduling of the fast kernel.  Path lengths differ by 20x between tiles (sky: one segment; between two
// mirror spheres: the full reflection depth), and the hardware starts CTAs in index order, so the long tiles of the image
// centre start late and the GPU drains for ~17 % of the kernel while they finish.  Every CTA therefore files itself, at its
// end, into one of four cost classes (longest path among its pixels); the next launch over the same grid starts the
// expensive classes first.  Results do not depend on the order; the first launch over a grid runs in index order.
constexpr int TILE_CLASSES = 4;
struct TileOrder
{
  const uint32_t * inLists = nullptr;   // [TILE_CLASSES][capacity] packed (tileRow << 16 | tileColumnGroup); NULL = index order
  const uint32_t * inCounts = nullptr;  // [TILE_CLASSES], sums to the grid size
  uint32_t * outLists = nullptr;        // [TILE_CLASSES][capacity], NULL = do not record
  uint32_t * outCounts = nullptr;       // [TILE_CLASSES], zero when the launch starts (the previous launch cleared it)
  uint32_t * zeroCounts = nullptr;      // [TILE_CLASSES] the NEXT launch records into: this launch clears it (no memset between frames)
  uint32_t capacity = 0;
};

// Blob scenes: candidate spheres of the FIRST query of a path (origin = eye) per screen cell of 2^shift x 2^shift pixels, built for every
// camera, image size and sphere update from the primary-ray screen bounds of the spheres: on the device (rfx_eye_grid.cu), or binned by the
// host (option "eye_grid_device" 0).  cellStart == NULL: none (the query walks the hierarchy).  The dims are the host's; whether the items
// fitted their region is known on the device only, so the kernels read the drop word after the offsets: non-zero, the build was dropped
// and the first queries walk the hierarchy.
struct EyeGrid
{
  const uint32_t * cellStart;   // [nx * ny + 2]: the cells' item offsets, the item total, the drop word
  const float4 * itemSphere;    // (cx, cy, cz, r^2) per (cell, sphere)
  const int * itemIndex;        // position in the sorted sphere array
  int nx, ny, shift;
};

struct TraceWork
{
  const void * sceneBlob;       // device scene blob (SceneHeader first)
  uint32_t sceneBytes;
  FrameParams fp;
  const uint32_t * sampleStates;// K1 output for this slice (one per Scene::trace call, call order)
  float * image;                // device W*H*3 float image (row 0 = bottom), may be NULL when argbOut is set
  uint32_t * argbOut;           // optional direct ARGB target (non-additive, whole-pixel results)
  uint32_t * sigOut;            // optional per-pixel hit-path signature
  unsigned long long * counters;// device [32][2] striped {bounces, shadowRays}
  TileOrder order;              // fast constant-bank kernel only
  uint32_t frames = 1;          // fast constant-bank kernel: consecutive frames of this one camera (fastBatchOk); frame f's states
                                // and ARGB frame lie f whole frames after sampleStates / argbOut
  bool lightGrids = false;      // blob scenes: the header carries candidate grids for some light (picks the kernel instantiation)
  bool triBvh = false;          // blob scenes: the header carries a hierarchy over the triangles (picks the kernel instantiation)
  bool far = false;             // blob scenes: the scene has a plane and a hierarchy, so a query can start outside the reach box (FAR)
  EyeGrid eyeGrid = { nullptr, nullptr, nullptr, 0, 0, 0 };
};
// blob scenes (rfx_trace_blob.cu).  launchTraceBlobFast: row-aligned slices (one sample per pixel, grid SSAA, additive jitter; ARGB
// and/or float image out); one-sample ARGB slices run as a wavefront pair when queue scratch is given (persistentCtas: grid of
// the queue-driven kernel in 128-thread CTAs).  Returns the
// number of kernels launched, 0 when the work does not qualify (the caller uses launchTraceBlobAny).  BVH depth is bounded by the host
// (BLOB_MAX_BVH_DEPTH): the traversal stack holds 24 entries per thread.
constexpr int BLOB_MAX_BVH_DEPTH = 22;
uint64_t blobWavePixels(const TraceWork & w);
#ifndef RFX_BLOB_WAVE_MIN_DEPTH
#define RFX_BLOB_WAVE_MIN_DEPTH 3
#endif
constexpr int BLOB_WAVE_MIN_DEPTH = RFX_BLOB_WAVE_MIN_DEPTH;       // shallower reflection limits render with the single tile kernel (the wavefront gains from depth 3 on: 2.73 against 2.77 ms, profiles/r2_grid)
// queueRecords: blobWavePixels(w) records of 64 bytes, queueCounters: 2 words
int launchTraceBlobFast(const TraceWork & w, cudaStream_t st, void * queueRecords = nullptr, uint32_t * queueCounters = nullptr, uint32_t persistentCtas = 0,
                        int firstSegments = 2,    // segments the tile kernel renders before it queues a path (0: no wavefront)
                        uint32_t bvhFloat4 = 0);  // SceneHeader::bvhFloat4 of the blob (0: no hierarchy): small hierarchies are copied to shared memory
int launchTraceBlobAny(const TraceWork & w, cudaStream_t st);     // every renderNext mode: ragged slices, block preview, signatures
// Scene::trace for a list of rays (rfx_trace_rays): rays[i] uses sampleStates[i]
int launchTraceBlobRays(const void * sceneBlob, int n, const float * origins, const float * rays, int reflNum,
                        const uint32_t * sampleStates, float * rgbOut, unsigned long long * counters, cudaStream_t st, bool triBvh, bool far);
// small scenes: constant-bank resident; *fastGrid (optional) receives the CTA count of the fast kernel's grid, 0 when the
// general kernel ran (the caller keeps tile-order history only for fast launches)
int launchTraceSmall(const SmallScene & sc, const TraceWork & w, cudaStream_t st, uint32_t * fastGrid = nullptr);
// CTA count the fast kernel would use for this work, 0 if the work does not qualify for it
uint32_t fastGridSize(const TraceWork & w);
#ifndef RFX_FRAME_BATCH
#define RFX_FRAME_BATCH 16      // most frames of one camera a fast-kernel launch renders (rfx_render_frames_device)
#endif
// whether the fast kernel can render several frames of this work's camera in one launch (whole one-sample ARGB frames)
bool fastBatchOk(const TraceWork & w);
// per launch of the fast kernel: pixel rectangles outside of which no primary ray can hit sphere i (rect[i]) / triangle k
// (rect[SMALL_MAX_SPHERES + k]); rfx_trace_small.cu has the derivation
struct PrimaryCull
{
  int4 rect[SMALL_MAX_SPHERES + SMALL_MAX_TRIS];   // x0, x1, y0, y1 (inclusive, frame pixels); x0 > x1: no pixel
};
PrimaryCull makePrimaryCull(const SmallScene & sc, const FrameParams & fp);
// (the same bounds one sphere at a time, which blob scenes bin into the screen grid of the first query: primarySphereBounds, rfx_eye_grid.h)

// rows a launch over `rows` whole rows enumerates: all of them, or in a split frame (fp.stripWorld > 0) the rows of this rank's
// strips, full strips plus the (possibly shorter) last strip, rounded up to whole strips
inline uint64_t ownedRows(const FrameParams & fp, uint64_t rows)
{
  if (!fp.stripWorld) return rows;
  const uint64_t nStrips = (rows + fp.stripRows - 1) / fp.stripRows;
  const uint64_t mine = nStrips > fp.stripRank ? (nStrips - fp.stripRank + fp.stripWorld - 1) / fp.stripWorld : 0;
  return mine * fp.stripRows;
}

// threads of a general K2 kernel (k_trace_small_any, k_trace_blob_any) for this work, 0 = nothing to render.  tiled = 1: the slice
// is whole rows and each warp renders a tile of tileW x (32 / tileW) pixels; tiled = 0: one thread per pixel or block origin
inline uint64_t anyThreads(const FrameParams & fp, uint32_t tileW, int & tiled)
{
  tiled = 0;
  if (fp.sampleNum <= 0)
  {
    const uint32_t a = (uint32_t)(-fp.sampleNum);
    const uint32_t bw = (fp.W + a - 1) / a, bh = (fp.H + a - 1) / a;
    return (uint64_t)bw * bh - fp.firstRank;   // upper bound; threads past p1 exit
  }
  if (fp.p0 % fp.W != 0 || fp.p1 % fp.W != 0) return fp.p1 - fp.p0;
  tiled = 1;
  const uint64_t rows = ownedRows(fp, (fp.p1 - fp.p0) / fp.W), tileH = 32u / tileW;
  return (uint64_t)((fp.W + tileW - 1) / tileW) * ((rows + tileH - 1) / tileH) * 32u;
}

// calls f(std::true_type()) or f(std::false_type()): a run-time flag picks a kernel instantiation
template <typename F> inline void withFlag(bool b, F && f)
{
  if (b) f(std::true_type());
  else f(std::false_type());
}

// ---- mesh updates (rfx_mesh.cu, rfx_update_mesh) ------------------------------------------------------------------
// k_mesh_setup sets up one mesh's triangles from new vertices into the blob and the hierarchy's leaf slots; k_tri_refit then
// recomputes every leaf's box and the pair nodes bottom-up.  The hierarchy keeps the topology of the last flatten.
struct MeshUpdate
{
  Triangle * tris;              // the blob's sorted triangle array
  SceneHeader * header;         // the blob's header (triReach, growT, nTriAlways of plane scenes)
  const float * xyz;            // the mesh's new vertices (device)
  const uint32_t * idx;         // its index list (device), 3 per triangle
  int triBase, nTris;           // its triangles' positions in the sorted array
  // the triangle hierarchy (triLeaf == NULL: none, only the blob is written)
  float4 * triLeaf, * triPairs;
  const int * triPrims, * triSlot;          // slot -> sorted position, sorted position -> slot (-1: none)
  const int * leafParent, * pairParent;     // 2 * parent pair node + side, -1: root
  uint32_t * arrive;                        // per pair node, zero before the refit
  int nLeaves;
  unsigned long long * red;                 // [7] orderedCode: union box lo xyz (min), hi xyz (max), largest kappa (max)
  bool far;                                 // plane scene: slivers leave the hierarchy for triAlways
  int * triAlways;                          // capacity: every triangle
  unsigned char * inAlways;                 // per sorted position: already appended to triAlways since the flatten
};
int launchMeshUpdate(const MeshUpdate & u, cudaStream_t st);   // returns the number of kernels launched

// ---- sphere updates (rfx_mesh.cu, rfx_update_spheres) -----------------------------------------------------------------------
// k_sphere_scatter writes the moved spheres' records into the blob's sphere array and the hierarchy's leaf slots; k_sphere_refit then
// recomputes every leaf's box and the pair nodes bottom-up, as k_tri_refit does.  The hierarchy keeps the topology of the last flatten.
struct SphereMove
{
  float4 rec;                   // (cx, cy, cz, r^2), as rfx_add_sphere stores it
  int pos;                      // the sphere's position in the sorted sphere array
  float radius;
  int pad[2];
};
struct SphereUpdate
{
  const SphereMove * moves;     // device, one per moved sphere (no duplicates)
  int nMoves;
  float4 * spheres;             // the blob's sorted sphere array
  float * radius;               // per sphere: its radius
  // the sphere hierarchy (leafSph == NULL: none, only the blob is written)
  float4 * leafSph, * pairs;
  const int * prims, * slot;                // slot -> sphere, sphere -> slot
  const int * leafParent, * pairParent;     // 2 * parent pair node + side, -1: root
  uint32_t * arrive;                        // per pair node, zero before the refit
  int nLeaves;
  double R;                                 // the margins' R of the last flatten
};
int launchSphereUpdate(const SphereUpdate & u, cudaStream_t st);   // returns the number of kernels launched

// ---- light grids on the device (rfx_light_grid.cu: rfx_update_lights, rfx_update_spheres) --------------------------------------------
// One far light's LightGrid built from the spheres of the blob, byte for byte what rfx_scene.cpp buildLightGrid builds for them, into the
// light's fixed regions (cells, items).  A grid with more items than itemCap is dropped: its header is NULL and *dropped set, *need
// raised to its item count.  A light without a grid (no disc, an empty extent, no finite bound) gets a NULL header.
struct LightGridBuild
{
  LightFrame f;                 // the light over the grid box (lightFrame, on the host)
  const float4 * spheres;       // the blob's sorted sphere array
  const float * radius;         // per sphere: its radius
  const int * prims;            // the sphere hierarchy's leaf slots: the sphere of each slot, -1 unused
  int nSlots;
  uint64_t nPrims;              // used slots (every sphere)
  double R;                     // the margins' R of the last flatten
  LightGrid * header;           // the light's header in the device array
  uint32_t * cells;             // the light's cell region [LIGHT_GRID_CELLS]
  float4 * itemSphere;          // its item regions [itemCap]
  int * itemIndex;
  uint32_t itemCap;
  uint32_t * need;              // raised to the item count of a grid that did not fit (read by the host at a synchronising call)
  uint32_t * dropped;           // the light's last build did not fit
  // scratch, shared by the builds on one stream
  double * disc;                // 3 per slot: pu, pv, rho
  uint32_t * span;              // 2 per slot: x0 | x1 << 16, y0 | y1 << 16 of the disc's cells (0xFFFF: none)
  double * blockSum;            // one per LIGHT_GRID_SUM_BLOCK slots
  unsigned long long * red;     // [5] orderedCode of ulo (min), uhi (max), vlo (min), vhi (max); non-zero: no finite bound.  Left at
                                // (1e300, -1e300, 1e300, -1e300, 0) by each build for the next
  LightGridDims * dims;         // nx == 0: no grid (or dropped)
};
int launchLightGridBuild(const LightGridBuild & b, cudaStream_t st);   // returns the number of kernels launched

// ---- the eye grid on the device (rfx_eye_grid.cu) -----------------------------------------------------------------------------------------
// The EyeGrid of one camera built from the spheres of the blob: exactly what rfx_scene.cpp binEyeGrid bins for them, into fixed regions.  A
// grid with more items than itemCap is dropped: its drop word is set, flags[0] raised to its item count and flags[1] counts the drop.
struct EyeGridBuild
{
  PrimaryCamera cam;            // makePrimaryCamera of the frame (ok: eyeGridDims gave nx, ny)
  uint32_t W, H;
  int nx, ny;
  const float4 * spheres;       // the blob's sorted sphere array
  int nSpheres;
  uint32_t * cells;             // [nx * ny + 2] (EyeGrid::cellStart)
  float4 * itemSphere;          // [itemCap]
  int * itemIndex;
  uint32_t itemCap;
  uint32_t * flags;             // [2]: the largest item count of a dropped build, builds dropped (read by the host at a synchronising call)
  // scratch
  int2 * xSpan;                 // per sphere: the columns of cells its rectangle touches (x0 > x1: none)
  uint32_t * rowMask;           // [ny][maskWords]: bit i of row y set when sphere i touches row y
  int maskWords;                // (nSpheres + 31) / 32
};
int launchEyeGridBuild(const EyeGridBuild & b, cudaStream_t st);      // returns the number of kernels launched

// ---- K3: resolve (imagePixel + argb)---------------------------------------------------------------------------
int launchResolve(const float * image, uint64_t nPixels, int additiveCounter, float * rgbfOut, uint32_t * argbOut, cudaStream_t st);
int launchClear(float * image, uint64_t nFloats, cudaStream_t st);

// host mirror of the LCG jump (n draws ahead)
uint32_t lcgJumpHost(uint32_t s, uint64_t n);

} // namespace rfx
