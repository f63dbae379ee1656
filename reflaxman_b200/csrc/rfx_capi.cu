// rfx_capi.cu — the C ABI of include/reflax_c.h: context, scene upload, slice scheduling.  The scene itself is flattened on the
// host by rfx_scene.cpp.
//
// Host-side float arithmetic in this file (envColor, sqRadius) restates what the reference's constructors compute once per object;
// it is compiled with -ffp-contract=off so every operation is the same IEEE binary32 operation the reference's build performs
// (reference Scene.cpp:10-15,47-58; Sphere.cpp:9-20; OmniLight.cpp:8-14).
#include "../../include/reflax_c.h"
#include "rfx_kernels.h"
#include "rfx_scene.h"

#include <cuda_runtime.h>
#include <float.h>
#include <math.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include <memory>
#include <stddef.h>

using namespace rfx;

namespace
{

std::string g_createError;

// A device array the context owns: freed when the context is deleted.  ensure() grows it.
template <typename T> struct DevArray
{
  T * p = nullptr;
  size_t cap = 0;                           // elements
  DevArray() = default;
  DevArray(DevArray && o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  DevArray(const DevArray &) = delete;
  DevArray & operator=(const DevArray &) = delete;
  ~DevArray() { cudaFree(p); }
  cudaError_t alloc(size_t n)               // exactly n elements, into an empty array
  {
    const cudaError_t e = cudaMalloc((void **)&p, n * sizeof(T));
    cap = e == cudaSuccess ? n : 0;
    return e;
  }
};

} // namespace

struct rfx_ctx
{
  int device = 0;
  cudaStream_t stream = nullptr, copyStream[2] = { nullptr, nullptr }, lastStream = nullptr;
  bool frameBatch = true;                   // rfx_set_option "frame_batch": rfx_render_frames_device renders runs of one camera in batched launches
  int copyStreams = 1;                      // D2H streams rfx_render_frames alternates between (rfx_set_option "copy_streams")
  cudaDeviceProp prop;
  mutable std::string err;

  HostScene scene;
  bool sceneDirty = true;

  // ---- device scene (uploadScene)
  SceneImage image;                         // what was uploaded, device pointers filled in (kept: the next upload rebuilds it in place)
  DevArray<unsigned char> dBlob;
  // cost-ordered tile scheduling of the fast kernel (TileOrder, rfx_kernels.h): two list sets, used alternately
  DevArray<uint32_t> dTileLists[2];
  DevArray<uint32_t> dTileCounts;           // [3][TILE_CLASSES]: recorded by the previous launch | recorded by this one | cleared by this one for the next
  int tileSlot = 0;                         // list set the NEXT launch records into
  int tileCountSlot = 0;                    // count set the NEXT launch records into (zero by then: cleared at creation or by the launch before)
  int tileRecordPeriod = 8;                 // rfx_set_option "tile_order_period": the cost classes are recorded on every k-th launch over a grid; the
                                            // launches in between replay the last recording (no CTA barrier, no atomic at their end: -2 % kernel time)
  int tileReuse = 0;                        // launches that reused the last recording
  bool tileHistory = false;                 // the other set holds the order recorded by the previous launch ...
  uint64_t tileKey[4] = { 0, 0, 0, 0 };     // ... over this grid (image size, row range, strip split)
  bool tileOrdering = true;
  int forcePath = 0;                        // 0 auto, 1 constant bank, 2 blob kernels, 3 blob, general kernel (k_trace_blob_any) only — tests exercise all
  DevArray<float> dLut;
  DevArray<float4> dBvhNodes;               // big scenes only: the hierarchy over the spheres, leaf slots then pair nodes
  DevArray<int> dBvhPrims;
  bool blobSmemBvh = true;                  // rfx_set_option "blob_smem_bvh"
  // shadow-ray candidate grids of the far lights (LightGrid, rfx_types.h): a header per light, and per light fixed regions of
  // LIGHT_GRID_CELLS cell offsets and gridItemAlloc items, which the flatten's grids are uploaded into and the device builder
  // (rfx_light_grid.cu) writes: light i's cells at dGridCells + i * LIGHT_GRID_CELLS, its items at i * gridItemAlloc
  DevArray<LightGrid> dLightGrids;
  DevArray<uint32_t> dGridCells;
  DevArray<float4> dGridSpheres;
  DevArray<int> dGridIndex;
  size_t gridItemAlloc = 0;                 // items per light region: twice the flatten's largest grid (at least 1024), grown on demand
  uint32_t gridItemCap = 0;                 // items a device build may write: gridItemAlloc, or fewer under gridItemLimit
  int64_t gridItemLimit = 0;                // rfx_set_option "light_grid_items" (test hook; 0: none)
  std::vector<char> lightGrid;              // per light: it has a grid now (the flatten built one, or its last update found it far)
  DevArray<uint32_t> dGridFlags;            // [1 + nLights]: the largest item count of a build that did not fit, then per light: dropped
  DevArray<double> dLgDisc, dLgBlockSum;    // the builder's scratch (LightGridBuild)
  DevArray<uint32_t> dLgSpan;
  DevArray<unsigned long long> dLgRed;
  DevArray<LightGridDims> dLgDims;
  // candidate spheres of the first query of a path per 32x32-pixel screen cell (EyeGrid, rfx_kernels.h), rebuilt when the camera,
  // the image size, the scene or the spheres change: on the device (rfx_eye_grid.cu) into a fixed item region of eyeItemAlloc items
  DevArray<uint32_t> dEyeCells;             // [nx * ny + 2]
  DevArray<float4> dEyeSpheres;
  DevArray<int> dEyeIndex;
  size_t eyeItemAlloc = 0;                  // items of the region: sized at the first build, grown at a synchronising call after a drop
  int64_t eyeItemLimit = 0;                 // rfx_set_option "eye_grid_items" (test hook; 0: none)
  DevArray<uint32_t> dEyeFlags;             // [2]: the largest item count of a dropped build, builds dropped since creation
  DevArray<int2> dEgSpan;                   // the builder's scratch (EyeGridBuild)
  DevArray<uint32_t> dEgRows;
  EyeGrid eyeGrid = { nullptr, nullptr, nullptr, 0, 0, 0 };
  uint32_t eyeKey[17] = { 0 }; uint64_t eyeSceneKey = 0, eyeSphereKey = 0; bool eyeValid = false;   // camera (eye, view, rz, wHalf, hHalf as bits) + W, H
  uint64_t sceneUploads = 0;                // bumped by uploadScene
  uint64_t sphereUpdates = 0;               // bumped by rfx_update_spheres when it updates the device scene
  bool eyeGridOn = true;                    // rfx_set_option "eye_grid"
  bool eyeGridDevice = true;                // rfx_set_option "eye_grid_device": 0 = binned on the host and uploaded
  uint64_t eyeGridBuilds = 0;
  // the last blob render (rfx_selftest_eye_grid): its camera, and the grid it used
  bool eyeRendered = false;
  FrameParams eyeFp;
  EyeGrid eyeUsed = { nullptr, nullptr, nullptr, 0, 0, 0 };
  DevArray<float4> dTriNodes;               // hierarchy over the triangles: leaf slots, then pair nodes
  DevArray<int> dTriPrims;
  DevArray<int> dTriAlways;                 // plane scenes: triangles tested after the triangle walk (SceneHeader::triAlways); with meshes
                                            // room for every triangle (rfx_update_mesh appends slivers)
  // mesh updates on the device (rfx_update_mesh, MeshUpdate): uploaded by uploadScene for blob scenes with meshes
  DevArray<uint32_t> dMeshIdx;              // every mesh's index list (SceneImage::meshIdx)
  DevArray<int> dTriSlot, dLeafParent, dPairParent;
  DevArray<unsigned char> dInAlways;        // per triangle: appended to triAlways since the flatten
  DevArray<uint32_t> dArrive;               // per pair node: refit arrival counters
  DevArray<unsigned long long> dMeshRed;    // [14]: an update's reduction record (MeshUpdate::red), then its value at the flatten
  DevArray<float> dVerts;                   // the vertices of the mesh being updated
  // sphere updates on the device (rfx_update_spheres, SphereUpdate): uploaded by uploadScene for blob scenes with spheres
  DevArray<float> dSphRadius;               // per sphere: its radius (SceneImage::sphRadius)
  DevArray<int> dSphSlot, dSphLeafParent, dSphPairParent;
  DevArray<uint32_t> dSphArrive;            // per pair node of the sphere hierarchy: refit arrival counters
  DevArray<SphereMove> dSphMoves;           // the moved spheres of an update
  std::vector<SphereMove> sphMoves;         // ... their host records (alive until the next update)
  std::vector<char> sphMoved;               // per sphere: scratch of the update's duplicate resolution

  // ---- camera + render state (reference Render.h:9-27); the eye is scene.eye
  float view[9] = { 1, 0, 0, 0, 1, 0, 0, 0, 1 }, fov = 1.0f;
  uint32_t W = 0, H = 0;
  DevArray<float> dImage;
  DevArray<uint32_t> dSig; bool sigOn = false;
  int reflNum = 0, sampleNum = 0; bool additive = false; int additiveCounter = 0; bool inProgress = false;
  uint64_t cursor = 0;
  FrameParams snap;           // camera snapshot taken by render_begin

  // ---- random streams
  DevArray<uint32_t> dRng;    // [2] ping-pong LCG state of the Vector3.cpp TU stream
  int rngSlot = 0;
  uint32_t seedRender = 12345u;
  DevArray<uint32_t> dRngPrefix;              // [3][RNG_CLASS_BLOCKS + 1] accept-count prefix sums of the LCG cycle (built at creation)
  DevArray<RngLocate> dRngLocate;
  DevArray<uint32_t> dSampleStates;
  DevArray<uint32_t> dOwnBlocks;              // split frames: K1's list of the blocks that hold this GPU's ranks
  DevArray<int> dStatus;
  DevArray<float> dRays;                      // rfx_trace_rays scratch

  // ---- staging for the host batch path
  static const int FRAME_SLOTS = 4;
  DevArray<uint32_t> dFrame[FRAME_SLOTS];
  DevArray<uint32_t> dResolve;                // K3 output of the Render-API read path
  uint64_t maxCallsPerLaunch = 1ull << 25;    // bounds the ranked-state scratch (128 MB) for huge SSAA factors / 8K frames
  // path queue of the blob scenes' wavefront kernel pair (rfx_trace_blob.cu): 64-byte records + {count, cursor}
  DevArray<uint4> dQueue;                     // in uint4 units (4 per record)
  DevArray<uint32_t> dQueueCtl;
  int blobWavefront = 2;                      // rfx_set_option "blob_wavefront": 0 off, k > 0: the tile kernel of the wavefront renders k segments
  cudaEvent_t evRendered[FRAME_SLOTS] = { nullptr, nullptr, nullptr, nullptr }, evCopied[FRAME_SLOTS] = { nullptr, nullptr, nullptr, nullptr };

  // ---- counters
  DevArray<unsigned long long> dCounters;     // [32][2]
  rfx_stats stats;
  bool profiling = false;
  std::vector<cudaEvent_t> evPool;            // pairs (start, stop) around K2 launches while profiling
  size_t evUsed = 0;
};

namespace
{

int fail(const rfx_ctx * c, int code, const std::string & msg)
{
  if (c) c->err = msg; else g_createError = msg;
  return code;
}

#define CK(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess)                                                                               \
      return fail(ctx, RFX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                \
  } while (0)

int useStream(rfx_ctx * ctx, cudaStream_t st)
{
  if (ctx->lastStream && ctx->lastStream != st) CK(cudaStreamSynchronize(ctx->lastStream));
  ctx->lastStream = st;
  return RFX_OK;
}

template <typename T> int ensure(rfx_ctx * ctx, DevArray<T> & a, size_t need)
{
  if (need <= a.cap) return RFX_OK;
  if (a.p) { CK(cudaDeviceSynchronize()); CK(cudaFree(a.p)); a.p = nullptr; a.cap = 0; }
  CK(a.alloc(need + need / 8));
  return RFX_OK;
}

// a host array to the front of a device array (an empty one still gets an address).  A pageable source is staged before the call
// returns; the caller keeps it alive until the stream has synchronised all the same.
template <typename T> int upload(rfx_ctx * ctx, DevArray<T> & a, const std::vector<T> & v, cudaStream_t st)
{
  int rc;
  if ((rc = ensure(ctx, a, std::max<size_t>(v.size(), 1))) != RFX_OK) return rc;
  if (!v.empty()) CK(cudaMemcpyAsync(a.p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, st));
  ctx->stats.h2d_bytes += v.size() * sizeof(T);
  return RFX_OK;
}

void setGridItemCap(rfx_ctx * ctx)
{
  size_t cap = ctx->gridItemAlloc;
  if (ctx->gridItemLimit > 0) cap = std::min<size_t>(cap, (size_t)ctx->gridItemLimit);
  ctx->gridItemCap = (uint32_t)std::min<size_t>(cap, UINT32_MAX);
}

// flatten the host scene (rfx_scene.cpp) and upload it
int uploadScene(rfx_ctx * ctx, cudaStream_t st)
{
  if (!ctx->sceneDirty) return RFX_OK;
  ctx->sceneUploads++;
  ctx->eyeValid = false;
  ctx->eyeRendered = false;

  for (HostTex & t : ctx->scene.tex)
    if (!t.uploaded)
    {
      if (!t.px.empty())
      {
        CK(cudaMalloc((void **)&t.dev, t.px.size() * 4));
        CK(cudaMemcpyAsync(t.dev, t.px.data(), t.px.size() * 4, cudaMemcpyHostToDevice, st));
        ctx->stats.h2d_bytes += t.px.size() * 4;
      }
      t.uploaded = true;
    }

  SceneImage & img = ctx->image;
  int rc;
  refreshMeshes(ctx->scene);
  if ((rc = buildSceneImage(ctx->scene, img, ctx->err)) != RFX_OK) return rc;
  SceneHeader & h = *reinterpret_cast<SceneHeader *>(img.blob.data());
  h.byteLut = ctx->dLut.p;
  if (!img.sphBvh.nodes.empty())
  {
    if ((rc = upload(ctx, ctx->dBvhNodes, img.sphBvh.nodes, st)) != RFX_OK || (rc = upload(ctx, ctx->dBvhPrims, img.sphBvh.prims, st)) != RFX_OK) return rc;
    h.bvhPrims = ctx->dBvhPrims.p;
    h.bvhLeafSph = ctx->dBvhNodes.p;
    h.bvhPairs = ctx->dBvhNodes.p + img.sphBvh.leafFloat4;
  }
  ctx->lightGrid.assign(ctx->scene.lights.size(), 0);
  std::vector<LightGrid> headers(img.grids);   // (alive until the synchronisation below)
  std::vector<uint32_t> flags;
  std::vector<unsigned long long> lgRed;
  if (!img.grids.empty())
  {
    // each light's grid into its regions (cellStart offsets are relative to the light's own items)
    const size_t nL = img.grids.size();
    size_t largest = 0;
    for (size_t li = 0; li < nL; li++)
      if (img.grids[li].nx) largest = std::max<size_t>(largest, img.gridCells[img.gridCellOff[li] + (size_t)img.grids[li].nx * img.grids[li].ny]);
    if ((rc = ensure(ctx, ctx->dGridCells, nL * LIGHT_GRID_CELLS)) != RFX_OK || (rc = ensure(ctx, ctx->dGridSpheres, nL * std::max<size_t>(2 * largest, 1024))) != RFX_OK ||
        (rc = ensure(ctx, ctx->dGridIndex, nL * std::max<size_t>(2 * largest, 1024))) != RFX_OK) return rc;
    ctx->gridItemAlloc = std::min(ctx->dGridSpheres.cap, ctx->dGridIndex.cap) / nL;
    setGridItemCap(ctx);
    flags.assign(1 + nL, 0);
    for (size_t li = 0; li < nL; li++)
    {
      if (!img.grids[li].nx) continue;
      ctx->lightGrid[li] = 1;
      const size_t nCells = (size_t)img.grids[li].nx * img.grids[li].ny + 1, nItems = img.gridCells[img.gridCellOff[li] + nCells - 1];
      if (nItems > ctx->gridItemCap)   // (only under the "light_grid_items" hook) dropped, as a device build that does not fit
      {
        headers[li] = LightGrid();
        flags[0] = std::max<uint32_t>(flags[0], (uint32_t)nItems); flags[1 + li] = 1;
        continue;
      }
      LightGrid & g = headers[li];
      g.cellStart = ctx->dGridCells.p + li * LIGHT_GRID_CELLS;
      g.itemSphere = ctx->dGridSpheres.p + li * ctx->gridItemAlloc;
      g.itemIndex = ctx->dGridIndex.p + li * ctx->gridItemAlloc;
      CK(cudaMemcpyAsync((void *)g.cellStart, &img.gridCells[img.gridCellOff[li]], nCells * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
      if (nItems)
      {
        CK(cudaMemcpyAsync((void *)g.itemSphere, &img.gridSpheres[img.gridItemOff[li]], nItems * sizeof(float4), cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync((void *)g.itemIndex, &img.gridIndex[img.gridItemOff[li]], nItems * sizeof(int), cudaMemcpyHostToDevice, st));
      }
      ctx->stats.h2d_bytes += nCells * sizeof(uint32_t) + nItems * (sizeof(float4) + sizeof(int));
    }
    if ((rc = upload(ctx, ctx->dLightGrids, headers, st)) != RFX_OK || (rc = upload(ctx, ctx->dGridFlags, flags, st)) != RFX_OK) return rc;
    h.lightGrids = ctx->dLightGrids.p;
    if (!img.smallOk)   // the device builder's scratch (rfx_update_lights, rfx_update_spheres)
    {
      const size_t nSlots = img.sphBvh.prims.size();
      lgRed = { orderedCode(1e300), orderedCode(-1e300), orderedCode(1e300), orderedCode(-1e300), 0ull };
      if ((rc = ensure(ctx, ctx->dLgDisc, 3 * nSlots)) != RFX_OK || (rc = ensure(ctx, ctx->dLgSpan, 2 * nSlots)) != RFX_OK ||
          (rc = ensure(ctx, ctx->dLgBlockSum, nSlots / LIGHT_GRID_SUM_BLOCK + 1)) != RFX_OK || (rc = ensure(ctx, ctx->dLgDims, 1)) != RFX_OK ||
          (rc = upload(ctx, ctx->dLgRed, lgRed, st)) != RFX_OK) return rc;
    }
  }
  if (!img.triBvh.nodes.empty())
  {
    if ((rc = upload(ctx, ctx->dTriNodes, img.triBvh.nodes, st)) != RFX_OK || (rc = upload(ctx, ctx->dTriPrims, img.triBvh.prims, st)) != RFX_OK) return rc;
    h.triPrims = ctx->dTriPrims.p;
    h.triLeaf = ctx->dTriNodes.p;
    h.triPairs = ctx->dTriNodes.p + img.triBvh.leafFloat4;
  }
  const bool meshUpdates = !img.meshes.empty() && !img.smallOk;   // rfx_update_mesh can update this scene on the device
  std::vector<unsigned long long> red;
  if (meshUpdates)
  {
    if ((rc = upload(ctx, ctx->dMeshIdx, img.meshIdx, st)) != RFX_OK) return rc;
    if (!img.triSlot.empty())
    {
      const size_t nTris = img.triSlot.size();
      if ((rc = upload(ctx, ctx->dTriSlot, img.triSlot, st)) != RFX_OK || (rc = upload(ctx, ctx->dLeafParent, img.leafParent, st)) != RFX_OK ||
          (rc = upload(ctx, ctx->dPairParent, img.pairParent, st)) != RFX_OK || (rc = ensure(ctx, ctx->dArrive, std::max<size_t>(img.pairParent.size(), 1))) != RFX_OK ||
          (rc = ensure(ctx, ctx->dInAlways, nTris)) != RFX_OK || (rc = ensure(ctx, ctx->dTriAlways, nTris)) != RFX_OK)
        return rc;
      CK(cudaMemsetAsync(ctx->dInAlways.p, 0, nTris, st));
      red.assign(14, 0);
      for (int k = 0; k < 6; k++) red[7 + k] = orderedCode(img.triUnion[k]);
      red[13] = orderedCode(0.0);
      if ((rc = upload(ctx, ctx->dMeshRed, red, st)) != RFX_OK) return rc;
      if (img.far) h.triAlways = ctx->dTriAlways.p;
    }
  }
  if (!img.smallOk && !img.spheres.empty())   // rfx_update_spheres can update this scene on the device
  {
    if ((rc = upload(ctx, ctx->dSphRadius, img.sphRadius, st)) != RFX_OK) return rc;
    if (!img.sphSlot.empty() &&
        ((rc = upload(ctx, ctx->dSphSlot, img.sphSlot, st)) != RFX_OK || (rc = upload(ctx, ctx->dSphLeafParent, img.sphLeafParent, st)) != RFX_OK ||
         (rc = upload(ctx, ctx->dSphPairParent, img.sphPairParent, st)) != RFX_OK ||
         (rc = ensure(ctx, ctx->dSphArrive, std::max<size_t>(img.sphPairParent.size(), 1))) != RFX_OK))
      return rc;
  }
  if (!img.triAlways.empty())
  {
    if ((rc = upload(ctx, ctx->dTriAlways, img.triAlways, st)) != RFX_OK) return rc;
    h.triAlways = ctx->dTriAlways.p;
  }
  if ((rc = upload(ctx, ctx->dBlob, img.blob, st)) != RFX_OK) return rc;
  CK(cudaStreamSynchronize(st));   // every copy above read from img, which the next upload overwrites
  img.small.byteLut = ctx->dLut.p;
  ctx->sceneDirty = false;
  return RFX_OK;
}

// number of block-preview origins (x % a == 0 && y % a == 0) with linear index < p, scan order
uint64_t originsBefore(uint64_t p, uint32_t W, uint32_t a)
{
  const uint64_t bw = (W + a - 1) / a;
  const uint64_t y = p / W, x = p % W;
  uint64_t n = ((y + a - 1) / a) * bw;            // complete origin rows below y
  if (y % a == 0) n += (x + a - 1) / a;           // origins left of x in this row
  return n;
}

// rank n Scene::trace calls on the randDir stream; the states land in ctx->dSampleStates.p (or nowhere when skipOnly)
int rankSamples(rfx_ctx * ctx, uint64_t n, bool skipOnly, cudaStream_t st, uint64_t ownPeriod = 0, uint32_t ownWorld = 0, uint32_t ownRank = 0)
{
  if (n == 0) return RFX_OK;
  const uint32_t nBlocks = rngBlocksFor(n);
  int rc;
  if (!skipOnly && (rc = ensure(ctx, ctx->dSampleStates, n)) != RFX_OK) return rc;
  RngWork w;
  w.stateIn = ctx->dRng.p + ctx->rngSlot;
  w.stateOut = ctx->dRng.p + (ctx->rngSlot ^ 1);
  w.prefix = ctx->dRngPrefix.p;
  w.locate = ctx->dRngLocate.p;
  w.sampleStates = skipOnly ? nullptr : ctx->dSampleStates.p;
  w.status = ctx->dStatus.p;
  w.n = n;
  w.nBlocks = nBlocks;
  w.ownPeriod = ownPeriod; w.ownWorld = ownWorld; w.ownRank = ownRank;
  if (ownWorld && !skipOnly)
  {
    const uint32_t bound = rngOwnBlocksBound(n, ownPeriod, ownWorld, nBlocks);
    if ((rc = ensure(ctx, ctx->dOwnBlocks, bound)) != RFX_OK) return rc;
    w.ownList = ctx->dOwnBlocks.p; w.ownListCap = (uint32_t)std::min<size_t>(ctx->dOwnBlocks.cap, 0xFFFFFFFFu);
  }
  ctx->stats.kernel_launches += launchRngRank(w, st);
  CK(cudaGetLastError());
  ctx->rngSlot ^= 1;
  return RFX_OK;
}

// advance the randDir stream by n Scene::trace calls without storing their states
int skipSamples(rfx_ctx * ctx, uint64_t n, cudaStream_t st)
{
  const uint64_t chunk = 1ull << 28;
  while (n > 0)
  {
    const uint64_t m = std::min(n, chunk);
    int rc;
    if ((rc = rankSamples(ctx, m, true, st)) != RFX_OK) return rc;
    n -= m;
  }
  return RFX_OK;
}

// The eye grid of the frame fp (EyeGrid), queued on st behind the kernels of the previous frame that still read the old one.  Cached
// per camera, image size, scene upload and sphere update.
int buildEyeGrid(rfx_ctx * ctx, const FrameParams & fp, cudaStream_t st)
{
  ctx->eyeGrid.cellStart = nullptr;
  if (!ctx->eyeGridOn || ctx->image.bvhDepth <= 0) return RFX_OK;
  uint32_t key[17];
  memcpy(key, fp.eye, 12); memcpy(key + 3, fp.view, 36);
  memcpy(key + 12, &fp.rz, 4); memcpy(key + 13, &fp.wHalf, 4); memcpy(key + 14, &fp.hHalf, 4);
  key[15] = fp.W; key[16] = fp.H;
  if (ctx->eyeValid && ctx->eyeSceneKey == ctx->sceneUploads && ctx->eyeSphereKey == ctx->sphereUpdates && !memcmp(key, ctx->eyeKey, sizeof(key)))
  {
    ctx->eyeGrid.cellStart = ctx->dEyeCells.p;
    return RFX_OK;
  }
  ctx->eyeValid = false;
  int nx = 0, ny = 0, rc;
  if (ctx->eyeGridDevice)
  {
    const PrimaryCamera cam = makePrimaryCamera(fp);
    if (!eyeGridDims(cam, fp.W, fp.H, nx, ny)) return RFX_OK;
    const size_t nS = ctx->image.spheres.size(), nCells = (size_t)nx * ny, words = (nS + 31) / 32;
    if (!ctx->eyeItemAlloc) ctx->eyeItemAlloc = std::max<size_t>(8 * nS + 2 * nCells, 1 << 16);   // grown after a build that did not fit
    if ((rc = ensure(ctx, ctx->dEyeCells, nCells + 2)) != RFX_OK || (rc = ensure(ctx, ctx->dEyeSpheres, ctx->eyeItemAlloc)) != RFX_OK ||
        (rc = ensure(ctx, ctx->dEyeIndex, ctx->eyeItemAlloc)) != RFX_OK || (rc = ensure(ctx, ctx->dEgSpan, std::max<size_t>(nS, 1))) != RFX_OK ||
        (rc = ensure(ctx, ctx->dEgRows, std::max<size_t>(ny * words, 1))) != RFX_OK) return rc;
    if (!ctx->dEyeFlags.p)
    {
      CK(ctx->dEyeFlags.alloc(2));
      CK(cudaMemsetAsync(ctx->dEyeFlags.p, 0, 2 * sizeof(uint32_t), st));
    }
    EyeGridBuild b;
    memset(&b, 0, sizeof(b));
    b.cam = cam; b.W = fp.W; b.H = fp.H; b.nx = nx; b.ny = ny;
    b.spheres = reinterpret_cast<const float4 *>(ctx->dBlob.p + reinterpret_cast<const SceneHeader *>(ctx->image.blob.data())->offSpheres);
    b.nSpheres = (int)nS;
    b.cells = ctx->dEyeCells.p; b.itemSphere = ctx->dEyeSpheres.p; b.itemIndex = ctx->dEyeIndex.p;
    size_t cap = std::min(ctx->dEyeSpheres.cap, ctx->dEyeIndex.cap);
    if (ctx->eyeItemLimit > 0) cap = std::min<size_t>(cap, (size_t)ctx->eyeItemLimit);
    b.itemCap = (uint32_t)std::min<size_t>(cap, UINT32_MAX);
    b.flags = ctx->dEyeFlags.p;
    b.xSpan = ctx->dEgSpan.p; b.rowMask = ctx->dEgRows.p; b.maskWords = (int)words;
    const int nl = launchEyeGridBuild(b, st);
    if (!nl) return fail(ctx, RFX_ERR_CUDA, "buildEyeGrid: the row masks could not be cleared");
    ctx->stats.kernel_launches += nl;
    CK(cudaGetLastError());
  }
  else
  {
    std::vector<uint32_t> cells;
    std::vector<float4> items;
    std::vector<int> index;
    if (!binEyeGrid(fp, ctx->image.spheres, nx, ny, cells, items, index)) return RFX_OK;
    cells.push_back(0u);                      // the drop word: the whole grid is uploaded
    if ((rc = upload(ctx, ctx->dEyeCells, cells, st)) != RFX_OK || (rc = upload(ctx, ctx->dEyeSpheres, items, st)) != RFX_OK ||
        (rc = upload(ctx, ctx->dEyeIndex, index, st)) != RFX_OK) return rc;
  }
  ctx->eyeGrid.cellStart = ctx->dEyeCells.p; ctx->eyeGrid.itemSphere = ctx->dEyeSpheres.p; ctx->eyeGrid.itemIndex = ctx->dEyeIndex.p;
  ctx->eyeGrid.nx = nx; ctx->eyeGrid.ny = ny; ctx->eyeGrid.shift = EYE_GRID_SHIFT;
  memcpy(ctx->eyeKey, key, sizeof(key)); ctx->eyeSceneKey = ctx->sceneUploads; ctx->eyeSphereKey = ctx->sphereUpdates; ctx->eyeValid = true;
  ctx->eyeGridBuilds++;
  return RFX_OK;
}

// At a synchronising call: after a device build that did not fit its item region (EyeGridBuild::flags), grow the region and forget the
// cached grid, so the next render builds it again.
int growEyeGrid(rfx_ctx * ctx)
{
  if (!ctx->dEyeFlags.p) return RFX_OK;
  uint32_t need = 0;
  CK(cudaMemcpy(&need, ctx->dEyeFlags.p, sizeof(need), cudaMemcpyDeviceToHost));
  if (!need) return RFX_OK;
  ctx->eyeValid = false;
  if (need > std::min(ctx->dEyeSpheres.cap, ctx->dEyeIndex.cap))
  {
    const size_t alloc = (size_t)need + need / 2;
    CK(cudaFree(ctx->dEyeSpheres.p)); ctx->dEyeSpheres.p = nullptr; ctx->dEyeSpheres.cap = 0;
    CK(cudaFree(ctx->dEyeIndex.p)); ctx->dEyeIndex.p = nullptr; ctx->dEyeIndex.cap = 0;
    CK(ctx->dEyeSpheres.alloc(alloc));
    CK(ctx->dEyeIndex.alloc(alloc));
    ctx->eyeItemAlloc = alloc;
    ctx->eyeRendered = false;                 // (the grid of the last render lived in the old region)
  }
  CK(cudaMemset(ctx->dEyeFlags.p, 0, sizeof(uint32_t)));
  return RFX_OK;
}

// Fills w.order for a fast-kernel launch and remembers what the launch will have recorded (see TileOrder).  History is
// only reused by a launch over exactly the same grid; any other launch of the fast kernel starts a new history.
int armTileOrder(rfx_ctx * ctx, TraceWork & w, cudaStream_t st)
{
  w.order = TileOrder();
  const uint32_t grid = ctx->image.smallOk && ctx->forcePath < 2 ? fastGridSize(w) : 0;
  if (!ctx->tileOrdering || grid == 0 || grid > (1u << 22)) { ctx->tileHistory = false; return RFX_OK; }
  const uint64_t key[4] = { ((uint64_t)w.fp.W << 32) | w.fp.H, w.fp.p0, w.fp.p1,
                            ((uint64_t)w.fp.stripRows << 40) | ((uint64_t)w.fp.stripWorld << 20) | w.fp.stripRank };
  int rc;
  const int out = ctx->tileSlot, in = out ^ 1;
  const int cOut = ctx->tileCountSlot, cIn = (cOut + 2) % 3, cNext = (cOut + 1) % 3;
  if (ctx->tileRecordPeriod > 1 && ctx->tileHistory && memcmp(key, ctx->tileKey, sizeof(key)) == 0 && ctx->tileReuse + 1 < ctx->tileRecordPeriod &&
      ctx->dTileLists[in].cap >= (size_t)grid * TILE_CLASSES)
  {
    // replay the last recording without recording again (the kernel then has no CTA barrier and no atomic at its end)
    w.order.inLists = ctx->dTileLists[in].p;
    w.order.inCounts = ctx->dTileCounts.p + cIn * TILE_CLASSES;
    w.order.capacity = grid;
    ctx->tileReuse++;
    return RFX_OK;
  }
  ctx->tileReuse = 0;
  if ((rc = ensure(ctx, ctx->dTileLists[out], (size_t)grid * TILE_CLASSES)) != RFX_OK) return rc;
  if (!ctx->dTileCounts.p)
  {
    CK(ctx->dTileCounts.alloc(3 * TILE_CLASSES));
    CK(cudaMemsetAsync(ctx->dTileCounts.p, 0, 3 * TILE_CLASSES * sizeof(uint32_t), st));
  }
  w.order.outLists = ctx->dTileLists[out].p;
  w.order.outCounts = ctx->dTileCounts.p + cOut * TILE_CLASSES;
  w.order.zeroCounts = ctx->dTileCounts.p + cNext * TILE_CLASSES;
  w.order.capacity = grid;
  if (ctx->tileHistory && memcmp(key, ctx->tileKey, sizeof(key)) == 0 && ctx->dTileLists[in].cap >= (size_t)grid * TILE_CLASSES)
  {
    w.order.inLists = ctx->dTileLists[in].p;
    w.order.inCounts = ctx->dTileCounts.p + cIn * TILE_CLASSES;
  }
  ctx->tileCountSlot = cNext;
  memcpy(ctx->tileKey, key, sizeof(key));
  ctx->tileHistory = true;
  ctx->tileSlot = in;
  return RFX_OK;
}

// the K2 work record of pixels [p0, p1) of the frame latched by render_begin
TraceWork traceWork(const rfx_ctx * ctx, uint64_t p0, uint64_t p1, uint64_t firstRank, const uint32_t * sampleStates, float * image, uint32_t * argbOut)
{
  TraceWork w;
  w.sceneBlob = ctx->dBlob.p;
  w.sceneBytes = (uint32_t)ctx->image.blob.size();
  w.fp = ctx->snap;
  w.fp.p0 = p0; w.fp.p1 = p1; w.fp.firstRank = firstRank;
  w.fp.seedRender = ctx->seedRender;
  w.sampleStates = sampleStates;
  w.image = image;
  w.argbOut = argbOut;
  w.sigOut = ctx->sigOn ? ctx->dSig.p : nullptr;
  w.counters = ctx->dCounters.p;
  w.lightGrids = ctx->image.lightGridsBuilt > 0 && std::count(ctx->lightGrid.begin(), ctx->lightGrid.end(), 1) > 0;   // (the lights with a grid now)
  w.triBvh = ctx->image.triBvhTris > 0;
  w.far = ctx->image.far;
  return w;
}

// while profiling, a K2 launch is bracketed by a (start, stop) pair of pooled events: records the start and hands out the stop
// (nullptr when not profiling)
int profileStart(rfx_ctx * ctx, cudaStream_t st, cudaEvent_t & stop)
{
  stop = nullptr;
  if (!ctx->profiling) return RFX_OK;
  if (ctx->evUsed + 2 > ctx->evPool.size())
    for (int i = 0; i < 2; i++) { cudaEvent_t e; CK(cudaEventCreate(&e)); ctx->evPool.push_back(e); }
  const cudaEvent_t start = ctx->evPool[ctx->evUsed++];
  stop = ctx->evPool[ctx->evUsed++];
  CK(cudaEventRecord(start, st));
  return RFX_OK;
}

// render pixels [p0, p1) of the frame latched by render_begin
// preStates: random states already ranked for exactly [p0, p1) (batch path ranks several frames per K1 pass); NULL = rank here
// frames > 1: that many whole frames of the latched camera in one launch (fastBatchOk), states and ARGB frames one after the other
int renderRange(rfx_ctx * ctx, uint64_t p0, uint64_t p1, uint32_t * argbOut, bool writeImage, cudaStream_t st,
                const uint32_t * preStates = nullptr, uint32_t frames = 1)
{
  int rc;
  const int sn = ctx->sampleNum;
  uint64_t cur = p0;
  while (cur < p1)
  {
    uint64_t end, nCalls, firstRank = 0;
    if (sn > 0)
    {
      const uint64_t per = (uint64_t)sn * sn;
      uint64_t pix = ctx->maxCallsPerLaunch / per;
      if (pix < 1) pix = 1;
      if (cur % ctx->W == 0 && pix >= ctx->W) pix -= pix % ctx->W;   // whole rows keep the chunk on the tiled fast kernel
      end = preStates ? p1 : std::min(p1, cur + pix);
      nCalls = (end - cur) * per;
    }
    else
    {
      const uint32_t a = (uint32_t)(-sn);
      end = p1;   // at most one call per a*a pixels: never exceeds the cap for any sane image
      firstRank = originsBefore(cur, ctx->W, a);
      nCalls = originsBefore(end, ctx->W, a) - firstRank;
    }
    if (nCalls > 0)
    {
      if (!preStates && (rc = rankSamples(ctx, nCalls, false, st)) != RFX_OK) return rc;
      TraceWork w = traceWork(ctx, cur, end, firstRank, preStates ? preStates : ctx->dSampleStates.p, writeImage ? ctx->dImage.p : nullptr, argbOut);
      w.frames = frames;
      cudaEvent_t evStop;
      if ((rc = profileStart(ctx, st, evStop)) != RFX_OK) return rc;
      const bool useSmall = ctx->forcePath >= 2 ? false : ctx->image.smallOk;
      if (useSmall && (rc = armTileOrder(ctx, w, st)) != RFX_OK) return rc;
      if (useSmall)
      {
        uint32_t fastGrid = 0;
        const int nl = launchTraceSmall(ctx->image.small, w, st, &fastGrid);
        ctx->stats.kernel_launches += nl;
        (fastGrid ? ctx->stats.launches_small_fast : ctx->stats.launches_small_any) += nl;
      }
      else
      {
        const uint64_t wavePixels = (ctx->blobWavefront && ctx->forcePath != 3) ? blobWavePixels(w) : 0;
        if (wavePixels)
        {
          if ((rc = ensure(ctx, ctx->dQueue, (size_t)wavePixels * 4)) != RFX_OK) return rc;   // 64-byte records
          if (!ctx->dQueueCtl.p) CK(ctx->dQueueCtl.alloc(2));
        }
        if ((rc = buildEyeGrid(ctx, w.fp, st)) != RFX_OK) return rc;
        w.eyeGrid = ctx->eyeGrid;
        ctx->eyeRendered = true; ctx->eyeFp = w.fp; ctx->eyeUsed = ctx->eyeGrid;
        int nl = ctx->forcePath == 3 ? 0 : launchTraceBlobFast(w, st, wavePixels ? ctx->dQueue.p : nullptr, ctx->dQueueCtl.p, (uint32_t)ctx->prop.multiProcessorCount * 8u,
                                                               ctx->blobWavefront, ctx->blobSmemBvh ? ctx->image.bvhFloat4 : 0u);
        if (nl) ctx->stats.launches_blob_fast += nl;
        else { nl = launchTraceBlobAny(w, st); ctx->stats.launches_blob_any += nl; }
        ctx->stats.kernel_launches += nl;
      }
      if (evStop) CK(cudaEventRecord(evStop, st));
      CK(cudaGetLastError());
      ctx->stats.samples += nCalls * frames;
      if (ctx->snap.jitter && sn > 0) ctx->seedRender = lcgJumpHost(ctx->seedRender, 2 * (end - cur));
    }
    cur = end;
  }
  return RFX_OK;
}

void meshBox(HostMesh & m)
{
  float * b = m.box;
  for (int k = 0; k < 3; k++) { b[k] = FLT_MAX; b[3 + k] = -FLT_MAX; }
  for (size_t i = 0; i < m.xyz.size(); i++) { b[i % 3] = std::min(b[i % 3], m.xyz[i]); b[3 + i % 3] = std::max(b[3 + i % 3], m.xyz[i]); }
}

// Whether the light grids (if any) were built for a drop-point box that still holds every object: the triangles outside meshes,
// the spheres (their current box: sph, or img.dropSpheres) and the meshes' current boxes.
bool gridBoxHolds(const rfx_ctx * ctx, const double * sph = nullptr)
{
  const SceneImage & img = ctx->image;
  if (!img.lightGridsBuilt) return true;
  if (!sph) sph = img.dropSpheres;
  double b[6];
  for (int k = 0; k < 3; k++) { b[k] = std::min(img.dropTris[k], sph[k]); b[3 + k] = std::max(img.dropTris[3 + k], sph[3 + k]); }
  for (const HostMesh & o : ctx->scene.meshes)
    for (int k = 0; k < 3; k++) { b[k] = std::min(b[k], (double)o.box[k]); b[3 + k] = std::max(b[3 + k], (double)o.box[3 + k]); }
  padDropBox(b);
  for (int k = 0; k < 3; k++)
    if (!(b[k] >= img.gridBox[k] && b[3 + k] <= img.gridBox[3 + k])) return false;
  return true;
}

// Light li's grid after it or the spheres moved (a scene whose flatten built grids): built on the device over the flatten's box when the
// light is far from it, else a NULL header.  Queued on st.
int updateLightGrid(rfx_ctx * ctx, size_t li, cudaStream_t st)
{
  const SceneImage & img = ctx->image;
  const double blo[3] = { img.gridBox[0], img.gridBox[1], img.gridBox[2] }, bhi[3] = { img.gridBox[3], img.gridBox[4], img.gridBox[5] };
  LightFrame f;
  ctx->lightGrid[li] = lightFrame(ctx->scene.lights[li], blo, bhi, f);
  if (!ctx->lightGrid[li])
  {
    CK(cudaMemsetAsync(ctx->dLightGrids.p + li, 0, sizeof(LightGrid), st));
    CK(cudaMemsetAsync(ctx->dGridFlags.p + 1 + li, 0, sizeof(uint32_t), st));
    return RFX_OK;
  }
  const SceneHeader & h = *reinterpret_cast<const SceneHeader *>(img.blob.data());
  LightGridBuild b;
  memset(&b, 0, sizeof(b));
  b.f = f;
  b.spheres = reinterpret_cast<const float4 *>(ctx->dBlob.p + h.offSpheres);
  b.radius = ctx->dSphRadius.p;
  b.prims = ctx->dBvhPrims.p;
  b.nSlots = (int)img.sphBvh.prims.size();
  b.nPrims = img.bvhSpheres;
  b.R = img.sphR;
  b.header = ctx->dLightGrids.p + li;
  b.cells = ctx->dGridCells.p + li * LIGHT_GRID_CELLS;
  b.itemSphere = ctx->dGridSpheres.p + li * ctx->gridItemAlloc;
  b.itemIndex = ctx->dGridIndex.p + li * ctx->gridItemAlloc;
  b.itemCap = ctx->gridItemCap;
  b.need = ctx->dGridFlags.p;
  b.dropped = ctx->dGridFlags.p + 1 + li;
  b.disc = ctx->dLgDisc.p; b.span = ctx->dLgSpan.p; b.blockSum = ctx->dLgBlockSum.p; b.red = ctx->dLgRed.p; b.dims = ctx->dLgDims.p;
  ctx->stats.kernel_launches += launchLightGridBuild(b, st);
  CK(cudaGetLastError());
  return RFX_OK;
}

// At a synchronising call: a device build that did not fit its item region (LightGridBuild::need) grows every light's regions for the
// later builds.  The grids already built move with their regions; the dropped one returns at its light's next build.
int growLightGrids(rfx_ctx * ctx)
{
  const SceneImage & img = ctx->image;
  if (ctx->sceneDirty || !img.lightGridsBuilt || !ctx->dGridFlags.p) return RFX_OK;   // (a pending flatten sizes its own regions)
  uint32_t need = 0;
  CK(cudaMemcpy(&need, ctx->dGridFlags.p, sizeof(need), cudaMemcpyDeviceToHost));
  if (need <= ctx->gridItemAlloc) return RFX_OK;
  const size_t nL = ctx->scene.lights.size(), old = ctx->gridItemAlloc, alloc = (size_t)need + need / 2;
  DevArray<float4> sp;
  DevArray<int> ix;
  CK(sp.alloc(nL * alloc));
  CK(ix.alloc(nL * alloc));
  CK(cudaMemcpy2D(sp.p, alloc * sizeof(float4), ctx->dGridSpheres.p, old * sizeof(float4), old * sizeof(float4), nL, cudaMemcpyDeviceToDevice));
  CK(cudaMemcpy2D(ix.p, alloc * sizeof(int), ctx->dGridIndex.p, old * sizeof(int), old * sizeof(int), nL, cudaMemcpyDeviceToDevice));
  std::vector<LightGrid> hdr(nL);
  CK(cudaMemcpy(hdr.data(), ctx->dLightGrids.p, nL * sizeof(LightGrid), cudaMemcpyDeviceToHost));
  for (size_t li = 0; li < nL; li++)
    if (hdr[li].cellStart) { hdr[li].itemSphere = sp.p + li * alloc; hdr[li].itemIndex = ix.p + li * alloc; }
  CK(cudaMemcpy(ctx->dLightGrids.p, hdr.data(), nL * sizeof(LightGrid), cudaMemcpyHostToDevice));
  CK(cudaFree(ctx->dGridSpheres.p)); CK(cudaFree(ctx->dGridIndex.p));
  ctx->dGridSpheres.p = sp.p; ctx->dGridSpheres.cap = sp.cap; sp.p = nullptr; sp.cap = 0;
  ctx->dGridIndex.p = ix.p; ctx->dGridIndex.cap = ix.cap; ix.p = nullptr; ix.cap = 0;
  ctx->gridItemAlloc = alloc;
  setGridItemCap(ctx);
  CK(cudaMemset(ctx->dGridFlags.p, 0, sizeof(uint32_t)));
  return RFX_OK;
}

// lights whose shadow queries use a grid: the headers on the device that are not NULL (after a synchronisation)
int countLightGrids(rfx_ctx * ctx, uint64_t & n)
{
  n = 0;
  if (!ctx->image.lightGridsBuilt || ctx->image.grids.empty()) return RFX_OK;
  std::vector<LightGrid> hdr(ctx->image.grids.size());
  CK(cudaMemcpy(hdr.data(), ctx->dLightGrids.p, hdr.size() * sizeof(LightGrid), cudaMemcpyDeviceToHost));
  for (const LightGrid & g : hdr) n += g.cellStart != nullptr;
  return RFX_OK;
}

// recompute envColor from the lights' current colours and powers as Scene's constructor and addLight do (Scene.cpp:12,54): the
// ambient term, then colour * (unclamped) power added light after light in insertion order
void recomputeEnv(HostScene & s)
{
  for (int k = 0; k < 3; k++) s.env[k] = s.ambient[k] * s.ambientPower;
  for (size_t i = 0; i < s.lights.size(); i++)
  {
    const Light & L = s.lights[i];
    const float rgb[3] = { L.r, L.g, L.b };
    for (int k = 0; k < 3; k++) s.env[k] = s.env[k] + rgb[k] * s.lightPower[i];
  }
}

// Whether the structures of the last flatten still serve the scene after mesh m moved (rfx_update_mesh updates it on the device):
// a blob scene whose hierarchies' margins were sized for a reach box that still holds m's vertices (every drop point on them), and
// whose light grids were built for a drop-point box that still holds every object.
bool deviceUpdateValid(const rfx_ctx * ctx, const HostMesh & m)
{
  const SceneImage & img = ctx->image;
  if (img.smallOk || img.meshes.size() != ctx->scene.meshes.size()) return false;
  if (img.bvhDepth > 0 || img.triBvhTris > 0)
    for (int k = 0; k < 3; k++)
      if (!(m.box[k] >= img.reach[k] && m.box[3 + k] <= img.reach[3 + k])) return false;
  return gridBoxHolds(ctx);
}

int checkStatus(rfx_ctx * ctx)
{
  int status = 0;
  CK(cudaMemcpy(&status, ctx->dStatus.p, sizeof(int), cudaMemcpyDeviceToHost));
  if (status) return fail(ctx, RFX_ERR_RNG, "random-stream ranking ran out of over-provisioned draws");
  return RFX_OK;
}

} // namespace

// =====================================================================================================================
extern "C"
{

const char * rfx_version(void) { return "reflaxman_b200 0.1 (sm_100a)"; }

int rfx_create(rfx_ctx ** out, int device)
{
  rfx_ctx * ctx = nullptr;   // for CK
  if (!out) return fail(nullptr, RFX_ERR_ARG, "rfx_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return fail(nullptr, RFX_ERR_NODEV, std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= n) return fail(nullptr, RFX_ERR_ARG, "rfx_create: bad device ordinal");
  cudaDeviceProp prop;
  CK(cudaSetDevice(device));
  CK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(nullptr, RFX_ERR_NODEV, std::string("device is sm_") + std::to_string(prop.major) + std::to_string(prop.minor) +
                ", this library carries sm_100a code only (there is no CPU fallback)");
  ctx = new rfx_ctx();
  ctx->device = device;
  ctx->prop = prop;
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  memset(&ctx->snap, 0, sizeof(ctx->snap));
  cudaError_t err = cudaSuccess;
  auto step = [&](cudaError_t r) { if (err == cudaSuccess) err = r; };
  step(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) step(cudaStreamCreateWithFlags(&ctx->copyStream[i], cudaStreamNonBlocking));
  if (initRngTables() != 0) step(cudaErrorUnknown);
  step(ctx->dRng.alloc(2));
  step(ctx->dRngPrefix.alloc(3 * (size_t)(RNG_CLASS_BLOCKS + 1)));
  step(ctx->dRngLocate.alloc(1));
  if (err == cudaSuccess)
  {
    // accept counts of the whole LCG cycle: ~5 ms once per context; every later ranking or skip is a table lookup away
    DevArray<uint32_t> counts;
    step(counts.alloc(3 * (size_t)RNG_CLASS_BLOCKS));
    if (err == cudaSuccess) { launchRngTable(counts.p, ctx->dRngPrefix.p, ctx->stream); step(cudaStreamSynchronize(ctx->stream)); step(cudaGetLastError()); }
  }
  step(ctx->dStatus.alloc(1));
  step(ctx->dCounters.alloc(64));
  step(ctx->dLut.alloc(256));
  for (int i = 0; i < rfx_ctx::FRAME_SLOTS; i++)
  {
    step(cudaEventCreateWithFlags(&ctx->evRendered[i], cudaEventDisableTiming));
    step(cudaEventCreateWithFlags(&ctx->evCopied[i], cudaEventDisableTiming));
  }
  if (err == cudaSuccess)
  {
    float lut[256];
    for (int i = 0; i < 256; i++) lut[i] = float(i) / 255.0f;   // Color(ARGB), Color.cpp:11-13
    const uint32_t seeds[2] = { 12345u, 12345u };
    step(cudaMemcpy(ctx->dLut.p, lut, sizeof(lut), cudaMemcpyHostToDevice));
    step(cudaMemcpy(ctx->dRng.p, seeds, sizeof(seeds), cudaMemcpyHostToDevice));
    step(cudaMemset(ctx->dStatus.p, 0, sizeof(int)));
    step(cudaMemset(ctx->dCounters.p, 0, 64 * sizeof(unsigned long long)));
  }
  if (err != cudaSuccess)
  {
    std::string msg = std::string("rfx_create: ") + cudaGetErrorString(err);
    rfx_destroy(ctx);
    return fail(nullptr, RFX_ERR_CUDA, msg);
  }
  *out = ctx;
  return RFX_OK;
}

void rfx_destroy(rfx_ctx * ctx)
{
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  for (HostTex & t : ctx->scene.tex) if (t.dev) cudaFree(t.dev);
  for (cudaEvent_t e : ctx->evPool) cudaEventDestroy(e);
  for (int i = 0; i < rfx_ctx::FRAME_SLOTS; i++)
  {
    if (ctx->evRendered[i]) cudaEventDestroy(ctx->evRendered[i]);
    if (ctx->evCopied[i]) cudaEventDestroy(ctx->evCopied[i]);
  }
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  for (int i = 0; i < 2; i++) if (ctx->copyStream[i]) cudaStreamDestroy(ctx->copyStream[i]);
  delete ctx;   // frees the device arrays
}

const char * rfx_last_error(const rfx_ctx * ctx) { return ctx ? ctx->err.c_str() : g_createError.c_str(); }

int rfx_get_device_info(const rfx_ctx * ctx, rfx_device_info * out)
{
  if (!ctx || !out) return RFX_ERR_ARG;
  memset(out, 0, sizeof(*out));
  out->device = ctx->device;
  out->sm_count = ctx->prop.multiProcessorCount;
  out->cc_major = ctx->prop.major; out->cc_minor = ctx->prop.minor;
  int khz = 0;
  cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, ctx->device);
  out->clock_khz = khz;
  out->total_mem = ctx->prop.totalGlobalMem;
  strncpy(out->name, ctx->prop.name, sizeof(out->name) - 1);
  return RFX_OK;
}

// ---------------------------------------------------------------------------------------------------------- scene
int rfx_scene_reset(rfx_ctx * ctx, const float ambient_rgb[3], float ambient_power)
{
  if (!ctx || !ambient_rgb) return fail(ctx, RFX_ERR_ARG, "rfx_scene_reset: NULL argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  for (HostTex & t : ctx->scene.tex) if (t.dev) cudaFree(t.dev);
  ctx->scene.tex.clear(); ctx->scene.objs.clear(); ctx->scene.lights.clear(); ctx->scene.lightPower.clear(); ctx->scene.meshes.clear();
  ctx->scene.skyTex = -1;
  for (int i = 0; i < 3; i++) { ctx->scene.extraOrigins[i] = FLT_MAX; ctx->scene.extraOrigins[3 + i] = -FLT_MAX; }
  for (int i = 0; i < 3; i++)
  {
    ctx->scene.ambient[i] = ambient_rgb[i];
    ctx->scene.env[i] = ambient_rgb[i] * ambient_power;   // envColor(diffLightColor * diffLightPower), Scene.cpp:12
  }
  ctx->scene.ambientPower = ambient_power;
  ctx->sceneDirty = true;
  return RFX_OK;
}

int rfx_add_light(rfx_ctx * ctx, const float o[3], float radius, const float rgb[3], float power)
{
  if (!ctx || !o || !rgb) return fail(ctx, RFX_ERR_ARG, "rfx_add_light: NULL argument");
  if (radius <= VSN) radius = VSN;                              // Scene.cpp:51-52
  for (int i = 0; i < 3; i++) ctx->scene.env[i] = ctx->scene.env[i] + rgb[i] * power;   // envColor += color * power, Scene.cpp:54
  Light l;
  l.ox = o[0]; l.oy = o[1]; l.oz = o[2]; l.radius = radius;
  l.r = rgb[0]; l.g = rgb[1]; l.b = rgb[2];
  l.power = clampf(power, 0.0f, 1.0f);                          // OmniLight.cpp:13
  ctx->scene.lights.push_back(l);
  ctx->scene.lightPower.push_back(power);
  ctx->sceneDirty = true;
  return (int)ctx->scene.lights.size() - 1;
}

int rfx_update_lights(rfx_ctx * ctx, uint32_t n, const int32_t * lights, const float * records)
{
  if (!ctx || !lights || !records || n == 0) return fail(ctx, RFX_ERR_ARG, "rfx_update_lights: NULL argument or no light");
  HostScene & s = ctx->scene;
  for (uint32_t i = 0; i < n; i++)
    if (lights[i] < 0 || lights[i] >= (int)s.lights.size())
      return fail(ctx, RFX_ERR_ARG, "rfx_update_lights: light " + std::to_string(lights[i]) + " is not a light of this scene");
  // the host records, as rfx_add_light makes them (a later entry for the same light overwrites an earlier one)
  std::vector<char> moved(s.lights.size(), 0);
  for (uint32_t i = 0; i < n; i++)
  {
    const float * r = records + 8 * (size_t)i;
    Light & l = s.lights[lights[i]];
    float radius = r[3];
    if (radius <= VSN) radius = VSN;                              // Scene.cpp:51-52
    l.ox = r[0]; l.oy = r[1]; l.oz = r[2]; l.radius = radius;
    l.r = r[4]; l.g = r[5]; l.b = r[6];
    l.power = clampf(r[7], 0.0f, 1.0f);                           // OmniLight.cpp:13
    s.lightPower[lights[i]] = r[7];
    moved[lights[i]] = 1;
  }
  recomputeEnv(s);
  if (ctx->sceneDirty || ctx->image.smallOk) { ctx->sceneDirty = true; return 0; }
  SceneImage & img = ctx->image;
  SceneHeader & h = *reinterpret_cast<SceneHeader *>(img.blob.data());
  // Light positions enter neither the reach box nor the hierarchies' margins nor the eye grid: only the light grids can change.  A
  // light that becomes far in a scene whose flatten built no grid (no header array on the device) re-flattens the scene.
  if (!img.lightGridsBuilt && img.bvhDepth > 0 && s.lightGridsOn && h.nPlanes == 0)
  {
    const double blo[3] = { img.gridBox[0], img.gridBox[1], img.gridBox[2] }, bhi[3] = { img.gridBox[3], img.gridBox[4], img.gridBox[5] };
    LightFrame f;
    for (size_t li = 0; li < moved.size(); li++)
      if (moved[li] && lightFrame(s.lights[li], blo, bhi, f)) { ctx->sceneDirty = true; return 0; }
  }
  CK(cudaSetDevice(ctx->device));
  // the stream the renders use: the update is ordered after the frames already queued there
  cudaStream_t st = ctx->lastStream ? ctx->lastStream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  // the records and envColor into the blob (the host copy first: the copies read from it, staged before they return)
  memcpy(img.blob.data() + h.offLights, s.lights.data(), sizeof(Light) * s.lights.size());
  memcpy(h.env, s.env, sizeof(h.env));
  CK(cudaMemcpyAsync(ctx->dBlob.p + h.offLights, img.blob.data() + h.offLights, sizeof(Light) * s.lights.size(), cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(ctx->dBlob.p + offsetof(SceneHeader, env), h.env, sizeof(h.env), cudaMemcpyHostToDevice, st));
  ctx->stats.h2d_bytes += sizeof(Light) * s.lights.size() + sizeof(h.env);
  if (img.lightGridsBuilt)
    for (size_t li = 0; li < moved.size(); li++)
      if (moved[li] && (rc = updateLightGrid(ctx, li, st)) != RFX_OK) return rc;
  return 1;
}

int rfx_add_sphere(rfx_ctx * ctx, const float c[3], float radius, int mtype, const float rgb[3], float refl, float transp)
{
  if (!ctx || !c || !rgb) return fail(ctx, RFX_ERR_ARG, "rfx_add_sphere: NULL argument");
  if (radius <= VSN) radius = VSN;                              // Scene.cpp:33-34
  HostObj o;
  memset(&o, 0, sizeof(o));
  o.kind = 0;
  o.mat = makeMaterial(mtype, rgb, refl, transp, (int)ctx->scene.objs.size());
  o.center[0] = c[0]; o.center[1] = c[1]; o.center[2] = c[2];
  o.sqRadius = radius * radius;                                 // Sphere.cpp:19
  o.radius = radius;
  ctx->scene.objs.push_back(o);
  ctx->sceneDirty = true;
  return (int)ctx->scene.objs.size() - 1;
}

int rfx_add_triangle(rfx_ctx * ctx, const float v[9], int mtype, const float rgb[3], float refl, float transp)
{
  if (!ctx || !v || !rgb) return fail(ctx, RFX_ERR_ARG, "rfx_add_triangle: NULL argument");
  HostObj o;
  memset(&o, 0, sizeof(o));
  o.kind = 1;
  o.mat = makeMaterial(mtype, rgb, refl, transp, (int)ctx->scene.objs.size());
  setupTriangle(v, o.tri);                                      // Triangle.cpp:11-21
  memcpy(o.triVerts, v, sizeof(o.triVerts));
  ctx->scene.objs.push_back(o);
  ctx->sceneDirty = true;
  return (int)ctx->scene.objs.size() - 1;
}

int rfx_add_mesh(rfx_ctx * ctx, uint32_t n_vertices, const float * xyz, uint32_t n_tris, const uint32_t * idx, int mtype, const float rgb[3],
                 float refl, float transp)
{
  if (!ctx || !xyz || !idx || !rgb || n_tris == 0) return fail(ctx, RFX_ERR_ARG, "rfx_add_mesh: NULL argument or no triangle");
  if ((uint64_t)ctx->scene.objs.size() + n_tris > (uint64_t)INT32_MAX) return fail(ctx, RFX_ERR_ARG, "rfx_add_mesh: too many objects");
  for (uint64_t k = 0; k < 3ull * n_tris; k++)
    if (idx[k] >= n_vertices) return fail(ctx, RFX_ERR_ARG, "rfx_add_mesh: vertex index out of range");
  const int first = (int)ctx->scene.objs.size();
  ctx->scene.objs.reserve(ctx->scene.objs.size() + n_tris);
  for (uint32_t k = 0; k < n_tris; k++)
  {
    float v[9];
    for (int j = 0; j < 3; j++) memcpy(v + 3 * j, xyz + 3 * (size_t)idx[3 * (size_t)k + j], 12);
    const int rc = rfx_add_triangle(ctx, v, mtype, rgb, refl, transp);
    if (rc < 0) return rc;
  }
  HostMesh m;
  m.first = first;
  m.idx.assign(idx, idx + 3 * (size_t)n_tris);
  m.xyz.assign(xyz, xyz + 3 * (size_t)n_vertices);
  meshBox(m);
  ctx->scene.meshes.push_back(std::move(m));
  return first;
}

int rfx_update_mesh(rfx_ctx * ctx, int first, const float * xyz)
{
  if (!ctx || !xyz) return fail(ctx, RFX_ERR_ARG, "rfx_update_mesh: NULL argument");
  HostScene & s = ctx->scene;
  size_t mi = 0;
  while (mi < s.meshes.size() && s.meshes[mi].first != first) mi++;
  if (mi == s.meshes.size()) return fail(ctx, RFX_ERR_ARG, "rfx_update_mesh: first does not start a mesh of this scene");
  HostMesh & m = s.meshes[mi];
  memcpy(m.xyz.data(), xyz, m.xyz.size() * sizeof(float));
  meshBox(m);
  m.stale = true;   // the host records follow at the next flatten (refreshMeshes)
  if (ctx->sceneDirty || !deviceUpdateValid(ctx, m)) { ctx->sceneDirty = true; return 0; }

  const SceneImage & img = ctx->image;
  const SceneImage::MeshImage & im = img.meshes[mi];
  CK(cudaSetDevice(ctx->device));
  // the stream the renders use: the update is ordered after the frames already queued there
  cudaStream_t st = ctx->lastStream ? ctx->lastStream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK || (rc = ensure(ctx, ctx->dVerts, m.xyz.size())) != RFX_OK) return rc;
  CK(cudaMemcpyAsync(ctx->dVerts.p, m.xyz.data(), m.xyz.size() * sizeof(float), cudaMemcpyHostToDevice, st));   // (staged before the call returns)
  ctx->stats.h2d_bytes += m.xyz.size() * sizeof(float);
  const SceneHeader & h = *reinterpret_cast<const SceneHeader *>(img.blob.data());
  MeshUpdate u;
  memset(&u, 0, sizeof(u));
  u.tris = reinterpret_cast<Triangle *>(ctx->dBlob.p + h.offTris);
  u.header = reinterpret_cast<SceneHeader *>(ctx->dBlob.p);
  u.xyz = ctx->dVerts.p;
  u.idx = ctx->dMeshIdx.p + im.idxOff;
  u.triBase = im.triBase; u.nTris = (int)im.nTris;
  if (!img.triSlot.empty())
  {
    u.triLeaf = ctx->dTriNodes.p; u.triPairs = ctx->dTriNodes.p + img.triBvh.leafFloat4;
    u.triPrims = ctx->dTriPrims.p; u.triSlot = ctx->dTriSlot.p;
    u.leafParent = ctx->dLeafParent.p; u.pairParent = ctx->dPairParent.p;
    u.arrive = ctx->dArrive.p;
    u.nLeaves = (int)img.leafParent.size();
    u.red = ctx->dMeshRed.p;
    u.far = img.far;
    u.triAlways = ctx->dTriAlways.p;
    u.inAlways = ctx->dInAlways.p;
    CK(cudaMemcpyAsync(ctx->dMeshRed.p, ctx->dMeshRed.p + 7, 7 * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, st));
    if (!img.pairParent.empty()) CK(cudaMemsetAsync(ctx->dArrive.p, 0, img.pairParent.size() * sizeof(uint32_t), st));
  }
  ctx->stats.kernel_launches += launchMeshUpdate(u, st);
  CK(cudaGetLastError());
  return 1;
}

int rfx_update_spheres(rfx_ctx * ctx, uint32_t n, const int32_t * objects, const float * spheres)
{
  if (!ctx || !objects || !spheres || n == 0) return fail(ctx, RFX_ERR_ARG, "rfx_update_spheres: NULL argument or no sphere");
  HostScene & s = ctx->scene;
  for (uint32_t i = 0; i < n; i++)
    if (objects[i] < 0 || objects[i] >= (int)s.objs.size() || s.objs[objects[i]].kind != 0)
      return fail(ctx, RFX_ERR_ARG, "rfx_update_spheres: object " + std::to_string(objects[i]) + " is not a sphere of this scene");
  // the host records, as rfx_add_sphere makes them (a later entry for the same object overwrites an earlier one)
  for (uint32_t i = 0; i < n; i++)
  {
    HostObj & o = s.objs[objects[i]];
    float radius = spheres[4 * i + 3];
    if (radius <= VSN) radius = VSN;                            // Scene.cpp:33-34
    memcpy(o.center, spheres + 4 * i, sizeof(o.center));
    o.sqRadius = radius * radius;                               // Sphere.cpp:19
    o.radius = radius;
  }
  if (ctx->sceneDirty || ctx->image.smallOk) { ctx->sceneDirty = true; return 0; }
  SceneImage & img = ctx->image;
  // the hierarchies' margins were sized for a reach box that must still hold every moved sphere (every drop point on it, its centre)
  if (img.bvhDepth > 0 || img.triBvhTris > 0)
    for (uint32_t i = 0; i < n; i++)
    {
      const HostObj & o = s.objs[objects[i]];
      for (int k = 0; k < 3; k++)
        if (!((double)o.center[k] - fabs((double)o.radius) >= img.reach[k] && (double)o.center[k] + fabs((double)o.radius) <= img.reach[3 + k]))
        {
          ctx->sceneDirty = true;
          return 0;
        }
    }
  double sphBox[6];
  if (img.lightGridsBuilt)
  {
    sphereDropBox(s, img, sphBox);
    if (!gridBoxHolds(ctx, sphBox)) { ctx->sceneDirty = true; return 0; }
  }

  // the moved spheres, once each, with their final records
  ctx->sphMoved.assign(img.spheres.size(), 0);
  ctx->sphMoves.clear();
  for (uint32_t i = n; i-- > 0;)
  {
    const int pos = (int)(std::lower_bound(img.sphObj.begin(), img.sphObj.end(), objects[i]) - img.sphObj.begin());
    if (ctx->sphMoved[pos]) continue;
    ctx->sphMoved[pos] = 1;
    const HostObj & o = s.objs[objects[i]];
    SphereMove m;
    memset(&m, 0, sizeof(m));
    m.rec = make_float4(o.center[0], o.center[1], o.center[2], o.sqRadius);
    m.pos = pos; m.radius = o.radius;
    ctx->sphMoves.push_back(m);
    img.spheres[pos] = m.rec;                                  // the eye grid's records
    img.sphRadius[pos] = o.radius;
  }
  CK(cudaSetDevice(ctx->device));
  // the stream the renders use: the update is ordered after the frames already queued there
  cudaStream_t st = ctx->lastStream ? ctx->lastStream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK || (rc = upload(ctx, ctx->dSphMoves, ctx->sphMoves, st)) != RFX_OK) return rc;
  const SceneHeader & h = *reinterpret_cast<const SceneHeader *>(img.blob.data());
  SphereUpdate u;
  memset(&u, 0, sizeof(u));
  u.moves = ctx->dSphMoves.p; u.nMoves = (int)ctx->sphMoves.size();
  u.spheres = reinterpret_cast<float4 *>(ctx->dBlob.p + h.offSpheres);
  u.radius = ctx->dSphRadius.p;
  if (!img.sphSlot.empty())
  {
    u.leafSph = ctx->dBvhNodes.p; u.pairs = ctx->dBvhNodes.p + img.sphBvh.leafFloat4;
    u.prims = ctx->dBvhPrims.p; u.slot = ctx->dSphSlot.p;
    u.leafParent = ctx->dSphLeafParent.p; u.pairParent = ctx->dSphPairParent.p;
    u.arrive = ctx->dSphArrive.p;
    u.nLeaves = (int)img.sphLeafParent.size();
    u.R = img.sphR;
    if (!img.sphPairParent.empty()) CK(cudaMemsetAsync(ctx->dSphArrive.p, 0, img.sphPairParent.size() * sizeof(uint32_t), st));
  }
  ctx->stats.kernel_launches += launchSphereUpdate(u, st);
  CK(cudaGetLastError());

  // The grids of the lights that have one are rebuilt on the device for the new spheres, over the box they were built for (which still
  // holds every drop point).  Re-binning into the old cells would miss spheres that moved out of a grid's rectangle.
  if (img.lightGridsBuilt)
  {
    memcpy(img.dropSpheres, sphBox, sizeof(sphBox));
    for (size_t li = 0; li < s.lights.size(); li++)
      if (ctx->lightGrid[li] && (rc = updateLightGrid(ctx, li, st)) != RFX_OK) return rc;
  }
  // the eye grid is built again at the next render, from the blob's spheres (img.spheres on the host path)
  ctx->sphereUpdates++;
  return 1;
}

int rfx_set_triangle_texture(rfx_ctx * ctx, int object, int texture, const float uv[6])
{
  if (!ctx || !uv) return fail(ctx, RFX_ERR_ARG, "rfx_set_triangle_texture: NULL argument");
  if (object < 0 || object >= (int)ctx->scene.objs.size() || ctx->scene.objs[object].kind != 1)
    return fail(ctx, RFX_ERR_ARG, "rfx_set_triangle_texture: object is not a triangle");
  if (texture < 0 || texture >= (int)ctx->scene.tex.size()) return fail(ctx, RFX_ERR_ARG, "rfx_set_triangle_texture: unknown texture");
  HostObj & o = ctx->scene.objs[object];
  // tuvTrans = Matrix33(v3 - v1, v2 - v1, (0,0,-1)) with v_i = (tu_i, tv_i, 0), Triangle.cpp:116-119
  o.tri.tuv[0] = uv[4] - uv[0]; o.tri.tuv[1] = uv[2] - uv[0];
  o.tri.tuv[2] = uv[5] - uv[1]; o.tri.tuv[3] = uv[3] - uv[1];
  o.tri.tu0 = uv[0]; o.tri.tv0 = uv[1];
  o.mat.tex = texture;
  ctx->sceneDirty = true;
  return RFX_OK;
}

int rfx_add_plane(rfx_ctx * ctx, const float pos[3], const float norm[3], int mtype, const float rgb[3], float refl, float transp)
{
  if (!ctx || !pos || !norm || !rgb) return fail(ctx, RFX_ERR_ARG, "rfx_add_plane: NULL argument");
  HostObj o;
  memset(&o, 0, sizeof(o));
  o.kind = 2;
  o.mat = makeMaterial(mtype, rgb, refl, transp, (int)ctx->scene.objs.size());
  memcpy(o.plane.pos, pos, sizeof(float) * 3);
  memcpy(o.plane.n, norm, sizeof(float) * 3);
  ctx->scene.objs.push_back(o);
  ctx->sceneDirty = true;
  return (int)ctx->scene.objs.size() - 1;
}

int rfx_add_texture_argb(rfx_ctx * ctx, uint32_t w, uint32_t h, const uint32_t * argb)
{
  if (!ctx) return RFX_ERR_ARG;
  HostTex t;
  if (argb && w && h)
  {
    t.w = w; t.h = h;
    t.px.assign(argb, argb + (size_t)w * h);
  }
  ctx->scene.tex.push_back(std::move(t));
  ctx->sceneDirty = true;
  return (int)ctx->scene.tex.size() - 1;
}

int rfx_set_skybox(rfx_ctx * ctx, int texture)
{
  if (!ctx) return RFX_ERR_ARG;
  if (texture >= (int)ctx->scene.tex.size()) return fail(ctx, RFX_ERR_ARG, "rfx_set_skybox: unknown texture");
  // Skybox::loadTexture returns false and keeps the checker when the file failed to load (Skybox.cpp:30-36)
  ctx->scene.skyTex = (texture >= 0 && !ctx->scene.tex[texture].px.empty()) ? texture : -1;
  ctx->sceneDirty = true;
  return ctx->scene.skyTex >= 0 ? 1 : 0;
}

// --------------------------------------------------------------------------------------------------------- camera
int rfx_set_camera(rfx_ctx * ctx, const float eye[3], const float view[9], float fov)
{
  if (!ctx || !eye || !view) return fail(ctx, RFX_ERR_ARG, "rfx_set_camera: NULL argument");
  memcpy(ctx->scene.eye, eye, sizeof(float) * 3);
  memcpy(ctx->view, view, sizeof(float) * 9);
  ctx->fov = fov;
  // the hierarchies' box margins were sized for ray origins inside bvhReach (uploadScene): an eye outside it re-flattens the scene
  if (ctx->image.bvhDepth > 0 || ctx->image.triBvhTris > 0)
    for (int k = 0; k < 3; k++)
      if (!(eye[k] >= ctx->image.reach[k] && eye[k] <= ctx->image.reach[3 + k])) ctx->sceneDirty = true;
  return RFX_OK;
}

// ----------------------------------------------------------------------------------------------------------- seeds
int rfx_set_seeds(rfx_ctx * ctx, uint32_t seed_vector3, uint32_t seed_render)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(ctx->dRng.p + ctx->rngSlot, &seed_vector3, sizeof(uint32_t), cudaMemcpyHostToDevice));
  ctx->seedRender = seed_render;
  return RFX_OK;
}

int rfx_get_seeds(rfx_ctx * ctx, uint32_t out[2])
{
  if (!ctx || !out) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(&out[0], ctx->dRng.p + ctx->rngSlot, sizeof(uint32_t), cudaMemcpyDeviceToHost));
  out[1] = ctx->seedRender;
  return checkStatus(ctx);
}

int rfx_selftest_rng(rfx_ctx * ctx, uint64_t out[2])
{
  if (!ctx || !out) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  unsigned long long * d = nullptr;
  CK(cudaMalloc((void **)&d, 2 * sizeof(unsigned long long)));
  cudaError_t e = cudaMemset(d, 0, 2 * sizeof(unsigned long long));
  if (e == cudaSuccess) { ctx->stats.kernel_launches += launchRngSelftest(d, ctx->stream); e = cudaStreamSynchronize(ctx->stream); }
  unsigned long long h[2] = { 0, 0 };
  if (e == cudaSuccess) e = cudaMemcpy(h, d, sizeof(h), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail(ctx, RFX_ERR_CUDA, std::string("rfx_selftest_rng: ") + cudaGetErrorString(e));
  out[0] = h[0]; out[1] = h[1];
  return RFX_OK;
}

int rfx_selftest_light_grids(rfx_ctx * ctx, uint64_t out[3])
{
  if (!ctx || !out) return RFX_ERR_ARG;
  if (ctx->sceneDirty) return fail(ctx, RFX_ERR_ARG, "rfx_selftest_light_grids: the scene changed since its last flatten");
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  out[0] = out[1] = out[2] = 0;
  const SceneImage & img = ctx->image;
  if (!img.lightGridsBuilt) return RFX_OK;
  std::unique_ptr<SceneImage> ref(new SceneImage());
  rebuildLightGrids(ctx->scene, img, *ref);
  const size_t nL = ctx->scene.lights.size();
  std::vector<LightGrid> hdr(nL);
  std::vector<uint32_t> flags(1 + nL), cells;
  std::vector<float4> sp;
  std::vector<int> ix;
  CK(cudaMemcpy(hdr.data(), ctx->dLightGrids.p, nL * sizeof(LightGrid), cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(flags.data(), ctx->dGridFlags.p, flags.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  for (size_t li = 0; li < nL; li++)
  {
    const LightGrid & g = hdr[li];
    const bool dev = g.cellStart != nullptr, host = !ref->grids.empty() && ref->grids[li].nx != 0;
    out[1] += dev; out[2] += host;
    if (!dev && host && flags[1 + li]) continue;   // dropped for want of room: its queries walk the hierarchy until a build fits
    if (dev != host) { out[0]++; continue; }
    if (!dev) continue;
    const LightGrid & r = ref->grids[li];
    const size_t nCells = (size_t)r.nx * r.ny + 1, off = ref->gridCellOff[li], nItems = ref->gridCells[off + nCells - 1];
    if (memcmp(g.u, r.u, sizeof(g.u)) || memcmp(g.v, r.v, sizeof(g.v)) || g.nx != r.nx || g.ny != r.ny || nItems > ctx->gridItemAlloc) { out[0]++; continue; }
    cells.resize(nCells); sp.resize(nItems); ix.resize(nItems);
    CK(cudaMemcpy(cells.data(), g.cellStart, nCells * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    if (nItems)
    {
      CK(cudaMemcpy(sp.data(), g.itemSphere, nItems * sizeof(float4), cudaMemcpyDeviceToHost));
      CK(cudaMemcpy(ix.data(), g.itemIndex, nItems * sizeof(int), cudaMemcpyDeviceToHost));
    }
    const size_t io = ref->gridItemOff[li];
    if (memcmp(cells.data(), &ref->gridCells[off], nCells * sizeof(uint32_t)) ||
        (nItems && (memcmp(sp.data(), &ref->gridSpheres[io], nItems * sizeof(float4)) || memcmp(ix.data(), &ref->gridIndex[io], nItems * sizeof(int)))))
      out[0]++;
  }
  return RFX_OK;
}

int rfx_selftest_eye_grid(rfx_ctx * ctx, uint64_t out[4])
{
  if (!ctx || !out) return RFX_ERR_ARG;
  if (ctx->sceneDirty) return fail(ctx, RFX_ERR_ARG, "rfx_selftest_eye_grid: the scene changed since its last flatten");
  if (!ctx->eyeRendered) return fail(ctx, RFX_ERR_ARG, "rfx_selftest_eye_grid: no blob frame has been rendered since the last flatten");
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  out[0] = out[1] = out[2] = out[3] = 0;
  uint32_t flags[2] = { 0, 0 };
  if (ctx->dEyeFlags.p) CK(cudaMemcpy(flags, ctx->dEyeFlags.p, sizeof(flags), cudaMemcpyDeviceToHost));
  out[3] = flags[1];
  // the host's binning for the camera of that render and the current spheres (none where buildEyeGrid builds none)
  int nx = 0, ny = 0;
  std::vector<uint32_t> cells, dev;
  std::vector<float4> items;
  std::vector<int> index;
  const bool host = ctx->eyeGridOn && ctx->image.bvhDepth > 0 && binEyeGrid(ctx->eyeFp, ctx->image.spheres, nx, ny, cells, items, index);
  const EyeGrid & g = ctx->eyeUsed;
  if (host) out[2] = cells.back();
  if ((g.cellStart != nullptr) != host) { out[0]++; return RFX_OK; }
  if (!host) return RFX_OK;
  if (g.nx != nx || g.ny != ny || g.shift != EYE_GRID_SHIFT) { out[0]++; return RFX_OK; }
  dev.resize(cells.size() + 1);
  CK(cudaMemcpy(dev.data(), g.cellStart, dev.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  if (dev.back() != 0u) return RFX_OK;                          // dropped for want of room: the first queries walked the hierarchy
  const uint32_t nDev = dev[cells.size() - 1];
  out[1] = nDev;
  for (size_t c = 0; c < cells.size(); c++) out[0] += dev[c] != cells[c];
  const size_t n = std::min<size_t>(nDev, cells.back());
  out[0] += std::max<size_t>(nDev, cells.back()) - n;            // items on one side only
  if (n)
  {
    std::vector<float4> sp(n);
    std::vector<int> ix(n);
    CK(cudaMemcpy(sp.data(), g.itemSphere, n * sizeof(float4), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(ix.data(), g.itemIndex, n * sizeof(int), cudaMemcpyDeviceToHost));
    for (size_t k = 0; k < n; k++) out[0] += ix[k] != index[k] || memcmp(&sp[k], &items[k], sizeof(float4)) != 0;
  }
  return RFX_OK;
}

int rfx_selftest_primary_bounds(rfx_ctx * ctx, int32_t out[96], int32_t counts[2])
{
  if (!ctx || !out || !counts) return RFX_ERR_ARG;
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "rfx_selftest_primary_bounds: image size not set");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, ctx->stream)) != RFX_OK) return rc;
  if (!ctx->image.smallOk) return fail(ctx, RFX_ERR_ARG, "rfx_selftest_primary_bounds: the scene does not fit the constant bank");
  const PrimaryCull pc = makePrimaryCull(ctx->image.small, frameFromCamera(ctx->scene.eye, ctx->view, ctx->fov, ctx->W, ctx->H));
  static_assert(sizeof(pc.rect) == 96 * sizeof(int32_t), "24 rectangles of 4 ints");
  memcpy(out, pc.rect, sizeof(pc.rect));
  counts[0] = (int32_t)ctx->image.spheres.size(); counts[1] = ctx->image.small.nT;   // (small.nS is padded to whole quads)
  return RFX_OK;
}

int rfx_skip_samples(rfx_ctx * ctx, uint64_t n)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  int rc;
  // the stream state lives on the device and advances in stream order: stay on the stream the renders use
  cudaStream_t st = ctx->lastStream ? ctx->lastStream : ctx->stream;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  return skipSamples(ctx, n, st);
}

// ---------------------------------------------------------------------------------------------------------- Render
int rfx_set_image_size(rfx_ctx * ctx, uint32_t width, uint32_t height)
{
  if (!ctx) return RFX_ERR_ARG;
  if (!width || !height) return fail(ctx, RFX_ERR_ARG, "rfx_set_image_size: zero size");   // Render.cpp:59-62: ignored
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  const size_t n = (size_t)width * height;
  if ((rc = ensure(ctx, ctx->dImage, n * 3)) != RFX_OK) return rc;
  ctx->stats.kernel_launches += launchClear(ctx->dImage.p, n * 3, ctx->stream);   // Render.cpp:67-71
  CK(cudaGetLastError());
  ctx->W = width; ctx->H = height;
  ctx->additiveCounter = 0;
  ctx->inProgress = false;
  ctx->cursor = 0;
  return RFX_OK;
}

int rfx_render_begin(rfx_ctx * ctx, int reflect_num, int sample_num, int additive)
{
  if (!ctx) return RFX_ERR_ARG;
  if (reflect_num <= 0 || sample_num == 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_begin: reflect_num must be > 0 and sample_num != 0");
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "rfx_render_begin: image size not set");
  if (sample_num > 1024 || sample_num < -4096) return fail(ctx, RFX_ERR_ARG, "rfx_render_begin: sample_num out of range");
  ctx->reflNum = reflect_num;
  ctx->sampleNum = sample_num;
  ctx->additive = additive != 0;
  ctx->inProgress = true;
  ctx->cursor = 0;
  if (additive) ctx->additiveCounter++; else ctx->additiveCounter = 0;     // Render.cpp:130-133

  // renderCameraEye / renderCameraView snapshot, Render.cpp:125-126.  NOTE the reference evaluates rz (Render.cpp:148-150) with the
  // LIVE camera.fov inside renderNext; Pulse never changes fov (Camera.cpp has no writer besides the constructors), so latching it
  // here is equivalent.
  FrameParams & fp = ctx->snap;
  fp = frameFromCamera(ctx->scene.eye, ctx->view, ctx->fov, ctx->W, ctx->H);
  fp.reflNum = reflect_num;
  fp.sampleNum = sample_num;
  fp.jitter = additive ? 1 : 0;
  fp.accumulate = ctx->additiveCounter > 1 ? 1 : 0;
  return RFX_OK;
}

int rfx_render_next(rfx_ctx * ctx, uint32_t pixels)
{
  if (!ctx) return RFX_ERR_ARG;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  if (!pixels || !ctx->inProgress || ctx->cursor >= total) return 0;     // Render.cpp:143-144: returns false
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, ctx->stream)) != RFX_OK) return rc;
  if (ctx->sigOn && (rc = ensure(ctx, ctx->dSig, (size_t)total)) != RFX_OK) return rc;
  const uint64_t end = std::min(total, ctx->cursor + pixels);
  if ((rc = renderRange(ctx, ctx->cursor, end, nullptr, true, ctx->stream)) != RFX_OK) return rc;
  ctx->cursor = end;
  if (ctx->cursor >= total) ctx->inProgress = false;                     // Render.cpp:207-211
  return ctx->inProgress ? 1 : 0;
}

// number of Scene::trace calls the reference makes for pixels [p0, p1) of the latched frame
static uint64_t callsIn(const rfx_ctx * ctx, uint64_t p0, uint64_t p1)
{
  if (ctx->sampleNum > 0) return (p1 - p0) * (uint64_t)ctx->sampleNum * (uint64_t)ctx->sampleNum;
  const uint32_t a = (uint32_t)(-ctx->sampleNum);
  return originsBefore(p1, ctx->W, a) - originsBefore(p0, ctx->W, a);
}

static int skipPixels(rfx_ctx * ctx, uint64_t p0, uint64_t p1, cudaStream_t st)
{
  int rc;
  if ((rc = skipSamples(ctx, callsIn(ctx, p0, p1), st)) != RFX_OK) return rc;
  if (ctx->snap.jitter && ctx->sampleNum > 0) ctx->seedRender = lcgJumpHost(ctx->seedRender, 2 * (p1 - p0));
  return RFX_OK;
}

int rfx_render_range(rfx_ctx * ctx, uint64_t p0, uint64_t p1, uint32_t * argb_device, void * stream)
{
  if (!ctx) return RFX_ERR_ARG;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  if (!ctx->inProgress) return fail(ctx, RFX_ERR_ARG, "rfx_render_range: no frame in progress");
  if (p0 > p1 || p1 > total || p0 < ctx->cursor) return fail(ctx, RFX_ERR_ARG, "rfx_render_range: ranges must be increasing and inside the frame");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  if (ctx->sigOn && (rc = ensure(ctx, ctx->dSig, (size_t)total)) != RFX_OK) return rc;
  if (p0 > ctx->cursor && (rc = skipPixels(ctx, ctx->cursor, p0, st)) != RFX_OK) return rc;
  if ((rc = renderRange(ctx, p0, p1, argb_device, argb_device == nullptr, st)) != RFX_OK) return rc;
  ctx->cursor = p1;
  return RFX_OK;
}

int rfx_render_strips(rfx_ctx * ctx, uint32_t strip_rows, uint32_t world, uint32_t rank, uint32_t * argb_device, void * stream)
{
  if (!ctx || !argb_device || !strip_rows || !world || rank >= world) return fail(ctx, RFX_ERR_ARG, "rfx_render_strips: bad argument");
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  if (!ctx->inProgress || ctx->cursor != 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_strips: needs a freshly begun frame");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  const uint64_t calls = ctx->sampleNum > 0 ? callsIn(ctx, 0, total) : 0;
  const bool fast = ctx->sampleNum > 0 && ctx->image.smallOk && ctx->forcePath < 2 && !ctx->snap.jitter && !ctx->sigOn &&
                    strip_rows % 8 == 0 && calls <= (1ull << 26);
  if (!fast)
  {
    // general path: one range per strip (block preview, big scenes, huge SSAA factors)
    const uint32_t nStrips = (ctx->H + strip_rows - 1) / strip_rows;
    for (uint32_t s = rank; s < nStrips; s += world)
    {
      const uint64_t p0 = (uint64_t)s * strip_rows * ctx->W, p1 = std::min<uint64_t>(total, (uint64_t)(s + 1) * strip_rows * ctx->W);
      if ((rc = rfx_render_range(ctx, p0, p1, argb_device, stream)) != RFX_OK) return rc;
    }
    return rfx_render_finish(ctx);
  }
  const uint64_t perPixel = (uint64_t)ctx->sampleNum * ctx->sampleNum;
  // K1 once over the whole frame (every GPU needs the accept counts of everything before its rows); only the states of
  // this rank's strips are stored
  if ((rc = rankSamples(ctx, calls, false, st, (uint64_t)strip_rows * ctx->W * perPixel, world, rank)) != RFX_OK) return rc;
  TraceWork w = traceWork(ctx, 0, total, 0, ctx->dSampleStates.p, nullptr, argb_device);
  w.fp.stripRows = strip_rows; w.fp.stripWorld = world; w.fp.stripRank = rank;
  cudaEvent_t evStop;
  if ((rc = profileStart(ctx, st, evStop)) != RFX_OK) return rc;
  if ((rc = armTileOrder(ctx, w, st)) != RFX_OK) return rc;
  {
    uint32_t fastGrid = 0;   // 0: the fast kernel declined (a 4-byte aligned frame) and the general kernel ran
    const int nl = launchTraceSmall(ctx->image.small, w, st, &fastGrid);
    ctx->stats.kernel_launches += nl;
    (fastGrid ? ctx->stats.launches_small_fast : ctx->stats.launches_small_any) += nl;
  }
  if (evStop) CK(cudaEventRecord(evStop, st));
  CK(cudaGetLastError());
  // the Scene::trace calls of this rank's own rows: its whole strips, less what the frame cuts off its last strip
  const uint32_t nStrips = (ctx->H + strip_rows - 1) / strip_rows;
  uint64_t ownRows = ownedRows(w.fp, ctx->H);
  if ((nStrips - 1) % world == rank) ownRows -= (uint64_t)nStrips * strip_rows - ctx->H;
  ctx->stats.samples += ownRows * ctx->W * perPixel;
  ctx->cursor = total;
  ctx->inProgress = false;
  return RFX_OK;
}

int rfx_render_finish(rfx_ctx * ctx)
{
  if (!ctx) return RFX_ERR_ARG;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  if (!ctx->inProgress) return RFX_OK;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->lastStream ? ctx->lastStream : ctx->stream;
  int rc;
  if (ctx->cursor < total && (rc = skipPixels(ctx, ctx->cursor, total, st)) != RFX_OK) return rc;
  ctx->cursor = total;
  ctx->inProgress = false;
  return RFX_OK;
}

int rfx_buffer_alloc(rfx_ctx * ctx, uint64_t bytes, void ** device_ptr)
{
  if (!ctx || !device_ptr || !bytes) return fail(ctx, RFX_ERR_ARG, "rfx_buffer_alloc: bad argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMalloc(device_ptr, bytes));
  CK(cudaMemset(*device_ptr, 0, bytes));
  return RFX_OK;
}

int rfx_buffer_free(rfx_ctx * ctx, void * device_ptr)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaFree(device_ptr));
  return RFX_OK;
}

int rfx_buffer_read(rfx_ctx * ctx, const void * device_ptr, void * host_dst, uint64_t bytes)
{
  if (!ctx || !device_ptr || !host_dst) return fail(ctx, RFX_ERR_ARG, "rfx_buffer_read: NULL argument");
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemcpy(host_dst, device_ptr, bytes, cudaMemcpyDeviceToHost));
  ctx->stats.d2h_bytes += bytes;
  return RFX_OK;
}

int rfx_ipc_export(rfx_ctx * ctx, void * device_ptr, unsigned char handle[64])
{
  if (!ctx || !device_ptr || !handle) return fail(ctx, RFX_ERR_ARG, "rfx_ipc_export: NULL argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  CK(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, device_ptr));
  memcpy(handle, &h, 64);
  return RFX_OK;
}

int rfx_ipc_import(rfx_ctx * ctx, const unsigned char handle[64], void ** device_ptr)
{
  if (!ctx || !device_ptr || !handle) return fail(ctx, RFX_ERR_ARG, "rfx_ipc_import: NULL argument");
  CK(cudaSetDevice(ctx->device));
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, 64);
  CK(cudaIpcOpenMemHandle(device_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return RFX_OK;
}

int rfx_ipc_close(rfx_ctx * ctx, void * device_ptr)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaIpcCloseMemHandle(device_ptr));
  return RFX_OK;
}

float rfx_progress(const rfx_ctx * ctx)
{
  if (!ctx || !ctx->W || !ctx->H) return 0.0f;
  // float(curx + cury * imageWidth) * 100.0f / imageWidth / imageHeight, Render.cpp:223-226; a finished frame leaves the
  // cursor at (0, imageHeight) upstream, i.e. 100 %
  return float(ctx->cursor) * 100.0f / ctx->W / ctx->H;
}

int rfx_additive_counter(const rfx_ctx * ctx) { return ctx ? ctx->additiveCounter : 0; }
int rfx_in_progress(const rfx_ctx * ctx) { return ctx && ctx->inProgress ? 1 : 0; }

static int readResolved(rfx_ctx * ctx, float * rgbf, uint32_t * argb, int divide = 1)
{
  const int counter = divide ? ctx->additiveCounter : 0;
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "image size not set");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  const size_t n = (size_t)ctx->W * ctx->H;
  if (argb)
  {
    if ((rc = ensure(ctx, ctx->dResolve, n)) != RFX_OK) return rc;
    ctx->stats.kernel_launches += launchResolve(ctx->dImage.p, n, counter, nullptr, ctx->dResolve.p, ctx->stream);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(argb, ctx->dResolve.p, n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->stats.d2h_bytes += n * 4;
  }
  if (rgbf)
  {
    if (counter > 1)
    {
      // divide on the device into the ranked-state scratch (reused as a float buffer), then copy
      size_t need = n * 3;
      if ((rc = ensure(ctx, ctx->dSampleStates, need)) != RFX_OK) return rc;
      ctx->stats.kernel_launches += launchResolve(ctx->dImage.p, n, counter, reinterpret_cast<float *>(ctx->dSampleStates.p), nullptr, ctx->stream);
      CK(cudaGetLastError());
      CK(cudaMemcpyAsync(rgbf, ctx->dSampleStates.p, n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    }
    else
      CK(cudaMemcpyAsync(rgbf, ctx->dImage.p, n * 12, cudaMemcpyDeviceToHost, ctx->stream));
    ctx->stats.d2h_bytes += n * 12;
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return checkStatus(ctx);
}

int rfx_read_argb(rfx_ctx * ctx, uint32_t * dst)
{
  if (!ctx || !dst) return fail(ctx, RFX_ERR_ARG, "rfx_read_argb: NULL argument");
  return readResolved(ctx, nullptr, dst);
}

int rfx_read_rgbf(rfx_ctx * ctx, float * dst)
{
  if (!ctx || !dst) return fail(ctx, RFX_ERR_ARG, "rfx_read_rgbf: NULL argument");
  return readResolved(ctx, dst, nullptr);
}

int rfx_read_image(rfx_ctx * ctx, float * rgbf, uint32_t * argb, int divide)
{
  if (!ctx || (!rgbf && !argb)) return fail(ctx, RFX_ERR_ARG, "rfx_read_image: NULL argument");
  return readResolved(ctx, rgbf, argb, divide);
}

int rfx_trace_rays(rfx_ctx * ctx, int n, const float * origins, const float * rays, int reflect_num, float * rgb)
{
  if (!ctx || n < 0 || !origins || !rays || !rgb || reflect_num <= 0) return fail(ctx, RFX_ERR_ARG, "rfx_trace_rays: bad argument");
  if (n == 0) return RFX_OK;
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  if (ctx->image.bvhDepth > 0 || ctx->image.triBvhTris > 0)
  {
    // the hierarchies' box margins are sized for ray origins inside bvhReach: origins outside it widen the region and re-flatten
    bool outside = false;
    for (int i = 0; i < n; i++)
      for (int k = 0; k < 3; k++)
      {
        const float v = origins[3 * (size_t)i + k];
        if (!(v >= ctx->image.reach[k] && v <= ctx->image.reach[3 + k]) && v == v && fabsf(v) <= FLT_MAX)
        {
          outside = true;
          ctx->scene.extraOrigins[k] = std::min(ctx->scene.extraOrigins[k], v);
          ctx->scene.extraOrigins[3 + k] = std::max(ctx->scene.extraOrigins[3 + k], v);
        }
      }
    if (outside)
    {
      ctx->sceneDirty = true;
      if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
    }
  }
  if ((rc = rankSamples(ctx, (uint64_t)n, false, st)) != RFX_OK) return rc;
  // ray buffers: origins | rays | rgb in one scratch allocation
  if ((rc = ensure(ctx, ctx->dRays, (size_t)n * 9)) != RFX_OK) return rc;
  float * dO = ctx->dRays.p, * dR = ctx->dRays.p + (size_t)n * 3, * dC = ctx->dRays.p + (size_t)n * 6;
  CK(cudaMemcpyAsync(dO, origins, (size_t)n * 12, cudaMemcpyHostToDevice, st));
  CK(cudaMemcpyAsync(dR, rays, (size_t)n * 12, cudaMemcpyHostToDevice, st));
  ctx->stats.h2d_bytes += (uint64_t)n * 24;
  ctx->stats.kernel_launches += launchTraceBlobRays(ctx->dBlob.p, n, dO, dR, reflect_num, ctx->dSampleStates.p, dC, ctx->dCounters.p, st, ctx->image.triBvhTris > 0,
                                                    ctx->image.far);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(rgb, dC, (size_t)n * 12, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  ctx->stats.d2h_bytes += (uint64_t)n * 12;
  ctx->stats.samples += (uint64_t)n;
  return checkStatus(ctx);
}

int rfx_read_pixel(rfx_ctx * ctx, int x, int y, float rgb[3])
{
  if (!ctx || !rgb) return RFX_ERR_ARG;
  rgb[0] = rgb[1] = rgb[2] = 0.0f;                                        // Render.cpp:112-113
  if (x < 0 || y < 0 || (uint32_t)x >= ctx->W || (uint32_t)y >= ctx->H) return RFX_OK;
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  CK(cudaMemcpyAsync(rgb, ctx->dImage.p + ((size_t)y * ctx->W + x) * 3, 12, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  ctx->stats.d2h_bytes += 12;
  if (ctx->additiveCounter > 1)
  {
    const float d = float(ctx->additiveCounter);                         // Render.cpp:109-110, Color.cpp:99-107
    rgb[0] = rgb[0] / d; rgb[1] = rgb[1] / d; rgb[2] = rgb[2] / d;
  }
  return RFX_OK;
}

int rfx_enable_signatures(rfx_ctx * ctx, int on)
{
  if (!ctx) return RFX_ERR_ARG;
  ctx->sigOn = on != 0;
  return RFX_OK;
}

int rfx_read_signatures(rfx_ctx * ctx, uint32_t * dst)
{
  if (!ctx || !dst) return RFX_ERR_ARG;
  if (!ctx->sigOn || !ctx->dSig.p) return fail(ctx, RFX_ERR_ARG, "rfx_read_signatures: signatures are not enabled");
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = useStream(ctx, ctx->stream)) != RFX_OK) return rc;
  CK(cudaMemcpyAsync(dst, ctx->dSig.p, (size_t)ctx->W * ctx->H * 4, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return RFX_OK;
}

// ----------------------------------------------------------------------------------------------------- batch path
static int beginFrame(rfx_ctx * ctx, const float * cam, int reflect_num, int sample_num)
{
  int rc;
  if ((rc = rfx_set_camera(ctx, cam, cam + 3, cam[12])) != RFX_OK) return rc;
  ctx->additiveCounter = 0;   // each frame is a fresh setImageSize-sized, non-additive screenshot render (Pulse.cpp:174-176)
  return rfx_render_begin(ctx, reflect_num, sample_num, 0);
}

int rfx_render_frames_device(rfx_ctx * ctx, int n_frames, const float * cams, int reflect_num, int sample_num,
                             uint32_t * argb_device, void * stream)
{
  if (!ctx || !cams || !argb_device || n_frames < 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames_device: bad argument");
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames_device: image size not set");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  // one K1 pass ranks the random states of a whole group of frames (the stream simply continues from frame to frame)
  if (reflect_num <= 0 || sample_num == 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames_device: reflect_num must be > 0 and sample_num != 0");
  ctx->sampleNum = sample_num;
  const uint64_t perFrame = callsIn(ctx, 0, total);
  const int group = (int)std::max<uint64_t>(1, ctx->maxCallsPerLaunch / std::max<uint64_t>(perFrame, 1));
  for (int f0 = 0; f0 < n_frames; f0 += group)
  {
    const int g = std::min(group, n_frames - f0);
    const bool pre = perFrame <= ctx->maxCallsPerLaunch;
    if (pre && (rc = rankSamples(ctx, perFrame * g, false, st)) != RFX_OK) return rc;
    for (int f = f0; f < f0 + g;)
    {
      const float * cam = cams + 13 * (size_t)f;
      if ((rc = beginFrame(ctx, cam, reflect_num, sample_num)) != RFX_OK) return rc;
      if (ctx->sceneDirty && (rc = uploadScene(ctx, st)) != RFX_OK) return rc;   // this frame's eye left the box the BVH margins were sized for
      uint32_t * out = argb_device + (size_t)f * total;
      const uint32_t * states = pre ? ctx->dSampleStates.p + (size_t)(f - f0) * perFrame : nullptr;
      // the following frames that repeat this camera (bit for bit) share their first segments: one launch renders up to
      // RFX_FRAME_BATCH of them (k_trace_small, BATCH)
      int n = 1;
      if (ctx->frameBatch && pre)
        while (n < std::min(RFX_FRAME_BATCH, f0 + g - f) && memcmp(cam, cam + 13 * (size_t)n, 13 * sizeof(float)) == 0) n++;
      if (n > 1)
      {
        // a repeat whose eye would re-flatten the scene (outside the box the hierarchy margins were sized for) renders on its own
        if ((rc = rfx_set_camera(ctx, cam, cam + 3, cam[12])) != RFX_OK) return rc;
        const bool useSmall = ctx->forcePath >= 2 ? false : ctx->image.smallOk;
        if (ctx->sceneDirty || !useSmall || !fastBatchOk(traceWork(ctx, 0, total, 0, states, nullptr, out))) n = 1;
      }
      if ((rc = renderRange(ctx, 0, total, out, false, st, states, (uint32_t)n)) != RFX_OK) return rc;
      ctx->cursor = total;
      ctx->inProgress = false;
      f += n;
    }
  }
  return RFX_OK;
}

int rfx_render_frames(rfx_ctx * ctx, int n_frames, const float * cams, int reflect_num, int sample_num, uint32_t * argb_host)
{
  if (!ctx || !cams || !argb_host || n_frames < 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames: bad argument");
  if (!ctx->W || !ctx->H) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames: image size not set");
  CK(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  int rc;
  if ((rc = useStream(ctx, st)) != RFX_OK) return rc;
  if ((rc = uploadScene(ctx, st)) != RFX_OK) return rc;
  const uint64_t total = (uint64_t)ctx->W * ctx->H;
  // FRAME_SLOTS device frame slots: render frame f into slot f % FRAME_SLOTS on the compute stream while the copy stream(s)
  // drain older slots into the caller's host buffer
  const int NS = rfx_ctx::FRAME_SLOTS;
  for (int j = 0; j < NS; j++)
    if ((rc = ensure(ctx, ctx->dFrame[j], total)) != RFX_OK) return rc;
  if (reflect_num <= 0 || sample_num == 0) return fail(ctx, RFX_ERR_ARG, "rfx_render_frames: reflect_num must be > 0 and sample_num != 0");
  ctx->sampleNum = sample_num;
  const uint64_t perFrame = callsIn(ctx, 0, total);
  const int group = (int)std::max<uint64_t>(1, ctx->maxCallsPerLaunch / std::max<uint64_t>(perFrame, 1));
  const bool pre = perFrame <= ctx->maxCallsPerLaunch;
  for (int f = 0; f < n_frames; f++)
  {
    const int slot = f % NS;
    cudaStream_t cs = ctx->copyStream[ctx->copyStreams > 1 ? (f & 1) : 0];
    if (pre && f % group == 0 && (rc = rankSamples(ctx, perFrame * std::min(group, n_frames - f), false, st)) != RFX_OK) return rc;
    if (f >= NS) CK(cudaStreamWaitEvent(st, ctx->evCopied[slot], 0));   // slot free again?
    if ((rc = beginFrame(ctx, cams + 13 * (size_t)f, reflect_num, sample_num)) != RFX_OK) return rc;
    if (ctx->sceneDirty && (rc = uploadScene(ctx, st)) != RFX_OK) return rc;   // this frame's eye left the box the BVH margins were sized for
    if ((rc = renderRange(ctx, 0, total, ctx->dFrame[slot].p, false, st,
                          pre ? ctx->dSampleStates.p + (size_t)(f % group) * perFrame : nullptr)) != RFX_OK) return rc;
    ctx->cursor = total;
    ctx->inProgress = false;
    CK(cudaEventRecord(ctx->evRendered[slot], st));
    CK(cudaStreamWaitEvent(cs, ctx->evRendered[slot], 0));
    CK(cudaMemcpyAsync(argb_host + (size_t)f * total, ctx->dFrame[slot].p, total * 4, cudaMemcpyDeviceToHost, cs));
    CK(cudaEventRecord(ctx->evCopied[slot], cs));
    ctx->stats.d2h_bytes += total * 4;
  }
  for (int i = 0; i < 2; i++) CK(cudaStreamSynchronize(ctx->copyStream[i]));
  CK(cudaStreamSynchronize(st));
  return checkStatus(ctx);
}

int rfx_synchronize(rfx_ctx * ctx)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  if (ctx->lastStream) CK(cudaStreamSynchronize(ctx->lastStream));
  CK(cudaStreamSynchronize(ctx->stream));
  int rc;
  if ((rc = growLightGrids(ctx)) != RFX_OK || (rc = growEyeGrid(ctx)) != RFX_OK) return rc;
  return checkStatus(ctx);
}

// ----------------------------------------------------------------------------------------------------------- stats
int rfx_get_stats(rfx_ctx * ctx, rfx_stats * out)
{
  if (!ctx || !out) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  unsigned long long c[64];
  CK(cudaMemcpy(c, ctx->dCounters.p, sizeof(c), cudaMemcpyDeviceToHost));
  uint64_t b = 0, s = 0;
  for (int i = 0; i < 32; i++) { b += c[2 * i]; s += c[2 * i + 1]; }
  ctx->stats.bounces = b;
  ctx->stats.shadow_rays = s;
  ctx->stats.rays = b + s;
  for (size_t i = 0; i + 1 < ctx->evUsed; i += 2)
  {
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ctx->evPool[i], ctx->evPool[i + 1]));
    ctx->stats.trace_kernel_ms += ms;
    ctx->stats.trace_kernels++;
  }
  ctx->evUsed = 0;
  int rc;
  if ((rc = countLightGrids(ctx, ctx->stats.light_grids)) != RFX_OK || (rc = growLightGrids(ctx)) != RFX_OK ||
      (rc = growEyeGrid(ctx)) != RFX_OK) return rc;
  ctx->stats.bvh_triangles = ctx->image.triBvhTris;
  ctx->stats.bvh_spheres = ctx->image.bvhSpheres;
  *out = ctx->stats;
  return RFX_OK;
}

int rfx_stats_reset(rfx_ctx * ctx)
{
  if (!ctx) return RFX_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  CK(cudaMemset(ctx->dCounters.p, 0, 64 * sizeof(unsigned long long)));
  memset(&ctx->stats, 0, sizeof(ctx->stats));
  ctx->evUsed = 0;
  return RFX_OK;
}

int rfx_force_path(rfx_ctx * ctx, int path)
{
  if (!ctx || path < 0 || path > 3) return RFX_ERR_ARG;
  ctx->forcePath = path;
  return RFX_OK;
}

int rfx_set_tile_ordering(rfx_ctx * ctx, int on)
{
  if (!ctx) return RFX_ERR_ARG;
  ctx->tileOrdering = on != 0;
  ctx->tileHistory = false;
  return RFX_OK;
}

int rfx_set_bvh_mode(rfx_ctx * ctx, int mode)
{
  if (!ctx || mode < 0 || mode > 2) return RFX_ERR_ARG;
  ctx->scene.bvhMode = mode;
  ctx->sceneDirty = true;
  return RFX_OK;
}

int rfx_set_option(rfx_ctx * ctx, const char * name, int64_t value)
{
  if (!ctx || !name) return RFX_ERR_ARG;
  if (!strcmp(name, "max_calls_per_launch"))
  {
    if (value < 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: max_calls_per_launch must be >= 1");
    ctx->maxCallsPerLaunch = (uint64_t)value;
    return RFX_OK;
  }
  if (!strcmp(name, "light_grids"))
  {
    if (value != 0 && value != 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: light_grids must be 0 or 1");
    if (ctx->scene.lightGridsOn != (value != 0)) ctx->sceneDirty = true;
    ctx->scene.lightGridsOn = value != 0;
    return RFX_OK;
  }
  if (!strcmp(name, "light_grid_items"))
  {
    if (value < 0) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: light_grid_items must be >= 0 (0: no limit)");
    ctx->gridItemLimit = value;
    setGridItemCap(ctx);
    return RFX_OK;
  }
  if (!strcmp(name, "eye_grid"))
  {
    if (value != 0 && value != 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: eye_grid must be 0 or 1");
    ctx->eyeGridOn = value != 0;
    ctx->eyeValid = false;
    return RFX_OK;
  }
  if (!strcmp(name, "eye_grid_device"))
  {
    if (value != 0 && value != 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: eye_grid_device must be 0 or 1");
    ctx->eyeGridDevice = value != 0;
    ctx->eyeValid = false;
    return RFX_OK;
  }
  if (!strcmp(name, "eye_grid_items"))
  {
    if (value < 0) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: eye_grid_items must be >= 0 (0: no limit)");
    ctx->eyeItemLimit = value;
    ctx->eyeValid = false;
    return RFX_OK;
  }
  if (!strcmp(name, "blob_wavefront"))
  {
    if (value < 0 || value > 64) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: blob_wavefront must be 0 (off) or the number of first segments (1..64)");
    ctx->blobWavefront = (int)value;
    return RFX_OK;
  }
  if (!strcmp(name, "tile_order_period"))
  {
    if (value < 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: tile_order_period must be >= 1");
    ctx->tileRecordPeriod = (int)std::min<int64_t>(value, 1 << 30);
    return RFX_OK;
  }
  if (!strcmp(name, "blob_smem_bvh"))
  {
    ctx->blobSmemBvh = value != 0;
    return RFX_OK;
  }
  if (!strcmp(name, "frame_batch"))
  {
    if (value != 0 && value != 1) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: frame_batch must be 0 or 1");
    ctx->frameBatch = value != 0;
    return RFX_OK;
  }
  if (!strcmp(name, "copy_streams"))
  {
    if (value < 1 || value > 2) return fail(ctx, RFX_ERR_ARG, "rfx_set_option: copy_streams must be 1 or 2");
    ctx->copyStreams = (int)value;
    return RFX_OK;
  }
  return fail(ctx, RFX_ERR_ARG, std::string("rfx_set_option: unknown option ") + name);
}

int rfx_enable_profiling(rfx_ctx * ctx, int on)
{
  if (!ctx) return RFX_ERR_ARG;
  ctx->profiling = on != 0;
  return RFX_OK;
}

} // extern "C"
