// rfx_eye_grid.cu — the screen grid of a path's first query (EyeGrid) built on the device for a new camera, a new image size or moved
// spheres, from the sphere records of the blob (which k_sphere_scatter keeps current).  The grid is the one rfx_scene.cpp binEyeGrid bins
// for the same camera and spheres: the same dims, cell offsets and items, the items of a cell in ascending sphere index.  Both sides run
// the arithmetic of rfx_eye_grid.h (--fmad=false here, -ffp-contract=off there; the header comment has the caveat on atan2, asin and tan).
// The host decides in O(1) whether the camera gets a grid at all (eyeGridDims) and how many cells it has.
//
// One build is four launches and a memset on the caller's stream, no synchronisation:
//   (memset)      the row masks
//   k_eg_span     one thread per sphere: the cells its rectangle touches; each warp writes its 32 spheres' bits into the mask word of
//                 every row they touch (bit i of row y: sphere i touches row y) — the rows' sphere lists, in index order, without atomics
//   k_eg_rows     one CTA per row (and per ROW_THREADS columns), one thread per cell: the row's spheres taken from its mask in index
//                 order, each tested against the thread's column — a count per cell, then (FILL) the items
//   k_eg_scan     one CTA: the cell offsets (exclusive scan, in place), the total, and the drop word: a grid with more items than its
//                 region holds is dropped (its first queries walk the hierarchy)
//   k_eg_rows<FILL>
#include "rfx_kernels.h"
#include "rfx_eye_grid.h"

namespace rfx
{

namespace
{

constexpr int SPAN_THREADS = 256;
constexpr int ROW_THREADS = 256;                     // columns per CTA of k_eg_rows (1080p: 60 columns, 8K: 240)
constexpr int ROW_BATCH = 1024;                      // spheres of a row staged in shared memory at a time
constexpr int SCAN_THREADS = 1024;

__global__ void __launch_bounds__(SPAN_THREADS) k_eg_span(const EyeGridBuild b)
{
  const int i = blockIdx.x * SPAN_THREADS + threadIdx.x;
  int4 sp = make_int4(1, 0, 1, 0);
  if (i < b.nSpheres)
  {
    sp = eyeCellSpan(primarySphereBounds(b.cam, b.spheres[i]), b.W, b.H);
    b.xSpan[i] = make_int2(sp.x, sp.y);
  }
  // the warp owns mask word i / 32 of every row: one ballot per row the warp's spheres touch
  const bool any = sp.x <= sp.y && sp.z <= sp.w;
  const int lo = __reduce_min_sync(0xFFFFFFFFu, any ? sp.z : 0x7FFFFFFF), hi = __reduce_max_sync(0xFFFFFFFFu, any ? sp.w : -1);
  for (int y = lo; y <= hi; y++)
  {
    const uint32_t bits = __ballot_sync(0xFFFFFFFFu, any && sp.z <= y && y <= sp.w);
    if ((threadIdx.x & 31u) == 0u && bits) b.rowMask[(size_t)y * b.maskWords + i / 32] = bits;
  }
}

// One CTA per (row y, ROW_THREADS columns), thread x for cell (x, y).  The CTA reads the row's mask ROW_THREADS words at a time, stages
// the spheres of their set bits (in index order) ROW_BATCH at a time in shared memory, and every thread tests those against its column.
// The count pass stores the number of spheres per cell; the fill pass writes them from the cell's offset on, in index order.
template <bool FILL>
__global__ void __launch_bounds__(ROW_THREADS) k_eg_rows(const EyeGridBuild b)
{
  const int chunks = (b.nx + ROW_THREADS - 1) / ROW_THREADS;
  const int y = blockIdx.x / chunks, x = (blockIdx.x % chunks) * ROW_THREADS + threadIdx.x;
  const size_t nCells = (size_t)b.nx * b.ny;
  if (FILL && b.cells[nCells + 1] != 0u) return;    // dropped: nothing to fill
  __shared__ int sIdx[ROW_BATCH];
  __shared__ int2 sX[ROW_BATCH];
  __shared__ uint32_t sWarp[ROW_THREADS / 32];
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const size_t cell = (size_t)y * b.nx + x;
  uint32_t run = (FILL && x < b.nx) ? b.cells[cell] : 0u;
  const uint32_t * mask = b.rowMask + (size_t)y * b.maskWords;
  for (int base = 0; base < b.maskWords; base += ROW_THREADS)
  {
    const int w = base + threadIdx.x;
    const uint32_t bits = w < b.maskWords ? mask[w] : 0u;
    const uint32_t cnt = __popc(bits);
    // exclusive scan of the words' bit counts
    uint32_t inc = cnt;
    for (int o = 1; o < 32; o <<= 1)
    {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) sWarp[warp] = inc;
    __syncthreads();
    uint32_t off = inc - cnt, total = 0;
    for (int k = 0; k < ROW_THREADS / 32; k++) { off += k < warp ? sWarp[k] : 0u; total += sWarp[k]; }
    __syncthreads();
    for (uint32_t done = 0; done < total; done += ROW_BATCH)
    {
      uint32_t m = bits, k = off;
      while (m && k < done + ROW_BATCH)
      {
        const int s = w * 32 + __ffs(m) - 1;
        m &= m - 1u;
        if (k >= done) { sIdx[k - done] = s; sX[k - done] = b.xSpan[s]; }
        k++;
      }
      __syncthreads();
      const int n = (int)min((uint32_t)ROW_BATCH, total - done);
      if (x < b.nx)
        for (int j = 0; j < n; j++)
        {
          const int2 xs = sX[j];
          if (xs.x <= x && x <= xs.y)
          {
            if (FILL)
            {
              const int s = sIdx[j];
              b.itemSphere[run] = b.spheres[s];
              b.itemIndex[run] = s;
            }
            run++;
          }
        }
      __syncthreads();
    }
  }
  if (!FILL && x < b.nx) b.cells[cell] = run;
}

// the cell offsets: an exclusive scan of the counts in place, the total after the last cell, then the drop word.  A grid with more items
// than its region holds is dropped: drop word 1 (the trace kernels then walk the hierarchy), flags[0] raised to its item count, flags[1]
// counts it.
__global__ void __launch_bounds__(SCAN_THREADS) k_eg_scan(const EyeGridBuild b)
{
  const uint32_t n = (uint32_t)b.nx * (uint32_t)b.ny, per = (n + SCAN_THREADS - 1) / SCAN_THREADS;
  const uint32_t t0 = min(n, threadIdx.x * per), t1 = min(n, t0 + per);
  uint32_t sum = 0;
  for (uint32_t c = t0; c < t1; c++) sum += b.cells[c];
  __shared__ uint32_t sWarp[SCAN_THREADS / 32];
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  uint32_t inc = sum;
  for (int o = 1; o < 32; o <<= 1)
  {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, o);
    if (lane >= o) inc += t;
  }
  if (lane == 31) sWarp[warp] = inc;
  __syncthreads();
  if (warp == 0)
  {
    uint32_t w = sWarp[lane], wi = w;
    for (int o = 1; o < 32; o <<= 1)
    {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, wi, o);
      if (lane >= o) wi += t;
    }
    sWarp[lane] = wi - w;   // exclusive
  }
  __syncthreads();
  uint32_t run = sWarp[warp] + inc - sum;
  for (uint32_t c = t0; c < t1; c++) { const uint32_t k = b.cells[c]; b.cells[c] = run; run += k; }
  if (threadIdx.x != SCAN_THREADS - 1) return;
  b.cells[n] = run;
  const bool drop = run > b.itemCap;
  b.cells[n + 1] = drop ? 1u : 0u;
  if (drop)
  {
    atomicMax(b.flags, run);
    atomicAdd(b.flags + 1, 1u);
  }
}

} // namespace

int launchEyeGridBuild(const EyeGridBuild & b, cudaStream_t st)
{
  const size_t maskBytes = (size_t)b.ny * b.maskWords * sizeof(uint32_t);
  if (maskBytes && cudaMemsetAsync(b.rowMask, 0, maskBytes, st) != cudaSuccess) return 0;
  int n = 0;
  if (b.nSpheres) { k_eg_span<<<(b.nSpheres + SPAN_THREADS - 1) / SPAN_THREADS, SPAN_THREADS, 0, st>>>(b); n++; }
  const unsigned rowCtas = (unsigned)b.ny * (unsigned)((b.nx + ROW_THREADS - 1) / ROW_THREADS);
  k_eg_rows<false><<<rowCtas, ROW_THREADS, 0, st>>>(b);
  k_eg_scan<<<1, SCAN_THREADS, 0, st>>>(b);
  k_eg_rows<true><<<rowCtas, ROW_THREADS, 0, st>>>(b);
  return n + 3;
}

} // namespace rfx
