// rfx_light_grid.cu — a far light's shadow-ray candidate grid (LightGrid) built on the device, from the spheres of the blob and the
// sphere hierarchy's leaf slots: rfx_update_lights (a light moved) and rfx_update_spheres (the spheres moved) rebuild grids here instead
// of on the host.  The grid is byte for byte the one rfx_scene.cpp buildLightGrid builds for the same spheres, box and R: both run the
// arithmetic of rfx_light_grid.h (--fmad=false here, -ffp-contract=off there), minima and maxima do not depend on their order, the sum of
// the disc radii has the one shape both sides use (LIGHT_GRID_SUM_BLOCK), and the items of a cell are listed in leaf-slot order.
//
// One build is six launches on the caller's stream, no synchronisation:
//   k_lg_disc   one thread per leaf slot: the sphere's disc (pu, pv, rho), the extent's minima / maxima, each block's sum of rho
//   k_lg_dims   one thread: the sum over the blocks, the cells (lightGridDims) and the header, or a NULL header (no grid)
//   k_lg_rect   one thread per leaf slot: the disc's rectangle of cells
//   k_lg_rows   one CTA per grid row, one thread per cell of the row: the row's discs in slot order, each tested against the thread's
//               cell — a count per cell, then (FILL) the items.  A disc that covers 257 x 257 cells is 257 CTAs' work, one test per thread.
//   k_lg_scan   one CTA: the cell offsets (exclusive scan, in place); a grid that does not fit its region loses its header (NULL)
//   k_lg_rows<FILL>
#include "rfx_kernels.h"
#include "rfx_light_grid.h"

namespace rfx
{

namespace
{

constexpr int DISC_THREADS = LIGHT_GRID_SUM_BLOCK;   // one CTA per block of the rho sum
constexpr int ROW_THREADS = 288;                     // >= LIGHT_GRID_MAX_DIM: one thread per cell of a row
constexpr int SCAN_THREADS = 1024;
constexpr uint32_t EMPTY_SPAN = 0xFFFFu;             // lo = 0xFFFF > hi = 0

static_assert(ROW_THREADS >= LIGHT_GRID_MAX_DIM && ROW_THREADS % 32 == 0, "one thread per cell of a row");

__global__ void __launch_bounds__(DISC_THREADS) k_lg_disc(const LightGridBuild b)
{
  const int s = blockIdx.x * DISC_THREADS + threadIdx.x;
  __shared__ double sRho[DISC_THREADS];
  __shared__ bool sUsed[DISC_THREADS];
  __shared__ double sRed[4][DISC_THREADS / 32];
  double pu = 0.0, pv = 0.0, rho = 0.0;
  bool used = false;
  if (s < b.nSlots)
  {
    const int p = b.prims[s];
    if (p >= 0)
    {
      const float4 q = b.spheres[p];
      const float c[3] = { q.x, q.y, q.z };
      const float r = b.radius[p];
      if (lightDisc(b.f, c, r, sphereMargin(r, b.R), pu, pv, rho)) used = true;
      else b.red[4] = 1ull;                             // no finite sMax: no grid
    }
  }
  if (used) { b.disc[3 * (size_t)s] = pu; b.disc[3 * (size_t)s + 1] = pv; b.disc[3 * (size_t)s + 2] = rho; }
  sRho[threadIdx.x] = rho; sUsed[threadIdx.x] = used;
  // the extent: minima and maxima (NaN ignored, as std::min / std::max over a finite start ignore it)
  double v[4] = { 1e300, -1e300, 1e300, -1e300 };
  if (used)
  {
    const double a = pu - rho, bb = pu + rho, c = pv - rho, d = pv + rho;
    if (a == a) v[0] = a;
    if (bb == bb) v[1] = bb;
    if (c == c) v[2] = c;
    if (d == d) v[3] = d;
  }
  for (int o = 16; o > 0; o >>= 1)
  {
    v[0] = dmin(v[0], __shfl_xor_sync(0xFFFFFFFFu, v[0], o)); v[1] = dmax(v[1], __shfl_xor_sync(0xFFFFFFFFu, v[1], o));
    v[2] = dmin(v[2], __shfl_xor_sync(0xFFFFFFFFu, v[2], o)); v[3] = dmax(v[3], __shfl_xor_sync(0xFFFFFFFFu, v[3], o));
  }
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  if (lane == 0)
    for (int k = 0; k < 4; k++) sRed[k][warp] = v[k];
  __syncthreads();
  if (threadIdx.x != 0) return;
  for (int w = 1; w < DISC_THREADS / 32; w++)
  {
    v[0] = dmin(v[0], sRed[0][w]); v[1] = dmax(v[1], sRed[1][w]);
    v[2] = dmin(v[2], sRed[2][w]); v[3] = dmax(v[3], sRed[3][w]);
  }
  atomicMin(b.red + 0, orderedCode(v[0])); atomicMax(b.red + 1, orderedCode(v[1]));
  atomicMin(b.red + 2, orderedCode(v[2])); atomicMax(b.red + 3, orderedCode(v[3]));
  // this block's part of the rho sum: sequential in slot order over the used slots
  double part = 0.0;
  for (int k = 0; k < DISC_THREADS; k++)
    if (sUsed[k]) part += sRho[k];
  b.blockSum[blockIdx.x] = part;
}

__global__ void k_lg_dims(const LightGridBuild b, int nBlocks)
{
  double e[4];
  for (int k = 0; k < 4; k++) e[k] = orderedValue(b.red[k]);
  const bool bad = b.red[4] != 0ull;
  // ready for the next build (k_lg_disc of this one has finished)
  b.red[0] = orderedCode(1e300); b.red[1] = orderedCode(-1e300); b.red[2] = orderedCode(1e300); b.red[3] = orderedCode(-1e300); b.red[4] = 0ull;
  double rhoSum = 0.0;
  for (int k = 0; k < nBlocks; k++) rhoSum += b.blockSum[k];
  LightGridDims d;
  memset(&d, 0, sizeof(d));
  LightGrid g;
  memset(&g, 0, sizeof(g));
  if (!bad && lightGridDims(e[0], e[1], e[2], e[3], rhoSum, b.nPrims, d))
  {
    lightGridHeader(b.f, d, g);
    g.cellStart = b.cells; g.itemSphere = b.itemSphere; g.itemIndex = b.itemIndex;
  }
  else
    d.nx = d.ny = 0;
  *b.header = g;
  *b.dims = d;
  *b.dropped = 0u;
}

__global__ void __launch_bounds__(DISC_THREADS) k_lg_rect(const LightGridBuild b)
{
  const int s = blockIdx.x * DISC_THREADS + threadIdx.x;
  if (s >= b.nSlots) return;
  const LightGridDims d = *b.dims;
  if (d.nx == 0) return;
  uint32_t xs = EMPTY_SPAN, ys = EMPTY_SPAN;
  if (b.prims[s] >= 0)
  {
    int x0, x1, y0, y1;
    lightCellsOf(d, b.disc[3 * (size_t)s], b.disc[3 * (size_t)s + 1], b.disc[3 * (size_t)s + 2], x0, x1, y0, y1);
    if (x0 <= x1 && y0 <= y1) { xs = (uint32_t)x0 | ((uint32_t)x1 << 16); ys = (uint32_t)y0 | ((uint32_t)y1 << 16); }
  }
  b.span[2 * (size_t)s] = xs; b.span[2 * (size_t)s + 1] = ys;
}

// One CTA per row y, thread x for cell (x, y).  The CTA walks the leaf slots in chunks of ROW_THREADS, compacts the chunk's discs whose
// rectangle covers row y (in slot order) into shared memory, and every thread tests those that cover its column against its cell.
// The count pass stores the number of discs per cell; the fill pass writes them from the cell's offset on, in slot order.
template <bool FILL>
__global__ void __launch_bounds__(ROW_THREADS) k_lg_rows(const LightGridBuild b)
{
  const LightGridDims d = *b.dims;
  const int y = blockIdx.x, x = threadIdx.x;
  if (d.nx == 0 || y >= d.ny) return;
  __shared__ int sSlot[ROW_THREADS];
  __shared__ uint32_t sX[ROW_THREADS];
  __shared__ double sPu[ROW_THREADS], sPv[ROW_THREADS], sRho[ROW_THREADS];
  __shared__ int sWarp[ROW_THREADS / 32];
  const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const size_t cell = (size_t)y * d.nx + x;
  uint32_t run = (FILL && x < d.nx) ? b.cells[cell] : 0u;
  for (int base = 0; base < b.nSlots; base += ROW_THREADS)
  {
    const int s = base + threadIdx.x;
    bool in = false;
    if (s < b.nSlots)
    {
      const uint32_t ys = b.span[2 * (size_t)s + 1];
      in = (int)(ys & 0xFFFFu) <= y && y <= (int)(ys >> 16);
    }
    const uint32_t ballot = __ballot_sync(0xFFFFFFFFu, in);
    if (lane == 0) sWarp[warp] = __popc(ballot);
    __syncthreads();
    int off = 0, total = 0;
    for (int w = 0; w < ROW_THREADS / 32; w++) { off += w < warp ? sWarp[w] : 0; total += sWarp[w]; }
    if (in)
    {
      const int k = off + __popc(ballot & ((1u << lane) - 1u));
      sSlot[k] = s;
      sX[k] = b.span[2 * (size_t)s];
      sPu[k] = b.disc[3 * (size_t)s]; sPv[k] = b.disc[3 * (size_t)s + 1]; sRho[k] = b.disc[3 * (size_t)s + 2];
    }
    __syncthreads();
    if (x < d.nx)
      for (int k = 0; k < total; k++)
      {
        const uint32_t xs = sX[k];
        if ((int)(xs & 0xFFFFu) <= x && x <= (int)(xs >> 16) && lightTouches(d, sPu[k], sPv[k], sRho[k], x, y))
        {
          if (FILL)
          {
            const int p = b.prims[sSlot[k]];
            b.itemSphere[run] = b.spheres[p];
            b.itemIndex[run] = p;
          }
          run++;
        }
      }
  }
  if (!FILL && x < d.nx) b.cells[cell] = run;
}

// the cell offsets: an exclusive scan of the counts in place, the total after the last cell.  A grid with more items than its region
// holds is dropped: NULL header (its shadow queries walk the hierarchy), *dropped set, *need raised to its item count.
__global__ void __launch_bounds__(SCAN_THREADS) k_lg_scan(const LightGridBuild b)
{
  const LightGridDims d = *b.dims;
  if (d.nx == 0) return;
  const uint32_t n = (uint32_t)d.nx * (uint32_t)d.ny, per = (n + SCAN_THREADS - 1) / SCAN_THREADS;
  const uint32_t t0 = min(n, threadIdx.x * per), t1 = min(n, t0 + per);
  uint32_t sum = 0;
  for (uint32_t c = t0; c < t1; c++) sum += b.cells[c];
  // exclusive scan of the threads' sums: within each warp, then over the warps
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
  // the last thread's running sum is the item count
  b.cells[n] = run;
  if (run > b.itemCap)
  {
    LightGrid g;
    memset(&g, 0, sizeof(g));
    *b.header = g;
    b.dims->nx = 0;                                  // the fill pass writes nothing
    *b.dropped = 1u;
    atomicMax(b.need, run);
  }
}

} // namespace

int launchLightGridBuild(const LightGridBuild & b, cudaStream_t st)
{
  const int blocks = (b.nSlots + DISC_THREADS - 1) / DISC_THREADS;
  if (blocks) k_lg_disc<<<blocks, DISC_THREADS, 0, st>>>(b);
  k_lg_dims<<<1, 1, 0, st>>>(b, blocks);
  if (!blocks) return 2;
  k_lg_rect<<<blocks, DISC_THREADS, 0, st>>>(b);
  k_lg_rows<false><<<LIGHT_GRID_MAX_DIM, ROW_THREADS, 0, st>>>(b);
  k_lg_scan<<<1, SCAN_THREADS, 0, st>>>(b);
  k_lg_rows<true><<<LIGHT_GRID_MAX_DIM, ROW_THREADS, 0, st>>>(b);
  return 6;
}

} // namespace rfx
