// Connected regions of a cluster map (mdkm_bind_regions): maximal 4- or 8-connected sets of
// pixels of one day with the same non-zero map value (label + 1), numbered 1..R in the raster
// order (day, y, x) of each region's first pixel, and their point statistics.
//
// Block-based union-find (Playne & Hawick 2018; Allegretti, Bolelli & Grana 2019) on int32
// parents that are global pixel indices of the whole stack; a parent is never larger than its
// child, so every tree's root is its region's smallest pixel index -- the first pixel in raster
// order -- and the region id is one plus the number of roots before it:
//   region_tile_kernel     one CTA per 32 x 32 tile of a day: union-find on tile-local indices
//                          in shared memory, each pixel's parent = its tile component's root;
//   region_border_kernel   one warp per tile: the pixels of its top row and left column union
//                          with their neighbours across the border (global atomicMin links);
//   region_number_kernel   roots (parent == self) counted per 4096-pixel chunk, a decoupled
//                          look-back scan over the chunks, every root gets its id;
//   region_resolve_kernel  every pixel takes its root's id (path splitting on the way), 0 where
//                          the pixel has no point;
//   region_stats_kernel    over the resident points: count, fixed-point coordinate sums and
//                          bounds of each point's region;
//   region_finish_kernel   the table and the means.
#pragma once
#include "common.cuh"
#include "lloyd.cuh"
#include "ptx.cuh"

namespace mdkm {

constexpr int kRegTile = 32;                        // tile side: one warp-wide row
constexpr int kRegChunk = kThreads * 16;            // pixels per chunk of the numbering scan

struct RegionParams {
  const void* map;                // [D][H][W] cluster map of the whole stack, 1 or 2 bytes a pixel
  int* parent;                    // [n_px] union-find parents (global pixel index; -1: no point)
  int* ids;                       // [n_px] region ids, 0 where the pixel has no point
  long long n_px;                 // D * H * W (< 2^31)
  long long HW;
  int H, W;
  int tiles_x, tiles_y;
  long long n_tiles;
  unsigned long long* status;     // [chunks] look-back words of the numbering, zeroed before it
  unsigned int* ticket;           // [0] chunk ticket, [1] fault flag (look-back timed out); zeroed
  unsigned long long* n_regions;  // R, written by the CTA of the last chunk
};

__device__ __forceinline__ void region_tile_of(const RegionParams& p, long long t, int& x0, int& y0,
                                               long long& day_base) {
  const int tx = (int)(t % p.tiles_x);
  t /= p.tiles_x;
  const int ty = (int)(t % p.tiles_y);
  x0 = tx * kRegTile;
  y0 = ty * kRegTile;
  day_base = (t / p.tiles_y) * p.HW;
}

__device__ __forceinline__ int tile_find(const volatile int* s, int i) {
  int q;
  while ((q = s[i]) != i) i = q;
  return i;
}

// links the trees of a and b: the larger root under the smaller one, retried when another
// thread relinked the root first
__device__ __forceinline__ void tile_union(int* s, int a, int b) {
  for (;;) {
    a = tile_find(s, a);
    b = tile_find(s, b);
    if (a == b) return;
    if (a > b) { const int t = a; a = b; b = t; }
    const int old = atomicMin(s + b, a);
    if (old == b) return;
    b = old;
  }
}

__device__ __forceinline__ int grid_find(const int* parent, int i) {
  for (;;) {
    const int q = (int)ld_relaxed_gpu_u32(parent + i);
    if (q == i) return i;
    i = q;
  }
}

__device__ __forceinline__ void grid_union(int* parent, int a, int b) {
  for (;;) {
    a = grid_find(parent, a);
    b = grid_find(parent, b);
    if (a == b) return;
    if (a > b) { const int t = a; a = b; b = t; }
    const int old = atomicMin(parent + b, a);
    if (old == b) return;
    b = old;
  }
}

// ---------------------------------------------------------------------------------------
// Tile-local labelling.  A warp reads a row of the tile (coalesced), and the pixels that
// continue their left neighbour's run point straight at the run's first pixel (one ballot), so
// only the links between rows need union-find: a pixel links to the row above only where the
// pixel to its left in the same run has not already linked that run above.  Pixels outside the
// day (H, W not multiples of the tile) are value 0 and are not written.
// ---------------------------------------------------------------------------------------
template <typename T, bool kConn8>
__global__ void __launch_bounds__(kThreads) region_tile_kernel(const RegionParams p) {
  __shared__ int s_par[kRegTile * kRegTile];
  __shared__ unsigned short s_val[kRegTile * kRegTile];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int x0, y0;
  long long day_base;
  region_tile_of(p, blockIdx.x, x0, y0, day_base);
  const T* map = static_cast<const T*>(p.map) + day_base;
  const int x = x0 + lane;
  for (int r = warp; r < kRegTile; r += kThreads / 32) {
    const int y = y0 + r, i = r * kRegTile + lane;
    const unsigned int v = (x < p.W && y < p.H) ? (unsigned int)map[(long long)y * p.W + x] : 0u;
    const unsigned int left = __shfl_up_sync(0xffffffffu, v, 1);
    const unsigned int runs = __ballot_sync(0xffffffffu, lane > 0 && v != 0u && left == v);
    // the run's first lane: the highest lane up to this one that does not continue its left neighbour
    const int start = 31 - __clz(~runs & (0xffffffffu >> (31 - lane)));
    s_val[i] = (unsigned short)v;
    s_par[i] = r * kRegTile + start;
  }
  __syncthreads();
  for (int r = warp; r < kRegTile; r += kThreads / 32) {
    const int i = r * kRegTile + lane;
    const unsigned int v = s_val[i];
    if (r == 0 || v == 0u) continue;
    const bool left = lane > 0 && s_val[i - 1] == v;
    const bool up = s_val[i - kRegTile] == v;
    const bool up_left = lane > 0 && s_val[i - kRegTile - 1] == v;
    if (kConn8) {
      const bool up_right = lane < kRegTile - 1 && s_val[i - kRegTile + 1] == v;
      if (left) {
        if (!up && up_right) tile_union(s_par, i, i - kRegTile + 1);
      } else if (up) {
        tile_union(s_par, i, i - kRegTile);
      } else {
        if (up_left) tile_union(s_par, i, i - kRegTile - 1);
        if (up_right) tile_union(s_par, i, i - kRegTile + 1);
      }
    } else if (up && !(left && up_left)) {
      tile_union(s_par, i, i - kRegTile);
    }
  }
  __syncthreads();
  for (int r = warp; r < kRegTile; r += kThreads / 32) {
    const int y = y0 + r, i = r * kRegTile + lane;
    if (x >= p.W || y >= p.H) continue;
    int out = -1;
    if (s_val[i]) {
      const int root = tile_find(s_par, i);
      out = (int)(day_base + (long long)(y0 + root / kRegTile) * p.W + x0 + root % kRegTile);
    }
    p.parent[day_base + (long long)y * p.W + x] = out;
  }
}

// ---------------------------------------------------------------------------------------
// Links across tile borders.  Lane l of the warp of a tile takes pixel l of the tile's top row
// (its neighbours in the row above) and pixel l of its left column (its neighbours in the column
// to the left).  Every edge between two tiles has an end on one of these; with 8-connectivity a
// neighbour run that the direct neighbour continues is linked through that neighbour.
// ---------------------------------------------------------------------------------------
template <typename T, bool kConn8>
__global__ void __launch_bounds__(kThreads) region_border_kernel(const RegionParams p) {
  const int lane = threadIdx.x & 31;
  const long long t = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  if (t >= p.n_tiles) return;
  int x0, y0;
  long long day_base;
  region_tile_of(p, t, x0, y0, day_base);
  const T* map = static_cast<const T*>(p.map) + day_base;
  const int W = p.W, H = p.H;
  auto link = [&](int y, int x, int yn, int xn) {  // (the caller checked that both are in the day)
    grid_union(p.parent, (int)(day_base + (long long)y * W + x), (int)(day_base + (long long)yn * W + xn));
  };
  if (y0 > 0 && x0 + lane < W) {
    const int y = y0, x = x0 + lane;
    const T v = map[(long long)y * W + x];
    const T* above = map + (long long)(y - 1) * W;
    if (v) {
      if (above[x] == v) {
        link(y, x, y - 1, x);
      } else if (kConn8) {
        if (x > 0 && above[x - 1] == v) link(y, x, y - 1, x - 1);
        if (x + 1 < W && above[x + 1] == v) link(y, x, y - 1, x + 1);
      }
    }
  }
  if (x0 > 0 && y0 + lane < H) {
    const int y = y0 + lane, x = x0;
    const T v = map[(long long)y * W + x];
    if (v) {
      if (map[(long long)y * W + x - 1] == v) {
        link(y, x, y, x - 1);
      } else if (kConn8) {
        if (y > 0 && map[(long long)(y - 1) * W + x - 1] == v) link(y, x, y - 1, x - 1);
        if (y + 1 < H && map[(long long)(y + 1) * W + x - 1] == v) link(y, x, y + 1, x - 1);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// Region ids of the roots: thread j of a chunk's CTA takes 16 consecutive pixels, a root is a
// pixel that is its own parent; CTA scan, then the look-back over the chunks (handed out in
// order by the ticket), then id = 1 + roots before it.  The CTA of the last chunk writes R.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) region_number_kernel(const RegionParams p) {
  __shared__ unsigned int s_warp[kThreads / 32];
  __shared__ long long s_chunk;
  __shared__ unsigned long long s_base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_chunk = atomicAdd(p.ticket, 1u);
  __syncthreads();
  const long long c = s_chunk;
  const long long i0 = c * kRegChunk + (long long)tid * 16;
  unsigned int roots = 0u;
  if (i0 + 16 <= p.n_px) {
    const int4* v = reinterpret_cast<const int4*>(p.parent + i0);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int4 q = __ldg(v + j);
      const long long b = i0 + 4 * j;
      roots |= ((q.x == (int)b) ? 1u : 0u) << (4 * j);
      roots |= ((q.y == (int)(b + 1)) ? 1u : 0u) << (4 * j + 1);
      roots |= ((q.z == (int)(b + 2)) ? 1u : 0u) << (4 * j + 2);
      roots |= ((q.w == (int)(b + 3)) ? 1u : 0u) << (4 * j + 3);
    }
  } else {
    for (int e = 0; e < 16; ++e)
      if (i0 + e < p.n_px && __ldg(p.parent + i0 + e) == (int)(i0 + e)) roots |= 1u << e;
  }
  const unsigned int cnt = (unsigned int)__popc(roots);
  unsigned int incl = cnt;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const unsigned int o = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += o;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  unsigned int before = 0u, agg = 0u;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    before += w < warp ? s_warp[w] : 0u;
    agg += s_warp[w];
  }
  if (warp == 0) {
    unsigned long long excl = 0ull;
    if (c == 0) {
      if (lane == 0) st_status(p.status, kStPrefix | agg);
    } else {
      if (lane == 0) st_status(p.status + c, kStAggregate | agg);
      excl = tile_lookback(p.status, c, agg, lane, p.ticket + 1);
    }
    if (lane == 0) {
      s_base = excl;
      if ((c + 1) * kRegChunk >= p.n_px) *p.n_regions = excl + agg;
    }
  }
  __syncthreads();
  int id = (int)(1ull + s_base + before + incl - cnt);
  while (roots) {
    const int e = __ffs(roots) - 1;
    roots &= roots - 1u;
    p.ids[i0 + e] = id++;
  }
}

// ---------------------------------------------------------------------------------------
// Every pixel -> its root's id.  A warp takes 128 consecutive pixels, lane l pixels l, l + 32,
// l + 64, l + 96 (coalesced).  Path splitting: each parent on the way is replaced by its
// grandparent, so later walks through the same trees are shorter (parents stay ancestors).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) region_resolve_kernel(const RegionParams p) {
  const int lane = threadIdx.x & 31;
  const long long n_warps = (long long)gridDim.x * (kThreads / 32);
  for (long long w = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); w * 128 < p.n_px; w += n_warps) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const long long i = w * 128 + e * 32 + lane;
      if (i >= p.n_px) continue;
      int x = (int)i;
      int q = (int)ld_relaxed_gpu_u32(p.parent + i);
      if (q < 0) {
        p.ids[i] = 0;
        continue;
      }
      if (q == x) continue;  // a root: region_number_kernel wrote its id
      for (;;) {
        const int g = (int)ld_relaxed_gpu_u32(p.parent + q);
        if (g == q) break;
        st_relaxed_gpu_u32(p.parent + x, (unsigned int)g);
        x = q;
        q = g;
      }
      p.ids[i] = p.ids[q];
    }
  }
}

struct RegionStatsParams {
  const float* pts;           // resident cloud (blocked), reference point order
  long long n;
  const long long* seg;       // [nseg + 1] point offsets of the days of the range
  int nseg;
  long long pix0;             // global pixel (0, 0) of segment 0's day
  long long HW;
  int W;
  const int* ids;             // [stack pixels] region ids
  double origin[3], scale[3]; // the fixed-point frame (Frame)
  unsigned long long* acc;    // [R][4] (qx, qy, qz, count), cleared by the host
  unsigned int* box;          // [R][5] first pixel, y_min, x_min, ~y_max, ~x_max (min), set to ~0 by the host
};

// A coordinate on the fixed-point grid: q = rint((x - origin) * scale), evaluated exactly in FP64
// ((double)x - origin and the power-of-two scale lose nothing), so every point moves to its
// nearest grid point and a region's mean is within half a grid step of the exact mean even for a
// region of one point.  (The FP32 form of the Lloyd sums rounds x - origin first, which can add
// up to a quarter of a step per point.)  On-grid coordinates give the same q either way.
__device__ __forceinline__ int grid_coord(float x, double origin, double scale) {
  return __double2int_rn(((double)x - origin) * scale);
}

// ---------------------------------------------------------------------------------------
// Per-region sums over this rank's points.  A warp walks a contiguous run of 128-point groups;
// lane l takes points 4l..4l+3 of a group.  The day comes from a forward-only cursor over the
// segment offsets, the pixel from the exact x, y.  Lanes with equal regions are combined first
// (__match_any_sync, as in stats_add), and the leader adds the group's sums with 64-bit atomics
// and its bounds with 32-bit atomicMin.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) region_stats_kernel(const RegionStatsParams p) {
  const int lane = threadIdx.x & 31;
  const long long n_groups = (p.n + kGroup - 1) / kGroup;
  const long long n_warps = (long long)gridDim.x * (kThreads / 32);
  const long long per_warp = (n_groups + n_warps - 1) / n_warps;
  const long long g_first = ((long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5)) * per_warp;
  const long long g_last = min(n_groups, g_first + per_warp);
  if (g_first >= g_last) return;
  int day = 0;
  {
    const long long i = g_first * kGroup + lane * 4;
    int lo = 0, hi = p.nseg;
    while (hi - lo > 1) {
      const int mid = (lo + hi) >> 1;
      if (__ldg(p.seg + mid) <= i) lo = mid; else hi = mid;
    }
    day = lo;
  }
  long long next = __ldg(p.seg + day + 1);
  for (long long g = g_first; g < g_last; ++g) {
    const float* blk = p.pts + g * kBlockFloats + lane * 4;
    const float4 vx = ldg_stream_f4(blk), vy = ldg_stream_f4(blk + kGroup), vz = ldg_stream_f4(blk + 2 * kGroup);
    const float xo[4] = {vx.x, vx.y, vx.z, vx.w}, yo[4] = {vy.x, vy.y, vy.z, vy.w}, zo[4] = {vz.x, vz.y, vz.z, vz.w};
    const long long i0 = g * kGroup + lane * 4;
    int key[4], qx[4], qy[4], qz[4], px[4], py[4];
    unsigned int gpix[4], rem = 0u;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      key[e] = -1;
      px[e] = pixel_index(xo[e]);
      py[e] = pixel_index(yo[e]);
      gpix[e] = ~0u;
      if (i0 + e < p.n) {
        while (i0 + e >= next) next = __ldg(p.seg + ++day + 1);
        const long long pix = p.pix0 + (long long)day * p.HW + (long long)py[e] * p.W + px[e];
        gpix[e] = (unsigned int)pix;
        key[e] = __ldg(p.ids + pix) - 1;
        rem |= 1u << e;
      }
      qx[e] = grid_coord(xo[e], p.origin[0], p.scale[0]);
      qy[e] = grid_coord(yo[e], p.origin[1], p.scale[1]);
      qz[e] = grid_coord(zo[e], p.origin[2], p.scale[2]);
    }
    while (__any_sync(0xffffffffu, rem != 0u)) {
      const int mine = (rem & 1u) ? key[0] : ((rem & 2u) ? key[1] : ((rem & 4u) ? key[2] : ((rem & 8u) ? key[3] : -1)));
      int sx = 0, sy = 0, sz = 0, sc = 0;
      unsigned int first = ~0u, y_min = ~0u, x_min = ~0u, ny_max = ~0u, nx_max = ~0u;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const bool hit = ((rem >> e) & 1u) && key[e] == mine;
        if (hit) {
          first = min(first, gpix[e]);  // the region's first pixel: its smallest global index
          sx += qx[e];
          sy += qy[e];
          sz += qz[e];
          ++sc;
          y_min = min(y_min, (unsigned int)py[e]);
          x_min = min(x_min, (unsigned int)px[e]);
          ny_max = min(ny_max, ~(unsigned int)py[e]);
          nx_max = min(nx_max, ~(unsigned int)px[e]);
          rem &= ~(1u << e);
        }
      }
      const unsigned int peers = __match_any_sync(0xffffffffu, mine);
      sx = __reduce_add_sync(peers, sx);
      sy = __reduce_add_sync(peers, sy);
      sz = __reduce_add_sync(peers, sz);
      sc = __reduce_add_sync(peers, sc);
      first = __reduce_min_sync(peers, first);
      y_min = __reduce_min_sync(peers, y_min);
      x_min = __reduce_min_sync(peers, x_min);
      ny_max = __reduce_min_sync(peers, ny_max);
      nx_max = __reduce_min_sync(peers, nx_max);
      if (mine >= 0 && lane == __ffs(peers) - 1) {
        unsigned long long* a = p.acc + (size_t)mine * 4;
        atomicAdd(a + 0, (unsigned long long)(long long)sx);
        atomicAdd(a + 1, (unsigned long long)(long long)sy);
        atomicAdd(a + 2, (unsigned long long)(long long)sz);
        atomicAdd(a + 3, (unsigned long long)sc);
        unsigned int* b = p.box + (size_t)mine * 5;
        atomicMin(b + 0, first);
        atomicMin(b + 1, y_min);
        atomicMin(b + 2, x_min);
        atomicMin(b + 3, ny_max);
        atomicMin(b + 4, nx_max);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// Region table (int64 [R][7]: day, cluster, pixels, y_min, x_min, y_max, x_max) and means
// (float64 [R][3], the clustered frame) from the summed slots; the means as day_stats_kernel
// computes them.  The day and the cluster come from the region's first pixel.
// ---------------------------------------------------------------------------------------
__global__ void region_finish_kernel(const unsigned long long* acc, const unsigned int* box, long long n_regions,
                                     const void* map, int map_elem, long long HW, Frame fr, long long* table,
                                     double* means) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < n_regions;
       r += (long long)gridDim.x * blockDim.x) {
    const long long cnt = (long long)acc[r * 4 + 3];
    const unsigned int* b = box + r * 5;
    const long long first = (long long)b[0];
    const int v = map_elem == 1 ? (int)static_cast<const unsigned char*>(map)[first]
                                : (int)static_cast<const unsigned short*>(map)[first];
    long long* t = table + r * 7;
    t[0] = first / HW;
    t[1] = v - 1;
    t[2] = cnt;
    t[3] = (long long)b[1];
    t[4] = (long long)b[2];
    t[5] = (long long)~b[3];
    t[6] = (long long)~b[4];
    for (int d = 0; d < 3; ++d) {
      const double sum = __dadd_rn(__ddiv_rn((double)(long long)acc[r * 4 + d], fr.scale[d]),
                                   __dmul_rn((double)cnt, fr.origin[d]));
      means[r * 3 + d] = __ddiv_rn(sum, (double)cnt);
    }
  }
}

}  // namespace mdkm
