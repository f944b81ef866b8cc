// Tile-ordered mirror of the resident cloud -- the copy the Lloyd iterations stream.
//
// The resident cloud keeps the reference's point order (np.where order: day-major, row-major,
// members/rafael/disparity/plugin.py:157), because labels, k-means++ draws and relocation ties
// are defined in that order.  In that order a group of 128 consecutive points is a 128 x 1
// pixel strip: long and thin, so a cluster boundary crosses many groups and each of them
// needs the per-point pass.  The mirror holds the same points re-ordered by the cells of an
// x-y grid with about 256 points per cell (the points of all days at those pixels): 128 consecutive
// points of the mirror are compact in x and y, far fewer groups touch a boundary, and most of
// them are settled from their cached summaries alone.  Sums are integers and the labels are
// recomputed in the reference's order at the end of a fit, so results do not depend on this
// order (nor on the arrival order of the points inside a cell, which the atomic cursors leave
// open).
//
// Built once per (cloud, frame): histogram of the points over the cells, exclusive scan,
// scatter -- two reads of the cloud and one write.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace mdkm {

constexpr int kMirrorMaxSeg = 1024;  // segment table held in shared memory
constexpr int kMirrorGpb = 32;       // groups per band and segment

struct MirrorGrid {
  float x0, y0;          // lower corner of the cloud's bounding box
  float inv_cx, inv_cy;  // 1 / cell size
  int gx, gy;            // cells per dimension
  int n_seg;
  const long long* seg_off;  // [n_seg + 1] point offsets of the segments (device)
  long long n_virtual;       // n_bands * n_seg * kMirrorGpb
};

// Cell of a point.  Cells are wide in x (a raster row contributes a run of consecutive points
// to a cell, which keeps the scattered writes sector-sized) and short in y.  The rows of cells
// are numbered in serpentine order (odd rows right to left): the group of 128 mirror points that
// straddles the end of one row of cells and the start of the next then covers two cells at the
// same edge of the frame -- in plain row-major order it would span the whole width of the cloud,
// touch every cluster along the row and never be settled (measured: the step kernel of
// config 4, k = 1024, went from 1.22 to 0.61 ms per iteration; the few hundred such groups were
// the tail every iteration waited for).
__device__ __forceinline__ int mirror_cell(const MirrorGrid& g, float x, float y) {
  const int cx = min(g.gx - 1, max(0, (int)((x - g.x0) * g.inv_cx)));
  const int cy = min(g.gy - 1, max(0, (int)((y - g.y0) * g.inv_cy)));
  return cy * g.gx + ((cy & 1) ? g.gx - 1 - cx : cx);
}

// Traversal order of the two passes below: band of rows outermost, segment (day) inside.  The
// points of a cell come from the same few raster rows of EVERY day; visiting those rows of all
// days together keeps the partial writes to the cell's range close in time, so they merge in
// L2 instead of being evicted half-filled.  Days are cut into n_bands runs of kMirrorGpb groups;
// virtual index v = (band * n_seg + seg) * kMirrorGpb + j  ->  group seg_first[seg] + band * kMirrorGpb + j.
// (32-bit arithmetic: v / kMirrorGpb is below 2^32 for any cloud that fits the device.)
__device__ __forceinline__ long long mirror_group_of(const MirrorGrid& g, const long long* s_off, long long v) {
  const unsigned int t = (unsigned int)(v / kMirrorGpb);
  const unsigned int j = (unsigned int)v & (kMirrorGpb - 1);
  const unsigned int band = t / (unsigned int)g.n_seg;
  const unsigned int seg = t - band * (unsigned int)g.n_seg;
  // groups that START inside the segment belong to it (a straddling group goes with its first point)
  const long long first = (s_off[seg] + kGroup - 1) / kGroup;
  const long long last = (s_off[seg + 1] + kGroup - 1) / kGroup;  // exclusive
  const long long grp = first + (long long)band * kMirrorGpb + j;
  return grp < last ? grp : -1;
}

// Runs of equal cells among the 32 consecutive points a warp holds in one round (one point per
// lane).  Consecutive points of a raster row share a cell for cell-width pixels, so a round
// holds a few runs; the first lane of every run acts for it.  `head_lane`: the first lane of
// this lane's run; `run_len`: the length of the run (valid in its first lane).
__device__ __forceinline__ bool mirror_runs(int cell, int lane, int& head_lane, int& run_len) {
  const int prev = __shfl_up_sync(0xffffffffu, cell, 1);
  const bool head = lane == 0 || cell != prev;
  const unsigned int heads = __ballot_sync(0xffffffffu, head);
  head_lane = 31 - __clz(heads & (0xffffffffu >> (31 - lane)));
  const unsigned int later = heads & ~((2u << lane) - 1u);  // heads after this lane
  run_len = (later ? __ffs(later) - 1 : 32) - lane;
  return head;
}

// counts[cell] += 1 for every point: one atomic per run of equal cells.
__global__ void __launch_bounds__(kThreads) mirror_count_kernel(const float* pts, long long n, MirrorGrid g,
                                                                unsigned int* counts) {
  __shared__ long long s_off[kMirrorMaxSeg + 1];
  for (int i = threadIdx.x; i <= g.n_seg; i += kThreads) s_off[i] = g.seg_off[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long stride = (long long)gridDim.x * (kThreads / 32);
  for (long long v = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); v < g.n_virtual; v += stride) {
    const long long grp = mirror_group_of(g, s_off, v);
    if (grp < 0) continue;  // warp-uniform
    const float* blk = pts + grp * kBlockFloats + lane;
    float xs[4], ys[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      xs[r] = __ldg(blk + r * 32);
      ys[r] = __ldg(blk + kGroup + r * 32);
    }
    const bool full = (grp + 1) * kGroup <= n;  // warp-uniform; only the cloud's last group is not
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int cell = (full || grp * kGroup + r * 32 + lane < n) ? mirror_cell(g, xs[r], ys[r]) : -1;
      int head_lane, run_len;
      if (mirror_runs(cell, lane, head_lane, run_len) && cell >= 0) atomicAdd(&counts[cell], (unsigned int)run_len);
    }
  }
}

// Exclusive scan of n 32-bit counts into 64-bit offsets in two launches: per-CTA totals of
// kScanTile counts, then every CTA adds up the totals before it (a few dozen values) and
// scans its own tile.
constexpr int kScanItems = 4;
constexpr int kScanTile = 1024 * kScanItems;

__global__ void __launch_bounds__(1024) mirror_tile_sums_kernel(const unsigned int* counts, long long n,
                                                                long long* tile_sums) {
  __shared__ long long s_warp[32];
  const long long base = (long long)blockIdx.x * kScanTile;
  long long mine = 0;
  for (int e = 0; e < kScanItems; ++e) {
    const long long i = base + (long long)e * 1024 + threadIdx.x;  // coalesced
    mine += i < n ? counts[i] : 0u;
  }
  for (int o = 16; o > 0; o >>= 1) mine += __shfl_down_sync(0xffffffffu, mine, o);
  if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = mine;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long t = 0;
    for (int w = 0; w < 32; ++w) t += s_warp[w];
    tile_sums[blockIdx.x] = t;
  }
}

// counts: capacity padded to a whole tile (the 128-bit loads of the last tile stay inside it).
__global__ void __launch_bounds__(1024) mirror_scan_kernel(const unsigned int* counts, long long n, long long* offsets,
                                                           const long long* tile_sums) {
  static_assert(kScanItems == 4, "one 128-bit load per thread");
  __shared__ long long s_warp[32];
  __shared__ long long s_carry;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid < 32) {  // totals of the tiles before this one
    long long t = 0;
    for (int b = tid; b < (int)blockIdx.x; b += 32) t += tile_sums[b];
    for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
    if (tid == 0) s_carry = t;
  }
  const long long i0 = (long long)blockIdx.x * kScanTile + (long long)tid * kScanItems;
  const uint4 raw = *reinterpret_cast<const uint4*>(counts + i0);
  const unsigned int v[4] = {i0 < n ? raw.x : 0u, i0 + 1 < n ? raw.y : 0u, i0 + 2 < n ? raw.z : 0u,
                             i0 + 3 < n ? raw.w : 0u};
  const long long mine = (long long)v[0] + v[1] + v[2] + v[3];
  long long incl = mine;
  for (int o = 1; o < 32; o <<= 1) {
    const long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[w] = incl;
  __syncthreads();
  if (w == 0) {
    long long ws = s_warp[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const long long t = __shfl_up_sync(0xffffffffu, ws, o);
      if (lane >= o) ws += t;
    }
    s_warp[lane] = ws;
  }
  __syncthreads();
  long long run = s_carry + (w ? s_warp[w - 1] : 0) + (incl - mine);
#pragma unroll
  for (int e = 0; e < kScanItems; ++e) {
    if (i0 + e < n) offsets[i0 + e] = run;
    run += v[e];
  }
}

// dst = (cursor of the cell)++ ; copies x, y, z into the mirror.  `cursors` enters as the
// cells' start offsets (the scan's output) and is consumed: every run of equal cells takes its
// slots with ONE 64-bit atomic on the cell's cursor.  One point per lane and round (four rounds
// per group): the lanes of a run hold consecutive points of a raster row and get consecutive
// slots, so every store instruction writes whole runs instead of 4-byte fragments.  The four
// atomics of a group are issued back to back, before the first result is needed: their round
// trips overlap.
__global__ void __launch_bounds__(kThreads) mirror_scatter_kernel(const float* pts, long long n, MirrorGrid g,
                                                                  unsigned long long* cursors, float* tpts) {
  __shared__ long long s_off[kMirrorMaxSeg + 1];
  for (int i = threadIdx.x; i <= g.n_seg; i += kThreads) s_off[i] = g.seg_off[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long stride = (long long)gridDim.x * (kThreads / 32);
  for (long long v = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); v < g.n_virtual; v += stride) {
    const long long grp = mirror_group_of(g, s_off, v);
    if (grp < 0) continue;  // warp-uniform
    const float* blk = pts + grp * kBlockFloats + lane;
    float xs[4], ys[4], zs[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      xs[r] = __ldg(blk + r * 32);
      ys[r] = __ldg(blk + kGroup + r * 32);
      zs[r] = __ldg(blk + 2 * kGroup + r * 32);
    }
    const bool full = (grp + 1) * kGroup <= n;  // warp-uniform
    int head_lane[4];
    bool valid[4];
    unsigned long long base[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int cell = (full || grp * kGroup + r * 32 + lane < n) ? mirror_cell(g, xs[r], ys[r]) : -1;
      int run_len;
      const bool head = mirror_runs(cell, lane, head_lane[r], run_len);
      valid[r] = cell >= 0;
      base[r] = 0;
      if (head && valid[r]) base[r] = atomicAdd(&cursors[cell], (unsigned long long)run_len);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const unsigned long long b = __shfl_sync(0xffffffffu, base[r], head_lane[r]);
      if (valid[r]) {
        float* q = tpts + pt_off((long long)b + (lane - head_lane[r]));
        q[0] = xs[r];
        q[kGroup] = ys[r];
        q[2 * kGroup] = zs[r];
      }
    }
  }
}

// =======================================================================================
// Raster clouds: the mirror without a histogram pass, atomics or scattered writes.
//
// A cloud that mdkm_unproject produced from whole raster rows comes with a run table
// (UnprojParams::run_src): for every 8 pixels of the range, how many points the pixels before
// them produced.  The points of an 8- or 16-pixel run of one row are consecutive in the cloud,
// the table says where they start and how many there are -- so the size of every cell, and the
// place of every run inside its cell, follow from the table alone (one scan over the runs,
// nothing per point), and the copy itself is a GATHER BY DESTINATION: one warp per group
// of 128 mirror points looks up the handful of runs that make up the group, fetches them
// (64-byte pieces of the cloud), writes the 1536-byte block in one piece and, having the whole
// group in registers, also emits the group's summary (box + fixed-point sums) -- what used to
// be mirror_count + mirror_scatter + group_summary_kernel.  The order inside a cell is fixed
// (day, row, x), so the mirror is deterministic.
// =======================================================================================
#ifndef MDKM_GATHER_CTAS
#define MDKM_GATHER_CTAS 6
#endif
struct RasterGeom {
  const unsigned int* run_src;  // [n_rows * nb8 + 1]
  long long row0;   // global row (day * H + y) of the first row of the range
  long long n_rows; // rows in the range
  int W, H;
  int nb8;          // 8-pixel bins per row (W / 8)
  int cb;           // bins per cell: 1 (8 px) or 2 (16 px)
  int gx;           // cells per row of cells
  int rpc;          // raster rows per cell
  int yshift, yext; // the rows of y the range covers: (yshift + i) mod H for i in [0, yext) -- all H of them
                    // once the range holds a whole day, else the n_rows rows from its first one on
  int gy;           // rows of cells: ceil(yext / rpc)
  int d0, nd;       // first day and number of days the range touches
};

// serpentine numbering of the cells, as above
__device__ __forceinline__ int raster_cell_index(const RasterGeom& g, int cxi, int cyi) {
  return cyi * g.gx + ((cyi & 1) ? g.gx - 1 - cxi : cxi);
}

// points of the run (day d0 + dd, covered row cyi * rpc + ry, bins [cxi * cb, cxi * cb + cb)) and
// the index of its first point in the cloud; 0 points when the row is outside the range
__device__ __forceinline__ unsigned int raster_run(const RasterGeom& g, int cxi, int cyi, int dd, int ry,
                                                   unsigned int& src) {
  src = 0u;
  const int yi = cyi * g.rpc + ry;
  if (yi >= g.yext) return 0u;
  int y = yi + g.yshift;
  if (y >= g.H) y -= g.H;
  const long long lr = (long long)(g.d0 + dd) * g.H + y - g.row0;
  if (lr < 0 || lr >= g.n_rows) return 0u;
  // (the table has pix_count / 8 + 1 < 2^29 + 1 entries: 32-bit indices)
  const unsigned int j0 = (unsigned int)lr * (unsigned int)g.nb8 + (unsigned int)(cxi * g.cb);
  const unsigned int j1 = min(j0 + (unsigned int)g.cb, ((unsigned int)lr + 1u) * (unsigned int)g.nb8);
  src = __ldg(g.run_src + j0);
  return __ldg(g.run_src + j1) - src;
}

// The run list in ONE pass over the run table.  Entries in destination order (cell, day, row):
// entry E = (first mirror slot, first cloud index); an entry's length is the next entry's slot
// minus its own (entry n_entries closes the list).  gfirst[g] = the entry that holds mirror slot
// 128 g.  The slot of an entry is the number of points of all entries before it -- cells are
// consecutive in the mirror -- so the list is an exclusive scan over the entries: a CTA takes a
// tile of kIndexTile consecutive entries by ticket, reads its runs (kIndexItems per thread, all
// loads in flight together), publishes the tile's total and obtains the points of all earlier
// tiles by a decoupled look-back (ptx.cuh).  No per-cell count array, no separate scan launch.
constexpr int kIndexItems = 8;
constexpr int kIndexTile = kThreads * kIndexItems;

// status: [n_tiles] look-back words; ticket[0] = tile counter, ticket[1] = fault flag (look-back
// timed out); all zero before the launch.  n_entries + kIndexTile < 2^32.
__global__ void __launch_bounds__(kThreads) raster_index_kernel(const RasterGeom g, long long n, unsigned int n_entries,
                                                                unsigned long long* status, unsigned int* ticket,
                                                                uint2* druns, unsigned int* gfirst) {
  __shared__ unsigned int s_tile;
  __shared__ unsigned int s_warp[kThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_tile = atomicAdd(ticket, 1u);
  __syncthreads();
  const unsigned int t = s_tile;
  // the gather behind this kernel may be set up (it waits for the whole grid before it reads)
  grid_launch_dependents();
  const unsigned int per_cell = (unsigned int)(g.nd * g.rpc), rpc = (unsigned int)g.rpc, gx = (unsigned int)g.gx;
  const unsigned int e0 = t * kIndexTile + tid * kIndexItems;
  unsigned int cnt[kIndexItems], src[kIndexItems];
  unsigned int tot = 0;
#pragma unroll
  for (int i = 0; i < kIndexItems; ++i) {
    const unsigned int E = e0 + i;
    cnt[i] = 0u;
    src[i] = 0u;
    if (E < n_entries) {
      const unsigned int lin = E / per_cell, e = E - lin * per_cell;
      const unsigned int dd = e / rpc, ry = e - dd * rpc;
      const unsigned int cyi = lin / gx, pos = lin - cyi * gx;
      const unsigned int cxi = (cyi & 1u) ? gx - 1u - pos : pos;  // serpentine, as raster_cell_index
      cnt[i] = raster_run(g, (int)cxi, (int)cyi, (int)dd, (int)ry, src[i]);
    }
    tot += cnt[i];
  }
  unsigned int incl = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int v = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += v;
  }
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    const unsigned int w = lane < kThreads / 32 ? s_warp[lane] : 0u;
    unsigned int ws = w;
#pragma unroll
    for (int o = 1; o < kThreads / 32; o <<= 1) {
      const unsigned int v = __shfl_up_sync(0xffffffffu, ws, o);
      if (lane >= o) ws += v;
    }
    const unsigned int agg = __shfl_sync(0xffffffffu, ws, kThreads / 32 - 1);
    if (t > 0 && lane == 0) st_status(status + t, kStAggregate | agg);
    const unsigned int base = (unsigned int)tile_lookback(status, t, agg, lane, ticket + 1);
    __syncwarp();
    if (lane < kThreads / 32) s_warp[lane] = base + ws - w;  // points before the warp's first entry
  }
  __syncthreads();
  unsigned int dst = s_warp[warp] + incl - tot;
  uint2 out[kIndexItems];
#pragma unroll
  for (int i = 0; i < kIndexItems; ++i) {
    out[i] = make_uint2(dst, src[i]);
    if (cnt[i]) {  // a run is shorter than a group: it holds at most one group start
      const unsigned long long gs = ((unsigned long long)dst + (kGroup - 1)) / kGroup;
      if (gs * kGroup < (unsigned long long)dst + cnt[i]) gfirst[gs] = e0 + i;
    }
    dst += cnt[i];
  }
  if (e0 + kIndexItems <= n_entries) {
    uint4* o4 = reinterpret_cast<uint4*>(druns + e0);  // 64-byte aligned
#pragma unroll
    for (int i = 0; i < kIndexItems / 2; ++i)
      o4[i] = make_uint4(out[2 * i].x, out[2 * i].y, out[2 * i + 1].x, out[2 * i + 1].y);
  } else {
#pragma unroll
    for (int i = 0; i < kIndexItems; ++i)
      if (e0 + i < n_entries) druns[e0 + i] = out[i];
  }
  if (t == 0 && tid == 0) druns[n_entries] = make_uint2((unsigned int)n, 0u);
}

// One warp per group of 128 mirror points: resolve the group's slots to cloud indices through
// the run list (32 entries per window, binary search by shuffles), fetch, write the block, emit
// the summary.  `summaries` is an array of 48-byte GroupSummary records (lloyd.cuh), written as
// three float4 here to keep this header independent of it.
__global__ void __launch_bounds__(kThreads, MDKM_GATHER_CTAS) raster_gather_kernel(const float* __restrict__ pts, long long n,
                                                                 const uint2* __restrict__ druns, long long n_entries,
                                                                 const unsigned int* __restrict__ gfirst, FrameF f,
                                                                 float* __restrict__ tpts, float4* __restrict__ summaries) {
  // launched behind raster_index_kernel with programmatic stream serialisation: nothing of its
  // output is read before the whole index grid has finished
  grid_dependency_wait();
  const int lane = threadIdx.x & 31;
  const long long n_groups = (n + kGroup - 1) / kGroup;
  const long long stride = (long long)gridDim.x * (kThreads / 32);
  // the first window of the NEXT group of this warp (its index entry, then 32 run-list entries) is
  // requested while the current group is worked on: two of the three dependent round trips per
  // group (index -> run list -> points) are off the critical path
  long long grp = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5);
  long long j_next = grp < n_groups ? (long long)__ldg(gfirst + grp) : 0;
  uint2 e_next = make_uint2(0xffffffffu, 0u);
  unsigned int w_end_next = 0;
  if (grp < n_groups) {
    if (j_next + lane < n_entries) e_next = __ldg(druns + j_next + lane);
    w_end_next = __ldg(&druns[min(j_next + 32, n_entries)].x);
  }
  for (; grp < n_groups; grp += stride) {
    const unsigned int base = (unsigned int)(grp * kGroup);
    const unsigned int n32 = (unsigned int)n;
    unsigned int srcs[4] = {0u, 0u, 0u, 0u};
    unsigned int todo = 0;  // rounds whose slot still has to be resolved (bit r)
#pragma unroll
    for (int r = 0; r < 4; ++r)
      if (base + r * 32 + lane < n32) todo |= 1u << r;
    long long j = j_next;
    uint2 e = e_next;
    unsigned int w_end = w_end_next;  // first slot behind the window
    {  // request the next group's first window
      const long long gn = grp + stride;
      if (gn < n_groups) {
        j_next = (long long)__ldg(gfirst + gn);
        e_next = j_next + lane < n_entries ? __ldg(druns + j_next + lane) : make_uint2(0xffffffffu, 0u);
        w_end_next = __ldg(&druns[min(j_next + 32, n_entries)].x);
      }
    }
    bool first_window = true;
    while (__any_sync(0xffffffffu, todo != 0)) {
      if (j >= n_entries) break;  // (cannot happen with a consistent run list; never read out of bounds)
      if (!first_window) {
        const long long jj = j + lane;
        e = jj < n_entries ? __ldg(druns + jj) : make_uint2(0xffffffffu, 0u);
        w_end = __ldg(&druns[min(j + 32, n_entries)].x);
      }
      first_window = false;
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const unsigned int s = base + r * 32 + lane;
        // last entry of the window whose first slot is <= s (empty entries share their successor's slot)
        int t = 0;
#pragma unroll
        for (int step = 16; step > 0; step >>= 1) {
          const unsigned int v = __shfl_sync(0xffffffffu, e.x, t + step);
          if (v <= s) t += step;
        }
        const unsigned int d0 = __shfl_sync(0xffffffffu, e.x, t), s0 = __shfl_sync(0xffffffffu, e.y, t);
        if (((todo >> r) & 1u) && s < w_end) {
          srcs[r] = s0 + (s - d0);
          todo &= ~(1u << r);
        }
      }
      j += 32;
    }
    float xs[4], ys[4], zs[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const bool live = base + r * 32 + lane < n32;
      const float* q = pts + pt_off((long long)srcs[r]);
      xs[r] = live ? __ldg(q) : 0.f;
      ys[r] = live ? __ldg(q + kGroup) : 0.f;
      zs[r] = live ? __ldg(q + 2 * kGroup) : 0.f;
    }
    float* tb = tpts + grp * kBlockFloats + lane;
    float lo[3] = {__int_as_float(0x7f800000), __int_as_float(0x7f800000), __int_as_float(0x7f800000)};
    float hi[3] = {__int_as_float(0xff800000), __int_as_float(0xff800000), __int_as_float(0xff800000)};
    int q3[3] = {0, 0, 0};
    int cnt = 0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      tb[r * 32] = xs[r];
      tb[kGroup + r * 32] = ys[r];
      tb[2 * kGroup + r * 32] = zs[r];
      // summary, exactly as group_summary_kernel computes it (the zero-filled tail belongs to the
      // box, not to the sums)
      const float xc = xs[r] - f.ox, yc = ys[r] - f.oy, zc = zs[r] - f.oz;
      lo[0] = fminf(lo[0], xc); hi[0] = fmaxf(hi[0], xc);
      lo[1] = fminf(lo[1], yc); hi[1] = fmaxf(hi[1], yc);
      lo[2] = fminf(lo[2], zc); hi[2] = fmaxf(hi[2], zc);
      if (base + r * 32 + lane < n32) {
        q3[0] += (int)(__float_as_uint(fmaf(xc, f.sx, kMagic)) - kMagicBits);
        q3[1] += (int)(__float_as_uint(fmaf(yc, f.sy, kMagic)) - kMagicBits);
        q3[2] += (int)(__float_as_uint(fmaf(zc, f.sz, kMagic)) - kMagicBits);
        ++cnt;
      }
    }
    float blo[3], bhi[3];
    int bq[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      blo[d] = redux_min_f32(lo[d]);
      bhi[d] = redux_max_f32(hi[d]);
      bq[d] = __reduce_add_sync(0xffffffffu, q3[d]);
    }
    const int bn = __reduce_add_sync(0xffffffffu, cnt);
    if (lane == 0) {
      float4* o = summaries + grp * 3;  // GroupSummary: lo[3] hi[3] | q[3] n | pad[2]
      o[0] = make_float4(blo[0], blo[1], blo[2], bhi[0]);
      o[1] = make_float4(bhi[1], bhi[2], __int_as_float(bq[0]), __int_as_float(bq[1]));
      o[2] = make_float4(__int_as_float(bq[2]), __int_as_float(bn), 0.f, 0.f);
    }
  }
}

}  // namespace mdkm
