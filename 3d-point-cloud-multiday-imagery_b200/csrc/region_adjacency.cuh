// Region adjacency within a day (mdkm_bind_region_adjacency): for every unordered pair of distinct
// regions r < s of one day that are joined by at least one edge, one row with the number of edges
// between them and their first edge; and for every region its perimeter, split by what lies on the
// other side of each edge.  An edge joins two 4-neighbouring pixels of one day: direction 0 joins
// (y, x) and (y, x+1), direction 1 joins (y, x) and (y+1, x); its index within the day is
// e = 2 (y W + x) + direction.  Read from the whole-stack region map that run_regions has just
// resolved.  The passes are those of the region overlaps (region_overlaps.cuh) with a day in place
// of a pair and the first edge in place of the first pixel:
//
//   adjacency_bound_kernel   per day, the run starts along each image row of the horizontal key
//                            (id[p], id[p+1]) and of the vertical key (id[p], id[p+W]), counting
//                            only keys of two different non-zero ids: an upper bound on the day's
//                            distinct keys, which sizes its hash table;
//   adjacency_insert_kernel  one open-addressing table per day (overlap slot layout, key min << 32
//                            | max); keys are combined in a lane, across the warp and along the
//                            warp's span, and their leaders insert them with ov_insert.  The same
//                            pass adds each pixel's background and raster-border sides to its
//                            region, aggregated per warp;
//   overlap_mark_kernel /    unchanged, with D "pairs" of 2 H W-bit masks (wpp = ceil(2 H W / 32));
//   overlap_scan_kernel      2 H W - 1 < 2^32 - 2 because the stack has fewer than 2^31 pixels;
//   adjacency_emit_kernel    every slot writes its row at its rank and adds its edges to both
//                            regions' region_edges;
//   adjacency_finish_kernel  per region: the perimeter, the sum of its three kinds of side.
#pragma once
#include "common.cuh"
#include "region_overlaps.cuh"

namespace mdkm {

struct AdjacencyParams {
  OverlapParams ov;          // ids, HW, W, n_pairs = D, bounds, tab, slots, bits, wpp, scan words, rows [M][6]
  unsigned long long* sides; // [R][4] boundaries, zeroed: column 0 holds background | border << 32 until the
                             // finish pass (each < 2^32: a day has fewer than 2^32 edges), column 1 region edges
  long long n_regions;
};

// the key of an edge between ids a and b: min << 32 | max when both are regions and differ, else 0
__device__ __forceinline__ unsigned long long adj_key(int a, int b) {
  return (a > 0 && b > 0 && a != b)
             ? ((unsigned long long)(unsigned int)min(a, b) << 32) | (unsigned int)max(a, b)
             : 0ull;
}

// The ids a warp lane needs for pixels i0..i0+3 of a day (i0 a multiple of 4, the span [.., s1)):
// the pixels (0 past s1), the pixel right of the last one, and the row below (0 past the last row).
__device__ __forceinline__ void adj_load(const AdjacencyParams& p, const int* day, long long i0, long long s1,
                                         int lane, int a[4], int& right, int b[4]) {
  const long long HW = p.ov.HW, W = p.ov.W;
  ov_load4(day, i0, s1, ov_aligned(day), a);
  ov_load4(day + W, i0, min(s1, HW - W), ov_aligned(day + W), b);
  right = __shfl_down_sync(0xffffffffu, a[0], 1);
  // (lanes below 31 have i0 + 4 < s1 or i0 + 3 >= HW - 1, where no pixel has a right neighbour)
  if (lane == 31) right = i0 + 4 < HW ? __ldg(day + i0 + 4) : 0;
}

// ---------------------------------------------------------------------------------------
// Bound: a warp takes kOvSpan pixels of a day, 128 at a time, lane l pixels 4l..4l+3 (16-byte
// loads of the row and of the row below where the day allows them).  The keys left of a lane's
// first pixel come from the lane before it, or from memory for lane 0.  One 64-bit atomic per warp
// and day.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) adjacency_bound_kernel(const AdjacencyParams p) {
  const int lane = threadIdx.x & 31;
  const long long HW = p.ov.HW, below_end = HW - p.ov.W;
  const long long s0 = ((long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5)) * kOvSpan;
  if (s0 >= HW) return;
  const long long s1 = min(HW, s0 + kOvSpan);
  for (int q = blockIdx.y; q < p.ov.n_pairs; q += gridDim.y) {
    const int* day = p.ov.ids + (long long)q * HW;
    unsigned int starts = 0u;
    for (long long g0 = s0; g0 < s1; g0 += kGroup) {
      const long long i0 = g0 + lane * 4;
      int a[4], b[4], right;
      adj_load(p, day, i0, s1, lane, a, right, b);
      const unsigned int x0 = (unsigned int)i0 % (unsigned int)p.ov.W;  // (HW < 2^31)
      unsigned int x = x0;
      unsigned long long hk[4], vk[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        hk[e] = x + 1u < (unsigned int)p.ov.W ? adj_key(a[e], e < 3 ? a[e + 1] : right) : 0ull;
        vk[e] = adj_key(a[e], b[e]);
        if (++x == (unsigned int)p.ov.W) x = 0u;
      }
      x = x0;
      unsigned long long hl = __shfl_up_sync(0xffffffffu, hk[3], 1), vl = __shfl_up_sync(0xffffffffu, vk[3], 1);
      if (lane == 0) {
        hl = vl = 0ull;
        if (x != 0u && i0 < s1) {
          const int l = __ldg(day + i0 - 1);
          hl = adj_key(l, a[0]);
          vl = i0 - 1 < below_end ? adj_key(l, __ldg(day + i0 - 1 + p.ov.W)) : 0ull;
        }
      }
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (hk[e] != 0ull && (x == 0u || hk[e] != hl)) ++starts;
        if (vk[e] != 0ull && (x == 0u || vk[e] != vl)) ++starts;
        hl = hk[e];
        vl = vk[e];
        if (++x == (unsigned int)p.ov.W) x = 0u;
      }
    }
    starts = __reduce_add_sync(0xffffffffu, starts);
    if (lane == 0 && starts) atomicAdd(p.ov.bounds + q, (unsigned long long)starts);
  }
}

// Adds `v` (background | border << 32) to region `id`'s side counts.
__device__ __forceinline__ void adj_add_sides(const AdjacencyParams& p, int id, unsigned long long v) {
  atomicAdd(p.sides + 4 * (long long)(id - 1), v);
}

// ---------------------------------------------------------------------------------------
// Insert: the warp walks its span as the bound pass does; lane l holds the 8 edges 2 (i0 + e) + dir
// of its pixels, in edge order.  Keys are combined as in overlap_insert_kernel: the carried key of
// the span (ckey, with its count and first edge), the group's last key, the rest in each lane and
// then across lanes (__match_any_sync), inserted by their leaders.  Each pixel also adds its sides
// on the raster border and towards pixels without a point: a region pixel to itself, a pixel
// without a point to its right and lower neighbours' regions.  Runs of one region in a lane are
// summed there, and the lane's last run over the warp before one 64-bit atomic per region.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) adjacency_insert_kernel(const AdjacencyParams p) {
  const int lane = threadIdx.x & 31;
  const long long HW = p.ov.HW, W = p.ov.W, below_end = HW - W;
  const long long s0 = ((long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5)) * kOvSpan;
  if (s0 >= HW) return;
  const long long s1 = min(HW, s0 + kOvSpan);
  for (int q = blockIdx.y; q < p.ov.n_pairs; q += gridDim.y) {
    const long long t0 = __ldg(p.ov.tab + q), cap = __ldg(p.ov.tab + q + 1) - t0;
    const bool keyed = cap >= 2;  // (else the day has no edge between two regions)
    const int lg = keyed ? 63 - __clzll(cap) : 1;
    unsigned long long* table = p.ov.slots + 2 * t0;
    const int* day = p.ov.ids + (long long)q * HW;
    unsigned long long ckey = 0ull;
    unsigned int ccnt = 0u, cfirst = ~0u;
    for (long long g0 = s0; g0 < s1; g0 += kGroup) {
      const long long i0 = g0 + lane * 4;
      int a[4], b[4], right;
      adj_load(p, day, i0, s1, lane, a, right, b);
      unsigned int x = (unsigned int)i0 % (unsigned int)W;  // (HW < 2^31)
      unsigned long long key[8];
      int run_id = 0;
      unsigned long long run_v = 0ull;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const long long i = i0 + e;
        const bool has_right = x + 1u < (unsigned int)W, has_below = i < below_end;
        const int r = e < 3 ? a[e + 1] : right;
        key[2 * e] = keyed && has_right ? adj_key(a[e], r) : 0ull;
        key[2 * e + 1] = keyed ? adj_key(a[e], b[e]) : 0ull;
        // sides: (id, background | border << 32) items, summed while the id repeats
        int id[2] = {0, 0};
        unsigned long long v[2] = {0ull, 0ull};
        if (a[e] > 0) {
          const unsigned int border = (x == 0u) + !has_right + (i < W) + !has_below;
          id[0] = a[e];
          v[0] = ((unsigned long long)border << 32) + (has_right && r == 0) + (has_below && b[e] == 0);
        } else if (i < s1) {
          if (has_right && r > 0) id[0] = r, v[0] = 1ull;
          if (has_below && b[e] > 0) id[1] = b[e], v[1] = 1ull;
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          if (id[j] == 0) continue;
          if (id[j] != run_id) {
            if (run_id) adj_add_sides(p, run_id, run_v);
            run_id = id[j];
            run_v = 0ull;
          }
          run_v += v[j];
        }
        if (++x == (unsigned int)W) x = 0u;
      }
      {
        const unsigned int peers = __match_any_sync(0xffffffffu, run_id);
        const unsigned int bg = __reduce_add_sync(peers, (unsigned int)run_v);
        const unsigned int border = __reduce_add_sync(peers, (unsigned int)(run_v >> 32));
        if (run_id && lane == __ffs(peers) - 1) adj_add_sides(p, run_id, ((unsigned long long)border << 32) | bg);
      }
      const unsigned long long tail = __shfl_sync(0xffffffffu, key[7], 31);
      unsigned int cc = 0u, cf = ~0u, tc = 0u, tf = ~0u, rem = 0u;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const unsigned int edge = 2u * (unsigned int)i0 + e;
        if (key[e] == 0ull) continue;
        if (key[e] == ckey) {
          ++cc;
          cf = min(cf, edge);
        } else if (key[e] == tail) {
          ++tc;
          tf = min(tf, edge);
        } else {
          rem |= 1u << e;
        }
      }
      while (__any_sync(0xffffffffu, rem != 0u)) {
        unsigned long long mine = 0ull;
#pragma unroll
        for (int e = 7; e >= 0; --e)
          if ((rem >> e) & 1u) mine = key[e];
        unsigned int cnt = 0u, first = ~0u;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          if (((rem >> e) & 1u) && key[e] == mine) {
            ++cnt;
            first = min(first, 2u * (unsigned int)i0 + e);
            rem &= ~(1u << e);
          }
        }
        const unsigned int peers = __match_any_sync(0xffffffffu, mine);
        cnt = __reduce_add_sync(peers, cnt);
        first = __reduce_min_sync(peers, first);
        if (mine != 0ull && lane == __ffs(peers) - 1) ov_insert(p.ov, table, lg, mine, cnt, first);
      }
      cc = __reduce_add_sync(0xffffffffu, cc);
      cf = __reduce_min_sync(0xffffffffu, cf);
      ccnt += cc;
      cfirst = min(cfirst, cf);
      if (tail != ckey) {
        tc = __reduce_add_sync(0xffffffffu, tc);
        tf = __reduce_min_sync(0xffffffffu, tf);
        if (ckey != 0ull && lane == 0) ov_insert(p.ov, table, lg, ckey, ccnt, cfirst);
        ckey = tail;
        ccnt = tc;
        cfirst = tf;
      }
    }
    if (ckey != 0ull && lane == 0) ov_insert(p.ov, table, lg, ckey, ccnt, cfirst);
  }
}

// ---------------------------------------------------------------------------------------
// Every occupied slot writes its row at the rank of its first edge's bit and adds its edges to the
// region_edges of both regions.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) adjacency_emit_kernel(const AdjacencyParams p) {
  for (int q = blockIdx.y; q < p.ov.n_pairs; q += gridDim.y) {
    const long long t0 = __ldg(p.ov.tab + q), t1 = __ldg(p.ov.tab + q + 1);
    for (long long s = t0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; s < t1;
         s += (long long)gridDim.x * blockDim.x) {
      const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(p.ov.slots + 2 * s);
      if (v.x == 0ull) continue;
      const unsigned int first = ~(unsigned int)(v.y >> 32);
      const long long w = (long long)q * p.ov.wpp + (first >> 5);
      const unsigned long long row = p.ov.chunk_base[w / kOvChunkWords] + p.ov.word_rel[w] +
                                     __popc(p.ov.bits[w] & ((1u << (first & 31u)) - 1u));
      const long long ra = (long long)(v.x >> 32), rb = (long long)(v.x & 0xffffffffull);
      const unsigned long long cnt = v.y & 0xffffffffull;
      const unsigned int px = first >> 1;
      long long* r = p.ov.rows + row * 6;
      r[0] = q;
      r[1] = ra;
      r[2] = rb;
      r[3] = (long long)cnt;
      r[4] = px / (unsigned int)p.ov.W;
      r[5] = px % (unsigned int)p.ov.W;
      atomicAdd(p.sides + 4 * (ra - 1) + 1, cnt);
      atomicAdd(p.sides + 4 * (rb - 1) + 1, cnt);
    }
  }
}

// ---------------------------------------------------------------------------------------
// Per region: (perimeter, region_edges, background_edges, border_edges).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) adjacency_finish_kernel(const AdjacencyParams p) {
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < p.n_regions;
       r += (long long)gridDim.x * blockDim.x) {
    unsigned long long* s = p.sides + 4 * r;
    const unsigned long long packed = s[0], region = s[1];
    const unsigned long long bg = packed & 0xffffffffull, border = packed >> 32;
    s[0] = region + bg + border;
    s[2] = bg;
    s[3] = border;
  }
}

}  // namespace mdkm
