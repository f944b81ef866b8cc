// Object tracks (mdkm_bind_tracks): regions of consecutive days linked by overlap, numbered over
// the stack.  Region r of day d and region s of day d+1 are linked when they have the same
// cluster and share at least one pixel with shared / (pixels_r + pixels_s - shared) >= min_iou
// in FP64; a track is a connected component of the links, numbered 1..T in the order of its
// smallest region id.  Read from the overlap rows of the consecutive pairs (region_overlaps.cuh)
// and the region table (region_finish_kernel).
//
//   track_init_kernel  every region its own parent, no links;
//   track_link_kernel  one thread per overlap row: the rule, then union-find on region indices
//                      (grid_union: the root is the smallest index) and the link counts that give
//                      `branched`; it also finds the end of the caller's rows (their count);
//   region_number_kernel / region_resolve_kernel on the R parents: roots numbered by the
//                      decoupled look-back, every region its root's id (region_tracks), T;
//   track_table_kernel one thread per region: its track's row, with integer atomics into R
//                      zeroed row slots (no T needed before the pass);
//   track_map_kernel   every pixel of this rank's range: its region's track, 0 where no point.
#pragma once
#include "common.cuh"
#include "region_overlaps.cuh"
#include "regions.cuh"

namespace mdkm {

struct TrackParams {
  const long long* rows;         // [n_rows][6] overlap rows: pair, region_a, region_b, pixels, y, x
  long long n_rows;
  const int* link_day;           // [n_pairs] d when the pair is the counted (d, d+1), else -1
  int n_user;                    // the caller's pairs come first: rows with pair < n_user are theirs
  unsigned long long* user_rows; // their count, written by the thread of their last row (zeroed)
  const long long* regions;      // [R][7] region table: day, cluster, pixels, ...
  long long n_regions;
  double min_iou;
  int* parent;                   // [R] union-find parents (region index)
  unsigned int* links;           // [2R] links forward (to the next day), then backward
  const int* tracks;             // [R] track id of each region
  long long* table;              // [R][7] track rows, zeroed: cluster, first_day, last_day, regions,
                                 // pixels, first_region, branched
};

__global__ void __launch_bounds__(kThreads) track_init_kernel(const TrackParams p) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < p.n_regions;
       r += (long long)gridDim.x * blockDim.x) {
    p.parent[r] = (int)r;
    p.links[r] = 0u;
    p.links[p.n_regions + r] = 0u;
  }
}

// ---------------------------------------------------------------------------------------
// Links.  The counts are exact integers below 2^31, so the FP64 quotient is the correctly rounded
// IoU and a numpy restatement gives the same decision.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) track_link_kernel(const TrackParams p) {
  for (long long m = blockIdx.x * (long long)blockDim.x + threadIdx.x; m < p.n_rows;
       m += (long long)gridDim.x * blockDim.x) {
    const long long* row = p.rows + m * 6;
    const int q = (int)row[0];
    if (q < p.n_user && (m + 1 == p.n_rows || row[6] >= p.n_user)) *p.user_rows = (unsigned long long)(m + 1);
    if (__ldg(p.link_day + q) < 0) continue;
    const long long r = row[1] - 1, s = row[2] - 1, shared = row[3];
    const long long* a = p.regions + r * 7;
    const long long* b = p.regions + s * 7;
    if (a[1] != b[1]) continue;
    if (__ddiv_rn((double)shared, (double)(a[2] + b[2] - shared)) < p.min_iou) continue;
    grid_union(p.parent, (int)r, (int)s);
    atomicAdd(p.links + r, 1u);
    atomicAdd(p.links + p.n_regions + s, 1u);
  }
}

// ---------------------------------------------------------------------------------------
// Track rows.  A track's smallest region id is its root, and region ids run in day order, so the
// root alone writes the cluster, the first day and the first region; the others are sums, a
// maximum and an or over the track's regions.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) track_table_kernel(const TrackParams p) {
  for (long long r = blockIdx.x * (long long)blockDim.x + threadIdx.x; r < p.n_regions;
       r += (long long)gridDim.x * blockDim.x) {
    const long long* g = p.regions + r * 7;
    long long* t = p.table + (long long)(p.tracks[r] - 1) * 7;
    if (p.parent[r] == (int)r) {
      t[0] = g[1];
      t[1] = g[0];
      t[5] = r + 1;
    }
    atomicMax(t + 2, g[0]);
    atomicAdd(reinterpret_cast<unsigned long long*>(t + 3), 1ull);
    atomicAdd(reinterpret_cast<unsigned long long*>(t + 4), (unsigned long long)g[2]);
    if (p.links[r] > 1u || p.links[p.n_regions + r] > 1u) atomicOr(reinterpret_cast<unsigned long long*>(t + 6), 1ull);
  }
}

// ---------------------------------------------------------------------------------------
// Track map: out[i] = ids[i] ? tracks[ids[i] - 1] : 0 over n pixels.  Thread j of the body takes
// four pixels from the first 16-byte boundary of `out` on (one 16-byte store; one 16-byte load
// when `ids` is aligned there too, else four); the thread after the body takes the head and
// the tail (up to three pixels each).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ int track_of(const int* tracks, int id) { return id ? __ldg(tracks + id - 1) : 0; }

__global__ void __launch_bounds__(kThreads) track_map_kernel(const int* ids, const int* tracks, int* out, long long n) {
  const long long head = min(n, (long long)((16u - (reinterpret_cast<size_t>(out) & 15u)) & 15u) / 4);
  const long long body = (n - head) / 4;
  const bool vec = (reinterpret_cast<size_t>(ids + head) & 15u) == 0;
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j <= body;
       j += (long long)gridDim.x * blockDim.x) {
    if (j < body) {
      int v[4];
      ov_load4(ids, head + 4 * j, n, vec, v);
      *reinterpret_cast<int4*>(out + head + 4 * j) =
          make_int4(track_of(tracks, v[0]), track_of(tracks, v[1]), track_of(tracks, v[2]), track_of(tracks, v[3]));
    } else {
      for (long long i = 0; i < head; ++i) out[i] = track_of(tracks, __ldg(ids + i));
      for (long long i = head + 4 * body; i < n; ++i) out[i] = track_of(tracks, __ldg(ids + i));
    }
  }
}

}  // namespace mdkm
