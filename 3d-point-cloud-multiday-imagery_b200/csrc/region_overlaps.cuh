// Region overlaps between days (mdkm_bind_region_overlaps): for a pair of days (a, b), one row for
// every pair of regions (r of day a, s of day b) that share at least one pixel (y, x), with the
// number of shared pixels and the first shared pixel in raster order; rows sorted by pair, then by
// that first pixel.  Read from the whole-stack region map that run_regions has just resolved.
//
//   overlap_bound_kernel   per pair, the pixels where both ids are non-zero and the key (id_a,
//                          id_b) differs from the left neighbour's or x == 0: an upper bound on
//                          the pair's distinct keys, which sizes its hash table;
//   overlap_insert_kernel  one open-addressing table per pair (capacity: the smallest power of two
//                          >= 2 x bound); keys are combined in a lane, across the warp
//                          (__match_any_sync) and along the warp's span (a carried run), and the
//                          leader of a key adds its pixels and lowers its first pixel with atomics:
//                          integer sums and a minimum, so the contents do not depend on the schedule;
//   overlap_mark_kernel    every occupied slot sets the bit of its first pixel in the pair's H*W-bit
//                          mask (a pixel lies in exactly one key, so no two slots share a bit);
//   overlap_scan_kernel    exclusive popcount scan over the masks of all pairs (decoupled
//                          look-back): every set bit's rank is its row, and the total is M;
//   overlap_emit_kernel    every slot writes its row at that rank -- no sort.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace mdkm {

constexpr int kOvSpan = kGroup * 16;         // pixels of a pair per warp of the bound / insert passes
constexpr int kOvChunkWords = kThreads * 4;  // mask words per CTA of the scan

struct OverlapParams {
  const int* ids;                 // [D][H][W] region ids of the whole stack, 0 where no point
  long long HW;
  int W;
  const int* pairs;               // [n_pairs][2] days
  int n_pairs;
  unsigned long long* bounds;     // [n_pairs] run starts, zeroed before the bound pass
  const long long* tab;           // [n_pairs + 1] slot offsets of the pairs' tables (power-of-two sizes)
  unsigned long long* slots;      // [slots][2]: key (r << 32 | s; 0: empty), then count | ~first << 32; zeroed
  unsigned int* bits;             // [n_pairs * wpp, padded to the scan chunk] first-pixel masks, zeroed
  long long wpp;                  // mask words per pair: ceil(HW / 32)
  unsigned int* word_rel;         // [mask words] set bits before the word within its scan chunk
  unsigned long long* status;     // [chunks] look-back words of the scan
  unsigned long long* chunk_base; // [chunks] set bits before the chunk
  unsigned int* ticket;           // [0] chunk ticket, [1] fault flag (look-back timed out)
  unsigned long long* total;      // M, written by the CTA of the last chunk
  unsigned int* probe_fault;      // set when a table had no free slot (a bound below the keys)
  long long* rows;                // [M][6] pair, region_a, region_b, pixels, y_first, x_first
};

// Four consecutive ids of one day from pixel i (a multiple of 4): one 16-byte load when the day
// is 16-byte aligned and the four are inside [0, end), else one by one, 0 past end.
__device__ __forceinline__ void ov_load4(const int* day, long long i, long long end, bool vec, int v[4]) {
  if (vec && i + 4 <= end) {
    const int4 q = __ldg(reinterpret_cast<const int4*>(day + i));
    v[0] = q.x;
    v[1] = q.y;
    v[2] = q.z;
    v[3] = q.w;
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = i + e < end ? __ldg(day + i + e) : 0;
  }
}

__device__ __forceinline__ unsigned long long ov_key(int a, int b) {
  return (a > 0 && b > 0) ? ((unsigned long long)(unsigned int)a << 32) | (unsigned int)b : 0ull;
}

__device__ __forceinline__ bool ov_aligned(const int* p) { return (reinterpret_cast<size_t>(p) & 15) == 0; }

// ---------------------------------------------------------------------------------------
// Bound: a warp takes kOvSpan pixels of a pair, 128 at a time, lane l pixels 4l..4l+3 (coalesced
// 16-byte loads of both days).  The left neighbour of a lane's first pixel comes from the lane
// before it, or from memory for lane 0.  One 64-bit atomic per warp and pair.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) overlap_bound_kernel(const OverlapParams p) {
  const int lane = threadIdx.x & 31;
  const long long s0 = ((long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5)) * kOvSpan;
  if (s0 >= p.HW) return;
  const long long s1 = min(p.HW, s0 + kOvSpan);
  for (int q = blockIdx.y; q < p.n_pairs; q += gridDim.y) {
    const int* da = p.ids + (long long)__ldg(p.pairs + 2 * q) * p.HW;
    const int* db = p.ids + (long long)__ldg(p.pairs + 2 * q + 1) * p.HW;
    const bool vec = ov_aligned(da) && ov_aligned(db);
    unsigned int starts = 0u;
    for (long long g0 = s0; g0 < s1; g0 += kGroup) {
      const long long i0 = g0 + lane * 4;
      int a[4], b[4];
      ov_load4(da, i0, s1, vec, a);
      ov_load4(db, i0, s1, vec, b);
      unsigned long long key[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) key[e] = ov_key(a[e], b[e]);
      unsigned long long left = __shfl_up_sync(0xffffffffu, key[3], 1);
      if (lane == 0) left = i0 > 0 ? ov_key(__ldg(da + i0 - 1), __ldg(db + i0 - 1)) : 0ull;
      unsigned int x = (unsigned int)i0 % (unsigned int)p.W;  // (HW < 2^31)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (key[e] != 0ull && (x == 0u || key[e] != left)) ++starts;
        left = key[e];
        if (++x == (unsigned int)p.W) x = 0u;
      }
    }
    starts = __reduce_add_sync(0xffffffffu, starts);
    if (lane == 0 && starts) atomicAdd(p.bounds + q, (unsigned long long)starts);
  }
}

// Adds `cnt` pixels with first pixel `first` to the key's slot (claimed with atomicCAS, linear
// probing).  A table holds at least twice its pair's keys, so a free slot is always found; a full
// walk without one flags the fault instead of looping.
__device__ __forceinline__ void ov_insert(const OverlapParams& p, unsigned long long* table, int lg,
                                          unsigned long long key, unsigned int cnt, unsigned int first) {
  const unsigned long long mask = (1ull << lg) - 1ull;
  unsigned long long s = (key * 0x9E3779B97F4A7C15ull) >> (64 - lg);
  for (unsigned long long n = 0; n <= mask; ++n, s = (s + 1ull) & mask) {
    unsigned long long* slot = table + 2 * s;
    unsigned long long k = *reinterpret_cast<volatile unsigned long long*>(slot);
    if (k == 0ull) {
      k = atomicCAS(slot, 0ull, key);
      if (k == 0ull) k = key;
    }
    if (k == key) {
      unsigned int* v = reinterpret_cast<unsigned int*>(slot + 1);
      atomicAdd(v, cnt);
      atomicMax(v + 1, ~first);
      return;
    }
  }
  atomicExch(p.probe_fault, 1u);
}

// ---------------------------------------------------------------------------------------
// Insert: the warp walks its span as the bound pass does.  It carries the key of the last pixel
// it has read (ckey, with its count and first pixel) from one group of 128 pixels to the next, so
// a run of one key across groups costs no atomics; pixels of the carried key and of the group's
// last key are summed over the warp with two reductions.  The other keys of a group are combined
// in each lane and then across lanes (__match_any_sync, as in region_stats_kernel), and their
// leaders insert them.  The carry is inserted when the group's last key differs from it, and at
// the end of the span.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) overlap_insert_kernel(const OverlapParams p) {
  const int lane = threadIdx.x & 31;
  const long long s0 = ((long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5)) * kOvSpan;
  if (s0 >= p.HW) return;
  const long long s1 = min(p.HW, s0 + kOvSpan);
  for (int q = blockIdx.y; q < p.n_pairs; q += gridDim.y) {
    const long long t0 = __ldg(p.tab + q), cap = __ldg(p.tab + q + 1) - t0;
    if (cap < 2) continue;  // (no pixel has ids on both days)
    const int lg = 63 - __clzll(cap);
    unsigned long long* table = p.slots + 2 * t0;
    const int* da = p.ids + (long long)__ldg(p.pairs + 2 * q) * p.HW;
    const int* db = p.ids + (long long)__ldg(p.pairs + 2 * q + 1) * p.HW;
    const bool vec = ov_aligned(da) && ov_aligned(db);
    unsigned long long ckey = 0ull;
    unsigned int ccnt = 0u, cfirst = ~0u;
    for (long long g0 = s0; g0 < s1; g0 += kGroup) {
      const long long i0 = g0 + lane * 4;
      int a[4], b[4];
      ov_load4(da, i0, s1, vec, a);
      ov_load4(db, i0, s1, vec, b);
      unsigned long long key[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) key[e] = ov_key(a[e], b[e]);
      const unsigned long long tail = __shfl_sync(0xffffffffu, key[3], 31);
      unsigned int cc = 0u, cf = ~0u, tc = 0u, tf = ~0u, rem = 0u;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const unsigned int px = (unsigned int)(i0 + e);
        if (key[e] == 0ull) continue;
        if (key[e] == ckey) {
          ++cc;
          cf = min(cf, px);
        } else if (key[e] == tail) {
          ++tc;
          tf = min(tf, px);
        } else {
          rem |= 1u << e;
        }
      }
      while (__any_sync(0xffffffffu, rem != 0u)) {
        const unsigned long long mine =
            (rem & 1u) ? key[0] : ((rem & 2u) ? key[1] : ((rem & 4u) ? key[2] : ((rem & 8u) ? key[3] : 0ull)));
        unsigned int cnt = 0u, first = ~0u;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          if (((rem >> e) & 1u) && key[e] == mine) {
            ++cnt;
            first = min(first, (unsigned int)(i0 + e));
            rem &= ~(1u << e);
          }
        }
        const unsigned int peers = __match_any_sync(0xffffffffu, mine);
        cnt = __reduce_add_sync(peers, cnt);
        first = __reduce_min_sync(peers, first);
        if (mine != 0ull && lane == __ffs(peers) - 1) ov_insert(p, table, lg, mine, cnt, first);
      }
      cc = __reduce_add_sync(0xffffffffu, cc);
      cf = __reduce_min_sync(0xffffffffu, cf);
      ccnt += cc;
      cfirst = min(cfirst, cf);
      if (tail != ckey) {
        tc = __reduce_add_sync(0xffffffffu, tc);
        tf = __reduce_min_sync(0xffffffffu, tf);
        if (ckey != 0ull && lane == 0) ov_insert(p, table, lg, ckey, ccnt, cfirst);
        ckey = tail;
        ccnt = tc;
        cfirst = tf;
      }
    }
    if (ckey != 0ull && lane == 0) ov_insert(p, table, lg, ckey, ccnt, cfirst);
  }
}

// ---------------------------------------------------------------------------------------
// Every occupied slot of pair q sets the bit of its first pixel in the pair's mask.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) overlap_mark_kernel(const OverlapParams p) {
  for (int q = blockIdx.y; q < p.n_pairs; q += gridDim.y) {
    const long long t0 = __ldg(p.tab + q), t1 = __ldg(p.tab + q + 1);
    unsigned int* bits = p.bits + (long long)q * p.wpp;
    for (long long s = t0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; s < t1;
         s += (long long)gridDim.x * blockDim.x) {
      const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(p.slots + 2 * s);
      if (v.x == 0ull) continue;
      const unsigned int first = ~(unsigned int)(v.y >> 32);
      atomicOr(bits + (first >> 5), 1u << (first & 31u));
    }
  }
}

// ---------------------------------------------------------------------------------------
// Exclusive popcount scan over the masks of all pairs, pair after pair: thread j of a chunk's CTA
// takes 4 words (one 16-byte load; the masks are padded to whole chunks), CTA scan, look-back over
// the chunks (handed out in order by the ticket), as region_number_kernel.  word_rel gets each
// word's offset within its chunk, chunk_base the chunk's offset; the last chunk writes M.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) overlap_scan_kernel(const OverlapParams p, long long n_chunks) {
  __shared__ unsigned int s_warp[kThreads / 32];
  __shared__ long long s_chunk;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) s_chunk = atomicAdd(p.ticket, 1u);
  __syncthreads();
  const long long c = s_chunk;
  const long long w0 = c * kOvChunkWords + (long long)tid * 4;
  const uint4 v = *reinterpret_cast<const uint4*>(p.bits + w0);
  const unsigned int n0 = __popc(v.x), n1 = __popc(v.y), n2 = __popc(v.z), n3 = __popc(v.w);
  const unsigned int cnt = n0 + n1 + n2 + n3;
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
  const unsigned int excl = before + incl - cnt;
  *reinterpret_cast<uint4*>(p.word_rel + w0) = make_uint4(excl, excl + n0, excl + n0 + n1, excl + n0 + n1 + n2);
  if (warp == 0) {
    unsigned long long base = 0ull;
    if (c == 0) {
      if (lane == 0) st_status(p.status, kStPrefix | agg);
    } else {
      if (lane == 0) st_status(p.status + c, kStAggregate | agg);
      base = tile_lookback(p.status, c, agg, lane, p.ticket + 1);
    }
    if (lane == 0) {
      p.chunk_base[c] = base;
      if (c + 1 == n_chunks) *p.total = base + agg;
    }
  }
}

// ---------------------------------------------------------------------------------------
// Every occupied slot writes its row at the rank of its first pixel's bit.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) overlap_emit_kernel(const OverlapParams p) {
  for (int q = blockIdx.y; q < p.n_pairs; q += gridDim.y) {
    const long long t0 = __ldg(p.tab + q), t1 = __ldg(p.tab + q + 1);
    for (long long s = t0 + (long long)blockIdx.x * blockDim.x + threadIdx.x; s < t1;
         s += (long long)gridDim.x * blockDim.x) {
      const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(p.slots + 2 * s);
      if (v.x == 0ull) continue;
      const unsigned int first = ~(unsigned int)(v.y >> 32);
      const long long w = (long long)q * p.wpp + (first >> 5);
      const unsigned long long row = p.chunk_base[w / kOvChunkWords] + p.word_rel[w] +
                                     __popc(p.bits[w] & ((1u << (first & 31u)) - 1u));
      long long* r = p.rows + row * 6;
      r[0] = q;
      r[1] = (long long)(v.x >> 32);
      r[2] = (long long)(v.x & 0xffffffffull);
      r[3] = (long long)(v.y & 0xffffffffull);
      r[4] = first / (unsigned int)p.W;
      r[5] = first % (unsigned int)p.W;
    }
  }
}

}  // namespace mdkm
