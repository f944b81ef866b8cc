// K1: height-map stack -> XYZ points with NaN / nodata / range masking fused in, stable
// (np.where-order) compaction, optional per-day plane detrend.
//
// Replaces members/rafael/disparity/plugin.py:148 (h = -disp/16), :151-152 (validity),
// :157-160 (np.where + stack), :161-171 (SVD plane fit, via 9 moments + a 3x3 symmetric
// eigen-solve) for every day of the stack, and concatenates the days (absent in the
// reference, SURVEY.md F1).
//
// ONE pass over the rasters (4 B read + 12 B written per pixel, the algorithmic minimum): a warp
// takes a tile of kTile = 1024 consecutive pixels, one pixel per lane and step (heights and validity
// bits in registers), counts its valid pixels, obtains the number of points of all earlier tiles by
// a decoupled look-back over status words (tiles are handed out by a ticket counter, so every
// predecessor of a running tile is itself running or done; the look-back works on super-tiles of
// eight warp tiles = one CTA), and stores x, y, z at offset + rank, step by step -- dense 128-byte
// runs in exactly np.where's order.  The loop is software-pipelined (the next super-tile is loaded
// and announced before the look-back of the current one): the pass is bound by HBM, not by the
// look-back chain.  Offsets at every kChunk = 4096 pixels are kept for the day boundaries.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace mdkm {

constexpr int kChunk = 4096;
// (measured on config 2, 41.9 M pixels: 1024-pixel tiles with two 256-thread CTAs of 127-register
// threads per SM 0.160 ms; 512-pixel tiles with four CTAs of 64 registers 0.164 ms)
#ifndef MDKM_TILE
#define MDKM_TILE 1024
#endif
#ifndef MDKM_UNPROJ_CTAS
#define MDKM_UNPROJ_CTAS 2
#endif
constexpr int kTile = MDKM_TILE;  // pixels per warp tile of the fused pass
struct UnprojParams {
  const void* hm;         // points at pixel pix_begin
  const uint8_t* mask;    // idem, or nullptr
  long long pix_begin;    // global flat index of the first pixel
  long long pix_count;
  long long HW;
  int W, H;
  int dtype;              // MDKM_HM_F32 / MDKM_HM_I16 / MDKM_HM_F32_GTIFF3
  float scale;            // for I16
  float max_abs;
  long long* chunk_offsets;  // [n_chunks]: points produced before every kChunk-th pixel of the range
  float* pts;             // blocked cloud (common.cuh)
  const double* planes;   // [n_days][8]: centre xyz, normal xyz, pad -- or nullptr
  int day0;               // day index of planes[0]
  long long chunk_begin;  // this launch handles chunks [chunk_begin, chunk_end) of the range
  long long chunk_end;
  unsigned int* run_src;  // optional [pix_count / 8 + 1]: entry i = points produced by the pixels before
                          // local pixel 8 i (the raster mirror build reads runs of pixels from it, mirror.cuh)
  // fused pass: this launch handles tiles [tile_begin, tile_end) of the range
  long long tile_begin, tile_end;
  unsigned long long* status;  // [n_tiles / 8] look-back words (one per super-tile), zeroed once per mdkm_unproject
  unsigned int* ticket;        // zeroed before every launch; ticket[1] = fault flag (look-back timed out)
  long long* total_out;        // points of all tiles up to tile_end - 1 (running total of the range)
  unsigned int* minmax;        // optional [6]: ordered-uint min x,y,z / max x,y,z of the points written
                               // (pre-filled with 0xffffffff / 0 by the host, as minmax_kernel expects)
};

// One pixel: height and validity (plugin.py:151-152).  dtype 2 is the reference's own
// "5-out-F.tif" raster (disparity.py:213-224): three pixel-interleaved float32 bands, band 0
// the height (-disp/16), band 2 `final_defined`.
__device__ __forceinline__ bool load_height1(const UnprojParams& p, long long i, float& hv) {
  bool ok = true;
  if (p.dtype == 0) {
    hv = __ldg(reinterpret_cast<const float*>(p.hm) + i);
  } else if (p.dtype == 1) {
    hv = p.scale * (float)__ldg(reinterpret_cast<const short*>(p.hm) + i);
  } else {
    const float* s3 = reinterpret_cast<const float*>(p.hm) + 3 * i;
    hv = __ldg(s3);
    ok = __ldg(s3 + 2) != 0.f;
  }
  ok = ok && (fabsf(hv) <= p.max_abs);
  if (p.mask) ok = ok && (__ldg(p.mask + i) != 0);
  return ok;
}

__device__ __forceinline__ unsigned int f2ord(float f) {
  const unsigned int b = __float_as_uint(f);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
// plugin.py:171: height_rel = dot(P - center, normal), in a fixed evaluation order
__device__ __forceinline__ float plane_height(const double* __restrict__ pl, unsigned int col, unsigned int row, float z) {
  double v = __dmul_rn((double)z - pl[2], pl[5]);
  v = __fma_rn((double)row - pl[1], pl[4], v);
  v = __fma_rn((double)col - pl[0], pl[3], v);
  return (float)v;
}

__device__ __forceinline__ float ldg_stream_f32(const float* p) {
  float r;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ unsigned int ldg_stream_u16(const void* p) {
  unsigned short r;
  asm volatile("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ unsigned int ldg_stream_u8(const void* p) {
  unsigned int r;
  asm volatile("ld.global.nc.L1::no_allocate.u8 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}

// One tile's pixels: heights into registers (all loads of a lane in flight at once), validity
// (plugin.py:151-152: isfinite(h) & (|h| <= limit) & validity_mask; NaN and inf fail the <= test)
// as one bit per step.  `limit` = pixels of the tile inside the range.
template <int kSteps>
__device__ __forceinline__ void load_tile(const UnprojParams& p, long long pix0, int lane, float (&hv)[kSteps],
                                          unsigned int& vmask, unsigned int& limit) {
  const long long left = p.pix_count - pix0;
  limit = left < (long long)(kSteps * 32) ? (unsigned int)left : (unsigned int)(kSteps * 32);
  // (the mask bytes first: folded into one word before the heights are requested, so that only
  // one set of loads occupies registers at a time)
  unsigned int keep = 0xffffffffu;
  if (p.mask) {
    const uint8_t* ms = p.mask + pix0 + lane;
    unsigned int mb[kSteps];
#pragma unroll
    for (int s = 0; s < kSteps; ++s) mb[s] = (unsigned int)(s * 32 + lane) < limit ? ldg_stream_u8(ms + s * 32) : 0u;
    keep = 0u;
#pragma unroll
    for (int s = 0; s < kSteps; ++s) keep |= mb[s] ? (1u << s) : 0u;
  }
  if (p.dtype == 0) {
    const float* src = reinterpret_cast<const float*>(p.hm) + pix0 + lane;
#pragma unroll
    for (int s = 0; s < kSteps; ++s)
      hv[s] = (unsigned int)(s * 32 + lane) < limit ? ldg_stream_f32(src + s * 32) : __int_as_float(0x7fc00000);
  } else if (p.dtype == 1) {
    const short* src = reinterpret_cast<const short*>(p.hm) + pix0 + lane;
#pragma unroll
    for (int s = 0; s < kSteps; ++s)
      hv[s] = (unsigned int)(s * 32 + lane) < limit ? p.scale * (float)(short)ldg_stream_u16(src + s * 32)
                                                      : __int_as_float(0x7fc00000);
  } else {
    // the reference's own 5-out-F.tif: (height, -, final_defined) per pixel; `final_defined`
    // first, folded into the keep bits like the mask
    const float* src = reinterpret_cast<const float*>(p.hm) + 3 * (pix0 + lane);
    {
      float dd[kSteps];
#pragma unroll
      for (int s = 0; s < kSteps; ++s) dd[s] = (unsigned int)(s * 32 + lane) < limit ? ldg_stream_f32(src + 3 * s * 32 + 2) : 0.f;
#pragma unroll
      for (int s = 0; s < kSteps; ++s) keep &= dd[s] != 0.f ? 0xffffffffu : ~(1u << s);  // not `final_defined` -> nodata
    }
#pragma unroll
    for (int s = 0; s < kSteps; ++s)
      hv[s] = (unsigned int)(s * 32 + lane) < limit ? ldg_stream_f32(src + 3 * s * 32) : __int_as_float(0x7fc00000);
  }
  vmask = 0;
#pragma unroll
  for (int s = 0; s < kSteps; ++s) vmask |= (fabsf(hv[s]) <= p.max_abs) ? (1u << s) : 0u;  // (outside the range: NaN)
  vmask &= keep;
}

// The fused pass.  A warp takes a tile of kTile consecutive pixels as kSteps steps of 32 pixels, ONE
// pixel per lane and step (coalesced 128-byte requests, all of a lane's loads in flight at once);
// heights and validity bits stay in registers.  A CTA takes a super-tile of 8 warp tiles per ticket:
// the warps count their valid pixels (one POPC + one REDUX), the super-tile's aggregate is published,
// ONE look-back per super-tile (by warp 0) yields the CTA's offset -- its depth is bounded by the
// number of resident CTAs -- and the warps' own offsets follow from the eight counts in shared
// memory.  Then every step ranks its valid pixels with one ballot and the lanes store x, y, z at
// offset + rank: the 32 outputs of a step are consecutive, so the scalar stores of a step form dense
// 128-byte runs, in np.where's order.  No staging in shared memory, no index list.
//
// The loop is software-pipelined: the NEXT super-tile is requested, counted and its aggregate
// published BEFORE the look-back of the current one, so the wait for the predecessors' status words
// overlaps the next tile's DRAM latency, and no aggregate ever waits for a look-back.
//
// kMode 0: W and pix_begin are multiples of 32 -- a step never straddles a raster row, the row / day
//          bookkeeping is per step (warp-uniform);
//       1: W >= 32 -- at most one row boundary inside a step;
//       2: any W (per-pixel division).
template <int kMode, bool kPlanes>
__global__ void __launch_bounds__(kThreads, MDKM_UNPROJ_CTAS) unproject_fused_kernel(const UnprojParams p) {
  constexpr int kWarps = kThreads / 32;
  constexpr int kSteps = kTile / 32;
  static_assert(kSteps <= 32, "one validity bit per step in a 32-bit word");
  __shared__ unsigned int s_cnt[2][kWarps];
  __shared__ unsigned long long s_base;
  __shared__ long long s_super;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned int lt = (1u << lane) - 1u;
  // bounding box of the points this thread writes (the frame of the cloud needs it: no extra pass)
  float mn[3] = {__int_as_float(0x7f800000), __int_as_float(0x7f800000), __int_as_float(0x7f800000)};
  float mx[3] = {__int_as_float(0xff800000), __int_as_float(0xff800000), __int_as_float(0xff800000)};
  const long long super_begin = p.tile_begin / kWarps;  // (launch boundaries are whole super-tiles)
  const unsigned int W = (unsigned int)p.W, H = (unsigned int)p.H;

  // prologue: the first super-tile of this CTA, counted and announced
  if (threadIdx.x == 0) s_super = super_begin + (long long)atomicAdd(p.ticket, 1u);
  __syncthreads();
  long long sup = s_super;
  float hv[kSteps];
  unsigned int vmask = 0, limit = 0, cnt = 0;
  bool have = sup * kWarps < p.tile_end;  // CTA-uniform
  if (have) {
    if (sup * kWarps + warp < p.tile_end) load_tile<kSteps>(p, (sup * kWarps + warp) * kTile, lane, hv, vmask, limit);
    cnt = __reduce_add_sync(0xffffffffu, (unsigned int)__popc(vmask));
    if (lane == 0) s_cnt[0][warp] = cnt;
  }
  __syncthreads();  // (also: everybody has read s_super)
  if (have && threadIdx.x == 0 && sup > 0) {
    unsigned int agg = 0;
    for (int w = 0; w < kWarps; ++w) agg += s_cnt[0][w];
    st_status(p.status + sup, kStAggregate | agg);
  }
  for (int par = 0; have; par ^= 1) {
    // 1. the next super-tile: ticket, pixels, counts, aggregate -- before this one's look-back
    if (threadIdx.x == 0) s_super = super_begin + (long long)atomicAdd(p.ticket, 1u);
    __syncthreads();
    const long long sup_n = s_super;
    const bool have_n = sup_n * kWarps < p.tile_end;  // CTA-uniform
    float hn[kSteps];
    unsigned int vmask_n = 0, limit_n = 0, cnt_n = 0;
    if (have_n) {
      if (sup_n * kWarps + warp < p.tile_end) load_tile<kSteps>(p, (sup_n * kWarps + warp) * kTile, lane, hn, vmask_n, limit_n);
      cnt_n = __reduce_add_sync(0xffffffffu, (unsigned int)__popc(vmask_n));
      if (lane == 0) s_cnt[par ^ 1][warp] = cnt_n;
    }
    __syncthreads();  // (also: everybody has read s_super)
    // 2. points of all earlier super-tiles (one look-back per CTA), then of the earlier warps
    if (warp == 0) {
      if (have_n) {
        const unsigned int agg_n = __reduce_add_sync(0xffffffffu, lane < kWarps ? s_cnt[par ^ 1][lane] : 0u);
        if (lane == 0) st_status(p.status + sup_n, kStAggregate | agg_n);
      }
      const unsigned int agg = __reduce_add_sync(0xffffffffu, lane < kWarps ? s_cnt[par][lane] : 0u);
#ifdef MDKM_NO_LOOKBACK  // timing experiment only (wrong offsets): the pass without its look-back
      const unsigned long long base = (unsigned long long)sup * ((kThreads / 32) * kTile);
#else
      const unsigned long long base = tile_lookback(p.status, sup, agg, lane, p.ticket + 1);
#endif
      if (lane == 0) s_base = base;
    }
    __syncthreads();
    const long long t = sup * kWarps + warp;
    if (t < p.tile_end) {  // warp-uniform
      const long long pix0 = t * kTile;  // local index of the tile's first pixel
      unsigned long long excl = s_base;
      for (int w = 0; w < warp; ++w) excl += s_cnt[par][w];
      if (lane == 0) {
        if ((t & (kChunk / kTile - 1)) == 0) p.chunk_offsets[t / (kChunk / kTile)] = (long long)excl;
        if (t == p.tile_end - 1 && p.total_out) *p.total_out = (long long)(excl + cnt);
      }
      // 3. x, y, z of the valid pixels at offset + rank.  Position of the tile's first pixel once per
      // tile (64-bit); per step / pixel only 32-bit arithmetic
      const long long gp0 = p.pix_begin + pix0;
      const long long day0 = gp0 / p.HW;
      const long long rem0 = gp0 - day0 * p.HW;
      unsigned int rowb = (unsigned int)(rem0 / p.W);                 // row, column, day of the step's first pixel
      unsigned int cb = (unsigned int)(rem0 - (long long)rowb * p.W);
      int dayb = (int)(day0 - p.day0);
      // (offsets inside the cloud relative to the block of the tile's first output: 32-bit)
      float* const tile_dst = p.pts + (long long)(excl >> 7) * kBlockFloats;
      unsigned int rel = (unsigned int)(excl & 127ull);                // offset of the step's first output
      const unsigned int run_base = (unsigned int)excl - rel;
      unsigned int* const run_dst = p.run_src ? p.run_src + (pix0 >> 3) + (lane >> 3) : nullptr;
#pragma unroll
      for (int s = 0; s < kSteps; ++s) {
        const bool ok = (vmask >> s) & 1u;
        const unsigned int m = __ballot_sync(0xffffffffu, ok);
        const unsigned int o = rel + (unsigned int)__popc(m & lt);
        unsigned int col = cb + (unsigned int)lane, row = rowb;
        int day = dayb;
        if (kMode == 1) {
          if (col >= W) {
            col -= W;
            if (++row == H) { row = 0; ++day; }
          }
        } else if (kMode == 2) {
          const unsigned int q = col / W;
          col -= q * W;
          row += q;
          while (row >= H) { row -= H; ++day; }
        }
        if (ok) {
          float z = hv[s];
          if (kPlanes) z = plane_height(p.planes + (size_t)day * 8, col, row, z);
          const float fx = (float)col, fy = (float)row;
          float* dst = tile_dst + (o >> 7) * (unsigned int)kBlockFloats + (o & 127u);
          dst[0] = fx;
          dst[kGroup] = fy;
          dst[2 * kGroup] = z;
          mn[0] = fminf(mn[0], fx); mx[0] = fmaxf(mx[0], fx);
          mn[1] = fminf(mn[1], fy); mx[1] = fmaxf(mx[1], fy);
          mn[2] = fminf(mn[2], z); mx[2] = fmaxf(mx[2], z);
        }
        // run table: points produced before every 8th pixel of the range
        if (run_dst && (lane & 7) == 0 && (unsigned int)(s * 32 + lane) < limit) run_dst[s * 4] = run_base + o;
        rel += (unsigned int)__popc(m);
        // first pixel of the next step
        cb += 32u;
        if (kMode == 0) {
          if (cb >= W) {  // (== W: a step never straddles a row)
            cb = 0;
            if (++rowb == H) { rowb = 0; ++dayb; }
          }
        } else if (kMode == 1) {
          if (cb >= W) {
            cb -= W;
            if (++rowb == H) { rowb = 0; ++dayb; }
          }
        } else {
          const unsigned int q = cb / W;
          cb -= q * W;
          rowb += q;
          while (rowb >= H) { rowb -= H; ++dayb; }
        }
      }
    }
    // 4. the next super-tile becomes the current one
#pragma unroll
    for (int s = 0; s < kSteps; ++s) hv[s] = hn[s];
    vmask = vmask_n; limit = limit_n; cnt = cnt_n;
    sup = sup_n;
    have = have_n;
  }
  if (p.minmax) {
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      const unsigned int a = __reduce_min_sync(0xffffffffu, f2ord(mn[d]));
      const unsigned int b = __reduce_max_sync(0xffffffffu, f2ord(mx[d]));
      if (lane == 0) {
        atomicMin(&p.minmax[d], a);
        atomicMax(&p.minmax[3 + d], b);
      }
    }
  }
}

// ---------------------------------------------------------------------------------------
// Per-day plane fit (plugin.py:161-171) from 9 moments.  Grid (kPlaneBlocks, n_days): CTA b of
// day d reduces a fixed slice of the day's pixels in a fixed order -> deterministic partials;
// plane_solve_kernel adds them in order and solves the 3x3 symmetric eigenproblem (Jacobi).
// ---------------------------------------------------------------------------------------
constexpr int kPlaneBlocks = 64;

__global__ void __launch_bounds__(kThreads) plane_moments_kernel(const UnprojParams p, int n_days,
                                                                 double* partials /*[d][b][10]*/) {
  __shared__ double s_red[kThreads / 32];
  const int d = blockIdx.y;
  const long long day_begin = (long long)(p.day0 + d) * p.HW - p.pix_begin;  // local index
  const long long quads = (p.HW + 3) / 4;
  const double px = 0.5 * (double)(p.W - 1), py = 0.5 * (double)(p.H - 1);
  double m[10];
#pragma unroll
  for (int i = 0; i < 10; ++i) m[i] = 0.0;
  for (long long q = (long long)blockIdx.x * kThreads + threadIdx.x; q < quads;
       q += (long long)gridDim.x * kThreads) {
    const long long li = q * 4;  // index inside the day
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const long long l = li + e;
      if (l >= p.HW) break;
      const long long i = day_begin + l;
      float hv;
      if (load_height1(p, i, hv)) {
        const int row = (int)(l / p.W);
        const int col = (int)(l - (long long)row * p.W);
        const double X = (double)col - px, Y = (double)row - py, Z = (double)hv;
        m[0] += 1.0; m[1] += X; m[2] += Y; m[3] += Z;
        m[4] += X * X; m[5] += X * Y; m[6] += X * Z; m[7] += Y * Y; m[8] += Y * Z; m[9] += Z * Z;
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    double v = m[i];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < kThreads / 32; ++w) t += s_red[w];
      partials[((size_t)d * gridDim.x + blockIdx.x) * 10 + i] = t;
    }
  }
}

__global__ void plane_solve_kernel(const double* partials, int n_blocks, int W, int H,
                                   double* planes /*[d][8]*/) {
  const int d = blockIdx.x;
  if (threadIdx.x != 0) return;
  double m[10];
  for (int i = 0; i < 10; ++i) {
    double t = 0.0;
    for (int b = 0; b < n_blocks; ++b) t += partials[((size_t)d * n_blocks + b) * 10 + i];
    m[i] = t;
  }
  double* pl = planes + (size_t)d * 8;
  const double px = 0.5 * (double)(W - 1), py = 0.5 * (double)(H - 1);
  const double n = m[0];
  if (n < 3.0) {  // oracle skips the fit for < 3 points: identity plane z_rel = z
    pl[0] = px; pl[1] = py; pl[2] = 0.0; pl[3] = 0.0; pl[4] = 0.0; pl[5] = 1.0; pl[6] = n; pl[7] = 0.0;
    return;
  }
  const double cx = m[1] / n, cy = m[2] / n, cz = m[3] / n;
  // scatter matrix of the centred points
  double A[3][3];
  A[0][0] = m[4] - n * cx * cx; A[0][1] = m[5] - n * cx * cy; A[0][2] = m[6] - n * cx * cz;
  A[1][1] = m[7] - n * cy * cy; A[1][2] = m[8] - n * cy * cz; A[2][2] = m[9] - n * cz * cz;
  A[1][0] = A[0][1]; A[2][0] = A[0][2]; A[2][1] = A[1][2];
  double V[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  for (int sweep = 0; sweep < 30; ++sweep) {
    const double off = fabs(A[0][1]) + fabs(A[0][2]) + fabs(A[1][2]);
    if (off < 1e-300) break;
    for (int pi = 0; pi < 2; ++pi)
      for (int qi = pi + 1; qi < 3; ++qi) {
        if (fabs(A[pi][qi]) < 1e-300) continue;
        const double theta = (A[qi][qi] - A[pi][pi]) / (2.0 * A[pi][qi]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 3; ++k) {
          const double akp = A[k][pi], akq = A[k][qi];
          A[k][pi] = c * akp - s * akq;
          A[k][qi] = s * akp + c * akq;
        }
        for (int k = 0; k < 3; ++k) {
          const double apk = A[pi][k], aqk = A[qi][k];
          A[pi][k] = c * apk - s * aqk;
          A[qi][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 3; ++k) {
          const double vkp = V[k][pi], vkq = V[k][qi];
          V[k][pi] = c * vkp - s * vkq;
          V[k][qi] = s * vkp + c * vkq;
        }
      }
  }
  int mi = 0;
  if (A[1][1] < A[mi][mi]) mi = 1;
  if (A[2][2] < A[mi][mi]) mi = 2;
  double nx = V[0][mi], ny = V[1][mi], nz = V[2][mi];
  const double nn = sqrt(nx * nx + ny * ny + nz * nz);
  nx /= nn; ny /= nn; nz /= nn;
  if (nz < 0) { nx = -nx; ny = -ny; nz = -nz; }  // plugin.py:167-168
  pl[0] = cx + px; pl[1] = cy + py; pl[2] = cz; pl[3] = nx; pl[4] = ny; pl[5] = nz; pl[6] = n; pl[7] = 0.0;
}

// ---------------------------------------------------------------------------------------
// Cloud statistics: per-dimension min / max (frame + error bound) and first/second moments
// about the frame origin (mean, and var(X) for sklearn's tolerance, _kmeans.py:285-293).
// ---------------------------------------------------------------------------------------
__host__ __device__ inline float ord2f(unsigned int u) {
  const unsigned int b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  float f;
  memcpy(&f, &b, 4);
  return f;
#endif
}

// out[0..2] = ordered min x,y,z ; out[3..5] = ordered max.  Caller pre-fills min with
// 0xffffffff and max with 0.  One warp per 128-point block of the blocked cloud.
__global__ void __launch_bounds__(kThreads) minmax_kernel(const float* pts, long long n, unsigned int* out) {
  float mn[3] = {__int_as_float(0x7f800000), __int_as_float(0x7f800000), __int_as_float(0x7f800000)};
  float mx[3] = {__int_as_float(0xff800000), __int_as_float(0xff800000), __int_as_float(0xff800000)};
  const int lane = threadIdx.x & 31;
  const long long n_groups = (n + kGroup - 1) / kGroup;
  const long long stride = (long long)gridDim.x * (kThreads / 32);
  for (long long g = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); g < n_groups; g += stride) {
    const float* blk = pts + g * kBlockFloats + lane * 4;
    const float4 vx = ldg_stream_f4(blk), vy = ldg_stream_f4(blk + kGroup), vz = ldg_stream_f4(blk + 2 * kGroup);
    const float ax[4] = {vx.x, vx.y, vx.z, vx.w}, ay[4] = {vy.x, vy.y, vy.z, vy.w}, az[4] = {vz.x, vz.y, vz.z, vz.w};
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (g * kGroup + lane * 4 + e < n) {
        mn[0] = fminf(mn[0], ax[e]); mx[0] = fmaxf(mx[0], ax[e]);
        mn[1] = fminf(mn[1], ay[e]); mx[1] = fmaxf(mx[1], ay[e]);
        mn[2] = fminf(mn[2], az[e]); mx[2] = fmaxf(mx[2], az[e]);
      }
  }
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const unsigned int a = __reduce_min_sync(0xffffffffu, f2ord(mn[d]));
    const unsigned int b = __reduce_max_sync(0xffffffffu, f2ord(mx[d]));
    if (lane == 0) {
      atomicMin(&out[d], a);
      atomicMax(&out[3 + d], b);
    }
  }
}

// partials[b][6] = sum (x-o), sum (x-o)^2 per dim, in FP64, fixed order inside the CTA;
// the last CTA adds the partials in CTA order into out[6].
__global__ void __launch_bounds__(kThreads) moments_kernel(const float* pts, long long n, FrameF f, double* partials,
                                                           unsigned int* ticket, double* out) {
  __shared__ double s_red[kThreads / 32];
  __shared__ bool s_last;
  double m[6] = {0, 0, 0, 0, 0, 0};
  const int lane = threadIdx.x & 31;
  const long long n_groups = (n + kGroup - 1) / kGroup;
  const long long stride = (long long)gridDim.x * (kThreads / 32);
  for (long long g = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); g < n_groups; g += stride) {
    const float* blk = pts + g * kBlockFloats + lane * 4;
    const float4 vx = ldg_stream_f4(blk), vy = ldg_stream_f4(blk + kGroup), vz = ldg_stream_f4(blk + 2 * kGroup);
    const float ax[4] = {vx.x, vx.y, vx.z, vx.w}, ay[4] = {vy.x, vy.y, vy.z, vy.w}, az[4] = {vz.x, vz.y, vz.z, vz.w};
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (g * kGroup + lane * 4 + e < n) {
        const double X = (double)ax[e] - (double)f.ox, Y = (double)ay[e] - (double)f.oy,
                     Z = (double)az[e] - (double)f.oz;
        m[0] += X; m[1] += Y; m[2] += Z;
        m[3] += X * X; m[4] += Y * Y; m[5] += Z * Z;
      }
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    double v = m[i];
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < kThreads / 32; ++w) t += s_red[w];
      partials[(size_t)blockIdx.x * 6 + i] = t;
    }
  }
  if (threadIdx.x == 0) {
    __threadfence();
    s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last && threadIdx.x < 6) {
    __threadfence();
    double t = 0.0;
    for (unsigned int b = 0; b < gridDim.x; ++b) t += partials[(size_t)b * 6 + threadIdx.x];
    out[threadIdx.x] = t;
    if (threadIdx.x == 0) *ticket = 0u;
  }
}

// [n][3] (x,y,z) or SoA x[n] y[n] z[n]  ->  blocked cloud
__global__ void __launch_bounds__(kThreads) to_blocked_kernel(const float* src, long long n, int soa, float* pts) {
  const long long total = n * 3;
  for (long long t = (long long)blockIdx.x * kThreads + threadIdx.x; t < total; t += (long long)gridDim.x * kThreads) {
    long long i;
    int c;
    if (soa) {
      c = (int)(t / n);
      i = t - (long long)c * n;
    } else {
      i = t / 3;
      c = (int)(t - i * 3);
    }
    pts[pt_off(i) + c * kGroup] = src[t];  // coalesced reads
  }
}

// out[i] = (x, y, z) of point idx[i]  (X[seeds] of init="random", sklearn/_kmeans.py:1014-1021)
// idx are global indices; a rank owns [rank_offset, rank_offset + n) and writes zeros elsewhere
__global__ void gather_points_kernel(const float* pts, const long long* idx, int m, long long rank_offset,
                                     long long n, float* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= m) return;
  const long long l = idx[i] - rank_offset;
  const bool mine = l >= 0 && l < n;
  const float* q = pts + pt_off(mine ? l : 0);
  out[3 * i + 0] = mine ? q[0] : 0.f;
  out[3 * i + 1] = mine ? q[kGroup] : 0.f;
  out[3 * i + 2] = mine ? q[2 * kGroup] : 0.f;
}

// zero the unused tail of the last block (and nothing else)
__global__ void zero_tail_kernel(float* pts, long long n) {
  const long long cap = (n + kGroup - 1) / kGroup * kGroup;
  for (long long i = n + threadIdx.x; i < cap; i += blockDim.x) {
    float* d = pts + pt_off(i);
    d[0] = 0.f;
    d[kGroup] = 0.f;
    d[2 * kGroup] = 0.f;
  }
}

// blocked cloud -> [n][3] in (x,y,z) or napari (z,y,x) order; coalesced stores
__global__ void __launch_bounds__(kThreads) blocked_to_aos_kernel(const float* pts, long long n, int napari,
                                                                  float* out) {
  const long long total = n * 3;
  for (long long t = (long long)blockIdx.x * kThreads + threadIdx.x; t < total; t += (long long)gridDim.x * kThreads) {
    const long long i = t / 3;
    const int c = (int)(t - i * 3);
    const int src = napari ? 2 - c : c;
    out[t] = pts[pt_off(i) + src * kGroup];
  }
}

// same for the points [range[0], range[1]) only (one slab of a streamed unprojection)
__global__ void __launch_bounds__(kThreads) blocked_to_aos_range_kernel(const float* pts, const long long* range,
                                                                        int napari, float* out) {
  const long long t0 = range[0] * 3, t1 = range[1] * 3;
  for (long long t = t0 + (long long)blockIdx.x * kThreads + threadIdx.x; t < t1; t += (long long)gridDim.x * kThreads) {
    const long long i = t / 3;
    const int c = (int)(t - i * 3);
    const int src = napari ? 2 - c : c;
    out[t] = pts[pt_off(i) + src * kGroup];
  }
}

}  // namespace mdkm
