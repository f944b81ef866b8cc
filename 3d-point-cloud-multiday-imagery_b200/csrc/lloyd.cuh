// Lloyd k-means kernels for d = 3 on sm_100a.
//
//   lloyd_step_kernel   ONE kernel per Lloyd iteration:
//                         prologue  the centroid update the PREVIOUS iteration left behind
//                                 (_k_means_common.pyx:274-311, _kmeans.py:721-738: average, centre
//                                 shift, convergence test, next centroid table), applied from its
//                                 sums -- gathered from the peer ranks' NVLink packets when there are
//                                 several -- by every CTA (deferred_update_rows / deferred_update);
//                         pass 1  classification: whole 128-point groups settled from their
//                                 cached summaries (box + fixed-point sums), no point read;
//                         --      grid barrier;
//                         pass 2  the groups a cluster boundary crosses, point by point:
//                                 nearest-centroid assignment + per-cluster sum / count
//                                 (sklearn/cluster/_k_means_lloyd.pyx:168-218; the reference
//                                 reaches it through KMeans.fit at
//                                 members/jasraj/land_use_classification/core.py:227-228);
//                         end     the sums go to acc[seq % 3]; with several ranks the last CTA
//                                 sends them to the peers; nobody waits.
//   lloyd_settle_kernel the update still pending behind the last launch of a run; table / buffers
//                       back to the layout every other kernel expects
//   lloyd_update_kernel the update alone (NCCL exchange path, and after a relocation)
//   lloyd_final_kernel  labels in the reference's point order from the final centroids +
//                       inertia + int32 labels (_kmeans.py:742-756, _k_means_common.pyx:94-124)
//   group_summary_kernel  the per-group summaries (once per cloud and frame)
//
// Work unit: a group of 128 consecutive points = one 1536-byte block of the blocked cloud
// (common.cuh: x[128] y[128] z[128]); the step kernel streams the tile-ordered mirror
// (mirror.cuh), where a group is compact in x and y.  In pass 2 a group is fetched with 1-D
// TMA bulk copies and everything inside it is warp-synchronous: no CTA barrier in the loop.
//
// Numerics (DESIGN.md "Exactness"):
//   * candidate pruning / classification: d_j(x) - d_ref(x) is linear in x, so its minimum
//     over a group's bounding box is a corner value; a centroid whose minimum gap exceeds a
//     margin covering every FP32 rounding involved cannot be the nearest of any point of the
//     group.  Conservative, so the result is identical to brute force.
//   * distances: FP32 CUDA cores, expanded form  ||c'||^2 - 2 x'.c'  (3 FFMA per pair) in a
//     frame whose origin makes pixel-grid coordinates exact.  A rigorous bound E on the
//     FP32 error of that expression is carried with every centroid table; a point whose best
//     and second-best FP32 distances are closer than 2E is re-decided in FP64 with the exact
//     centroids, so the label equals the FP64 argmin (lowest index on ties) up to FP64
//     rounding.
//   * sums: coordinates are rounded once to a 2^-22-of-range fixed-point grid and summed as
//     integers (warp REDUX -> shared int64 -> global int64).  Integer addition is
//     associative, so the sums are bit-identical for any point order, grid size, run, or
//     number of GPUs.
#pragma once
#include "common.cuh"
#include "ptx.cuh"

namespace mdkm {

// ---------------------------------------------------------------------------------------
// K4: centroid update + convergence.  One CTA.
// ---------------------------------------------------------------------------------------
struct UpdateParams {
  unsigned long long* acc;  // [kpad*4 + 8], global sums (already allreduced)
  unsigned long long* acc_saved;  // [kpad*4 + 8]: the sums as they were when the loop paused
  unsigned char* table;     // centroid table, updated in place
  DevStatus* st;
  Frame fr;
  double inv_scale[3];      // 1 / fr.scale (powers of two: multiplying is exact)
  double mean[3];           // data mean (only used for sklearn's empty-cluster copy quirk)
  int k, kpad;
  int allow_pause;          // 1: pause for relocation when a cluster is empty
  int ignore_status;
};

__device__ __forceinline__ double block_sum_fixed(double v, double* s_red) {
  // fixed-order reduction: shuffle tree inside the warp, warps combined in index order
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int w = threadIdx.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[w] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += s_red[i];
  return t;
}

__device__ __forceinline__ double block_max(double v, double* s_red) {
  for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_down_sync(0xffffffffu, v, o));
  const int w = threadIdx.x >> 5;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) s_red[w] = v;
  __syncthreads();
  double t = 0.0;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t = fmax(t, s_red[i]);
  return t;
}

// Buckets the k centroids whose fast rows are in `fast` (shared or global memory) by the x-y grid of
// common.cuh (for k >= kBucketMinK) into the bucket section `sec` (shared or global memory).
// Executed by all threads of ONE CTA right after that CTA wrote the fast rows.
__device__ __forceinline__ void build_centroid_buckets(const float4* fast, unsigned char* sec, int k, int kpad,
                                                       const Frame& fr) {
  if (k < kBucketMinK) return;
  __shared__ int s_cnt[32 * 32 + 1];
  const int g = bucket_g(k), cells = g * g, tid = threadIdx.x;
  BucketHdr hdr;
  hdr.hx = (float)fr.halfrange[0]; hdr.hy = (float)fr.halfrange[1];
  hdr.inv_x = (float)g / (2.0f * fmaxf(hdr.hx, 1e-30f));
  hdr.inv_y = (float)g / (2.0f * fmaxf(hdr.hy, 1e-30f));
  unsigned short* start = reinterpret_cast<unsigned short*>(sec + sizeof(BucketHdr));
  unsigned short* perm = start + cells + 1;
  __syncthreads();  // the fast rows of this CTA's other threads are visible
  for (int i = tid; i <= cells; i += blockDim.x) s_cnt[i] = 0;
  __syncthreads();
  for (int j = tid; j < k; j += blockDim.x) {
    const float4 r = fast[j];
    const int b = bucket_coord(-0.5f * r.y, hdr.hy, hdr.inv_y, g) * g + bucket_coord(-0.5f * r.x, hdr.hx, hdr.inv_x, g);
    atomicAdd(&s_cnt[b], 1);
  }
  __syncthreads();
  {
    // exclusive scan of the cell counts, in place (cells <= 1024: four per thread of a 256-thread CTA)
    __shared__ int s_wsum[32];
    int v[4], tsum = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid * 4 + e;
      v[e] = idx < cells ? s_cnt[idx] : 0;
      tsum += v[e];
    }
    int incl = tsum;
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if ((tid & 31) >= o) incl += t;
    }
    if ((tid & 31) == 31) s_wsum[tid >> 5] = incl;
    __syncthreads();
    int run = incl - tsum;
    for (int w = 0; w < (tid >> 5); ++w) run += s_wsum[w];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid * 4 + e;
      if (idx < cells) {
        s_cnt[idx] = run;
        start[idx] = (unsigned short)run;
        run += v[e];
      }
    }
    if (tid == 0) {
      start[cells] = (unsigned short)k;
      *reinterpret_cast<BucketHdr*>(sec) = hdr;
    }
  }
  __syncthreads();
  for (int j = tid; j < k; j += blockDim.x) {
    const float4 r = fast[j];
    const int b = bucket_coord(-0.5f * r.y, hdr.hy, hdr.inv_y, g) * g + bucket_coord(-0.5f * r.x, hdr.hx, hdr.inv_x, g);
    perm[atomicAdd(&s_cnt[b], 1)] = (unsigned short)j;
  }
  for (int j = k + tid; j < kpad; j += blockDim.x) perm[j] = 0;
}

// Executed by all kThreads threads of ONE CTA: the stand-alone update kernel, or the last CTA
// of a fused step kernel.  Reads the accumulators through L2 (they were produced by atomics).
// It sits on the critical path of every iteration, so global round trips are kept to one: a
// thread fetches the accumulator row and the old centroid of its cluster together, and the
// five block-wide reductions share one pair of barriers.
__device__ __forceinline__ void lloyd_update_body(const UpdateParams& u) {
  DevStatus* st = u.st;
  __shared__ double s_red[5][kThreads / 32];
  __shared__ int s_nempty;
  __shared__ unsigned long long s_maxcnt;  // (count << 13) | (2 * kMaxK - 1 - j): argmax, first wins
  const int tid = threadIdx.x;
  if (tid == 0) {
    s_nempty = 0;
    s_maxcnt = 0ull;
  }
  __syncthreads();
  float4* fast = reinterpret_cast<float4*>(u.table);
  double4* exact = reinterpret_cast<double4*>(u.table + exact_offset(u.kpad));
  // rows of this thread's first cluster (the only one when k <= kThreads), fetched up front
  const bool have0 = tid < u.k;
  ulonglong2 a0 = make_ulonglong2(0ull, 0ull), b0 = a0;
  double4 old0 = make_double4(0.0, 0.0, 0.0, 0.0);
  const unsigned long long n_changed = __ldcg(&u.acc[u.kpad * 4 + 0]);  // (same round trip as the rows below)
  if (have0) {
    a0 = __ldcg(reinterpret_cast<const ulonglong2*>(u.acc + tid * 4));
    b0 = __ldcg(reinterpret_cast<const ulonglong2*>(u.acc + tid * 4 + 2));
    old0 = exact[tid];
  }
  // empty clusters and the heaviest cluster (np.argmax: first maximum)
  int my_empty = 0;
  unsigned long long my_max = 0ull;
  for (int j = tid; j < u.k; j += kThreads) {
    const unsigned long long cnt = j == tid ? b0.y : __ldcg(&u.acc[j * 4 + 3]);
    if (cnt == 0ull) ++my_empty;
    const unsigned long long key = (cnt << 13) | (unsigned long long)(kMaxK * 2 - 1 - j);
    my_max = key > my_max ? key : my_max;
  }
  my_empty = __reduce_add_sync(0xffffffffu, my_empty);
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long t = __shfl_down_sync(0xffffffffu, my_max, o);
    my_max = t > my_max ? t : my_max;
  }
  if ((tid & 31) == 0) {
    if (my_empty) atomicAdd(&s_nempty, my_empty);
    atomicMax(&s_maxcnt, my_max);
  }
  __syncthreads();
  const int n_empty = s_nempty;
  if (n_empty > 0 && u.allow_pause) {
    // the sums are parked: exchanges already enqueued behind this point (NCCL path) keep
    // running on `acc`, so the host restores it from here before it relocates
    for (int i = tid; i < u.kpad * 4 + 8; i += kThreads) u.acc_saved[i] = __ldcg(&u.acc[i]);
    if (tid == 0) {
      st->paused = 1;
      st->n_empty = n_empty;
    }
    return;  // the host sequences the relocation kernels and re-runs update
  }
  const int jmax = kMaxK * 2 - 1 - (int)(s_maxcnt & 0x1fffull);

  double shift2 = 0.0, m_cn = 0.0, m_cx = 0.0, m_cy = 0.0, m_cz = 0.0;
  for (int j = tid; j < u.kpad; j += kThreads) {
    if (j < u.k) {
      const bool first = j == tid;
      const double4 old = first ? old0 : exact[j];
      ulonglong2 a = first ? a0 : __ldcg(reinterpret_cast<const ulonglong2*>(u.acc + j * 4));
      ulonglong2 b = first ? b0 : __ldcg(reinterpret_cast<const ulonglong2*>(u.acc + j * 4 + 2));
      double cx, cy, cz;
      bool raw = false;
      if (b.y == 0ull) {
        // sklearn/_k_means_common.pyx:289-293: copy of the heaviest cluster's row -- which is
        // still the un-averaged sum when that row comes later in the loop.
        a = __ldcg(reinterpret_cast<const ulonglong2*>(u.acc + jmax * 4));
        b = __ldcg(reinterpret_cast<const ulonglong2*>(u.acc + jmax * 4 + 2));
        raw = jmax > j;
      }
      const double sc = (double)b.y;
      const double qx = (double)(long long)a.x * u.inv_scale[0];
      const double qy = (double)(long long)a.y * u.inv_scale[1];
      const double qz = (double)(long long)b.x * u.inv_scale[2];
      if (!raw) {
        const double alpha = 1.0 / sc;  // pyx:284-287: centers *= 1/weight
        cx = qx * alpha;
        cy = qy * alpha;
        cz = qz * alpha;
      } else {
        // raw sum in sklearn's mean-centred frame, expressed in ours
        cx = qx + sc * (u.fr.origin[0] - u.mean[0]) + (u.mean[0] - u.fr.origin[0]);
        cy = qy + sc * (u.fr.origin[1] - u.mean[1]) + (u.mean[1] - u.fr.origin[1]);
        cz = qz + sc * (u.fr.origin[2] - u.mean[2]) + (u.mean[2] - u.fr.origin[2]);
      }
      const double dx = cx - old.x, dy = cy - old.y, dz = cz - old.z;
      const double sh = sqrt(dx * dx + dy * dy + dz * dz);  // _center_shift, pyx:298-311
      shift2 += sh * sh;                                     // (center_shift**2).sum()
      const double cn = cx * cx + cy * cy + cz * cz;
      exact[j] = make_double4(cx, cy, cz, cn);
      fast[j] = make_float4((float)(-2.0 * cx), (float)(-2.0 * cy), (float)(-2.0 * cz), (float)cn);
      m_cn = fmax(m_cn, cn);
      m_cx = fmax(m_cx, fabs(cx));
      m_cy = fmax(m_cy, fabs(cy));
      m_cz = fmax(m_cz, fabs(cz));
    } else {
      fast[j] = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7f800000));
      exact[j] = make_double4(0.0, 0.0, 0.0, 1.0 / 0.0);
    }
  }
  build_centroid_buckets(fast, u.table + bucket_offset(u.kpad), u.k, u.kpad, u.fr);
  // fixed-order reductions: shuffle tree inside the warp, warps combined in index order
  for (int o = 16; o > 0; o >>= 1) {
    shift2 += __shfl_down_sync(0xffffffffu, shift2, o);
    m_cn = fmax(m_cn, __shfl_down_sync(0xffffffffu, m_cn, o));
    m_cx = fmax(m_cx, __shfl_down_sync(0xffffffffu, m_cx, o));
    m_cy = fmax(m_cy, __shfl_down_sync(0xffffffffu, m_cy, o));
    m_cz = fmax(m_cz, __shfl_down_sync(0xffffffffu, m_cz, o));
  }
  if ((tid & 31) == 0) {
    const int w = tid >> 5;
    s_red[0][w] = shift2; s_red[1][w] = m_cn; s_red[2][w] = m_cx; s_red[3][w] = m_cy; s_red[4][w] = m_cz;
  }
  __syncthreads();  // also: every thread has read its accumulator rows
  for (int i = tid; i < u.kpad * 4 + 8; i += kThreads) u.acc[i] = 0ull;
  if (tid == 0) {
    shift2 = 0.0; m_cn = 0.0; m_cx = 0.0; m_cy = 0.0; m_cz = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) {
      shift2 += s_red[0][w];
      m_cn = fmax(m_cn, s_red[1][w]);
      m_cx = fmax(m_cx, s_red[2][w]);
      m_cy = fmax(m_cy, s_red[3][w]);
      m_cz = fmax(m_cz, s_red[4][w]);
    }
    // FP32 error bound of the fast distances (DESIGN.md "Exactness"): u = 2^-24
    const double ue = 5.9604644775390625e-08;
    const double E = ue * (4.0 * m_cn + 10.0 * (u.fr.halfrange[0] * m_cx + u.fr.halfrange[1] * m_cy +
                                                 u.fr.halfrange[2] * m_cz));
    st->thresh = __double2float_ru(2.0 * E * 1.001 + 1e-37);
    st->shift2 = shift2;
    st->n_changed = n_changed;
    st->n_empty = n_empty;
    st->paused = 0;
    const int it = st->iter + 1;
    st->iter = it;
    if (!st->first && n_changed == 0ull) {  // _kmeans.py:721-726
      st->strict = 1;
      st->done = 1;
    } else if (shift2 <= st->tol) {         // _kmeans.py:729-738
      st->done = 1;
    }
    if (it >= st->max_iter) st->done = 1;
    st->first = 0;
  }
}

__global__ void __launch_bounds__(kThreads, 1) lloyd_update_kernel(const UpdateParams u) {
  if (!u.ignore_status && (u.st->done || (u.st->paused && u.allow_pause))) return;
  lloyd_update_body(u);
}



// exact centroid row: two plain 16 B loads (L1-cached; measured faster than the non-coherent
// path on the many-centroid configurations)
__device__ __forceinline__ double4 ld_c64(const double4* p) {
  const double2 a = *reinterpret_cast<const double2*>(p);
  const double2 b = *(reinterpret_cast<const double2*>(p) + 1);
  return make_double4(a.x, a.y, b.x, b.y);
}

// Can centroid `row` beat the reference centroid `ref` anywhere in the box?  Both rows are in
// the expanded form (-2c', ||c'||^2), so d_row(x) - d_ref(x) = a.w + a.xyz . x is LINEAR in x
// and its minimum over the box is attained at a corner, coordinate by coordinate.
__device__ __forceinline__ float min_gap_over_box(const float4 row, const float4 ref, float bx0, float bx1,
                                                  float by0, float by1, float bz0, float bz1) {
  const float ax = row.x - ref.x, ay = row.y - ref.y, az = row.z - ref.z, aw = row.w - ref.w;
  return aw + fminf(ax * bx0, ax * bx1) + fminf(ay * by0, ay * by1) + fminf(az * bz0, az * bz1);
}

struct __align__(16) GroupSummary {
  float lo[3], hi[3];  // box of the centred FP32 coordinates
  int q[3];            // sum of the fixed-point coordinates of the group's points
  int n;               // points in the group (128 except the cloud's tail)
  int pad[2];
};

struct StepParams {
  const float* pts;           // blocked cloud (common.cuh)
  long long n;
  void* labels;               // uint8 (k <= 256) or uint16, capacity = whole groups
  unsigned char* table;       // TWO centroid tables (see common.cuh), table_stride bytes apart: launch `seq` assigns
  size_t table_stride;        //   with table[seq & 1]
  unsigned long long* acc;    // THREE accumulators of acc_slot words: [kpad*4] (qx,qy,qz,count) + [kpad*4 + 0] n_changed;
  int acc_slot;               //   launch `seq` adds into acc[seq % 3]
  int seq;                    // index of this launch among the fused launches since the last settle kernel (0 otherwise)
  DevStatus* st;
  FrameF f;
  int k, kpad;
  int ignore_status;          // 1: test hook (run even when done/paused)
  int fuse_update;            // 1: fused run -- this launch applies the update the previous one left behind (seq > 0),
                              //    adds into the rotating accumulators and, with several ranks, sends its sums to the
                              //    peers (NVLink, no host, no NCCL); 0: the host exchanges and updates between launches
  int two_level;              // 1: classification pass walks super-groups first (large clouds)
  int settle;                 // 0: measurement mode, no group is settled from its summary --
                              //    every point goes through the per-point pass (MDKM_OPT_SETTLE_GROUPS)
  const GroupSummary* gsum;   // per-group box + cached sums (static per cloud and frame)
  const void* ssum;           // SuperSummary per kSuper groups (defined with the classification pass)
  int* worklist;              // groups the classification pass could not settle
  int* work_count;            // TWO counters of entries: launch `seq` uses work_count[seq & 1] and clears the other
  int* glabel;                // per group: the label that owns its whole box, else -1
  unsigned int* grid_bar;     // arrival counter of the in-kernel grid barrier
  UpdateParams upd;
  PeerXchg px;
};

// ---------------------------------------------------------------------------------------
// Group summaries.  A group's bounding box and fixed-point coordinate sums never change while
// the cloud and its frame stay the same, so they are computed once (48 B per 128 points).
// With them a whole group can be settled WITHOUT touching its points: if one centroid beats
// every other one over the whole box (the same conservative linear-gap test assign_group
// uses), all 128 points take that label and the cached sums are added to its accumulator.
// On raster-ordered clouds that covers most groups; only the rest (a cluster boundary crosses
// them) are streamed through the per-point kernel.  Results are identical to brute force.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) group_summary_kernel(const float* pts, long long n, FrameF f,
                                                                 GroupSummary* out) {
  const int lane = threadIdx.x & 31;
  const long long n_groups = (n + kGroup - 1) / kGroup;
  const long long stride = (long long)gridDim.x * (kThreads / 32);
  for (long long g = (long long)blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5); g < n_groups; g += stride) {
    const float* blk = pts + g * kBlockFloats + lane * 4;
    const float4 vx = ldg_stream_f4(blk), vy = ldg_stream_f4(blk + kGroup), vz = ldg_stream_f4(blk + 2 * kGroup);
    const float xs[4] = {vx.x, vx.y, vx.z, vx.w}, ys[4] = {vy.x, vy.y, vy.z, vy.w}, zs[4] = {vz.x, vz.y, vz.z, vz.w};
    float lo[3] = {__int_as_float(0x7f800000), __int_as_float(0x7f800000), __int_as_float(0x7f800000)};
    float hi[3] = {__int_as_float(0xff800000), __int_as_float(0xff800000), __int_as_float(0xff800000)};
    int q[3] = {0, 0, 0};
    int cnt = 0;
    const long long i0 = g * kGroup + lane * 4;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      // the unused tail of the last block is zero-filled and belongs to the box, exactly as
      // the per-point kernel sees it; it does not belong to the sums
      const float xc = xs[e] - f.ox, yc = ys[e] - f.oy, zc = zs[e] - f.oz;
      lo[0] = fminf(lo[0], xc); hi[0] = fmaxf(hi[0], xc);
      lo[1] = fminf(lo[1], yc); hi[1] = fmaxf(hi[1], yc);
      lo[2] = fminf(lo[2], zc); hi[2] = fmaxf(hi[2], zc);
      if (i0 + e < n) {
        q[0] += (int)(__float_as_uint(fmaf(xc, f.sx, kMagic)) - kMagicBits);
        q[1] += (int)(__float_as_uint(fmaf(yc, f.sy, kMagic)) - kMagicBits);
        q[2] += (int)(__float_as_uint(fmaf(zc, f.sz, kMagic)) - kMagicBits);
        ++cnt;
      }
    }
    GroupSummary gs;
#pragma unroll
    for (int d = 0; d < 3; ++d) {
      gs.lo[d] = redux_min_f32(lo[d]);
      gs.hi[d] = redux_max_f32(hi[d]);
      gs.q[d] = __reduce_add_sync(0xffffffffu, q[d]);
    }
    gs.n = __reduce_add_sync(0xffffffffu, cnt);
    gs.pad[0] = gs.pad[1] = 0;
    if (lane == 0) out[g] = gs;
  }
}

// Classification pass, run by every CTA of the step kernel before the per-point work.
// One THREAD per group.  A group that was settled with label L in the previous iteration is
// re-tested against L only (one pass over the centroid table); a group that was not settled
// goes straight to the per-point pass, which hands it back here (glabel >= 0) as soon as one
// centroid owns its whole box.  In the first iteration every group is tested against the
// centroid nearest to its box centre.  Settled groups add their cached sums to `s_acc` (the
// warp's accumulator slice) and never touch their points; the others are appended to the
// global worklist (staged per warp in shared memory).
constexpr int kClassifyList = 2048;  // shared-memory staging of the worklist (entries per CTA)

// The same summaries one level up: kSuper consecutive groups (1024 points) with the union of
// their boxes and the sum of their sums.  Most of the cloud lies deep inside one cluster, so the
// classification pass first tests whole super-groups -- one box test settles eight groups -- and
// only looks at the groups of the super-groups that fail.  Static per cloud and frame, like the
// group summaries.
constexpr int kSuper = 8;
struct __align__(16) SuperSummary {
  float lo[3], hi[3];  // union of the groups' boxes
  int n;               // points (kSuper * kGroup unless the cloud ends inside)
  int pad;
  long long q[3];      // sum of the fixed-point coordinates
  long long pad2;
};
static_assert(sizeof(SuperSummary) == 64, "SuperSummary is read as four 16-byte words");

// One lane per group (coalesced 48-byte reads), the eight lanes of a super-group combined by shuffles.
__global__ void __launch_bounds__(kThreads) super_summary_kernel(const GroupSummary* __restrict__ gsum, int n_groups,
                                                                 SuperSummary* __restrict__ out) {
  static_assert(kSuper == 8, "eight lanes per super-group");
  const int n_pad = (n_groups + 31) / 32 * 32;  // whole warps: the shuffles below need all 32 lanes
  const int n_super = (n_groups + kSuper - 1) / kSuper;
  for (int g = blockIdx.x * kThreads + threadIdx.x; g < n_pad; g += gridDim.x * kThreads) {  // warp-uniform trip count
    float lo[3] = {__int_as_float(0x7f800000), __int_as_float(0x7f800000), __int_as_float(0x7f800000)};
    float hi[3] = {__int_as_float(0xff800000), __int_as_float(0xff800000), __int_as_float(0xff800000)};
    long long q[3] = {0, 0, 0};
    int n = 0;
    if (g < n_groups) {
      const float4* src = reinterpret_cast<const float4*>(gsum + g);
      const float4 a = __ldg(src), b = __ldg(src + 1), c = __ldg(src + 2);
      lo[0] = a.x; lo[1] = a.y; lo[2] = a.z; hi[0] = a.w; hi[1] = b.x; hi[2] = b.y;
      q[0] = __float_as_int(b.z); q[1] = __float_as_int(b.w); q[2] = __float_as_int(c.x);
      n = __float_as_int(c.y);
    }
#pragma unroll
    for (int o = 1; o < kSuper; o <<= 1) {
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        lo[d] = fminf(lo[d], __shfl_xor_sync(0xffffffffu, lo[d], o));
        hi[d] = fmaxf(hi[d], __shfl_xor_sync(0xffffffffu, hi[d], o));
        q[d] += __shfl_xor_sync(0xffffffffu, q[d], o);
      }
      n += __shfl_xor_sync(0xffffffffu, n, o);
    }
    if ((threadIdx.x & (kSuper - 1)) == 0 && g / kSuper < n_super) {
      SuperSummary s;
      for (int d = 0; d < 3; ++d) { s.lo[d] = lo[d]; s.hi[d] = hi[d]; s.q[d] = q[d]; }
      s.n = n; s.pad = 0; s.pad2 = 0;
      out[g / kSuper] = s;
    }
  }
}

template <bool kPrivate>
__device__ __forceinline__ void acc_add(unsigned long long* s_acc, int lab, long long sx, long long sy,
                                        long long sz, unsigned int cnt);

// The centroid nearest to the centre of a box (lowest index on ties).
__device__ __forceinline__ int nearest_to_box_centre(const float4* __restrict__ s_fast, int k, float lo0, float lo1,
                                                     float lo2, float hi0, float hi1, float hi2) {
  const float mx = 0.5f * (lo0 + hi0), my = 0.5f * (lo1 + hi1), mz = 0.5f * (lo2 + hi2);
  float dmin = __int_as_float(0x7f800000);
  int ref = 0;
  for (int j = 0; j < k; ++j) {
    const float4 r = s_fast[j];
    const float d = fmaf(mx, r.x, fmaf(my, r.y, fmaf(mz, r.z, r.w)));
    if (d < dmin) { dmin = d; ref = j; }
  }
  return ref;
}

// Is centroid `ref` the only one that can be nearest (within the margin) to a point of the box?
__device__ __forceinline__ bool box_owned_by(const float4* __restrict__ s_fast, int k, const unsigned char* s_bkt,
                                             int ref, float margin, float lo0, float lo1, float lo2, float hi0,
                                             float hi1, float hi2) {
  const float4 rr = s_fast[ref];
  int ncand = 0;
  if (s_bkt == nullptr) {
    // few centroids: all of them, with the box as centre + half-widths -- the minimum of the
    // (linear) gap over the box is its value at the centre minus sum_d |a_d| h_d.  The
    // rounding of this form is covered by a margin of 6 * thresh instead of 4 * thresh.
    // (A cheap "box inside the safe ball of c_ref" test in front of this loop was measured: one
    // thread per box means a warp skips the loop only when all its 32 boxes pass, and the extra
    // test cost more than those warps saved -- not kept.)
    const float mx = 0.5f * (lo0 + hi0), my = 0.5f * (lo1 + hi1), mz = 0.5f * (lo2 + hi2);
    const float hx = 0.5f * (hi0 - lo0), hy = 0.5f * (hi1 - lo1), hz = 0.5f * (hi2 - lo2);
    const float lim = fmaf(mx, rr.x, fmaf(my, rr.y, fmaf(mz, rr.z, rr.w))) + 1.5f * margin;
#pragma unroll 4
    for (int j = 0; j < k; ++j) {
      const float4 r = s_fast[j];
      const float dj = fmaf(mx, r.x, fmaf(my, r.y, fmaf(mz, r.z, r.w)));
      const float reach = fmaf(fabsf(r.x - rr.x), hx, fmaf(fabsf(r.y - rr.y), hy, fabsf(r.z - rr.z) * hz));
      ncand += (dj - reach <= lim) ? 1 : 0;  // j == ref: reach = 0, dj <= lim: counted once
    }
  } else {
    // Only centroids near the box can win: d_j(x) <= d_ref(x) + margin at some x of the box
    // implies |x - c_j| <= sqrt(r^2 + margin), r = largest distance from c_ref to the box;
    // so c_j lies in the box grown by that reach, and only those buckets are visited.
    const BucketHdr hdr = *reinterpret_cast<const BucketHdr*>(s_bkt);
    const int g = bucket_g(k);
    const unsigned short* start = reinterpret_cast<const unsigned short*>(s_bkt + sizeof(BucketHdr));
    const unsigned short* perm = start + g * g + 1;
    const float cx = -0.5f * rr.x, cy = -0.5f * rr.y, cz = -0.5f * rr.z;
    const float dx = fmaxf(fabsf(lo0 - cx), fabsf(hi0 - cx)), dy = fmaxf(fabsf(lo1 - cy), fabsf(hi1 - cy)),
                dz = fmaxf(fabsf(lo2 - cz), fabsf(hi2 - cz));
    const float reach = sqrtf(fmaf(dx, dx, fmaf(dy, dy, dz * dz)) + 2.0f * margin) * 1.0001f + 1e-3f / hdr.inv_x;
    const int bx0 = bucket_coord(lo0 - reach, hdr.hx, hdr.inv_x, g), bx1 = bucket_coord(hi0 + reach, hdr.hx, hdr.inv_x, g);
    const int by0 = bucket_coord(lo1 - reach, hdr.hy, hdr.inv_y, g), by1 = bucket_coord(hi1 + reach, hdr.hy, hdr.inv_y, g);
    ncand = 1;  // ref itself
    for (int by = by0; by <= by1 && ncand <= 1; ++by) {
      const int i1 = start[by * g + bx1 + 1];
      for (int i = start[by * g + bx0]; i < i1; ++i) {
        const int j = perm[i];
        if (j != ref && min_gap_over_box(s_fast[j], rr, lo0, hi0, lo1, hi1, lo2, hi2) <= margin) {
          ++ncand;
          break;
        }
      }
    }
  }
  return ncand <= 1;  // only ref itself can win anywhere in the box
}

// One level: one thread per group, the next group's summary requested while the current one is
// worked on.  The better choice while every thread has only a few groups (the two-level walk
// below is a chain of dependent rounds: super-group test, then its failed groups).
template <typename LabT, bool kPrivate>
__device__ __forceinline__ void classify_groups_flat(const GroupSummary* __restrict__ gsum, int n_groups,
                                                LabT* labels, int* glabel, int* worklist, int* work_count,
                                                const float4* __restrict__ s_fast, int k, float margin,
                                                bool first_iter, unsigned long long* s_acc, int* s_list,
                                                const unsigned char* s_bkt, unsigned int& n_chg, bool settle,
                                                float4 a, float4 b, float4 c, int prev) {
  // a, b, c, prev: summary and previous label of this thread's FIRST group (block * kThreads + tid),
  // requested by the caller before it waited for the centroid table
  const int tid = threadIdx.x, lane = tid & 31;
  int* w_list = s_list + (tid >> 5) * (kClassifyList / (kThreads / 32));  // this warp's slice
  int w_count = 0;                                                         // warp-uniform
  const int span = (int)gridDim.x * kThreads;
  int g = (int)blockIdx.x * kThreads + tid;
  for (int base = (int)blockIdx.x * kThreads; base < n_groups; base += span) {  // CTA-uniform trip count
    const bool valid = g < n_groups;
    int label = -1;  // settled label, or -1: needs the per-point pass
    const int q[3] = {__float_as_int(b.z), __float_as_int(b.w), __float_as_int(c.x)};
    if (settle && valid && __float_as_int(c.y) == kGroup && (first_iter || prev >= 0)) {
      const float lo0 = a.x, lo1 = a.y, lo2 = a.z, hi0 = a.w, hi1 = b.x, hi2 = b.y;
      const int ref = prev >= 0 ? prev : nearest_to_box_centre(s_fast, k, lo0, lo1, lo2, hi0, hi1, hi2);
      if (box_owned_by(s_fast, k, s_bkt, ref, margin, lo0, lo1, lo2, hi0, hi1, hi2)) label = ref;
    }
    if (label >= 0 && first_iter) {  // later iterations: label == prev, nothing to write
      n_chg += kGroup;
      uint4* lp = reinterpret_cast<uint4*>(labels + (size_t)g * kGroup);
      constexpr int kVec = kGroup * (int)sizeof(LabT) / 16;
      const unsigned int fillw = sizeof(LabT) == 1 ? (unsigned int)label * 0x01010101u : (unsigned int)label * 0x00010001u;
#pragma unroll
      for (int v = 0; v < kVec; ++v) lp[v] = make_uint4(fillw, fillw, fillw, fillw);
      glabel[g] = label;
    }
    const int g_now = g;
    // next group of this thread: its summary loads overlap the bookkeeping below
    g += span;
    if (g < n_groups) {
      const float4* src = reinterpret_cast<const float4*>(gsum + g);
      a = __ldg(src); b = __ldg(src + 1); c = __ldg(src + 2);
      prev = first_iter ? -1 : glabel[g];
    }
    // cached sums, one round per distinct label in the warp (usually one)
    unsigned int todo = __ballot_sync(0xffffffffu, label >= 0);
    while (todo) {
      const int L = __shfl_sync(0xffffffffu, label, __ffs(todo) - 1);
      const bool hit = label == L;
      long long sum[3];
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        // 32 groups x 2^29 overflows 32 bits: reduce the two halves of q separately
        const int hi = __reduce_add_sync(0xffffffffu, hit ? (q[d] >> 15) : 0);
        const int lo = __reduce_add_sync(0xffffffffu, hit ? (q[d] & 0x7fff) : 0);
        sum[d] = ((long long)hi << 15) + (long long)lo;
      }
      const unsigned int hits = __ballot_sync(0xffffffffu, hit);
      // the warp's private slice when there is one (plain read-modify-write): 64-bit
      // shared-memory atomics are compare-and-swap loops and collapse under contention
      if (lane == 0) acc_add<kPrivate>(s_acc, L, sum[0], sum[1], sum[2], (unsigned int)__popc(hits) * kGroup);
      todo &= ~hits;
    }
    // the rest goes to the per-point pass: every warp collects its groups in its own slice of
    // shared memory and hands them to the global worklist with one atomic per flush (not one
    // per trip: the round trip of a global atomic would dominate this pass) -- no CTA barrier
    const unsigned int heavy = __ballot_sync(0xffffffffu, valid && label < 0);
    if (valid && label < 0) w_list[w_count + __popc(heavy & ((1u << lane) - 1u))] = g_now;
    w_count += __popc(heavy);
    const bool last_trip = base + span >= n_groups;
    if (last_trip || w_count + 32 > kClassifyList / (kThreads / 32)) {  // warp-uniform
      __syncwarp();
      int dst = 0;
      if (lane == 0 && w_count) dst = atomicAdd(work_count, w_count);
      dst = __shfl_sync(0xffffffffu, dst, 0);
      for (int i = lane; i < w_count; i += 32) worklist[dst + i] = w_list[i];
      __syncwarp();
      w_count = 0;
    }
  }
}

// Two levels: super-groups first, groups only where a super-group fails.  Pays once a thread
// has many groups to look at (large clouds).
template <typename LabT, bool kPrivate>
__device__ __forceinline__ void classify_groups_two_level(const GroupSummary* __restrict__ gsum,
                                                const SuperSummary* __restrict__ ssum, int n_groups,
                                                LabT* labels, int* glabel, int* worklist, int* work_count,
                                                const float4* __restrict__ s_fast, int k, float margin,
                                                bool first_iter, unsigned long long* s_acc, int* s_list,
                                                const unsigned char* s_bkt, unsigned int& n_chg, bool settle) {
  const int tid = threadIdx.x, lane = tid & 31;
  int* w_list = s_list + (tid >> 5) * (kClassifyList / (kThreads / 32));  // this warp's slice
  int w_count = 0;                                                         // warp-uniform
  constexpr int kVec = kGroup * (int)sizeof(LabT) / 16;                    // 16-byte words of a group's labels

  // hands the staged worklist entries of this warp to the global list (one atomic per flush, not
  // one per round: the round trip of a global atomic would dominate this pass) -- no CTA barrier
  auto flush = [&]() {
    __syncwarp();
    int dst = 0;
    if (lane == 0 && w_count) dst = atomicAdd(work_count, w_count);
    dst = __shfl_sync(0xffffffffu, dst, 0);
    for (int i = lane; i < w_count; i += 32) worklist[dst + i] = w_list[i];
    __syncwarp();
    w_count = 0;
  };

  // One group per lane (warp-synchronous): test it against the label it was settled with, add the
  // cached sums of the settled ones, stage the others for the per-point pass.
  auto group_round = [&](int g, bool valid) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a, c = a;
    int prev = -1;
    if (valid) {
      const float4* src = reinterpret_cast<const float4*>(gsum + g);
      a = __ldg(src); b = __ldg(src + 1); c = __ldg(src + 2);
      prev = first_iter ? -1 : glabel[g];
    }
    int label = -1;  // settled label, or -1: needs the per-point pass
    const int q[3] = {__float_as_int(b.z), __float_as_int(b.w), __float_as_int(c.x)};
    if (settle && valid && __float_as_int(c.y) == kGroup && (first_iter || prev >= 0)) {
      const int ref = prev >= 0 ? prev : nearest_to_box_centre(s_fast, k, a.x, a.y, a.z, a.w, b.x, b.y);
      if (box_owned_by(s_fast, k, s_bkt, ref, margin, a.x, a.y, a.z, a.w, b.x, b.y)) label = ref;
    }
    if (label >= 0 && first_iter) {  // later iterations: label == prev, nothing to write
      n_chg += kGroup;
      uint4* lp = reinterpret_cast<uint4*>(labels + (size_t)g * kGroup);
      const unsigned int fillw = sizeof(LabT) == 1 ? (unsigned int)label * 0x01010101u : (unsigned int)label * 0x00010001u;
#pragma unroll
      for (int v = 0; v < kVec; ++v) lp[v] = make_uint4(fillw, fillw, fillw, fillw);
      glabel[g] = label;
    }
    // cached sums, one round per distinct label in the warp (usually one)
    unsigned int todo = __ballot_sync(0xffffffffu, label >= 0);
    while (todo) {
      const int L = __shfl_sync(0xffffffffu, label, __ffs(todo) - 1);
      const bool hit = label == L;
      long long sum[3];
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        // 32 groups x 2^29 overflows 32 bits: reduce the two halves of q separately
        const int hi = __reduce_add_sync(0xffffffffu, hit ? (q[d] >> 15) : 0);
        const int lo = __reduce_add_sync(0xffffffffu, hit ? (q[d] & 0x7fff) : 0);
        sum[d] = ((long long)hi << 15) + (long long)lo;
      }
      const unsigned int hits = __ballot_sync(0xffffffffu, hit);
      // the warp's private slice when there is one (plain read-modify-write): 64-bit
      // shared-memory atomics are compare-and-swap loops and collapse under contention
      if (lane == 0) acc_add<kPrivate>(s_acc, L, sum[0], sum[1], sum[2], (unsigned int)__popc(hits) * kGroup);
      todo &= ~hits;
    }
    const unsigned int heavy = __ballot_sync(0xffffffffu, valid && label < 0);
    if (valid && label < 0) w_list[w_count + __popc(heavy & ((1u << lane) - 1u))] = g;
    w_count += __popc(heavy);
    if (w_count + 32 > kClassifyList / (kThreads / 32)) flush();  // warp-uniform
  };

  const int n_super = (n_groups + kSuper - 1) / kSuper;
  const int span = (int)gridDim.x * kThreads;
  for (int sbase = (int)blockIdx.x * kThreads; sbase < n_super; sbase += span) {  // CTA-uniform trip count
    // ---- one SUPER-group per lane ------------------------------------------------------------
    const int sg = sbase + tid;
    bool fail = sg < n_super;  // its groups have to be looked at one by one
    int label = -1;
    long long sq[3] = {0, 0, 0};
    if (settle && fail) {
      const float4* src = reinterpret_cast<const float4*>(ssum + sg);
      const float4 a = __ldg(src), b = __ldg(src + 1);  // lo[3] hi[0] | hi[1] hi[2] n pad
      if (__float_as_int(b.z) == kSuper * kGroup) {
        int ref = -1;
        if (first_iter) {
          ref = nearest_to_box_centre(s_fast, k, a.x, a.y, a.z, a.w, b.x, b.y);
        } else {
          // settled as a whole only if all its groups were settled with one label
          const int4* gl = reinterpret_cast<const int4*>(glabel + (size_t)sg * kSuper);
          const int4 u = gl[0], v = gl[1];
          static_assert(kSuper == 8, "two int4 of group labels per super-group");
          const bool same = u.x == u.y && u.x == u.z && u.x == u.w && u.x == v.x && u.x == v.y && u.x == v.z && u.x == v.w;
          ref = same ? u.x : -1;
        }
        if (ref >= 0 && box_owned_by(s_fast, k, s_bkt, ref, margin, a.x, a.y, a.z, a.w, b.x, b.y)) {
          label = ref;
          fail = false;
          const longlong2 q01 = *reinterpret_cast<const longlong2*>(src + 2);
          sq[0] = q01.x; sq[1] = q01.y;
          sq[2] = *reinterpret_cast<const long long*>(src + 3);
        }
      }
    }
    if (label >= 0 && first_iter) {
      n_chg += kSuper * kGroup;
      uint4* lp = reinterpret_cast<uint4*>(labels + (size_t)sg * kSuper * kGroup);
      const unsigned int fillw = sizeof(LabT) == 1 ? (unsigned int)label * 0x01010101u : (unsigned int)label * 0x00010001u;
      for (int v = 0; v < kSuper * kVec; ++v) lp[v] = make_uint4(fillw, fillw, fillw, fillw);
      int4* gl = reinterpret_cast<int4*>(glabel + (size_t)sg * kSuper);
      gl[0] = make_int4(label, label, label, label);
      gl[1] = make_int4(label, label, label, label);
    }
    // cached sums of the settled super-groups, one round per distinct label in the warp
    unsigned int todo = __ballot_sync(0xffffffffu, label >= 0);
    while (todo) {
      const int L = __shfl_sync(0xffffffffu, label, __ffs(todo) - 1);
      const bool hit = label == L;
      long long sum[3];
#pragma unroll
      for (int d = 0; d < 3; ++d) {
        // |q| < 2^32 per super-group, 32 of them: the two halves are reduced separately
        const int hi = __reduce_add_sync(0xffffffffu, hit ? (int)(sq[d] >> 16) : 0);
        const int lo = __reduce_add_sync(0xffffffffu, hit ? (int)(sq[d] & 0xffff) : 0);
        sum[d] = ((long long)hi << 16) + (long long)lo;
      }
      const unsigned int hits = __ballot_sync(0xffffffffu, hit);
      if (lane == 0) acc_add<kPrivate>(s_acc, L, sum[0], sum[1], sum[2], (unsigned int)__popc(hits) * (kSuper * kGroup));
      todo &= ~hits;
    }
    // ---- the groups of the super-groups that failed: four super-groups (32 groups) per round ----
    unsigned int fm = __ballot_sync(0xffffffffu, fail);
    const int wbase = sbase + (tid & ~31);  // first super-group of this warp
    while (fm) {                            // warp-uniform
      unsigned int m = fm;
      for (int i = 0; i < (lane >> 3); ++i) m &= m - 1u;  // drop the lane / 8 lowest set bits
      const int sl = m ? __ffs(m) - 1 : -1;
      const int g = sl >= 0 ? (wbase + sl) * kSuper + (lane & (kSuper - 1)) : n_groups;
      group_round(g, g < n_groups);
#pragma unroll
      for (int i = 0; i < 4; ++i) fm &= fm - 1u;  // (x & (x - 1) of 0 is 0)
    }
  }
  flush();
}

// Grid-wide barrier of a cooperatively launched (fully resident) grid: a monotonically
// increasing arrival counter, one generation per use.
__device__ __forceinline__ void grid_barrier(unsigned int* counter, int* timeout_flag) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    const unsigned int arrived = atomicAdd(counter, 1u) + 1u;
    const unsigned int target = (arrived + gridDim.x - 1u) / gridDim.x * gridDim.x;
    // bounded wait (about 4 s): the launch is cooperative, so every CTA is resident and this
    // never triggers; if it ever did, a flagged wrong result beats a hung GPU
    const long long t0 = clock64();
    while ((int)(*reinterpret_cast<volatile unsigned int*>(counter) - target) < 0) {
      if (clock64() - t0 > (8ll << 30)) {
        *timeout_flag = 1;
        break;
      }
    }
    __threadfence();
  }
  __syncthreads();
}

#ifndef MDKM_FINAL_CTAS0
#define MDKM_FINAL_CTAS0 3
#endif
struct FinalParams {
  const float* pts;           // resident cloud, reference point order
  long long n;
  int* labels_out;            // int32[n] or nullptr
  const unsigned char* table;
  double* partials;           // [gridDim.x] inertia partials
  unsigned int* ticket;
  DevStatus* st;
  FrameF f;
  int k, kpad;
  int split_rows;             // 1: raster-ordered cloud (row-major runs of pixels)
  // the end of a fit, enqueued right behind its last batch of iterations:
  int skip_paused;            // 1: do nothing but publish the status when it says paused && !done
  DevStatus* status_host;     // or nullptr: the last CTA copies the status here (device-visible host memory)
  double* centroids_host;     // or nullptr: the last CTA writes the k x 3 centroids (original coordinates) here
  double origin[3];           // Frame::origin, for centroids_host
  // cluster map (lloyd_final_kernel<kChunks, true>): label + 1 at the pixel of every point, local
  // pixel (day - map_day0) * map_HW + y * map_W + x - (map_pix_begin - map_day0 * map_HW)
  void* map_out;              // uint8 / uint16 per pixel of the range of the last unprojection
  int map_elem;               // 1 or 2 bytes
  int map_W;
  long long map_pix_begin;    // global index of the range's first pixel
  long long map_HW;
  long long map_day0;         // day of map_pix_begin
  const long long* map_seg;   // [map_nseg + 1] point offsets of the days of the range (device; also
  int map_nseg;               // read by the statistics below)
  // per-(day, cluster) statistics (lloyd_final_kernel<kChunks, kMap, true>): every point adds
  // (qx, qy, qz, 1) to the four int64 words of slot (stats_day0 + day) * k + label
  unsigned long long* stats_acc;  // [slots * 4], cleared by the host
  long long stats_day0;           // global day of segment 0 of the cloud
  int stats_slots;                // days of the stack * k
  int stats_smem_off;             // > 0: per-warp copies of the slots at this byte offset of the dynamic shared
                                  // memory, flushed once per CTA at the end; 0: points go to stats_acc directly
};

// Day of this lane's points in the cluster map: segment `day` holds the points before `next`,
// and its pixel (0, 0) is element `base` of the map.  A warp walks its groups in point order, so
// the cursor only moves forward.
struct MapCursor {
  int day;
  long long next;
  long long base;
};

// the cursor of point i: the last segment that starts at or before i (empty days are skipped)
__device__ __forceinline__ MapCursor map_cursor(const FinalParams& p, long long i) {
  int lo = 0, hi = p.map_nseg;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(p.map_seg + mid) <= i) lo = mid; else hi = mid;
  }
  return MapCursor{lo, __ldg(p.map_seg + lo + 1), (long long)lo * p.map_HW - (p.map_pix_begin - p.map_day0 * p.map_HW)};
}

// exact pixel coordinate (an integer in [0, 2^23), mdkm_bind_cluster_map checks H and W) -> int,
// with one FADD instead of a float-to-int conversion
__device__ __forceinline__ int pixel_index(float v) { return __float_as_int(v + 8388608.0f) - 0x4B000000; }

// Copies the status block into device-visible host memory (one thread).  L2 reads: other CTAs
// updated it with atomics.
__device__ __forceinline__ void publish_status(const DevStatus* st, DevStatus* dst) {
  static_assert(sizeof(DevStatus) % 8 == 0, "status copied in 8-byte words");
  const unsigned long long* s = reinterpret_cast<const unsigned long long*>(st);
  unsigned long long* d = reinterpret_cast<unsigned long long*>(dst);
#pragma unroll 4
  for (int i = 0; i < (int)(sizeof(DevStatus) / 8); ++i) d[i] = __ldcg(s + i);
  __threadfence_system();
}

// ---------------------------------------------------------------------------------------
// Assignment of one warp-group.  xc/yc/zc: centred FP32 coordinates of this lane's 4 points;
// orig_*: this lane's four ORIGINAL coordinates (shared-memory stage or registers), read only
// by the FP64 refine.  s_fast: expanded rows (-2c', ||c'||^2) padded with (0,0,0,+inf) rows to
// a multiple of 32.  kChunks = rows/32 when known at compile time (straight-line code),
// 0 = run-time loop.  Warp-synchronous: all 32 lanes must call it.
//
// Pruning: take the centroid i nearest to the centre of the group's bounding box; centroid j
// stays a candidate only if it can beat i somewhere in the box (min_gap_over_box <= margin).
// The true nearest centroid of every point, and every centroid within the FP32 error band of
// it, beats-or-ties i at that point, so it is a candidate: the result equals brute force.
// Returns the number of candidates; the labels of this lane's points are in lab[].
// count_mask: bit e clear = point e of this lane is a stand-in (see lloyd_final_kernel) and is
// left out of the n_refined statistic.
// ---------------------------------------------------------------------------------------
template <int kChunks>
__device__ __forceinline__ int assign_group(const float (&xc)[4], const float (&yc)[4], const float (&zc)[4],
                                            const float* orig_x, const float* orig_y, const float* orig_z,
                                            const FrameF& f, const float4* __restrict__ s_fast,
                                            const double4* __restrict__ c64, int k, int kp32, float thresh,
                                            int lane, int (&lab)[4], unsigned int& n_refined,
                                            unsigned int count_mask = 0xfu) {
  // bounding box of the group (FMNMX3 + CREDUX.F32)
  const float bx0 = redux_min_f32(fminf(fminf(xc[0], xc[1]), fminf(xc[2], xc[3])));
  const float bx1 = redux_max_f32(fmaxf(fmaxf(xc[0], xc[1]), fmaxf(xc[2], xc[3])));
  const float by0 = redux_min_f32(fminf(fminf(yc[0], yc[1]), fminf(yc[2], yc[3])));
  const float by1 = redux_max_f32(fmaxf(fmaxf(yc[0], yc[1]), fmaxf(yc[2], yc[3])));
  const float bz0 = redux_min_f32(fminf(fminf(zc[0], zc[1]), fminf(zc[2], zc[3])));
  const float bz1 = redux_max_f32(fmaxf(fmaxf(zc[0], zc[1]), fmaxf(zc[2], zc[3])));
  const float mx = 0.5f * (bx0 + bx1), my = 0.5f * (by0 + by1), mz = 0.5f * (bz0 + bz1);
  // margin: 4*thresh = 8E covers the FP32 rounding of the gap expression and of the fast
  // distances themselves (E bounds the error of one fast distance, DESIGN.md "Exactness")
  const float margin = 4.0f * thresh;

  constexpr int kM = kChunks > 0 ? kChunks : 1;
  unsigned int masks[kM];
  int ncand = 0, first = 0;
  float4 ref;
  if (kChunks > 0) {
    float4 row[kM];
    float dc[kM];
    float dmin = __int_as_float(0x7f800000);
#pragma unroll
    for (int c = 0; c < kM; ++c) {
      row[c] = s_fast[c * 32 + lane];
      dc[c] = fmaf(mx, row[c].x, fmaf(my, row[c].y, fmaf(mz, row[c].z, row[c].w)));
      dmin = fminf(dmin, dc[c]);
    }
    dmin = redux_min_f32(dmin);
    int iref = 0;
#pragma unroll
    for (int c = kM - 1; c >= 0; --c) {
      const unsigned int m = __ballot_sync(0xffffffffu, dc[c] == dmin);
      if (m) iref = c * 32 + __ffs(m) - 1;
    }
    ref = s_fast[iref];
#pragma unroll
    for (int c = kM - 1; c >= 0; --c) {
      const float gap = min_gap_over_box(row[c], ref, bx0, bx1, by0, by1, bz0, bz1);
      masks[c] = __ballot_sync(0xffffffffu, gap <= margin);
      ncand += __popc(masks[c]);
      if (masks[c]) first = c * 32 + __ffs(masks[c]) - 1;
    }
  } else {
    float dmin = __int_as_float(0x7f800000);
    for (int j = lane; j < kp32; j += 32) {
      const float4 r = s_fast[j];
      dmin = fminf(dmin, fmaf(mx, r.x, fmaf(my, r.y, fmaf(mz, r.z, r.w))));
    }
    dmin = redux_min_f32(dmin);
    int iref = -1;
    for (int base = 0; base < kp32 && iref < 0; base += 32) {
      const float4 r = s_fast[base + lane];
      const unsigned int m =
          __ballot_sync(0xffffffffu, fmaf(mx, r.x, fmaf(my, r.y, fmaf(mz, r.z, r.w))) == dmin);
      if (m) iref = base + __ffs(m) - 1;
    }
    ref = s_fast[iref < 0 ? 0 : iref];
    for (int base = 0; base < kp32; base += 32) {
      const float gap = min_gap_over_box(s_fast[base + lane], ref, bx0, bx1, by0, by1, bz0, bz1);
      const unsigned int m = __ballot_sync(0xffffffffu, gap <= margin);
      if (ncand == 0 && m) first = base + __ffs(m) - 1;
      ncand += __popc(m);
    }
    masks[0] = 0;
  }
  if (ncand <= 1) {  // interior group: one possible owner, no distance evaluation at all
#pragma unroll
    for (int e = 0; e < 4; ++e) lab[e] = first;
    return ncand;
  }
  // evaluate the candidates in ascending index (strict '<' keeps the lowest index on ties,
  // pyx:205-213), tracking best and second best per point
  float best[4], second[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    best[e] = __int_as_float(0x7f800000);
    second[e] = __int_as_float(0x7f800000);
    lab[e] = 0;
  }
  auto eval = [&](int j) {
    const float4 cf = s_fast[j];  // LDS.128, warp broadcast
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float d = fmaf(xc[e], cf.x, fmaf(yc[e], cf.y, fmaf(zc[e], cf.z, cf.w)));
      const bool lt = d < best[e];
      second[e] = fminf(second[e], fmaxf(d, best[e]));
      best[e] = fminf(best[e], d);
      lab[e] = lt ? j : lab[e];
    }
  };
  if (kChunks > 0) {
#pragma unroll
    for (int c = 0; c < kM; ++c) {
      unsigned int m = masks[c];
      while (m) {
        eval(c * 32 + __ffs(m) - 1);
        m &= m - 1;
      }
    }
  } else {
    for (int base = 0; base < kp32; base += 32) {
      const float gap = min_gap_over_box(s_fast[base + lane], ref, bx0, bx1, by0, by1, bz0, bz1);
      unsigned int m = __ballot_sync(0xffffffffu, gap <= margin);
      while (m) {
        eval(base + __ffs(m) - 1);
        m &= m - 1;
      }
    }
  }
  // FP64 refine of the points the FP32 pass cannot decide (rare; see file header), from the
  // ORIGINAL coordinates, so no FP32 rounding of x - origin enters.  Only the group's
  // candidates can be the exact nearest (see above), so only they are re-evaluated, and the
  // warp walks them together: the cost does not grow with k.
  bool ambig[4];
  bool amb = false;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    ambig[e] = !(second[e] - best[e] > thresh);
    amb |= ambig[e];
  }
  if (__any_sync(0xffffffffu, amb)) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (!__any_sync(0xffffffffu, ambig[e])) continue;  // warp-uniform
      const double X = (double)orig_x[e] - (double)f.ox;
      const double Y = (double)orig_y[e] - (double)f.oy;
      const double Z = (double)orig_z[e] - (double)f.oz;
      double bd = 1.0 / 0.0;
      int bi = 0;
      auto eval64 = [&](int j) {  // ascending j, strict '<': lowest index on exact ties
        const double4 c = ld_c64(&c64[j]);
        const double d = fma(-2.0, fma(X, c.x, fma(Y, c.y, Z * c.z)), c.w);
        if (d < bd) {
          bd = d;
          bi = j;
        }
      };
      if (kChunks > 0) {
#pragma unroll
        for (int c = 0; c < kM; ++c) {
          unsigned int m = masks[c];
          while (m) {
            eval64(c * 32 + __ffs(m) - 1);
            m &= m - 1;
          }
        }
      } else {
        for (int base = 0; base < kp32; base += 32) {
          const float gap = min_gap_over_box(s_fast[base + lane], ref, bx0, bx1, by0, by1, bz0, bz1);
          unsigned int m = __ballot_sync(0xffffffffu, gap <= margin);
          while (m) {
            eval64(base + __ffs(m) - 1);
            m &= m - 1;
          }
        }
      }
      if (ambig[e]) {
        lab[e] = bi;
        n_refined += (count_mask >> e) & 1u;  // (stand-in points of a split group are not counted)
      }
    }
  }
  return ncand;
}

// ---------------------------------------------------------------------------------------
// Assignment of one warp-group when the centroids are bucketed (many centroids): the
// candidates are collected from the buckets the group's box, grown by its reach, touches --
// a handful of centroids instead of three passes over all k.  `ref_hint` is any centroid index
// (the label a point of the group had before: a good reference) or -1 to search the nearest
// to the box centre.  Candidates come in bucket order, so ties are broken on the index
// explicitly (lowest index wins, pyx:205-213).  `s_cand`: this warp's kCandCap slots.
// Returns the number of candidates, or -1 when there are more than kCandCap (the caller then
// takes the generic path).  Warp-synchronous.
// ---------------------------------------------------------------------------------------
constexpr int kCandCap = 64;

__device__ __forceinline__ int assign_group_bucketed(const float (&xc)[4], const float (&yc)[4], const float (&zc)[4],
                                                     const float* orig_x, const float* orig_y, const float* orig_z,
                                                     const FrameF& f, const float4* __restrict__ s_fast,
                                                     const double4* __restrict__ c64, const unsigned char* s_bkt,
                                                     int k, int kp32, float thresh, int ref_hint,
                                                     unsigned short* s_cand, int lane, int (&lab)[4],
                                                     unsigned int& n_refined, unsigned int count_mask = 0xfu) {
  const float bx0 = redux_min_f32(fminf(fminf(xc[0], xc[1]), fminf(xc[2], xc[3])));
  const float bx1 = redux_max_f32(fmaxf(fmaxf(xc[0], xc[1]), fmaxf(xc[2], xc[3])));
  const float by0 = redux_min_f32(fminf(fminf(yc[0], yc[1]), fminf(yc[2], yc[3])));
  const float by1 = redux_max_f32(fmaxf(fmaxf(yc[0], yc[1]), fmaxf(yc[2], yc[3])));
  const float bz0 = redux_min_f32(fminf(fminf(zc[0], zc[1]), fminf(zc[2], zc[3])));
  const float bz1 = redux_max_f32(fmaxf(fmaxf(zc[0], zc[1]), fmaxf(zc[2], zc[3])));
  const float margin = 4.0f * thresh;
  int iref = ref_hint;
  if (iref < 0) {  // nearest centroid to the box centre (first iteration, final pass)
    const float mx = 0.5f * (bx0 + bx1), my = 0.5f * (by0 + by1), mz = 0.5f * (bz0 + bz1);
    float dmin = __int_as_float(0x7f800000);
    for (int j = lane; j < kp32; j += 32) {
      const float4 r = s_fast[j];
      dmin = fminf(dmin, fmaf(mx, r.x, fmaf(my, r.y, fmaf(mz, r.z, r.w))));
    }
    dmin = redux_min_f32(dmin);
    for (int base = 0; base < kp32 && iref < 0; base += 32) {
      const float4 r = s_fast[base + lane];
      const unsigned int m =
          __ballot_sync(0xffffffffu, fmaf(mx, r.x, fmaf(my, r.y, fmaf(mz, r.z, r.w))) == dmin);
      if (m) iref = base + __ffs(m) - 1;
    }
    if (iref < 0) iref = 0;
  }
  const float4 ref = s_fast[iref];
  const BucketHdr hdr = *reinterpret_cast<const BucketHdr*>(s_bkt);
  const int g = bucket_g(k);
  const unsigned short* start = reinterpret_cast<const unsigned short*>(s_bkt + sizeof(BucketHdr));
  const unsigned short* perm = start + g * g + 1;
  const float cx = -0.5f * ref.x, cy = -0.5f * ref.y, cz = -0.5f * ref.z;
  const float dx = fmaxf(fabsf(bx0 - cx), fabsf(bx1 - cx)), dy = fmaxf(fabsf(by0 - cy), fabsf(by1 - cy)),
              dz = fmaxf(fabsf(bz0 - cz), fabsf(bz1 - cz));
  const float reach = sqrtf(fmaf(dx, dx, fmaf(dy, dy, dz * dz)) + 2.0f * margin) * 1.0001f + 1e-3f / hdr.inv_x;
  const int cx0 = bucket_coord(bx0 - reach, hdr.hx, hdr.inv_x, g), cx1 = bucket_coord(bx1 + reach, hdr.hx, hdr.inv_x, g);
  const int cy0 = bucket_coord(by0 - reach, hdr.hy, hdr.inv_y, g), cy1 = bucket_coord(by1 + reach, hdr.hy, hdr.inv_y, g);
  int ncand = 0;
  for (int cyi = cy0; cyi <= cy1; ++cyi) {
    const int i1 = start[cyi * g + cx1 + 1];
    for (int base = start[cyi * g + cx0]; base < i1; base += 32) {
      const int i = base + lane;
      const int j = i < i1 ? (int)perm[i] : -1;
      const bool pass = j >= 0 && min_gap_over_box(s_fast[j < 0 ? 0 : j], ref, bx0, bx1, by0, by1, bz0, bz1) <= margin;
      const unsigned int m = __ballot_sync(0xffffffffu, pass);
      if (ncand + __popc(m) > kCandCap) return -1;  // warp-uniform
      if (pass) s_cand[ncand + __popc(m & ((1u << lane) - 1u))] = (unsigned short)j;
      ncand += __popc(m);
    }
  }
  __syncwarp();
  if (ncand <= 1) {  // one possible owner (the reference is always a candidate)
    const int only = ncand == 1 ? (int)s_cand[0] : iref;
#pragma unroll
    for (int e = 0; e < 4; ++e) lab[e] = only;
    return ncand;
  }
  float best[4], second[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    best[e] = __int_as_float(0x7f800000);
    second[e] = __int_as_float(0x7f800000);
    lab[e] = 0x7fffffff;
  }
  for (int c = 0; c < ncand; ++c) {
    const int j = s_cand[c];
    const float4 cf = s_fast[j];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float d = fmaf(xc[e], cf.x, fmaf(yc[e], cf.y, fmaf(zc[e], cf.z, cf.w)));
      const bool lt = d < best[e] || (d == best[e] && j < lab[e]);
      second[e] = fminf(second[e], fmaxf(d, best[e]));
      best[e] = fminf(best[e], d);
      lab[e] = lt ? j : lab[e];
    }
  }
  bool ambig[4];
  bool amb = false;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    ambig[e] = !(second[e] - best[e] > thresh);
    amb |= ambig[e];
  }
  if (__any_sync(0xffffffffu, amb)) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (!__any_sync(0xffffffffu, ambig[e])) continue;  // warp-uniform
      const double X = (double)orig_x[e] - (double)f.ox;
      const double Y = (double)orig_y[e] - (double)f.oy;
      const double Z = (double)orig_z[e] - (double)f.oz;
      double bd = 1.0 / 0.0;
      int bi = 0x7fffffff;
      for (int c = 0; c < ncand; ++c) {
        const int j = s_cand[c];
        const double4 cc = ld_c64(&c64[j]);
        const double d = fma(-2.0, fma(X, cc.x, fma(Y, cc.y, Z * cc.z)), cc.w);
        if (d < bd || (d == bd && j < bi)) {
          bd = d;
          bi = j;
        }
      }
      if (ambig[e]) {
        lab[e] = bi;
        n_refined += (count_mask >> e) & 1u;  // (stand-in points of a split group are not counted)
      }
    }
  }
  return ncand;
}

template <typename LabT>
struct LabPack;
template <>
struct LabPack<unsigned char> {
  using V = unsigned int;  // 4 labels
  static constexpr int kBytes = 4;
  static __device__ __forceinline__ V load(const void* p) { return *reinterpret_cast<const unsigned int*>(p); }
  static __device__ __forceinline__ V pack(const int (&l)[4]) {
    return (unsigned)l[0] | ((unsigned)l[1] << 8) | ((unsigned)l[2] << 16) | ((unsigned)l[3] << 24);
  }
  static __device__ __forceinline__ void store(unsigned char* p, V v) {
    *reinterpret_cast<unsigned int*>(p) = v;
  }
  static __device__ __forceinline__ bool same(V a, V b) { return a == b; }
  static __device__ __forceinline__ int get(V v, int e) { return (v >> (8 * e)) & 0xff; }
};
template <>
struct LabPack<unsigned short> {
  using V = uint2;
  static constexpr int kBytes = 8;
  static __device__ __forceinline__ V load(const void* p) { return *reinterpret_cast<const uint2*>(p); }
  static __device__ __forceinline__ V pack(const int (&l)[4]) {
    uint2 v;
    v.x = (unsigned)l[0] | ((unsigned)l[1] << 16);
    v.y = (unsigned)l[2] | ((unsigned)l[3] << 16);
    return v;
  }
  static __device__ __forceinline__ void store(unsigned short* p, V v) { *reinterpret_cast<uint2*>(p) = v; }
  static __device__ __forceinline__ bool same(V a, V b) { return a.x == b.x && a.y == b.y; }
  static __device__ __forceinline__ int get(V v, int e) {
    const unsigned w = (e < 2) ? v.x : v.y;
    return (w >> (16 * (e & 1))) & 0xffff;
  }
};

// Adds (sx,sy,sz,cnt) to row `lab` of an accumulator slice.  kPrivate: the slice belongs to
// this warp and only lane 0 ever touches it -> plain read-modify-write; otherwise the slice is
// shared by the CTA -> shared-memory atomics.
template <bool kPrivate>
__device__ __forceinline__ void acc_add(unsigned long long* s_acc, int lab, long long sx, long long sy,
                                        long long sz, unsigned int cnt) {
  unsigned long long* row = s_acc + lab * 4;
  if (kPrivate) {
    ulonglong2 a = *reinterpret_cast<ulonglong2*>(row);
    ulonglong2 b = *reinterpret_cast<ulonglong2*>(row + 2);
    a.x += (unsigned long long)sx;
    a.y += (unsigned long long)sy;
    b.x += (unsigned long long)sz;
    b.y += (unsigned long long)cnt;
    *reinterpret_cast<ulonglong2*>(row) = a;
    *reinterpret_cast<ulonglong2*>(row + 2) = b;
  } else {
    atomicAdd(row + 0, (unsigned long long)sx);
    atomicAdd(row + 1, (unsigned long long)sy);
    atomicAdd(row + 2, (unsigned long long)sz);
    atomicAdd(row + 3, (unsigned long long)cnt);
  }
}

// ---------------------------------------------------------------------------------------
// K2 + K3: assignment and per-cluster sums in one pass.
//
// Each warp streams its own sequence of 128-point groups through a kStages-deep ring in
// shared memory: lane 0 issues two 1-D TMA bulk copies per group (the 1536-byte xyz block
// and the previous labels) and arms the stage's mbarrier with the byte count; the warp waits
// on the barrier, works on the group from shared memory / registers, and re-arms the stage
// for the group kStages ahead.  No CTA-wide barrier inside the loop; HBM latency is covered
// by the copies in flight, not by occupancy.
// ---------------------------------------------------------------------------------------
constexpr int kStages = 3;

// All-gather + sum of the ranks' partial sums without a collective call.  Every 64-bit word travels
// as two 8-byte packets (32 bits of the value, 32 bits of the step's epoch) written with ONE store
// each straight into the peers' buffers over NVLink (peer-mapped memory): value and flag arrive
// together, so there is no separate flag, no fence and no second round trip -- a receiver polls
// the packet itself until it carries the step's epoch (the "LL" scheme of collective libraries).
// Slots are double-buffered by the epoch's parity: a rank can run at most one step ahead of the
// slowest one.  Integer sums: every rank ends with bit-identical totals.
//
// peer_send_sums: the SENDING half, run by the last CTA of a step kernel to finish (it owns the
// complete local sums); nobody waits here -- the packets fly while the kernel drains and the next
// one starts.  Thread t owns word t, t + kThreads, ...
__device__ __forceinline__ void peer_send_sums(const PeerXchg& px, const unsigned long long* acc, int n,
                                               unsigned int tag) {
  const int tid = threadIdx.x, R = px.n_ranks;
  const int par = (int)(tag & 1u);
  // packets of (parity, source rank): 2 * slot of them, 8 bytes each
  const size_t mine = ((size_t)par * R + px.rank) * (size_t)px.slot * 2;
  for (int i = tid; i < n; i += kThreads) {
    const unsigned long long v = __ldcg(acc + i);
    for (int q = 0; q < R; ++q) {
      if (q == px.rank) continue;
      unsigned long long* dst = px.data[q] + mine + 2 * (size_t)i;
      st_relaxed_sys_v2u32(dst, (unsigned int)v, tag);
      st_relaxed_sys_v2u32(dst + 1, (unsigned int)(v >> 32), tag);
    }
  }
}

// The RECEIVING half: word i of the global sums = this rank's word + the peers' packets of epoch
// `tag`.  All peers' packets of the word are requested together (2 (R - 1) independent loads in
// flight: one L2 round trip when everything has arrived); only what is still missing is asked again.
__device__ __forceinline__ unsigned long long gather_sum_word(const PeerXchg& px, const unsigned long long* acc,
                                                              int i, unsigned int tag, long long t0, bool& timed_out) {
  unsigned long long s = __ldcg(acc + i);
  const int R = px.n_ranks;
  if (R <= 1) return s;
  const int par = (int)(tag & 1u);
  uint2 lo[kMaxRanks], hi[kMaxRanks];
  const unsigned long long* base = px.data[px.rank] + (size_t)par * R * (size_t)px.slot * 2 + 2 * (size_t)i;
  unsigned int missing = 0;
#pragma unroll
  for (int q = 0; q < kMaxRanks; ++q)
    if (q < R && q != px.rank) {
      const unsigned long long* src = base + (size_t)q * (size_t)px.slot * 2;
      lo[q] = ld_relaxed_sys_v2u32(src);
      hi[q] = ld_relaxed_sys_v2u32(src + 1);
    }
#pragma unroll
  for (int q = 0; q < kMaxRanks; ++q)
    if (q < R && q != px.rank && (lo[q].y != tag || hi[q].y != tag)) missing |= 1u << q;
  while (missing && !timed_out) {
    // bounded wait (about 4 s): a missing peer must not hang the GPU
    if (clock64() - t0 > (8ll << 30)) timed_out = true;
#pragma unroll
    for (int q = 0; q < kMaxRanks; ++q)
      if ((missing >> q) & 1u) {
        const unsigned long long* src = base + (size_t)q * (size_t)px.slot * 2;
        lo[q] = ld_relaxed_sys_v2u32(src);
        hi[q] = ld_relaxed_sys_v2u32(src + 1);
      }
#pragma unroll
    for (int q = 0; q < kMaxRanks; ++q)
      if (((missing >> q) & 1u) && lo[q].y == tag && hi[q].y == tag) missing &= ~(1u << q);
  }
#pragma unroll
  for (int q = 0; q < kMaxRanks; ++q)
    if (q < R && q != px.rank) s += (unsigned long long)lo[q].x | ((unsigned long long)hi[q].x << 32);
  return s;
}

// ---------------------------------------------------------------------------------------
// Deferred centroid update.  A fused step kernel ends as soon as its sums are in acc[seq % 3]
// (and, with several ranks, on their way to the peers): there is no last-CTA tail.  The update
// that turns those sums into the next centroid table (_k_means_common.pyx:274-311,
// _kmeans.py:721-738) runs in the PROLOGUE of the next launch, redundantly in every CTA: each
// one gathers the K x 4 sums (one L2 round trip, the same one the table load used to cost),
// computes the new rows straight into its shared-memory table and takes the same decisions
// (converged / max_iter / empty cluster) from the same integers.  CTA 0 (`writer`) additionally
// writes the new table to table[seq & 1] (the FP64 rows are read from there in pass 2, behind the
// grid barrier) and the status block.  The latency chain of an iteration loses the ticket, the
// fence and two dependent L2 round trips of the old tail, and the peers' packets travel during
// the launch boundary.
//
// Returns 0: go on with the E-step (fast rows and buckets are in shared memory, threshold in
// ds.thresh; the writer publishes ds.* after the grid barrier), 1: converged or max_iter reached
// (status written, final table in `new_table`), 2: an empty cluster needs the host (sums parked in
// acc_saved, status paused, update NOT applied).  Executed by all kThreads threads of a CTA.
// ---------------------------------------------------------------------------------------
struct DeferredShared {
  double red[5][kThreads / 32];
  unsigned long long nchg;
  unsigned long long maxcnt;  // (count << 13) | (2 * kMaxK - 1 - j): argmax, first wins
  double shift2;
  int nempty;
  int verdict;
  int iter;
  float thresh;
};

// What the writer CTA publishes once every CTA of the launch has read the status block (behind the
// grid barrier of a step kernel, or at the end of the settle kernel).
__device__ __forceinline__ void publish_update(DevStatus* st, const DeferredShared& ds) {
  st->thresh = ds.thresh;
  st->shift2 = ds.shift2;
  st->n_changed = ds.nchg;
  st->n_empty = ds.nempty;
  st->iter = ds.iter;
  st->first = 0;
}

__device__ __forceinline__ int deferred_update(const UpdateParams& u, const PeerXchg& px,
                                               const unsigned long long* acc_src, const unsigned char* old_table,
                                               unsigned char* new_table, float4* s_fast, unsigned char* s_bkt,
                                               unsigned long long* s_sums, DeferredShared& ds, bool writer, int seq) {
  DevStatus* st = u.st;
  const int tid = threadIdx.x;
  const unsigned int tag = (unsigned int)st->epoch;  // the epoch the pending E-step's packets carry
  const int was_first = st->first, iter_old = st->iter, max_iter = st->max_iter;
  const double tol = st->tol;
  if (tid == 0) {
    ds.nempty = 0;
    ds.maxcnt = 0ull;
  }
  {
    bool timed_out = false;
    const long long t0 = clock64();
    for (int i = tid; i < u.kpad * 4 + 1; i += kThreads) {
      const unsigned long long v = gather_sum_word(px, acc_src, i, tag, t0, timed_out);
      if (i < u.kpad * 4) s_sums[i] = v;
      else ds.nchg = v;
    }
    if (timed_out) st->xchg_timeout = 1;
  }
  __syncthreads();
  // empty clusters and the heaviest cluster (np.argmax: first maximum)
  int my_empty = 0;
  unsigned long long my_max = 0ull;
  for (int j = tid; j < u.k; j += kThreads) {
    const unsigned long long cnt = s_sums[j * 4 + 3];
    if (cnt == 0ull) ++my_empty;
    const unsigned long long key = (cnt << 13) | (unsigned long long)(kMaxK * 2 - 1 - j);
    my_max = key > my_max ? key : my_max;
  }
  my_empty = __reduce_add_sync(0xffffffffu, my_empty);
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long t = __shfl_down_sync(0xffffffffu, my_max, o);
    my_max = t > my_max ? t : my_max;
  }
  if ((tid & 31) == 0) {
    if (my_empty) atomicAdd(&ds.nempty, my_empty);
    atomicMax(&ds.maxcnt, my_max);
  }
  __syncthreads();
  const int n_empty = ds.nempty;
  const unsigned long long n_changed = ds.nchg;
  if (n_empty > 0 && u.allow_pause) {
    // the host sequences the relocation kernels on the parked (global) sums and re-runs the update
    if (writer) {
      for (int i = tid; i < u.kpad * 4 + 8; i += kThreads)
        u.acc_saved[i] = i < u.kpad * 4 ? s_sums[i] : (i == u.kpad * 4 ? n_changed : 0ull);
      __syncthreads();
      if (tid == 0) {
        st->n_empty = n_empty;
        __threadfence();
        st->paused = 1;
      }
    }
    return 2;
  }
  const int jmax = kMaxK * 2 - 1 - (int)(ds.maxcnt & 0x1fffull);
  const double4* old_exact = reinterpret_cast<const double4*>(old_table + exact_offset(u.kpad));
  double4* new_exact = reinterpret_cast<double4*>(new_table + exact_offset(u.kpad));
  float4* new_fast = reinterpret_cast<float4*>(new_table);
  double shift2 = 0.0, m_cn = 0.0, m_cx = 0.0, m_cy = 0.0, m_cz = 0.0;
  for (int j = tid; j < u.kpad; j += kThreads) {
    float4 fr4 = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7f800000));
    double4 ex4 = make_double4(0.0, 0.0, 0.0, 1.0 / 0.0);
    if (j < u.k) {
      const double4 old = old_exact[j];
      int row = j;
      bool raw = false;
      if (s_sums[j * 4 + 3] == 0ull) {
        // sklearn/_k_means_common.pyx:289-293: copy of the heaviest cluster's row -- which is
        // still the un-averaged sum when that row comes later in the loop.
        row = jmax;
        raw = jmax > j;
      }
      const unsigned long long ax = s_sums[row * 4 + 0], ay = s_sums[row * 4 + 1], az = s_sums[row * 4 + 2];
      const double sc = (double)s_sums[row * 4 + 3];
      const double qx = (double)(long long)ax * u.inv_scale[0];
      const double qy = (double)(long long)ay * u.inv_scale[1];
      const double qz = (double)(long long)az * u.inv_scale[2];
      double cx, cy, cz;
      if (!raw) {
        const double alpha = 1.0 / sc;  // pyx:284-287: centers *= 1/weight
        cx = qx * alpha;
        cy = qy * alpha;
        cz = qz * alpha;
      } else {
        // raw sum in sklearn's mean-centred frame, expressed in ours
        cx = qx + sc * (u.fr.origin[0] - u.mean[0]) + (u.mean[0] - u.fr.origin[0]);
        cy = qy + sc * (u.fr.origin[1] - u.mean[1]) + (u.mean[1] - u.fr.origin[1]);
        cz = qz + sc * (u.fr.origin[2] - u.mean[2]) + (u.mean[2] - u.fr.origin[2]);
      }
      const double dx = cx - old.x, dy = cy - old.y, dz = cz - old.z;
      const double sh = sqrt(dx * dx + dy * dy + dz * dz);  // _center_shift, pyx:298-311
      shift2 += sh * sh;                                     // (center_shift**2).sum()
      const double cn = cx * cx + cy * cy + cz * cz;
      ex4 = make_double4(cx, cy, cz, cn);
      fr4 = make_float4((float)(-2.0 * cx), (float)(-2.0 * cy), (float)(-2.0 * cz), (float)cn);
      m_cn = fmax(m_cn, cn);
      m_cx = fmax(m_cx, fabs(cx));
      m_cy = fmax(m_cy, fabs(cy));
      m_cz = fmax(m_cz, fabs(cz));
    }
    s_fast[j] = fr4;
    if (writer) {
      new_exact[j] = ex4;
      new_fast[j] = fr4;
    }
  }
  if (s_bkt) {
    build_centroid_buckets(s_fast, s_bkt, u.k, u.kpad, u.fr);
    if (writer) {
      __syncthreads();
      const uint4* src = reinterpret_cast<const uint4*>(s_bkt);
      uint4* dst = reinterpret_cast<uint4*>(new_table + bucket_offset(u.kpad));
      for (int i = tid; i < (int)(bucket_bytes(u.k, u.kpad) / 16); i += kThreads) dst[i] = src[i];
    }
  }
  // fixed-order reductions: shuffle tree inside the warp, warps combined in index order
  for (int o = 16; o > 0; o >>= 1) {
    shift2 += __shfl_down_sync(0xffffffffu, shift2, o);
    m_cn = fmax(m_cn, __shfl_down_sync(0xffffffffu, m_cn, o));
    m_cx = fmax(m_cx, __shfl_down_sync(0xffffffffu, m_cx, o));
    m_cy = fmax(m_cy, __shfl_down_sync(0xffffffffu, m_cy, o));
    m_cz = fmax(m_cz, __shfl_down_sync(0xffffffffu, m_cz, o));
  }
  if ((tid & 31) == 0) {
    const int w = tid >> 5;
    ds.red[0][w] = shift2; ds.red[1][w] = m_cn; ds.red[2][w] = m_cx; ds.red[3][w] = m_cy; ds.red[4][w] = m_cz;
  }
  __syncthreads();
  if (tid == 0) {
    shift2 = 0.0; m_cn = 0.0; m_cx = 0.0; m_cy = 0.0; m_cz = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) {
      shift2 += ds.red[0][w];
      m_cn = fmax(m_cn, ds.red[1][w]);
      m_cx = fmax(m_cx, ds.red[2][w]);
      m_cy = fmax(m_cy, ds.red[3][w]);
      m_cz = fmax(m_cz, ds.red[4][w]);
    }
    // FP32 error bound of the fast distances (DESIGN.md "Exactness"): u = 2^-24
    const double ue = 5.9604644775390625e-08;
    const double E = ue * (4.0 * m_cn + 10.0 * (u.fr.halfrange[0] * m_cx + u.fr.halfrange[1] * m_cy +
                                                 u.fr.halfrange[2] * m_cz));
    ds.thresh = __double2float_ru(2.0 * E * 1.001 + 1e-37);
    ds.shift2 = shift2;
    const int it = iter_old + 1;
    ds.iter = it;
    const bool strict = !was_first && n_changed == 0ull;  // _kmeans.py:721-726
    const bool done = strict || shift2 <= tol || it >= max_iter;  // _kmeans.py:729-738
    ds.verdict = done ? 1 : 0;
    if (done && writer) {
      // `done` first: a CTA that starts late leaves at once whatever else it reads
      st->done = 1;
      if (strict) st->strict = 1;
      __threadfence();
      st->thresh = ds.thresh;
      st->shift2 = shift2;
      st->n_changed = n_changed;
      st->n_empty = n_empty;
      st->iter = it;
      st->first = 0;
      st->last_seq = seq;  // (the final table sits in table[seq & 1])
      // `pending` stays as it is: a CTA of this launch that starts late and sees neither `done` nor
      // a cleared `pending` must still come to the same verdict; the settle kernel clears it
    }
  }
  __syncthreads();
  return ds.verdict;
}

// The same update for tables of at most 128 rows (the step kernels with private accumulator
// slices: every CTA runs it), ONE row per thread.  The row's sums and its old centroid are
// requested by deferred_prefetch at the very top of the kernel, together with the status words,
// so the whole prologue costs one L2 round trip; two CTA barriers (the first doubles as the
// "any empty cluster" vote).  Same arithmetic, same reduction order as deferred_update.
struct RowRegs {
  ulonglong2 a, b;          // (sum qx, sum qy), (sum qz, count) of row threadIdx.x
  double4 old;              // its centroid before the update
  unsigned long long nchg;  // changed-label count (thread kThreads - 1 only)
};

__device__ __forceinline__ void deferred_prefetch(RowRegs& r, const unsigned long long* acc_src,
                                                  const unsigned char* old_table, int k, int kpad) {
  const int tid = threadIdx.x;
  r.a = make_ulonglong2(0ull, 0ull);
  r.b = r.a;
  r.old = make_double4(0.0, 0.0, 0.0, 0.0);
  r.nchg = 0ull;
  if (tid < kpad) {
    r.a = __ldcg(reinterpret_cast<const ulonglong2*>(acc_src + tid * 4));
    r.b = __ldcg(reinterpret_cast<const ulonglong2*>(acc_src + tid * 4 + 2));
  }
  if (tid < k) {
    const double2* src = reinterpret_cast<const double2*>(old_table + exact_offset(kpad)) + 2 * tid;
    const double2 o0 = __ldcg(src), o1 = __ldcg(src + 1);
    r.old = make_double4(o0.x, o0.y, o1.x, o1.y);
  }
  if (tid == kThreads - 1) r.nchg = __ldcg(acc_src + kpad * 4);
}

// The peers' shares of all n words (epoch `tag`), spread over the CTA: a thread takes (peer, word)
// pairs, requests both packets of up to kPairs pairs at once (so the whole gather is one round trip
// through L2 when everything has arrived; only what is missing is asked again) and parks the 64-bit
// values in shared memory, stash[peer_index * n + word].  Ends with a CTA barrier.
__device__ __forceinline__ void gather_peer_words(const PeerXchg& px, int n, unsigned int tag,
                                                  unsigned long long* stash, DevStatus* st) {
  constexpr int kPairs = 4;
  const int tid = threadIdx.x, R = px.n_ranks, par = (int)(tag & 1u);
  const unsigned long long* mybuf = px.data[px.rank] + (size_t)par * R * (size_t)px.slot * 2;
  const int total = (R - 1) * n;
  const long long t0 = clock64();
  bool timed_out = false;
  for (int base = 0; base < total; base += kThreads * kPairs) {
    const unsigned long long* src[kPairs];
    uint2 lo[kPairs], hi[kPairs];
    int idx[kPairs];
#pragma unroll
    for (int u = 0; u < kPairs; ++u) {
      idx[u] = base + u * kThreads + tid;
      if (idx[u] < total) {
        const int qi = idx[u] / n, w = idx[u] - qi * n;
        const int q = qi + (qi >= px.rank ? 1 : 0);
        src[u] = mybuf + ((size_t)q * (size_t)px.slot + (size_t)w) * 2;
        lo[u] = ld_relaxed_sys_v2u32(src[u]);
        hi[u] = ld_relaxed_sys_v2u32(src[u] + 1);
      }
    }
#pragma unroll
    for (int u = 0; u < kPairs; ++u) {
      if (idx[u] < total) {
        while ((lo[u].y != tag || hi[u].y != tag) && !timed_out) {
          if (clock64() - t0 > (8ll << 30)) timed_out = true;  // bounded wait (about 4 s): a missing peer must not hang the GPU
          lo[u] = ld_relaxed_sys_v2u32(src[u]);
          hi[u] = ld_relaxed_sys_v2u32(src[u] + 1);
        }
        stash[idx[u]] = (unsigned long long)lo[u].x | ((unsigned long long)hi[u].x << 32);
      }
    }
  }
  if (timed_out) st->xchg_timeout = 1;
  __syncthreads();
}

// the status words a step kernel needs, requested together at its very top
struct StatusSnap {
  int done, paused, first, iter, max_iter;
  float thresh;
  double tol;
  unsigned long long epoch;
};
__device__ __forceinline__ StatusSnap status_snapshot(const DevStatus* st) {
  StatusSnap s;
  s.done = st->done; s.paused = st->paused; s.first = st->first; s.iter = st->iter; s.max_iter = st->max_iter;
  s.thresh = st->thresh; s.tol = st->tol; s.epoch = st->epoch;
  return s;
}

__device__ __forceinline__ int deferred_update_rows(const UpdateParams& u, const PeerXchg& px, RowRegs& r,
                                                    const StatusSnap& snap, unsigned char* new_table, float4* s_fast,
                                                    unsigned char* s_bkt, unsigned long long* s_stash,
                                                    DeferredShared& ds, bool writer, int seq, float& thresh_out) {
  DevStatus* st = u.st;
  const int tid = threadIdx.x;
  const int was_first = snap.first, iter_old = snap.iter, max_iter = snap.max_iter;
  const double tol = snap.tol;
  if (px.n_ranks > 1) {
    // (s_stash: the idle accumulator slices, (n_ranks - 1) * (kpad * 4 + 1) words)
    const int n = u.kpad * 4 + 1;
    gather_peer_words(px, n, (unsigned int)snap.epoch, s_stash, st);  // the epoch the pending E-step's packets carry
    for (int qi = 0; qi < px.n_ranks - 1; ++qi) {
      const unsigned long long* row = s_stash + (size_t)qi * n;
      if (tid < u.kpad) {
        r.a.x += row[tid * 4 + 0];
        r.a.y += row[tid * 4 + 1];
        r.b.x += row[tid * 4 + 2];
        r.b.y += row[tid * 4 + 3];
      }
      if (tid == kThreads - 1) r.nchg += row[u.kpad * 4];
    }
  }
  if (tid == kThreads - 1) ds.nchg = r.nchg;
  const int n_empty = __syncthreads_count(tid < u.k && r.b.y == 0ull);
#ifdef MDKM_TIMING
  if (writer && tid == 0) st->t_a = globaltimer_ns();
#endif
  if (n_empty > 0) {
    // the host sequences the relocation kernels on the parked (global) sums and re-runs the update
    if (writer) {
      if (tid < u.kpad) {
        *reinterpret_cast<ulonglong2*>(u.acc_saved + tid * 4) = r.a;
        *reinterpret_cast<ulonglong2*>(u.acc_saved + tid * 4 + 2) = r.b;
      }
      if (tid >= kThreads - 8)  // the changed-label count and the unused words behind it
        u.acc_saved[u.kpad * 4 + (tid - (kThreads - 8))] = tid == kThreads - 8 ? ds.nchg : 0ull;
      __syncthreads();
      if (tid == 0) {
        st->n_empty = n_empty;
        __threadfence();
        st->paused = 1;
      }
    }
    return 2;
  }
  double shift2 = 0.0, m_cn = 0.0, m_cx = 0.0, m_cy = 0.0, m_cz = 0.0;
  if (tid < u.kpad) {
    float4 fr4 = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7f800000));
    double4 ex4 = make_double4(0.0, 0.0, 0.0, 1.0 / 0.0);
    if (tid < u.k) {
      const double sc = (double)r.b.y;
      const double qx = (double)(long long)r.a.x * u.inv_scale[0];
      const double qy = (double)(long long)r.a.y * u.inv_scale[1];
      const double qz = (double)(long long)r.b.x * u.inv_scale[2];
      const double alpha = 1.0 / sc;  // pyx:284-287: centers *= 1/weight
      const double cx = qx * alpha, cy = qy * alpha, cz = qz * alpha;
      const double dx = cx - r.old.x, dy = cy - r.old.y, dz = cz - r.old.z;
      const double sh = sqrt(dx * dx + dy * dy + dz * dz);  // _center_shift, pyx:298-311
      shift2 = sh * sh;                                      // (center_shift**2).sum()
      const double cn = cx * cx + cy * cy + cz * cz;
      ex4 = make_double4(cx, cy, cz, cn);
      fr4 = make_float4((float)(-2.0 * cx), (float)(-2.0 * cy), (float)(-2.0 * cz), (float)cn);
      m_cn = cn; m_cx = fabs(cx); m_cy = fabs(cy); m_cz = fabs(cz);
    }
    s_fast[tid] = fr4;
    if (writer) {
      reinterpret_cast<double4*>(new_table + exact_offset(u.kpad))[tid] = ex4;
      reinterpret_cast<float4*>(new_table)[tid] = fr4;
    }
  }
  if (s_bkt) {
    build_centroid_buckets(s_fast, s_bkt, u.k, u.kpad, u.fr);
    if (writer) {
      __syncthreads();
      const uint4* src = reinterpret_cast<const uint4*>(s_bkt);
      uint4* dst = reinterpret_cast<uint4*>(new_table + bucket_offset(u.kpad));
      for (int i = tid; i < (int)(bucket_bytes(u.k, u.kpad) / 16); i += kThreads) dst[i] = src[i];
    }
  }
  // fixed-order reductions: shuffle tree inside the warp, warps combined in index order
  for (int o = 16; o > 0; o >>= 1) {
    shift2 += __shfl_down_sync(0xffffffffu, shift2, o);
    m_cn = fmax(m_cn, __shfl_down_sync(0xffffffffu, m_cn, o));
    m_cx = fmax(m_cx, __shfl_down_sync(0xffffffffu, m_cx, o));
    m_cy = fmax(m_cy, __shfl_down_sync(0xffffffffu, m_cy, o));
    m_cz = fmax(m_cz, __shfl_down_sync(0xffffffffu, m_cz, o));
  }
  if ((tid & 31) == 0) {
    const int w = tid >> 5;
    ds.red[0][w] = shift2; ds.red[1][w] = m_cn; ds.red[2][w] = m_cx; ds.red[3][w] = m_cy; ds.red[4][w] = m_cz;
  }
  __syncthreads();
#ifdef MDKM_TIMING
  if (writer && tid == 0) st->t_b = globaltimer_ns();
#endif
  // every thread combines the warps' partials itself (no broadcast barrier)
  shift2 = 0.0; m_cn = 0.0; m_cx = 0.0; m_cy = 0.0; m_cz = 0.0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) {
    shift2 += ds.red[0][w];
    m_cn = fmax(m_cn, ds.red[1][w]);
    m_cx = fmax(m_cx, ds.red[2][w]);
    m_cy = fmax(m_cy, ds.red[3][w]);
    m_cz = fmax(m_cz, ds.red[4][w]);
  }
  // FP32 error bound of the fast distances (DESIGN.md "Exactness"): u = 2^-24
  const double ue = 5.9604644775390625e-08;
  const double E = ue * (4.0 * m_cn + 10.0 * (u.fr.halfrange[0] * m_cx + u.fr.halfrange[1] * m_cy +
                                               u.fr.halfrange[2] * m_cz));
  thresh_out = __double2float_ru(2.0 * E * 1.001 + 1e-37);
  const unsigned long long n_changed = ds.nchg;
  const int it = iter_old + 1;
  const bool strict = !was_first && n_changed == 0ull;           // _kmeans.py:721-726
  const bool done = strict || shift2 <= tol || it >= max_iter;  // _kmeans.py:729-738
  if (writer && tid == 0) {
    ds.thresh = thresh_out;
    ds.shift2 = shift2;
    ds.iter = it;
    ds.nempty = 0;
    if (done) {
      // `done` first: a CTA that starts late leaves at once whatever else it reads
      st->done = 1;
      if (strict) st->strict = 1;
      __threadfence();
      publish_update(st, ds);
      st->last_seq = seq;  // (the final table sits in table[seq & 1]; `pending` is cleared by the settle kernel)
    }
  }
  return done ? 1 : 0;
}

template <typename LabT>
__host__ __device__ constexpr int stage_bytes() { return kBlockFloats * 4 + kGroup * (int)sizeof(LabT); }

// (Handing the tail of the worklist out dynamically -- an atomic claim per entry, 16 counters, two
// steps ahead of the ring -- was measured: the claims' latency under load stalls the warps more than
// the static round-robin's imbalance costs; config 2 +3.7 us, config 5 +67 us per iteration.  Not kept.)
// (Two more hand-out schemes were measured after that: the warps of a CTA drawing their CTA's share from a
// shared-memory counter -- no change --, and a quarter of the list kept as a pool the CTAs draw from in chunks
// of eight entries, one global atomic per chunk -- the CTAs then finish within 5 instead of 8 us of each
// other on the config-3 shape, but all of them later: the pass is bound by the SMs' issue rate, an early
// CTA's slots were being used by its neighbours on the SM all along.)
// (Letting the last label of a mixed group take what the others left of the group's totals -- one round
// of masked sums less -- was measured too: +0.6 us on config 2, +2 us on the config-3 shape.  Not kept.)
// Tables of more than 256 rows (16-bit labels) leave room for two CTAs per SM only (shared memory), so
// those kernels may use up to 128 registers.
template <typename LabT, bool kPrivate, int kChunks>
__global__ void __launch_bounds__(kThreads, sizeof(LabT) == 2 ? 2 : 3) lloyd_step_kernel(const StepParams p) {
  constexpr int kWarps = kThreads / 32;
  constexpr int kStageB = stage_bytes<LabT>();
  constexpr int kLabB = kGroup * (int)sizeof(LabT);

  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int kp32 = kChunks > 0 ? kChunks * 32 : ((p.kpad + 31) & ~31);  // rows staged in shared memory
  float4* s_fast = reinterpret_cast<float4*>(smem_raw);
  unsigned char* s_ring = reinterpret_cast<unsigned char*>(s_fast + kp32);
  unsigned long long* s_acc_all = reinterpret_cast<unsigned long long*>(s_ring + kWarps * kStages * kStageB);
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ __align__(8) uint64_t s_gbar[kWarps * kStages];
  __shared__ unsigned int s_changed;
  __shared__ unsigned int s_refined;
  __shared__ unsigned short s_cand[kWarps * kCandCap];
  __shared__ bool s_is_last;
  __shared__ DeferredShared s_def;

  // the next kernel of the stream may be set up while this one runs (it waits for this grid's end
  // before it reads anything, see grid_dependency_wait below)
  grid_launch_dependents();
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);  // warp-uniform by construction
  const int n_slices = kPrivate ? kWarps : 1;
  unsigned long long* s_acc = s_acc_all + (kPrivate ? warp * p.kpad * 4 : 0);
  // bucket index of the centroids (k >= kBucketMinK), behind the accumulator slices
  const uint32_t bkt_bytes = (uint32_t)bucket_bytes(p.k, p.kpad);
  unsigned char* s_bkt = reinterpret_cast<unsigned char*>(s_acc_all + (size_t)(kPrivate ? kWarps : 1) * p.kpad * 4);
  // this launch's table, accumulator and worklist counter (see StepParams)
  const int seq = p.seq;
  unsigned char* table_cur = p.table + (size_t)(seq & 1) * p.table_stride;
  unsigned long long* acc_w = p.acc + (size_t)(seq % 3) * p.acc_slot;
  int* work_count = p.work_count + (seq & 1);
  const double4* c64 = reinterpret_cast<const double4*>(table_cur + exact_offset(p.kpad));
  const FrameF f = p.f;
  // (One launch = one Lloyd iteration.  Running a batch of iterations inside one launch, with a
  // grid barrier instead of the kernel boundary, was measured: 0.9 us per iteration at best, and
  // the loop-carried state pushed the kernel over its register budget -- not kept.)
  // the update of the previous E-step is still to be applied (see deferred_update): true for every
  // fused launch but the first one behind a settle kernel.  Tables of at most 128 rows: every CTA
  // applies it, one row per thread -- the row's sums and old centroid are requested right here,
  // together with the status words below
  const bool pending = p.fuse_update && seq > 0;  // the same for every CTA
  const unsigned long long* acc_prev = p.acc + (size_t)((seq + 2) % 3) * p.acc_slot;
  const unsigned char* table_prev = p.table + (size_t)((seq & 1) ^ 1) * p.table_stride;
  RowRegs rr;
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    for (int i = 0; i < kWarps * kStages; ++i) mbar_init(&s_gbar[i], 1);
    fence_mbar_init();
    s_changed = 0;
    s_refined = 0;
  }
  // rows [kpad, kp32) are not covered by the table: make them non-candidates
  for (int i = p.kpad + tid; i < kp32; i += kThreads) {
    s_fast[i] = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7f800000));
  }
  // (launched with programmatic stream serialisation: the previous kernel of the stream may still be
  // draining -- nothing it wrote is read before this point)
  grid_dependency_wait();
  if (kPrivate && pending) deferred_prefetch(rr, acc_prev, table_prev, p.k, p.kpad);
  const StatusSnap snap = status_snapshot(p.st);
  if (!p.ignore_status && (snap.done | snap.paused)) return;  // the same for every CTA
#ifdef MDKM_TIMING
  if (blockIdx.x == 0 && tid == 0) {
    p.st->t_start = globaltimer_ns();
    p.st->t_update_done = 0ull;
  }
#endif

  // group bookkeeping is 32-bit and warp-uniform (the host guarantees n < 2^38 points)
  const int n_groups = (int)((p.n + kGroup - 1) / kGroup);
  const int n_full = (int)(p.n / kGroup);  // groups below this index have 128 real points
  LabT* labels = reinterpret_cast<LabT*>(p.labels);
  unsigned int n_chg = 0, n_ref = 0;
  // (one-level walk: the first group's summary travels while the centroid table does)
  float4 pa = make_float4(0.f, 0.f, 0.f, 0.f), pb = pa, pc = pa;
  int pprev = -1;
  if (!p.two_level && (int)blockIdx.x * kThreads + tid < n_groups) {
    const int g_first = (int)blockIdx.x * kThreads + tid;
    const float4* src = reinterpret_cast<const float4*>(p.gsum + g_first);
    pa = __ldg(src); pb = __ldg(src + 1); pc = __ldg(src + 2);
    pprev = (!pending && snap.first != 0) ? -1 : p.glabel[g_first];
  }
  float thresh = 0.f;
  bool first_iter = false;
  bool table_by_tma = !pending;
  if (pending) {
    int verdict;
    if (kPrivate) {
      verdict = deferred_update_rows(p.upd, p.px, rr, snap, table_cur, s_fast, bkt_bytes ? s_bkt : nullptr, s_acc_all,
                                     s_def, blockIdx.x == 0, seq, thresh);
    } else if (blockIdx.x == 0) {
      // larger tables: CTA 0 alone applies the update and announces the verdict (the iteration is
      // long, the redundant work would cost more than the wait)
      verdict = deferred_update(p.upd, p.px, acc_prev, table_prev, table_cur, s_fast, bkt_bytes ? s_bkt : nullptr,
                                s_acc_all, s_def, true, seq);
      thresh = s_def.thresh;
      __threadfence();
      __syncthreads();
      if (tid == 0) {
        p.st->next_thresh = thresh;
        __threadfence();
        st_release_gpu_u32(&p.st->upd_flag, ((unsigned int)snap.epoch << 2) | (unsigned int)verdict);
      }
    } else {
      if (tid == 0) {
        const unsigned int want = (unsigned int)snap.epoch << 2;
        unsigned int fl;
        const long long t0 = clock64();
        do {
          fl = ld_acquire_gpu_u32(&p.st->upd_flag);
          if (clock64() - t0 > (8ll << 30)) {  // bounded wait (about 4 s); never triggers: CTA 0 is resident
            p.st->xchg_timeout = 1;
            fl = want | 1u;
          }
        } while ((fl & ~3u) != want);
        s_def.verdict = (int)(fl & 3u);
        s_def.thresh = *reinterpret_cast<volatile float*>(&p.st->next_thresh);
      }
      __syncthreads();
      verdict = s_def.verdict;
      thresh = s_def.thresh;
      if (verdict == 0) {
        // the table CTA 0 has just written: plain loads through L2 (not the TMA unit: the writes were
        // made through the generic proxy inside this very kernel)
        const uint4* src = reinterpret_cast<const uint4*>(table_cur);
        uint4* dst = reinterpret_cast<uint4*>(s_fast);
        for (int i = tid; i < p.kpad; i += kThreads) dst[i] = __ldcg(src + i);
        if (bkt_bytes) {
          const uint4* bs = reinterpret_cast<const uint4*>(table_cur + bucket_offset(p.kpad));
          uint4* bd = reinterpret_cast<uint4*>(s_bkt);
          for (int i = tid; i < (int)(bkt_bytes / 16); i += kThreads) bd[i] = __ldcg(bs + i);
        }
      }
    }
    if (verdict != 0) return;  // converged / max_iter / paused: the same for every CTA
  } else {
    __syncthreads();
    if (tid == 0) {
      // centroid rows (and their bucket index): global -> shared through the TMA unit (1-D bulk copies)
      mbar_expect_tx(&s_bar, (uint32_t)p.kpad * 16u + bkt_bytes);
      tma_load_1d(s_fast, table_cur, (uint32_t)p.kpad * 16u, &s_bar);
      if (bkt_bytes) tma_load_1d(s_bkt, table_cur + bucket_offset(p.kpad), bkt_bytes, &s_bar);
    }
    thresh = snap.thresh;
    first_iter = snap.first != 0;
  }
  // (the accumulator slices held the gathered sums during the update)
  for (int i = tid; i < n_slices * p.kpad * 4; i += kThreads) s_acc_all[i] = 0ull;
  if (blockIdx.x == 0 && p.fuse_update) {
    // the accumulator the NEXT launch adds into (last read by the previous launch) and the previous
    // launch's worklist counter
    unsigned long long* acc_z = p.acc + (size_t)((seq + 1) % 3) * p.acc_slot;
    for (int i = tid; i < p.kpad * 4 + 8; i += kThreads) acc_z[i] = 0ull;
    if (tid == 0) p.work_count[(seq & 1) ^ 1] = 0;
  }
  __syncthreads();
  if (table_by_tma) mbar_wait(&s_bar, 0);
#ifdef MDKM_TIMING
  if (blockIdx.x == 0 && tid == 0) p.st->t_classify_start = globaltimer_ns();  // table ready
#endif
  // ---- pass 1: settle whole groups from their summaries (no point is read) ----------------
  // the ring is idle during pass 1: its first bytes stage the worklist entries
  static_assert(kWarps * kStages * kStageB >= kClassifyList * 4, "worklist staging does not fit the ring");
  if (p.two_level)
    classify_groups_two_level<LabT, kPrivate>(p.gsum, reinterpret_cast<const SuperSummary*>(p.ssum), n_groups, labels,
                                              p.glabel, p.worklist, work_count, s_fast, p.k, 4.0f * thresh, first_iter,
                                              s_acc, reinterpret_cast<int*>(s_ring), bkt_bytes ? s_bkt : nullptr, n_chg,
                                              p.settle != 0);
  else
    classify_groups_flat<LabT, kPrivate>(p.gsum, n_groups, labels, p.glabel, p.worklist, work_count, s_fast, p.k,
                                         4.0f * thresh, first_iter, s_acc, reinterpret_cast<int*>(s_ring),
                                         bkt_bytes ? s_bkt : nullptr, n_chg, p.settle != 0, pa, pb, pc, pprev);
#ifdef MDKM_TIMING
  if (tid == 0) atomicMax(&p.st->t_first_done, globaltimer_ns());  // latest end of pass 1 (reused field)
#endif
  grid_barrier(p.grid_bar, &p.st->xchg_timeout);  // the worklist is complete
#ifdef MDKM_TIMING
  if (blockIdx.x == 0 && tid == 0) p.st->t_classify_done = globaltimer_ns();
#endif
  // ---- pass 2: the groups a cluster boundary crosses, point by point -----------------------
  // (the "groups" below are positions in the worklist)
  const int n_items = *reinterpret_cast<volatile int*>(work_count);
  if (p.fuse_update && blockIdx.x == 0 && tid == 0) {
    // every CTA has read the status block by now: the applied update and this E-step become visible
    if (pending) publish_update(p.st, s_def);
    p.st->pending = 1;
    p.st->last_seq = seq;
    p.st->epoch = p.st->epoch + 1ull;  // the epoch this E-step's packets carry
    p.st->work_sum += (unsigned long long)n_items;
  }
  // round-robin over the warps of the grid: neighbouring list entries are neighbouring groups
  // with similar cost, so interleaving them evens out the warps' loads
  const int stride = (int)gridDim.x * kWarps;
  const int g0 = (int)blockIdx.x * kWarps + warp;
  const int g_end = n_items;
  const int* __restrict__ wl = p.worklist;
  const uint32_t ring_a = smem_u32(s_ring) + warp * (kStages * kStageB);
  const uint32_t gbar_a = smem_u32(s_gbar) + warp * (kStages * 8);
  const float* pts = p.pts;
  int g_fetch = g0;

  // one elected lane fetches group `gf` into `stage`: the 1536-byte xyz block and its labels
  auto issue = [&](int stage, int gf) {
    if (elect_one()) {
      const uint32_t dst = ring_a + stage * kStageB, bar = gbar_a + stage * 8;
      mbar_expect_tx_a(bar, (uint32_t)kStageB);
      tma_load_1d_a(dst, pts + (size_t)gf * kBlockFloats, kBlockFloats * 4, bar);
      tma_load_1d_a(dst + kBlockFloats * 4, labels + (size_t)gf * kGroup, kLabB, bar);
    }
  };
  // group index of the three stages in flight (warp-uniform registers)
  int gq0 = 0, gq1 = 0, gq2 = 0;
  static_assert(kStages == 3, "the group-index queue below is written for three stages");
  // (the list was written by other CTAs of this very kernel: read it through L2, not the
  // non-coherent path)
  if (g_fetch < g_end) { gq0 = __ldcg(wl + g_fetch); issue(0, gq0); }
  g_fetch += stride;
  if (g_fetch < g_end) { gq1 = __ldcg(wl + g_fetch); issue(1, gq1); }
  g_fetch += stride;
  if (g_fetch < g_end) { gq2 = __ldcg(wl + g_fetch); issue(2, gq2); }
  g_fetch += stride;
  int g_pref = g_fetch < g_end ? __ldcg(wl + g_fetch) : 0;  // list entry of the next fetch

  // run accumulator: while consecutive groups of this warp carry one label, every lane just
  // adds its own four fixed-point coordinates (int32, no cross-lane traffic); the run is
  // reduced with three REDUX and added to shared memory only when the label changes, a mixed
  // group arrives, or after kRunMax groups (int32 headroom: 4 * 2^22 * 64 = 2^30)
  constexpr int kRunMax = 64;
  int rx = 0, ry = 0, rz = 0;
  int run_groups = 0;
  int wlab = -1;
  auto flush_run = [&]() {
    if (run_groups > 0) {
      // a lane's partial can reach 2^30 and the points of a run usually lie on one side of the
      // origin: the warp total does not fit 32 bits, so the two halves are reduced separately
      const long long sx = ((long long)__reduce_add_sync(0xffffffffu, rx >> 15) << 15) +
                           (long long)__reduce_add_sync(0xffffffffu, rx & 0x7fff);
      const long long sy = ((long long)__reduce_add_sync(0xffffffffu, ry >> 15) << 15) +
                           (long long)__reduce_add_sync(0xffffffffu, ry & 0x7fff);
      const long long sz = ((long long)__reduce_add_sync(0xffffffffu, rz >> 15) << 15) +
                           (long long)__reduce_add_sync(0xffffffffu, rz & 0x7fff);
      if (lane == 0) acc_add<kPrivate>(s_acc, wlab, sx, sy, sz, (unsigned int)run_groups * kGroup);
      rx = ry = rz = 0;
      run_groups = 0;
    }
  };
  int stage = 0;
  uint32_t parity = 0;

  for (int it = g0; it < g_end; it += stride) {
    const int g = gq0;
    const uint32_t st_a = ring_a + stage * kStageB + lane * 16;
    mbar_wait_a(gbar_a + stage * 8, parity);
    const float4 vx = lds_f4(st_a);
    const float4 vy = lds_f4(st_a + kGroup * 4);
    const float4 vz = lds_f4(st_a + kGroup * 8);
    const unsigned char* src = s_ring + warp * (kStages * kStageB) + stage * kStageB;
    const typename LabPack<LabT>::V oldl = LabPack<LabT>::load(src + kBlockFloats * 4 + lane * LabPack<LabT>::kBytes);
    const float xc[4] = {vx.x - f.ox, vx.y - f.ox, vx.z - f.ox, vx.w - f.ox};
    const float yc[4] = {vy.x - f.oy, vy.y - f.oy, vy.z - f.oy, vy.w - f.oy};
    const float zc[4] = {vz.x - f.oz, vz.y - f.oz, vz.z - f.oz, vz.w - f.oz};
    int lab[4];
    int ncand = -1;
    if (kChunks == 0 && bkt_bytes) {
      // many centroids: candidates from the bucket index, reference = a label the group had
      const int hint = first_iter ? -1 : __shfl_sync(0xffffffffu, LabPack<LabT>::get(oldl, 0), 0);
      ncand = assign_group_bucketed(xc, yc, zc, reinterpret_cast<const float*>(src + lane * 16),
                                    reinterpret_cast<const float*>(src + kGroup * 4 + lane * 16),
                                    reinterpret_cast<const float*>(src + kGroup * 8 + lane * 16), f, s_fast, c64,
                                    s_bkt, p.k, kp32, thresh, hint, s_cand + warp * kCandCap, lane, lab, n_ref);
    }
    if (ncand < 0)
      ncand = assign_group<kChunks>(xc, yc, zc, reinterpret_cast<const float*>(src + lane * 16),
                                    reinterpret_cast<const float*>(src + kGroup * 4 + lane * 16),
                                    reinterpret_cast<const float*>(src + kGroup * 8 + lane * 16), f, s_fast, c64,
                                    p.k, kp32, thresh, lane, lab, n_ref);
    // every value read from the stage has been consumed: refill it with the group kStages
    // ahead (the reads completed before this point, so the async-proxy write cannot race)
    __syncwarp();
    gq0 = gq1;
    gq1 = gq2;
    gq2 = g_pref;
    if (g_fetch < g_end) issue(stage, g_pref);
    g_fetch += stride;
    g_pref = g_fetch < g_end ? __ldcg(wl + g_fetch) : 0;
    if (++stage == kStages) {
      stage = 0;
      parity ^= 1u;
    }

    const bool full = g < n_full;  // warp-uniform
    const typename LabPack<LabT>::V newl = LabPack<LabT>::pack(lab);
    LabPack<LabT>::store(labels + (size_t)g * kGroup + lane * 4, newl);
    if (first_iter) {
      n_chg += full ? 4u : (unsigned int)max(0LL, min(4LL, p.n - ((long long)g * kGroup + lane * 4)));
    } else if (!LabPack<LabT>::same(newl, oldl)) {
      const long long i0 = (long long)g * kGroup + lane * 4;
#pragma unroll
      for (int e = 0; e < 4; ++e)
        n_chg += ((full || i0 + e < p.n) && lab[e] != LabPack<LabT>::get(oldl, e)) ? 1u : 0u;
    }

    // fixed-point coordinates: q = rint(x' * scale) by mantissa alignment (|q| < 2^22):
    // bits(x'*s + 1.5*2^23) - bits(1.5*2^23); the bias is removed once per sum
    unsigned int ux[4], uy[4], uz[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      ux[e] = __float_as_uint(fmaf(xc[e], f.sx, kMagic));
      uy[e] = __float_as_uint(fmaf(yc[e], f.sy, kMagic));
      uz[e] = __float_as_uint(fmaf(zc[e], f.sz, kMagic));
    }
    const int tx = (int)(ux[0] + ux[1] + ux[2] + ux[3] - 4u * kMagicBits);
    const int ty = (int)(uy[0] + uy[1] + uy[2] + uy[3] - 4u * kMagicBits);
    const int tz = (int)(uz[0] + uz[1] + uz[2] + uz[3] - 4u * kMagicBits);
    // is the whole group one label?  (a lone candidate labels it without looking)
    bool uniform = full && (ncand <= 1);
    int l0 = lab[0];
    if (full && !uniform) {
      l0 = __shfl_sync(0xffffffffu, lab[0], 0);
      uniform = __all_sync(0xffffffffu, (lab[0] == l0) && (lab[1] == l0) && (lab[2] == l0) && (lab[3] == l0));
    }
    // settled (one centroid owns the whole box): the classification pass takes over from here
    if (lane == 0) p.glabel[g] = (full && ncand <= 1) ? lab[0] : -1;
    if (uniform) {
      if (l0 != wlab || run_groups == kRunMax) {  // warp-uniform
        flush_run();
        wlab = l0;
      }
      rx += tx;
      ry += ty;
      rz += tz;
      ++run_groups;
    } else {
      // mixed group (a cluster boundary crosses it) or the partial tail group: one round per
      // distinct label, each lane contributing the points it has with that label
      flush_run();
      const long long i0 = (long long)g * kGroup + lane * 4;
      bool act[4];
      unsigned int rem = 0;
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        act[e] = full || (i0 + e < p.n);
        rem |= act[e] ? (1u << e) : 0u;
      }
      unsigned int todo = __ballot_sync(0xffffffffu, rem != 0);
      while (todo) {
        const int src_lane = __ffs(todo) - 1;
        // this lane's first unprocessed label (selects, not a dynamically indexed array)
        const int mine_first = (rem & 1u) ? lab[0] : ((rem & 2u) ? lab[1] : ((rem & 4u) ? lab[2] : lab[3]));
        const int L = __shfl_sync(0xffffffffu, mine_first, src_lane);
        int sx = 0, sy = 0, sz = 0, sc = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const bool hit = ((rem >> e) & 1u) && (lab[e] == L);
          sx += hit ? (int)(ux[e] - kMagicBits) : 0;
          sy += hit ? (int)(uy[e] - kMagicBits) : 0;
          sz += hit ? (int)(uz[e] - kMagicBits) : 0;
          sc += hit ? 1 : 0;
          rem &= hit ? ~(1u << e) : ~0u;
        }
        sx = __reduce_add_sync(0xffffffffu, sx);
        sy = __reduce_add_sync(0xffffffffu, sy);
        sz = __reduce_add_sync(0xffffffffu, sz);
        sc = __reduce_add_sync(0xffffffffu, sc);
        if (lane == 0) acc_add<kPrivate>(s_acc, L, sx, sy, sz, (unsigned int)sc);
        todo = __ballot_sync(0xffffffffu, rem != 0);
      }
    }
  }
  flush_run();
  n_chg = __reduce_add_sync(0xffffffffu, n_chg);
  n_ref = __reduce_add_sync(0xffffffffu, n_ref);
  if (lane == 0) {
    if (n_chg) atomicAdd(&s_changed, n_chg);
    if (n_ref) atomicAdd(&s_refined, n_ref);
  }
  __syncthreads();
  // CTA partials -> global int64 accumulators (RED.ADD.64; order-independent, exact)
  for (int i = tid; i < p.kpad * 4; i += kThreads) {
    unsigned long long v = 0ull;
    for (int s = 0; s < n_slices; ++s) v += s_acc_all[s * p.kpad * 4 + i];
    if (v) atomicAdd(&acc_w[i], v);
  }
  if (tid == 0) {
    if (s_changed) atomicAdd(&acc_w[p.kpad * 4 + 0], (unsigned long long)s_changed);
    if (s_refined) atomicAdd(&p.st->n_refined, (unsigned long long)s_refined);
#ifdef MDKM_TIMING
    atomicAdd(&p.st->t_update_done, globaltimer_ns() - p.st->t_start);  // sum of the CTAs' finish times
    atomicMax(&p.st->t_last_done, globaltimer_ns());
#endif
  }
  // One rank: nothing else -- the next launch (or the settle kernel) turns the sums into centroids.
  if (!p.fuse_update || p.px.n_ranks <= 1) return;
  // ---- several ranks: the last CTA to get here owns the complete local sums and sends them ----
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const unsigned int t = atomicAdd(&p.st->ticket, 1u);
    s_is_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (s_is_last) {  // CTA-uniform
    __threadfence();
    if (tid == 0) p.st->ticket = 0u;
    const unsigned int tag = (unsigned int)__ldcg(&p.st->epoch);  // (incremented by CTA 0 behind the grid barrier)
    peer_send_sums(p.px, acc_w, p.kpad * 4 + 8, tag);
  }
}

// ---------------------------------------------------------------------------------------
// Settle kernel (one CTA), enqueued by the host behind a run of fused step launches and before
// anything else reads the table: applies the update that is still pending (the last E-step's
// sums), moves the current table to table[0] and clears the rotating buffers, so that every
// other kernel -- final pass, relocation, stand-alone update, the next run of fused launches
// starting at seq 0 -- finds the classic layout: table[0], acc[0], pending = 0.
// ---------------------------------------------------------------------------------------
struct SettleParams {
  UpdateParams upd;     // acc = acc[0], table = table[0]
  PeerXchg px;
  size_t table_stride;
  int acc_slot;
  int* work_count;      // two counters
};

__global__ void __launch_bounds__(kThreads, 1) lloyd_settle_kernel(const SettleParams sp) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  __shared__ DeferredShared s_def;
  const UpdateParams& u = sp.upd;
  DevStatus* st = u.st;
  const int tid = threadIdx.x;
  float4* s_fast = reinterpret_cast<float4*>(smem_raw);
  unsigned long long* s_sums = reinterpret_cast<unsigned long long*>(s_fast + u.kpad);
  unsigned char* s_bkt = reinterpret_cast<unsigned char*>(s_sums + u.kpad * 4);
  const uint32_t bkt_bytes = (uint32_t)bucket_bytes(u.k, u.kpad);
  const int last = st->last_seq;
  const bool apply = st->pending != 0 && !st->paused && !st->done;
  unsigned char* t_last = u.table + (size_t)(last & 1) * sp.table_stride;
  int verdict = -1;
  if (apply) {
    verdict = deferred_update(u, sp.px, u.acc + (size_t)(last % 3) * sp.acc_slot, t_last, u.table, s_fast,
                              bkt_bytes ? s_bkt : nullptr, s_sums, s_def, true, 0);
    if (verdict == 0 && tid == 0) publish_update(st, s_def);  // (more iterations to come)
  }
  __syncthreads();
  if ((last & 1) && (!apply || verdict == 2)) {
    // the table the last E-step used (final, or the one a paused update starts from) -> table[0]
    const uint4* src = reinterpret_cast<const uint4*>(t_last);
    uint4* dst = reinterpret_cast<uint4*>(u.table);
    for (int i = tid; i < (int)(table_bytes(u.k, u.kpad) / 16); i += kThreads) dst[i] = src[i];
  }
  for (int i = tid; i < 3 * sp.acc_slot; i += kThreads) u.acc[i] = 0ull;
  if (tid == 0) {
    sp.work_count[0] = 0;
    sp.work_count[1] = 0;
    st->pending = 0;
    st->last_seq = 0;
  }
}

// Start of a fit (one launch): the status block, cleared accumulators and counters, and the
// centroid table from K x 3 float64 centroids in ORIGINAL coordinates.
struct InitTableParams {
  const double* centers;  // k*3, device or device-visible host memory
  unsigned char* table;
  DevStatus* st;
  Frame fr;
  int k, kpad;
  DevStatus st0;                    // written to *st
  unsigned long long* acc;          // acc_words words zeroed (or nullptr)
  long long acc_words;
  int* work_count;                  // two counters zeroed (or nullptr)
  unsigned int* final_ticket;       // zeroed (lloyd_final_kernel)
  const unsigned int* index_fault;  // or nullptr: nonzero when the raster mirror index timed out -> status done + fault
};

__global__ void __launch_bounds__(kThreads, 1) init_table_kernel(const InitTableParams u) {
  __shared__ double s_red[kThreads / 32];
  if (threadIdx.x == 0) {
    DevStatus s = u.st0;
    if (u.index_fault && *u.index_fault) {
      s.done = 1;
      s.xchg_timeout = 2;
    }
    *u.st = s;
    *u.final_ticket = 0u;
    if (u.work_count) {
      u.work_count[0] = 0;
      u.work_count[1] = 0;
    }
  }
  for (long long i = threadIdx.x; i < u.acc_words; i += kThreads) u.acc[i] = 0ull;
  float4* fast = reinterpret_cast<float4*>(u.table);
  double4* exact = reinterpret_cast<double4*>(u.table + exact_offset(u.kpad));
  double m_cn = 0.0, m_cx = 0.0, m_cy = 0.0, m_cz = 0.0;
  for (int j = threadIdx.x; j < u.kpad; j += kThreads) {
    if (j < u.k) {
      const double cx = u.centers[3 * j + 0] - u.fr.origin[0];
      const double cy = u.centers[3 * j + 1] - u.fr.origin[1];
      const double cz = u.centers[3 * j + 2] - u.fr.origin[2];
      const double cn = cx * cx + cy * cy + cz * cz;
      exact[j] = make_double4(cx, cy, cz, cn);
      fast[j] = make_float4((float)(-2.0 * cx), (float)(-2.0 * cy), (float)(-2.0 * cz), (float)cn);
      m_cn = fmax(m_cn, cn);
      m_cx = fmax(m_cx, fabs(cx));
      m_cy = fmax(m_cy, fabs(cy));
      m_cz = fmax(m_cz, fabs(cz));
    } else {
      fast[j] = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7f800000));
      exact[j] = make_double4(0.0, 0.0, 0.0, 1.0 / 0.0);
    }
  }
  m_cn = block_max(m_cn, s_red);
  m_cx = block_max(m_cx, s_red);
  m_cy = block_max(m_cy, s_red);
  m_cz = block_max(m_cz, s_red);
  if (threadIdx.x == 0) {
    const double ue = 5.9604644775390625e-08;
    const double E = ue * (4.0 * m_cn + 10.0 * (u.fr.halfrange[0] * m_cx + u.fr.halfrange[1] * m_cy +
                                                 u.fr.halfrange[2] * m_cz));
    u.st->thresh = __double2float_ru(2.0 * E * 1.001 + 1e-37);
  }
  build_centroid_buckets(fast, u.table + bucket_offset(u.kpad), u.k, u.kpad, u.fr);
}

// Reads the table back as K x 3 float64 centroids in original coordinates.
__global__ void read_table_kernel(const unsigned char* table, int k, int kpad, Frame fr,
                                  double* centers_out) {
  const double4* exact = reinterpret_cast<const double4*>(table + exact_offset(kpad));
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < k; j += gridDim.x * blockDim.x) {
    const double4 c = exact[j];
    centers_out[3 * j + 0] = c.x + fr.origin[0];
    centers_out[3 * j + 1] = c.y + fr.origin[1];
    centers_out[3 * j + 2] = c.z + fr.origin[2];
  }
}

// Converts the int64 accumulators into float64 coordinate sums (original frame) + counts.
__global__ void read_sums_kernel(const unsigned long long* acc, int k, Frame fr, double* sums_out,
                                 long long* counts_out) {
  for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < k; j += gridDim.x * blockDim.x) {
    const long long cnt = (long long)acc[j * 4 + 3];
    for (int d = 0; d < 3; ++d)
      sums_out[3 * j + d] = (double)(long long)acc[j * 4 + d] / fr.scale[d] + (double)cnt * fr.origin[d];
    counts_out[j] = cnt;
  }
}

// Per-(day, cluster) slots of the final pass -> counts and means (original frame).  The exact
// coordinate sum is rebuilt first and divided once: exact whenever it fits 53 bits, so the mean
// is then the correctly rounded mean of the grid points.  Explicit roundings: no FMA contraction.
__global__ void day_stats_kernel(const unsigned long long* acc, long long slots, Frame fr, long long* counts_out,
                                 double* means_out) {
  for (long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x; j < slots; j += (long long)gridDim.x * blockDim.x) {
    const long long cnt = (long long)acc[j * 4 + 3];
    counts_out[j] = cnt;
    for (int d = 0; d < 3; ++d) {
      const double sum = __dadd_rn(__ddiv_rn((double)(long long)acc[j * 4 + d], fr.scale[d]),
                                   __dmul_rn((double)cnt, fr.origin[d]));
      means_out[3 * j + d] = cnt ? __ddiv_rn(sum, (double)cnt) : __longlong_as_double(0x7ff8000000000000ll);
    }
  }
}

// ---------------------------------------------------------------------------------------
// In raster order a group is a strip of one row -- except the one that runs over the end of a
// row (one in W/128): its box spans the whole width of the frame, every cluster along the row
// becomes a candidate and the group costs as much as dozens of others.  Such a group is
// assigned in two halves (the points of its first row, then the rest), each with its own small
// box; in each half the points of the other one are replaced by a stand-in from this half,
// whose result is dropped.  Same labels as the one-box form: both are exact.
// ---------------------------------------------------------------------------------------
template <int kChunks>
__device__ __forceinline__ void assign_split_group(const float (&xo)[4], const float (&yo)[4], const float (&zo)[4],
                                                   const FrameF& f, const float4* __restrict__ s_fast,
                                                   const double4* __restrict__ c64, const unsigned char* s_bkt,
                                                   int k, int kp32, float thresh, unsigned short* s_cand, int lane,
                                                   int (&lab)[4], unsigned int& n_ref) {
  const float y_head = __shfl_sync(0xffffffffu, yo[0], 0);
#pragma unroll 1
  for (int half = 0; half < 2; ++half) {
    const int src_lane = half ? 31 : 0;  // the group's first / last point belongs to this half
    const float sx = __shfl_sync(0xffffffffu, half ? xo[3] : xo[0], src_lane);
    const float sy = __shfl_sync(0xffffffffu, half ? yo[3] : yo[0], src_lane);
    const float sz = __shfl_sync(0xffffffffu, half ? zo[3] : zo[0], src_lane);
    float hx[4], hy[4], hz[4], hxc[4], hyc[4], hzc[4];
    unsigned int mine = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const bool in_half = (yo[e] == y_head) == (half == 0);
      mine |= in_half ? (1u << e) : 0u;
      hx[e] = in_half ? xo[e] : sx;
      hy[e] = in_half ? yo[e] : sy;
      hz[e] = in_half ? zo[e] : sz;
      hxc[e] = hx[e] - f.ox; hyc[e] = hy[e] - f.oy; hzc[e] = hz[e] - f.oz;
    }
    int hl[4];
    int ncand = -1;
    if (kChunks == 0 && s_bkt)
      ncand = assign_group_bucketed(hxc, hyc, hzc, hx, hy, hz, f, s_fast, c64, s_bkt, k, kp32, thresh, -1, s_cand,
                                    lane, hl, n_ref, mine);
    if (ncand < 0) assign_group<kChunks>(hxc, hyc, hzc, hx, hy, hz, f, s_fast, c64, k, kp32, thresh, lane, hl, n_ref, mine);
#pragma unroll
    for (int e = 0; e < 4; ++e) lab[e] = ((mine >> e) & 1u) ? hl[e] : lab[e];
  }
}

// Adds this lane's points to their (day, cluster) slots; key[e] < 0 for a point past the end.
// Warp-synchronous.  Lanes with equal keys are summed first (__match_any_sync, one key per lane
// and round, so at most four rounds): consecutive points mostly share a raster row and a
// cluster, and a group of one key costs one slot update.  32-bit partial sums: a round sums at
// most 128 points of |q| < 2^22.  kPrivate: `acc` is this warp's own copy of the slots (shared
// memory), updated without atomics -- the keys of one round are distinct, and __syncwarp orders
// the rounds; otherwise the global slots, with 64-bit atomic adds.
template <bool kPrivate>
__device__ __forceinline__ void stats_add(unsigned long long* acc, const int (&key)[4], const int (&qx)[4],
                                          const int (&qy)[4], const int (&qz)[4], int lane) {
  unsigned int rem = (key[0] >= 0 ? 1u : 0u) | (key[1] >= 0 ? 2u : 0u) | (key[2] >= 0 ? 4u : 0u) |
                     (key[3] >= 0 ? 8u : 0u);
  while (__any_sync(0xffffffffu, rem != 0)) {
    const int mine = (rem & 1u) ? key[0] : ((rem & 2u) ? key[1] : ((rem & 4u) ? key[2] : ((rem & 8u) ? key[3] : -1)));
    int sx = 0, sy = 0, sz = 0, sc = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const bool hit = ((rem >> e) & 1u) && key[e] == mine;
      sx += hit ? qx[e] : 0;
      sy += hit ? qy[e] : 0;
      sz += hit ? qz[e] : 0;
      sc += hit ? 1 : 0;
      rem &= hit ? ~(1u << e) : ~0u;
    }
    const unsigned int peers = __match_any_sync(0xffffffffu, mine);
    sx = __reduce_add_sync(peers, sx);
    sy = __reduce_add_sync(peers, sy);
    sz = __reduce_add_sync(peers, sz);
    sc = __reduce_add_sync(peers, sc);
    if (mine >= 0 && lane == __ffs(peers) - 1) acc_add<kPrivate>(acc, mine, sx, sy, sz, (unsigned int)sc);
    if (kPrivate) __syncwarp();
  }
}

// labels and FP64 inertia (direct form) of this lane's four points of a group; with kMap also
// label + 1 at each point's pixel of the cluster map (x and y are exact pixel coordinates); with
// kStats also the point's fixed-point coordinates into its (day, label) slot.  Warp-synchronous
// with kStats.
template <bool kMap, bool kStats>
__device__ __forceinline__ void final_emit(const FinalParams& p, const double4* __restrict__ c64, const FrameF& f,
                                           long long i0, const float (&xo)[4], const float (&yo)[4],
                                           const float (&zo)[4], const int (&lab)[4], double& inert,
                                           MapCursor& mc, unsigned long long* s_stats, int lane) {
  int day[4] = {-1, -1, -1, -1};
  if (kMap || kStats) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const long long i = i0 + e;
      if (i < p.n) {
        while (i >= mc.next) {
          mc.next = __ldg(p.map_seg + ++mc.day + 1);
          if (kMap) mc.base += p.map_HW;
        }
        if (kStats) day[e] = mc.day;
        if (kMap) {
          const long long pix = mc.base + (long long)pixel_index(yo[e]) * p.map_W + pixel_index(xo[e]);
          if (p.map_elem == 1) static_cast<unsigned char*>(p.map_out)[pix] = (unsigned char)(lab[e] + 1);
          else static_cast<unsigned short*>(p.map_out)[pix] = (unsigned short)(lab[e] + 1);
        }
      }
    }
  }
  if (kStats) {
    // q = rint(x' * scale) exactly as the Lloyd step's sums take it (lloyd_step_kernel)
    int key[4], qx[4], qy[4], qz[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      key[e] = day[e] >= 0 ? (int)(p.stats_day0 + day[e]) * p.k + lab[e] : -1;
      qx[e] = (int)(__float_as_uint(fmaf(xo[e] - f.ox, f.sx, kMagic)) - kMagicBits);
      qy[e] = (int)(__float_as_uint(fmaf(yo[e] - f.oy, f.sy, kMagic)) - kMagicBits);
      qz[e] = (int)(__float_as_uint(fmaf(zo[e] - f.oz, f.sz, kMagic)) - kMagicBits);
    }
    if (s_stats) stats_add<true>(s_stats, key, qx, qy, qz, lane);
    else stats_add<false>(p.stats_acc, key, qx, qy, qz, lane);
  }
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    if (i0 + e < p.n) {
      const double4 c = ld_c64(&c64[lab[e]]);
      const double dx = ((double)xo[e] - (double)f.ox) - c.x;
      const double dy = ((double)yo[e] - (double)f.oy) - c.y;
      const double dz = ((double)zo[e] - (double)f.oz) - c.z;
      inert += dx * dx + dy * dy + dz * dz;
    }
  }
  if (p.labels_out) {
    if (i0 + 3 < p.n && ((reinterpret_cast<uintptr_t>(p.labels_out) & 15) == 0)) {
      *reinterpret_cast<int4*>(p.labels_out + i0) = make_int4(lab[0], lab[1], lab[2], lab[3]);
    } else {
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (i0 + e < p.n) p.labels_out[i0 + e] = lab[e];
    }
  }
}

// ---------------------------------------------------------------------------------------
// Final pass over the resident cloud (reference point order): E-step with the final centroids
// -> int32 labels, and the inertia in FP64 (direct form, fixed-order reduction).  kMap: the
// labels also go to the cluster map (FinalParams::map_out, cleared by the host beforehand).
// kStats: per-(day, cluster) counts and fixed-point coordinate sums (FinalParams::stats_acc,
// cleared by the host beforehand); integers, so the same for any grid or point order.
// ---------------------------------------------------------------------------------------
template <int kChunks, bool kMap, bool kStats>
__global__ void __launch_bounds__(kThreads, kChunks == 0 ? MDKM_FINAL_CTAS0 : 3) lloyd_final_kernel(const FinalParams p) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int kp32 = kChunks > 0 ? kChunks * 32 : ((p.kpad + 31) & ~31);
  float4* s_fast = reinterpret_cast<float4*>(smem_raw);
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ double s_red[kThreads / 32];
  __shared__ unsigned int s_refined;
  __shared__ bool s_last;
  __shared__ unsigned short s_cand[(kThreads / 32) * kCandCap];
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const uint32_t bkt_bytes = kChunks == 0 ? (uint32_t)bucket_bytes(p.k, p.kpad) : 0u;
  unsigned char* s_bkt = reinterpret_cast<unsigned char*>(s_fast + kp32);
  if (p.skip_paused && p.st->paused && !p.st->done) {  // (grid-uniform) the host relocates and runs the tail again
    if (blockIdx.x == 0 && tid == 0 && p.status_host) publish_status(p.st, p.status_host);
    return;
  }
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    fence_mbar_init();
    s_refined = 0;
  }
  for (int i = p.kpad + tid; i < kp32; i += kThreads) {
    s_fast[i] = make_float4(0.f, 0.f, 0.f, __int_as_float(0x7f800000));
  }
  unsigned long long* s_stats = nullptr;  // this warp's slots
  if (kStats && p.stats_smem_off) {
    unsigned long long* s_all = reinterpret_cast<unsigned long long*>(smem_raw + p.stats_smem_off);
    for (int i = tid; i < (kThreads / 32) * p.stats_slots * 4; i += kThreads) s_all[i] = 0ull;
    s_stats = s_all + (size_t)warp * p.stats_slots * 4;
  }
  __syncthreads();
  if (tid == 0) {
    mbar_expect_tx(&s_bar, (uint32_t)p.kpad * 16u + bkt_bytes);
    tma_load_1d(s_fast, p.table, (uint32_t)p.kpad * 16u, &s_bar);
    if (bkt_bytes) tma_load_1d(s_bkt, p.table + bucket_offset(p.kpad), bkt_bytes, &s_bar);
  }
  const double4* c64 = reinterpret_cast<const double4*>(p.table + exact_offset(p.kpad));
  const float thresh = p.st->thresh;
  const FrameF f = p.f;
  mbar_wait(&s_bar, 0);

  double inert = 0.0;
  unsigned int n_ref = 0;
  int hint = -1;  // many centroids: the previous group's label is the reference of the next one
  const long long n_groups = (p.n + kGroup - 1) / kGroup;
  // every warp owns a contiguous run of groups: neighbours in the raster, so the label of one
  // group is a good reference centroid for the next (bucketed path)
  const long long n_warps = (long long)gridDim.x * (kThreads / 32);
  const long long per_warp = (n_groups + n_warps - 1) / n_warps;
  const long long g_first = ((long long)blockIdx.x * (kThreads / 32) + warp) * per_warp;
  const long long g_last = min(n_groups, g_first + per_warp);
  MapCursor mc{0, 0, 0};
  if ((kMap || kStats) && g_first < g_last) mc = map_cursor(p, g_first * kGroup + lane * 4);
  // few centroids: the next group's block is requested before this one is worked on (one group
  // of look-ahead in registers) -- a warp walks its run serially, so without it every group pays
  // a DRAM round trip.  With many centroids the pass is bound by the candidate walk instead and
  // the registers are better spent there.
  constexpr bool kAhead = kChunks > 0;
  float4 nx = make_float4(0.f, 0.f, 0.f, 0.f), ny = nx, nz = nx;
  if (kAhead && g_first < g_last) {
    const float* blk = p.pts + g_first * kBlockFloats + lane * 4;
    nx = ldg_stream_f4(blk); ny = ldg_stream_f4(blk + kGroup); nz = ldg_stream_f4(blk + 2 * kGroup);
  }
  for (long long g = g_first; g < g_last; ++g) {
    float4 vx, vy, vz;
    if (kAhead) {
      vx = nx; vy = ny; vz = nz;
      if (g + 1 < g_last) {
        const float* blk = p.pts + (g + 1) * kBlockFloats + lane * 4;
        nx = ldg_stream_f4(blk); ny = ldg_stream_f4(blk + kGroup); nz = ldg_stream_f4(blk + 2 * kGroup);
      }
    } else {
      const float* blk = p.pts + g * kBlockFloats + lane * 4;
      vx = ldg_stream_f4(blk); vy = ldg_stream_f4(blk + kGroup); vz = ldg_stream_f4(blk + 2 * kGroup);
    }
    const float xo[4] = {vx.x, vx.y, vx.z, vx.w}, yo[4] = {vy.x, vy.y, vy.z, vy.w}, zo[4] = {vz.x, vz.y, vz.z, vz.w};
    const long long i0 = g * kGroup + lane * 4;
    int lab[4];
    // a raster-order group that runs over the end of a row is left to the second loop below
    if (p.split_rows && __shfl_sync(0xffffffffu, yo[0], 0) != __shfl_sync(0xffffffffu, yo[3], 31)) continue;
    const float xc[4] = {xo[0] - f.ox, xo[1] - f.ox, xo[2] - f.ox, xo[3] - f.ox};
    const float yc[4] = {yo[0] - f.oy, yo[1] - f.oy, yo[2] - f.oy, yo[3] - f.oy};
    const float zc[4] = {zo[0] - f.oz, zo[1] - f.oz, zo[2] - f.oz, zo[3] - f.oz};
    int ncand = -1;
    if (kChunks == 0 && bkt_bytes)
      ncand = assign_group_bucketed(xc, yc, zc, xo, yo, zo, f, s_fast, c64, s_bkt, p.k, kp32, thresh, hint,
                                    s_cand + warp * kCandCap, lane, lab, n_ref);
    if (ncand < 0) assign_group<kChunks>(xc, yc, zc, xo, yo, zo, f, s_fast, c64, p.k, kp32, thresh, lane, lab, n_ref);
    hint = __shfl_sync(0xffffffffu, lab[0], 0);
    final_emit<kMap, kStats>(p, c64, f, i0, xo, yo, zo, lab, inert, mc, s_stats, lane);
  }
  // second loop: the groups that run over the end of a raster row (one in W/128), two halves each
  if (p.split_rows) {
    if ((kMap || kStats) && g_first < g_last) mc = map_cursor(p, g_first * kGroup + lane * 4);  // (walks the run again)
    for (long long gb = g_first; gb < g_last; gb += 32) {
      bool sp = false;
      if (gb + lane < g_last) {
        const float* ys = p.pts + (gb + lane) * kBlockFloats + kGroup;
        sp = __ldg(ys) != __ldg(ys + kGroup - 1);
      }
      unsigned int todo = __ballot_sync(0xffffffffu, sp);
      while (todo) {  // warp-uniform
        const long long g = gb + __ffs(todo) - 1;
        todo &= todo - 1;
        const float* blk = p.pts + g * kBlockFloats + lane * 4;
        const float4 vx = ldg_stream_f4(blk), vy = ldg_stream_f4(blk + kGroup), vz = ldg_stream_f4(blk + 2 * kGroup);
        const float xo[4] = {vx.x, vx.y, vx.z, vx.w}, yo[4] = {vy.x, vy.y, vy.z, vy.w}, zo[4] = {vz.x, vz.y, vz.z, vz.w};
        int lab[4] = {0, 0, 0, 0};
        assign_split_group<kChunks>(xo, yo, zo, f, s_fast, c64, bkt_bytes ? s_bkt : nullptr, p.k, kp32, thresh,
                                    s_cand + warp * kCandCap, lane, lab, n_ref);
        final_emit<kMap, kStats>(p, c64, f, g * kGroup + lane * 4, xo, yo, zo, lab, inert, mc, s_stats, lane);
      }
    }
  }
  const double bsum = block_sum_fixed(inert, s_red);
  n_ref = __reduce_add_sync(0xffffffffu, n_ref);
  if (lane == 0 && n_ref) atomicAdd(&s_refined, n_ref);
  __syncthreads();
  if (s_stats) {  // (block_sum_fixed synchronised the CTA: every point is in the warps' slots)
    const unsigned long long* s_all = reinterpret_cast<const unsigned long long*>(smem_raw + p.stats_smem_off);
    const int words = p.stats_slots * 4;
    for (int i = tid; i < words; i += kThreads) {
      unsigned long long v = 0ull;
      for (int w = 0; w < kThreads / 32; ++w) v += s_all[w * words + i];
      if (v) atomicAdd(&p.stats_acc[i], v);
    }
  }
  if (tid == 0) {
    p.partials[blockIdx.x] = bsum;
    if (s_refined) atomicAdd(&p.st->n_refined, (unsigned long long)s_refined);
    __threadfence();
    const unsigned int t = atomicAdd(p.ticket, 1u);
    s_last = (t == gridDim.x - 1);
  }
  __syncthreads();
  if (s_last) {
    // last CTA: add the per-CTA partials in CTA-index order (deterministic)
    __threadfence();
    double v = 0.0;
    for (int i = tid; i < (int)gridDim.x; i += kThreads) v += p.partials[i];
    const double tot = block_sum_fixed(v, s_red);
    if (p.centroids_host) {
      for (int j = tid; j < p.k; j += kThreads) {
        const double4 c = c64[j];
        p.centroids_host[3 * j + 0] = c.x + p.origin[0];
        p.centroids_host[3 * j + 1] = c.y + p.origin[1];
        p.centroids_host[3 * j + 2] = c.z + p.origin[2];
      }
    }
    if (tid == 0) {
      p.st->inertia = tot;
      *p.ticket = 0u;
      if (p.status_host) publish_status(p.st, p.status_host);
    }
  }
}

}  // namespace mdkm
