// libmdkm.so -- host side of the C ABI declared in include/mdkm.h.
// One handle = one B200 = one rank.  All arithmetic runs in the CUDA kernels of lloyd.cuh /
// unproject.cuh / extras.cuh; this file only allocates, sequences launches and moves bytes.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cstdlib>
#include <string>
#include <map>
#include <utility>
#include <vector>

#include "../../include/mdkm.h"
#include "common.cuh"
#include "extras.cuh"
#include "levelling.cuh"
#include "lloyd.cuh"
#include "mirror.cuh"
#include "nccl_shim.h"
#include "region_adjacency.cuh"
#include "region_overlaps.cuh"
#include "regions.cuh"
#include "seeding.cuh"
#include "tracks.cuh"
#include "transitions.cuh"
#include "unproject.cuh"

using namespace mdkm;

namespace {

constexpr int kBatch = 10;                          // Lloyd iterations enqueued between status polls
constexpr size_t kMappedBytes = 256 << 10;          // device-visible host buffer for small results
constexpr int kMaxOvPairs = 8192;                   // day pairs of region overlaps (their bounds: one small copy)
constexpr int kMaxTrackDays = 16384;                // days of a stack with tracks: their D - 1 consecutive pairs are
                                                    // counted with the caller's, and all the bounds share that copy
static_assert((2 + kMaxOvPairs + kMaxTrackDays) * 8 <= kMappedBytes, "overlap bounds exceed the small result buffer");

// copies `bytes` (a multiple of 4) from device memory into device-visible host memory
__global__ void publish_kernel(void* dst_host, const void* src, int bytes) {
  const int n4 = bytes >> 2;
  for (int i = threadIdx.x; i < n4; i += blockDim.x)
    reinterpret_cast<unsigned int*>(dst_host)[i] = reinterpret_cast<const unsigned int*>(src)[i];
  __threadfence_system();
}

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;  // elements
};

// The outputs bound for the next fit / predict.  Each mdkm_bind_* call clears and sets its own
// part; the next fit / predict moves the whole struct out (take_outputs), so every binding is
// consumed by that call whatever happens.
struct OutputBindings {
  // cluster map (mdkm_bind_cluster_map)
  void* map = nullptr;
  int map_elem = 0, map_mem = MDKM_MEM_HOST;
  // per-(day, cluster) statistics (mdkm_bind_day_stats)
  int64_t* counts = nullptr;
  double* means = nullptr;
  int stats_kcap = 0;
  // day-pair transition counts (mdkm_bind_day_transitions)
  std::vector<int> pairs;  // [n_pairs][2] days, copied when bound
  int64_t* trans = nullptr;
  int trans_kcap = 0;
  // connected regions (mdkm_bind_regions)
  int regions = 0;  // connectivity 4 or 8; 0: not bound
  int32_t* region_map = nullptr;
  int region_map_mem = MDKM_MEM_HOST;
  // region overlaps (mdkm_bind_region_overlaps)
  std::vector<int> ov_pairs;  // [n_pairs][2] days, copied when bound; empty: not bound
  // object tracks (mdkm_bind_tracks)
  double track_iou = 0.0;  // min_iou; 0: not bound
  int32_t* track_map = nullptr;
  int track_map_mem = MDKM_MEM_HOST;
  // region adjacency (mdkm_bind_region_adjacency)
  bool adjacency = false;
};

}  // namespace

struct mdkm_handle {
  int device = 0;
  int sm_count = 148;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;

  // resident cloud (SoA, capacity padded to the tile)
  DevBuf<float> pts;  // blocked cloud (common.cuh), capacity = whole 128-point blocks
  long long n = 0;        // points on this rank
  long long n_total = 0;  // points over all ranks
  long long rank_offset = 0;            // global index of this rank's first point
  std::vector<long long> shard_sizes;   // points per rank (valid with the frame)
  bool have_points = false;
  bool frame_ok = false;
  Frame fr{};
  FrameF ff{};
  double mean[3] = {0, 0, 0};
  bool mean_ok = false;

  // k-means state
  DevBuf<unsigned char> labels;  // uint8 / uint16 per point
  DevBuf<unsigned char> table;
  DevBuf<unsigned long long> acc;
  DevBuf<int> labels32;
  DevBuf<double> dscratch;    // init / centroid read-back / sums
  DevBuf<double> partials;    // inertia / moments partials
  DevBuf<unsigned int> uscratch;  // tickets, minmax
  DevBuf<unsigned long long> reloc;  // relocation scratch
  DevBuf<unsigned char> gsum;        // GroupSummary per 128-point group (static per cloud + frame)
  DevBuf<unsigned char> ssum;        // SuperSummary per kSuper groups
  DevBuf<int> glabel;                // per group: uniform label or -1
  DevBuf<int> worklist;              // [n_groups] + 1 counter at the end
  bool summary_ok = false;
  bool ssum_ok = false;  // super-group summaries built for the current mirror
  // tile-ordered mirror of the cloud (mirror.cuh): what the Lloyd iterations stream
  DevBuf<float> tpts;
  int raster_w = 0;  // width of the raster the cloud was unprojected from (0: generic cloud)
  DevBuf<unsigned int> cell_counts;
  DevBuf<long long> cell_offsets;
  // raster clouds (mdkm_unproject of whole rows): run table written by the unprojection, and the
  // run list / group index the raster mirror build derives from it (mirror.cuh)
  DevBuf<unsigned int> run_src;
  bool runs_ok = false;
  long long run_row0 = 0, run_rows = 0;  // first global row (day * H + y) and number of rows of the range
  int run_H = 0;
  DevBuf<unsigned char> druns;
  DevBuf<unsigned int> gfirst;
  DevBuf<unsigned long long> index_status;  // raster_index_kernel: ticket + fault flag, look-back words
  int opt_raster_mirror = 1;  // MDKM_OPT_RASTER_MIRROR
  int opt_cell_px = 0, opt_cell_rows = 0;  // MDKM_OPT_CELL_PX / MDKM_OPT_CELL_ROWS (0 = automatic)
  int opt_two_level = -1;                  // MDKM_OPT_TWO_LEVEL (-1 = automatic)
  int opt_pdl = 1;                         // MDKM_OPT_DEPENDENT_LAUNCH
  float bounds[6] = {0, 0, 0, 0, 0, 0};  // global min x,y,z / max x,y,z of the cloud
  DevStatus* d_status = nullptr;
  DevStatus* h_status = nullptr;  // pinned, 2 slots
  cudaEvent_t batch_ev[2] = {nullptr, nullptr};
  int last_k = 0;
  int occ_k = -1, occ_step = 0, occ_final = 0;  // occupancy of the step / final kernels for occ_k clusters
  long long stat_refined = 0, stat_reloc = 0, stat_work = 0, stat_groups = 0;
  double stat_tol = 0.0;
  int opt_settle = 1;  // MDKM_OPT_SETTLE_GROUPS

  // unprojection scratch
  DevBuf<long long> chunk_offsets;
  DevBuf<unsigned long long> tile_status;  // look-back words of the fused unprojection pass (+ its ticket)
  DevBuf<unsigned char> staging;  // host inputs staged here
  DevBuf<double> planes;
  long long* h_total = nullptr;  // pinned

  // segments of the resident cloud (one per day of the unprojected range; one for set_points)
  std::vector<long long> seg_off;  // [n_seg + 1] point offsets
  bool seg_whole = false;          // every segment is a whole day / the whole cloud
  DevBuf<long long> d_seg_off;
  DevBuf<unsigned int> sel_hist;
  DevBuf<unsigned char> sel_targets;

  // k-means++ state
  DevBuf<double> kpp_closest, kpp_cell, kpp_blk, kpp_prefix, kpp_partials, kpp_rand;
  DevBuf<unsigned char> kpp_state;

  // small device->host results (status words, totals, centroids) never use the copy engine --
  // it may be busy for milliseconds with a bulk result copy -- but are written by a tiny
  // kernel straight into this page-locked, device-visible (UVA) host buffer
  unsigned char* mapped = nullptr;
  size_t mapped_used = 0;
  struct SmallCopy { void* dst; size_t off, bytes; };
  std::vector<SmallCopy> small_pending;

  // asynchronous result copies (cloud): side stream + staging that outlives the call
  cudaStream_t d2h_stream = nullptr;
  cudaEvent_t ev_ready = nullptr;   // compute stream -> d2h stream
  bool d2h_pending = false;
  DevBuf<float> cloud_aos;
  // slab pipeline of mdkm_unproject: H2D copies on their own stream, per-slab events
  cudaStream_t h2d_stream = nullptr;
  std::vector<cudaEvent_t> slab_ev;
  DevBuf<long long> slab_totals;     // [n_slabs + 1] running point totals (device)
  long long* h_slab_totals = nullptr;  // pinned mirror
  size_t h_slab_cap = 0;
  float* bound_cloud_out = nullptr;  // mdkm_bind_cloud_output
  long long bound_cloud_cap = 0;
  int bound_cloud_napari = 1;
  OutputBindings bound;              // the outputs of the next fit / predict
  // cluster map (mdkm_bind_cluster_map) over the pixel range of the last mdkm_unproject
  long long raster_pix_begin = 0, raster_pix_count = 0;
  int raster_H = 0;                  // (the width is raster_w)
  DevBuf<unsigned char> map_stage;   // host outputs are written here, then copied
  DevBuf<long long> map_seg;         // the days' point offsets (d_seg_off may hold merged segments)
  // per-(day, cluster) statistics (mdkm_bind_day_stats) of the next fit / predict
  int stack_days = 0;                // days of the stack of the last mdkm_unproject (1 after mdkm_set_points)
  long long day0 = 0;                // global day of the resident cloud's first segment
  DevBuf<unsigned long long> stats_acc;  // [days * k * 4] (qx, qy, qz, count) per slot
  DevBuf<unsigned char> stats_dev;       // counts, then means, converted on the device
  unsigned char* stats_host = nullptr;   // pinned: their copy, handed to the caller after the sync
  size_t stats_host_cap = 0;
  // day-pair transition counts (mdkm_bind_day_transitions) of the next fit / predict
  DevBuf<int> trans_pairs;
  DevBuf<unsigned long long> trans_bins;  // [n_pairs][(k+1)^2]
  unsigned char* trans_host = nullptr;    // pinned: their copy, handed to the caller after the sync
  size_t trans_host_cap = 0;
  // the whole-stack cluster map that day transitions and regions read (take_stack_map)
  int stack_cover = -1;                  // the ranks' pixel ranges cover the stack (1) or not (0); -1: not checked
  DevBuf<unsigned char> stack_map;       // the map the final pass writes when none is bound; the whole stack with
                                         // several ranks
  // connected regions of the cluster map (mdkm_bind_regions) of the next fit / predict, and those
  // of the last fit / predict that had them, kept on the device until the next unproject /
  // set_points / fit or predict with regions
  DevBuf<int> region_parent;             // [stack pixels] union-find parents
  DevBuf<int> region_ids;                // [stack pixels] region map of the whole stack
  DevBuf<unsigned long long> region_scan;  // look-back words of the numbering, then ticket + fault, then R
  DevBuf<unsigned long long> region_acc;   // [R][4] (qx, qy, qz, count)
  DevBuf<unsigned int> region_box;         // [R][5] first pixel, y_min, x_min, ~y_max, ~x_max
  DevBuf<unsigned char> region_out;        // table int64 [R][7], then means float64 [R][3]
  long long n_regions = -1;              // R of the last fit / predict with regions; -1: none
  // region overlaps between days (mdkm_bind_region_overlaps) of the next fit / predict, and those
  // of the last fit / predict that had them, with the lifecycle of the regions
  DevBuf<int> ov_pairs;
  DevBuf<long long> ov_tab;              // [n_pairs + 1] slot offsets of the pairs' hash tables
  DevBuf<unsigned long long> ov_slots;   // [slots][2] key, count | ~first << 32
  DevBuf<unsigned int> ov_bits;          // first-pixel masks, then word offsets within the scan chunks
  DevBuf<unsigned long long> ov_scan;    // look-back words, chunk offsets, ticket + fault, M, probe fault
  DevBuf<long long> ov_rows;             // int64 [M][6]
  long long n_overlaps = -1;             // M of the last fit / predict with overlaps; -1: none
  // object tracks (mdkm_bind_tracks) of the next fit / predict, and those of the last fit / predict
  // that had them, with the lifecycle of the regions
  DevBuf<int> track_link_day;            // [counted pairs] d of the counted pair (d, d+1), else -1
  DevBuf<int> track_parent;              // [R] union-find parents (region index)
  DevBuf<unsigned int> track_links;      // [2R] links forward, then backward
  DevBuf<int> track_ids;                 // [R] track of each region (region_tracks)
  DevBuf<unsigned long long> track_scan; // look-back words of the numbering, ticket + fault, T, caller's M
  DevBuf<long long> track_tab;           // int64 [R][7]: the first T rows are the track table
  DevBuf<int> track_stage;               // a host track map is written here, then copied
  long long n_tracks = -1;               // T of the last fit / predict with tracks; -1: none
  // region adjacency within a day (mdkm_bind_region_adjacency) of the next fit / predict, and that
  // of the last fit / predict that had it, with the lifecycle of the regions
  DevBuf<long long> adj_tab;             // [D + 1] slot offsets of the days' hash tables
  DevBuf<unsigned long long> adj_slots;  // [slots][2] key, count | ~first edge << 32
  DevBuf<unsigned int> adj_bits;         // first-edge masks, then word offsets within the scan chunks
  DevBuf<unsigned long long> adj_scan;   // look-back words, chunk offsets, ticket + fault, M, probe fault
  DevBuf<long long> adj_rows;            // int64 [M][6]
  DevBuf<unsigned long long> adj_sides;  // int64 [R][4] region boundaries
  unsigned char* adj_bounds = nullptr;   // pinned: the days' bounds, read with R
  size_t adj_bounds_cap = 0;
  long long n_adjacency = -1;            // M of the last fit / predict with adjacency; -1: none

  // communicator
  ncclComm_t comm = nullptr;
  int n_ranks = 1, rank = 0;
  // NVLink peer exchange of the partial sums (CUDA IPC): own buffer, peers' mappings
  unsigned long long* xchg = nullptr;
  void* peer_base[kMaxRanks] = {};  // mappings opened with cudaIpcOpenMemHandle (closed by close_p2p)
  PeerXchg px{};
  bool p2p_ok = false;
  unsigned long long epoch_base = 0;  // fused steps completed on this communicator
  int step_seq = 0;                   // fused step launches since the last settle kernel (StepParams::seq)
  size_t settle_smem = 0;
  std::map<const void*, int> occ_cache;  // resident CTAs per SM of the grid-stride kernels

  // profiling: CUDA-event spans around the kernels of a phase (mdkm_profile_*)
  bool prof = false;
  std::vector<cudaEvent_t> prof_ev;  // pool, two per span
  struct ProfSpan { int phase; long long count; };
  std::vector<ProfSpan> prof_spans;
  double prof_ms[MDKM_PHASE_COUNT] = {};
  long long prof_count[MDKM_PHASE_COUNT] = {};
  int launches = 0;
};

namespace {

int fail(mdkm_handle* h, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (h) h->err = buf;
  return code;
}

#define CU(call)                                                                              \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return fail(h, e__ == cudaErrorMemoryAllocation ? MDKM_ERR_OOM : MDKM_ERR_CUDA,         \
                  "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

#define NC(call)                                                                               \
  do {                                                                                         \
    ncclResult_t r__ = (call);                                                                 \
    if (r__ != 0)                                                                              \
      return fail(h, MDKM_ERR_NCCL, "%s failed: %s", #call,                                    \
                  nccl_api().GetErrorString ? nccl_api().GetErrorString(r__) : "nccl error");  \
  } while (0)

#define OK(call)              \
  do {                        \
    int rc__ = (call);        \
    if (rc__ != MDKM_OK) return rc__; \
  } while (0)

// Enqueue a small device->host result on the compute stream without the copy engine.
// `pinned_dst` (optional) is a page-locked destination written directly; otherwise the bytes
// land in the handle's mapped buffer and sync_small() hands them to `dst`.
int small_d2h(mdkm_handle* h, void* dst, const void* dev_src, size_t bytes, bool dst_is_pinned = false) {
  if (bytes == 0) return MDKM_OK;
  if (bytes % 4 != 0) return fail(h, MDKM_ERR_INVALID, "small_d2h: size must be a multiple of 4");
  void* target = dst;
  if (!dst_is_pinned) {
    const size_t off = (h->mapped_used + 15) & ~(size_t)15;
    if (off + bytes > kMappedBytes) return fail(h, MDKM_ERR_INVALID, "small result buffer exhausted");
    target = h->mapped + off;
    h->mapped_used = off + bytes;
    h->small_pending.push_back({dst, off, bytes});
  }
  publish_kernel<<<1, 256, 0, h->stream>>>(target, dev_src, (int)bytes);
  CU(cudaGetLastError());
  return MDKM_OK;
}

// Synchronise the compute stream and deliver the pending small results.
int sync_small(mdkm_handle* h) {
  CU(cudaStreamSynchronize(h->stream));
  for (const auto& c : h->small_pending) memcpy(c.dst, h->mapped + c.off, c.bytes);
  h->small_pending.clear();
  h->mapped_used = 0;
  return MDKM_OK;
}

template <typename T>
int ensure(mdkm_handle* h, DevBuf<T>& b, size_t elems) {
  if (b.cap >= elems && b.p) return MDKM_OK;
  if (b.p) {
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
  }
  if (elems == 0) elems = 1;
  CU(cudaMalloc(&b.p, elems * sizeof(T)));
  b.cap = elems;
  return MDKM_OK;
}

template <typename T>
void release(DevBuf<T>& b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr;
  b.cap = 0;
}

inline long long round_up(long long v, long long m) { return (v + m - 1) / m * m; }

int prof_begin(mdkm_handle* h, int phase, long long count);
void prof_end(mdkm_handle* h, int idx);

int grid_for(const mdkm_handle* h, long long work_items, int per_sm) {
  long long g = std::min<long long>(work_items, (long long)h->sm_count * per_sm);
  return (int)std::max<long long>(1, g);
}

// CTAs of `fn` (kThreads threads, `smem` bytes of dynamic shared memory) that are resident on one SM
// at a time, as the runtime reports it (cached per kernel).  Grid-stride kernels are launched as ONE
// full wave: a grid of 8 CTAs per SM for a kernel of which 6 fit runs a second, one-third-full wave
// at a fraction of the bandwidth (raster_gather_kernel: 213 -> 19x us on config 2).
template <typename Kernel>
int resident_per_sm(mdkm_handle* h, Kernel fn, size_t smem = 0) {
  const void* key = reinterpret_cast<const void*>(fn);
  auto it = h->occ_cache.find(key);
  if (it != h->occ_cache.end()) return it->second;
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, kThreads, smem) != cudaSuccess || occ < 1) {
    cudaGetLastError();
    occ = 4;
  }
  h->occ_cache[key] = occ;
  return occ;
}

// Blocks until the asynchronous result copies issued so far have landed in host memory.
int wait_pending(mdkm_handle* h) {
  if (h->d2h_pending) {
    CU(cudaStreamSynchronize(h->d2h_stream));
    h->d2h_pending = false;
  }
  return MDKM_OK;
}

void close_p2p(mdkm_handle* h) {
  for (int q = 0; q < kMaxRanks; ++q)
    if (h->peer_base[q]) {
      cudaIpcCloseMemHandle(h->peer_base[q]);
      h->peer_base[q] = nullptr;
    }
  if (h->xchg) cudaFree(h->xchg);
  h->xchg = nullptr;
  h->p2p_ok = false;
  h->px = PeerXchg{};
  h->epoch_base = 0;
}

int alloc_points(mdkm_handle* h, long long n) {
  const size_t cap = (size_t)round_up(std::max<long long>(n, 1), kGroup);
  OK(ensure(h, h->pts, cap * 3));
  return MDKM_OK;
}

// zero the unused tail of the last block so that it only loosens that group's bounding box
int zero_tail(mdkm_handle* h) {
  if (h->n % kGroup != 0 || h->n == 0) {
    if (h->n == 0) {
      CU(cudaMemsetAsync(h->pts.p, 0, kBlockFloats * 4, h->stream));
    } else {
      zero_tail_kernel<<<1, 128, 0, h->stream>>>(h->pts.p, h->n);
      ++h->launches;
      CU(cudaGetLastError());
    }
  }
  return MDKM_OK;
}

int allreduce(mdkm_handle* h, void* buf, size_t count, int dtype, int op) {
  if (h->n_ranks <= 1) return MDKM_OK;
  NC(nccl_api().AllReduce(buf, buf, count, dtype, op, h->comm, h->stream));
  return MDKM_OK;
}

// Frame of the resident cloud: origin / fixed-point scale / half-range from the global
// per-dimension min and max.
// `minmax_ready`: uscratch[4..9] already holds the ordered min / max of the points (the fused
// unprojection pass collects them while it writes the cloud).
int compute_frame(mdkm_handle* h, bool minmax_ready = false) {
  OK(ensure(h, h->uscratch, 16));
  OK(ensure(h, h->dscratch, 64 + (size_t)h->n_ranks));
  unsigned int init[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};
  if (!minmax_ready) CU(cudaMemcpyAsync(h->uscratch.p + 4, init, sizeof(init), cudaMemcpyHostToDevice, h->stream));
  if (h->n > 0 && !minmax_ready) {
    minmax_kernel<<<grid_for(h, (h->n + 1023) / 1024, resident_per_sm(h, minmax_kernel)), kThreads, 0, h->stream>>>(h->pts.p, h->n,
                                                                                     h->uscratch.p + 4);
    ++h->launches;
    CU(cudaGetLastError());
  }
  unsigned int ord[6];
  OK(small_d2h(h, ord, h->uscratch.p + 4, sizeof(ord)));
  OK(sync_small(h));
  float mm[6];
  for (int i = 0; i < 6; ++i) mm[i] = ord2f(ord[i]);
  long long ntot = h->n;
  h->shard_sizes.assign((size_t)h->n_ranks, 0);
  h->shard_sizes[h->rank] = h->n;
  h->rank_offset = 0;
  if (h->n_ranks > 1) {
    // exchange min / max / shard sizes (tiny, once per cloud)
    float* dmm = reinterpret_cast<float*>(h->dscratch.p);
    long long* dn = reinterpret_cast<long long*>(h->dscratch.p + 8);
    CU(cudaMemcpyAsync(dmm, mm, sizeof(mm), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(dn, h->shard_sizes.data(), 8 * (size_t)h->n_ranks, cudaMemcpyHostToDevice, h->stream));
    OK(allreduce(h, dmm, 3, kNcclFloat32, kNcclMin));
    OK(allreduce(h, dmm + 3, 3, kNcclFloat32, kNcclMax));
    OK(allreduce(h, dn, h->n_ranks, kNcclInt64, kNcclSum));
    OK(small_d2h(h, mm, dmm, sizeof(mm)));
    OK(small_d2h(h, h->shard_sizes.data(), dn, 8 * (size_t)h->n_ranks));
    OK(sync_small(h));
    ntot = 0;
    for (int r = 0; r < h->n_ranks; ++r) {
      if (r == h->rank) h->rank_offset = ntot;
      ntot += h->shard_sizes[r];
    }
  }
  h->n_total = ntot;
  for (int i = 0; i < 6; ++i) h->bounds[i] = mm[i];
  for (int d = 0; d < 3; ++d) {
    double lo = mm[d], hi = mm[3 + d];
    if (!(lo <= hi)) { lo = 0.0; hi = 0.0; }  // empty cloud
    if (!isfinite(lo) || !isfinite(hi)) return fail(h, MDKM_ERR_INVALID, "points contain non-finite coordinates");
    // origin: midrange rounded to an integer (exactly representable in FP32, makes pixel
    // coordinates exact); kept at 0 when that would not shorten the range noticeably.
    double mid = 0.5 * (lo + hi);
    double half = 0.5 * (hi - lo);
    double o = (fabs(mid) > 0.25 * half) ? nearbyint(mid) : 0.0;
    o = (double)(float)o;
    // A cloud narrower than a unit and away from an integer (extent 1e-3 around 0.5): the integer
    // origin would leave a half-range of up to 0.5 and a quantum set by it instead of by the
    // extent.  Then the origin is a multiple of the largest power of two not above the half-range
    // (half-range below 1.5x the cloud's), provided x - o stays exact in FP32: that step is no
    // finer than the ulp of the largest |x| (x - o is a multiple of the ulp of x) and every |x|
    // exceeds the new half-range (so x - o needs no more bits than x).
    if (half > 0.0 && fabs(mid - o) > half) {
      const double step = ldexp(1.0, ilogb(half));
      const double o2 = nearbyint(mid / step) * step;
      const double hr2 = std::max(fabs(lo - o2), fabs(hi - o2));
      const double amin = lo > 0.0 ? lo : (hi < 0.0 ? -hi : 0.0);
      const double amax = std::max(fabs(lo), fabs(hi));
      const double ulp_max = ldexp(1.0, ilogb(amax) - 23);
      if (hr2 < amin && step >= ulp_max && (double)(float)o2 == o2) o = o2;
    }
    double hr = std::max(fabs(lo - o), fabs(hi - o));
    hr = hr * (1.0 + 1e-6) + 1e-30;  // FP32 rounding of x - o
    int e = (int)floor(log2((double)((1 << kQuantBits) - 2) / hr));
    e = std::max(-100, std::min(100, e));
    h->fr.origin[d] = o;
    h->fr.scale[d] = ldexp(1.0, e);
    h->fr.halfrange[d] = hr;
  }
  h->ff.ox = (float)h->fr.origin[0]; h->ff.oy = (float)h->fr.origin[1]; h->ff.oz = (float)h->fr.origin[2];
  h->ff.sx = (float)h->fr.scale[0]; h->ff.sy = (float)h->fr.scale[1]; h->ff.sz = (float)h->fr.scale[2];
  h->frame_ok = true;
  h->mean_ok = false;
  h->summary_ok = false;
  return MDKM_OK;
}

// mean and mean(var) of the global cloud (sklearn/_kmeans.py:285-293 and :1487-1490)
int compute_moments(mdkm_handle* h, double* mean_var_out) {
  const int g = grid_for(h, (h->n + 1023) / 1024, 4);
  OK(ensure(h, h->partials, (size_t)std::max(g, h->sm_count * 8) * 8 + 16));
  OK(ensure(h, h->uscratch, 16));
  OK(ensure(h, h->dscratch, 64));
  CU(cudaMemsetAsync(h->uscratch.p, 0, 4, h->stream));
  CU(cudaMemsetAsync(h->dscratch.p, 0, 8 * sizeof(double), h->stream));
  if (h->n > 0) {
    moments_kernel<<<g, kThreads, 0, h->stream>>>(h->pts.p, h->n, h->ff, h->partials.p, h->uscratch.p,
                                                  h->dscratch.p);
    ++h->launches;
    CU(cudaGetLastError());
  }
  OK(allreduce(h, h->dscratch.p, 6, kNcclFloat64, kNcclSum));
  double m[6];
  OK(small_d2h(h, m, h->dscratch.p, sizeof(m)));
  OK(sync_small(h));
  const double N = (double)std::max<long long>(h->n_total, 1);
  double mv = 0.0;
  for (int d = 0; d < 3; ++d) {
    const double mu = m[d] / N;
    h->mean[d] = mu + h->fr.origin[d];
    mv += m[3 + d] / N - mu * mu;
  }
  h->mean_ok = true;
  if (mean_var_out) *mean_var_out = mv / 3.0;
  return MDKM_OK;
}

// Step-kernel variants: label width x accumulator slices x compile-time table chunks.
typedef void (*StepKernel)(const StepParams);
StepKernel pick_step_kernel(bool wide, bool priv, int kpad) {
  const int chunks = kpad <= 32 ? 1 : (kpad <= 64 ? 2 : 0);
  if (wide) return lloyd_step_kernel<unsigned short, false, 0>;
  if (priv) {
    if (chunks == 1) return lloyd_step_kernel<unsigned char, true, 1>;
    if (chunks == 2) return lloyd_step_kernel<unsigned char, true, 2>;
    return lloyd_step_kernel<unsigned char, true, 0>;
  }
  return lloyd_step_kernel<unsigned char, false, 0>;
}

int step_occupancy(mdkm_handle* h, StepKernel fn, size_t smem, int* occ) {
  CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, fn, kThreads, smem));
  return MDKM_OK;
}

typedef void (*FinalKernel)(const FinalParams);
template <bool kMap, bool kStats>
FinalKernel pick_final_chunks(int kpad) {
  if (kpad <= 32) return lloyd_final_kernel<1, kMap, kStats>;
  if (kpad <= 64) return lloyd_final_kernel<2, kMap, kStats>;
  return lloyd_final_kernel<0, kMap, kStats>;
}
FinalKernel pick_final_kernel(int kpad, bool map = false, bool stats = false) {
  if (stats) return map ? pick_final_chunks<true, true>(kpad) : pick_final_chunks<false, true>(kpad);
  return map ? pick_final_chunks<true, false>(kpad) : pick_final_chunks<false, false>(kpad);
}

struct KmBuffers {
  int k, kpad;
  size_t step_smem, final_smem;
  int step_grid, final_grid;
  bool wide;     // uint16 labels
  bool priv;     // per-warp accumulator slices in shared memory
  bool two_level;  // classification pass walks super-groups first
  StepKernel step_fn;
  FinalKernel final_fn;
  long long n_groups;
};

// Re-orders the resident cloud, segment by segment, by the cells of an x-y grid (about 256
// points per cell) into h->tpts; see mirror.cuh.  Once per (cloud, frame).
int build_mirror(mdkm_handle* h, int cell_px) {
  const long long cap = round_up(std::max<long long>(h->n, 1), kGroup);
  OK(ensure(h, h->tpts, (size_t)cap * 3));
  CU(cudaMemsetAsync(h->tpts.p + (cap - kGroup) * 3, 0, kBlockFloats * 4, h->stream));  // tail of the last block
  if (h->n == 0) return MDKM_OK;
  // segments: the days of the unprojected range (merged into one when there are too many)
  std::vector<long long> seg = h->seg_off;
  if (seg.size() < 2 || seg.back() != h->n || (int)seg.size() - 1 > kMirrorMaxSeg) seg.assign({0, h->n});
  const int n_seg = (int)seg.size() - 1;
  OK(ensure(h, h->d_seg_off, (size_t)n_seg + 1));
  CU(cudaMemcpyAsync(h->d_seg_off.p, seg.data(), (size_t)(n_seg + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  const double xr = std::max((double)h->bounds[3] - (double)h->bounds[0], 1e-30);
  const double yr = std::max((double)h->bounds[4] - (double)h->bounds[1], 1e-30);
  const double target = std::max(1.0, (double)h->n / 256.0);  // cells (each holds points of every segment)
  long long gx = (long long)llround(sqrt(target * xr / yr));
  // raster clouds: cells a fixed number of pixels wide, so that every row adds a run of that
  // many consecutive points to a cell.  Wider cells are cheaper to build (longer write runs),
  // narrower ones are more compact and leave fewer boundary groups per iteration, which pays
  // once there are many centroids.
  if (h->raster_w > 0) gx = (long long)ceil(xr / (double)cell_px);
  gx = std::max<long long>(1, std::min<long long>(gx, 1 << 15));
  long long gy = (long long)ceil(target / (double)gx);
  gy = std::max<long long>(1, std::min<long long>(gy, 1 << 15));
  if (!(xr > 1e-20)) gx = 1;
  if (!(yr > 1e-20)) gy = 1;
  MirrorGrid g{};
  g.x0 = h->bounds[0]; g.y0 = h->bounds[1];
  g.inv_cx = (float)((double)gx / xr);
  g.inv_cy = (float)((double)gy / yr);
  g.gx = (int)gx; g.gy = (int)gy;
  g.n_seg = n_seg;
  g.seg_off = h->d_seg_off.p;
  const long long n_cells = gx * gy;
  // bands of rows: kMirrorGpb groups of every segment per band
  long long max_groups = 1;
  for (int sgm = 0; sgm < n_seg; ++sgm)
    max_groups = std::max(max_groups, (seg[sgm + 1] + kGroup - 1) / kGroup - (seg[sgm] + kGroup - 1) / kGroup + 1);
  const long long n_bands = (max_groups + kMirrorGpb - 1) / kMirrorGpb;
  g.n_virtual = n_bands * n_seg * kMirrorGpb;
  const int n_tiles = (int)((n_cells + kScanTile - 1) / kScanTile);
  OK(ensure(h, h->cell_counts, (size_t)n_tiles * kScanTile));  // whole tiles: the scan reads 128-bit words
  OK(ensure(h, h->cell_offsets, (size_t)n_cells + 2));
  CU(cudaMemsetAsync(h->cell_counts.p, 0, (size_t)n_cells * 4, h->stream));
  const int grid = grid_for(h, (h->n + 1023) / 1024, 8);
  mirror_count_kernel<<<grid, kThreads, 0, h->stream>>>(h->pts.p, h->n, g, h->cell_counts.p);
  OK(ensure(h, h->partials, (size_t)std::max(n_tiles, h->sm_count * 8) * 8 + 16));
  long long* tile_sums = reinterpret_cast<long long*>(h->partials.p);
  mirror_tile_sums_kernel<<<n_tiles, 1024, 0, h->stream>>>(h->cell_counts.p, n_cells, tile_sums);
  mirror_scan_kernel<<<n_tiles, 1024, 0, h->stream>>>(h->cell_counts.p, n_cells, h->cell_offsets.p, tile_sums);
  ++h->launches;
  // the cells' start offsets become their arrival cursors
  mirror_scatter_kernel<<<grid, kThreads, 0, h->stream>>>(
      h->pts.p, h->n, g, reinterpret_cast<unsigned long long*>(h->cell_offsets.p), h->tpts.p);
  h->launches += 3;
  CU(cudaGetLastError());
  return MDKM_OK;
}

// The same for a raster cloud that came with a run table: cell sizes and the place of every run
// follow from the table (one scan over the runs), the copy is a gather by destination that
// also writes the group summaries.  No histogram pass over the points, no atomics.
int build_mirror_raster(mdkm_handle* h, int cell_px) {
  const long long cap = round_up(std::max<long long>(h->n, 1), kGroup);
  OK(ensure(h, h->tpts, (size_t)cap * 3));
  const long long n_groups = cap / kGroup;
  OK(ensure(h, h->gsum, (size_t)n_groups * sizeof(GroupSummary)));
  RasterGeom g{};
  g.run_src = h->run_src.p;
  g.row0 = h->run_row0; g.n_rows = h->run_rows;
  g.W = h->raster_w; g.H = h->run_H;
  g.nb8 = g.W / 8;
  g.cb = cell_px / 8;
  g.gx = (g.nb8 + g.cb - 1) / g.cb;
  g.d0 = (int)(g.row0 / g.H);
  g.nd = (int)((g.row0 + g.n_rows - 1) / g.H) - g.d0 + 1;
  // rows of y the range covers: all of them once it holds a whole day, else its n_rows rows
  // counted (cyclically) from the first one
  g.yshift = g.n_rows >= g.H ? 0 : (int)(g.row0 % g.H);
  g.yext = (int)std::min<long long>(g.n_rows, g.H);
  // rows per cell: about 400 points per cell (measured optimum of fit time over cell shapes, configs 2-4),
  // counting every day that covers a row
  const double per_row = (double)h->n / (double)g.yext / (double)g.gx;  // points per cell and row of y
  g.rpc = (int)std::max(1.0, std::min(64.0, nearbyint(400.0 / std::max(per_row, 1e-9))));
  if (h->opt_cell_rows > 0) g.rpc = std::min(64, h->opt_cell_rows);
  g.gy = (g.yext + g.rpc - 1) / g.rpc;
  const long long n_cells = (long long)g.gx * g.gy;
  const long long n_entries = n_cells * g.nd * g.rpc;
  if (n_cells >= (1ll << 31) || n_entries + kIndexTile >= (1ll << 32)) return fail(h, MDKM_ERR_INVALID, "raster too large for the run list");
  const long long n_tiles = (n_entries + kIndexTile - 1) / kIndexTile;
  OK(ensure(h, h->druns, ((size_t)n_entries + 1) * sizeof(uint2)));
  OK(ensure(h, h->gfirst, (size_t)n_groups));
  OK(ensure(h, h->index_status, (size_t)n_tiles + 1));  // ticket + fault flag, then the look-back words
  if (h->n == 0) {
    CU(cudaMemsetAsync(h->tpts.p, 0, kBlockFloats * 4, h->stream));
    group_summary_kernel<<<1, kThreads, 0, h->stream>>>(h->tpts.p, h->n, h->ff, reinterpret_cast<GroupSummary*>(h->gsum.p));
    ++h->launches;
    CU(cudaGetLastError());
    return MDKM_OK;
  }
  CU(cudaMemsetAsync(h->index_status.p, 0, ((size_t)n_tiles + 1) * 8, h->stream));
  raster_index_kernel<<<(unsigned int)n_tiles, kThreads, 0, h->stream>>>(
      g, h->n, (unsigned int)n_entries, h->index_status.p + 1, reinterpret_cast<unsigned int*>(h->index_status.p),
      reinterpret_cast<uint2*>(h->druns.p), h->gfirst.p);
  CU(cudaGetLastError());
  // the gather is set up while the index kernel drains (it waits for the whole grid before it reads)
  const uint2* druns = reinterpret_cast<const uint2*>(h->druns.p);
  const unsigned int* gfirst = h->gfirst.p;
  float4* gsum = reinterpret_cast<float4*>(h->gsum.p);
  void* args[] = {&h->pts.p, &h->n, &druns, const_cast<long long*>(&n_entries), &gfirst, &h->ff, &h->tpts.p, &gsum};
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid_for(h, (n_groups + 7) / 8, resident_per_sm(h, raster_gather_kernel)));
  cfg.blockDim = dim3(kThreads);
  cfg.stream = h->stream;
  cudaLaunchAttribute attr;
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = h->opt_pdl ? 1 : 0;
  CU(cudaLaunchKernelExC(&cfg, reinterpret_cast<const void*>(raster_gather_kernel), args));
  h->launches += 2;
  CU(cudaGetLastError());
  return MDKM_OK;
}

// The k x 3 centroids a caller hands in: a NaN or an infinity would go straight into the tables
// (scikit-learn rejects such an init; the points get the same check in compute_frame).
int check_centroids(mdkm_handle* h, int k, const double* c, const char* what) {
  if (k < 1 || k > kMaxK) return fail(h, MDKM_ERR_INVALID, "k must be in [1, %d]", kMaxK);
  for (long long i = 0; i < 3ll * k; ++i)
    if (!isfinite(c[i])) return fail(h, MDKM_ERR_INVALID, "%s row %lld has a non-finite coordinate", what, i / 3);
  return MDKM_OK;
}

int prepare_kmeans(mdkm_handle* h, int k, KmBuffers& kb) {
  if (!h->have_points) return fail(h, MDKM_ERR_STATE, "no points resident: call mdkm_unproject or mdkm_set_points first");
  if (k < 1 || k > kMaxK) return fail(h, MDKM_ERR_INVALID, "k must be in [1, %d]", kMaxK);
  if (!h->frame_ok) OK(compute_frame(h));
  if ((long long)k > h->n_total) return fail(h, MDKM_ERR_INVALID, "n_samples=%lld should be >= n_clusters=%d", h->n_total, k);
  kb.k = k;
  kb.kpad = pad_k(k);
  kb.wide = k > 256;
  const size_t kp32 = (size_t)((kb.kpad + 31) & ~31);
  kb.priv = !kb.wide && kb.kpad <= 128;
  const size_t ring = (size_t)(kThreads / 32) * kStages * (kb.wide ? stage_bytes<unsigned short>() : stage_bytes<unsigned char>());
  kb.step_smem = kp32 * 16 + ring + (size_t)kb.kpad * 32 * (kb.priv ? (kThreads / 32) : 1) + bucket_bytes(k, kb.kpad);
  kb.final_smem = kp32 * 16 + bucket_bytes(k, kb.kpad);
  const long long cap = round_up(std::max<long long>(h->n, 1), kGroup);
  OK(ensure(h, h->labels, (size_t)cap * (kb.wide ? 2 : 1)));
  OK(ensure(h, h->table, 2 * table_bytes(k, kb.kpad)));  // fused launches alternate between two tables
  OK(ensure(h, h->acc, 4 * ((size_t)kb.kpad * 4 + 8)));  // three rotating accumulators + the copy parked on a pause
  OK(ensure(h, h->dscratch, (size_t)std::max(64, k * 4 + 16)));
  OK(ensure(h, h->uscratch, 16));
  const long long tiles = (h->n + kThreads * 4 - 1) / (kThreads * 4);  // 8 warp-groups per CTA pass
  // persistent grids: one full wave of resident CTAs (occupancy queried from the runtime)
  int occ_step = 1, occ_final = 1;
  kb.step_fn = pick_step_kernel(kb.wide, kb.priv, kb.kpad);
  kb.final_fn = pick_final_kernel(kb.kpad);
  if (h->occ_k == k) {  // same kernels and shared-memory sizes as the last fit on this handle
    occ_step = h->occ_step;
    occ_final = h->occ_final;
  } else {
    OK(step_occupancy(h, kb.step_fn, kb.step_smem, &occ_step));
    CU(cudaFuncSetAttribute(kb.final_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kb.final_smem));
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_final, kb.final_fn, kThreads, kb.final_smem));
    h->occ_k = k;
    h->occ_step = occ_step;
    h->occ_final = occ_final;
  }
  if (occ_step < 1) return fail(h, MDKM_ERR_INVALID, "k=%d does not fit the shared-memory tables", k);
  kb.step_grid = grid_for(h, tiles, std::max(1, occ_step));
  kb.final_grid = grid_for(h, tiles, std::max(1, occ_final));
  OK(ensure(h, h->partials, (size_t)std::max(kb.final_grid, h->sm_count * 8) * 8 + 16));
  // group summaries for the classification pass
  kb.n_groups = cap / kGroup;
  OK(ensure(h, h->gsum, (size_t)kb.n_groups * sizeof(GroupSummary)));
  const long long n_super = (kb.n_groups + kSuper - 1) / kSuper;
  OK(ensure(h, h->ssum, (size_t)n_super * sizeof(SuperSummary)));
  OK(ensure(h, h->glabel, (size_t)n_super * kSuper));  // (whole super-groups: read eight at a time)
  OK(ensure(h, h->worklist, (size_t)kb.n_groups + 4));
  if (!h->summary_ok) {
    const int span = prof_begin(h, MDKM_PHASE_BUILD, h->n);
    if (h->runs_ok && h->raster_w > 0 && h->opt_raster_mirror) {
      int cell_px = k <= 16 && h->raster_w % 16 == 0 ? 16 : 8;
      if (h->opt_cell_px == 8 || (h->opt_cell_px == 16 && h->raster_w % 16 == 0)) cell_px = h->opt_cell_px;
      OK(build_mirror_raster(h, cell_px));
    } else {
      OK(build_mirror(h, k <= 16 ? 16 : 8));
      group_summary_kernel<<<grid_for(h, (kb.n_groups + 7) / 8, resident_per_sm(h, group_summary_kernel)), kThreads, 0, h->stream>>>(
          h->tpts.p, h->n, h->ff, reinterpret_cast<GroupSummary*>(h->gsum.p));
      ++h->launches;
      CU(cudaGetLastError());
    }
    prof_end(h, span);
    h->summary_ok = true;
    h->ssum_ok = false;
  }
  // two-level classification once every thread of the grid has more than a handful of groups
  // (measured on one box: config 2, 2.8 groups per thread, is 4 us per iteration faster with one
  // level; config 3 / 5, 11 / 34 groups per thread, are 3 / 47 us faster with two)
  kb.two_level = h->opt_two_level >= 0 ? h->opt_two_level != 0 : kb.n_groups > 6ll * kb.step_grid * kThreads;
  if (kb.two_level && !h->ssum_ok) {  // super-group summaries: only when they will be used
    const int span = prof_begin(h, MDKM_PHASE_BUILD, 0);
    super_summary_kernel<<<grid_for(h, (kb.n_groups + kThreads - 1) / kThreads, resident_per_sm(h, super_summary_kernel)), kThreads, 0, h->stream>>>(
        reinterpret_cast<const GroupSummary*>(h->gsum.p), (int)kb.n_groups, reinterpret_cast<SuperSummary*>(h->ssum.p));
    ++h->launches;
    CU(cudaGetLastError());
    prof_end(h, span);
    h->ssum_ok = true;
  }
  if (!h->d_status) {
    CU(cudaMalloc(&h->d_status, sizeof(DevStatus)));
    CU(cudaMallocHost(&h->h_status, 2 * sizeof(DevStatus)));
    CU(cudaEventCreateWithFlags(&h->batch_ev[0], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->batch_ev[1], cudaEventDisableTiming));
  }
  h->last_k = k;
  return MDKM_OK;
}

UpdateParams make_update_params(mdkm_handle* h, const KmBuffers& kb, int allow_pause, int ignore_status) {
  UpdateParams up{};
  up.acc = h->acc.p;
  up.acc_saved = h->acc.p + 3 * ((size_t)kb.kpad * 4 + 8);
  up.table = h->table.p;
  up.st = h->d_status;
  up.fr = h->fr;
  for (int d = 0; d < 3; ++d) up.inv_scale[d] = 1.0 / h->fr.scale[d];
  for (int d = 0; d < 3; ++d) up.mean[d] = h->mean_ok ? h->mean[d] : h->fr.origin[d];
  up.k = kb.k; up.kpad = kb.kpad;
  up.allow_pause = allow_pause;
  up.ignore_status = ignore_status;
  return up;
}

// The Lloyd iteration is ONE kernel when the sums can be completed inside it: a single rank,
// or ranks whose exchange buffers are mapped into each other (NVLink, CUDA IPC).
bool can_fuse(const mdkm_handle* h) { return h->n_ranks == 1 || h->p2p_ok; }

int launch_step(mdkm_handle* h, const KmBuffers& kb, int ignore_status, int fuse_update = 0) {
  StepParams sp{};
  sp.pts = h->tpts.p; sp.n = h->n;  // the tile-ordered mirror; labels / summaries / worklist follow its order
  sp.labels = h->labels.p;
  sp.table = h->table.p;
  sp.table_stride = table_bytes(kb.k, kb.kpad);
  sp.acc = h->acc.p;
  sp.acc_slot = kb.kpad * 4 + 8;
  sp.seq = fuse_update ? h->step_seq++ : 0;
  sp.st = h->d_status;
  sp.f = h->ff;
  sp.k = kb.k; sp.kpad = kb.kpad;
  sp.ignore_status = ignore_status;
  sp.fuse_update = fuse_update;
  sp.settle = h->opt_settle;
  sp.two_level = kb.two_level ? 1 : 0;
  if (fuse_update) {
    sp.upd = make_update_params(h, kb, /*allow_pause=*/1, 0);
    sp.px = h->px;
    if (h->n_ranks == 1) sp.px.n_ranks = 1;
  }
  // pass 1 (inside the kernel): whole groups settled from their summaries; the rest lands in
  // the worklist that pass 2 streams point by point
  int* work_count = h->worklist.p + kb.n_groups;  // two counters (StepParams)
  sp.gsum = reinterpret_cast<const GroupSummary*>(h->gsum.p);
  sp.ssum = h->ssum.p;
  sp.worklist = h->worklist.p;
  sp.work_count = work_count;
  sp.glabel = h->glabel.p;
  sp.grid_bar = &h->d_status->grid_bar;
  // cooperative launch: the grid barrier between the two passes needs every CTA resident
  // The first launch behind a settle kernel is cooperative (the runtime guarantees that the whole grid
  // is resident, which the in-kernel grid barrier needs).  The following launches of the run use
  // programmatic stream serialisation instead -- the runtime does not combine the two (measured: the
  // cooperative attribute silently wins) --: the next kernel is set up while the current one drains
  // (CTAs take the SM slots as the previous kernel's retire, shared memory is initialised) and waits
  // for the previous grid's end before it reads anything (griddepcontrol.wait).  Its grid is the
  // same full wave the cooperative launch was accepted with; the barrier's bounded wait flags the
  // error if a foreign kernel ever kept part of it from becoming resident.  1.7 us per iteration.
  void* args[] = {&sp};
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(kb.step_grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kb.step_smem;
  cfg.stream = h->stream;
  cudaLaunchAttribute attr;
  if (fuse_update && h->opt_pdl && sp.seq > 0) {
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
  } else {
    attr.id = cudaLaunchAttributeCooperative;
    attr.val.cooperative = 1;
  }
  cfg.attrs = &attr;
  cfg.numAttrs = 1;
  const cudaError_t le = cudaLaunchKernelExC(&cfg, reinterpret_cast<const void*>(kb.step_fn), args);
  CU(le);
  ++h->launches;
  if (!fuse_update) CU(cudaMemsetAsync(work_count, 0, 4, h->stream));
  return MDKM_OK;
}

int launch_update(mdkm_handle* h, const KmBuffers& kb, int allow_pause, int ignore_status) {
  const UpdateParams up = make_update_params(h, kb, allow_pause, ignore_status);
  lloyd_update_kernel<<<1, kThreads, 0, h->stream>>>(up);
  ++h->launches;
  CU(cudaGetLastError());
  return MDKM_OK;
}

// Behind a run of fused step launches: applies the pending update, restores the classic layout
// (table[0], acc[0]) and restarts the launch numbering (lloyd.cuh: lloyd_settle_kernel).
int launch_settle(mdkm_handle* h, const KmBuffers& kb) {
  SettleParams sp{};
  sp.upd = make_update_params(h, kb, /*allow_pause=*/1, 0);
  sp.px = h->px;
  if (h->n_ranks == 1 || !can_fuse(h)) sp.px.n_ranks = 1;
  sp.table_stride = table_bytes(kb.k, kb.kpad);
  sp.acc_slot = kb.kpad * 4 + 8;
  sp.work_count = h->worklist.p + kb.n_groups;
  const size_t smem = (size_t)kb.kpad * 48 + bucket_bytes(kb.k, kb.kpad);
  if (smem > 48 * 1024 && h->settle_smem < smem) {
    CU(cudaFuncSetAttribute(lloyd_settle_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    h->settle_smem = smem;
  }
  lloyd_settle_kernel<<<1, kThreads, smem, h->stream>>>(sp);
  ++h->launches;
  CU(cudaGetLastError());
  h->step_seq = 0;
  return MDKM_OK;
}

// Start of a fit / step / prediction in one launch: the status block `st0`, the first `acc_slots`
// accumulator slots and the work counters cleared, the centroid table built from `centers_host`
// (staged in the device-visible host buffer: no pageable copy on the stream).
int fit_head(mdkm_handle* h, const KmBuffers& kb, const DevStatus& st0, const double* centers_host, int acc_slots) {
  const size_t bytes = (size_t)kb.k * 3 * sizeof(double);
  const size_t off = (h->mapped_used + 15) & ~(size_t)15;
  if (off + bytes > kMappedBytes) return fail(h, MDKM_ERR_INVALID, "small result buffer exhausted");
  memcpy(h->mapped + off, centers_host, bytes);  // (free: sync_small waited for every earlier reader)
  h->mapped_used = off + bytes;
  InitTableParams ip{};
  ip.centers = reinterpret_cast<const double*>(h->mapped + off);
  ip.table = h->table.p;
  ip.st = h->d_status;
  ip.fr = h->fr;
  ip.k = kb.k; ip.kpad = kb.kpad;
  ip.st0 = st0;
  ip.acc = h->acc.p;
  ip.acc_words = (long long)acc_slots * (kb.kpad * 4 + 8);
  ip.work_count = acc_slots ? h->worklist.p + kb.n_groups : nullptr;
  ip.final_ticket = h->uscratch.p;
  ip.index_fault = h->index_status.p ? reinterpret_cast<const unsigned int*>(h->index_status.p) + 1 : nullptr;
  init_table_kernel<<<1, kThreads, 0, h->stream>>>(ip);
  ++h->launches;
  CU(cudaGetLastError());
  return MDKM_OK;
}

// The raster mirror index of this cloud timed out in its look-back (fit_head turned that into a
// finished run with status xchg_timeout = 2): report it; the next call rebuilds the mirror.
int index_fault(mdkm_handle* h) {
  h->summary_ok = false;
  CU(cudaMemsetAsync(h->index_status.p, 0, 8, h->stream));
  return fail(h, MDKM_ERR_CUDA, "raster mirror index: a tile's look-back timed out");
}

// Profiling spans: prof_begin records an event on the compute stream and returns the span's
// index (-1 when profiling is off), prof_end records the closing event; collect_profile (after
// the stream has been synchronised) adds the elapsed times to the phases' totals.
int prof_begin(mdkm_handle* h, int phase, long long count) {
  if (!h->prof) return -1;
  const int idx = (int)h->prof_spans.size();
  while (h->prof_ev.size() < (size_t)(idx + 1) * 2) {
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return -1;
    h->prof_ev.push_back(e);
  }
  if (cudaEventRecord(h->prof_ev[2 * idx], h->stream) != cudaSuccess) return -1;
  h->prof_spans.push_back({phase, count});
  return idx;
}

void prof_end(mdkm_handle* h, int idx) {
  if (idx >= 0) cudaEventRecord(h->prof_ev[2 * idx + 1], h->stream);
}

int collect_profile(mdkm_handle* h) {
  for (size_t i = 0; i < h->prof_spans.size(); ++i) {
    float ms = 0.f;
    CU(cudaEventElapsedTime(&ms, h->prof_ev[2 * i], h->prof_ev[2 * i + 1]));
    h->prof_ms[h->prof_spans[i].phase] += ms;
    h->prof_count[h->prof_spans[i].phase] += h->prof_spans[i].count;
  }
  h->prof_spans.clear();
  return MDKM_OK;
}

// A cluster map taken by one fit / predict: written at `dev` by the final pass, then copied to
// `host` unless that is null (device output).
struct MapOut {
  void* dev = nullptr;
  void* host = nullptr;
  int elem = 0;
  size_t bytes = 0;
  // several ranks with day transitions: `dev` is this rank's band of the whole-stack map `stack`,
  // which the final pass clears; a device output receives the band afterwards at `dev_out`
  unsigned char* stack = nullptr;
  size_t stack_bytes = 0;
  void* dev_out = nullptr;
  // day transitions / regions: the whole stack's map (device), once take_stack_map has set it up
  const unsigned char* whole = nullptr;
};

// Per-(day, cluster) statistics taken by one fit / predict (mdkm_bind_day_stats): accumulated by
// the final pass, summed over the ranks, converted on the device and copied to the pinned
// stage; `counts` / `means` receive them after the call's synchronisation.
struct StatsOut {
  long long slots = 0;  // days * k
  int64_t* counts = nullptr;
  double* means = nullptr;
};

// Day-pair transition counts taken by one fit / predict (mdkm_bind_day_transitions): binned from
// the cluster map behind the final pass, summed over the ranks and copied to the pinned stage;
// `out` receives them after the call's synchronisation.
struct TransOut {
  int64_t* out = nullptr;
  int n_pairs = 0;
  int k1 = 0;  // states: k + 1
};

// Connected regions taken by one fit / predict (mdkm_bind_regions): labelled from the whole-stack
// cluster map after the call's synchronisation; `map` (optional) receives this rank's range of
// the region map.
struct RegOut {
  int conn = 0;  // 4 or 8; 0: not asked for
  int32_t* map = nullptr;
  int mem = MDKM_MEM_HOST;
};

// Region overlaps taken by one fit / predict (mdkm_bind_region_overlaps): counted from the
// whole-stack region map that run_regions resolves; the rows stay on the device, where
// mdkm_region_overlap_table finds them.
struct OvOut {
  std::vector<int> pairs;  // [n_pairs][2] days; empty: not asked for
  int n_pairs() const { return (int)(pairs.size() / 2); }
};

// Object tracks taken by one fit / predict (mdkm_bind_tracks): linked from the overlap rows of the
// consecutive pairs, which are counted behind the caller's own pairs; `map` (optional) receives
// this rank's range of the track map.
struct TrackOut {
  double iou = 0.0;             // min_iou; 0: not asked for
  int32_t* map = nullptr;
  int mem = MDKM_MEM_HOST;
  int n_user = 0;               // the caller's overlap pairs, which come first
  std::vector<int> link_day;    // [counted pairs] d of the counted pair (d, d+1), else -1
};

// The optional outputs taken by one fit / predict (take_outputs).
struct CallOutputs {
  MapOut map;
  StatsOut stats;
  TransOut trans;
  RegOut reg;
  OvOut ov;
  TrackOut trk;
  bool adj = false;  // region adjacency (mdkm_bind_region_adjacency)
};

// page-locked host buffer of at least `bytes` (the stages of results handed over after a sync)
int ensure_pinned(mdkm_handle* h, unsigned char*& p, size_t& cap, size_t bytes) {
  if (cap >= bytes && p) return MDKM_OK;
  if (p) {
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaFreeHost(p));
    p = nullptr;
    cap = 0;
  }
  CU(cudaMallocHost(&p, std::max<size_t>(bytes, 1)));
  cap = std::max<size_t>(bytes, 1);
  return MDKM_OK;
}

int run_final(mdkm_handle* h, const KmBuffers& kb, int* labels_dev, bool skip_paused = false,
              double* centroids_host = nullptr, DevStatus* status_host = nullptr, const MapOut* map = nullptr,
              const StatsOut* stats = nullptr);

// the days' point offsets on the device, for the day cursor of the final pass
int upload_day_offsets(mdkm_handle* h) {
  const size_t n_off = h->seg_off.size();
  OK(ensure(h, h->map_seg, n_off));
  CU(cudaMemcpyAsync(h->map_seg.p, h->seg_off.data(), n_off * 8, cudaMemcpyHostToDevice, h->stream));
  return MDKM_OK;
}

// Takes the cluster map of the bindings `b` for a call with k clusters: checks that k fits the
// element type, stages host outputs, uploads the days' point offsets.
int take_cluster_map(mdkm_handle* h, int k, const OutputBindings& b, MapOut& m) {
  void* out = b.map;
  const int elem = b.map_elem, mem = b.map_mem;
  if (!out) return MDKM_OK;
  if (k > (elem == 1 ? 255 : 65535))
    return fail(h, MDKM_ERR_INVALID, "k=%d labels do not fit a cluster map of %d-byte elements", k, elem);
  CU(cudaSetDevice(h->device));
  m.elem = elem;
  m.bytes = (size_t)h->raster_pix_count * elem;
  if (mem == MDKM_MEM_DEVICE) {
    m.dev = out;
  } else {
    OK(ensure(h, h->map_stage, std::max<size_t>(m.bytes, 1)));
    m.dev = h->map_stage.p;
    m.host = out;
  }
  return upload_day_offsets(h);
}

// Takes the day statistics of the bindings `b` for a call with k clusters: checks k against the
// bound capacity, sizes the accumulators, uploads the days' point offsets.
int take_day_stats(mdkm_handle* h, int k, const OutputBindings& b, StatsOut& s) {
  int64_t* counts = b.counts;
  double* means = b.means;
  const int kcap = b.stats_kcap;
  if (!counts) return MDKM_OK;
  if (k > kcap) return fail(h, MDKM_ERR_INVALID, "k=%d exceeds the k_capacity %d of the bound day statistics", k, kcap);
  if (k < 1 || k > kMaxK) return MDKM_OK;  // (rejected with the call's own message)
  CU(cudaSetDevice(h->device));
  s.slots = (long long)h->stack_days * k;
  s.counts = counts;
  s.means = means;
  OK(ensure(h, h->stats_acc, (size_t)s.slots * 4));
  OK(ensure(h, h->stats_dev, (size_t)s.slots * 32));
  OK(ensure_pinned(h, h->stats_host, h->stats_host_cap, (size_t)s.slots * 32));
  return upload_day_offsets(h);
}

// The whole-stack cluster map that day transitions and regions read, taken once per call for
// both: checks, once per cloud, that the ranks' pixel ranges cover the stack (one all-reduce).
// With one rank it is the call's map: the bound one, or an internal one the final pass writes
// when none is bound.  With several ranks it is a whole-stack map of which every rank writes its
// band (a bound device output then receives that band), merged by merge_stack_map.
int take_stack_map(mdkm_handle* h, int k, MapOut& m) {
  if (m.whole) return MDKM_OK;
  CU(cudaSetDevice(h->device));
  const long long HW = (long long)h->raster_H * h->raster_w, stack_px = (long long)h->stack_days * HW;
  if (h->stack_cover < 0) {
    long long px = h->raster_pix_count;
    if (h->n_ranks > 1) {
      OK(ensure(h, h->dscratch, 64));
      long long* d = reinterpret_cast<long long*>(h->dscratch.p);
      CU(cudaMemcpyAsync(d, &px, 8, cudaMemcpyHostToDevice, h->stream));
      OK(allreduce(h, d, 1, kNcclInt64, kNcclSum));
      OK(small_d2h(h, &px, d, 8));
      OK(sync_small(h));
    }
    h->stack_cover = px == stack_px ? 1 : 0;
  }
  if (!h->stack_cover)
    return fail(h, MDKM_ERR_STATE, "day transitions and regions need the pixel ranges of the ranks to cover the whole stack");
  if (h->n_ranks == 1) {
    if (!m.dev) {
      m.elem = k <= 255 ? 1 : 2;
      m.bytes = (size_t)h->raster_pix_count * m.elem;
      OK(ensure(h, h->stack_map, std::max<size_t>(m.bytes, 1)));
      m.dev = h->stack_map.p;
      OK(upload_day_offsets(h));
    }
    m.whole = static_cast<const unsigned char*>(m.dev);
    return MDKM_OK;
  }
  const int elem = m.dev ? m.elem : (k <= 255 ? 1 : 2);
  const size_t stack_bytes = (size_t)stack_px * elem;
  OK(ensure(h, h->stack_map, std::max<size_t>(stack_bytes, 1)));
  if (m.dev && !m.host) m.dev_out = m.dev;
  if (!m.dev) OK(upload_day_offsets(h));
  m.dev = h->stack_map.p + (size_t)h->raster_pix_begin * elem;
  m.elem = elem;
  m.bytes = (size_t)h->raster_pix_count * elem;
  m.stack = h->stack_map.p;
  m.stack_bytes = stack_bytes;
  m.whole = h->stack_map.p;
  return MDKM_OK;
}

// Behind the final pass, on the stream: with several ranks the bands of the whole-stack map summed
// over the ranks.  The bands are disjoint: their byte-wise sum is their union, for 16-bit maps too.
int merge_stack_map(mdkm_handle* h, const MapOut& m) {
  if (m.stack) OK(allreduce(h, m.stack, m.stack_bytes, kNcclUint8, kNcclSum));
  return MDKM_OK;
}

// Takes the day transitions of the bindings `b` for a call with k clusters and its cluster map
// `m`: checks k against the bound capacity, sets up the whole-stack map, sizes the bins, uploads
// the pairs.
int take_transitions(mdkm_handle* h, int k, const OutputBindings& b, MapOut& m, TransOut& t) {
  if (!b.trans) return MDKM_OK;
  const int kcap = b.trans_kcap;
  if (k > kcap) return fail(h, MDKM_ERR_INVALID, "k=%d exceeds the k_capacity %d of the bound day transitions", k, kcap);
  if (k < 1 || k > kMaxK) return MDKM_OK;  // (rejected with the call's own message)
  OK(take_stack_map(h, k, m));
  t.out = b.trans;
  t.n_pairs = (int)(b.pairs.size() / 2);
  t.k1 = k + 1;
  const size_t words = (size_t)t.n_pairs * t.k1 * t.k1;
  OK(ensure(h, h->trans_bins, words));
  OK(ensure(h, h->trans_pairs, b.pairs.size()));
  CU(cudaMemcpyAsync(h->trans_pairs.p, b.pairs.data(), b.pairs.size() * 4, cudaMemcpyHostToDevice, h->stream));
  OK(ensure_pinned(h, h->trans_host, h->trans_host_cap, words * 8));
  return MDKM_OK;
}

// The regions, region overlaps, tracks and region adjacency of an earlier call are dropped.
void drop_results(mdkm_handle* h) {
  h->n_regions = -1;
  h->n_overlaps = -1;
  h->n_tracks = -1;
  h->n_adjacency = -1;
}

// Takes the regions `g` for a call with k clusters and its cluster map `m`: sets up the
// whole-stack map; the results of an earlier call are dropped.
int take_regions(mdkm_handle* h, int k, MapOut& m, RegOut& g) {
  if (!g.conn) return MDKM_OK;
  if (k < 1 || k > kMaxK) {  // (rejected with the call's own message)
    g.conn = 0;
    return MDKM_OK;
  }
  drop_results(h);
  return take_stack_map(h, k, m);
}

// Takes the region overlaps `o` of a call whose regions are `g` (before take_regions): they need
// the regions of the same call; uploads the pairs.
int take_overlaps(mdkm_handle* h, const RegOut& g, const OvOut& o) {
  if (o.pairs.empty()) return MDKM_OK;
  if (!g.conn) return fail(h, MDKM_ERR_STATE, "region overlaps need regions bound for the same call (mdkm_bind_regions)");
  CU(cudaSetDevice(h->device));
  OK(ensure(h, h->ov_pairs, o.pairs.size()));
  CU(cudaMemcpyAsync(h->ov_pairs.p, o.pairs.data(), o.pairs.size() * 4, cudaMemcpyHostToDevice, h->stream));
  return MDKM_OK;
}

// Takes the tracks `t` of a call whose regions are `g` and overlaps `o` (before take_overlaps):
// they need the regions of the same call.  The consecutive pairs (d, d+1) that the caller did not
// ask for are counted after the caller's pairs, whose rows stay a prefix; the link pass finds the
// counted pair of every d through link_day.
int take_tracks(mdkm_handle* h, const RegOut& g, OvOut& o, TrackOut& t) {
  if (!t.iou) return MDKM_OK;
  if (!g.conn) return fail(h, MDKM_ERR_STATE, "tracks need regions bound for the same call (mdkm_bind_regions)");
  const int D = h->stack_days;
  t.n_user = o.n_pairs();
  std::vector<int> pair_of(std::max(D - 1, 0), -1);
  for (int q = 0; q < t.n_user; ++q) {
    const int a = o.pairs[2 * q], b = o.pairs[2 * q + 1];
    if (b == a + 1 && pair_of[a] < 0) pair_of[a] = q;
  }
  for (int d = 0; d + 1 < D; ++d) {
    if (pair_of[d] >= 0) continue;
    pair_of[d] = o.n_pairs();
    o.pairs.push_back(d);
    o.pairs.push_back(d + 1);
  }
  t.link_day.assign(std::max(o.n_pairs(), 1), -1);
  for (int d = 0; d + 1 < D; ++d) t.link_day[pair_of[d]] = d;
  CU(cudaSetDevice(h->device));
  OK(ensure(h, h->track_link_day, t.link_day.size()));
  CU(cudaMemcpyAsync(h->track_link_day.p, t.link_day.data(), t.link_day.size() * 4, cudaMemcpyHostToDevice,
                     h->stream));
  return MDKM_OK;
}

// Takes the region adjacency of a call whose regions are `g` (before take_regions): it needs the
// regions of the same call; sizes the pinned stage of the days' bounds.
int take_adjacency(mdkm_handle* h, const RegOut& g, bool adj) {
  if (!adj) return MDKM_OK;
  if (!g.conn) return fail(h, MDKM_ERR_STATE, "region adjacency needs regions bound for the same call (mdkm_bind_regions)");
  CU(cudaSetDevice(h->device));
  return ensure_pinned(h, h->adj_bounds, h->adj_bounds_cap, (size_t)h->stack_days * 8);
}

typedef void (*TransKernel)(const TransParams);
template <typename T>
TransKernel pick_trans_kernel(int mode) {
  if (mode == kTransWarpBins) return day_transitions_kernel<T, kTransWarpBins>;
  if (mode == kTransCtaBins) return day_transitions_kernel<T, kTransCtaBins>;
  return day_transitions_kernel<T, kTransGlobalBins>;
}

// Behind the final pass and merge_stack_map, on the stream: the bins of this rank's share of the
// pixels of every day of the whole-stack map, their sum over the ranks, the copy to the pinned
// stage.  (Behind a final pass that returned early for a relocation this bins a map of zeros; the
// pass after the relocation runs it again.)
int run_transitions(mdkm_handle* h, const TransOut& t, const MapOut& m) {
  if (!t.out) return MDKM_OK;
  const long long HW = (long long)h->raster_H * h->raster_w;
  const size_t nb = (size_t)t.k1 * t.k1, words = nb * t.n_pairs;
  CU(cudaMemsetAsync(h->trans_bins.p, 0, words * 8, h->stream));
  TransParams tp{};
  tp.map = m.whole;
  tp.HW = HW;
  tp.q_begin = HW * h->rank / h->n_ranks;
  tp.q_end = HW * (h->rank + 1) / h->n_ranks;
  tp.pairs = h->trans_pairs.p;
  tp.n_pairs = t.n_pairs;
  tp.k1 = t.k1;
  tp.bins = h->trans_bins.p;
  // bins in shared memory when they do not cost a resident CTA (run-time occupancy query): a copy
  // per warp, else one per CTA; otherwise straight to the global bins
  auto pick = [&](int mode) { return m.elem == 2 ? pick_trans_kernel<unsigned short>(mode) : pick_trans_kernel<unsigned char>(mode); };
  int base = 0, optin = 0;
  CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&base, pick(kTransGlobalBins), kThreads, 0));
  CU(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
  int mode = kTransGlobalBins, occ = base;
  size_t smem = 0;
  for (int md = kTransWarpBins; md < kTransGlobalBins; ++md) {
    const size_t bytes = nb * 4 * (md == kTransWarpBins ? kThreads / 32 : 1);
    int o = 0;
    if (bytes <= (size_t)optin) {
      CU(cudaFuncSetAttribute(pick(md), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, pick(md), kThreads, bytes));
    }
    if (o >= base) {
      mode = md;
      occ = o;
      smem = bytes;
      break;
    }
  }
  // one wave of resident CTAs over (pairs, chunks); shared bins count in 32 bits, so no CTA
  // bins more than 2^30 + 30 pixels of a pair
  const long long chunks = (tp.q_end - tp.q_begin) / kTransPx + 1;
  const int gy = (int)std::min<long long>(t.n_pairs, 65535);
  long long gx = std::max<long long>(1, (long long)h->sm_count * std::max(occ, 1) / gy);
  gx = std::min(gx, (chunks + kThreads - 1) / kThreads);
  gx = std::max(gx, chunks * kTransPx / (1ll << 30) + 1);
  pick(mode)<<<dim3((unsigned int)gx, (unsigned int)gy), kThreads, smem, h->stream>>>(tp);
  ++h->launches;
  CU(cudaGetLastError());
  OK(allreduce(h, h->trans_bins.p, words, kNcclInt64, kNcclSum));
  CU(cudaMemcpyAsync(h->trans_host, h->trans_bins.p, words * 8, cudaMemcpyDeviceToHost, h->stream));
  return MDKM_OK;
}

// After the call's synchronisation: the pinned stage -> the caller's counts.
void deliver_transitions(mdkm_handle* h, const TransOut& t) {
  if (t.out) memcpy(t.out, h->trans_host, (size_t)t.n_pairs * t.k1 * t.k1 * 8);
}

// Behind the final pass, on the stream: the sums over the ranks, counts and means, their copy
// to the pinned stage.  (A final pass that returned early for a relocation leaves zeros; the
// pass after the relocation runs this again.)
int reduce_day_stats(mdkm_handle* h, const StatsOut& s) {
  if (!s.counts) return MDKM_OK;
  OK(allreduce(h, h->stats_acc.p, (size_t)s.slots * 4, kNcclInt64, kNcclSum));
  long long* d_counts = reinterpret_cast<long long*>(h->stats_dev.p);
  double* d_means = reinterpret_cast<double*>(h->stats_dev.p + (size_t)s.slots * 8);
  day_stats_kernel<<<grid_for(h, (s.slots + kThreads - 1) / kThreads, 4), kThreads, 0, h->stream>>>(
      h->stats_acc.p, s.slots, h->fr, d_counts, d_means);
  ++h->launches;
  CU(cudaGetLastError());
  CU(cudaMemcpyAsync(h->stats_host, h->stats_dev.p, (size_t)s.slots * 32, cudaMemcpyDeviceToHost, h->stream));
  return MDKM_OK;
}

// After the call's synchronisation: the pinned stage -> the caller's arrays.
void deliver_day_stats(mdkm_handle* h, const StatsOut& s) {
  if (!s.counts) return;
  memcpy(s.counts, h->stats_host, (size_t)s.slots * 8);
  memcpy(s.means, h->stats_host + (size_t)s.slots * 8, (size_t)s.slots * 24);
}

int run_overlaps(mdkm_handle* h, const OvOut& o, const int* ids, const unsigned long long* bounds);
int run_tracks(mdkm_handle* h, const TrackOut& t, const OvOut& o, const int* ids);
int run_adjacency(mdkm_handle* h, bool adj, const int* ids, const unsigned long long* bounds);

// The pair-independent part of the overlap kernels' parameters.
OverlapParams overlap_params(mdkm_handle* h, const int* ids, int n_pairs) {
  OverlapParams op{};
  op.ids = ids;
  op.HW = (long long)h->raster_H * h->raster_w;
  op.W = h->raster_w;
  op.pairs = h->ov_pairs.p;
  op.n_pairs = n_pairs;
  op.wpp = (op.HW + 31) / 32;
  return op;
}

// grid of the overlap passes that give a warp kOvSpan pixels of every pair (pairs along y)
dim3 overlap_span_grid(long long HW, int n_pairs) {
  const long long warps = (HW + kOvSpan - 1) / kOvSpan;
  return dim3((unsigned int)((warps + kThreads / 32 - 1) / (kThreads / 32)), (unsigned int)std::min(n_pairs, 65535));
}

// The regions `g` of the whole-stack map `m`, after the call's synchronisation (the map is final,
// also after a relocation).  Every rank labels the whole stack: tile-local union-find, links
// across the tile borders, ids of the roots, every pixel's id (regions.cuh); the caller's region
// map receives this rank's range.  One synchronisation reads R -- and, with region overlaps `o` or
// adjacency `adj`, the bounds of their pairs or days, counted right behind the ids -- then this
// rank's points are summed into per-region slots, the slots are reduced over the ranks (sums;
// minima of the first pixel and the bounds) and the table and means are written on the device,
// where mdkm_region_table finds them.  The overlaps follow (run_overlaps), then the tracks (run_tracks),
// then the adjacency (run_adjacency).
int run_regions(mdkm_handle* h, const RegOut& g, const MapOut& m, const OvOut& o, const TrackOut& t, bool adj) {
  if (!g.conn) return MDKM_OK;
  const long long HW = (long long)h->raster_H * h->raster_w, n_px = (long long)h->stack_days * HW;
  const bool in_place = g.map && g.mem == MDKM_MEM_DEVICE && h->n_ranks == 1;  // (one rank holds the whole stack)
  OK(ensure(h, h->region_parent, (size_t)n_px));
  if (!in_place) OK(ensure(h, h->region_ids, (size_t)n_px));
  const long long n_chunks = (n_px + kRegChunk - 1) / kRegChunk;
  const int n_pairs = o.n_pairs(), n_adj = adj ? h->stack_days : 0;
  // look-back words of the numbering, ticket + fault, R, the overlap bounds of the pairs, then the
  // adjacency bounds of the days
  OK(ensure(h, h->region_scan, (size_t)n_chunks + 2 + n_pairs + n_adj));
  RegionParams rp{};
  rp.map = m.whole;
  rp.parent = h->region_parent.p;
  rp.ids = in_place ? g.map : h->region_ids.p;
  rp.n_px = n_px;
  rp.HW = HW;
  rp.H = h->raster_H;
  rp.W = h->raster_w;
  rp.tiles_x = (h->raster_w + kRegTile - 1) / kRegTile;
  rp.tiles_y = (h->raster_H + kRegTile - 1) / kRegTile;
  rp.n_tiles = (long long)h->stack_days * rp.tiles_x * rp.tiles_y;
  rp.status = h->region_scan.p;
  rp.ticket = reinterpret_cast<unsigned int*>(h->region_scan.p + n_chunks);
  rp.n_regions = h->region_scan.p + n_chunks + 1;
  const bool c8 = g.conn == 8, wide = m.elem == 2;
  auto tile_fn = wide ? (c8 ? region_tile_kernel<unsigned short, true> : region_tile_kernel<unsigned short, false>)
                      : (c8 ? region_tile_kernel<unsigned char, true> : region_tile_kernel<unsigned char, false>);
  auto border_fn = wide ? (c8 ? region_border_kernel<unsigned short, true> : region_border_kernel<unsigned short, false>)
                        : (c8 ? region_border_kernel<unsigned char, true> : region_border_kernel<unsigned char, false>);
  tile_fn<<<(unsigned int)rp.n_tiles, kThreads, 0, h->stream>>>(rp);
  border_fn<<<(unsigned int)((rp.n_tiles + kThreads / 32 - 1) / (kThreads / 32)), kThreads, 0, h->stream>>>(rp);
  CU(cudaMemsetAsync(h->region_scan.p, 0, ((size_t)n_chunks + 2 + n_pairs + n_adj) * 8, h->stream));
  region_number_kernel<<<(unsigned int)n_chunks, kThreads, 0, h->stream>>>(rp);
  region_resolve_kernel<<<grid_for(h, (n_px + 1023) / 1024, resident_per_sm(h, region_resolve_kernel)), kThreads, 0,
                          h->stream>>>(rp);
  h->launches += 4;
  if (n_pairs) {
    OverlapParams op = overlap_params(h, rp.ids, n_pairs);
    op.bounds = h->region_scan.p + n_chunks + 2;
    overlap_bound_kernel<<<overlap_span_grid(HW, n_pairs), kThreads, 0, h->stream>>>(op);
    ++h->launches;
  }
  unsigned long long* adj_bounds = reinterpret_cast<unsigned long long*>(h->adj_bounds);
  if (n_adj) {
    AdjacencyParams ap{};
    ap.ov = overlap_params(h, rp.ids, n_adj);
    ap.ov.bounds = h->region_scan.p + n_chunks + 2 + n_pairs;
    adjacency_bound_kernel<<<overlap_span_grid(HW, n_adj), kThreads, 0, h->stream>>>(ap);
    ++h->launches;
    OK(small_d2h(h, adj_bounds, ap.ov.bounds, (size_t)n_adj * 8, /*dst_is_pinned=*/true));
  }
  CU(cudaGetLastError());
  if (g.map && !in_place)
    CU(cudaMemcpyAsync(g.map, rp.ids + h->raster_pix_begin, (size_t)h->raster_pix_count * 4,
                       g.mem == MDKM_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
  std::vector<unsigned long long> got(2 + (size_t)n_pairs, 0ull);  // ticket | fault << 32, R, the overlap bounds
  OK(small_d2h(h, got.data(), h->region_scan.p + n_chunks, got.size() * 8));
  OK(sync_small(h));
  if (got[0] >> 32) return fail(h, MDKM_ERR_CUDA, "region numbering: the look-back over the chunks timed out");
  const long long R = (long long)got[1];
  if (R > 0) {
    OK(ensure(h, h->region_acc, (size_t)R * 4));
    OK(ensure(h, h->region_box, (size_t)R * 5));
    OK(ensure(h, h->region_out, (size_t)R * 80));
    CU(cudaMemsetAsync(h->region_acc.p, 0, (size_t)R * 32, h->stream));
    CU(cudaMemsetAsync(h->region_box.p, 0xff, (size_t)R * 20, h->stream));
    if (h->n > 0) {
      RegionStatsParams sp{};
      sp.pts = h->pts.p;
      sp.n = h->n;
      sp.seg = h->map_seg.p;
      sp.nseg = (int)h->seg_off.size() - 1;
      sp.pix0 = h->day0 * HW;
      sp.HW = HW;
      sp.W = h->raster_w;
      sp.ids = rp.ids;
      for (int d = 0; d < 3; ++d) {
        sp.origin[d] = h->fr.origin[d];
        sp.scale[d] = h->fr.scale[d];
      }
      sp.acc = h->region_acc.p;
      sp.box = h->region_box.p;
      const long long n_groups = (h->n + kGroup - 1) / kGroup;
      region_stats_kernel<<<grid_for(h, (n_groups + 7) / 8, resident_per_sm(h, region_stats_kernel)), kThreads, 0,
                            h->stream>>>(sp);
      ++h->launches;
    }
    OK(allreduce(h, h->region_acc.p, (size_t)R * 4, kNcclInt64, kNcclSum));
    OK(allreduce(h, h->region_box.p, (size_t)R * 5, kNcclUint32, kNcclMin));
    long long* table = reinterpret_cast<long long*>(h->region_out.p);
    region_finish_kernel<<<grid_for(h, (R + kThreads - 1) / kThreads, 4), kThreads, 0, h->stream>>>(
        h->region_acc.p, h->region_box.p, R, m.whole, m.elem, HW, h->fr, table,
        reinterpret_cast<double*>(table + R * 7));
    ++h->launches;
    CU(cudaGetLastError());
  }
  h->n_regions = R;
  OK(run_overlaps(h, o, rp.ids, got.data() + 2));
  OK(run_tracks(h, t, o, rp.ids));
  return run_adjacency(h, adj, rp.ids, adj_bounds);
}

// The region overlaps `o` of the region map `ids` (the whole stack, on every rank), behind the
// region table on the stream, given the bounds of the pairs (region_overlaps.cuh): one hash table
// per pair sized from its bound, the keys inserted, their first pixels marked, the masks scanned;
// one synchronisation reads M, then the rows are written on the device, where
// mdkm_region_overlap_table finds them.  Every rank builds the whole table on its own.
int run_overlaps(mdkm_handle* h, const OvOut& o, const int* ids, const unsigned long long* bounds) {
  const int n_pairs = o.n_pairs();
  if (!n_pairs) return MDKM_OK;
  std::vector<long long> tab((size_t)n_pairs + 1, 0);
  long long max_cap = 0;
  for (int q = 0; q < n_pairs; ++q) {
    long long cap = 0;
    if (bounds[q]) for (cap = 2; cap < 2 * (long long)bounds[q]; cap <<= 1) {}
    tab[q + 1] = tab[q] + cap;
    max_cap = std::max(max_cap, cap);
  }
  if (tab[n_pairs] == 0) {  // no pixel has ids on both days of any pair
    h->n_overlaps = 0;
    return MDKM_OK;
  }
  OverlapParams op = overlap_params(h, ids, n_pairs);
  const long long n_words = (long long)n_pairs * op.wpp;
  const long long n_chunks = (n_words + kOvChunkWords - 1) / kOvChunkWords, padded = n_chunks * kOvChunkWords;
  OK(ensure(h, h->ov_tab, tab.size()));
  OK(ensure(h, h->ov_slots, 2 * (size_t)tab[n_pairs]));
  OK(ensure(h, h->ov_bits, 2 * (size_t)padded));
  OK(ensure(h, h->ov_scan, 2 * (size_t)n_chunks + 3));
  CU(cudaMemcpyAsync(h->ov_tab.p, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(h->ov_slots.p, 0, (size_t)tab[n_pairs] * 16, h->stream));
  CU(cudaMemsetAsync(h->ov_bits.p, 0, (size_t)padded * 4, h->stream));
  CU(cudaMemsetAsync(h->ov_scan.p, 0, (2 * (size_t)n_chunks + 3) * 8, h->stream));
  op.tab = h->ov_tab.p;
  op.slots = h->ov_slots.p;
  op.bits = h->ov_bits.p;
  op.word_rel = h->ov_bits.p + padded;
  op.status = h->ov_scan.p;
  op.chunk_base = h->ov_scan.p + n_chunks;
  op.ticket = reinterpret_cast<unsigned int*>(h->ov_scan.p + 2 * n_chunks);
  op.total = h->ov_scan.p + 2 * n_chunks + 1;
  op.probe_fault = reinterpret_cast<unsigned int*>(h->ov_scan.p + 2 * n_chunks + 2);
  const dim3 slot_grid((unsigned int)grid_for(h, (max_cap + kThreads - 1) / kThreads, 4),
                       (unsigned int)std::min(n_pairs, 65535));
  overlap_insert_kernel<<<overlap_span_grid(op.HW, n_pairs), kThreads, 0, h->stream>>>(op);
  overlap_mark_kernel<<<slot_grid, kThreads, 0, h->stream>>>(op);
  overlap_scan_kernel<<<(unsigned int)n_chunks, kThreads, 0, h->stream>>>(op, n_chunks);
  h->launches += 3;
  CU(cudaGetLastError());
  unsigned long long got[3] = {0, 0, 0};  // ticket | fault << 32, M, probe fault
  OK(small_d2h(h, got, op.ticket, 24));
  OK(sync_small(h));
  if (got[0] >> 32) return fail(h, MDKM_ERR_CUDA, "region overlaps: the look-back over the chunks timed out");
  if (got[2]) return fail(h, MDKM_ERR_CUDA, "region overlaps: a hash table had no free slot");
  const long long M = (long long)got[1];
  OK(ensure(h, h->ov_rows, (size_t)M * 6));
  op.rows = h->ov_rows.p;
  overlap_emit_kernel<<<slot_grid, kThreads, 0, h->stream>>>(op);
  ++h->launches;
  CU(cudaGetLastError());
  h->n_overlaps = M;
  return MDKM_OK;
}

// The tracks `t` of the R regions of the last run_regions, behind the overlap rows of the
// counted pairs `o` on the stream (tracks.cuh): links, the numbering passes of the regions on the
// R parents, the table into R zeroed rows, this rank's range of the track map from the region
// map `ids` (the whole stack).  One synchronisation reads T and the number of the caller's rows,
// which becomes the count mdkm_region_overlap_count reports.  Every rank builds the same tracks.
int run_tracks(mdkm_handle* h, const TrackOut& t, const OvOut& o, const int* ids) {
  if (!t.iou) return MDKM_OK;
  const long long R = h->n_regions, M = o.n_pairs() ? h->n_overlaps : 0;
  const long long n_chunks = (R + kRegChunk - 1) / kRegChunk;
  OK(ensure(h, h->track_parent, (size_t)R));
  OK(ensure(h, h->track_links, 2 * (size_t)R));
  OK(ensure(h, h->track_ids, (size_t)R));
  OK(ensure(h, h->track_tab, 7 * (size_t)R));
  OK(ensure(h, h->track_scan, (size_t)n_chunks + 3));  // look-back words, ticket + fault, T, caller's M
  CU(cudaMemsetAsync(h->track_scan.p, 0, ((size_t)n_chunks + 3) * 8, h->stream));
  CU(cudaMemsetAsync(h->track_tab.p, 0, (size_t)R * 56, h->stream));
  TrackParams tp{};
  tp.rows = h->ov_rows.p;
  tp.n_rows = M;
  tp.link_day = h->track_link_day.p;
  tp.n_user = t.n_user;
  tp.user_rows = h->track_scan.p + n_chunks + 2;
  tp.regions = reinterpret_cast<const long long*>(h->region_out.p);
  tp.n_regions = R;
  tp.min_iou = t.iou;
  tp.parent = h->track_parent.p;
  tp.links = h->track_links.p;
  tp.tracks = h->track_ids.p;
  tp.table = h->track_tab.p;
  if (R > 0) {
    RegionParams np{};
    np.parent = h->track_parent.p;
    np.ids = h->track_ids.p;
    np.n_px = R;
    np.status = h->track_scan.p;
    np.ticket = reinterpret_cast<unsigned int*>(h->track_scan.p + n_chunks);
    np.n_regions = h->track_scan.p + n_chunks + 1;
    const int per_region = grid_for(h, (R + kThreads - 1) / kThreads, resident_per_sm(h, track_table_kernel));
    track_init_kernel<<<per_region, kThreads, 0, h->stream>>>(tp);
    if (M > 0)
      track_link_kernel<<<grid_for(h, (M + kThreads - 1) / kThreads, resident_per_sm(h, track_link_kernel)), kThreads, 0,
                          h->stream>>>(tp);
    region_number_kernel<<<(unsigned int)n_chunks, kThreads, 0, h->stream>>>(np);
    region_resolve_kernel<<<grid_for(h, (R + 1023) / 1024, resident_per_sm(h, region_resolve_kernel)), kThreads, 0,
                            h->stream>>>(np);
    track_table_kernel<<<per_region, kThreads, 0, h->stream>>>(tp);
    h->launches += M > 0 ? 5 : 4;
  }
  const long long n = h->raster_pix_count;
  if (t.map && n > 0) {
    int* out = t.map;
    if (t.mem != MDKM_MEM_DEVICE) {
      OK(ensure(h, h->track_stage, (size_t)n));
      out = h->track_stage.p;
    }
    track_map_kernel<<<grid_for(h, (n / 4 + kThreads) / kThreads, resident_per_sm(h, track_map_kernel)), kThreads, 0,
                       h->stream>>>(ids + h->raster_pix_begin, h->track_ids.p, out, n);
    ++h->launches;
    if (t.mem != MDKM_MEM_DEVICE)
      CU(cudaMemcpyAsync(t.map, out, (size_t)n * 4, cudaMemcpyDeviceToHost, h->stream));
  }
  CU(cudaGetLastError());
  unsigned long long got[3] = {0, 0, 0};  // ticket | fault << 32, T, the caller's rows
  OK(small_d2h(h, got, h->track_scan.p + n_chunks, 24));
  OK(sync_small(h));
  if (got[0] >> 32) return fail(h, MDKM_ERR_CUDA, "track numbering: the look-back over the chunks timed out");
  h->n_tracks = (long long)got[1];
  h->n_overlaps = t.n_user ? (long long)got[2] : -1;
  return MDKM_OK;
}

// The region adjacency of the R regions of the last run_regions in the region map `ids` (the
// whole stack, on every rank), given the bounds of the days (region_adjacency.cuh): one hash table
// per day sized from its bound, the keys inserted while the sides towards pixels without a point
// and the raster border are summed, their first edges marked and the masks scanned (the overlap
// passes, a day in place of a pair); one synchronisation reads M, then the rows are written and
// the boundaries finished on the device, where mdkm_region_adjacency_table finds them.  Every rank
// builds the whole table on its own.
int run_adjacency(mdkm_handle* h, bool adj, const int* ids, const unsigned long long* bounds) {
  if (!adj) return MDKM_OK;
  const int D = h->stack_days;
  const long long R = h->n_regions;
  h->n_adjacency = 0;
  if (R == 0) return MDKM_OK;
  std::vector<long long> tab((size_t)D + 1, 0);
  long long max_cap = 0;
  for (int d = 0; d < D; ++d) {
    long long cap = 0;
    if (bounds[d]) for (cap = 2; cap < 2 * (long long)bounds[d]; cap <<= 1) {}
    tab[d + 1] = tab[d] + cap;
    max_cap = std::max(max_cap, cap);
  }
  AdjacencyParams ap{};
  ap.ov = overlap_params(h, ids, D);
  ap.ov.wpp = (2 * ap.ov.HW + 31) / 32;
  const long long n_words = (long long)D * ap.ov.wpp;
  const long long n_chunks = (n_words + kOvChunkWords - 1) / kOvChunkWords, padded = n_chunks * kOvChunkWords;
  const bool keyed = tab[D] > 0;  // some day has an edge between two regions
  OK(ensure(h, h->adj_tab, tab.size()));
  OK(ensure(h, h->adj_sides, 4 * (size_t)R));
  if (keyed) {
    OK(ensure(h, h->adj_slots, 2 * (size_t)tab[D]));
    OK(ensure(h, h->adj_bits, 2 * (size_t)padded));
    OK(ensure(h, h->adj_scan, 2 * (size_t)n_chunks + 3));
  }
  CU(cudaMemcpyAsync(h->adj_tab.p, tab.data(), tab.size() * 8, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(h->adj_sides.p, 0, (size_t)R * 32, h->stream));
  ap.ov.tab = h->adj_tab.p;
  ap.sides = h->adj_sides.p;
  ap.n_regions = R;
  if (keyed) {
    CU(cudaMemsetAsync(h->adj_slots.p, 0, (size_t)tab[D] * 16, h->stream));
    CU(cudaMemsetAsync(h->adj_bits.p, 0, (size_t)padded * 4, h->stream));
    CU(cudaMemsetAsync(h->adj_scan.p, 0, (2 * (size_t)n_chunks + 3) * 8, h->stream));
    ap.ov.slots = h->adj_slots.p;
    ap.ov.bits = h->adj_bits.p;
    ap.ov.word_rel = h->adj_bits.p + padded;
    ap.ov.status = h->adj_scan.p;
    ap.ov.chunk_base = h->adj_scan.p + n_chunks;
    ap.ov.ticket = reinterpret_cast<unsigned int*>(h->adj_scan.p + 2 * n_chunks);
    ap.ov.total = h->adj_scan.p + 2 * n_chunks + 1;
    ap.ov.probe_fault = reinterpret_cast<unsigned int*>(h->adj_scan.p + 2 * n_chunks + 2);
  }
  const dim3 slot_grid((unsigned int)grid_for(h, (max_cap + kThreads - 1) / kThreads, 4),
                       (unsigned int)std::min(D, 65535));
  const int per_region = grid_for(h, (R + kThreads - 1) / kThreads, 4);
  adjacency_insert_kernel<<<overlap_span_grid(ap.ov.HW, D), kThreads, 0, h->stream>>>(ap);
  ++h->launches;
  if (keyed) {
    overlap_mark_kernel<<<slot_grid, kThreads, 0, h->stream>>>(ap.ov);
    overlap_scan_kernel<<<(unsigned int)n_chunks, kThreads, 0, h->stream>>>(ap.ov, n_chunks);
    h->launches += 2;
    CU(cudaGetLastError());
    unsigned long long got[3] = {0, 0, 0};  // ticket | fault << 32, M, probe fault
    OK(small_d2h(h, got, ap.ov.ticket, 24));
    OK(sync_small(h));
    if (got[0] >> 32) return fail(h, MDKM_ERR_CUDA, "region adjacency: the look-back over the chunks timed out");
    if (got[2]) return fail(h, MDKM_ERR_CUDA, "region adjacency: a hash table had no free slot");
    const long long M = (long long)got[1];
    OK(ensure(h, h->adj_rows, (size_t)M * 6));
    ap.ov.rows = h->adj_rows.p;
    adjacency_emit_kernel<<<slot_grid, kThreads, 0, h->stream>>>(ap);
    ++h->launches;
    h->n_adjacency = M;
  }
  adjacency_finish_kernel<<<per_region, kThreads, 0, h->stream>>>(ap);
  ++h->launches;
  CU(cudaGetLastError());
  return MDKM_OK;
}

// Takes the outputs bound for a call with k clusters into `o`.  The bindings are moved out of the
// handle first, so the call consumes every one of them whatever happens.  When several checks
// fail the first in this order is reported, except that the cluster map's comes after the day
// statistics'.
int take_outputs(mdkm_handle* h, int k, CallOutputs& o) {
  OutputBindings b = std::exchange(h->bound, OutputBindings{});
  o.reg = {b.regions, b.region_map, b.region_map_mem};
  o.ov.pairs = std::move(b.ov_pairs);
  o.trk = {b.track_iou, b.track_map, b.track_map_mem};
  o.adj = b.adjacency;
  const int map_rc = take_cluster_map(h, k, b, o.map);
  OK(take_day_stats(h, k, b, o.stats));
  OK(map_rc);
  OK(take_transitions(h, k, b, o.map, o.trans));
  OK(take_tracks(h, o.reg, o.ov, o.trk));
  OK(take_overlaps(h, o.reg, o.ov));
  OK(take_adjacency(h, o.reg, o.adj));
  return take_regions(h, k, o.map, o.reg);
}

// Behind the final pass, on the stream: the day statistics, the whole-stack map and the day
// transitions of `o`.
int reduce_outputs(mdkm_handle* h, const CallOutputs& o) {
  OK(reduce_day_stats(h, o.stats));
  OK(merge_stack_map(h, o.map));
  return run_transitions(h, o.trans, o.map);
}

// After the call's synchronisation: the regions of `o` with their overlaps, tracks and adjacency,
// then the day statistics and transitions handed to the caller.
int deliver_outputs(mdkm_handle* h, const CallOutputs& o) {
  OK(run_regions(h, o.reg, o.map, o.ov, o.trk, o.adj));
  deliver_day_stats(h, o.stats);
  deliver_transitions(h, o.trans);
  return MDKM_OK;
}

// The map's device->host copy (host outputs), on the compute stream behind the final pass.
int copy_cluster_map(mdkm_handle* h, const MapOut& m) {
  if (m.host && m.bytes) CU(cudaMemcpyAsync(m.host, m.dev, m.bytes, cudaMemcpyDeviceToHost, h->stream));
  if (m.dev_out && m.bytes) CU(cudaMemcpyAsync(m.dev_out, m.dev, m.bytes, cudaMemcpyDeviceToDevice, h->stream));
  return MDKM_OK;
}

// Empty-cluster relocation (sklearn/_k_means_common.pyx:167-211), sequenced from the host
// while the Lloyd loop is paused.  All arithmetic on the device (extras.cuh).
int relocate_empty(mdkm_handle* h, const KmBuffers& kb, int n_empty) {
  // scratch: [0] best distance bits, [1] best global index, [2..5] payload (qx,qy,qz,old label),
  //          [6] taken count, [8 .. 8+kMaxK) taken global indices
  OK(ensure(h, h->reloc, 8 + 2 * (size_t)kMaxK));
  CU(cudaMemsetAsync(h->reloc.p, 0, (8 + 2 * (size_t)kMaxK) * 8, h->stream));
  const long long rank_offset = h->rank_offset;  // global index of this rank's first point
  // labels in the reference's order under the OLD centroids (the paused update has not touched
  // the table yet): what the step just assigned, recomputed point by point
  OK(ensure(h, h->labels32, (size_t)std::max<long long>(h->n, 1)));
  OK(run_final(h, kb, h->labels32.p));
  RelocParams rp{};
  rp.pts = h->pts.p; rp.n = h->n;
  rp.labels = h->labels32.p;
  rp.table = h->table.p; rp.kpad = kb.kpad; rp.k = kb.k;
  rp.f = h->ff;
  rp.scratch = h->reloc.p;
  rp.acc = h->acc.p;
  rp.rank_offset = rank_offset;
  const int g = grid_for(h, (h->n + 1023) / 1024, 4);
  for (int e = 0; e < n_empty; ++e) {
    rp.round = e;
    CU(cudaMemsetAsync(h->reloc.p, 0, 6 * 8, h->stream));
    CU(cudaMemsetAsync(h->reloc.p + 1, 0xff, 8, h->stream));
    reloc_maxdist_kernel<<<g, kThreads, 0, h->stream>>>(rp);
    ++h->launches;
    OK(allreduce(h, h->reloc.p, 1, kNcclUint64, kNcclMax));
    reloc_argidx_kernel<<<g, kThreads, 0, h->stream>>>(rp);
    ++h->launches;
    OK(allreduce(h, h->reloc.p + 1, 1, kNcclUint64, kNcclMin));
    reloc_payload_kernel<<<1, 32, 0, h->stream>>>(rp);
    ++h->launches;
    OK(allreduce(h, h->reloc.p + 2, 4, kNcclUint64, kNcclSum));
    reloc_apply_kernel<<<1, 32, 0, h->stream>>>(rp, h->d_status);
    ++h->launches;
    CU(cudaGetLastError());
  }
  return MDKM_OK;
}

// (the ticket is zero: fit_head clears it, every final pass leaves it so)
int run_final(mdkm_handle* h, const KmBuffers& kb, int* labels_dev, bool skip_paused, double* centroids_host,
              DevStatus* status_host, const MapOut* map, const StatsOut* stats) {
  FinalParams fp{};
  FinalKernel fn = kb.final_fn;
  size_t smem = kb.final_smem;
  const bool want_map = map && map->dev, want_stats = stats && stats->counts;
  if (want_map) {
    // pixels without a point stay 0 (napari's background label)
    if (map->stack) CU(cudaMemsetAsync(map->stack, 0, map->stack_bytes, h->stream));
    else if (map->bytes) CU(cudaMemsetAsync(map->dev, 0, map->bytes, h->stream));
    fp.map_out = map->dev;
    fp.map_elem = map->elem;
    fp.map_W = h->raster_w;
    fp.map_pix_begin = h->raster_pix_begin;
    fp.map_HW = (long long)h->raster_H * h->raster_w;
    fp.map_day0 = h->raster_pix_begin / fp.map_HW;
  }
  if (want_map || want_stats) {
    fn = pick_final_kernel(kb.kpad, want_map, want_stats);
    fp.map_seg = h->map_seg.p;
    fp.map_nseg = (int)h->seg_off.size() - 1;
  }
  if (want_stats) {
    CU(cudaMemsetAsync(h->stats_acc.p, 0, (size_t)stats->slots * 32, h->stream));
    fp.stats_acc = h->stats_acc.p;
    fp.stats_day0 = h->day0;
    fp.stats_slots = (int)stats->slots;
    // a copy of the slots per warp in shared memory when they fit without costing a resident CTA;
    // otherwise straight to the global slots (many days x many clusters)
    const size_t with_slots = kb.final_smem + (size_t)(kThreads / 32) * stats->slots * 32;
    int optin = 0, occ = 0;
    CU(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
    if (with_slots <= (size_t)optin) {
      CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)with_slots));
      CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, kThreads, with_slots));
    }
    if (occ >= h->occ_final) {
      smem = with_slots;
      fp.stats_smem_off = (int)kb.final_smem;
    }
  }
  if (fn != kb.final_fn) CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fp.pts = h->pts.p; fp.n = h->n;
  fp.labels_out = labels_dev;
  fp.table = h->table.p;
  fp.partials = h->partials.p;
  fp.ticket = h->uscratch.p;
  fp.st = h->d_status;
  fp.f = h->ff;
  fp.k = kb.k; fp.kpad = kb.kpad;
  fp.split_rows = h->raster_w > 0 ? 1 : 0;
  fp.skip_paused = skip_paused ? 1 : 0;
  fp.status_host = status_host;
  fp.centroids_host = centroids_host;
  for (int d = 0; d < 3; ++d) fp.origin[d] = h->fr.origin[d];
  fn<<<kb.final_grid, kThreads, smem, h->stream>>>(fp);
  ++h->launches;
  CU(cudaGetLastError());
  return MDKM_OK;
}

}  // namespace

// =========================================================================================
// C ABI
// =========================================================================================
extern "C" {

const char* mdkm_version(void) { return "mdkm 0.1 sm_100a"; }

int mdkm_create(mdkm_handle** out, int device, void* cuda_stream) {
  if (!out) return MDKM_ERR_INVALID;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return MDKM_ERR_NO_DEVICE;
  if (device < 0 || device >= count) return MDKM_ERR_INVALID;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return MDKM_ERR_CUDA;
  if (prop.major != 10) return MDKM_ERR_NO_DEVICE;  // kernels are sm_100a only; no fallback
  if (cudaSetDevice(device) != cudaSuccess) return MDKM_ERR_CUDA;
  mdkm_handle* h = new mdkm_handle();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  if (cuda_stream) {
    h->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  } else {
    if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
      delete h;
      return MDKM_ERR_CUDA;
    }
    h->own_stream = true;
  }
  if (cudaMallocHost(&h->h_total, 64) != cudaSuccess ||
      cudaHostAlloc(&h->mapped, kMappedBytes, cudaHostAllocMapped) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_ready, cudaEventDisableTiming) != cudaSuccess) {
    delete h;
    return MDKM_ERR_CUDA;
  }
  *out = h;
  return MDKM_OK;
}

void mdkm_destroy(mdkm_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  if (h->d2h_stream) cudaStreamSynchronize(h->d2h_stream);
  if (h->comm && nccl_api().ok) nccl_api().CommDestroy(h->comm);
  close_p2p(h);
  if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
  if (h->h2d_stream) {
    cudaStreamSynchronize(h->h2d_stream);
    cudaStreamDestroy(h->h2d_stream);
  }
  if (h->ev_ready) cudaEventDestroy(h->ev_ready);
  for (auto e : h->slab_ev) cudaEventDestroy(e);
  if (h->h_slab_totals) cudaFreeHost(h->h_slab_totals);
  release(h->slab_totals);
  release(h->cloud_aos);
  release(h->pts);
  release(h->labels); release(h->table); release(h->acc); release(h->labels32);
  release(h->dscratch); release(h->partials); release(h->uscratch); release(h->reloc);
  release(h->gsum); release(h->ssum); release(h->glabel); release(h->worklist);
  release(h->tpts); release(h->cell_counts); release(h->cell_offsets); release(h->index_status);
  release(h->run_src); release(h->druns); release(h->gfirst);
  release(h->tile_status); release(h->chunk_offsets); release(h->staging); release(h->planes);
  release(h->d_seg_off); release(h->sel_hist); release(h->sel_targets);
  release(h->map_stage); release(h->map_seg); release(h->stats_acc); release(h->stats_dev);
  if (h->stats_host) cudaFreeHost(h->stats_host);
  release(h->stack_map); release(h->trans_pairs); release(h->trans_bins);
  if (h->trans_host) cudaFreeHost(h->trans_host);
  release(h->region_parent); release(h->region_ids); release(h->region_scan); release(h->region_acc);
  release(h->region_box); release(h->region_out);
  release(h->ov_pairs); release(h->ov_tab); release(h->ov_slots); release(h->ov_bits); release(h->ov_scan);
  release(h->ov_rows);
  release(h->track_link_day); release(h->track_parent); release(h->track_links); release(h->track_ids);
  release(h->track_scan); release(h->track_tab); release(h->track_stage);
  release(h->adj_tab); release(h->adj_slots); release(h->adj_bits); release(h->adj_scan); release(h->adj_rows);
  release(h->adj_sides);
  if (h->adj_bounds) cudaFreeHost(h->adj_bounds);
  release(h->kpp_closest); release(h->kpp_cell); release(h->kpp_blk); release(h->kpp_prefix);
  release(h->kpp_partials); release(h->kpp_rand); release(h->kpp_state);
  if (h->d_status) cudaFree(h->d_status);
  if (h->h_status) cudaFreeHost(h->h_status);
  if (h->h_total) cudaFreeHost(h->h_total);
  if (h->mapped) cudaFreeHost(h->mapped);
  for (auto e : h->batch_ev)
    if (e) cudaEventDestroy(e);
  for (auto e : h->prof_ev) cudaEventDestroy(e);
  if (h->own_stream) cudaStreamDestroy(h->stream);
  delete h;
}

const char* mdkm_last_error(const mdkm_handle* h) { return h ? h->err.c_str() : "null handle"; }

int mdkm_comm_unique_id(unsigned char out[MDKM_NCCL_UNIQUE_ID_BYTES]) {
  if (!out) return MDKM_ERR_INVALID;
  NcclApi& api = nccl_api();
  if (!api.ok) return MDKM_ERR_NCCL;
  ncclUniqueId id;
  if (api.GetUniqueId(&id) != 0) return MDKM_ERR_NCCL;
  memcpy(out, id.internal, MDKM_NCCL_UNIQUE_ID_BYTES);
  return MDKM_OK;
}

int mdkm_comm_init(mdkm_handle* h, int n_ranks, int rank, const unsigned char id[MDKM_NCCL_UNIQUE_ID_BYTES]) {
  if (!h || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(h, MDKM_ERR_INVALID, "bad rank/world size");
  CU(cudaSetDevice(h->device));
  if (h->comm) {
    nccl_api().CommDestroy(h->comm);
    h->comm = nullptr;
  }
  h->n_ranks = n_ranks;
  h->rank = rank;
  h->frame_ok = false;
  h->stack_cover = -1;
  close_p2p(h);
  if (n_ranks == 1) return MDKM_OK;
  if (!id) return fail(h, MDKM_ERR_INVALID, "unique id required");
  NcclApi& api = nccl_api();
  if (!api.ok) return fail(h, MDKM_ERR_NCCL, "libnccl.so.2 not found (set MDKM_NCCL_LIB)");
  ncclUniqueId uid;
  memcpy(uid.internal, id, MDKM_NCCL_UNIQUE_ID_BYTES);
  NC(api.CommInitRank(&h->comm, n_ranks, uid, rank));
  if (h->have_points) OK(compute_frame(h));
  return MDKM_OK;
}

int mdkm_comm_p2p_handle(mdkm_handle* h, unsigned char out[MDKM_IPC_HANDLE_BYTES]) {
  if (!h || !out) return MDKM_ERR_INVALID;
  if (h->n_ranks < 2 || h->n_ranks > kMaxRanks)
    return fail(h, MDKM_ERR_STATE, "peer exchange needs 2..%d ranks (mdkm_comm_init first)", kMaxRanks);
  CU(cudaSetDevice(h->device));
  close_p2p(h);
  const size_t slot = (size_t)kMaxK * 4 + 8;
  const size_t words = 4 * (size_t)h->n_ranks * slot + 2 * (size_t)h->n_ranks;  // two 8-byte packets per word
  CU(cudaMalloc(&h->xchg, words * 8));
  CU(cudaMemset(h->xchg, 0, words * 8));
  cudaIpcMemHandle_t ih;
  CU(cudaIpcGetMemHandle(&ih, h->xchg));
  static_assert(sizeof(ih) == MDKM_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
  memcpy(out, &ih, sizeof(ih));
  return MDKM_OK;
}

int mdkm_comm_p2p_open(mdkm_handle* h, const unsigned char* handles) {
  if (!h || !handles) return MDKM_ERR_INVALID;
  if (!h->xchg) return fail(h, MDKM_ERR_STATE, "call mdkm_comm_p2p_handle first");
  CU(cudaSetDevice(h->device));
  const size_t slot = (size_t)kMaxK * 4 + 8;
  PeerXchg px{};
  px.n_ranks = h->n_ranks; px.rank = h->rank; px.slot = (int)slot;
  for (int q = 0; q < h->n_ranks; ++q) {
    void* base = h->xchg;
    if (q != h->rank) {
      cudaIpcMemHandle_t ih;
      memcpy(&ih, handles + (size_t)q * MDKM_IPC_HANDLE_BYTES, sizeof(ih));
      cudaError_t e = cudaIpcOpenMemHandle(&base, ih, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        cudaGetLastError();
        for (int r = 0; r < q; ++r)
          if (h->peer_base[r]) { cudaIpcCloseMemHandle(h->peer_base[r]); h->peer_base[r] = nullptr; }
        return fail(h, MDKM_ERR_NCCL, "cudaIpcOpenMemHandle(rank %d) failed: %s -- the NCCL exchange stays in use", q,
                    cudaGetErrorString(e));
      }
      h->peer_base[q] = base;
    }
    px.data[q] = static_cast<unsigned long long*>(base);
    px.flags[q] = px.data[q] + 4 * (size_t)h->n_ranks * slot;
  }
  h->px = px;
  h->p2p_ok = true;
  h->epoch_base = 0;
  return MDKM_OK;
}

int mdkm_comm_p2p_close(mdkm_handle* h) {
  if (!h) return MDKM_ERR_INVALID;
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  close_p2p(h);
  return MDKM_OK;
}

int mdkm_comm_p2p_buffer(mdkm_handle* h, void** out_device_ptr) {
  if (!h || !out_device_ptr) return MDKM_ERR_INVALID;
  if (!h->xchg) return fail(h, MDKM_ERR_STATE, "call mdkm_comm_p2p_handle first");
  *out_device_ptr = h->xchg;
  return MDKM_OK;
}

int mdkm_comm_p2p_open_ptrs(mdkm_handle* h, void* const* buffers) {
  if (!h || !buffers) return MDKM_ERR_INVALID;
  if (!h->xchg) return fail(h, MDKM_ERR_STATE, "call mdkm_comm_p2p_handle first");
  CU(cudaSetDevice(h->device));
  const size_t slot = (size_t)kMaxK * 4 + 8;
  PeerXchg px{};
  px.n_ranks = h->n_ranks; px.rank = h->rank; px.slot = (int)slot;
  for (int q = 0; q < h->n_ranks; ++q) {
    void* base = buffers[q];
    if (!base) return fail(h, MDKM_ERR_INVALID, "null exchange buffer for rank %d", q);
    if (q == h->rank) {
      if (base != h->xchg) return fail(h, MDKM_ERR_INVALID, "buffers[rank] is not this handle's exchange buffer");
    } else {
      cudaPointerAttributes at{};
      CU(cudaPointerGetAttributes(&at, base));
      if (at.type != cudaMemoryTypeDevice) return fail(h, MDKM_ERR_INVALID, "buffers[%d] is not device memory", q);
      if (at.device != h->device) {
        int can = 0;
        CU(cudaDeviceCanAccessPeer(&can, h->device, at.device));
        if (!can) return fail(h, MDKM_ERR_NCCL, "device %d cannot access device %d -- the NCCL exchange stays in use", h->device, at.device);
        cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
          return fail(h, MDKM_ERR_NCCL, "cudaDeviceEnablePeerAccess(%d) failed: %s", at.device, cudaGetErrorString(e));
        cudaGetLastError();
      }
    }
    px.data[q] = static_cast<unsigned long long*>(base);
    px.flags[q] = px.data[q] + 4 * (size_t)h->n_ranks * slot;
  }
  h->px = px;
  h->p2p_ok = true;
  h->epoch_base = 0;
  return MDKM_OK;
}

void* mdkm_get_stream(const mdkm_handle* h) { return h ? reinterpret_cast<void*>(h->stream) : nullptr; }

int mdkm_set_option(mdkm_handle* h, int option, long long value) {
  if (!h) return MDKM_ERR_INVALID;
  switch (option) {
    case MDKM_OPT_SETTLE_GROUPS:
      h->opt_settle = value != 0;
      return MDKM_OK;
    case MDKM_OPT_RASTER_MIRROR:
      h->opt_raster_mirror = value != 0;
      h->summary_ok = false;
      return MDKM_OK;
    case MDKM_OPT_TWO_LEVEL:
      h->opt_two_level = value < 0 ? -1 : (value != 0);
      return MDKM_OK;
    case MDKM_OPT_DEPENDENT_LAUNCH:
      h->opt_pdl = value != 0;
      return MDKM_OK;
    case MDKM_OPT_CELL_PX:
      if (value != 0 && value != 8 && value != 16) return fail(h, MDKM_ERR_INVALID, "cell width must be 0 (automatic), 8 or 16 pixels");
      h->opt_cell_px = (int)value;
      h->summary_ok = false;
      return MDKM_OK;
    case MDKM_OPT_CELL_ROWS:
      if (value < 0 || value > 64) return fail(h, MDKM_ERR_INVALID, "rows per cell must be in [0, 64]");
      h->opt_cell_rows = (int)value;
      h->summary_ok = false;
      return MDKM_OK;
    default:
      return fail(h, MDKM_ERR_INVALID, "unknown option %d", option);
  }
}

int mdkm_set_points(mdkm_handle* h, const float* xyz, int64_t n, int layout, int mem) {
  if (!h) return MDKM_ERR_INVALID;
  if (n < 0 || (n > 0 && !xyz)) return fail(h, MDKM_ERR_INVALID, "bad points argument");
  CU(cudaSetDevice(h->device));
  OK(alloc_points(h, n));
  h->n = n;
  if (n > 0) {
    const float* src = xyz;
    if (mem != MDKM_MEM_DEVICE) {
      OK(ensure(h, h->staging, (size_t)n * 12));
      CU(cudaMemcpyAsync(h->staging.p, xyz, (size_t)n * 12, cudaMemcpyHostToDevice, h->stream));
      src = reinterpret_cast<const float*>(h->staging.p);
    }
    to_blocked_kernel<<<grid_for(h, (n * 3 + kThreads - 1) / kThreads, 8), kThreads, 0, h->stream>>>(
        src, n, layout == MDKM_POINTS_SOA ? 1 : 0, h->pts.p);
    ++h->launches;
    CU(cudaGetLastError());
  }
  OK(zero_tail(h));
  h->seg_off.assign({0, (long long)n});
  h->seg_whole = true;
  h->raster_w = 0;
  h->bound = {};
  h->stack_cover = -1;
  drop_results(h);
  h->stack_days = 1;
  h->day0 = 0;
  h->runs_ok = false;
  h->have_points = true;
  h->frame_ok = false;
  OK(compute_frame(h));
  return MDKM_OK;
}

int64_t mdkm_num_points(const mdkm_handle* h) { return h ? h->n : -1; }

int64_t mdkm_num_points_global(mdkm_handle* h) {
  if (!h || !h->have_points) return -1;
  if (!h->frame_ok && compute_frame(h) != MDKM_OK) return -1;
  return h->n_total;
}

int mdkm_gather_points(mdkm_handle* h, const int64_t* idx, int m, float* out_xyz) {
  if (!h || !idx || !out_xyz || m < 0) return fail(h, MDKM_ERR_INVALID, "bad gather argument");
  if (!h->have_points) return fail(h, MDKM_ERR_STATE, "no points resident");
  CU(cudaSetDevice(h->device));
  if (!h->frame_ok) OK(compute_frame(h));
  for (int i = 0; i < m; ++i)
    if (idx[i] < 0 || idx[i] >= h->n_total)
      return fail(h, MDKM_ERR_INVALID, "gather index %lld out of range", (long long)idx[i]);
  if (m == 0) return MDKM_OK;
  if ((size_t)m * 12 > kMappedBytes / 2) return fail(h, MDKM_ERR_INVALID, "gather of %d points is too large", m);
  OK(ensure(h, h->dscratch, (size_t)m * 3 + 16));
  long long* d_idx = reinterpret_cast<long long*>(h->dscratch.p);
  float* d_out = reinterpret_cast<float*>(h->dscratch.p + m);
  CU(cudaMemcpyAsync(d_idx, idx, (size_t)m * 8, cudaMemcpyHostToDevice, h->stream));
  // indices are global: a rank contributes the points it owns and zeros for the others
  gather_points_kernel<<<(m + 255) / 256, 256, 0, h->stream>>>(h->pts.p, d_idx, m, h->rank_offset, h->n, d_out);
  ++h->launches;
  CU(cudaGetLastError());
  OK(allreduce(h, d_out, (size_t)m * 3, kNcclFloat32, kNcclSum));
  OK(small_d2h(h, out_xyz, d_out, (size_t)m * 12));
  OK(sync_small(h));
  return MDKM_OK;
}

int mdkm_bind_cloud_output(mdkm_handle* h, float* out_host, int64_t capacity_points, int napari_order) {
  if (!h) return MDKM_ERR_INVALID;
  if (out_host && capacity_points < 0) return fail(h, MDKM_ERR_INVALID, "bad capacity");
  h->bound_cloud_out = out_host;
  h->bound_cloud_cap = out_host ? capacity_points : 0;
  h->bound_cloud_napari = napari_order;
  return MDKM_OK;
}

int mdkm_bind_cluster_map(mdkm_handle* h, void* out, int elem_bytes, int64_t capacity_pixels, int mem) {
  if (!h) return MDKM_ERR_INVALID;
  h->bound.map = nullptr;
  if (!out) return MDKM_OK;
  if (!h->have_points || h->raster_w <= 0)
    return fail(h, MDKM_ERR_STATE, "a cluster map needs a resident cloud from mdkm_unproject");
  if (elem_bytes != 1 && elem_bytes != 2) return fail(h, MDKM_ERR_INVALID, "elem_bytes must be 1 or 2");
  if (h->raster_w >= (1 << 23) || h->raster_H >= (1 << 23))  // (the final pass converts x, y with an FADD)
    return fail(h, MDKM_ERR_INVALID, "cluster maps need rasters narrower and shorter than 2^23 pixels");
  if (capacity_pixels < h->raster_pix_count)
    return fail(h, MDKM_ERR_INVALID, "cluster map holds %lld pixels, the range has %lld", (long long)capacity_pixels,
                h->raster_pix_count);
  h->bound.map = out;
  h->bound.map_elem = elem_bytes;
  h->bound.map_mem = mem;
  return MDKM_OK;
}

int mdkm_bind_day_transitions(mdkm_handle* h, const int32_t* pairs, int n_pairs, int64_t* counts_out, int k_capacity) {
  if (!h) return MDKM_ERR_INVALID;
  h->bound.trans = nullptr;
  if (!counts_out) return MDKM_OK;
  if (!h->have_points || h->raster_w <= 0)
    return fail(h, MDKM_ERR_STATE, "day transitions need a resident cloud from mdkm_unproject");
  if (!pairs || n_pairs < 1 || k_capacity < 1 ||
      (double)n_pairs * ((double)k_capacity + 1.0) * ((double)k_capacity + 1.0) >= 2147483648.0)
    return fail(h, MDKM_ERR_INVALID, "day transitions need n_pairs >= 1, k_capacity >= 1 and n_pairs * (k_capacity + 1)^2 < 2^31");
  if (h->raster_w >= (1 << 23) || h->raster_H >= (1 << 23))  // (the final pass writes the map they are binned from)
    return fail(h, MDKM_ERR_INVALID, "day transitions need rasters narrower and shorter than 2^23 pixels");
  for (int i = 0; i < 2 * n_pairs; ++i)
    if (pairs[i] < 0 || pairs[i] >= h->stack_days)
      return fail(h, MDKM_ERR_INVALID, "pair %d: day %d is not in [0, %d)", i / 2, (int)pairs[i], h->stack_days);
  h->bound.pairs.assign(pairs, pairs + 2 * (size_t)n_pairs);
  h->bound.trans = counts_out;
  h->bound.trans_kcap = k_capacity;
  return MDKM_OK;
}

int mdkm_bind_regions(mdkm_handle* h, int connectivity, int32_t* map_out, int64_t capacity_pixels, int mem) {
  if (!h) return MDKM_ERR_INVALID;
  h->bound.regions = 0;
  h->bound.region_map = nullptr;
  if (!connectivity && !map_out) return MDKM_OK;
  if (!h->have_points || h->raster_w <= 0)
    return fail(h, MDKM_ERR_STATE, "regions need a resident cloud from mdkm_unproject");
  if (connectivity != 4 && connectivity != 8)
    return fail(h, MDKM_ERR_INVALID, "regions: connectivity must be 4 or 8, got %d", connectivity);
  if ((long long)h->stack_days * h->raster_H * h->raster_w >= (1ll << 31))
    return fail(h, MDKM_ERR_INVALID, "regions need a stack of fewer than 2^31 pixels");
  if (h->raster_w >= (1 << 23) || h->raster_H >= (1 << 23))  // (the final pass writes the map they are labelled from)
    return fail(h, MDKM_ERR_INVALID, "regions need rasters narrower and shorter than 2^23 pixels");
  if (map_out && (capacity_pixels < h->raster_pix_count || (mem != MDKM_MEM_HOST && mem != MDKM_MEM_DEVICE)))
    return fail(h, MDKM_ERR_INVALID, "region map: capacity %lld < %lld pixels, or bad memory kind",
                (long long)capacity_pixels, h->raster_pix_count);
  h->bound.regions = connectivity;
  h->bound.region_map = map_out;
  h->bound.region_map_mem = mem;
  return MDKM_OK;
}

int mdkm_region_count(const mdkm_handle* h, int64_t* n_regions) {
  if (!h || !n_regions) return MDKM_ERR_INVALID;
  if (h->n_regions < 0) return fail(const_cast<mdkm_handle*>(h), MDKM_ERR_STATE, "no regions: no fit / predict with regions since the last unproject / set_points");
  *n_regions = h->n_regions;
  return MDKM_OK;
}

int mdkm_region_table(mdkm_handle* h, int64_t* table_out, double* means_out, int64_t capacity_regions) {
  if (!h) return MDKM_ERR_INVALID;
  if (h->n_regions < 0) return fail(h, MDKM_ERR_STATE, "no regions: no fit / predict with regions since the last unproject / set_points");
  const long long R = h->n_regions;
  if (capacity_regions < R) return fail(h, MDKM_ERR_INVALID, "region table: capacity %lld < %lld regions", (long long)capacity_regions, R);
  if (R == 0) return MDKM_OK;
  CU(cudaSetDevice(h->device));
  if (table_out) CU(cudaMemcpyAsync(table_out, h->region_out.p, (size_t)R * 56, cudaMemcpyDeviceToHost, h->stream));
  if (means_out)
    CU(cudaMemcpyAsync(means_out, h->region_out.p + (size_t)R * 56, (size_t)R * 24, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return MDKM_OK;
}

int mdkm_bind_region_overlaps(mdkm_handle* h, const int32_t* pairs, int n_pairs) {
  if (!h) return MDKM_ERR_INVALID;
  h->bound.ov_pairs.clear();
  if (!pairs) return MDKM_OK;
  if (!h->have_points || h->raster_w <= 0)
    return fail(h, MDKM_ERR_STATE, "region overlaps need a resident cloud from mdkm_unproject");
  if (n_pairs < 1 || n_pairs > kMaxOvPairs)
    return fail(h, MDKM_ERR_INVALID, "region overlaps need 1 <= n_pairs <= %d, got %d", kMaxOvPairs, n_pairs);
  for (int i = 0; i < 2 * n_pairs; ++i)
    if (pairs[i] < 0 || pairs[i] >= h->stack_days)
      return fail(h, MDKM_ERR_INVALID, "region overlap pair %d: day %d is not in [0, %d)", i / 2, (int)pairs[i],
                  h->stack_days);
  h->bound.ov_pairs.assign(pairs, pairs + 2 * (size_t)n_pairs);
  return MDKM_OK;
}

int mdkm_region_overlap_count(const mdkm_handle* h, int64_t* n_rows) {
  if (!h || !n_rows) return MDKM_ERR_INVALID;
  if (h->n_overlaps < 0)
    return fail(const_cast<mdkm_handle*>(h), MDKM_ERR_STATE, "no region overlaps: no fit / predict with region overlaps since the last unproject / set_points or fit / predict with regions");
  *n_rows = h->n_overlaps;
  return MDKM_OK;
}

int mdkm_region_overlap_table(mdkm_handle* h, int64_t* table_out, int64_t capacity_rows) {
  if (!h) return MDKM_ERR_INVALID;
  if (h->n_overlaps < 0)
    return fail(h, MDKM_ERR_STATE, "no region overlaps: no fit / predict with region overlaps since the last unproject / set_points or fit / predict with regions");
  const long long M = h->n_overlaps;
  if (capacity_rows < M) return fail(h, MDKM_ERR_INVALID, "region overlap table: capacity %lld < %lld rows", (long long)capacity_rows, M);
  if (M == 0 || !table_out) return MDKM_OK;
  CU(cudaSetDevice(h->device));
  CU(cudaMemcpyAsync(table_out, h->ov_rows.p, (size_t)M * 48, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return MDKM_OK;
}

int mdkm_bind_tracks(mdkm_handle* h, double min_iou, int32_t* map_out, int64_t capacity_pixels, int mem) {
  if (!h) return MDKM_ERR_INVALID;
  h->bound.track_iou = 0.0;
  h->bound.track_map = nullptr;
  if (min_iou == 0.0 && !map_out) return MDKM_OK;
  if (!h->have_points || h->raster_w <= 0)
    return fail(h, MDKM_ERR_STATE, "tracks need a resident cloud from mdkm_unproject");
  if (!(min_iou > 0.0 && min_iou <= 1.0))
    return fail(h, MDKM_ERR_INVALID, "tracks: min_iou must be in (0, 1], got %g", min_iou);
  if (h->stack_days > kMaxTrackDays)
    return fail(h, MDKM_ERR_INVALID, "tracks need a stack of at most %d days, got %d", kMaxTrackDays, h->stack_days);
  if (map_out && (capacity_pixels < h->raster_pix_count || (mem != MDKM_MEM_HOST && mem != MDKM_MEM_DEVICE)))
    return fail(h, MDKM_ERR_INVALID, "track map: capacity %lld < %lld pixels, or bad memory kind",
                (long long)capacity_pixels, h->raster_pix_count);
  h->bound.track_iou = min_iou;
  h->bound.track_map = map_out;
  h->bound.track_map_mem = mem;
  return MDKM_OK;
}

int mdkm_track_count(const mdkm_handle* h, int64_t* n_tracks) {
  if (!h || !n_tracks) return MDKM_ERR_INVALID;
  if (h->n_tracks < 0)
    return fail(const_cast<mdkm_handle*>(h), MDKM_ERR_STATE, "no tracks: no fit / predict with tracks since the last unproject / set_points or fit / predict with regions");
  *n_tracks = h->n_tracks;
  return MDKM_OK;
}

int mdkm_track_table(mdkm_handle* h, int64_t* table_out, int32_t* region_tracks_out, int64_t capacity_tracks,
                     int64_t capacity_regions) {
  if (!h) return MDKM_ERR_INVALID;
  if (h->n_tracks < 0)
    return fail(h, MDKM_ERR_STATE, "no tracks: no fit / predict with tracks since the last unproject / set_points or fit / predict with regions");
  const long long T = h->n_tracks, R = h->n_regions;
  if (table_out && capacity_tracks < T)
    return fail(h, MDKM_ERR_INVALID, "track table: capacity %lld < %lld tracks", (long long)capacity_tracks, T);
  if (region_tracks_out && capacity_regions < R)
    return fail(h, MDKM_ERR_INVALID, "region tracks: capacity %lld < %lld regions", (long long)capacity_regions, R);
  if (R == 0) return MDKM_OK;
  CU(cudaSetDevice(h->device));
  if (table_out) CU(cudaMemcpyAsync(table_out, h->track_tab.p, (size_t)T * 56, cudaMemcpyDeviceToHost, h->stream));
  if (region_tracks_out)
    CU(cudaMemcpyAsync(region_tracks_out, h->track_ids.p, (size_t)R * 4, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return MDKM_OK;
}

int mdkm_bind_region_adjacency(mdkm_handle* h, int on) {
  if (!h) return MDKM_ERR_INVALID;
  h->bound.adjacency = false;
  if (!on) return MDKM_OK;
  if (!h->have_points || h->raster_w <= 0)
    return fail(h, MDKM_ERR_STATE, "region adjacency needs a resident cloud from mdkm_unproject");
  h->bound.adjacency = true;
  return MDKM_OK;
}

int mdkm_region_adjacency_count(const mdkm_handle* h, int64_t* n_rows) {
  if (!h || !n_rows) return MDKM_ERR_INVALID;
  if (h->n_adjacency < 0)
    return fail(const_cast<mdkm_handle*>(h), MDKM_ERR_STATE, "no region adjacency: no fit / predict with region adjacency since the last unproject / set_points or fit / predict with regions");
  *n_rows = h->n_adjacency;
  return MDKM_OK;
}

int mdkm_region_adjacency_table(mdkm_handle* h, int64_t* rows_out, int64_t* boundaries_out, int64_t capacity_rows,
                                int64_t capacity_regions) {
  if (!h) return MDKM_ERR_INVALID;
  if (h->n_adjacency < 0)
    return fail(h, MDKM_ERR_STATE, "no region adjacency: no fit / predict with region adjacency since the last unproject / set_points or fit / predict with regions");
  const long long M = h->n_adjacency, R = h->n_regions;
  if (rows_out && capacity_rows < M)
    return fail(h, MDKM_ERR_INVALID, "region adjacency table: capacity %lld < %lld rows", (long long)capacity_rows, M);
  if (boundaries_out && capacity_regions < R)
    return fail(h, MDKM_ERR_INVALID, "region boundaries: capacity %lld < %lld regions", (long long)capacity_regions, R);
  CU(cudaSetDevice(h->device));
  if (rows_out && M) CU(cudaMemcpyAsync(rows_out, h->adj_rows.p, (size_t)M * 48, cudaMemcpyDeviceToHost, h->stream));
  if (boundaries_out && R)
    CU(cudaMemcpyAsync(boundaries_out, h->adj_sides.p, (size_t)R * 32, cudaMemcpyDeviceToHost, h->stream));
  CU(cudaStreamSynchronize(h->stream));
  return MDKM_OK;
}

int mdkm_bind_day_stats(mdkm_handle* h, int64_t* counts_out, double* means_out, int n_days, int k_capacity) {
  if (!h) return MDKM_ERR_INVALID;
  h->bound.counts = nullptr;
  h->bound.means = nullptr;
  if (!counts_out) return MDKM_OK;
  if (!h->have_points) return fail(h, MDKM_ERR_STATE, "day statistics need a resident cloud");
  if (!means_out) return fail(h, MDKM_ERR_INVALID, "day statistics need a means array");
  if (n_days != h->stack_days)
    return fail(h, MDKM_ERR_INVALID, "n_days=%d, the resident cloud's stack has %d days", n_days, h->stack_days);
  if (k_capacity < 1 || (long long)n_days * k_capacity >= (1ll << 29))  // (slot indices are int32 on the device)
    return fail(h, MDKM_ERR_INVALID, "k_capacity must be >= 1 and n_days * k_capacity < 2^29");
  h->bound.counts = counts_out;
  h->bound.means = means_out;
  h->bound.stats_kcap = k_capacity;
  return MDKM_OK;
}

// Unprojection as a pipeline of slabs: the host->device copy of slab s+1 (copy stream) overlaps
// the kernels of slab s (compute stream) and, when a cloud output is bound, the device->host
// copy of the points slab s-1 produced (result stream).  PCIe is full duplex, so the two copy
// directions proceed together; the kernels are negligible next to either.
int mdkm_unproject(mdkm_handle* h, const void* hm, int hm_dtype, float hm_scale, const uint8_t* mask, int D, int H,
                   int W, int64_t pix_begin, int64_t pix_count, float max_abs, int detrend, int mem,
                   int64_t* n_points_out) {
  if (!h) return MDKM_ERR_INVALID;
  float* cloud_out = h->bound_cloud_out;  // a binding is consumed by this call, whatever happens
  const long long cloud_cap = h->bound_cloud_cap;
  const int cloud_napari = h->bound_cloud_napari;
  h->bound_cloud_out = nullptr;
  h->bound_cloud_cap = 0;
  h->bound = {};  // (the outputs describe the range and the stack they were bound for)
  h->stack_cover = -1;
  drop_results(h);
  if (D < 0 || H <= 0 || W <= 0 || pix_begin < 0 || pix_count < 0 ||
      pix_begin + pix_count > (int64_t)D * H * W || (pix_count > 0 && !hm))
    return fail(h, MDKM_ERR_INVALID, "bad stack geometry");
  if (hm_dtype != MDKM_HM_F32 && hm_dtype != MDKM_HM_I16 && hm_dtype != MDKM_HM_F32_GTIFF3)
    return fail(h, MDKM_ERR_INVALID, "bad hm_dtype");
  const long long HW = (long long)H * W;
  if (detrend && ((pix_begin % HW) != 0 || (pix_count % HW) != 0))
    return fail(h, MDKM_ERR_INVALID, "detrend needs whole days in [pix_begin, pix_begin+pix_count)");
  if (cloud_out && cloud_cap < pix_count)
    return fail(h, MDKM_ERR_INVALID, "bound cloud output holds %lld points, the range has %lld pixels", cloud_cap,
                (long long)pix_count);
  CU(cudaSetDevice(h->device));
  OK(wait_pending(h));
  const size_t esz = hm_dtype == MDKM_HM_F32 ? 4 : (hm_dtype == MDKM_HM_I16 ? 2 : 12);
  const bool from_host = mem != MDKM_MEM_DEVICE;
  const void* d_hm = hm;
  const uint8_t* d_mask = mask;
  const size_t hm_bytes = (size_t)pix_count * esz;
  const size_t hm_pad = (hm_bytes + 255) / 256 * 256;
  if (from_host && pix_count > 0) {
    OK(ensure(h, h->staging, hm_pad + (mask ? (size_t)pix_count : 0) + 256));
    d_hm = h->staging.p;
    if (mask) d_mask = h->staging.p + hm_pad;
  }
  OK(alloc_points(h, pix_count));
  const long long n_chunks = (pix_count + kChunk - 1) / kChunk;
  const long long n_tiles = (pix_count + kTile - 1) / kTile;
  constexpr int kSuper = kThreads / 32;  // warp tiles per super-tile (one CTA, one look-back)
  const long long n_super = (n_tiles + kSuper - 1) / kSuper;
  OK(ensure(h, h->chunk_offsets, (size_t)n_chunks + 2));
  OK(ensure(h, h->tile_status, (size_t)n_super + 2));  // [n_super] status words, then the ticket counter
  UnprojParams up{};
  up.hm = d_hm; up.mask = d_mask;
  up.pix_begin = pix_begin; up.pix_count = pix_count; up.HW = HW; up.W = W; up.H = H;
  up.dtype = hm_dtype;
  up.scale = hm_scale; up.max_abs = max_abs;
  up.chunk_offsets = h->chunk_offsets.p;
  up.status = h->tile_status.p;
  up.ticket = reinterpret_cast<unsigned int*>(h->tile_status.p + n_super);
  up.pts = h->pts.p;
  up.planes = nullptr;
  up.day0 = (int)(pix_begin / HW);
  // run table for the raster mirror build: whole rows of a raster whose width is a multiple of 8
  h->runs_ok = false;
  const bool want_runs = pix_count > 0 && (W % 8) == 0 && (pix_begin % W) == 0 && (pix_count % W) == 0 &&
                         pix_count < (1ll << 32);
  if (want_runs) {
    OK(ensure(h, h->run_src, (size_t)(pix_count / 8) + 1));
    up.run_src = h->run_src.p;
  }
  long long n_out = 0;
  if (pix_count > 0) {
    const int n_days = detrend ? (int)(pix_count / HW) : 0;
    if (detrend) {
      OK(ensure(h, h->planes, (size_t)n_days * 8));
      OK(ensure(h, h->partials, (size_t)n_days * kPlaneBlocks * 10 + 16));
    }
    // slab boundaries (pixels of the range): every kSlabPix, plus the day ends when detrending
    // (a day's plane needs the whole day).  Device input without a bound output: one slab.
    constexpr long long kSlabPix = 4ll << 20;
    std::vector<long long> cut;  // exclusive ends
    if (!from_host && !cloud_out) {
      cut.push_back(pix_count);
    } else {
      long long next_day = detrend ? HW : pix_count;
      // (the first slabs are small so that the result copies start early: the end-to-end call is bound
      // by the device-to-host link, which idles until the first slab has been unprojected)
      long long slab = kSlabPix / 8;
      for (long long p = 0; p < pix_count;) {
        long long e = std::min<long long>(pix_count, p + slab);
        slab = std::min<long long>(kSlabPix, slab * 2);
        if (detrend && e > next_day) e = next_day;
        if (e == next_day) next_day += HW;
        cut.push_back(e);
        p = e;
      }
    }
    const int n_slabs = (int)cut.size();
    OK(ensure(h, h->slab_totals, (size_t)n_slabs + 1));
    if (h->h_slab_cap < (size_t)n_slabs + 1) {
      if (h->h_slab_totals) cudaFreeHost(h->h_slab_totals);
      h->h_slab_totals = nullptr;
      h->h_slab_cap = 0;
      CU(cudaMallocHost(&h->h_slab_totals, ((size_t)n_slabs + 1) * 8));
      h->h_slab_cap = (size_t)n_slabs + 1;
    }
    while (h->slab_ev.size() < (size_t)n_slabs * 2) {
      cudaEvent_t e;
      CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      h->slab_ev.push_back(e);
    }
    if (cloud_out) OK(ensure(h, h->cloud_aos, (size_t)pix_count * 3));
    CU(cudaMemsetAsync(h->slab_totals.p, 0, 8, h->stream));
    CU(cudaMemsetAsync(h->tile_status.p, 0, ((size_t)n_super + 1) * 8, h->stream));  // look-back words + ticket
    {  // bounding box of the cloud, collected by the fused pass
      OK(ensure(h, h->uscratch, 16));
      CU(cudaMemsetAsync(h->uscratch.p + 4, 0xff, 12, h->stream));
      CU(cudaMemsetAsync(h->uscratch.p + 7, 0, 12, h->stream));
      up.minmax = h->uscratch.p + 4;
    }
    // copies of this call must not start before earlier work on the compute stream that still
    // reads the staging buffer has finished
    if (from_host) {
      CU(cudaEventRecord(h->ev_ready, h->stream));
      CU(cudaStreamWaitEvent(h->h2d_stream, h->ev_ready, 0));
    }
    long long done_chunks = 0, days_solved = 0, begin = 0;
    for (int s = 0; s < n_slabs; ++s) {
      const long long end = cut[s];
      if (from_host) {
        CU(cudaMemcpyAsync(h->staging.p + (size_t)begin * esz, static_cast<const char*>(hm) + (size_t)begin * esz,
                           (size_t)(end - begin) * esz, cudaMemcpyHostToDevice, h->h2d_stream));
        if (mask)
          CU(cudaMemcpyAsync(h->staging.p + hm_pad + begin, mask + begin, (size_t)(end - begin),
                             cudaMemcpyHostToDevice, h->h2d_stream));
        CU(cudaEventRecord(h->slab_ev[2 * s], h->h2d_stream));
        CU(cudaStreamWaitEvent(h->stream, h->slab_ev[2 * s], 0));
      }
      long long ready = end;  // pixels whose chunks may be processed now
      if (detrend) {
        const long long days_in = end / HW;
        if (days_in > days_solved) {
          UnprojParams upd = up;
          upd.day0 = up.day0 + (int)days_solved;
          const int nd = (int)(days_in - days_solved);
          plane_moments_kernel<<<dim3(kPlaneBlocks, nd), kThreads, 0, h->stream>>>(
              upd, nd, h->partials.p + (size_t)days_solved * kPlaneBlocks * 10);
          plane_solve_kernel<<<nd, 32, 0, h->stream>>>(h->partials.p + (size_t)days_solved * kPlaneBlocks * 10,
                                                       kPlaneBlocks, W, H, h->planes.p + (size_t)days_solved * 8);
          h->launches += 2;
          days_solved = days_in;
        }
        ready = days_solved * HW;
        up.planes = h->planes.p;
      }
      // (whole super-tiles = an even number of chunks, except at the very end of the range)
      const long long c_end = (s == n_slabs - 1) ? n_chunks : (ready / kChunk) / (kSuper * kTile / kChunk) * (kSuper * kTile / kChunk);
      if (c_end > done_chunks) {
        up.chunk_begin = done_chunks;
        up.chunk_end = c_end;
        // the tiles of these chunks, in one fused pass (rank, look-back, write)
        up.tile_begin = done_chunks * (kChunk / kTile);
        up.tile_end = std::min<long long>(c_end * (kChunk / kTile), n_tiles);
        up.total_out = h->slab_totals.p + s + 1;
        const long long nt = up.tile_end - up.tile_begin;
        const int g = grid_for(h, (nt + kSuper - 1) / kSuper, MDKM_UNPROJ_CTAS);  // resident CTAs per SM (register budget)
        if (s > 0) CU(cudaMemsetAsync(up.ticket, 0, 4, h->stream));
        const int span = prof_begin(h, MDKM_PHASE_UNPROJECT, std::min<long long>(c_end * kChunk, pix_count) - done_chunks * kChunk);
        // row / day bookkeeping per step when a step of 32 pixels never straddles a raster row
        const int mode = (W % 32 == 0 && pix_begin % 32 == 0) ? 0 : (W >= 32 ? 1 : 2);
        if (up.planes) {
          if (mode == 0) unproject_fused_kernel<0, true><<<g, kThreads, 0, h->stream>>>(up);
          else if (mode == 1) unproject_fused_kernel<1, true><<<g, kThreads, 0, h->stream>>>(up);
          else unproject_fused_kernel<2, true><<<g, kThreads, 0, h->stream>>>(up);
        } else {
          if (mode == 0) unproject_fused_kernel<0, false><<<g, kThreads, 0, h->stream>>>(up);
          else if (mode == 1) unproject_fused_kernel<1, false><<<g, kThreads, 0, h->stream>>>(up);
          else unproject_fused_kernel<2, false><<<g, kThreads, 0, h->stream>>>(up);
        }
        prof_end(h, span);
        ++h->launches;
        if (cloud_out) {
          blocked_to_aos_range_kernel<<<g, kThreads, 0, h->stream>>>(h->pts.p, h->slab_totals.p + s, cloud_napari,
                                                                     h->cloud_aos.p);
          ++h->launches;
        }
        done_chunks = c_end;
      } else {
        CU(cudaMemcpyAsync(h->slab_totals.p + s + 1, h->slab_totals.p + s, 8, cudaMemcpyDeviceToDevice, h->stream));
      }
      CU(cudaGetLastError());
      OK(small_d2h(h, h->h_slab_totals + s + 1, h->slab_totals.p + s + 1, 8, /*dst_is_pinned=*/true));
      CU(cudaEventRecord(h->slab_ev[2 * s + 1], h->stream));
      begin = end;
    }
    h->h_slab_totals[0] = 0;
    // segments: where each day of the range starts in the output
    const long long d_first = pix_begin / HW, d_last = (pix_begin + pix_count - 1) / HW;
    const int n_seg = (int)(d_last - d_first + 1);
    OK(ensure(h, h->d_seg_off, (size_t)n_seg + 1));
    if (n_seg > 1) {
      day_offsets_kernel<<<n_seg - 1, 32, 0, h->stream>>>(up, n_seg, h->d_seg_off.p);
      ++h->launches;
      CU(cudaGetLastError());
    }
    h->seg_off.assign((size_t)n_seg + 1, 0);
    if (n_seg > 1) OK(small_d2h(h, h->seg_off.data() + 1, h->d_seg_off.p + 1, (size_t)(n_seg - 1) * 8));
    // result copies: as soon as the host knows how many points a slab produced
    for (int s = 0; s < n_slabs; ++s) {
      CU(cudaEventSynchronize(h->slab_ev[2 * s + 1]));
      const long long a = h->h_slab_totals[s], b = h->h_slab_totals[s + 1];
      if (cloud_out && b > a) {
        CU(cudaStreamWaitEvent(h->d2h_stream, h->slab_ev[2 * s + 1], 0));
        CU(cudaMemcpyAsync(cloud_out + a * 3, h->cloud_aos.p + a * 3, (size_t)(b - a) * 12, cudaMemcpyDeviceToHost,
                           h->d2h_stream));
        h->d2h_pending = true;
      }
    }
    unsigned int lookback_fault = 0;
    OK(small_d2h(h, &lookback_fault, up.ticket + 1, 4));
    OK(sync_small(h));
    if (lookback_fault) return fail(h, MDKM_ERR_CUDA, "unprojection: a tile's look-back timed out");
    n_out = h->h_slab_totals[n_slabs];
    h->seg_off[n_seg] = n_out;
    h->seg_whole = (pix_begin % HW) == 0 && (pix_count % HW) == 0;
  } else {
    h->seg_off.assign({0, 0});
    h->seg_whole = true;
  }
  h->n = n_out;
  h->raster_w = W;
  h->raster_H = H;
  h->raster_pix_begin = pix_begin;
  h->raster_pix_count = pix_count;
  h->stack_days = D;
  h->day0 = pix_begin / ((long long)H * W);
  if (want_runs) {
    const unsigned int n32 = (unsigned int)n_out;  // closes the table
    CU(cudaMemcpyAsync(h->run_src.p + pix_count / 8, &n32, 4, cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));  // (n32 lives on this stack frame)
    h->runs_ok = true;
    h->run_row0 = pix_begin / W;
    h->run_rows = pix_count / W;
    h->run_H = H;
  }
  OK(zero_tail(h));
  h->have_points = true;
  h->frame_ok = false;
  OK(compute_frame(h, /*minmax_ready=*/pix_count > 0));
  if (n_points_out) *n_points_out = n_out;
  return MDKM_OK;
}

static int get_cloud_impl(mdkm_handle* h, float* out, int napari_order, int mem, bool async) {
  if (!h || !out) return fail(h, MDKM_ERR_INVALID, "null argument");
  if (!h->have_points) return fail(h, MDKM_ERR_STATE, "no points resident");
  CU(cudaSetDevice(h->device));
  OK(wait_pending(h));  // the staging buffer below may still be in flight
  if (h->n == 0) return MDKM_OK;
  float* dst = out;
  if (mem != MDKM_MEM_DEVICE) {
    OK(ensure(h, h->cloud_aos, (size_t)h->n * 3));
    dst = h->cloud_aos.p;
  }
  blocked_to_aos_kernel<<<grid_for(h, (h->n * 3 + kThreads - 1) / kThreads, resident_per_sm(h, blocked_to_aos_kernel)), kThreads, 0, h->stream>>>(
      h->pts.p, h->n, napari_order, dst);
  ++h->launches;
  CU(cudaGetLastError());
  if (mem != MDKM_MEM_DEVICE) {
    // the copy runs on the side stream so that later kernels of this handle overlap it
    CU(cudaEventRecord(h->ev_ready, h->stream));
    CU(cudaStreamWaitEvent(h->d2h_stream, h->ev_ready, 0));
    CU(cudaMemcpyAsync(out, dst, (size_t)h->n * 12, cudaMemcpyDeviceToHost, h->d2h_stream));
    h->d2h_pending = true;
    if (!async) OK(wait_pending(h));
  } else if (!async) {
    CU(cudaStreamSynchronize(h->stream));
  }
  return MDKM_OK;
}

int mdkm_get_cloud(mdkm_handle* h, float* out, int napari_order, int mem) {
  return get_cloud_impl(h, out, napari_order, mem, false);
}

int mdkm_get_cloud_async(mdkm_handle* h, float* out, int napari_order, int mem) {
  return get_cloud_impl(h, out, napari_order, mem, true);
}

int mdkm_wait(mdkm_handle* h) {
  if (!h) return MDKM_ERR_INVALID;
  CU(cudaSetDevice(h->device));
  OK(wait_pending(h));
  CU(cudaStreamSynchronize(h->stream));
  return MDKM_OK;
}

int mdkm_fit(mdkm_handle* h, int k, const double* init, int max_iter, double tol, int32_t* labels_out,
             int labels_mem, double* centroids_out, int* n_iter_out, double* inertia_out) {
  if (!h) return MDKM_ERR_INVALID;
  CallOutputs outs;
  OK(take_outputs(h, k, outs));
  if (!init) return fail(h, MDKM_ERR_INVALID, "init centroids required");
  OK(check_centroids(h, k, init, "init"));
  if (max_iter < 1) return fail(h, MDKM_ERR_INVALID, "max_iter must be >= 1");
  if (tol < 0) return fail(h, MDKM_ERR_INVALID, "tol must be >= 0");
  CU(cudaSetDevice(h->device));
  KmBuffers kb{};
  OK(prepare_kmeans(h, k, kb));

  // sklearn/_kmeans.py:285-293: _tol = mean(var(X, axis=0)) * tol  (0 when tol == 0)
  double tol_scaled = 0.0;
  if (tol > 0) {
    double mv = 0.0;
    OK(compute_moments(h, &mv));
    tol_scaled = mv * tol;
  }
  h->stat_tol = tol_scaled;

  DevStatus st0{};
  st0.max_iter = max_iter;
  st0.k = k;
  st0.first = 1;
  st0.tol = tol_scaled;
  st0.epoch = h->epoch_base;
  const size_t acc_slot = (size_t)kb.kpad * 4 + 8;
  h->step_seq = 0;
  OK(fit_head(h, kb, st0, init, /*acc_slots=*/3));

  // the host-sequenced rare path (empty cluster): everything behind the pause has left early;
  // relocate on the device from the parked global sums, finish the paused iteration
  long long relocs = 0;
  int guard = 0;
  auto relocate_and_resume = [&](const DevStatus& s, int& enq) -> int {
    if (!h->mean_ok) OK(compute_moments(h, nullptr));
    CU(cudaMemcpyAsync(h->acc.p, h->acc.p + 3 * acc_slot, acc_slot * 8, cudaMemcpyDeviceToDevice, h->stream));
    OK(relocate_empty(h, kb, s.n_empty));
    relocs += s.n_empty;
    OK(launch_update(h, kb, /*allow_pause=*/0, 0));
    enq = s.iter + 1;
    if (++guard > max_iter + 8) return fail(h, MDKM_ERR_STATE, "relocation loop did not terminate");
    return MDKM_OK;
  };

  // Lloyd loop: batches of iterations are enqueued back to back; the host only looks at the
  // device status between batches, one batch behind the GPU (no per-iteration sync).  Once the last
  // batch is enqueued the end of the fit goes right behind it, without waiting: a pause or an early
  // exit makes every later kernel return at once, the final pass does nothing on a pause, and the
  // host, after its one synchronisation, relocates and runs the end again.
  int enq = 0;  // iterations enqueued that can still complete
  for (;;) {  // (one pass, unless an update finds an empty cluster in the last batch)
    int inflight = 0, head = 0, tail = 0;
    while (true) {
      while (inflight < 2 && enq < max_iter) {
        const int nb = std::min(kBatch, max_iter - enq);
        // profiling: one event pair around the batch's step kernels (back-to-back launches, so
        // the figure is immune to host-side enqueue gaps); only fused batches are bracketed
        const int span = can_fuse(h) ? prof_begin(h, MDKM_PHASE_STEP, nb) : -1;
        for (int b = 0; b < nb; ++b) {
          if (can_fuse(h)) {
            OK(launch_step(h, kb, 0, /*fuse_update=*/1));
          } else {
            OK(launch_step(h, kb, 0));
            OK(allreduce(h, h->acc.p, acc_slot, kNcclUint64, kNcclSum));
            OK(launch_update(h, kb, /*allow_pause=*/1, 0));
          }
        }
        prof_end(h, span);
        enq += nb;
        if (enq >= max_iter) break;  // (the end of the fit publishes the status of the last batch)
        OK(small_d2h(h, &h->h_status[tail], h->d_status, sizeof(DevStatus), /*dst_is_pinned=*/true));
        CU(cudaEventRecord(h->batch_ev[tail], h->stream));
        tail ^= 1;
        ++inflight;
      }
      if (enq >= max_iter) break;
      CU(cudaEventSynchronize(h->batch_ev[head]));
      const DevStatus s = h->h_status[head];
      head ^= 1;
      --inflight;
      if (s.paused && !s.done) {
        CU(cudaStreamSynchronize(h->stream));
        inflight = 0;
        head = tail = 0;
        if (can_fuse(h)) OK(launch_settle(h, kb));  // the table the paused update starts from -> table[0]
        OK(relocate_and_resume(s, enq));
        continue;
      }
      if (s.done) break;
    }
    // (no synchronisation here: everything below is ordered behind the loop on the stream)
    // fused launches leave the last E-step's update to their successor: apply it now
    if (can_fuse(h)) OK(launch_settle(h, kb));

    // final E-step (unless strict) + inertia + int32 labels
    int* labels_dev = nullptr;
    if (labels_out) {
      if (labels_mem == MDKM_MEM_DEVICE) {
        labels_dev = labels_out;
      } else {
        OK(ensure(h, h->labels32, (size_t)std::max<long long>(h->n, 1)));
        labels_dev = h->labels32.p;
      }
    }
    // one rank: the final kernel's last CTA also writes the centroids and the status to the host;
    // several: the inertia is summed over the ranks first
    const bool one_rank = h->n_ranks == 1;
    double* centroids_host = nullptr;
    if (one_rank && centroids_out) {
      const size_t bytes = (size_t)k * 3 * sizeof(double);
      const size_t off = (h->mapped_used + 15) & ~(size_t)15;
      if (off + bytes > kMappedBytes) return fail(h, MDKM_ERR_INVALID, "small result buffer exhausted");
      h->mapped_used = off + bytes;
      h->small_pending.push_back({centroids_out, off, bytes});
      centroids_host = reinterpret_cast<double*>(h->mapped + off);
    }
    // labels in the reference's point order: always recomputed from the final centroids (the
    // stored ones follow the mirror's order).  After a strict exit the table equals the one the
    // last E-step used -- the sums are integers -- so this reproduces that step's labels exactly.
    {
      const int span = prof_begin(h, MDKM_PHASE_FINAL, h->n);
      // (a pause leaves the map alone: the pass after the relocation writes it)
      OK(run_final(h, kb, labels_dev, /*skip_paused=*/true, centroids_host, one_rank ? &h->h_status[0] : nullptr,
                   &outs.map, &outs.stats));
      prof_end(h, span);
    }
    OK(reduce_outputs(h, outs));
    if (!one_rank) {
      OK(ensure(h, h->dscratch, (size_t)k * 3 + 16));
      read_table_kernel<<<(k + 255) / 256, 256, 0, h->stream>>>(h->table.p, k, kb.kpad, h->fr, h->dscratch.p);
      ++h->launches;
      CU(cudaGetLastError());
      OK(allreduce(h, &h->d_status->inertia, 1, kNcclFloat64, kNcclSum));
      if (centroids_out) OK(small_d2h(h, centroids_out, h->dscratch.p, (size_t)k * 3 * sizeof(double)));
      OK(small_d2h(h, &h->h_status[0], h->d_status, sizeof(DevStatus), /*dst_is_pinned=*/true));
    }
    if (labels_out && labels_mem != MDKM_MEM_DEVICE && h->n > 0)
      CU(cudaMemcpyAsync(labels_out, labels_dev, (size_t)h->n * 4, cudaMemcpyDeviceToHost, h->stream));
    OK(copy_cluster_map(h, outs.map));
    OK(sync_small(h));
    if (h->h_status[0].paused && !h->h_status[0].done && !h->h_status[0].xchg_timeout) {
      // an update of the last batch, or the settle kernel, found an empty cluster: relocate, go on
      const DevStatus s = h->h_status[0];
      OK(relocate_and_resume(s, enq));
      continue;
    }
    break;
  }
  const DevStatus& fin = h->h_status[0];
  h->epoch_base = fin.epoch;
#ifdef MDKM_TIMING
  fprintf(stderr, "[mdkm timing] deferred update: sums and vote +%.2f us | rows and reductions +%.2f us\n",
          ((double)fin.t_a - (double)fin.t_start) * 1e-3, ((double)fin.t_b - (double)fin.t_start) * 1e-3);
  fprintf(stderr, "[mdkm timing] last iteration: table ready +%.1f us | latest end of pass 1 +%.1f us | after grid barrier +%.1f us | CTAs done on average +%.1f us, last +%.1f us\n",
          ((double)fin.t_classify_start - (double)fin.t_start) * 1e-3, ((double)fin.t_first_done - (double)fin.t_start) * 1e-3,
          (fin.t_classify_done - fin.t_start) * 1e-3, (double)fin.t_update_done * 1e-3 / std::max(1, kb.step_grid),
          (fin.t_last_done - fin.t_start) * 1e-3);
#endif
  if (fin.xchg_timeout == 2) return index_fault(h);
  if (fin.xchg_timeout) return fail(h, MDKM_ERR_NCCL, "a kernel-side wait timed out (peer exchange of the partial sums: a rank is missing; or the grid barrier)");
  OK(deliver_outputs(h, outs));
  if (n_iter_out) *n_iter_out = fin.iter;
  if (inertia_out) *inertia_out = fin.inertia;
  h->stat_refined = (long long)fin.n_refined;
  h->stat_reloc = relocs;
  h->stat_work = (long long)fin.work_sum;
  h->stat_groups = kb.n_groups;
  OK(collect_profile(h));
  return MDKM_OK;
}

int mdkm_fit_worklist(const mdkm_handle* h, int64_t* worklist_groups, int64_t* groups) {
  if (!h) return MDKM_ERR_INVALID;
  if (worklist_groups) *worklist_groups = h->stat_work;
  if (groups) *groups = h->stat_groups;
  return MDKM_OK;
}

int mdkm_fit_stats(const mdkm_handle* h, int64_t* n_refined, int64_t* n_relocations, double* tol_scaled) {
  if (!h) return MDKM_ERR_INVALID;
  if (n_refined) *n_refined = h->stat_refined;
  if (n_relocations) *n_relocations = h->stat_reloc;
  if (tol_scaled) *tol_scaled = h->stat_tol;
  return MDKM_OK;
}

int mdkm_lloyd_step(mdkm_handle* h, int k, const double* centroids, int32_t* labels_out, int labels_mem,
                    double* sums_out, int64_t* counts_out) {
  if (!h) return MDKM_ERR_INVALID;
  if (!centroids) return fail(h, MDKM_ERR_INVALID, "centroids required");
  OK(check_centroids(h, k, centroids, "centroids"));
  CU(cudaSetDevice(h->device));
  KmBuffers kb{};
  OK(prepare_kmeans(h, k, kb));
  DevStatus st0{};
  st0.max_iter = 1;
  st0.k = k;
  st0.first = 1;
  st0.epoch = h->epoch_base;
  OK(fit_head(h, kb, st0, centroids, /*acc_slots=*/1));
  OK(launch_step(h, kb, 1));
  OK(allreduce(h, h->acc.p, (size_t)kb.kpad * 4 + 8, kNcclUint64, kNcclSum));
  OK(ensure(h, h->dscratch, (size_t)k * 4 + 16));
  long long* d_counts = reinterpret_cast<long long*>(h->dscratch.p + (size_t)k * 3);
  read_sums_kernel<<<(k + 255) / 256, 256, 0, h->stream>>>(h->acc.p, k, h->fr, h->dscratch.p, d_counts);
  ++h->launches;
  CU(cudaGetLastError());
  if (sums_out) OK(small_d2h(h, sums_out, h->dscratch.p, (size_t)k * 3 * sizeof(double)));
  if (counts_out) OK(small_d2h(h, counts_out, d_counts, (size_t)k * 8));
  if (labels_out) {
    // widen the stored labels: the final kernel in "use stored labels" mode
    int* labels_dev = labels_out;
    if (labels_mem != MDKM_MEM_DEVICE) {
      OK(ensure(h, h->labels32, (size_t)std::max<long long>(h->n, 1)));
      labels_dev = h->labels32.p;
    }
    OK(run_final(h, kb, labels_dev));
    if (labels_mem != MDKM_MEM_DEVICE && h->n > 0)
      CU(cudaMemcpyAsync(labels_out, labels_dev, (size_t)h->n * 4, cudaMemcpyDeviceToHost, h->stream));
  }
  OK(small_d2h(h, &h->h_status[0], h->d_status, sizeof(DevStatus), /*dst_is_pinned=*/true));
  OK(sync_small(h));
  h->stat_refined = (long long)h->h_status[0].n_refined;
  h->stat_reloc = 0;
  OK(collect_profile(h));
  if (h->h_status[0].xchg_timeout == 2) return index_fault(h);
  if (h->h_status[0].xchg_timeout) return fail(h, MDKM_ERR_CUDA, "the step kernel's grid barrier timed out");
  return MDKM_OK;
}

int mdkm_predict(mdkm_handle* h, int k, const double* centroids, int32_t* labels_out, int labels_mem,
                 double* inertia_out) {
  if (!h) return MDKM_ERR_INVALID;
  CallOutputs outs;
  OK(take_outputs(h, k, outs));
  if (!centroids) return fail(h, MDKM_ERR_INVALID, "centroids required");
  OK(check_centroids(h, k, centroids, "centroids"));
  CU(cudaSetDevice(h->device));
  KmBuffers kb{};
  OK(prepare_kmeans(h, k, kb));
  DevStatus st0{};
  st0.max_iter = 1;
  st0.k = k;
  st0.first = 1;
  st0.epoch = h->epoch_base;
  OK(fit_head(h, kb, st0, centroids, /*acc_slots=*/0));
  int* labels_dev = nullptr;
  if (labels_out) {
    labels_dev = labels_out;
    if (labels_mem != MDKM_MEM_DEVICE) {
      OK(ensure(h, h->labels32, (size_t)std::max<long long>(h->n, 1)));
      labels_dev = h->labels32.p;
    }
  }
  OK(run_final(h, kb, labels_dev, false, nullptr, nullptr, &outs.map, &outs.stats));
  if (h->n_ranks > 1) OK(allreduce(h, &h->d_status->inertia, 1, kNcclFloat64, kNcclSum));
  OK(reduce_outputs(h, outs));
  OK(small_d2h(h, &h->h_status[0], h->d_status, sizeof(DevStatus), /*dst_is_pinned=*/true));
  if (labels_out && labels_mem != MDKM_MEM_DEVICE && h->n > 0)
    CU(cudaMemcpyAsync(labels_out, labels_dev, (size_t)h->n * 4, cudaMemcpyDeviceToHost, h->stream));
  OK(copy_cluster_map(h, outs.map));
  OK(sync_small(h));
  if (h->h_status[0].xchg_timeout == 2) return index_fault(h);
  OK(deliver_outputs(h, outs));
  if (inertia_out) *inertia_out = h->h_status[0].inertia;
  h->stat_refined = (long long)h->h_status[0].n_refined;
  h->stat_reloc = 0;
  return MDKM_OK;
}

int mdkm_num_segments(const mdkm_handle* h) { return h && h->have_points ? (int)h->seg_off.size() - 1 : -1; }

int mdkm_segment_offsets(const mdkm_handle* h, int64_t* out) {
  if (!h || !out || !h->have_points) return MDKM_ERR_INVALID;
  for (size_t i = 0; i < h->seg_off.size(); ++i) out[i] = h->seg_off[i];
  return MDKM_OK;
}

int mdkm_ground_level(mdkm_handle* h, float* height_norm_out, int mem, double* h_min_out, double* h_max_out) {
  if (!h) return MDKM_ERR_INVALID;
  if (!h->have_points) return fail(h, MDKM_ERR_STATE, "no points resident");
  if (!h->seg_whole)
    return fail(h, MDKM_ERR_STATE, "mdkm_ground_level needs whole days on this rank (shard the stack by days)");
  CU(cudaSetDevice(h->device));
  const int n_seg = (int)h->seg_off.size() - 1;
  OK(ensure(h, h->d_seg_off, (size_t)n_seg + 1));
  OK(ensure(h, h->sel_hist, (size_t)n_seg * kSelTargets * kSelBins));
  OK(ensure(h, h->sel_targets, (size_t)n_seg * kSelTargets * sizeof(SelTarget)));
  OK(ensure(h, h->planes, (size_t)n_seg * 2 + 8));
  CU(cudaMemcpyAsync(h->d_seg_off.p, h->seg_off.data(), (size_t)(n_seg + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemsetAsync(h->sel_hist.p, 0, (size_t)n_seg * kSelTargets * kSelBins * 4, h->stream));
  // numpy "linear" percentile: virtual index (n-1)*q, neighbours floor / floor+1
  // (numpy/lib/_function_base_impl.py: _QuantileMethods['linear'], _get_indexes, _lerp)
  const double qs[2] = {2.0 / 100.0, 98.0 / 100.0};
  std::vector<SelTarget> tg((size_t)n_seg * kSelTargets);
  std::vector<double> gam((size_t)n_seg * 2, 0.0);
  for (int s = 0; s < n_seg; ++s) {
    const long long ns = h->seg_off[s + 1] - h->seg_off[s];
    for (int q = 0; q < 2; ++q) {
      long long prev = 0, next = 0;
      double g = 0.0;
      if (ns > 0) {
        const double v = (double)(ns - 1) * qs[q];
        prev = (long long)floor(v);
        next = prev + 1;
        g = v - (double)prev;
        if (v >= (double)(ns - 1)) { prev = next = ns - 1; g = v - (-1.0); }
        if (v < 0) { prev = next = 0; }
      }
      tg[(size_t)s * kSelTargets + 2 * q + 0] = SelTarget{0u, 0u, prev};
      tg[(size_t)s * kSelTargets + 2 * q + 1] = SelTarget{0u, 0u, next};
      gam[(size_t)s * 2 + q] = g;
    }
  }
  CU(cudaMemcpyAsync(h->sel_targets.p, tg.data(), tg.size() * sizeof(SelTarget), cudaMemcpyHostToDevice, h->stream));
  SelParams sp{};
  sp.pts = h->pts.p;
  sp.seg_off = h->d_seg_off.p;
  sp.hist = h->sel_hist.p;
  sp.targets = reinterpret_cast<SelTarget*>(h->sel_targets.p);
  sp.n_seg = n_seg;
  const int shifts[3] = {21, 10, 0}, bits[3] = {11, 11, 10}, pshift[3] = {32, 21, 10};
  for (int pass = 0; pass < 3; ++pass) {
    sp.shift = shifts[pass]; sp.bits = bits[pass]; sp.prefix_shift = pshift[pass];
    select_hist_kernel<<<dim3(kSelCtasPerSeg, n_seg), kThreads, 0, h->stream>>>(sp);
    select_pick_kernel<<<n_seg, kSelTargets * 32, 0, h->stream>>>(sp);
    h->launches += 2;
    CU(cudaGetLastError());
  }
  OK(small_d2h(h, tg.data(), h->sel_targets.p, tg.size() * sizeof(SelTarget)));
  OK(sync_small(h));
  std::vector<double> levels((size_t)n_seg * 2, 0.0);
  for (int s = 0; s < n_seg; ++s) {
    const long long ns = h->seg_off[s + 1] - h->seg_off[s];
    double pc[2] = {NAN, NAN};
    if (ns > 0) {
      for (int q = 0; q < 2; ++q) {
        const double a = (double)ord2f(tg[(size_t)s * kSelTargets + 2 * q + 0].prefix);
        const double b = (double)ord2f(tg[(size_t)s * kSelTargets + 2 * q + 1].prefix);
        const double t = gam[(size_t)s * 2 + q];
        const double diff = b - a;
        double r = a + diff * t;              // numpy _lerp
        if (t >= 0.5) r = b - diff * (1.0 - t);
        pc[q] = r;
      }
    }
    if (h_min_out) h_min_out[s] = pc[0];
    if (h_max_out) h_max_out[s] = pc[1];
    levels[(size_t)s * 2 + 0] = ns > 0 ? pc[0] : 0.0;
    levels[(size_t)s * 2 + 1] = ns > 0 ? (pc[1] - pc[0] + 1e-6) : 1.0;  // plugin.py:183
  }
  if (h->n > 0) {
    CU(cudaMemcpyAsync(h->planes.p, levels.data(), levels.size() * 8, cudaMemcpyHostToDevice, h->stream));
    float* hn_dev = height_norm_out;
    if (height_norm_out && mem != MDKM_MEM_DEVICE) {
      OK(ensure(h, h->staging, (size_t)h->n * 4));
      hn_dev = reinterpret_cast<float*>(h->staging.p);
    }
    LevelParams lp{};
    lp.pts = h->pts.p; lp.seg_off = h->d_seg_off.p; lp.levels = h->planes.p;
    lp.height_norm = hn_dev; lp.n = h->n; lp.n_seg = n_seg;
    level_apply_kernel<<<grid_for(h, (h->n + 1023) / 1024, 8), kThreads, (size_t)(n_seg + 1) * 8, h->stream>>>(lp);
    ++h->launches;
    CU(cudaGetLastError());
    OK(zero_tail(h));
    if (height_norm_out && mem != MDKM_MEM_DEVICE)
      CU(cudaMemcpyAsync(height_norm_out, hn_dev, (size_t)h->n * 4, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
  }
  h->frame_ok = false;
  return compute_frame(h);
}

int mdkm_kmeans_plusplus(mdkm_handle* h, int k, int64_t first_index, const double* rand_vals, int n_local_trials,
                         double* centers_out, int64_t* indices_out) {
  if (!h) return MDKM_ERR_INVALID;
  if (!h->have_points) return fail(h, MDKM_ERR_STATE, "no points resident");
  if (!h->frame_ok) OK(compute_frame(h));  // also counts the points of all ranks
  if (k < 1 || k > kMaxK || (long long)k > h->n_total) return fail(h, MDKM_ERR_INVALID, "bad k");
  if (first_index < 0 || first_index >= h->n_total) return fail(h, MDKM_ERR_INVALID, "first_index out of range");
  if (k > 1 && (!rand_vals || n_local_trials < 1 || n_local_trials > kKppMaxTrials))
    return fail(h, MDKM_ERR_INVALID, "rand_vals required and 1 <= n_local_trials <= %d", kKppMaxTrials);
  if (!centers_out) return fail(h, MDKM_ERR_INVALID, "centers_out required");
  if (h->n_ranks > kMaxRanks) return fail(h, MDKM_ERR_STATE, "at most %d ranks", kMaxRanks);
  CU(cudaSetDevice(h->device));
  const bool sharded = h->n_ranks > 1;
  const long long cap = round_up(std::max<long long>(h->n, 1), kGroup);
  const long long n_cells = cap / kGroup;
  const long long n_blk = (n_cells + kKppCellsPerBlock - 1) / kKppCellsPerBlock;
  const int T = k > 1 ? n_local_trials : 1;
  const int grid = grid_for(h, (n_cells + 7) / 8, 8);
  OK(ensure(h, h->kpp_closest, (size_t)cap));
  OK(ensure(h, h->kpp_cell, (size_t)n_cells));
  OK(ensure(h, h->kpp_blk, (size_t)n_blk));
  OK(ensure(h, h->kpp_prefix, (size_t)n_blk));
  OK(ensure(h, h->kpp_partials, (size_t)grid * kKppMaxTrials + kXWords));
  OK(ensure(h, h->kpp_rand, (size_t)std::max(1, (k - 1) * T)));
  OK(ensure(h, h->kpp_state, sizeof(KppState)));
  OK(ensure(h, h->dscratch, (size_t)k * 4 + 16 + 2 * kMaxRanks));
  CU(cudaMemsetAsync(h->kpp_state.p, 0, sizeof(KppState), h->stream));
  if (k > 1)
    CU(cudaMemcpyAsync(h->kpp_rand.p, rand_vals, (size_t)(k - 1) * T * 8, cudaMemcpyHostToDevice, h->stream));
  KppParams kp{};
  kp.pts = h->pts.p; kp.n = h->n;
  kp.closest = h->kpp_closest.p; kp.cell_sum = h->kpp_cell.p; kp.blk_sum = h->kpp_blk.p;
  kp.blk_prefix = h->kpp_prefix.p; kp.partials = h->kpp_partials.p; kp.rand_vals = h->kpp_rand.p;
  kp.st = reinterpret_cast<KppState*>(h->kpp_state.p);
  kp.centers_out = h->dscratch.p;
  kp.indices_out = reinterpret_cast<long long*>(h->dscratch.p + (size_t)k * 3);
  kp.n_trials = T;
  kp.first_index = first_index;
  kp.n_ranks = h->n_ranks; kp.rank = h->rank;
  kp.xbuf = h->kpp_partials.p + (size_t)grid * kKppMaxTrials;
  kp.choose = sharded ? 0 : 1;
  double* d_pots = reinterpret_cast<double*>(h->kpp_state.p + offsetof(KppState, pots));
  if (sharded) {
    // who owns centre 0, and which ranks have points at all
    double cnt[kMaxRanks] = {};
    for (int r = 0; r < h->n_ranks; ++r) cnt[r] = (double)h->shard_sizes[r];
    kp.rank_offset = h->rank_offset;
    const long long local = first_index - kp.rank_offset;
    kp.first_index = (local >= 0 && local < h->n) ? local : -1;
    CU(cudaMemsetAsync(kp.xbuf, 0, kXWords * 8, h->stream));
    CU(cudaMemcpyAsync(kp.xbuf + kXCnt, cnt, sizeof(cnt), cudaMemcpyHostToDevice, h->stream));
  }
  KppPotKernel pot_fn = kpp_pot_variant(T);
  // all k rounds are enqueued back to back; nothing returns to the host until the end
  for (int c = 0; c < k; ++c) {
    kp.round = c;
    if (sharded) CU(cudaMemsetAsync(kp.xbuf, 0, kXCnt * 8, h->stream));
    if (c == 0) {
      if (sharded) {
        kpp_first_candidate_kernel<<<1, 32, 0, h->stream>>>(kp);
        OK(allreduce(h, kp.xbuf + kXCand, 4, kNcclFloat64, kNcclSum));
        kpp_unpack_candidates_kernel<<<1, 32, 0, h->stream>>>(kp);
        kpp_choose_kernel<<<1, 32, 0, h->stream>>>(kp);
        h->launches += 3;
      }
    } else {
      kpp_search_kernel<<<1, 1024, 0, h->stream>>>(kp, n_blk);
      ++h->launches;
      if (sharded) {
        OK(allreduce(h, kp.xbuf + kXTot, kMaxRanks, kNcclFloat64, kNcclSum));
        kpp_search_sharded_kernel<<<1, kKppMaxTrials * 32, 0, h->stream>>>(kp, n_blk);
        OK(allreduce(h, kp.xbuf + kXCand, (size_t)T * 4, kNcclFloat64, kNcclSum));
        kpp_unpack_candidates_kernel<<<1, 32, 0, h->stream>>>(kp);
        h->launches += 2;
      }
      pot_fn<<<grid, kThreads, 0, h->stream>>>(kp);
      ++h->launches;
      if (sharded) {
        OK(allreduce(h, d_pots, T, kNcclFloat64, kNcclSum));
        kpp_choose_kernel<<<1, 32, 0, h->stream>>>(kp);
        ++h->launches;
      }
    }
    if (c == 0 || c < k - 1) {  // the last centre has no later draw to prepare
      kpp_commit_kernel<<<(unsigned int)n_blk, kThreads, 0, h->stream>>>(kp);
      ++h->launches;
    }
    CU(cudaGetLastError());
  }
  OK(small_d2h(h, centers_out, kp.centers_out, (size_t)k * 3 * 8));
  if (indices_out) OK(small_d2h(h, indices_out, kp.indices_out, (size_t)k * 8));
  OK(sync_small(h));
  return MDKM_OK;
}

int mdkm_drop_caches(mdkm_handle* h) {
  if (!h) return MDKM_ERR_INVALID;
  h->summary_ok = false;  // tile-ordered mirror + group summaries are rebuilt by the next fit
  return MDKM_OK;
}

int mdkm_profile_enable(mdkm_handle* h, int on) {
  if (!h) return MDKM_ERR_INVALID;
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  h->prof = on != 0;
  h->prof_spans.clear();
  for (int i = 0; i < MDKM_PHASE_COUNT; ++i) {
    h->prof_ms[i] = 0.0;
    h->prof_count[i] = 0;
  }
  return MDKM_OK;
}

int mdkm_profile_read(mdkm_handle* h, double* step_kernel_ms, int* n_step_launches, int* n_kernel_launches_total) {
  if (!h) return MDKM_ERR_INVALID;
  if (step_kernel_ms) *step_kernel_ms = h->prof_ms[MDKM_PHASE_STEP];
  if (n_step_launches) *n_step_launches = (int)h->prof_count[MDKM_PHASE_STEP];
  if (n_kernel_launches_total) *n_kernel_launches_total = h->launches;
  h->prof_ms[MDKM_PHASE_STEP] = 0.0;
  h->prof_count[MDKM_PHASE_STEP] = 0;
  h->launches = 0;
  return MDKM_OK;
}

int mdkm_profile_phase(mdkm_handle* h, int phase, double* ms, int64_t* count) {
  if (!h || phase < 0 || phase >= MDKM_PHASE_COUNT) return MDKM_ERR_INVALID;
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  OK(collect_profile(h));
  if (ms) *ms = h->prof_ms[phase];
  if (count) *count = h->prof_count[phase];
  h->prof_ms[phase] = 0.0;
  h->prof_count[phase] = 0;
  return MDKM_OK;
}

}  // extern "C"
