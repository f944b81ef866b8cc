/* mdkm.h -- C ABI of libmdkm.so: multi-day height-map -> XYZ unprojection + Lloyd k-means
 * on one NVIDIA B200 (sm_100a) per handle.
 *
 * This is the drop-in boundary for the ONE hot path of
 * rafael-alani/3d-point-cloud-multiday-imagery that this project accelerates
 * (SURVEY.md section 8).  The reference is pure Python and has no FFI of its own; each
 * entry point below replaces the Python/NumPy/scikit-learn code it cites, and
 * INTEGRATION.md shows the ctypes stub a maintainer would add to
 * members/rafael/disparity/plugin.py.
 *
 * Conventions
 *   - plain C, no exceptions, no torch types; every call returns MDKM_OK (0) or a negative
 *     mdkm_status; mdkm_last_error(h) gives the text for the last failure on that handle.
 *   - one handle == one CUDA device == one rank.  A handle is used by one host thread at a
 *     time (the reference calls the path from a single napari worker thread,
 *     members/rafael/disparity/widget.py:116-147).
 *   - pointers are host pointers unless the call takes a `mem` argument, in which case
 *     MDKM_MEM_DEVICE means "device pointer on the handle's device" (e.g. a torch tensor's
 *     data_ptr()).  The library never keeps a caller pointer after the call returns.
 *   - there is no CPU fallback: without a usable CUDA device mdkm_create fails.
 */
#ifndef MDKM_H_
#define MDKM_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mdkm_handle mdkm_handle;

typedef enum mdkm_status {
  MDKM_OK = 0,
  MDKM_ERR_INVALID = -1,   /* bad argument */
  MDKM_ERR_CUDA = -2,      /* CUDA runtime error (see mdkm_last_error) */
  MDKM_ERR_NO_DEVICE = -3, /* no CUDA device / wrong architecture */
  MDKM_ERR_STATE = -4,     /* call order (e.g. fit before points are set) */
  MDKM_ERR_NCCL = -5,      /* NCCL missing or failed */
  MDKM_ERR_OOM = -6
} mdkm_status;

enum { MDKM_MEM_HOST = 0, MDKM_MEM_DEVICE = 1 };
/* height raster element type: float32 heights; int16 OpenCV fixed-point disparity; or the
 * reference's own "5-out-F.tif" pixel layout (disparity.py:213-224): three pixel-interleaved
 * float32 bands per pixel, band 0 = height (-disp/16), band 2 = final_defined (0 = invalid) */
enum { MDKM_HM_F32 = 0, MDKM_HM_I16 = 1, MDKM_HM_F32_GTIFF3 = 2 };
enum { MDKM_POINTS_AOS = 0, MDKM_POINTS_SOA = 1 }; /* xyzxyz... or x[n] y[n] z[n] */

#define MDKM_NCCL_UNIQUE_ID_BYTES 128
#define MDKM_IPC_HANDLE_BYTES 64

/* Library / build identification ("mdkm <ver> sm_100a"). */
const char* mdkm_version(void);

/* Create a handle on CUDA device `device`.  `cuda_stream` is an optional cudaStream_t the
 * library should enqueue on (NULL: it creates its own non-blocking stream). */
int mdkm_create(mdkm_handle** out, int device, void* cuda_stream);
void mdkm_destroy(mdkm_handle* h);
const char* mdkm_last_error(const mdkm_handle* h);

/* ---- multi-GPU: one rank per handle, NCCL over NVLink ------------------------------- */
/* Rank 0 makes the id; the caller ships the 128 bytes to the other ranks (the Python
 * host uses torch.distributed for that) and every rank calls mdkm_comm_init. */
int mdkm_comm_unique_id(unsigned char out[MDKM_NCCL_UNIQUE_ID_BYTES]);
int mdkm_comm_init(mdkm_handle* h, int n_ranks, int rank,
                   const unsigned char id[MDKM_NCCL_UNIQUE_ID_BYTES]);

/* Optional, after mdkm_comm_init on every rank (one process per GPU, one node): let the Lloyd
 * step kernel exchange the K x 4 partial sums itself, by stores into peer memory over
 * NVLink, instead of an ncclAllReduce between two kernels.  Each rank exports a CUDA IPC
 * handle of its exchange buffer (mdkm_comm_p2p_handle), the caller gathers the 64-byte
 * handles of all ranks in rank order (the Python host uses torch.distributed) and hands the
 * n_ranks * 64 bytes to mdkm_comm_p2p_open.  If the open fails (no peer access) the call
 * returns MDKM_ERR_NCCL and the NCCL path stays in use.  Collective: all ranks or none. */
int mdkm_comm_p2p_handle(mdkm_handle* h, unsigned char out[MDKM_IPC_HANDLE_BYTES]);
int mdkm_comm_p2p_open(mdkm_handle* h, const unsigned char* handles);
/* Drops the peer mappings (and this rank's exchange buffer) again and keeps the NCCL
 * communicator: the Lloyd iteration goes back to step kernel -> ncclAllReduce -> update kernel.
 * The caller uses it to make the fallback collective: when mdkm_comm_p2p_open failed on ANY
 * rank, EVERY rank calls this (no-op where nothing is open). */
int mdkm_comm_p2p_close(mdkm_handle* h);

/* The same exchange for ranks that live in ONE process (one handle per device, each driven by
 * its own host thread -- the in-process caller of the reference, widget.py:116-147): after
 * mdkm_comm_p2p_handle on every handle, mdkm_comm_p2p_buffer returns the device pointer of this
 * rank's exchange buffer, and mdkm_comm_p2p_open_ptrs takes the n_ranks pointers in rank order
 * (peer access between the devices is enabled by the call; no CUDA IPC involved). */
int mdkm_comm_p2p_buffer(mdkm_handle* h, void** out_device_ptr);
int mdkm_comm_p2p_open_ptrs(mdkm_handle* h, void* const* buffers);

/* The CUDA stream (cudaStream_t) the handle enqueues on, so that a caller that produces inputs
 * or consumes device-resident outputs on another stream can order the two with events. */
void* mdkm_get_stream(const mdkm_handle* h);

/* Tuning / measurement switches.  MDKM_OPT_SETTLE_GROUPS (default 1): 0 disables the
 * classification pass's settling of whole 128-point groups from their cached summaries, so
 * that EVERY point is read and assigned by the per-point pass in every iteration (the
 * streaming path bench.py reports its HBM fraction for); results are identical either way. */
/* MDKM_OPT_RASTER_MIRROR (default 1): 0 makes clouds that came from mdkm_unproject use the generic
 * (histogram + scatter) build of the tile-ordered mirror instead of the run-table build; a test
 * hook, the results are identical.
 * MDKM_OPT_CELL_PX (0 = automatic, 8 or 16) / MDKM_OPT_CELL_ROWS (0 = automatic, 1..64): width and
 * height, in pixels, of the x-y cells the mirror of a raster cloud is ordered by (tuning).
 * MDKM_OPT_TWO_LEVEL (-1 = automatic by cloud size, 0, 1): whether the classification pass of the
 * Lloyd kernel tests super-groups of 1024 points before it looks at 128-point groups.
 * MDKM_OPT_DEPENDENT_LAUNCH (default 1): after the first (cooperative) Lloyd kernel of a fit, the
 * following ones are launched with programmatic stream serialisation -- the next iteration's kernel
 * is set up while the current one drains -- instead of the cooperative attribute (the runtime does
 * not combine the two); 0 = every launch cooperative.  Results are identical. */
enum { MDKM_OPT_SETTLE_GROUPS = 1, MDKM_OPT_RASTER_MIRROR = 2, MDKM_OPT_CELL_PX = 3, MDKM_OPT_CELL_ROWS = 4,
       MDKM_OPT_TWO_LEVEL = 5, MDKM_OPT_DEPENDENT_LAUNCH = 6 };
int mdkm_set_option(mdkm_handle* h, int option, long long value);

/* ---- K1: unprojection ----------------------------------------------------------------
 * Replaces members/rafael/disparity/plugin.py:148 (h = -disp/16), :151-152 (validity:
 * isfinite & |h| <= max_abs & mask), :157-160 ((y,x)=np.where(valid), P=[x,y,z]) and the
 * (absent in the reference) multi-day concatenation, for the pixel range
 * [pix_begin, pix_begin+pix_count) of the flattened [D,H,W] stack.  `hm` / `mask` point at
 * pixel `pix_begin`.  hm_dtype MDKM_HM_F32: heights, used as is (hm_scale ignored);
 * MDKM_HM_I16: OpenCV fixed-point disparity, h = hm_scale * disp (the reference uses
 * -1/16); MDKM_HM_F32_GTIFF3: 12 bytes per pixel, band 2 acts as the validity mask (ANDed
 * with `mask` when that is given too).  mask may be NULL.  detrend != 0 additionally applies the per-day plane fit of
 * plugin.py:161-171 (z becomes the signed distance to the day's least-squares plane); it
 * needs whole days in the range.  The points stay resident in the handle, in np.where
 * order (day-major, row-major); *n_points_out receives how many there are on this rank. */
int mdkm_unproject(mdkm_handle* h, const void* hm, int hm_dtype, float hm_scale,
                   const uint8_t* mask, int D, int H, int W, int64_t pix_begin,
                   int64_t pix_count, float max_abs, int detrend, int mem,
                   int64_t* n_points_out);

/* Optional: have the NEXT mdkm_unproject also stream the cloud it produces into host memory
 * (float32 [n,3]; (z,y,x) columns when napari_order != 0, i.e. plugin.py:192's
 * `points_coords`), slab by slab while later slabs are still being uploaded and unprojected.
 * out_host must hold capacity_points >= pix_count points (the valid count is not known in
 * advance) and should be page-locked.  The binding is consumed by that one call; the array
 * is complete after mdkm_wait (or any later call that touches the cloud). */
int mdkm_bind_cloud_output(mdkm_handle* h, float* out_host, int64_t capacity_points,
                           int napari_order);

/* Optional: have the NEXT mdkm_fit or mdkm_predict on this handle also write its labels as a
 * cluster map over the pixel range [pix_begin, pix_begin + pix_count) of the last
 * mdkm_unproject: a pixel that produced a point holds that point's label + 1, every other
 * pixel 0 (napari's background label).  The map encodes exactly the labels the call returns.
 * elem_bytes: 1 (uint8, k <= 255) or 2 (uint16); out holds capacity_pixels >= pix_count
 * elements, in host or device memory per `mem` (device outputs are written in place on the
 * handle's stream).  The map is written by the final labelling pass itself, without a second
 * pass over the cloud.  out == NULL clears the binding.  The binding is consumed by that one
 * call, and dropped by mdkm_unproject / mdkm_set_points.  Errors: MDKM_ERR_STATE when the
 * resident cloud came from mdkm_set_points (it has no raster); MDKM_ERR_INVALID for a bad
 * elem_bytes or a capacity that is too small here, and from the mdkm_fit / mdkm_predict, before
 * any work is enqueued, when k labels do not fit elem_bytes. */
int mdkm_bind_cluster_map(mdkm_handle* h, void* out, int elem_bytes, int64_t capacity_pixels,
                          int mem);

/* Optional: have the NEXT mdkm_fit or mdkm_predict on this handle also return the composition
 * of every day by cluster.  counts_out (int64) receives n_days * k counts, means_out (float64)
 * n_days * k * 3 coordinates, both row-major [day][cluster] with the k of that call; both are
 * host memory holding at least n_days * k_capacity rows.  counts_out[d*k + j] is the number of
 * points of day d whose returned label is j; means_out[(d*k + j)*3 + c] is the mean of their
 * coordinate c (x, y, z) in the frame that was clustered (after detrending / ground levelling,
 * like the centroids), NaN where the count is 0.  Rows are the global days of the stack:
 * n_days is the D of the last mdkm_unproject (1 after mdkm_set_points), and with several ranks
 * every rank receives the sums over all ranks.
 * Where the numbers come from: the final labelling pass adds every point's fixed-point
 * coordinates (the integers the Lloyd sums use) into an int64 slot per (day, cluster); the
 * ranks' slots are summed with one all-reduce, and each mean is (sum_q / scale + count *
 * origin) / count in float64.  The integer sums do not depend on the point order, the number of
 * ranks or the schedule, so the results are bitwise reproducible; a mean is within half a grid
 * step of the exact mean, and is the correctly rounded exact mean when the points lie on the
 * grid.  Asking for them changes no other result of the call.
 * counts_out == NULL clears the binding.  The binding is consumed by that one call, and dropped
 * by mdkm_unproject / mdkm_set_points.  Errors: MDKM_ERR_STATE when no points are resident;
 * MDKM_ERR_INVALID when n_days is not the stack's day count, means_out is NULL or k_capacity < 1
 * (n_days * k_capacity < 2^29), and from the mdkm_fit / mdkm_predict, before any work is
 * enqueued, when its k exceeds k_capacity. */
int mdkm_bind_day_stats(mdkm_handle* h, int64_t* counts_out, double* means_out, int n_days,
                        int k_capacity);

/* Optional: have the NEXT mdkm_fit or mdkm_predict on this handle also return the from-to
 * (transition) counts of pairs of days.  A pixel's state on a day is label + 1 when the pixel
 * produced a point that day and 0 when it did not -- the value of the cluster map.  For pair p =
 * (a, b), pairs[2p] = a and pairs[2p+1] = b (global days of the stack; any order, repeats and
 * a == b allowed; copied by this call), counts_out[(p*(k+1) + s)*(k+1) + t] is the number of
 * pixels of the H x W grid with state s on day a and t on day b, with the k of that call: row 0
 * counts the pixels that gain their point, column 0 those that lose it.  counts_out is host
 * memory with room for n_pairs * (k_capacity + 1)^2 counts.  With several ranks every rank
 * receives the counts of the whole stack.
 * Where the numbers come from: the final labelling pass writes the cluster map (the bound one,
 * or an internal one when none is bound); a kernel bins it behind that pass.  With several ranks
 * each rank writes its band of a zeroed whole-stack map, the bands are merged with one byte-wise
 * all-reduce (a full-stack map on every rank), each rank bins 1/n_ranks of the pixels, and one
 * all-reduce of the int64 counts sums them: the same bits on any number of ranks.  Asking for
 * them changes no other result of the call.
 * counts_out == NULL clears the binding.  The binding is consumed by that one call, and dropped
 * by mdkm_unproject / mdkm_set_points.  Errors: MDKM_ERR_STATE when the resident cloud did not
 * come from mdkm_unproject; MDKM_ERR_INVALID when pairs is NULL, n_pairs < 1, k_capacity < 1, a
 * day is outside [0, D) or n_pairs * (k_capacity + 1)^2 >= 2^31; from the mdkm_fit /
 * mdkm_predict, before any work is enqueued, MDKM_ERR_INVALID when its k exceeds k_capacity, and
 * MDKM_ERR_STATE on every rank when the ranks' pixel ranges do not cover the whole stack (their
 * pixel counts summed by one all-reduce, once per cloud; one handle without a communicator must
 * hold the whole stack). */
int mdkm_bind_day_transitions(mdkm_handle* h, const int32_t* pairs, int n_pairs, int64_t* counts_out,
                              int k_capacity);

/* Optional: have the NEXT mdkm_fit or mdkm_predict on this handle also find the connected regions
 * of its cluster map.  A region is a maximal set of pixels of one day that all have the same
 * non-zero map value (label + 1) and are connected: connectivity 4 (edge neighbours) or 8 (edge
 * and corner neighbours).  Pixels without a point belong to no region; regions never span days.
 * Regions are numbered 1..R over the whole stack in the raster order (day, y, x) of each region's
 * first pixel, which does not depend on the schedule or the number of ranks.
 * map_out (optional, int32, host or device memory per mem, room for capacity_pixels >= the
 * pix_count of the last mdkm_unproject) receives the region map of that pixel range: the region
 * id of every pixel that produced a point, 0 elsewhere.
 * After the call, mdkm_region_count gives R and mdkm_region_table copies the table, int64
 * [R][7] rows (day, cluster (0-based label), pixels (= its point count), y_min, x_min, y_max,
 * x_max; inclusive bounds in pixel coordinates of the day), and the means, float64 [R][3], the
 * mean (x, y, z) of the region's points in the frame that was clustered -- computed as the means
 * of mdkm_bind_day_stats (int64 sums of fixed-point coordinates of the handle's frame, (sum_q /
 * scale + count * origin) / count), with every coordinate rounded to its nearest grid point in
 * FP64: bitwise the same on any number of ranks, within half a grid step of the exact mean even
 * for a region of one point, exact on the grid.  The
 * pixels of the regions of (day d, cluster j) add up to that day's count of cluster j.
 * Where the numbers come from: after the call's synchronisation, when the map is final, a
 * block-based union-find labels the whole-stack map on the device (tile-local union-find in
 * shared memory, links across tile borders with atomicMin, ids by a scan of the roots); one more
 * synchronisation reads R; a pass over the resident points sums each region's count, coordinates
 * and bounds; with several ranks every rank labels the whole stack (the map is merged as for day
 * transitions) and the sums are all-reduced.  Asking for regions changes no other result.
 * connectivity == 0 with map_out == NULL clears the binding.  The binding is consumed by that one
 * call, and dropped by mdkm_unproject / mdkm_set_points.  Errors: MDKM_ERR_STATE when the resident
 * cloud did not come from mdkm_unproject; MDKM_ERR_INVALID for a connectivity other than 4 or 8,
 * a stack of 2^31 pixels or more, H or W of 2^23 or more, a capacity below pix_count or a bad
 * mem; from the mdkm_fit / mdkm_predict, before any work is enqueued, MDKM_ERR_STATE on every
 * rank when the ranks' pixel ranges do not cover the whole stack (as for day transitions). */
int mdkm_bind_regions(mdkm_handle* h, int connectivity, int32_t* map_out, int64_t capacity_pixels, int mem);

/* The regions of the last mdkm_fit / mdkm_predict that had them bound, kept on the device until
 * the next mdkm_unproject / mdkm_set_points or fit / predict with regions.  mdkm_region_count:
 * their number R.  mdkm_region_table: copies the table (table_out, int64 [R][7]) and the means
 * (means_out, float64 [R][3]) to host memory; either may be NULL.  Errors: MDKM_ERR_STATE when
 * there are no regions (none computed since the last unproject / set_points);
 * MDKM_ERR_INVALID from mdkm_region_table when capacity_regions < R. */
int mdkm_region_count(const mdkm_handle* h, int64_t* n_regions);
int mdkm_region_table(mdkm_handle* h, int64_t* table_out, double* means_out, int64_t capacity_regions);

/* Optional: have the NEXT mdkm_fit or mdkm_predict on this handle, which must also have regions
 * bound (mdkm_bind_regions), return the overlaps of the regions of pairs of days: which object of
 * day a became which object of day b.  For pair p = (a, b), pairs[2p] = a and pairs[2p+1] = b
 * (global days of the stack; any order, repeats and a == b allowed; copied by this call), there is
 * one row for every pair of regions (r of day a, s of day b) such that at least one pixel (y, x)
 * lies in r on day a and in s on day b; r and s may have different clusters.
 * After the call, mdkm_region_overlap_count gives the number of rows M and
 * mdkm_region_overlap_table copies them, int64 [M][6]: pair, region_a, region_b, pixels (shared
 * pixels), y_first, x_first (the first shared pixel in raster order).  Rows are sorted by pair,
 * then by the raster order of their first shared pixel -- the rule that numbers the regions -- so
 * they do not depend on the schedule or the number of ranks.  For a == b the rows are (r, r,
 * pixels of r, first pixel of r) for every region of day a, in id order; the rows of (b, a) are
 * those of (a, b) with columns 1 and 2 swapped, in the same order; summed by (cluster of r,
 * cluster of s) the pixels are the transition counts of the pair without row and column 0.
 * Where the numbers come from: behind the region ids, a pass counts for every pair the pixels
 * where both ids are non-zero and the (id_a, id_b) key differs from the left neighbour's or x ==
 * 0, an upper bound on the pair's rows, read by the synchronisation that reads R (no extra one).
 * Each pair gets an open-addressing hash table of 16-byte slots (the smallest power of two >= 2 x
 * its bound); equal keys are combined in the warp, and their leaders add the pixels and lower the
 * first pixel with atomics.  Every occupied slot sets the bit of its first pixel in an H*W-bit mask
 * per pair, a popcount scan of the masks gives each slot its row, and one more synchronisation
 * reads M.  Memory: 16 B x table capacity (<= 64 B per pixel and pair) plus 8 B per 32 pixels and
 * pair (mask and scan offsets), plus 48 B per row; the worst case, where every pixel is a row, is
 * a one-pixel checkerboard against its one-pixel shift (about 112 B per pixel and pair).  A failed
 * allocation returns MDKM_ERR_OOM.  With several ranks every rank builds the whole table from its
 * whole-stack region map: no collective, the same bits on every rank, and every rank pays the
 * whole cost.  Asking for overlaps changes no other result of the call.
 * pairs == NULL clears the binding.  The binding is consumed by that one call, and dropped by
 * mdkm_unproject / mdkm_set_points.  Errors: MDKM_ERR_STATE when the resident cloud did not come
 * from mdkm_unproject; MDKM_ERR_INVALID when n_pairs < 1 or n_pairs > 8192, or a day is outside
 * [0, D); from the mdkm_fit / mdkm_predict, before any work is enqueued, MDKM_ERR_STATE when no
 * regions are bound for that call. */
int mdkm_bind_region_overlaps(mdkm_handle* h, const int32_t* pairs, int n_pairs);

/* The region overlaps of the last mdkm_fit / mdkm_predict that had them bound, kept on the device
 * until the next mdkm_unproject / mdkm_set_points or fit / predict with regions (a later call with
 * regions but without overlaps drops them).  mdkm_region_overlap_count: their number M.
 * mdkm_region_overlap_table: copies the rows (table_out, int64 [M][6]) to host memory.  Errors:
 * MDKM_ERR_STATE when there are none (none computed since the last unproject / set_points);
 * MDKM_ERR_INVALID from mdkm_region_overlap_table when capacity_rows < M. */
int mdkm_region_overlap_count(const mdkm_handle* h, int64_t* n_rows);
int mdkm_region_overlap_table(mdkm_handle* h, int64_t* table_out, int64_t capacity_rows);

/* Optional: have the NEXT mdkm_fit or mdkm_predict on this handle, which must also have regions
 * bound (mdkm_bind_regions), return object tracks: which region is the same object over the whole
 * stack.  Region r of day d and region s of day d+1 (consecutive global days) are linked when
 * cluster(r) == cluster(s) and they share at least one pixel with
 *   (double)shared / (double)(pixels_r + pixels_s - shared) >= min_iou
 * in FP64 (the counts are exact integers below 2^31 and the division is correctly rounded, so a
 * numpy restatement gives the same bits; pixels are column 2 of the region table).  A track is a
 * connected component of the graph whose nodes are the regions and whose edges are the links; a
 * region without links is a track of its own, so T <= R and every region is in exactly one
 * track.  Tracks do not bridge a gap: a day on which the object has no region ends its track.
 * Tracks are numbered 1..T in the order of their smallest region id, so the numbering does not
 * depend on the schedule or the number of ranks, and all regions of a track have one cluster.
 * Chains: with min_iou > 0.5 every region has at most one link forward and one back, so every
 * track is a chain with one region per day over [first_day, last_day].  If r linked to two
 * disjoint regions s1, s2 of day d+1, each IoU > 1/2 would force shared_i > pixels_r / 2, and
 * shared_1 + shared_2 > pixels_r is impossible; the FP64 rounding keeps this, because 0.5 is
 * representable and rounding is monotone, so a rounded quotient >= min_iou > 0.5 means an exact
 * quotient > 0.5.  With min_iou <= 0.5, splits and merges join tracks.
 * After the call, mdkm_track_count gives T and mdkm_track_table copies the track table, int64
 * [T][7]: cluster, first_day, last_day, regions (the number of regions in the track), pixels (the
 * sum of its regions' pixels), first_region (its smallest region id), branched (1 when some
 * region of the track has two or more links to the next day or to the previous day, else 0) --
 * and the region tracks, int32 [R]: the track id of region r at index r - 1.
 * map_out (optional, int32, capacity_pixels >= the pix_count of the last mdkm_unproject; host or
 * device memory as `mem` says) receives the track id of every pixel of this rank's range that
 * produced a point, 0 elsewhere: the region map with every id replaced by its track's.  A device
 * map is written in place; a host map is written into a device stage of 4 B per pixel and copied.
 * Where the numbers come from: the overlaps of the consecutive pairs (d, d+1) are counted with
 * those of mdkm_bind_region_overlaps (the caller's pairs first, then the consecutive pairs the
 * caller did not ask for; the caller's rows and their count are the same as without tracks), one
 * thread per row of a consecutive pair applies the rule and joins the two regions in a union-find
 * on the R regions (integer atomics: the root is the smallest region id), the numbering passes of
 * the regions give the roots their ids and every region its root's, and one pass over the regions
 * fills the table with integer atomics; then the map pass.  One more synchronisation reads T.
 * Memory: 72 B per region (parents, links, ids, table slots), the overlaps of the consecutive pairs
 * (see mdkm_bind_region_overlaps), and 4 B per pixel of the range for a host map.  With several
 * ranks every rank builds the same tracks from its whole-stack region map, with no collective.
 * Asking for tracks changes no other result of the call.
 * min_iou == 0 with map_out == NULL clears the binding.  The binding is consumed by that one call,
 * and dropped by mdkm_unproject / mdkm_set_points.  Errors: MDKM_ERR_STATE when the resident cloud
 * did not come from mdkm_unproject; MDKM_ERR_INVALID when min_iou is not in (0, 1] (NaN included),
 * the stack has more than 16384 days, capacity_pixels < pix_count, or `mem` is neither
 * MDKM_MEM_HOST nor MDKM_MEM_DEVICE; from the mdkm_fit / mdkm_predict, before any work is
 * enqueued, MDKM_ERR_STATE when no regions are bound for that call. */
int mdkm_bind_tracks(mdkm_handle* h, double min_iou, int32_t* map_out, int64_t capacity_pixels, int mem);

/* The tracks of the last mdkm_fit / mdkm_predict that had them bound, kept on the device until
 * the next mdkm_unproject / mdkm_set_points or fit / predict with regions (a later call with
 * regions but without tracks drops them).  mdkm_track_count: their number T.  mdkm_track_table:
 * copies the track table (table_out, int64 [T][7]) and the region tracks (region_tracks_out, int32
 * [R]) to host memory; either may be NULL.  Errors: MDKM_ERR_STATE when there are none (none
 * computed since the last unproject / set_points); MDKM_ERR_INVALID from mdkm_track_table when
 * table_out is given and capacity_tracks < T, or region_tracks_out is given and capacity_regions
 * < R. */
int mdkm_track_count(const mdkm_handle* h, int64_t* n_tracks);
int mdkm_track_table(mdkm_handle* h, int64_t* table_out, int32_t* region_tracks_out, int64_t capacity_tracks,
                     int64_t capacity_regions);

/* Optional: have the NEXT mdkm_fit or mdkm_predict on this handle, which must also have regions
 * bound (mdkm_bind_regions), return the adjacency of the regions within each day: which objects of
 * one day touch, along how long a border, and each region's perimeter.  An edge joins two
 * 4-neighbouring pixels of one day: direction 0 joins (y, x) and (y, x+1), direction 1 joins (y, x)
 * and (y+1, x); its index within the day is e = 2 (y W + x) + direction, and edges are ordered by
 * (day, e).  After the call, mdkm_region_adjacency_count gives the number of rows M and
 * mdkm_region_adjacency_table copies them, int64 [M][6]: day, region_a, region_b, edges, y_first,
 * x_first -- one row for every unordered pair of distinct regions r = region_a < s = region_b
 * joined by at least one edge, with the number of edges between them (their shared border in pixel
 * edges) and the upper or left pixel of their first edge.  Rows are sorted by that first edge;
 * every edge belongs to at most one row, so the order is total and does not depend on the schedule
 * or the number of ranks.  Regions that touch only at a corner have no row, under either
 * connectivity; regions that share an edge have different clusters.  It also copies the region
 * boundaries, int64 [R][4], row r - 1 for region r: perimeter (the sides of the region's pixels
 * whose other side is not in the region), region_edges (sides facing another region: the sum of
 * `edges` over the rows of r), background_edges (sides facing a pixel of the same day without a
 * point) and border_edges (sides on the edge of the H x W grid); perimeter = region_edges +
 * background_edges + border_edges, and 4 pixels = perimeter + 2 x (edges inside the region).
 * Where the numbers come from: behind the region ids, a pass counts for every day the run starts
 * along each image row of the horizontal key (id[p], id[p+1]) and of the vertical key (id[p],
 * id[p+W]) of two different non-zero ids, an upper bound on the day's rows, read by the
 * synchronisation that reads R (no extra one).  Each day gets an open-addressing hash table of
 * 16-byte slots keyed min << 32 | max (the smallest power of two >= 2 x its bound); equal keys are
 * combined in the warp, and their leaders add the edges and lower the first edge with atomics; the
 * same pass adds every pixel's background and border sides to its region, summed per warp.  Every
 * occupied slot sets the bit of its first edge in a 2 H W-bit mask per day, the popcount scan of
 * the region overlaps gives each slot its row, and one more synchronisation reads M; the rows are
 * then written and each row's edges added to both regions' region_edges.  Memory: 16 B x table
 * capacity (<= 128 B per pixel) plus 8 B per 16 pixels (mask and scan offsets), 48 B per row and
 * 32 B per region; the worst case, where every edge is a row of its own, is a one-pixel
 * checkerboard (2 rows per pixel: 96 B of rows and 64 to 128 B of table per pixel).  A failed
 * allocation returns MDKM_ERR_OOM.
 * With several ranks every rank builds the whole table from its whole-stack region map: no
 * collective, the same bits on every rank, and every rank pays the whole cost.  Asking for
 * adjacency changes no other result of the call.
 * on == 0 clears the binding.  The binding is consumed by that one call, and dropped by
 * mdkm_unproject / mdkm_set_points.  Errors: MDKM_ERR_STATE when the resident cloud did not come
 * from mdkm_unproject; from the mdkm_fit / mdkm_predict, before any work is enqueued,
 * MDKM_ERR_STATE when no regions are bound for that call. */
int mdkm_bind_region_adjacency(mdkm_handle* h, int on);

/* The region adjacency of the last mdkm_fit / mdkm_predict that had it bound, kept on the device
 * until the next mdkm_unproject / mdkm_set_points or fit / predict with regions (a later call with
 * regions but without adjacency drops it).  mdkm_region_adjacency_count: the number of rows M.
 * mdkm_region_adjacency_table: copies the rows (rows_out, int64 [M][6]) and the region boundaries
 * (boundaries_out, int64 [R][4]) to host memory; either may be NULL.  Errors: MDKM_ERR_STATE when
 * there is none (none computed since the last unproject / set_points); MDKM_ERR_INVALID from
 * mdkm_region_adjacency_table when rows_out is given and capacity_rows < M, or boundaries_out is
 * given and capacity_regions < R. */
int mdkm_region_adjacency_count(const mdkm_handle* h, int64_t* n_rows);
int mdkm_region_adjacency_table(mdkm_handle* h, int64_t* rows_out, int64_t* boundaries_out, int64_t capacity_rows,
                                int64_t capacity_regions);

/* Load an already unprojected cloud (this rank's shard).  Replaces the `X` argument of the
 * reference's KMeans(...).fit_predict(X) call (members/jasraj/land_use_classification/
 * core.py:227-228) for d = 3. */
int mdkm_set_points(mdkm_handle* h, const float* xyz, int64_t n, int layout, int mem);

/* Number of resident points on this rank / over all ranks of the communicator (the second
 * one is a collective the first time it is called for a cloud). */
int64_t mdkm_num_points(const mdkm_handle* h);
int64_t mdkm_num_points_global(mdkm_handle* h);

/* Fetch m points by index as float32 [m,3] (x,y,z) into host memory (what `X[seeds]` does for
 * init="random", sklearn/cluster/_kmeans.py:1014-1021).  With a communicator the indices
 * are global (shards concatenated in rank order), the call is collective and every rank
 * receives all m points. */
int mdkm_gather_points(mdkm_handle* h, const int64_t* idx, int m, float* out_xyz);

/* Copy the resident cloud out as float32 [n,3].  napari_order != 0 gives (z,y,x) columns as
 * plugin.py:192 builds `points_coords`; 0 gives (x,y,z). */
int mdkm_get_cloud(mdkm_handle* h, float* out, int napari_order, int mem);

/* Same, but returns as soon as the copy is enqueued: it proceeds on a side stream while
 * later calls on this handle (mdkm_fit) compute.  `out` (page-locked host memory for a real
 * overlap) holds the cloud once mdkm_wait -- or any later call that touches the cloud --
 * has returned. */
int mdkm_get_cloud_async(mdkm_handle* h, float* out, int napari_order, int mem);
int mdkm_wait(mdkm_handle* h);

/* Segments of the resident cloud: one per day of the unprojected pixel range (the reference
 * treats every stereo pair / day separately, plugin.py:106), one for mdkm_set_points.
 * mdkm_segment_offsets writes n_segments + 1 point offsets (the last one is n). */
int mdkm_num_segments(const mdkm_handle* h);
int mdkm_segment_offsets(const mdkm_handle* h, int64_t* out);

/* Ground-levelling of plugin.py:181-192, per segment (day): h_min / h_max =
 * np.percentile(z, 2) / np.percentile(z, 98) with numpy's linear interpolation (exact order
 * statistics by radix select on the device); z -= h_min in the resident cloud;
 * height_norm_out (optional, n floats, host or device per `mem`) =
 * clip((z - h_min) / (h_max - h_min + 1e-6), 0, 1), the 'height' colour property.
 * h_min_out / h_max_out: optional arrays of n_segments doubles.  Rank-local: needs whole days
 * on this rank (shard the stack by days).  Call it before mdkm_fit. */
int mdkm_ground_level(mdkm_handle* h, float* height_norm_out, int mem, double* h_min_out,
                      double* h_max_out);

/* ---- K2..K4: Lloyd k-means -----------------------------------------------------------
 * Replaces sklearn.cluster.KMeans(n_clusters=k, init=<array>, n_init=1,
 * algorithm="lloyd", max_iter, tol).fit(X) as the reference calls it (core.py:227-228;
 * algorithm in sklearn/cluster/_kmeans.py:630-758, 1436-1563 and _k_means_lloyd.pyx).
 * init: k x 3 float64, row-major, same coordinates as the points.
 * A NaN or infinite coordinate in init, or in the centroids of mdkm_lloyd_step / mdkm_predict, gives MDKM_ERR_INVALID.
 * labels_out: int32[n_local] (may be NULL); centroids_out: float64[k*3]; n_iter_out,
 * inertia_out as scikit-learn's n_iter_ / inertia_.  With a communicator the point set is
 * the union of all ranks' shards and every rank gets the same centroids / n_iter /
 * inertia and its own shard's labels.  No host synchronisation per iteration. */
int mdkm_fit(mdkm_handle* h, int k, const double* init, int max_iter, double tol,
             int32_t* labels_out, int labels_mem, double* centroids_out, int* n_iter_out,
             double* inertia_out);

/* Diagnostics of the last mdkm_fit / mdkm_lloyd_step on this rank:
 * n_refined = point-iterations whose FP32 distances were within the rounding-error bound
 * of a tie and were re-decided in float64; n_relocations = empty-cluster relocations. */
int mdkm_fit_stats(const mdkm_handle* h, int64_t* n_refined, int64_t* n_relocations,
                   double* tol_scaled);

/* More diagnostics of the last mdkm_fit on this rank: *worklist_groups = 128-point groups that
 * went through the per-point pass, summed over the iterations of the fit (fused iterations
 * only); *groups = groups of the cloud.  1 - worklist_groups / (groups * n_iter) is the share
 * of group-iterations settled from the cached summaries without reading a point. */
int mdkm_fit_worklist(const mdkm_handle* h, int64_t* worklist_groups, int64_t* groups);

/* One E-step + M-step sums with the given centroids (test hook for single-step parity;
 * mirrors sklearn.cluster._k_means_lloyd.lloyd_iter_chunked_dense up to the sums,
 * _k_means_lloyd.pyx:23-152).  sums_out: float64[k*3] = sum of member coordinates,
 * counts_out: int64[k]; both GLOBAL over ranks when a communicator is set. */
int mdkm_lloyd_step(mdkm_handle* h, int k, const double* centroids, int32_t* labels_out,
                    int labels_mem, double* sums_out, int64_t* counts_out);

/* Labels of the resident points for given centroids and the resulting inertia: the E-step
 * alone, i.e. KMeans.predict / -KMeans.score (sklearn/cluster/_kmeans.py:742-756, 1068-1095;
 * inertia: _k_means_common.pyx:94-124).  labels_out may be NULL; inertia is global over ranks. */
int mdkm_predict(mdkm_handle* h, int k, const double* centroids, int32_t* labels_out,
                 int labels_mem, double* inertia_out);

/* k-means++ seeding on the device (sklearn/cluster/_kmeans.py:180-278).  The random draws
 * of numpy.random.RandomState stay on the host and are supplied by the caller in
 * scikit-learn's order: `first_index` is the result of RandomState.choice(n) for the first
 * centre, then for each further centre `n_local_trials` uniforms in [0,1) from rand_vals
 * (row-major [(k-1), n_local_trials], n_local_trials <= 16; scikit-learn uses
 * 2 + int(ln k)); the device does the distances (float64), the potentials, the
 * cumulative-sum search and the greedy choice among the trials, all k centres without a
 * host round trip.  centers_out: float64[k*3]; indices_out: int64[k] (may be NULL).
 * With a communicator the cloud is the concatenation of the ranks' shards in rank order:
 * first_index and the returned indices are GLOBAL, every rank passes the same arguments and
 * gets the same centres (the ranks' sums are exchanged with NCCL, three small all-reduces
 * per centre). */
int mdkm_kmeans_plusplus(mdkm_handle* h, int k, int64_t first_index, const double* rand_vals,
                         int n_local_trials, double* centers_out, int64_t* indices_out);

/* The first fit on a cloud builds two acceleration structures that later fits on the same
 * cloud reuse: the tile-ordered mirror of the points and the per-group summaries (box +
 * fixed-point sums).  mdkm_drop_caches discards them, so that the next fit pays for them again
 * (bench.py times every fit that way). */
int mdkm_drop_caches(mdkm_handle* h);

/* Timing aid for bench.py: when enabled, CUDA events bracket every batch of back-to-back
 * launches of the Lloyd step kernel inside mdkm_fit; mdkm_profile_read returns the summed
 * duration and the number of launches it covers and resets both (average launch duration =
 * their ratio; batches that ended early on convergence make it a lower bound). */
int mdkm_profile_enable(mdkm_handle* h, int on);
int mdkm_profile_read(mdkm_handle* h, double* step_kernel_ms, int* n_step_launches,
                      int* n_kernel_launches_total);

/* The same for the other kernel groups of the path (CUDA events on the handle's stream around
 * the kernels only -- host work and copies between them are outside): summed duration and work
 * count since the last read of that phase.  count = pixels (UNPROJECT: count + scan + scatter
 * kernels of mdkm_unproject), points (BUILD: tile-ordered mirror + group summaries of a cold
 * fit; FINAL: the final labelling / inertia pass of mdkm_fit), launches (STEP). */
enum { MDKM_PHASE_UNPROJECT = 0, MDKM_PHASE_BUILD = 1, MDKM_PHASE_STEP = 2, MDKM_PHASE_FINAL = 3,
       MDKM_PHASE_COUNT = 4 };
int mdkm_profile_phase(mdkm_handle* h, int phase, double* ms, int64_t* count);

#ifdef __cplusplus
}
#endif
#endif /* MDKM_H_ */
