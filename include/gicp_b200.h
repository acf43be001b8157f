/*
 * gicp_b200.h - C ABI of libgicp_b200.so, the B200-native GICP registration engine.
 *
 * The reference (msi-se/generalized-icp) has no FFI: its boundary is the Python
 * call  gicp.gicp(source_points, target_points, ...)  (python-implementation/
 * gicp.py:78, returning the 7-tuple of gicp.py:174) and
 * gicp.apply_transformation (gicp.py:176).  This header is what a ctypes shim
 * standing in for that module binds (see INTEGRATION.md); every entry point
 * cites the reference lines it replaces.
 *
 * Conventions
 *  - every function returns 0 on success, non-zero on failure; the message of
 *    the last failure on the calling thread is gicpGetLastError().  No C++
 *    exception crosses the boundary.
 *  - all d_* pointers are DEVICE pointers owned by the caller (e.g. PyTorch
 *    allocations); h_* pointers are HOST pointers.  The library owns only the
 *    workspace behind its handle (grow-only, reused across calls).
 *  - `stream` is a cudaStream_t passed as void*; calls are asynchronous on it
 *    unless they return host data (those synchronise the stream).
 *  - a handle is bound to one device and one (dim, storage) pair and is not
 *    thread-safe: one handle per thread.  All calls on a handle must use the SAME
 *    stream (the source and target sides share the handle's scratch buffers;
 *    two streams would race on them).
 *  - clouds come as BATCHES: `n_clouds` clouds concatenated into one (n_total,
 *    dim) row-major array, with h_offsets[n_clouds+1] giving each cloud's row
 *    range.  A single pair is a batch of one.  Source cloud i is registered
 *    against target cloud i.
 *  - point indices reported by the library are cloud-local (0-based row within
 *    the cloud), -1 meaning "none".
 */
#ifndef GICP_B200_H
#define GICP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gicpContext* gicpHandle;

enum { GICP_STORAGE_F32 = 0, GICP_STORAGE_F64 = 1 };
enum { GICP_SOURCE = 0, GICP_TARGET = 1 };
enum { GICP_PLANE_TO_PLANE = 0, GICP_POINT_TO_POINT = 1, GICP_POINT_TO_PLANE = 2 };

/* Parameters; names follow gicp.py:78 where the reference has them. */
typedef struct gicpParams {
    int32_t k;                    /* neighbours INCLUDING the query point; gicp.py:24 hard-codes 6        */
    int32_t max_iterations;       /* gicp.py:78 max_iterations = 100                                      */
    double  tolerance;            /* gicp.py:78 tolerance = 1e-6 : stop when |last_loss - loss| < tol     */
    double  max_distance_correspondence;     /* gicp.py:78 (=150): reject when d > d_max (strict, :136)   */
    double  max_distance_nearest_neighbors;  /* gicp.py:78 (=50):  k-NN bound, exclusive (:24)            */
    double  lambda_tangent;       /* gicp.py:5   epsilon = 100                                            */
    double  lambda_normal;        /* gicp.py:11  epsilon * 0.1 = 10                                       */
    int32_t inner_max_iterations; /* LM iterations of the on-device inner solve (replaces fmin_cg, :152)  */
    int32_t covariance_model;     /* ICP family through the same kernels (presentation/main.typ:446-462):
                                   * 0 plane-to-plane = GICP (the reference), 1 point-to-point (C_A = 0, C_B = I),
                                   * 2 point-to-plane (C_A = 0, C_B = the target's surface-aligned covariance)    */
    double  knn_cell;             /* uniform-grid cell edge for the k-NN grid; 0 = auto (radius / 4);   */
                                  /* a given value is raised to at least radius / 8                       */
    double  nn_cell;              /* cell edge of the target's 1-NN grid;      0 = auto (d_max / 2)       */
    int64_t max_cells_per_cloud;  /* cell-table budget per cloud; 0 = auto                                */
} gicpParams;

#define GICP_NRED_2D 32   /* doubles per pair written by gicpNormalEquations, dim 2 */
#define GICP_NRED_3D 80   /* doubles per pair written by gicpNormalEquations, dim 3 */

/* ---- lifetime ------------------------------------------------------------------------- */
int gicpCreate(gicpHandle* out, int device, int dim /*2|3*/, int storage /*GICP_STORAGE_* */);
int gicpDestroy(gicpHandle h);
const char* gicpGetLastError(void);
int gicpVersion(void);
/* fills *p with the reference's defaults (gicp.py:78, :5, :11, :24) */
int gicpDefaultParams(gicpParams* p);
int gicpSetParams(gicpHandle h, const gicpParams* p);

/* ---- clouds: grid build (replaces KDTree(points), gicp.py:21,127) and per-point
 *      covariances (replaces compute_covariance_matrix, gicp.py:19-35) ---------------------
 * d_points: (n_total, dim) row-major, float32 or float64 according to `storage`.
 * The target call also builds the 1-NN grid used by the correspondence search.
 * The arrays must stay valid until the next gicpSet* call on the same side.              */
int gicpSetTarget(gicpHandle h, const void* d_points, const int64_t* h_offsets, int32_t n_clouds, void* stream);
int gicpSetSource(gicpHandle h, const void* d_points, const int64_t* h_offsets, int32_t n_clouds, void* stream);
/* Both sides of a batch of pairs in one call (gicp.py:104 + :111 of one gicp() call).  Same result as gicpSetTarget
 * followed by gicpSetSource.  While one side alone cannot fill the device (up to 2^20 points per side: the reference's
 * own scans, a 100k-point pair) the source side is set up on an internal stream, with its own scratch, concurrently
 * with the target side; `stream` is forked before and joined after, so the caller still sees one stream-ordered
 * operation.  Larger sides run one after the other.                                                                */
int gicpSetPair(gicpHandle h, const void* d_target_points, const int64_t* h_target_offsets, const void* d_source_points,
                const int64_t* h_source_offsets, int32_t n_clouds, void* stream);

/* Scan sequences (robot-visualization.py:246-252: "source <- target; target <- current scan"): the
 * target of pair k is the source of pair k+1, so its grids and covariances are reused instead of
 * being rebuilt (the reference recomputes both on every call, gicp.py:104,111).  After this call
 * the handle's source is the former target; set a new target with gicpSetTarget.             */
int gicpPromoteTargetToSource(gicpHandle h);

/* ---- the registration loop (replaces gicp.py:107-174) ------------------------------------
 * Runs all pairs to convergence / max_iterations on the device.
 *  h_T0        optional (n_clouds, dim+1, dim+1) initial transforms (NULL = identity, gicp.py:107)
 *  d_T         (n_clouds, dim+1, dim+1) f64: final transform (gicp.py:174 [0])
 *  d_n_outer   (n_clouds) i32: outer iterations executed = len(all_source_cov_matrices)
 *  d_converged (n_clouds) i32: iteration index printed by "Converged at iteration" (gicp.py:161) or -1
 *  d_loss_hist optional (n_clouds, max_iterations) f64: min_loss per outer iteration (gicp.py:154)
 *  d_T_hist    optional (n_clouds, max_iterations+1, dim+1, dim+1) f64: all_transformations (gicp.py:108,167)
 *  d_inliers   optional (n_clouds, max_iterations) i32: correspondences that passed the gate per iteration
 * Asynchronous on `stream`: large pairs are driven by a host loop that runs a few iterations ahead of 4-byte
 * progress polls (it returns once every pair has stopped); when every source cloud has <= 2048 points the whole
 * loop is ONE kernel (fused.cuh) and the call returns immediately - synchronise `stream` before reading the outputs. */
int gicpRegister(gicpHandle h, const double* h_T0, double* d_T, int32_t* d_n_outer, int32_t* d_converged,
                 double* d_loss_hist, double* d_T_hist, int32_t* d_inliers, void* stream);

/* ---- stage entry points (teacher-forced parity tests; each is one stage of the loop) -----
 * gicpKnn: k-NN lists of one side as computed for the covariances (gicp.py:24-25):
 *   d_idx (n_total, k) i32 cloud-local, ascending by (distance, index), -1 = missing;
 *   d_dist (n_total, k) f64 or NULL.                                                       */
int gicpKnn(gicpHandle h, int which, int32_t* d_idx, double* d_dist, void* stream);
/* covariances of one side in input order: (n_total, dim, dim) f64  (gicp.py:104,111)       */
int gicpCovariances(gicpHandle h, int which, double* d_cov, void* stream);
/* correspondences under the given transforms (gicp.py:119,129-145):
 *   h_T (n_clouds, dim+1, dim+1); d_idx (n_src_total) i32 matched target index or -1 when gated;
 *   d_dist (n_src_total) f64 1-NN distance (inf when nothing within the search bound);
 *   d_W optional (n_src_total, dim, dim) f64 weight matrices, 0 for gated rows.            */
int gicpCorrespond(gicpHandle h, const double* h_T, int32_t* d_idx, double* d_dist, double* d_W, void* stream);
/* the fused per-iteration reduction at the given transforms: h_out (n_clouds, GICP_NRED_xD).
 * Layout (dim 3; p~ = (1, p' - mu), p' = R p + t, e = q - p', v = W e):
 *   [0..59]  sum p~_a p~_b W_cd, ab in {00,01,02,03,11,12,13,22,23,33} (slow), cd in {00,01,02,11,12,22} (fast)
 *   [60..71] sum v_c p~_a  (c slow, a fast)      [72] sum e^T W e      [73] gated-in count
 *   [74..76] mu                                  [77..79] 0
 * dim 2: ab in {00,01,02,11,12,22}, cd in {00,01,11} -> [0..17]; [18..23] v_c p~_a; [24] loss; [25] count;
 *   [26..27] mu.  Synchronises the stream.                                                 */
int gicpNormalEquations(gicpHandle h, const double* h_T, double* h_out, void* stream);

/* source covariances as the reference recomputes them on the transformed cloud every outer
 * iteration (gicp.py:120): C_src,k = R_k C_src,0 R_k^T.  h_T (n_T, n_clouds, dim+1, dim+1);
 * d_out (n_T, n_src_total, dim, dim) f64 in input order.  all_source_cov_matrices, gicp.py:121. */
int gicpSourceCovariancesAt(gicpHandle h, const double* h_T, int32_t n_T, double* d_out, void* stream);

/* ---- voxel-grid downsampling (PCL's VoxelGrid filter), for clouds too dense to register raw ----------------
 * A batch in the layout of gicpSet*, in the handle's dim and storage.  For every cloud, with leaf L:
 *  - the voxel of a point is v_a = floor((double)p_a / L) per axis (IEEE float64 division, lattice anchored at the
 *    origin, so clouds share one lattice); rows with a non-finite coordinate are dropped;
 *  - a voxel with fewer than min_points points is dropped (1 keeps every voxel);
 *  - the output point of a voxel is the centroid of its points: a float64 sum in a fixed order, started from the
 *    first point, divided by the count, rounded to the storage type; bit-identical from run to run;
 *  - a cloud's output rows are ordered by each voxel's lowest input row, so with every point alone in its voxel the
 *    output is the finite input rows, bit for bit;
 *  - per cloud, floor(hi / L) - floor(lo / L) over its finite rows must be < 2^21 along each axis in 3-D (< 2^31 in
 *    2-D) and every voxel index must fit int64; otherwise the call fails naming the cloud and the axis.
 *  d_out         (n_total, dim) caller-allocated, same dtype as d_points, not d_points itself; the first
 *                h_out_offsets[n_clouds] rows are written
 *  h_out_offsets (n_clouds+1) host: row range of each cloud's output - directly usable as the offsets of gicpSet*
 *  d_voxel_of    optional (n_total) i32: cloud-local output row of each input point, -1 when dropped
 *  d_counts      optional (n_total) i32: points per output row
 * Synchronises the stream.  Uses scratch of its own: the handle's source / target (grids, covariances, loop state)
 * are untouched, so it may be called between gicpSetPair and gicpRegister.                                      */
int gicpVoxelDownsample(gicpHandle h, const void* d_points, const int64_t* h_offsets, int32_t n_clouds,
                        double voxel_size, int32_t min_points, void* d_out, int64_t* h_out_offsets,
                        int32_t* d_voxel_of, int32_t* d_counts, void* stream);

/* ---- multi-GPU: one large pair with the source sharded over ranks (BASELINE config 5) ----
 * Every rank holds both full clouds; rank r computes covariances for its slice of the
 * target (all-gathered once) and runs the per-iteration reduction on its slice of the
 * source, followed by one all-reduce of GICP_NRED_xD doubles per outer iteration.
 * NCCL is loaded at run time (libnccl.so.2, the one PyTorch ships).                        */
int gicpCommGetUniqueId(char id[128]);
int gicpCommInit(gicpHandle h, int32_t n_ranks, int32_t rank, const char id[128]);
int gicpCommDestroy(gicpHandle h);

/* ---- input generation for scan-sequence benchmarks: the robot demo's 2-D LiDAR ray caster ------
 * (robot-visualization.py:42-120 cast_ray, :222-237 scan loop), one thread per ray, all poses at once.
 *  d_poses (n_poses, 3) f64: x, y, yaw in degrees;  d_segments (n_seg, 4) f64: x3, y3, x4, y4;
 *  d_circles (n_circ, 3) f64: cx, cy, r;  d_noise optional (n_poses, num_rays) f64 additive range noise;
 *  d_rel_xy (n_poses, num_rays, 2) f64 robot-relative hit points;  d_hit (n_poses, num_rays) i32.     */
int gicpRayCast(int device, const double* d_poses, int32_t n_poses, int32_t num_rays, const double* d_segments,
                int32_t n_seg, const double* d_circles, int32_t n_circ, double max_range, const double* d_noise,
                double* d_rel_xy, int32_t* d_hit, void* stream);

/* number of kernels this library launched on this handle since creation (bench bookkeeping) */
int64_t gicpLaunchCount(gicpHandle h);

/* per-stage device timing with CUDA events on the launching stream (bench.py's roofline leg).
 * gicpProfile(h, 1) starts recording; gicpProfileRead synchronises the device, returns the summed
 * milliseconds and the number of timed launches/sections per stage, and clears the records.   */
enum { GICP_STAGE_GRID = 0, GICP_STAGE_KNN_COV = 1, GICP_STAGE_CORRESPOND = 2, GICP_STAGE_ACCUMULATE = 3,
       GICP_STAGE_SOLVE = 4, GICP_N_STAGES = 5 };
int gicpProfile(gicpHandle h, int enable);
int gicpProfileRead(gicpHandle h, double ms_out[GICP_N_STAGES], int64_t count_out[GICP_N_STAGES]);

#ifdef __cplusplus
}
#endif
#endif /* GICP_B200_H */
