/*
 * b200icp.h -- C ABI of the B200-native 2D ICP scan-matching path.
 *
 * Drop-in boundary for the reference's registration step
 * (DucVuUET04/ICP_SLAM-YOLO).  The reference has no FFI of its own: the boundary
 * is the Python call  icp(A, B, max_iterations, tolerance) -> (src, R, t)
 * (labels_segmentation/icp.py:28-53) built on best_fit_transform
 * (labels_segmentation/icp.py:5-26), fed by polar_to_cartesian_3d
 * (duc/ICP_LIDAR/process.py:38-52), plus the Open3D-shaped sibling
 * gicp(points1, points2, threshold, voxel, trans_init) -> (rmse, T4x4)
 * (duc/ICP_LIDAR/gicp_lidar.py:12-36, called at duc/ICP_LIDAR/mainn.py:311).
 * Every entry point below names the reference lines it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - All data pointers are DEVICE pointers owned by the caller (host pointers only
 *     where a parameter says "host").  The library allocates nothing, never writes
 *     its inputs, and is asynchronous on the CUDA stream passed as `stream`
 *     (a cudaStream_t cast to void*; NULL = legacy default stream).
 *   - Every call returns a b200icp_status (0 = OK).  No exceptions, no aborts.
 *     b200icp_last_error() returns a thread-local description of the last failure.
 *   - Degenerate pairs (no source or no target points, every correspondence gated
 *     out) do not fail the batch: they yield R = I, t = 0 (or the initial pose),
 *     error = +inf, iterations = number of completed updates.
 *   - Points are interleaved (x, y) pairs, float32 or float64.  All O(N) state
 *     (source points, sums, poses, errors) is float64 on the device; only the
 *     O(N*M) candidate search runs in float32 and every candidate is re-decided
 *     in float64, so correspondence indices equal a float64 brute-force argmin
 *     with lowest-index tie-break.
 */
#ifndef B200ICP_H_
#define B200ICP_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200ICP_VERSION_MAJOR 0
#define B200ICP_VERSION_MINOR 3   /* 0.3: W-warps-per-pair fused kernel; scan-to-map = exact culling +
                                     exact scan with the all-gather in the search epilogue */

typedef enum b200icp_status {
  B200ICP_OK = 0,
  B200ICP_ERR_INVALID_ARGUMENT = 1, /* NULL / negative size / bad enum            */
  B200ICP_ERR_UNSUPPORTED_SHAPE = 2,/* pitch beyond what the fused kernel handles  */
  B200ICP_ERR_CUDA = 3,             /* a CUDA runtime call failed (see last_error) */
  B200ICP_ERR_NO_DEVICE = 4         /* no sm_100 device / driver                   */
} b200icp_status;

typedef enum b200icp_dtype { B200ICP_F32 = 0, B200ICP_F64 = 1 } b200icp_dtype;

/* How pair p of a batch picks its source and target rows. */
typedef enum b200icp_pairing {
  B200ICP_PAIR_ROWWISE = 0,   /* src row p        , tgt row p                        */
  B200ICP_PAIR_EXPLICIT = 1,  /* src row src_row[p], tgt row tgt_row[p]               */
  B200ICP_PAIR_TRIANGLE = 2   /* q = first_pair + p enumerates (i < j) row-major over
                                 n_rows rows of ONE table: tgt = row i, src = row j
                                 (all-pairs loop-closure candidates)                  */
} b200icp_pairing;

/*
 * A batch of ICP problems over row tables of ragged scans in HBM.
 *   src_points : [src_rows][src_pitch][2]   tgt_points : [tgt_rows][tgt_pitch][2]
 *   src_len / tgt_len : valid points per row (NULL => every row is full, = pitch)
 * Sequence odometry (scan k+1 -> scan k, icp.py:28 called per consecutive pair) is
 * ROWWISE with src_points = table + one row and tgt_points = table.
 * Replaces the A, B arguments of icp() (labels_segmentation/icp.py:28).
 */
typedef struct b200icp_problem {
  const void* src_points;
  const void* tgt_points;
  const int32_t* src_len;
  const int32_t* tgt_len;
  int32_t src_pitch;        /* points per source row (>= every src_len)            */
  int32_t tgt_pitch;
  int32_t dtype;            /* b200icp_dtype of BOTH point tables                  */
  int32_t pairing;          /* b200icp_pairing                                     */
  const int32_t* src_row;   /* EXPLICIT only                                       */
  const int32_t* tgt_row;   /* EXPLICIT only                                       */
  int64_t first_pair;       /* TRIANGLE only: linear index of this shard's pair 0  */
  int32_t n_rows;           /* TRIANGLE only: rows in the table                    */
  int32_t reserved;
} b200icp_problem;

/* Replaces max_iterations / tolerance of icp() (icp.py:28) and adds the Open3D-shaped
 * trans_init / max_correspondence_distance of gicp() (gicp_lidar.py:12,29-34). */
#define B200ICP_FLAG_DENSE_SWEEP 1  /* evaluate every source-target pair (no culling of target
                                       groups).  Results are identical either way; the culled
                                       sweep is ~2x faster on spatially ordered scans (LiDAR beams)
                                       and ~15 % slower on unordered point sets.             */

#define B200ICP_FLAG_NO_SWEEP_REUSE 2  /* sweep every pass in every iteration.  By default a pass of
                                          64 source points skips its candidate sweep while none of
                                          them can have left the group of 8 targets that held its
                                          nearest neighbour at the last sweep (a bound on the motion
                                          since then against the gap to the nearest outside target);
                                          the correspondences are identical either way.            */

#define B200ICP_FLAG_WARP_KERNEL 4  /* force the throughput kernel (W warps per pair, shared tile)  */
#define B200ICP_FLAG_CTA_KERNEL 8   /* force the latency kernel (one CTA of up to 8 warps per pair).
                                       Default: chosen by the batch size -- the throughput kernel once
                                       the pairs fill the GPU (> 512), the latency kernel below that
                                       (one registration per frame).
                                       BATCH-SIZE DEPENDENCE: the two kernels find identical
                                       correspondences and iteration counts but add the float64 sums in
                                       a different order, so the pose bits of one pair may differ by
                                       ~1e-12 (relative) between a call of <= 512 pairs and a larger
                                       one.  Callers that need bit-stable poses across batch sizes
                                       force one kernel with these flags (HostPipeline does, on the
                                       size of the whole batch).                                   */
#define B200ICP_FLAG_PAIR_WARPS_SHIFT 8    /* tuning: bits 8..10 = warps per pair (1..4) of the
                                              throughput kernel; 0 = chosen from the number of passes */

typedef struct b200icp_options {
  int32_t max_iterations;   /* icp.py:28,35; reference default 20                   */
  int32_t flags;            /* B200ICP_FLAG_*                                        */
  double tolerance;         /* icp.py:49; < 0 forces all iterations                 */
  double max_corr_dist;     /* <= 0 or +inf: no gate (exactly the reference);
                               else keep pairs with distance < max_corr_dist        */
  const double* init_pose;  /* NULL or [n_pairs][6] = R00 R01 R10 R11 tx ty         */
} b200icp_options;

/* Any pointer except pose_total / error / iterations may be NULL. */
typedef struct b200icp_outputs {
  double* pose_total;   /* [n_pairs][6] cumulative R,t with src_final = R A + t          */
  double* pose_last;    /* [n_pairs][6] last increment: what icp() returns (icp.py:53)   */
  double* error;        /* [n_pairs] mean NN distance of the last search (icp.py:48)     */
  double* rmse;         /* [n_pairs] sqrt(mean d^2) over inliers of the last search      */
  int32_t* inliers;     /* [n_pairs] correspondences used by the last update             */
  int32_t* iterations;  /* [n_pairs] i+1 at break else max_iterations (icp.py:35,50)     */
  int32_t* indices;     /* [n_pairs][src_pitch] correspondences of the last search       */
  double* src_final;    /* [n_pairs][src_pitch][2] transformed source (icp.py:45,53)     */
  int32_t* index_history; /* [n_pairs][max_iterations][src_pitch] (diagnostics/parity)   */
  int64_t* evaluated_pairs; /* [n_pairs] source-target distance evaluations the candidate
                               sweep actually executed (all iterations); the brute-force
                               count is sum over iterations of n_src * n_tgt.  Diagnostics
                               for the pruned sweep (DESIGN.md 4.2)                      */
} b200icp_outputs;

/* ---- library ---------------------------------------------------------------- */
int b200icp_version(void);               /* major*1000 + minor                     */
const char* b200icp_last_error(void);    /* thread-local, never NULL               */

/* Largest pitches the fused per-pair kernel accepts (host query). */
int b200icp_max_src_pitch(void);
int b200icp_max_tgt_pitch(void);

/*
 * Nearest-neighbour correspondence search, one search per pair.
 * Replaces  tree = KDTree(B); distances, indices = tree.query(src)
 * (labels_segmentation/icp.py:37-38).
 *   idx_out   [n_pairs][src_pitch] int32, -1 beyond src_len
 *   dist2_out [n_pairs][src_pitch] float64 squared distance (NULL to skip)
 */
int b200icp_nn_batch(const b200icp_problem* prob, int64_t n_pairs,
                     int32_t* idx_out, double* dist2_out, int32_t flags /* B200ICP_FLAG_DENSE_SWEEP,
                     _WARP_KERNEL, _CTA_KERNEL; 0 = defaults */, void* stream);

/*
 * Whole ICP loop per pair, fused on the device (no host round trips).
 * Replaces icp() (labels_segmentation/icp.py:28-53) including
 * best_fit_transform() (icp.py:5-26).
 */
int b200icp_align_batch(const b200icp_problem* prob, int64_t n_pairs,
                        const b200icp_options* opt, const b200icp_outputs* out,
                        void* stream);

/*
 * 2D Generalized ICP (line-to-line), the registration objective of the reference's
 * gicp(points1, points2, threshold, voxel, trans_init) (duc/ICP_LIDAR/gicp_lidar.py:12-36, called at
 * slam_offline.py:382 and mainn.py:311).  Open3D is not vendored, so the model is defined by
 * oracle/gicp_oracle.py (parity-unpinned; DESIGN.md 4.8).
 *
 * b200icp_estimate_covariances: per point of every row of a table, the k nearest points of the same
 * row under the order (d^2, index) (the point itself included; all of them when the row has fewer
 * than k), their population covariance C (sums taken sequentially in that order, no contraction)
 * and the regularised  C_reg = u u^T + epsilon (I - u u^T),  u = (cos phi, sin phi),
 * phi = atan2(2 cxy, cxx - cyy) / 2.  C_reg = I when fewer than 3 neighbours or cxx + cyy = 0.
 *   points  [rows][pitch][2] (dtype);  len [rows] valid points per row (NULL = pitch)
 *   cov_out [rows][pitch][3] float64 (cxx, cxy, cyy); entries past len are 0.
 *   3 <= k <= 32; epsilon finite and > 0; pitch <= 65536 (O(n^2) per row: local maps and scans,
 *   not the scan-to-map map).
 */
int b200icp_estimate_covariances(const void* points, const int32_t* len, int32_t rows, int32_t pitch,
                                 int32_t dtype, int32_t k, double epsilon, double* cov_out, void* stream);

typedef struct b200icp_gicp_options {
  int32_t max_iterations;   /* updates (gicp_lidar.py:27: 50)                                   */
  int32_t reserved;
  double max_corr_dist;     /* <= 0 or +inf: no gate; else keep pairs with distance < it        */
  double relative_fitness;  /* stop when |d fitness| < relative_fitness AND                     */
  double relative_rmse;     /*           |d rmse| < relative_rmse (Open3D's defaults: 1e-6)    */
  const double* init_pose;  /* NULL or [n_pairs][6] = R00 R01 R10 R11 tx ty                     */
} b200icp_gicp_options;

/*
 * Whole GICP loop per pair, one CTA per pair (Open3D's RegistrationICP shape): evaluate at the
 * initial pose; then per update one float64 Gauss-Newton step in (dtheta, dx, dy) about the pivot
 * c = current pose applied to the centroid of the original source, with
 *   J = [[-(s_y - c_y), 1, 0], [s_x - c_x, 0, 1]],  r = b - s,  M = (C^B_j + R C^A_i R^T)^-1,
 *   H = sum J^T M J,  g = sum J^T M r,  H x = g by a 3x3 Cholesky factorisation;
 * apply s <- R(dtheta)(s - c) + c + dt and T <- dT o T (as increments: s + ((R(dtheta) - I)(s - c) + dt),
 * so a zero step changes nothing), and evaluate again.  An evaluation takes the
 * exact float64 nearest target of every source point (lowest index on ties, as b200icp_nn_batch),
 * the gate of b200icp_align_batch, fitness = inliers / n and rmse = sqrt(mean d^2) over inliers.
 * Stops when both relative criteria hold, after max_iterations updates, when an evaluation has
 * no inlier (error = rmse = +inf) or when a Cholesky pivot is not finite and positive (no update).
 * n = 0 or m = 0: the initial pose, iterations = 0, error = rmse = +inf.
 *   src_cov / tgt_cov: [rows][pitch][3] from b200icp_estimate_covariances, laid out like the point
 *   tables and indexed by the same rows (ROWWISE odometry offsets src_cov by one row, like
 *   src_points).  src_pitch <= 1024; tgt_pitch <= 65536 (targets are searched in shared-memory
 *   tiles of 4,096 and the results merged exactly).
 *   Outputs (b200icp_outputs): pose_total; pose_last = the last applied increment; error = mean
 *   inlier distance, rmse, inliers and indices at the FINAL pose; iterations = applied updates;
 *   index_history[it] = the correspondences update `it` used; evaluated_pairs unused (may be NULL).
 */
int b200icp_gicp_batch(const b200icp_problem* prob, int64_t n_pairs, const b200icp_gicp_options* opt,
                       const double* src_cov, const double* tgt_cov, const b200icp_outputs* out,
                       void* stream);

/*
 * Least-squares rigid transform between MATCHED rows (row i of the source onto row i of the
 * target, the first min(src_len, tgt_len) points of each pair).
 * Replaces best_fit_transform(A, B) (labels_segmentation/icp.py:5-26).
 *   pose_out [n_pairs][6] = R00 R01 R10 R11 tx ty.  Any pitch.  Degenerate H = 0 gives R = I.
 *   The sums take each cloud relative to its own first point, so clouds far apart (1e6 mm, 1 mm
 *   spread) keep the accuracy of clouds near the origin.
 */
int b200icp_best_fit_batch(const b200icp_problem* prob, int64_t n_pairs, double* pose_out,
                           void* stream);

/*
 * Scan preparation on the device: quality / range / front-arc filter and
 * polar -> Cartesian with order-preserving compaction.
 * Replaces polar_to_cartesian_3d (duc/ICP_LIDAR/process.py:38-52).
 *   raw      [n_scans][raw_pitch][3] float64 rows (quality, angle_deg, distance_mm)
 *   raw_len  [n_scans] valid rows per scan (NULL = raw_pitch; values above raw_pitch read raw_pitch rows)
 *   filter   NULL = the canonical thresholds of process.py:45-46; the reference's other copies of
 *            the function differ only in these constants: slam_offline.py:68-69 (0 < d < 10000,
 *            q > 13, arc), realtime_2.py:160-161 (0 < d < 5000, q > 5, no arc), realtime_1.py:164-167
 *            and b.py:173-177 (as realtime_2 with y = +d sin)
 *   xy_out   [n_scans][out_pitch][2] float64;  len_out [n_scans]
 *            The kept rows are written in input order.  A scan keeping more than out_pitch rows
 *            yields its first out_pitch kept points and len_out = out_pitch; rows of xy_out past
 *            len_out are zero.
 */
typedef struct b200icp_polar_filter {
  double min_dist, max_dist;    /* keep min_dist < distance < max_dist   (process.py:46: 1000, 9000) */
  double min_quality;           /* keep quality > min_quality            (process.py:46: 10)         */
  double arc_lo, arc_hi;        /* keep angle <= arc_lo or angle >= arc_hi (process.py:45: 135, 225) */
  int32_t use_arc;              /* 0: no arc test                                                    */
  int32_t y_sign;               /* -1: y = -d sin (process.py:49);  +1: y = +d sin                   */
} b200icp_polar_filter;

int b200icp_polar_to_cartesian(const double* raw, const int32_t* raw_len, int32_t n_scans,
                               int32_t raw_pitch, const b200icp_polar_filter* filter, double* xy_out,
                               int32_t* len_out, int32_t out_pitch, void* stream);

/* ---- scan-to-map ICP: a scan of a few thousand points against a map of millions, sharded
 * contiguously across GPUs (one process per GPU).  The scan-to-local-map call shape of
 * duc/ICP_LIDAR/mainn.py:297-318 / slam_offline.py:366-392 with the point-to-point loop of
 * labels_segmentation/icp.py:28-53 (KDTree(B).query(src), icp.py:37-38, is the search below).
 *
 * Once per map shard: b200icp_s2m_prepare_map -> one bounding circle per chunk of 1,024 consecutive
 * map points and one per 32 chunks.  The circle tables of all ranks (32 bytes per 1,024 points) are
 * gathered once by the caller and passed as b200icp_s2m_tables, so that every rank can bound a scan
 * point's nearest-neighbour distance over the WHOLE map without a per-iteration collective.
 * Per iteration and rank, two launches:
 *     b200icp_s2m_search  applies the pose increment the previous update left pending; per scan
 *                         point an upper bound of its NN distance (distance to the previous
 *                         iteration's nearest map point; circles in the first iteration); exhaustive
 *                         exact scan (float64 decisions; an FP32 test only skips points proven
 *                         farther than the bound) of every local chunk whose circle is within it ->
 *                         the exact nearest point of THIS shard among all that can matter (lowest
 *                         index on ties) or "none"; the 32-byte record goes to `records`, or, with
 *                         `peers`, straight into every rank's inbox over NVLink, followed by this
 *                         rank's flag (the all-gather is the kernel's epilogue).
 *     (caller)            without peers: all-gather of the records  -> records_all[ranks][n]
 *     b200icp_s2m_update  with `inbox`: waits for the flags of all ranks (2 s timeout -> state.done
 *                         = 2); global winner per point (distance, then lowest global index), pose
 *                         solve, convergence; bit-identical on every rank.
 * After the loop b200icp_s2m_finish applies the last pending increment to src64.
 * All are asynchronous and become no-ops once state->done is set, so a fixed-length loop needs no
 * host synchronisation (and can be captured in a CUDA graph). */
typedef struct b200icp_s2m_shard {
  const void* points;      /* [m][2] map points of this shard (dtype below)                    */
  int64_t m;               /* points in this shard                                             */
  int64_t global_offset;   /* index of points[0] in the whole map (contiguous sharding)        */
  int32_t dtype;           /* b200icp_dtype                                                    */
  int32_t reserved;
  /* filled by b200icp_s2m_prepare_map; caller-allocated, c = b200icp_s2m_padded_chunks(m):    */
  double* chunk_circle;    /* [c][4]: centroid x, y, bounding radius (< 0: padding), unused    */
  double* super_circle;    /* [c / 32][4]: the same for every 32 chunks                        */
  /* optional, both or neither (caller-allocated): a Morton-sorted copy of the shard, so that the
   * chunk circles are compact whatever the order of `points` (e.g. after a hash-based voxel filter).
   * Indices in the records and tie-breaking still refer to the ORIGINAL order.  m < 2^31.       */
  void* sorted_points;     /* [m][2], same dtype                                               */
  int32_t* order;          /* [m]: original local index of sorted point j                      */
} b200icp_s2m_shard;

typedef struct b200icp_s2m_tables {   /* circles of the whole map: every rank's, in rank order */
  const double* chunk_circle;   /* [n_chunks_total][4]                                         */
  const double* super_circle;   /* [n_chunks_total / 32][4]                                    */
  int32_t n_chunks_total;       /* multiple of 32                                              */
  int32_t first_local_chunk;    /* where this rank's (padded) chunks start; multiple of 32     */
  int32_t n_local_chunks;       /* = b200icp_s2m_padded_chunks(shard.m)                        */
  int32_t reserved;
} b200icp_s2m_tables;

typedef struct b200icp_s2m_record {   /* 32 bytes, one per scan point and rank */
  double d2;               /* exact float64 squared distance to the shard's nearest point, or
                              +inf when no chunk of the shard can hold the nearest neighbour    */
  int64_t gidx;            /* its global map index                                             */
  double bx, by;           /* its coordinates (so no rank needs another rank's shard)          */
} b200icp_s2m_record;

typedef struct b200icp_s2m_state {    /* device-resident, 136 bytes */
  double pose_total[6];    /* R00 R01 R10 R11 tx ty, cumulative                                */
  double pose_last[6];     /* last increment (what icp() returns, icp.py:53)                   */
  double error;            /* mean NN distance of the last search (icp.py:48)                  */
  double mean_d2;
  double prev_error;
  int32_t iterations;      /* completed updates                                                */
  int32_t inliers;
  int32_t done;            /* 1: converged / max_iterations / all gated out; 2: a peer timed out */
  int32_t applied;         /* increments already applied to src64 (iterations - 1 or iterations) */
} b200icp_s2m_state;

int b200icp_s2m_chunk(void);                                   /* 1024                          */
int64_t b200icp_s2m_padded_chunks(int64_t m);                  /* chunks of a shard, rounded up to 32 */
int64_t b200icp_s2m_scratch_bytes(int32_t n_scan);             /* tickets + partial sums; ZEROED once by the caller */
int64_t b200icp_s2m_prepare_workspace_bytes(int64_t m);        /* for the spatial sort; not needed without it */
int b200icp_s2m_prepare_map(const b200icp_s2m_shard* shard, void* workspace /*|NULL*/, int64_t workspace_bytes,
                            void* stream);
/* src64 [n][2] float64 scan state (written), prev_nn [n][2] float64 (written: "none"; may be NULL
 * for a one-shot search), state (written) */
int b200icp_s2m_init(const void* scan, int32_t dtype, int32_t n, const double* init_pose /*[6]|NULL*/,
                     double* src64, double* prev_nn, b200icp_s2m_state* state, void* stream);
/* records [n] (local output) or peers (DEVICE array of `world` inbox addresses, own inbox at
 * [rank]); exactly one of the two is used (peers wins). */
int b200icp_s2m_search(const b200icp_s2m_shard* shard, const b200icp_s2m_tables* tables, double* src64,
                       const double* prev_nn /*|NULL*/, int32_t n, b200icp_s2m_record* records,
                       void* const* peers, int32_t world, int32_t rank, b200icp_s2m_state* state,
                       void* scratch, void* stream);
/* records_all [n_ranks][n], or inbox (this rank's peer inbox; records_all ignored) */
int b200icp_s2m_update(const b200icp_s2m_record* records_all, void* inbox, int32_t n_ranks,
                       const double* src64, double* prev_nn, int32_t n, int32_t max_iterations,
                       double tolerance, double max_corr_dist, int32_t* idx_out /*[n]|NULL*/,
                       b200icp_s2m_state* state, void* scratch, void* stream);
int b200icp_s2m_finish(double* src64, int32_t n, b200icp_s2m_state* state, void* scratch, void* stream);

/*
 * Peer inboxes for scan-to-map: every rank allocates one peer-visible buffer of
 * b200icp_s2m_inbox_bytes(n, world) bytes (b200icp_peer_alloc: cudaMalloc + zero + IPC handle;
 * layout [2 slots][world][n] records, [2][world] int64 flags, one int64 exchange counter),
 * exchanges the 64-byte handles out of band, opens the others (b200icp_peer_open) and passes the
 * DEVICE array of the `world` addresses to b200icp_s2m_search.  Slots alternate per exchange; the
 * exchange counter is advanced by b200icp_s2m_update, so searches and updates must be paired and
 * every rank must issue the same sequence of calls.
 */
int64_t b200icp_s2m_inbox_bytes(int32_t n_scan, int32_t world);
int b200icp_peer_alloc(int64_t bytes, void** ptr_out /*host*/, void* handle_out /*host, 64 bytes*/);
int b200icp_peer_open(const void* handle /*host, 64 bytes*/, void** ptr_out /*host*/);
int b200icp_peer_close(void* ptr);
int b200icp_peer_free(void* ptr);

/*
 * Order-preserving selection of points (the steps either side of registration in the SLAM loop).
 *   mode 0: keep point i iff key[i] < threshold.  With key = squared NN distance to the previous
 *           scan (b200icp_nn_batch / b200icp_s2m_search) and threshold = d^2 this replaces
 *           remove_dynamic_points (duc/ICP_LIDAR/process.py:75-84: distances < distance_threshold).
 *   mode 1: keep point i iff |p_i - (cx, cy)|^2 < threshold: the local-map radius crop
 *           (duc/ICP_LIDAR/mainn.py:300-303: distances_sq < LOCAL_MAP_RADIUS_MM**2).  The squared
 *           distance is rounded as NumPy rounds it, (x - cx)^2 and (y - cy)^2 each rounded before
 *           the add (no FMA), so the kept set equals NumPy's bit for bit, on the circle too.
 * out_points [n][2] (same dtype), count_out: device int64, scratch: device int64[ceil(n/1024)+1].
 * n = 0 writes count_out = 0; points, key and out_points may then be NULL.
 */
int b200icp_select_points(const void* points, int32_t dtype, int64_t n, int32_t mode,
                          const double* key, double cx, double cy, double threshold,
                          void* out_points, int64_t* count_out, int64_t* scratch, void* stream);

/*
 * Sequence odometry: prefix composition of the pairwise poses of consecutive scans into global
 * poses, out[0] = identity, out[k+1] = out[k] o poses[k]  (the frame-to-frame pose carry of the
 * reference's SLAM loops, duc/ICP_LIDAR/slam_offline.py:382-392).
 *   poses [n][6], out [n+1][6], both R00 R01 R10 R11 tx ty, float64, device.  n = 0 writes the
 *   identity to out[0]; poses may then be NULL.
 */
int b200icp_chain_poses(const double* poses, int64_t n, double* out, void* stream);

/*
 * 2D voxel-grid down-sampling: one point per occupied cell (cell = floor(p / voxel_size)), the
 * mean of the points in it, cells ordered by (cell_y, cell_x).  Replaces
 * point_cloud.voxel_down_sample(voxel_size) as the reference uses it before registration
 * (duc/ICP_LIDAR/gicp_lidar.py:8-11,20-21) and for duplicate removal (process.py:68-73); the 2D
 * grid is labels_segmentation/d.py:10-16.  Parity-unpinned against Open3D (output order of
 * Open3D is unspecified).  out_points [n][2] (same dtype), count_out device int64.
 * Cells are int64 per axis, so cells 2^32 apart stay apart.  Points whose cell is not an int64
 * (non-finite coordinates, |p / voxel_size| >= 2^63) are skipped, like the non-finite points of
 * b200icp_occ_update; when every point is skipped, count_out = 0.
 */
int64_t b200icp_voxel_workspace_bytes(int64_t n);
int b200icp_voxel_downsample(const void* points, int32_t dtype, int64_t n, double voxel_size,
                             void* out_points, int64_t* count_out, void* workspace,
                             int64_t workspace_bytes, void* stream);

/*
 * Occupancy-grid ray casting (the mapping step that follows registration in the SLAM loop).
 * Replaces update_occupancy_map (duc/ICP_LIDAR/process.py:114-177; same body at
 * duc/ICP_LIDAR/slam_offline.py:174-236; called at mainn.py:340,749 and slam_offline.py:341,419)
 * including bresenham_line (process.py:86-112).  Bit-identical to the reference.
 *   probs : the reference keeps the probabilities in the function attribute
 *           update_occupancy_map.occupancy_probs (process.py:122-125), created as 0.5 everywhere;
 *           here the caller owns them.   image : the `occupancy_map` argument (h, w, 3) uint8; its
 *           window around the robot is re-rendered as grey levels after every frame
 *           (process.py:172-176).  NULL skips the rendering.
 * Per frame: window of +-area cells around the robot cell; for every point, in order, a ray
 * from the robot cell to the point's cell: cells before the end are multiplied by p_free_dec
 * until one is >= threshold_up (that ends the ray and the end cell is NOT raised), the end cell is
 * raised by p_occ_inc and clamped to 1.  Frames with no points change nothing.  Points with
 * non-finite coordinates are skipped (the reference raises on them).
 * float32 parameters: NumPy 2 evaluates `np.float32 * 0.9` with float32(0.9) (the caller passes
 * the rounded constants).
 */
typedef struct b200icp_occ_grid {
  float* probs;            /* [n_maps][h][w] float32, updated in place                       */
  uint8_t* image;          /* [n_maps][h][w][3] uint8 or NULL                                 */
  int32_t h, w;            /* cells; <= 32768 each                                            */
  double center_x, center_y; /* map_center_px (slam_offline.py:320)                           */
  double resolution;       /* mm per cell (Config.py:7)                                       */
  int32_t area;            /* half window in cells (process.py:115: 140); <= 10000            */
  float p_occ_inc;         /* process.py:115: float32(0.2)                                    */
  float p_free_dec;        /* process.py:115: float32(0.9)                                    */
  float threshold_up;      /* process.py:158: float32(0.65)                                   */
} b200icp_occ_grid;

/*
 * n_maps independent grids (one CTA each), n_frames frames applied to each in order:
 *   points   [n_maps][n_frames][pitch][2] map-frame coordinates (dtype f32/f64)
 *   len      [n_maps][n_frames] valid points per frame (NULL = pitch)
 *   robot_xy [n_maps][n_frames][2] float64 robot position (global_pose[:2, 3])
 */
int b200icp_occ_update(const b200icp_occ_grid* grid, int32_t n_maps, const void* points, int32_t dtype,
                       const int32_t* len, const double* robot_xy, int32_t n_frames, int32_t pitch,
                       void* stream);

/*
 * Point filter on cell probabilities.  Replaces filter_new_points_by_occupancy
 * (duc/ICP_LIDAR/process.py:203-226) and prune_global_map (process.py:228-249): point i is dropped
 * iff its cell lies inside the grid and probs[py, px] < free_threshold.
 *   points [n][cols] rows (x, y, ...), cols >= 2;  kept_index [n] int64: the kept row numbers in
 *   order (first *count_out entries);  scratch: int64[ceil(n/1024) + 1].
 */
int b200icp_occ_filter_points(const void* points, int32_t dtype, int32_t cols, int64_t n, const float* probs,
                              int32_t h, int32_t w, double center_x, double center_y, double resolution,
                              float free_threshold, int64_t* kept_index, int64_t* count_out,
                              int64_t* scratch, void* stream);

/*
 * FP32 FFMA throughput probe used as the roofline denominator of the NN phase
 * (MEASURED_PEAKS.json carries no FP32 figure).  Launches one kernel doing
 * `flop_out[0]` floating point operations (written to a HOST int64); the caller
 * times it with CUDA events on `stream`.  sink is a device float buffer of at
 * least 1 element.
 */
int b200icp_ffma_probe(float* sink, int32_t inner_iters, int64_t* flop_out /*host*/,
                       void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200ICP_H_ */
