/* coreslam_b200.h — C ABI of the B200-native CoreSLAM scan-to-map hot path.
 *
 * Drop-in boundary for SLAM.NET's CoreSLAMProcessor (C#).  The reference has no FFI layer; the
 * boundary is the public surface of CoreSLAM/CoreSLAMProcessor.cs, which a C# wrapper keeps verbatim
 * and forwards here through P/Invoke (see INTEGRATION.md for the [DllImport] stubs).  Plain C types
 * only: pointers, sizes, PODs.  Every entry point returns a cs_status (0 = ok); cs_last_error()
 * gives the text.  There is no CPU fallback: without a CUDA device cs_create fails with
 * CS_ERR_NO_DEVICE.
 *
 * Citations "file:line" are relative to the reference tree (mikkleini/slam.net @ 7abc587).
 *
 * Threading: calls on one handle are caller-serialised (CoreSLAMProcessor.Update is blocking and
 * non-reentrant, BaseSLAM/ParallelWorker.cs:94-97).  Distinct handles may be used from distinct
 * threads; each owns one CUDA stream.
 */
#ifndef CORESLAM_B200_H
#define CORESLAM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CS_ABI_VERSION 1

typedef enum cs_status {
  CS_OK = 0,
  CS_ERR_INVALID_ARGUMENT = 1,
  CS_ERR_NO_DEVICE = 2,   /* no CUDA device / driver: the product path never falls back to the CPU */
  CS_ERR_CUDA = 3,        /* sticky: the handle is unusable afterwards */
  CS_ERR_OUT_OF_MEMORY = 4,
  CS_ERR_CAPACITY = 5,    /* more points / candidates than the handle was created for */
  CS_ERR_STATE = 6,
  CS_ERR_NCCL = 7         /* multi-GPU exchange failed (peer mapping refused, or a rank of the group never delivered its key) */
} cs_status;

/* cs_config.flags */
#define CS_FLAG_ROW_MAJOR_MAP 0x1u /* keep the device map row-major (default: 8x8-cell tiled, one 128 B line per tile) */
#define CS_FLAG_TIMING 0x2u        /* record CUDA events around every kernel (cs_get_timing) */
#define CS_FLAG_KEEP_DISTANCES 0x4u /* cs_update also stores all per-candidate distances (cs_get_distances) */
#define CS_FLAG_NO_HOST_SPIN 0x8u  /* wait for the pose with cudaEventSynchronize instead of polling mapped memory */
#define CS_FLAG_L2_PERSIST 0x10u   /* put a persisting L2 access-policy window over the map */
#define CS_FLAG_DEBUG_RAYS 0x20u   /* keep x1,y1,x2,y2,xp,yp of every ray of the last integration (cs_get_rays) */
#define CS_FLAG_SEARCH_WARP 0x40u  /* always search with the warp-per-candidate kernel (default: by candidate count) */
#define CS_FLAG_SEARCH_SLAB 0x80u  /* always search with the heading-sorted slab kernels, whatever the candidate count */
#define CS_FLAG_DEBUG_BOUNDED_SPIN 0x100u /* debugging aid: every device-side poll between the kernels of a step (pose, ray
                                             arrival, cell hand-off) gives up after 2 s (CS_TUNE_SPIN_MS) instead of spinning
                                             for ever; the grid drains and the handle's next call returns CS_ERR_CUDA naming
                                             the poll.  For runs under MPS / time-slicing / a debugger, where the co-residency
                                             the polls rely on may not hold.  Costs one clock read per 1024 poll turns. */

typedef struct cs_processor cs_processor; /* opaque; replaces a CoreSLAMProcessor instance */
typedef struct cs_scanlog cs_scanlog;     /* opaque; device-resident scan log for replays */
typedef struct cs_batch cs_batch;         /* opaque; N independent sessions on one GPU */

/* Mirrors the constructor CoreSLAMProcessor(physicalMapSize, holeMapSize, obstacleMapSize, startPose,
 * sigmaXY, sigmaTheta, iterationsPerThread, numSearchThreads), CoreSLAMProcessor.cs:119-120.
 * obstacle_map_size = 0 leaves the ObstacleMap half of Update (:751) out (the scan-to-pose benchmarks do);
 * > 0 keeps a device-resident ObstacleMap and every Update / cs_integrate also runs UpdateObstacleMap. */
typedef struct cs_config {
  float physical_map_size;   /* metres, edge of the square map */
  int32_t hole_map_size;     /* pixels per edge (HoleMap.Size, HoleMap.cs:17-22) */
  float start_pose[3];       /* x, y (m), theta (rad) */
  float sigma_xy;            /* metres */
  float sigma_theta;         /* radians */
  int32_t iterations_per_thread;
  int32_t num_search_threads; /* <= 0: SingleMonteCarloSearch (:662-665), candidates = iterations */
  int32_t device;            /* CUDA device ordinal */
  int32_t max_points;        /* scan staging capacity; 0 -> 16384 */
  uint64_t seed;             /* Philox seed for production-mode candidates */
  void* stream;              /* optional cudaStream_t to run on; NULL -> the handle creates its own */
  uint32_t flags;            /* CS_FLAG_* */
  int32_t obstacle_map_size; /* pixels per edge of the ObstacleMap (ObstacleMap.cs:17-22), 0 = none */
} cs_config;

/* Result of one search / update.  distance = INT32_MAX and index = 0 when nothing was in bounds or
 * when the scan was integrated without a search (scanCount < PositionSearchBeginning, :726-743). */
typedef struct cs_result {
  float pose[3];      /* CoreSLAMProcessor.Pose after the call (theta normalised, :745-747) */
  int32_t distance;   /* winner's "distance" (:253) */
  int32_t index;      /* flat candidate index: 0 = searchPose, 1 + t*I + i (:674-710 tie-break order) */
  int32_t searched;   /* 1 if a pose search ran for this scan */
  int64_t visits;     /* HoleMap cells written by the integration (sum over rays of dxc+1) */
} cs_result;

typedef struct cs_timing {
  float search_ms, finalize_ms, integrate_ms; /* device time of the last call's kernels (CS_FLAG_TIMING); the glue
                                                 now runs inside the update kernel, so finalize_ms is 0 */
  float h2d_ms;
  float total_device_ms;
  double host_wait_ms;                        /* host wall time of the last cs_update until the pose was available */
  float obstacle_ms;                          /* UpdateObstacleMap kernels of the last call (0 without an ObstacleMap) */
  float reserved;
} cs_timing;

int32_t cs_abi_version(void);
const char* cs_last_error(const cs_processor* h); /* h may be NULL: error of the last failed create on this thread */
int32_t cs_device_count(void);                    /* number of CUDA devices, 0 when the driver is absent */

/* ---- lifetime: ctor :119-162, Reset :167-175, Dispose :757-773 ------------------------------------ */
cs_status cs_create(const cs_config* cfg, cs_processor** out);
cs_status cs_destroy(cs_processor* h);
cs_status cs_reset(cs_processor* h); /* map := 32750, Pose := startPose, lastOdometryPose := 0, scanCount := 0 */

/* ---- properties :40-106 ---------------------------------------------------------------------------- */
cs_status cs_set_quality(cs_processor* h, int32_t quality);                  /* Quality, 1..255, default 50 */
cs_status cs_set_hole_width(cs_processor* h, float metres);                  /* HoleWidth, default 0.6 */
cs_status cs_set_position_search_beginning(cs_processor* h, int32_t scans);  /* default 5 */
cs_status cs_get_pose(cs_processor* h, float pose[3]);                       /* Pose */
cs_status cs_set_pose(cs_processor* h, const float pose[3], const float last_odometry[3], int32_t scan_count);
cs_status cs_get_map_info(const cs_processor* h, int32_t* size, float* scale); /* HoleMap.Size / HoleMap.Scale */

/* ---- ObstacleMap: CoreSLAM/ObstacleMap.cs:11-44, CoreSLAMProcessor.cs:53 (needs cs_config.obstacle_map_size > 0) ----
 * UpdateObstacleMap (:540-593) and DrawLaserRayOnObstacleMap (:456-490) run on the device at the end of every
 * cs_update / cs_integrate / cs_replay step, after the HoleMap integration, from the same pose and cloud.   */
cs_status cs_set_unmapped_obstacle_hits(cs_processor* h, int32_t hits); /* UnmappedObstacleHits (:98), sbyte, default -5; used by the next cs_reset */
cs_status cs_set_max_obstacle_hits(cs_processor* h, int32_t hits);      /* MaxObstacleHits (:103), sbyte, default 10 */
cs_status cs_get_obstacle_map_info(const cs_processor* h, int32_t* size, float* scale); /* ObstacleMap.Size / .Scale (0 when absent) */
cs_status cs_obstacle_map_download(cs_processor* h, int8_t* pixels);      /* ObstacleMap.Pixels, Size*Size sbyte, [y, x] row-major */
cs_status cs_obstacle_map_upload(cs_processor* h, const int8_t* pixels);
cs_status cs_obstacle_map_fill(cs_processor* h, int32_t value);
cs_status cs_get_obstacle_visits(cs_processor* h, int64_t* touched);      /* map cells the rays touched since the last reset/fill (measurement) */

/* ---- the hot path ---------------------------------------------------------------------------------- */

/* ParallelMonteCarloSearch (:674-710) with explicit inputs: evaluates CalculateDistanceSISD
 * (:226-259) for searchPose (flat index 0) and n_cand candidate poses, returns the arg-min under the
 * reference's tie-break order.  Does not touch the processor state or the map.
 *   points       n_points * (x, y), metres, lidar frame (ScanCloud.Points, BaseSLAM/ScanCloud.cs:10-21)
 *   cand_poses   n_cand * (x, y, theta) absolute poses — "upload the reference's candidates" mode.
 *                NULL: the handle's Philox stream is used for scan index `scan_index` (n_cand must then
 *                be T*I).
 *   cand_cs      optional (n_cand+1) * (cos theta, sin theta), unscaled, entry 0 = searchPose: host libm
 *                values for callers whose libm is not glibc x86-64.  NULL: computed on the device with
 *                the glibc-identical routine.
 *   distances    optional out, n_cand+1 values in flat order.                                        */
cs_status cs_search(cs_processor* h, const float* points, int32_t n_points, const float search_pose[3],
                    const float* cand_poses, const float* cand_cs, int32_t n_cand, uint32_t scan_index,
                    cs_result* best, int32_t* distances);

/* ---- relocalisation on an existing map (no reference counterpart: its simulator only offers Reset) ----------------------
 * Where is this scan on the handle's map, from a pose nobody knows (a restart, a robot carried elsewhere, lost tracking)?
 * cs_relocalize evaluates CalculateDistanceSISD (:226-259) at every pose of a regular (x, y, theta) lattice on the device
 * and returns the best distinct hypotheses.
 *   Lattice pose  (ix, iy, it) = (origin[0] + (float)ix*step[0], origin[1] + (float)iy*step[1], origin[2] + (float)it*step[2]),
 *                 each multiply and add one f32 rounding, no FMA (an axis with count 1 is its origin, whatever its step).
 *                 Flat index (it*count[1] + iy)*count[0] + ix.  Poses may lie partly or wholly off the map; headings may lie
 *                 outside [-pi, pi].
 *   Distance      exactly what cs_search returns for the same pose passed as an absolute candidate: px = X*Scale + 0.5f,
 *                 c = cosf(theta)*Scale with the library's libm-identical cosf/sinf, the sum divided by ALL points;
 *                 INT32_MAX when no point is in bounds.
 *   Selection     the key of a pose is (distance, flat index).  A pose is reported when its distance is < INT32_MAX and its
 *                 key is strictly smaller than the key of every other lattice pose within +-window steps on each of the
 *                 three axes (the box clipped at the lattice edges; theta does not wrap).  window = 0 is a plain top-k.
 *                 hits receives at most k of them in ascending key order, *n_hits how many.  The result does not depend
 *                 on the launch shape.  (The window test reads every pose of the box of a minimum: a window as large as
 *                 the lattice costs as many reads as the lattice has poses, per minimum.)
 *   State         reads the HoleMap as it stands after everything already queued on the handle and changes nothing else:
 *                 map, pose, lastOdometryPose, scanCount, the Philox stream position, a candidate sort queued ahead, the
 *                 glue table and the CS_FLAG_KEEP_DISTANCES buffer stay as they were.  Either map layout.  Uses the
 *                 handle's own map only, also when it is attached to a candidate-split group.  Waits for its results.
 *   distances     optional out: count[0]*count[1]*count[2] values in flat order (one device-to-host copy).
 *   Errors        CS_ERR_INVALID_ARGUMENT: NULL arguments, n_points <= 0, a count < 1, a non-finite origin, a non-finite or
 *                 non-positive step on an axis with count > 1, window < 0, k outside 1..CS_LATTICE_MAX_HITS.
 *                 CS_ERR_CAPACITY: n_points > max_points, or more than CS_LATTICE_MAX_POSES poses (split a bigger lattice,
 *                 e.g. by heading range).  CS_ERR_OUT_OF_MEMORY: the distance volume (4 B per pose, kept by the handle
 *                 for later calls) could not be allocated.  The handle stays usable after any of these.
 * To resume tracking: cs_relocalize_bounded (below) with a fine lattice over the map, then
 * cs_set_pose(best, odometry of that scan, PositionSearchBeginning) and Update as usual (INTEGRATION.md). */
#define CS_LATTICE_MAX_POSES (1 << 28) /* poses per call */
#define CS_LATTICE_MAX_HITS 64

typedef struct cs_lattice {
  float origin[3];  /* pose of lattice point (0,0,0): x, y (m), theta (rad) */
  float step[3];    /* spacing along x, y (m), theta (rad) */
  int32_t count[3]; /* points along x, y, theta; each >= 1 */
} cs_lattice;

typedef struct cs_lattice_hit {
  float pose[3];    /* the lattice pose as evaluated (theta NOT normalised) */
  int32_t distance; /* CalculateDistanceSISD (:226-259) at that pose */
  int32_t index;    /* flat lattice index */
} cs_lattice_hit;

cs_status cs_relocalize(cs_processor* h, const float* points, int32_t n_points, const cs_lattice* lattice, int32_t window,
                        int32_t k, cs_lattice_hit* hits, int32_t* n_hits,
                        int32_t* distances /* optional: count[0]*count[1]*count[2] values in flat order */);

/* cs_relocalize_bounded returns exactly the hits of cs_relocalize (poses, distances, indices and order) for the same
 * lattice, window and k, and accepts lattices of up to CS_LATTICE_MAX_POSES_BOUNDED poses, so a whole room at a fine
 * step fits one call.  Most poses are never evaluated: it bounds the distance of blocks of poses from below and prunes
 * the blocks whose bound exceeds an upper bound U on the k-th hit (branch and bound, DESIGN section 4).
 *   Descent       the lattice is cut, per heading, into nodes of 2^L x 2^L (x, y) poses.  A node's bound is floor(1024 *
 *                 sum / n_points) over the points of the minimum of the HoleMap over the cells the point can reach from
 *                 the node's poses (0 for a point that may leave the map); it is <= the distance of every pose of the node.
 *                 A node whose bound is > U is dropped; the others are split down to 16 x 8 patches, whose poses are
 *                 evaluated exactly as in cs_relocalize.  A node whose every point lies wholly off the map is dropped at
 *                 any U: its poses are all int.MaxValue.
 *   Exactness     U starts as the k-th smallest exact distance of one pose per top-level node.  A pose that passes the
 *                 window test with distance <= U is a true window minimum.  When fewer than k pass, U is raised and the
 *                 descent runs again, at the latest with U = INT32_MAX - 1, which prunes only poses of distance int.MaxValue.
 *   Cost          besides the descent, every call rebuilds min-window grids of the map: up to 11 row-major copies of the
 *                 HoleMap (2 B per cell each; 11 x 8 MB for a 2048^2 map), kept by the handle like the other scratch.
 *   State         as cs_relocalize: reads the map as it stands after the queued work and changes nothing else on the handle;
 *                 either map layout; the handle's own map, also when it is attached to a group.  Waits for its results.
 *                 There is no distance-volume output: cs_relocalize returns the volume.
 *   stats         optional out (below).
 *   Errors        as cs_relocalize, with CS_LATTICE_MAX_POSES_BOUNDED for the pose limit, and CS_ERR_CAPACITY when more
 *                 than CS_LATTICE_BOUNDED_MAX_NODES nodes survive one level of the descent (at the last level a node is a
 *                 32 x 32 tile of one heading, so at most 2^30 poses are evaluated; a uniform map prunes nothing), or when
 *                 the lattice has more than 2^28 such tiles (count[0] and count[1] far below 32 with very many headings),
 *                 or count[0] or count[1] > 2^30.
 *                 The handle stays usable after any of these. */
#define CS_LATTICE_MAX_POSES_BOUNDED 2147483647 /* poses per cs_relocalize_bounded call: the flat index stays an int32 */
#define CS_LATTICE_BOUNDED_MAX_NODES (1 << 20)  /* nodes that may survive one level of cs_relocalize_bounded's descent */

typedef struct cs_relocalize_stats {
  int64_t poses;       /* count[0]*count[1]*count[2] */
  int64_t evaluated;   /* poses whose exact distance was computed, summed over the passes */
  int64_t bounded;     /* (node, level) bounds computed, summed over the passes */
  int32_t levels;      /* levels of the descent */
  int32_t passes;      /* 1, or more when U had to be raised */
  int32_t upper_bound; /* U of the last pass */
  int32_t reserved;
} cs_relocalize_stats;

cs_status cs_relocalize_bounded(cs_processor* h, const float* points, int32_t n_points, const cs_lattice* lattice,
                                int32_t window, int32_t k, cs_lattice_hit* hits, int32_t* n_hits,
                                cs_relocalize_stats* stats /* optional */);

/* cs_relocalize_sequence and cs_relocalize_sequence_bounded score every lattice pose with the last few scans instead of
 * one: a hypothesis that fits the newest scan but not what the robot saw a little earlier is rejected, which a single
 * scan cannot do in corridors of repeated doors, rows of shelves or identical rooms.
 *   Scans         K = n_scans scans, 1 <= K <= CS_SEQUENCE_MAX_SCANS.  points holds them back to back as (x, y) in metres,
 *                 each in its own lidar frame (ScanCloud.Points); scan k owns points [scan_first[k], scan_first[k+1]),
 *                 scan_first[0] = 0.  odometry[3k .. 3k+2] is the odometry pose of scan k.
 *   Anchor        the lattice pose is the pose of the LAST scan, a = odometry[K-1], so a hit is the pose to resume at:
 *                 cs_set_pose(hit.pose, odometry[K-1], ...).  Relative motion is SE(2) composition (the odometry frame's
 *                 heading may be unrelated to the map's).  All f32, one rounding per operation in this order, no FMA,
 *                 cosf/sinf the library's libm-identical ones.  Per scan k, once per call:
 *                   ca = cosf(a.theta), sa = sinf(a.theta), ex = o_k.x - a.x, ey = o_k.y - a.y,
 *                   dx_k = ca*ex + sa*ey, dy_k = ca*ey - sa*ex, dtheta_k = o_k.theta - a.theta.
 *                 At lattice pose (x, y, theta), with c = cosf(theta), s = sinf(theta) unscaled:
 *                   x_k = x + (c*dx_k - s*dy_k), y_k = y + (s*dx_k + c*dy_k), theta_k = theta + dtheta_k.
 *   Distance      D = sum over k of d_k, d_k exactly what cs_search returns for scan k at (x_k, y_k, theta_k) as an absolute
 *                 candidate (the sum divided by scan k's point count); INT32_MAX when some d_k is INT32_MAX.  D <= 32 *
 *                 1024 * 65535 = 2147450880 < INT32_MAX.
 *                 At K = 1 every scan sits at the lattice pose: the volume and hits are bit-identical to cs_relocalize's
 *                 (and the bounded call's hits to cs_relocalize_bounded's), whatever the odometry; such a call runs the
 *                 single-scan kernels.
 *   Lattice, window, k, selection, hit order, state, distances and stats
 *                 as cs_relocalize (cs_relocalize_sequence) and cs_relocalize_bounded (cs_relocalize_sequence_bounded).
 *                 stats.evaluated counts poses, not (pose, scan) pairs.  The bounded call's node bound is the sum of the
 *                 scans' bounds; a node where some scan lies wholly off the map at every pose is dropped at any U.
 *   Errors        as those calls, and CS_ERR_INVALID_ARGUMENT for NULL scan_first or odometry, n_scans outside
 *                 1..CS_SEQUENCE_MAX_SCANS, scan_first[0] != 0, a scan with fewer than 1 point or a non-finite odometry
 *                 value; CS_ERR_CAPACITY for a scan with more than max_points points.  The handle stays usable.
 *   Cost          grows with K: about K times the single-scan call, more when the bounded call needs another pass
 *                 (DESIGN section 5); the concatenated scans go to device scratch
 *                 that the handle keeps (8 B per point). */
#define CS_SEQUENCE_MAX_SCANS 32

cs_status cs_relocalize_sequence(cs_processor* h, const float* points, const int32_t* scan_first, const float* odometry,
                                 int32_t n_scans, const cs_lattice* lattice, int32_t window, int32_t k,
                                 cs_lattice_hit* hits, int32_t* n_hits,
                                 int32_t* distances /* optional: count[0]*count[1]*count[2] values in flat order */);
cs_status cs_relocalize_sequence_bounded(cs_processor* h, const float* points, const int32_t* scan_first, const float* odometry,
                                         int32_t n_scans, const cs_lattice* lattice, int32_t window, int32_t k,
                                         cs_lattice_hit* hits, int32_t* n_hits, cs_relocalize_stats* stats /* optional */);

/* UpdateHoleMap (:496-534) + DrawLaserRayOnHoleMap (:359-443) + ClipRay (:320-345) for an explicit
 * pose; uses the handle's HoleWidth and Quality.  pose_cs: optional host (cos, sin) of pose[2].
 * Asynchronous: returns after enqueueing; visits (optional) forces a wait for the count.            */
cs_status cs_integrate(cs_processor* h, const float* points, int32_t n_points, const float pose[3],
                       const float* pose_cs, int64_t* visits);

/* CoreSLAMProcessor.Update (:717-752) after ScanSegmentsToCloud: search gate, searchPose = Pose +
 * (odo - lastOdo), search, NormalizeAngle, state update, HoleMap integration.  Returns as soon as the
 * new pose is known; the integration keeps running on the stream and is ordered before the next call.
 *   cand_offsets  T*I * (dx, dy, dtheta): the values the reference would dequeue for this scan
 *                 (verification mode, :633-638).  NULL: on-device Philox Gaussian (production mode). */
cs_status cs_update(cs_processor* h, const float* points, int32_t n_points, const float odometry_pose[3],
                    const float* cand_offsets, cs_result* out);

/* CoreSLAMProcessor.Update(List<ScanSegment>) exactly as the reference declares it (:717-752), ScanSegmentsToCloud
 * (:187-207) included: the host uploads the raw rays and segment poses, the cloud is computed on the device (same f32
 * operations in the same order, libm-identical cosf/sinf) and feeds the search and both map integrations directly.
 *   rays        n_rays * (angle [rad], radius [m]) of all segments back to back (BaseSLAM/Ray.cs, ScanSegment.Rays)
 *   seg_first   n_segments + 1 indices: segment s owns rays [seg_first[s], seg_first[s+1]); seg_first[n_segments] = n_rays
 *   seg_poses   n_segments * (x, y, theta): ScanSegment.Pose; the odometry pose of the Update is the LAST segment's (:719)
 * n_segments = 0 fails like segments.Last() on an empty list does (InvalidOperationException -> CS_ERR_INVALID_ARGUMENT). */
cs_status cs_update_segments(cs_processor* h, const float* rays, const int32_t* seg_first, const float* seg_poses, int32_t n_rays,
                             int32_t n_segments, const float* cand_offsets, cs_result* out);
/* ScanSegmentsToCloud alone (:187-207) for an explicit odometry pose: points_out receives n_rays * (x, y). */
cs_status cs_segments_to_cloud(cs_processor* h, const float* rays, const int32_t* seg_first, const float* seg_poses, int32_t n_rays,
                               int32_t n_segments, const float odometry_pose[3], float* points_out);

/* Candidate-split GROUP: the same split as cs_update_begin / cs_update_finish below, but with the 8-byte exchange done
 * INSIDE the search kernel — the thread that owns this GPU's arg-min writes the packed key into every rank's table over
 * peer-mapped memory (NVLink), waits until its own table holds the world's keys, takes the minimum and publishes the
 * pose: no collective launch, no second kernel, the kernels of a scan stay chained.  After cs_group_attach every
 * cs_update / cs_update_segments / cs_replay of the handle evaluates this rank's slice
 * [rank*(T*I+1)/world, (rank+1)*(T*I+1)/world) and ends on the group's winner; all ranks must feed the same scans in the
 * same order (and, in verification mode, the same full candidate table).  A rank that waits longer than 2 s for the
 * others fails the call with CS_ERR_NCCL.  Replaces the cross-thread arg-min of ParallelMonteCarloSearch
 * (CoreSLAMProcessor.cs:694-705) at GPU granularity.
 *   one process per GPU:  cs_group_export on every rank, exchange the 64-byte handles by any means (MPI, a socket,
 *                         torch.distributed.all_gather), cs_group_attach(rank, world, handles) on every rank;
 *   one process, several handles (one per device, or several on one device): cs_group_attach_local(rank, world, peers). */
typedef struct { unsigned char bytes[64]; } cs_ipc_handle;
cs_status cs_group_export(cs_processor* h, cs_ipc_handle* out);
cs_status cs_group_attach(cs_processor* h, int32_t rank, int32_t world, const cs_ipc_handle* handles /* world entries */);
cs_status cs_group_attach_local(cs_processor* h, int32_t rank, int32_t world, cs_processor* const* peers /* world entries */);
cs_status cs_group_detach(cs_processor* h);

/* Multi-GPU candidate split (very large candidate sets, BASELINE cfg4): the map is replicated, GPU g
 * evaluates the flat candidate indices [cand_first, cand_first + cand_count) of the same scan, and ONE
 * 8-byte exchange picks the winner: the packed key (uint32 distance << 32 | uint32 flat index) is
 * min-reduced over the GPUs in place at *key_device between the two calls — on the handle's stream, e.g.
 * ncclAllReduce(key, key, 1, ncclUint64, ncclMin, comm, stream) or torch.distributed.all_reduce(MIN) on an
 * int64 view (the key is < 2^63).  cs_update_finish then decodes the same winner on every GPU, publishes
 * the pose and integrates the scan into this GPU's replica (deterministic, so replicas stay identical
 * without any map traffic).  In verification mode every GPU passes the full T*I offset table (the winner
 * is looked up by flat index); in Philox mode (cand_offsets = NULL) nothing is uploaded.
 * Replaces the cross-thread arg-min of ParallelMonteCarloSearch (:694-705) at GPU granularity. */
cs_status cs_update_begin(cs_processor* h, const float* points, int32_t n_points, const float odometry_pose[3],
                          const float* cand_offsets, int32_t cand_first, int32_t cand_count, uint64_t** key_device);
cs_status cs_update_finish(cs_processor* h, cs_result* out);

/* Wait until everything enqueued on the handle (including the last integration) has finished. */
cs_status cs_sync(cs_processor* h);

/* ---- map access: HoleMap.Pixels (public field, HoleMap.cs:27), row-major y*Size+x ------------------ */
cs_status cs_map_download(cs_processor* h, uint16_t* pixels);      /* Size*Size values */
cs_status cs_map_upload(cs_processor* h, const uint16_t* pixels);
cs_status cs_map_fill(cs_processor* h, uint16_t value);
cs_status cs_map_packed(cs_processor* h, uint8_t* packed);          /* HoleMap.GetPackedPixels, HoleMap.cs:44-55 */
/* Asynchronous export in the reference's viewer formats: a snapshot is taken in stream order (after the last
 * integration, before the next Update) and copied to `dst` on a side stream while the next Updates run.  `dst` should be
 * pinned (cs_pinned_alloc) for the copy to overlap; it is valid after cs_map_export_wait.  One export in flight per handle
 * (a second cs_map_export_begin queues behind the first). */
typedef enum cs_export_format {
  CS_EXPORT_GRAY16 = 0,      /* HoleMap.Pixels, Size*Size uint16 row-major: what MainWindow.xaml.cs:227-229 feeds a Gray16 bitmap */
  CS_EXPORT_PACKED4 = 1,     /* HoleMap.GetPackedPixels (HoleMap.cs:44-55), Size*Size/2 bytes */
  CS_EXPORT_OBSTACLE_I8 = 2  /* ObstacleMap.Pixels, Size*Size sbyte [y, x] */
} cs_export_format;
cs_status cs_map_export_begin(cs_processor* h, int32_t format, void* dst);
cs_status cs_map_export_wait(cs_processor* h);
cs_status cs_map_checksum(cs_processor* h, uint64_t* checksum);     /* position-dependent 64-bit hash computed on the device */
uint64_t cs_host_map_checksum(const uint16_t* pixels, int32_t size); /* same hash of a host row-major map */

/* ---- diagnostics ------------------------------------------------------------------------------------ */
cs_status cs_set_flags(cs_processor* h, uint32_t flags);   /* TIMING / KEEP_DISTANCES / NO_HOST_SPIN can change at run time */
cs_status cs_get_timing(cs_processor* h, cs_timing* t);
cs_status cs_get_distances(cs_processor* h, int32_t* distances, int32_t count); /* needs CS_FLAG_KEEP_DISTANCES */
cs_status cs_get_rays(cs_processor* h, int32_t* rays, int32_t n_points);         /* x1,y1,x2,y2,xp,yp of the last integration (CS_FLAG_DEBUG_RAYS) */
cs_status cs_get_visits(cs_processor* h, int64_t* visits);   /* cells written by the last integration (waits for it) */
/* Diagnostics (timeline of the last step; the first call enables the recording and returns nothing, later calls
 * copy `count` values).  Records of 8 int64 each:
 *   record b < Size             sub-task b of the draw kernel (cs_wedge_kernel): %globaltimer (ns) at [0] task start,
 *                               [1] candidates of its first piece found, [2] task end; [3] most candidates of a piece
 *                               | general path used << 16 | pieces << 20 | first ring << 32; %globaltimer of its block
 *                               at [4] block start, [5] rays ready, [6] task table ready; [7] SM id | block << 16
 *   record Size + b, b < 8192   block b of the search kernel: [0] SM id, %globaltimer at [1] start, [2] dependency
 *                               wait over, [3] scan staged, [4] warp 0 done, [5] block done, [6] pose published
 *                               (last block only), [7] 1 for the block that published */
cs_status cs_get_ring_cycles(cs_processor* h, int64_t* cycles, int32_t count);
/* Which search kernel and launch shape a scan of n_points points and n_cand random candidates gets on this handle:
 * plan[0] = 1 heading-sorted slab search (cs_sort_kernel + cs_search2_kernel), 0 warp-per-candidate (cs_search_kernel);
 * plan[1..2] = grid (x, y); plan[3] = threads per block; plan[4] = points per block. */
cs_status cs_get_search_plan(cs_processor* h, int32_t n_points, int32_t n_cand, int32_t plan[5]);
cs_status cs_get_launch_count(cs_processor* h, uint64_t* launches);              /* kernels launched so far by this handle */

/* ---- pinned staging so the C# side can fill ScanCloud points in place ------------------------------- */
cs_status cs_pinned_alloc(void** ptr, uint64_t bytes);
cs_status cs_pinned_free(void* ptr);

/* ---- device-resident scan logs: replays with no host round trip per scan ---------------------------- */
cs_status cs_scanlog_create(int32_t device, int32_t n_scans, int32_t max_points, int32_t n_offsets, cs_scanlog** out);
cs_status cs_scanlog_set(cs_scanlog* log, int32_t scan, const float* points, int32_t n_points,
                         const float odometry_pose[3], const float* cand_offsets /* n_offsets*3 or NULL */);
cs_status cs_scanlog_upload(cs_scanlog* log);
cs_status cs_scanlog_destroy(cs_scanlog* log);
/* Scan-log files (the reference has no log format — its simulator generates scans live, MainWindow.xaml.cs:380-407 —
 * so a recorded drive can be replayed through both implementations).  Little-endian:
 *   header 32 B : "CSLG", u32 version = 1, u32 n_scans, u32 max_points, u32 n_offsets, 12 B reserved (0)
 *   per scan    : u32 n_points, f32 odometry[3], f32 points[n_points][2] (metres, lidar frame, = ScanCloud.Points),
 *                 f32 offsets[n_offsets][3] (the candidate deviates the reference would dequeue; absent when n_offsets = 0)
 * cs_scanlog_file_info / cs_scanlog_file_read are host-only (no CUDA device needed). */
cs_status cs_scanlog_save(const cs_scanlog* log, const char* path);
cs_status cs_scanlog_load(int32_t device, const char* path, cs_scanlog** out); /* created, filled and uploaded */
cs_status cs_scanlog_file_info(const char* path, int32_t* n_scans, int32_t* max_points, int32_t* n_offsets);
cs_status cs_scanlog_file_read(const char* path, int32_t scan, float* points /* max_points*2 */, int32_t* n_points,
                               float odometry_pose[3], float* cand_offsets /* n_offsets*3 or NULL */);
/* Runs Update for scans [first, first+count) back to back on the device; results[count] optional.
 * With results == NULL the call only enqueues the work and returns (cs_sync waits for it). */
cs_status cs_replay(cs_processor* h, const cs_scanlog* log, int32_t first, int32_t count, cs_result* results);

/* ---- batches of independent sessions on one GPU (parameter sweeps / scan-log replays, BASELINE cfg5) ----
 * One launch per kernel for all sessions (grid.y = session); every session has its own HoleMap, ObstacleMap (when
 * obstacle_map_size > 0), pose, sigma_xy / sigma_theta / seed / start_pose (cfgs[j]), Quality, HoleWidth,
 * MaxObstacleHits and UnmappedObstacleHits.  Map size, obstacle_map_size, iterations, threads, device, max_points
 * and flags must be equal across cfgs.  No communication between sessions.  With obstacle_map_size > 0 every
 * batched Update (cs_batch_update, cs_batch_submit, cs_batch_replay) also runs UpdateObstacleMap (:751) for every
 * session, as cs_update does for one processor. */
cs_status cs_batch_create(const cs_config* cfgs, int32_t n_sessions, cs_batch** out);
cs_status cs_batch_destroy(cs_batch* b);
const char* cs_batch_last_error(const cs_batch* b);
int32_t cs_batch_size(const cs_batch* b);
cs_status cs_batch_set_params(cs_batch* b, int32_t session /* <0: all */, int32_t quality, float hole_width);
/* Update for every session: points n_sessions*max_points*(x,y) with max_points = cfgs[0].max_points exactly as passed to
 * cs_batch_create (odd or even; 0 means 16384): session j's points start at points + j*max_points*2 and it uses the first
 * n_points[j] of them, odometry n_sessions*3, cand_offsets n_sessions*T*I*3 or NULL (Philox), results optional n_sessions records. */
cs_status cs_batch_update(cs_batch* b, const float* points, const int32_t* n_points, const float* odometry,
                          const float* cand_offsets, cs_result* results);
/* The same Update, pipelined: cs_batch_submit stages and queues one step and returns; cs_batch_collect waits for the oldest
 * submitted step and copies out its n_sessions result records (NULL: only wait).  At most two steps may be waiting for
 * their collect (a third submit fails with CS_ERR_STATE).  A caller that alternates submit(k+1), collect(k) overlaps the host
 * staging of step k+1 with the device's work on step k.  (No reference counterpart: CoreSLAMProcessor.Update is blocking,
 * CoreSLAMProcessor.cs:717; this is the batched replay's throughput path.) */
cs_status cs_batch_submit(cs_batch* b, const float* points, const int32_t* n_points, const float* odometry,
                          const float* cand_offsets);
cs_status cs_batch_collect(cs_batch* b, cs_result* results);
/* Every session replays scans [first, first+count) of one shared device-resident log; results: optional
 * n_sessions records of the last scan. */
cs_status cs_batch_replay(cs_batch* b, const cs_scanlog* log, int32_t first, int32_t count, cs_result* results);
cs_status cs_batch_sync(cs_batch* b);
cs_status cs_batch_get_poses(cs_batch* b, float* poses /* n_sessions*3 */);
cs_status cs_batch_map_download(cs_batch* b, int32_t session, uint16_t* pixels);
cs_status cs_batch_map_checksums(cs_batch* b, uint64_t* checksums /* n_sessions */);
cs_status cs_batch_get_launch_count(cs_batch* b, uint64_t* launches);
/* CoreSLAMProcessor.Reset (:167-175) of every session at once (the sessions share one step state): HoleMap := 32750,
 * ObstacleMap := the session's UnmappedObstacleHits, Pose := its cfgs[j].start_pose, lastOdometryPose := 0,
 * scanCount := 0, and the Philox stream restarts at scan 0.  Quality, HoleWidth and MaxObstacleHits are kept.
 * CS_ERR_STATE while submitted steps wait for cs_batch_collect. */
cs_status cs_batch_reset(cs_batch* b);
/* The sessions' ObstacleMaps (need obstacle_map_size > 0, CS_ERR_STATE otherwise); session < 0: all sessions.
 * unmapped_hits: UnmappedObstacleHits (:98), sbyte, default -5, used by the next cs_batch_reset;
 * max_hits: MaxObstacleHits (:103), sbyte, default 10, used from the next step. */
cs_status cs_batch_set_obstacle_params(cs_batch* b, int32_t session, int32_t unmapped_hits, int32_t max_hits);
cs_status cs_batch_obstacle_map_download(cs_batch* b, int32_t session, int8_t* pixels); /* Size*Size sbyte, [y, x] row-major */
cs_status cs_batch_obstacle_checksums(cs_batch* b, uint64_t* checksums /* n_sessions */); /* cs_host_obstacle_checksum of each map */
cs_status cs_batch_get_obstacle_visits(cs_batch* b, int64_t* touched /* n_sessions */);  /* as cs_get_obstacle_visits, per session */
/* Host-only: sum over the row-major cells i of ((uint8_t)pixel + 1) * mix64(i), mod 2^64 (the hash of cs_host_map_checksum). */
uint64_t cs_host_obstacle_checksum(const int8_t* pixels, int32_t size);

/* ---- host twins of the device generators (for building verification tables; not a compute path) ----- */
/* offsets[n*3] = the Philox deviates the device uses for candidates 0..n-1 of scan `scan_index`. */
void cs_philox_offsets(uint64_t seed, uint32_t scan_index, int32_t n, float sigma_xy, float sigma_theta, float* offsets);
void cs_host_sincos(const float* angles, int32_t n, float* cos_out, float* sin_out); /* the library's cosf/sinf, host build */
cs_status cs_device_sincos(int32_t device, const float* angles, int32_t n, float* cos_out, float* sin_out);
float cs_host_normalize_angle(float a);
/* Measured ceiling for the search's access pattern: random 2-byte loads over a table of `cells`
 * uint16 (L2-resident when it fits), best of `repeats`.  Used by bench.py as the gather roofline. */
/* Host-only diagnostic: the number of rings the library sizes a scan's integration for — an upper bound of the longest clipped
 * ray in cells, + 1 (DrawLaserRayOnHoleMap walks x = 0..dxc, CoreSLAMProcessor.cs:404), from the scan's largest range, the map
 * scale (HoleMap.cs:20) and HoleWidth (:525).  A session batch launches exactly this many rings per session. */
int32_t cs_rings_hint(int32_t size_pixels, float size_meters, float hole_width, const float* points, int32_t n_points);
cs_status cs_gather_peak(int32_t device, int64_t cells, int32_t per_thread, int32_t repeats, double* lookups_per_s);

#ifdef __cplusplus
}
#endif
#endif /* CORESLAM_B200_H */
