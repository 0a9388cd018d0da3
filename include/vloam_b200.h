/* vloam_b200.h -- C ABI of the B200-native lidar registration hot path.
 *
 * Drop-in boundary for liuzm-slam/VLOAM-NOTED's per-frame chain
 *   scanRegistration -> laserOdometry -> laserMapping
 * (src/lidar_odometry_mapping).  The reference has no FFI: the path sits behind
 * three plain C++ classes driven by LidarOdometryMapping
 * (src/lidar_odometry_mapping.cpp:65-176).  Each entry point below names the
 * reference member function(s) it replaces; vloam_adapter.hpp re-creates the
 * classes on top of this ABI (see INTEGRATION.md).
 *
 * Conventions: every call returns 0 on success or a negative VLOAM_E_* code and
 * records a message readable with vloam_b200_last_error().  Quaternions are
 * x,y,z,w (the order of para_q, laser_odometry.cpp:84-91).  Points are
 * 16-byte {x,y,z,intensity} floats (pcl::PointXYZI without its padding,
 * common.h:42).  One context = one sequence; contexts are not thread-safe, like
 * the reference objects (different contexts may be driven from different
 * threads).  All compute runs in hand-written CUDA kernels; there is no CPU
 * fallback.
 *
 * Execution model.  A context owns several CUDA streams (the pose chain, side
 * streams for the stack filters / search structures / map update / look-ahead
 * scan registration and look-ahead odometry) and one helper host thread that issues side-stream launches.
 * The laserMapping sub-map is a persistent device voxel-hash grid that the per-sweep map update edits in place.
 * Calls queue work and return early where they can; the host blocks at
 *   S1  after scan registration, for the feature counts (inside laser_odometry),
 *   S2  after the mapping solve, for the pose and map sizes (inside
 *       laser_mapping on every MAPPED frame, with or without output pointers),
 * and inside every getter.  A frame on which mapping is skipped
 * (mapping_skip_frame > 1) with NULL output pointers returns without S2; the
 * device-side ordering between frames never depends on those host waits.
 * vloam_b200_publish_map() queues the assembly of the global map on a stream of
 * its own, behind the last map update, and returns; the next sweeps' map edits
 * wait for it on the device, so publishing neither blocks the caller nor
 * changes any result.  vloam_b200_get_map() is the only call that waits for it.
 * vloam_b200_synchronize() drains everything, including the helper thread.
 */
#ifndef VLOAM_B200_H_
#define VLOAM_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define VLOAM_OK 0
#define VLOAM_E_INVALID -1   /* bad argument / unsupported scan_line (SR.cpp:58-61, 255-259) */
#define VLOAM_E_CUDA -2      /* CUDA runtime error */
#define VLOAM_E_CAPACITY -3  /* a device buffer bound was exceeded */
#define VLOAM_E_NAME -4      /* unknown debug buffer name */

/* ROS parameters read by the three init() functions (SR.cpp:44-54,
 * LO.cpp:45-54, LM.cpp:44-45, 99-102, 125-128); defaults are the shipped KITTI
 * values (launch/loam_velodyne_HDL_64_kitti.launch:3-16). */
typedef struct vloam_b200_params {
  int n_scans;            /* scan_line: 16, 32, 64 (reference) or 128 (extension) */
  float minimum_range;    /* minimum_range */
  float line_res;         /* mapping_line_resolution */
  float plane_res;        /* mapping_plane_resolution */
  int mapping_skip_frame; /* mapping_skip_frame */
  int reserved;           /* flags: VLOAM_FLAG_DISTORTION | VLOAM_FLAG_TRANSFORM_TO_END, or 0 */
} vloam_b200_params;

/* LaserOdometry::DISTORTION (laser_odometry.h:90; a compile-time `false` in the reference): with this flag set in
 * vloam_b200_params.reserved the odometry de-skews every feature point by its sweep phase s = (intensity -
 * int(intensity)) / SCAN_PERIOD: TransformToStart uses Identity.slerp(s, q_last_curr) and s * t_last_curr
 * (laser_odometry.cpp:152-173) and the two odometry functors interpolate the same way (lidarFactor.hpp:29-33, 86-90). */
#define VLOAM_FLAG_DISTORTION 1
/* TransformToEnd (laser_odometry.cpp:176-193) applied as the block at laser_odometry.cpp:537-556 does (under `if (0)` in
 * the reference, whose KITTI sweeps come motion-compensated): after every odometry solve -- on the first frame too, with
 * identity -- every point of cornerPointsLessSharp, surfPointsLessFlat and laserCloudFullRes is moved into the frame of the
 * sweep's END: un = TransformToStart(p) (float; s from the intensity under VLOAM_FLAG_DISTORTION, s = 1 otherwise), then
 * q_last_curr.inverse() * (un - t_last_curr) in double, stored as float, intensity truncated to int(intensity).  Those clouds
 * become the "last" clouds of the next odometry solve and the mapping stage's input, and vloam_b200_register_full_cloud
 * registers the end-frame full-resolution cloud.  Set it together with VLOAM_FLAG_DISTORTION to de-skew sweeps that are not
 * motion-compensated; accepted with or without it. */
#define VLOAM_FLAG_TRANSFORM_TO_END 2

typedef struct vloam_b200_ctx vloam_b200_ctx;

/* Feature clouds handed between the stages (ScanRegistration::output SR.cpp:566-577,
 * LaserOdometry::output LO.cpp:660-679). */
enum {
  VLOAM_CLOUD_FULL = 0,        /* laserCloud: kept points, ring-major */
  VLOAM_CLOUD_SHARP = 1,       /* cornerPointsSharp */
  VLOAM_CLOUD_LESS_SHARP = 2,  /* cornerPointsLessSharp */
  VLOAM_CLOUD_FLAT = 3,        /* surfPointsFlat */
  VLOAM_CLOUD_LESS_FLAT = 4,   /* surfPointsLessFlat */
  VLOAM_CLOUD_CORNER_LAST = 5, /* laserCloudCornerLast (after solveLO's swap; end frame under VLOAM_FLAG_TRANSFORM_TO_END) */
  VLOAM_CLOUD_SURF_LAST = 6,   /* laserCloudSurfLast (same) */
  VLOAM_CLOUD_FULL_RES = 7     /* laserCloudFullRes as LaserOdometry::output hands it over: VLOAM_CLOUD_FULL, in the sweep-end
                                  frame under VLOAM_FLAG_TRANSFORM_TO_END (byte-equal to VLOAM_CLOUD_FULL without the flag) */
};

void vloam_b200_default_params(vloam_b200_params* p);

/* ScanRegistration::init + LaserOdometry::init + LaserMapping::init
 * (SR.cpp:42-92, LO.cpp:41-118, LM.cpp:40-129) on CUDA device `device`. */
int vloam_b200_create(const vloam_b200_params* p, int device, vloam_b200_ctx** out);
void vloam_b200_destroy(vloam_b200_ctx* c);
const char* vloam_b200_last_error(const vloam_b200_ctx* c);

/* LidarOdometryMapping::reset (LOM.cpp:65-71): ScanRegistration::reset +
 * LaserMapping::reset; call once per frame before scan_registration. */
int vloam_b200_begin_frame(vloam_b200_ctx* c);

/* ScanRegistration::input (SR.cpp:144-513).  xyz: HOST pointer to n points,
 * `stride` floats apart (3 for packed XYZ, 4 for KITTI x,y,z,r).  Asynchronous
 * with respect to the host unless a getter is called. */
int vloam_b200_scan_registration(vloam_b200_ctx* c, const float* xyz, int n, int stride);
/* Optional look-ahead for replays: register the NEXT sweep, or the next TWO sweeps in order (host pointer -- pinned for
 * an asynchronous copy -- or device pointer; registering a buffer that is already registered is a no-op, a third pending
 * registration replaces the second).  Upload and scan registration of a registered sweep are queued on a side stream from
 * inside the processing of the current sweep and run underneath that sweep's odometry and mapping; with two sweeps ahead the
 * odometry and the stack filters of sweep k+1 run beside the mapping of sweep k as well.  The scan_registration /
 * process_frame call with the same (pointer, n, stride) finds the work done; a call with any other buffer drops everything
 * that was registered or computed ahead and runs the plain path.  CONTRACT: adoption is keyed
 * on (pointer, n, stride) only -- the buffer must stay valid AND UNCHANGED from this call until the scan_registration /
 * process_frame call that consumes it returns; a caller that refills one buffer in place must not register it.
 * Results are bit-identical with or without the look-ahead.  No reference counterpart: the bag player hands over one
 * sweep at a time (MAIN.cpp:143). */
int vloam_b200_prefetch_scan(vloam_b200_ctx* c, const float* xyz, int n, int stride);
int vloam_b200_prefetch_scan_device(vloam_b200_ctx* c, const float* d_xyz, int n, int stride);
/* Same, but xyz is a DEVICE pointer already resident in HBM. */
int vloam_b200_scan_registration_device(vloam_b200_ctx* c, const float* d_xyz, int n, int stride);

/* ScanRegistration::output / LaserOdometry::output cloud hand-off: copies cloud
 * `which` to host memory (out may be NULL to query the size).  Returns the
 * number of points or a negative error. */
int vloam_b200_get_cloud(vloam_b200_ctx* c, int which, float* out_xyzi, int cap_points);

/* LaserOdometry::input + solveLO + output (LO.cpp:137-148, 199-584, 660-679).
 * prior_q/prior_t: velo_last_VOT_velo_curr, read when use_prior != 0
 * (detach_VO_LO == false, LO.cpp:237-250).  Outputs (any may be NULL): odometry
 * pose q_w_curr/t_w_curr, frame-to-frame q_last_curr/t_last_curr, skip_frame. */
int vloam_b200_laser_odometry(vloam_b200_ctx* c, const double* prior_q, const double* prior_t, int use_prior,
                              double* q_w_curr, double* t_w_curr, double* q_last_curr, double* t_last_curr,
                              int* skip_frame);

/* LaserMapping::input + solveMapping (LM.cpp:178-209, 212-814), fed from the
 * context's own odometry output as LOM.cpp:149-158 does, or from the caller's
 * vloam_b200_laser_mapping_input of this frame (below).  Outputs (may be
 * NULL): the mapped pose q_w_curr/t_w_curr (the high-frequency propagated pose
 * on skipped frames, LM.cpp:197-201). */
int vloam_b200_laser_mapping(vloam_b200_ctx* c, double* q_w_curr, double* t_w_curr);

/* Stage inputs from the caller.  The reference's LaserOdometry::input (LO.cpp:137-148) and LaserMapping::input
 * (LM.cpp:178-209) deep-copy whatever they are handed; these four calls do the same, so the stages can run on edited clouds
 * (moving objects removed), behind another odometry (a VO-fused or wheel / INS pose), on recorded odometry output, or as
 * separate contexts.
 *
 * Points: x, y, z at float offsets 0..2 and the intensity at float offset w_offset of records `stride` floats apart
 * (4, 3 = packed xyzi; 8, 4 = pcl::PointXYZI as PCL lays it out in memory).  Only those four floats are read; the copy moves
 * bits, so results are bit-identical to the same points produced on the device.
 * Copies: a host buffer may be reused as soon as the call returns.  Device buffers (the _device variants) are read on the
 * context's main stream (vloam_b200_stream) in the order of the context's calls.
 * Validation: VLOAM_E_INVALID with a message for n < 0, NULL with n > 0, stride < 4, w_offset outside [3, stride - 1], a
 * NULL pose and skip_frame other than 0 / 1.
 * No cost without them: a context that never makes these calls runs no extra launch, wait or allocation; their buffers are
 * reserved by the first call.
 *
 * Odometry input: the five ScanRegistration clouds in VLOAM_CLOUD_FULL .. VLOAM_CLOUD_LESS_FLAT order replace this frame's
 * vloam_b200_scan_registration (call it after begin_frame, before vloam_b200_laser_odometry); get_cloud(0..4) then returns
 * them.  Ring ids are int(intensity); the clouds need not be ring-major.  Under VLOAM_FLAG_TRANSFORM_TO_END they are moved to
 * the sweep end like scan-registration output.  The call drops every look-ahead registered or computed with
 * vloam_b200_prefetch_scan, as a scan_registration call with an unregistered buffer does; results stay bit-identical with or
 * without the look-ahead. */
int vloam_b200_laser_odometry_input(vloam_b200_ctx* c, const float* const clouds[5], const int n[5], int stride, int w_offset);
int vloam_b200_laser_odometry_input_device(vloam_b200_ctx* c, const float* const d_clouds[5], const int n[5], int stride, int w_offset);
/* Mapping input: laserCloudCornerLast, laserCloudSurfLast, laserCloudFullRes, q_wodom_curr (x,y,z,w), t_wodom_curr and
 * skip_frame, consumed by exactly one vloam_b200_laser_mapping call of this frame (skip_frame = 1: it returns the
 * high-frequency pose q_wmap_wodom * q_wodom_curr, LM.cpp:197-201).  An input that no mapping call consumes is dropped by the
 * next begin_frame; without one, laser_mapping reads the context's own odometry output.  The input never touches the
 * context's odometry (its "last" clouds, its pose, its frame count, the next frame's skip decision): a context may run its
 * own scan registration and odometry and still map the caller's clouds.  The clouds are used exactly as given (LaserMapping
 * applies no TransformToEnd), and vloam_b200_register_full_cloud after that mapping call registers the caller's `full`
 * cloud. */
int vloam_b200_laser_mapping_input(vloam_b200_ctx* c, const float* corner, int nc, const float* surf, int ns, const float* full, int nfull,
                                   int stride, int w_offset, const double* q_wodom, const double* t_wodom, int skip_frame);
int vloam_b200_laser_mapping_input_device(vloam_b200_ctx* c, const float* d_corner, int nc, const float* d_surf, int ns, const float* d_full,
                                          int nfull, int stride, int w_offset, const double* q_wodom, const double* t_wodom, int skip_frame);

/* The full-resolution cloud of this sweep registered into the map frame: LaserMapping::publish's loop
 * over laserCloudFullRes with pointAssociateToMap (LM.cpp:901-905; q_w_curr / t_w_curr after
 * solveMapping, the propagated pose on skipped frames).  Under VLOAM_FLAG_TRANSFORM_TO_END each point is
 * pointAssociateToMap(TransformToEnd(p)) with a float intermediate, the cloud LaserOdometry hands over.  out_xyzi: HOST buffer of cap_points points (NULL
 * to query the size).  Returns the number of points or a negative error. */
int vloam_b200_register_full_cloud(vloam_b200_ctx* c, float* out_xyzi, int cap_points);

/* LaserMapping::publish, LM.cpp:884-899: queue the assembly of laserCloudMap (all 4851 cubes, corner then surf per cube)
 * from the map as of the last mapped frame.  Returns at once; the device orders every later map edit behind it.  (A call
 * that has to grow the context's publication buffers -- the first one, or when the map outgrew them -- first waits for the
 * previous publication.) */
int vloam_b200_publish_map(vloam_b200_ctx* c);
/* Wait for the last publish_map and copy its cloud to host memory (out NULL: size query).  Returns the number of points,
 * VLOAM_E_CAPACITY when cap_points is too small, VLOAM_E_INVALID when nothing was published since create.  A second
 * publish_map before get_map replaces the first. */
int vloam_b200_get_map(vloam_b200_ctx* c, float* out_xyzi, int cap_points);

/* Prior maps: start from a map built earlier -- to continue mapping it in a later session, or to localize in it with the map held
 * fixed.  No reference counterpart (LaserMapping always starts empty, LM.h:75-78); a context that never makes these calls runs no
 * extra launch, wait or allocation, and their buffers are reserved by the first call.
 *
 * load_map replaces the context's map, both kinds, with world-frame (map-frame) clouds: `corner` for laserCloudCornerArray, `surf` for
 * laserCloudSurfArray, as (stride, w_offset) float records like the stage inputs above (host pointers; device pointers for the _device
 * variant, read on the context's main stream).  Each point goes to its cube by the insert formula (LM.cpp:747-756) at the context's
 * current window centre (laserCloudCen*); points outside the 21x21x11 grid (LM.cpp:758-761) and points with a non-finite x, y or z
 * are dropped, and dropped[2] (may be NULL) receives how many per kind.  Every non-empty cube is then pcl::VoxelGrid-filtered at
 * line_res / plane_res over its points in input order (LM.cpp:795-808): one centroid per occupied voxel, f32 sums in input order,
 * ascending voxel order.  Poses, odometry state, frame counts and the window centre are unchanged.  The call waits for the helper
 * thread, the map update in flight and a pending publish_map (whose get_map still returns the old map); the next mapped sweep
 * rebuilds its search structures.  Errors: VLOAM_E_INVALID as for the stage inputs, VLOAM_E_CAPACITY above 2097151 points of a kind;
 * on any error the map is unchanged.  Empty clouds clear the map.
 * A published map round-trips: load_map(get_map_kind(0), get_map_kind(1)) at the window centre it was published with gives back
 * the same cubes. */
int vloam_b200_load_map(vloam_b200_ctx* c, const float* corner, int nc, const float* surf, int ns, int stride, int w_offset,
                        long long dropped[2]);
int vloam_b200_load_map_device(vloam_b200_ctx* c, const float* d_corner, int nc, const float* d_surf, int ns, int stride, int w_offset,
                               long long dropped[2]);
/* The odometry-to-map transform q_wmap_wodom (x,y,z,w) / t_wmap_wodom the mapping stage keeps (transformUpdate, LM.cpp:147-151): it
 * forms the next initial guess (LM.cpp:206-207) and the skipped-frame pose (LM.cpp:197-201), i.e. where the sensor starts in a
 * loaded map.  Ordered on the device behind the last mapping; takes effect at the next laser_mapping.  VLOAM_E_INVALID for NULL or
 * non-finite values. */
int vloam_b200_set_map_pose(vloam_b200_ctx* c, const double q_wmap_wodom[4], const double t_wmap_wodom[3]);
/* enabled = 0: later mapped sweeps localize against the map without changing it -- LM.cpp:741-808 (insert, re-filter, raw appends
 * to cubes outside the window) is skipped; the solve, transformUpdate, register_full_cloud, publish_map, skipped frames and the
 * look-ahead are as before, and the window still rolls (LM.cpp:252-444), clearing the cubes that leave the grid.  enabled = 1
 * (the default) resumes normal updates on the current map. */
int vloam_b200_set_map_update(vloam_b200_ctx* c, int enabled);
/* The corner (which = 0) or surf (1) points of the last publish_map, in cube order: the get_map cloud without the other kind's
 * cubes.  Same waits and errors as get_map; VLOAM_E_INVALID for another `which`. */
int vloam_b200_get_map_kind(vloam_b200_ctx* c, int which, float* out_xyzi, int cap_points);

/* Relocalization: find the sensor in a loaded map without an initial guess -- after a restart inside a saved map, say.  No reference
 * counterpart.  Call order: load_map, set_map_update(c, 0), one process_frame (its mapped pose is meaningless: the map pose is still the
 * identity), relocalize with apply = 1, then keep calling process_frame; sweeps registered ahead with prefetch_scan stay valid.
 *
 * The search is exact over its discretisation (branch and bound over translation on the device; the scores are integers):
 *   Query points: the VoxelGrid-filtered stacks of the last mapped sweep (lm.cornerStack then lm.surfStack, in that sweep's sensor
 *   frame -- its end frame under VLOAM_FLAG_TRANSFORM_TO_END), the ones with (x*x + y*y) + z*z <= max_range^2 (double) in that order,
 *   every k-th of the n kept with k = ceil(n / max_points), each as u = R_c p in double.  R_c is Eigen's toRotationMatrix of q_c / |q_c|.
 *   Grid: cells of size r = resolution; N = floor(half_xy / r), Nz = floor(half_z / r); Gx = Gy = 2 (ceil(max_range / r) + N + 1),
 *   Gz = 2 (ceil(max |u_z| / r) + Nz + 1); origin o = t_c - r (G / 2) (integer G / 2).  A cell is occupied when a point of either
 *   kind of the map falls in it: floor((m - o) / r) in double.
 *   Candidates (j, iz, iy, ix), iz in [-Nz, Nz], iy and ix in [-N, N]: R = Rz(theta_j) R_c (roll and pitch of the centre are kept),
 *   t = t_c + r (ix, iy, iz).  Yaw step d = yaw_step_deg (degrees), or r / max_range radians when it is 0.  half_yaw_deg = 180: j in
 *   [0, ceil(2 pi / d - 1e-9)), theta_j = j d; otherwise J = floor(half_yaw_deg pi / 180 / d + 1e-9), j in [-J, J].  Linear index
 *   ((j' nZ + iz') S + iy') S + ix' with every coordinate counted from its lowest value, S = 2N + 1, nZ = 2Nz + 1.
 *   Score: the number of query points whose cell floor(((c u_x - s u_y) + t_c.x - o_x) / r), ... (c, s = cos, sin theta_j; z:
 *   floor((u_z + t_c.z - o_z) / r)) moved by (ix, iy, iz) is occupied (outside the grid: not).  best: the highest score, ties to the
 *   lowest index; runner-up: the same outside {max(|dx|, |dy|) < exclusion_m and |d theta| < exclusion_deg} around best (yaw distance
 *   taken around the circle when half_yaw_deg = 180).  found: best score >= min_score * n_points.
 * With apply and found, q/t_wmap_wodom (vloam_b200_set_map_pose's field) is set by transformUpdate (LM.cpp:147-151) from the found pose
 * and the odometry pose the last mapped sweep was mapped with; the next laser_mapping starts from there (LM.cpp:206-207) and its solve
 * refines the last half cell and half yaw step.  Nothing else changes: no map edit, no lm.pose write, no window move.
 * The call drains the context (vloam_b200_synchronize) and blocks until the result is on the host.  Errors: VLOAM_E_INVALID for NULL
 * pointers, non-finite or negative values, resolution / max_range / max_points <= 0, half_yaw_deg > 180, no mapped sweep since create or
 * the last load_map (or a skipped sweep last), an empty map and no query point within max_range; VLOAM_E_CAPACITY above 2^31 - 1
 * candidates or grid cells, or 16383 translation steps per side.  A context that never calls it makes no extra launch, wait or
 * allocation. */
typedef struct vloam_b200_reloc_params {
  double q_c[4], t_c[3];  /* centre pose T_map_sensor (q x,y,z,w): the caller's rough guess; default identity */
  double half_xy;         /* m, default 20 */
  double half_z;          /* m, default 1 */
  double half_yaw_deg;    /* 180 (default) = every heading */
  double resolution;      /* m: occupancy cell and translation step, default 1 */
  double yaw_step_deg;    /* 0 (default) = resolution / max_range radians */
  double max_range;       /* m, default 60 */
  double min_score;       /* fraction of the query points for `found`, default 0.3 */
  double exclusion_m;     /* runner-up exclusion zone, default 3 m ... */
  double exclusion_deg;   /* ... and 10 degrees */
  int max_points;         /* default 2048 */
  int apply;              /* default 1: set q/t_wmap_wodom when found */
} vloam_b200_reloc_params;
typedef struct vloam_b200_reloc_result {
  double q[4], t[3];                 /* best pose T_map_sensor */
  double runner_q[4], runner_t[3];   /* runner-up pose (zeros when every candidate lies in the exclusion zone) */
  long long index, runner_index;     /* linear candidate indices (-1: no runner-up) */
  long long candidates;              /* size of the search space */
  long long nodes;                   /* bounds and scores evaluated by both searches */
  int score, runner_score;           /* query points on occupied cells (runner_score -1: none) */
  int n_points;                      /* query points */
  int found;
} vloam_b200_reloc_result;
void vloam_b200_default_reloc_params(vloam_b200_reloc_params* p);
int vloam_b200_relocalize(vloam_b200_ctx* c, const vloam_b200_reloc_params* p, vloam_b200_reloc_result* result);

/* MAIN.cpp:143-144, 186-190 in one call: begin_frame, scan_registration,
 * laser_odometry, laser_mapping.  pose_out (may be NULL): 14 doubles
 * {odom q[4], odom t[3], mapped q[4], mapped t[3]}.  On a mapped frame the call
 * returns after sync point S2 (the pose is final; the map update continues on a
 * side stream); on a skipped frame it blocks only when pose_out is non-NULL. */
int vloam_b200_process_frame(vloam_b200_ctx* c, const float* xyz, int n, int stride, double* pose_out);
int vloam_b200_process_frame_device(vloam_b200_ctx* c, const float* d_xyz, int n, int stride, double* pose_out);

/* Block until all work queued on any of the context's streams (and by its helper thread) has finished. */
int vloam_b200_synchronize(vloam_b200_ctx* c);
/* The context's main (pose-chain) cudaStream_t (as void*), for timing with CUDA events after vloam_b200_synchronize. */
void* vloam_b200_stream(vloam_b200_ctx* c);
/* Number of kernels this context has launched since creation. */
long long vloam_b200_kernel_launches(const vloam_b200_ctx* c);
/* Per-stage device time of the last frame in ms {SR, LO, LM}; needs timing enabled. */
int vloam_b200_set_timing(vloam_b200_ctx* c, int enabled);
int vloam_b200_stage_ms(vloam_b200_ctx* c, float* ms3);

/* Measurement aid: record CUDA events around every launch of the kernel called `name`
 * (NULL switches it off); profile_result returns how many launches were timed, their
 * summed duration and the algorithmic bytes the launch sites declared for them. */
int vloam_b200_profile_kernel(vloam_b200_ctx* c, const char* name);
int vloam_b200_profile_result(vloam_b200_ctx* c, int* launches, double* total_ms, double* total_bytes);
/* After profile_kernel(c, "*") (every launch timed): text table "name count total_ms total_bytes" per line. */
int vloam_b200_profile_table(vloam_b200_ctx* c, char* buf, int cap);
/* Same launches as a timeline: "name stream start_us end_us" per line (stream 0 = main .. 3), relative to the first. */
int vloam_b200_profile_timeline(vloam_b200_ctx* c, char* buf, int cap);

/* State export / import and stage-level inspection, keyed by name.  The
 * reference keeps this state in private members (LO.h:90-147, LM.h:102-203);
 * teacher-forced parity tests inject the oracle's state through these.
 * get: returns the byte size (copying when out != NULL and cap suffices).
 * Names: sr.laserCloud sr.sharp sr.lessSharp sr.flat sr.lessFlat sr.curvature
 * sr.label sr.scanStartInd sr.scanEndInd lo.cornerLast lo.surfLast lo.pose
 * lo.assoc.corner{0,1} lo.assoc.surf{0,1} lm.pose lm.state lm.cornerStack
 * lm.surfStack lm.cornerFromMap lm.surfFromMap lm.validInd lm.cornerMap
 * lm.surfMap lm.knn.{cidx,sidx,cd2,sd2,cok,sok}{0,1} lm.costs lo.costs
 * lm.paths (int64 {in-place, pool-path} mapped sweeps since create);
 * of the last relocalize: rl.points (float64 u xyz per query point), rl.occ (float64 origin[3], int64 dims[3], then the level-0
 * occupancy bytes, x fastest), rl.yaw (float64 cos, sin per yaw), rl.levels (int64 frontier nodes kept per level [2][16], then the
 * nodes evaluated per pass [2]), rl.ms (float32 device ms {search, occupancy + pyramid});
 * set: lo.last lo.pose lm.pose lm.state lm.cornerMap lm.surfMap. */
long vloam_b200_debug_get(vloam_b200_ctx* c, const char* name, void* out, long cap_bytes);
int vloam_b200_debug_set(vloam_b200_ctx* c, const char* name, const void* data, long bytes);
/* Odometry association only (LO.cpp:282-485) at pose x = {qx,qy,qz,qw,tx,ty,tz}
 * of the current sharp/flat clouds against the last clouds; state untouched.
 * corner_idx: 2 ints per sharp point, surf_idx: 3 per flat point (-1 = none). */
int vloam_b200_lo_associate(vloam_b200_ctx* c, const double* x, int* corner_idx, int* surf_idx);

/* pcl::VoxelGrid on a host cloud (SR.cpp:497-501, LM.cpp:492-500, 795-808),
 * run by the same device kernels the stages use.  Returns the output count. */
int vloam_b200_voxel_grid(vloam_b200_ctx* c, const float* in_xyzi, int n, float leaf, float* out_xyzi, int cap_points);

/* One robustified evaluation of the normal equations (the per-iteration work
 * Ceres does for LO.cpp:500-509 / LM.cpp:710-717): factors are nf x 10 doubles
 * {type, p[3], a[3], b[3]} (type 0 LidarEdgeFactor, 1 LidarPlaneFactor,
 * 2 LidarPlaneNormFactor; lidarFactor.hpp:14-144).  Outputs cost, H[36], g[6]. */
int vloam_b200_evaluate(vloam_b200_ctx* c, const double* factors, int nf, const double* x, double* cost, double* H,
                        double* g);
/* ceres::Solve as configured by the reference on the same factor list. */
int vloam_b200_solve(vloam_b200_ctx* c, const double* factors, int nf, double* x, double* log4);
/* The same two calls with a per-factor interpolation ratio s[nf] (DISTORTION: LidarEdgeFactor / LidarPlaneFactor evaluate
 * Identity.slerp(s, q) * p + s t and are differentiated through the slerp, lidarFactor.hpp:29-36, 86-93); s == NULL is
 * the plain call. */
int vloam_b200_evaluate_deskew(vloam_b200_ctx* c, const double* factors, const double* s, int nf, const double* x, double* cost,
                               double* H, double* g);
int vloam_b200_solve_deskew(vloam_b200_ctx* c, const double* factors, const double* s, int nf, double* x, double* log4);

/* The two neighbourhood fits of solveMapping on caller-supplied five-point sets (float32[n][5][3], the map
 * neighbours as the kNN returns them): kind 0 = 3x3 covariance + SelfAdjointEigenSolver line test, accepted when
 * lambda_2 > 3 lambda_1 (LM.cpp:559-603); kind 1 = colPivHouseholderQr plane with the 0.2 m check (LM.cpp:637-680).
 * ok[n]: accept flags; params[n][6]: {a[3], b[3]} of the LidarEdgeFactor / {unit normal[3], d, 0, 0} of the
 * LidarPlaneNormFactor (zeros when rejected).  Same device code as the mapping stage. */
int vloam_b200_fit(vloam_b200_ctx* c, const float* near_xyz, int n, int kind, int* ok, double* params);

/* atanf(x[i]) and atan2f(y[i], x[i]) exactly as the scan-registration kernels evaluate them on the device (the reference
 * calls glibc's float routines at SR.cpp:185-187, 217, 263; a 1-ulp difference moves points across ring boundaries, so the
 * device code carries bit-identical fdlibm restatements).  Host arrays in and out; a test aid. */
int vloam_b200_exact_math(vloam_b200_ctx* c, const float* y, const float* x, int n, float* atan_x, float* atan2_yx);

#ifdef __cplusplus
}
#endif
#endif /* VLOAM_B200_H_ */
