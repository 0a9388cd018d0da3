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
 * context's own odometry output as LOM.cpp:149-158 does.  Outputs (may be
 * NULL): the mapped pose q_w_curr/t_w_curr (the high-frequency propagated pose
 * on skipped frames, LM.cpp:197-201). */
int vloam_b200_laser_mapping(vloam_b200_ctx* c, double* q_w_curr, double* t_w_curr);

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
