// vloam_adapter.hpp -- the reference's C++ stage classes re-created on top of the C ABI, WITH THE REFERENCE'S SIGNATURES.
//
// Drop-in for src/lidar_odometry_mapping/include/lidar_odometry_mapping/
//   {scan_registration.h, laser_odometry.h, laser_mapping.h, lidar_odometry_mapping.h}
// (forwarding headers of those names live in vloam-noted_b200/ros_include/lidar_odometry_mapping/): same class names,
// default constructors, init(std::shared_ptr<VloamTF>&), member functions, argument types and order
// (scan_registration.h:64-81, laser_odometry.h:63-87, laser_mapping.h:72-100, lidar_odometry_mapping.h:45-86), so the
// only caller -- vloam_main_node.cpp:118-124 (construction + init), 143-144 (reset), 186-190 (the three IO calls) --
// compiles unchanged.  tests/cpp/main_node_excerpt.cpp is that caller, verbatim, built against this header.
//
// What the header needs from its environment (a ROS / PCL / Eigen box provides the real ones; this repo's test box has
// none of them and compiles against the minimal stand-ins of tests/cpp/stubs/, which declare exactly the members used):
//   <pcl/point_cloud.h>, <pcl/point_types.h>   pcl::PointCloud<T>{points, Ptr}, pcl::PointXYZ, pcl::PointXYZI
//   <Eigen/Dense>                               Eigen::Quaterniond(w,x,y,z) / x() y() z() w(), Eigen::Vector3d(x,y,z)
//   <tf2/LinearMath/Transform.h>                tf2::Transform / Quaternion / Vector3 (setOrigin, setRotation, inverse, *)
//   <ros/ros.h>                                 ros::param::get (the default parameter source), ROS_BREAK
//   <vloam_tf/vloam_tf.h>                       vloam::VloamTF (fields written by publish(): LO.cpp:612-620, LM.cpp:834-861)
//
// Parameters: the three init() functions read the same global ROS parameters as the reference (SR.cpp:44-54,
// LO.cpp:45-54, LM.cpp:44-45, 99-102, 125-128) through vloam::adapter_param_source(), an injectable getter that defaults
// to ros::param::get; a missing parameter aborts like ROS_BREAK() does (AdapterError).  VLOAM_B200_DEVICE selects the GPU.
//
// Data flow: inside one Engine the feature clouds never leave the device; output() copies them out because the reference's
// callers (and publish()) expect PCL clouds.  input() then has three cases:
//   - its stage's predecessor never ran in this Engine (a stage constructed on its own, with a private Engine from init()):
//     the clouds and pose handed in are uploaded (vloam_b200_laser_odometry_input / vloam_b200_laser_mapping_input), as the
//     reference's input() deep-copies them (LO.cpp:137-148, LM.cpp:178-209);
//   - the shared Engine, `adapter_options().caller_clouds = true`: the clouds are compared in full with a private copy of
//     what output() produced, and the pose with the one it returned; when they are equal the device copy is kept, otherwise
//     the edited input is uploaded (feature clouds with moving objects removed, the mapping stage behind another odometry);
//   - the shared Engine by default: input() ASSERTS that the clouds are the ones output() produced (size + first / last
//     point) and throws on an edited copy, without keeping a copy of its own.
// Clouds are passed to the C ABI as PCL lays them out in memory (stride sizeof(PointType) / 4 floats, intensity at
// offsetof(PointType, intensity)): no host repack for the 16-byte stand-in or real PCL's 32-byte PointXYZI.
// `adapter_options().fetch_clouds = false` skips the copies (poses only); the stages then keep the device path.
//
// publish(): the VloamTF writes are done; ROS topic / tf broadcast plumbing (SR.cpp:516-564, LO.cpp:587-611, 621-657,
// LM.cpp:816-833, 862-920) stays with the caller -- the poses and clouds it would publish are the ones output() returns.
#pragma once
#include <stddef.h>
#include <string.h>
#include <functional>
#include <memory>
#include <stdexcept>
#include <stdlib.h>
#include <string>
#include <utility>
#include <vector>

#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#include <Eigen/Dense>
#include <ros/ros.h>
#include <tf2/LinearMath/Transform.h>
#include <vloam_tf/vloam_tf.h>

#include "vloam_b200.h"

namespace vloam {

typedef pcl::PointXYZI PointType;  // common.h:42

// The reference aborts (ROS_BREAK) on a missing parameter or a bad scan_line; the adapter throws.
struct AdapterError : std::runtime_error { using std::runtime_error::runtime_error; };

// ---- parameters ----------------------------------------------------------------------------------------------
struct AdapterParamSource {  // returns false when the parameter does not exist
  std::function<bool(const std::string&, double&)> get;
};
inline AdapterParamSource& adapter_param_source() {
  static AdapterParamSource s{[](const std::string& name, double& v) -> bool {
    // ros::param::get is typed: try the types the reference's launch files use for these names
    double d; int i; bool b; float f;
    if (ros::param::get(name, d)) { v = d; return true; }
    if (ros::param::get(name, i)) { v = i; return true; }
    if (ros::param::get(name, f)) { v = f; return true; }
    if (ros::param::get(name, b)) { v = b ? 1.0 : 0.0; return true; }
    return false;
  }};
  return s;
}
inline double adapter_param(const char* name) {
  double v = 0;
  if (!adapter_param_source().get(name, v)) throw AdapterError(std::string("missing ROS parameter '") + name + "' (the reference calls ROS_BREAK here)");
  return v;
}
struct AdapterOptions {
  bool fetch_clouds = true;    // output() copies the clouds to the host
  bool caller_clouds = false;  // input() in a shared Engine accepts edited clouds / another odometry pose (uploads them)
};
inline AdapterOptions& adapter_options() { static AdapterOptions o; return o; }

// Eigen's Quaterniond * Vector3d (uv = 2 u x v; v + w uv + u x uv), as the device code evaluates it.  Used only by
// the per-point helpers the reference exposes publicly (TransformToStart, pointAssociateToMap, ...): callers
// outside the pipeline may use them, the pipeline itself transforms whole clouds on the device.
inline void quat_rotate(const double q[4], const double v[3], double o[3]) {
  const double ux = q[0], uy = q[1], uz = q[2], w = q[3];
  double a = uy * v[2] - uz * v[1], b = uz * v[0] - ux * v[2], c = ux * v[1] - uy * v[0];
  a += a; b += b; c += c;
  o[0] = (v[0] + w * a) + (uy * c - uz * b);
  o[1] = (v[1] + w * b) + (uz * a - ux * c);
  o[2] = (v[2] + w * c) + (ux * b - uy * a);
}
inline void quat_inverse(const double q[4], double o[4]) {  // Eigen: conjugate / squaredNorm
  const double n2 = q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3];
  o[0] = -q[0] / n2; o[1] = -q[1] / n2; o[2] = -q[2] / n2; o[3] = q[3] / n2;
}

// ---- the shared context ------------------------------------------------------------------------------------------
// One vloam_b200_ctx per LidarOdometryMapping: in the reference the three stage objects are members of one
// LidarOdometryMapping (lidar_odometry_mapping.h:78-80) and only talk through it.  A stage constructed on its own
// creates a private Engine at init().
class Engine {
public:
  typedef pcl::PointCloud<PointType> Cloud;
  typedef Cloud::Ptr CloudPtr;
  struct Sig { size_t n = 0; float first[4] = {0, 0, 0, 0}, last[4] = {0, 0, 0, 0}; bool valid = false; };

  // reads scan_line, minimum_range, mapping_line_resolution, mapping_plane_resolution, mapping_skip_frame
  Engine() {
    vloam_b200_params p;
    vloam_b200_default_params(&p);
    p.n_scans = (int)adapter_param("scan_line");
    p.minimum_range = (float)adapter_param("minimum_range");
    p.line_res = (float)adapter_param("mapping_line_resolution");
    p.plane_res = (float)adapter_param("mapping_plane_resolution");
    p.mapping_skip_frame = (int)adapter_param("mapping_skip_frame");
    const char* dev = getenv("VLOAM_B200_DEVICE");
    create(p, dev ? atoi(dev) : 0);
  }
  // explicit parameters, e.g. p.reserved = VLOAM_FLAG_DISTORTION | VLOAM_FLAG_TRANSFORM_TO_END for sweeps that are not motion-compensated
  explicit Engine(const vloam_b200_params& p, int device = 0) { create(p, device); }
  ~Engine() { vloam_b200_destroy(ctx_); }
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;
  vloam_b200_ctx* ctx() const { return ctx_; }
  void check(int r) const { if (r < 0) throw AdapterError(vloam_b200_last_error(ctx_)); }

  // device cloud `which` -> *out (allocated when null); remembers its signature for the input() assertions, and under
  // caller_clouds the cloud itself
  void fetch(int which, CloudPtr& out) {
    if (!out) out = CloudPtr(new Cloud());
    const int n = vloam_b200_get_cloud(ctx_, which, nullptr, 0);
    check(n);
    if (which <= VLOAM_CLOUD_LESS_FLAT) produced_sr = true;
    Sig& s = sig_[which];
    s.n = (size_t)n; s.valid = true;
    copy_[which].clear();
    if (!adapter_options().fetch_clouds) { out->points.clear(); s.valid = false; return; }
    buf_.resize((size_t)n * 4);
    if (n) check(vloam_b200_get_cloud(ctx_, which, buf_.data(), n));
    if (adapter_options().caller_clouds) copy_[which] = buf_;
    out->points.resize(n);
    for (int i = 0; i < n; ++i) { PointType p; p.x = buf_[i * 4]; p.y = buf_[i * 4 + 1]; p.z = buf_[i * 4 + 2]; p.intensity = buf_[i * 4 + 3]; out->points[i] = p; }
    out->width = (unsigned)n; out->height = 1; out->is_dense = true;
    if (n) { for (int k = 0; k < 4; ++k) { s.first[k] = buf_[k]; s.last[k] = buf_[(size_t)(n - 1) * 4 + k]; } }
  }
  // input(): the cloud handed in must be the one output() produced from this context (it already lives on the device)
  void expect(int which, const CloudPtr& in, const char* what) const {
    const Sig& s = sig_[which];
    if (!s.valid) return;  // clouds were not fetched (adapter_options) or the producing stage has not run: nothing to compare
    bool same = in && in->points.size() == s.n;
    if (same && s.n) {
      const PointType &a = in->points.front(), &b = in->points.back();
      same = a.x == s.first[0] && a.y == s.first[1] && a.z == s.first[2] && a.intensity == s.first[3] && b.x == s.last[0] && b.y == s.last[1] &&
             b.z == s.last[2] && b.intensity == s.last[3];
    }
    if (!same) throw AdapterError(std::string("input(): ") + what + " is not the cloud the previous stage's output() returned; the CUDA path keeps the clouds on "
                                  "the device and cannot take edited copies (use vloam_b200_debug_set for state injection)");
  }
  // caller_clouds: is `in` bit for bit the cloud output() produced?  (false when it was not fetched: the clouds are uploaded)
  bool same(int which, const CloudPtr& in) const {
    const std::vector<float>& c = copy_[which];
    if (!sig_[which].valid || !in || in->points.size() * 4 != c.size()) return false;
    for (size_t i = 0; i < in->points.size(); ++i) {
      const PointType& p = in->points[i];
      const float v[4] = {p.x, p.y, p.z, p.intensity};
      if (memcmp(v, &c[i * 4], sizeof v) != 0) return false;
    }
    return true;
  }
  int skip_from_device = 0;  // skip_frame as LaserOdometry::output computed it (LO.cpp:668-678)
  double q_wodom[4] = {0, 0, 0, 1}, t_wodom[3] = {0, 0, 0};
  // the predecessor of a stage ran in this Engine: ScanRegistration::output fetched its clouds (also with fetch_clouds = false,
  // when they stay on the device) / LaserOdometry::solveLO ran.  A stage whose predecessor never ran here uploads its input.
  bool produced_sr = false, produced_lo = false;
  // PCL memory as the C ABI reads it
  static const float* points(const CloudPtr& c) { return c && !c->points.empty() ? reinterpret_cast<const float*>(c->points.data()) : nullptr; }
  static int count(const CloudPtr& c) { return c ? (int)c->points.size() : 0; }
  static const int kStride = (int)(sizeof(PointType) / sizeof(float)), kWOffset = (int)(offsetof(PointType, intensity) / sizeof(float));
private:
  void create(const vloam_b200_params& p, int device) {
    const int r = vloam_b200_create(&p, device, &ctx_);
    if (r != VLOAM_OK) throw AdapterError("vloam_b200_create failed (bad scan_line / resolution or no CUDA device): " + std::to_string(r));
  }
  vloam_b200_ctx* ctx_ = nullptr;
  Sig sig_[8];
  std::vector<float> buf_;
  std::vector<float> copy_[8];  // caller_clouds: what fetch() copied out, xyzi
};

// ---- scan_registration.h:64-81 -------------------------------------------------------------------------------------
class ScanRegistration {
public:
  typedef pcl::PointCloud<PointType>::Ptr CloudPtr;
  ScanRegistration() {}
  void attach(const std::shared_ptr<Engine>& e) { e_ = e; }  // adapter-only: share LidarOdometryMapping's context
  void init() {  // SR.cpp:42-92: parameters scan_line / minimum_range (read when the context is created)
    if (!e_) e_ = std::make_shared<Engine>();
    laserCloud = CloudPtr(new pcl::PointCloud<PointType>()); cornerPointsSharp = CloudPtr(new pcl::PointCloud<PointType>());
    cornerPointsLessSharp = CloudPtr(new pcl::PointCloud<PointType>()); surfPointsFlat = CloudPtr(new pcl::PointCloud<PointType>());
    surfPointsLessFlat = CloudPtr(new pcl::PointCloud<PointType>());
  }
  void reset() {}   // SR.cpp:95-104: the device buffers are overwritten by the next input()
  void input(const pcl::PointCloud<pcl::PointXYZ>& laserCloudIn_) {  // SR.cpp:144-513
    need();
    const size_t n = laserCloudIn_.points.size();
    xyz_.resize(n * 3);
    for (size_t i = 0; i < n; ++i) { xyz_[i * 3] = laserCloudIn_.points[i].x; xyz_[i * 3 + 1] = laserCloudIn_.points[i].y; xyz_[i * 3 + 2] = laserCloudIn_.points[i].z; }
    e_->check(vloam_b200_scan_registration(e_->ctx(), xyz_.data(), (int)n, 3));
    fresh_ = true;
  }
  // SR.cpp:107-141: order-preserving removal of points closer than thres
  template <typename PointT>
  void removeClosedPointCloud(const pcl::PointCloud<PointT>& cloud_in, pcl::PointCloud<PointT>& cloud_out, float thres) {
    if (&cloud_in != &cloud_out) cloud_out.points.resize(cloud_in.points.size());
    size_t j = 0;
    for (size_t i = 0; i < cloud_in.points.size(); ++i) {
      if (cloud_in.points[i].x * cloud_in.points[i].x + cloud_in.points[i].y * cloud_in.points[i].y + cloud_in.points[i].z * cloud_in.points[i].z < thres * thres) continue;
      cloud_out.points[j] = cloud_in.points[i];
      j++;
    }
    if (j != cloud_in.points.size()) cloud_out.points.resize(j);
    cloud_out.height = 1; cloud_out.width = static_cast<uint32_t>(j); cloud_out.is_dense = true;
  }
  void publish() {}  // SR.cpp:516-564: ROS topics only
  void output(CloudPtr& laserCloud_, CloudPtr& cornerPointsSharp_, CloudPtr& cornerPointsLessSharp_, CloudPtr& surfPointsFlat_,
              CloudPtr& surfPointsLessFlat_) {  // SR.cpp:566-577: aliases of the internal clouds
    need();
    if (fresh_) {
      e_->fetch(VLOAM_CLOUD_FULL, laserCloud); e_->fetch(VLOAM_CLOUD_SHARP, cornerPointsSharp); e_->fetch(VLOAM_CLOUD_LESS_SHARP, cornerPointsLessSharp);
      e_->fetch(VLOAM_CLOUD_FLAT, surfPointsFlat); e_->fetch(VLOAM_CLOUD_LESS_FLAT, surfPointsLessFlat);
      fresh_ = false;
    }
    laserCloud_ = laserCloud; cornerPointsSharp_ = cornerPointsSharp; cornerPointsLessSharp_ = cornerPointsLessSharp;
    surfPointsFlat_ = surfPointsFlat; surfPointsLessFlat_ = surfPointsLessFlat;
  }
  const std::shared_ptr<Engine>& engine() const { return e_; }
private:
  void need() const { if (!e_) throw AdapterError("ScanRegistration used before init()"); }
  std::shared_ptr<Engine> e_;
  std::vector<float> xyz_;
  bool fresh_ = false;
  CloudPtr laserCloud, cornerPointsSharp, cornerPointsLessSharp, surfPointsFlat, surfPointsLessFlat;
};

// ---- laser_odometry.h:63-87 ----------------------------------------------------------------------------------------
class LaserOdometry {
public:
  typedef pcl::PointCloud<PointType>::Ptr CloudPtr;
  LaserOdometry() {}
  void attach(const std::shared_ptr<Engine>& e) { e_ = e; }
  void init(std::shared_ptr<VloamTF>& vloam_tf_) {  // LO.cpp:41-118
    vloam_tf = vloam_tf_;
    (void)adapter_param("loam_verbose_level");
    detach_VO_LO = adapter_param("detach_VO_LO") != 0.0;
    (void)adapter_param("mapping_skip_frame");
    if (!e_) e_ = std::make_shared<Engine>();
    laserCloudCornerLast = CloudPtr(new pcl::PointCloud<PointType>()); laserCloudSurfLast = CloudPtr(new pcl::PointCloud<PointType>());
    laserCloudFullRes = CloudPtr(new pcl::PointCloud<PointType>());
  }
  // LO.cpp:137-148 deep-copies the five clouds.  In a shared Engine they already live on the device: by default the arguments
  // are checked to be ScanRegistration::output's clouds of this sweep; under caller_clouds an edited set is uploaded.  A stage
  // whose ScanRegistration never ran in its Engine uploads them.
  void input(const CloudPtr& laserCloud_, const CloudPtr& cornerPointsSharp_, const CloudPtr& cornerPointsLessSharp_, const CloudPtr& surfPointsFlat_,
             const CloudPtr& surfPointsLessFlat_) {
    need();
    const CloudPtr* in[5] = {&laserCloud_, &cornerPointsSharp_, &cornerPointsLessSharp_, &surfPointsFlat_, &surfPointsLessFlat_};
    bool upload = !e_->produced_sr;
    if (!upload && adapter_options().caller_clouds)
      for (int w = VLOAM_CLOUD_FULL; w <= VLOAM_CLOUD_LESS_FLAT; ++w) upload = upload || !e_->same(w, *in[w]);
    if (upload) {
      const float* p[5]; int n[5];
      for (int w = 0; w < 5; ++w) { p[w] = Engine::points(*in[w]); n[w] = Engine::count(*in[w]); }
      e_->check(vloam_b200_laser_odometry_input(e_->ctx(), p, n, Engine::kStride, Engine::kWOffset));
      return;
    }
    e_->expect(VLOAM_CLOUD_FULL, laserCloud_, "laserCloud"); e_->expect(VLOAM_CLOUD_SHARP, cornerPointsSharp_, "cornerPointsSharp");
    e_->expect(VLOAM_CLOUD_LESS_SHARP, cornerPointsLessSharp_, "cornerPointsLessSharp"); e_->expect(VLOAM_CLOUD_FLAT, surfPointsFlat_, "surfPointsFlat");
    e_->expect(VLOAM_CLOUD_LESS_FLAT, surfPointsLessFlat_, "surfPointsLessFlat");
  }
  void solveLO() {  // LO.cpp:199-584; detach_VO_LO == false: the VO prior velo_last_VOT_velo_curr overwrites para_q / para_t (LO.cpp:237-250)
    need();
    double pq[4] = {0, 0, 0, 1}, pt[3] = {0, 0, 0};
    const bool prior = !detach_VO_LO && vloam_tf;
    if (prior) {
      const tf2::Quaternion r = vloam_tf->velo_last_VOT_velo_curr.getRotation();
      const tf2::Vector3 o = vloam_tf->velo_last_VOT_velo_curr.getOrigin();
      pq[0] = r.x(); pq[1] = r.y(); pq[2] = r.z(); pq[3] = r.w(); pt[0] = o.x(); pt[1] = o.y(); pt[2] = o.z();
    }
    e_->check(vloam_b200_laser_odometry(e_->ctx(), pq, pt, prior ? 1 : 0, qw_, tw_, ql_, tl_, &skip_));
    e_->produced_lo = true;
    e_->skip_from_device = skip_;
    for (int k = 0; k < 4; ++k) e_->q_wodom[k] = qw_[k];
    for (int k = 0; k < 3; ++k) e_->t_wodom[k] = tw_[k];
    fresh_ = true;
  }
  void publish() {  // the VloamTF writes of LO.cpp:612-620 (the ROS messages around them stay with the caller)
    if (!vloam_tf) return;
    vloam_tf->base_prev_LOT_base_curr.setOrigin(tf2::Vector3(tl_[0], tl_[1], tl_[2]));
    vloam_tf->base_prev_LOT_base_curr.setRotation(tf2::Quaternion(ql_[0], ql_[1], ql_[2], ql_[3]));
    vloam_tf->cam0_curr_LOT_cam0_prev = vloam_tf->base_T_cam0.inverse() * vloam_tf->base_prev_LOT_base_curr.inverse() * vloam_tf->base_T_cam0;
    vloam_tf->world_LOT_base_last.setOrigin(tf2::Vector3(tw_[0], tw_[1], tw_[2]));
    vloam_tf->world_LOT_base_last.setRotation(tf2::Quaternion(qw_[0], qw_[1], qw_[2], qw_[3]));
  }
  void output(Eigen::Quaterniond& q_w_curr_, Eigen::Vector3d& t_w_curr_, CloudPtr& laserCloudCornerLast_, CloudPtr& laserCloudSurfLast_,
              CloudPtr& laserCloudFullRes_, bool& skip_frame) {  // LO.cpp:660-679
    need();
    q_w_curr_ = Eigen::Quaterniond(qw_[3], qw_[0], qw_[1], qw_[2]);
    t_w_curr_ = Eigen::Vector3d(tw_[0], tw_[1], tw_[2]);
    skip_frame = skip_ != 0;
    if (!skip_frame) {  // "no change if skip_frame"
      if (fresh_) {
        e_->fetch(VLOAM_CLOUD_CORNER_LAST, laserCloudCornerLast); e_->fetch(VLOAM_CLOUD_SURF_LAST, laserCloudSurfLast); e_->fetch(VLOAM_CLOUD_FULL_RES, laserCloudFullRes);
        fresh_ = false;
      }
      laserCloudCornerLast_ = laserCloudCornerLast; laserCloudSurfLast_ = laserCloudSurfLast; laserCloudFullRes_ = laserCloudFullRes;
    }
  }
  // LO.cpp:152-173 with DISTORTION == false (s = 1): the point of this sweep in the frame of the sweep's start
  void TransformToStart(PointType const* const pi, PointType* const po) {
    const double v[3] = {pi->x, pi->y, pi->z};
    double r[3]; quat_rotate(ql_, v, r);
    po->x = (float)(r[0] + tl_[0]); po->y = (float)(r[1] + tl_[1]); po->z = (float)(r[2] + tl_[2]); po->intensity = pi->intensity;
  }
  // LO.cpp:176-193: into the frame of the sweep's end (dead in the reference: only called under `if (0)`, LO.cpp:537)
  void TransformToEnd(PointType const* const pi, PointType* const po) {
    PointType un; TransformToStart(pi, &un);
    const double v[3] = {un.x - tl_[0], un.y - tl_[1], un.z - tl_[2]};
    double qi[4], r[3]; quat_inverse(ql_, qi); quat_rotate(qi, v, r);
    po->x = (float)r[0]; po->y = (float)r[1]; po->z = (float)r[2]; po->intensity = (float)(int)pi->intensity;
  }
  const std::shared_ptr<Engine>& engine() const { return e_; }
private:
  void need() const { if (!e_) throw AdapterError("LaserOdometry used before init()"); }
  std::shared_ptr<Engine> e_;
  std::shared_ptr<VloamTF> vloam_tf;
  bool detach_VO_LO = true, fresh_ = false;
  double qw_[4] = {0, 0, 0, 1}, tw_[3] = {0, 0, 0}, ql_[4] = {0, 0, 0, 1}, tl_[3] = {0, 0, 0};
  int skip_ = 0;
  CloudPtr laserCloudCornerLast, laserCloudSurfLast, laserCloudFullRes;
};

// ---- laser_mapping.h:72-100 ------------------------------------------------------------------------------------------
class LaserMapping {
public:
  typedef pcl::PointCloud<PointType>::Ptr CloudPtr;
  LaserMapping() {}
  void attach(const std::shared_ptr<Engine>& e) { e_ = e; }
  void init(std::shared_ptr<VloamTF>& vloam_tf_) {  // LM.cpp:40-129
    vloam_tf = vloam_tf_;
    (void)adapter_param("loam_verbose_level");
    (void)adapter_param("mapping_line_resolution"); (void)adapter_param("mapping_plane_resolution");
    (void)adapter_param("mapping_skip_frame");
    map_pub_number = (int)adapter_param("map_pub_number");
    if (!e_) e_ = std::make_shared<Engine>();
  }
  void reset() { need(); e_->check(vloam_b200_begin_frame(e_->ctx())); }  // LM.cpp:132-136
  // LM.cpp:178-209.  In a shared Engine by default the three clouds must be LaserOdometry::output's (they are on the device
  // already) and the odometry pose the one it returned (the device reads it from the shared context); under caller_clouds
  // anything else is uploaded, and a stage whose LaserOdometry never ran in its Engine always uploads (the reference deep-copies
  // both).  On a skipped frame this call computes the high-frequency pose (LM.cpp:197-201), as solveMapping is not called then.
  void input(const CloudPtr& laserCloudCornerLast_, const CloudPtr& laserCloudSurfLast_, const CloudPtr& laserCloudFullRes_, const Eigen::Quaterniond& q_wodom_curr_,
             const Eigen::Vector3d& t_wodom_curr_, const bool& skip_frame_) {
    need();
    skip_frame = skip_frame_;
    const double q[4] = {q_wodom_curr_.x(), q_wodom_curr_.y(), q_wodom_curr_.z(), q_wodom_curr_.w()}, t[3] = {t_wodom_curr_.x(), t_wodom_curr_.y(), t_wodom_curr_.z()};
    bool upload = !e_->produced_lo;
    if (!upload && adapter_options().caller_clouds) {
      upload = (e_->skip_from_device != 0) != skip_frame || memcmp(q, e_->q_wodom, sizeof q) != 0 || memcmp(t, e_->t_wodom, sizeof t) != 0;
      if (!skip_frame)
        upload = upload || !e_->same(VLOAM_CLOUD_CORNER_LAST, laserCloudCornerLast_) || !e_->same(VLOAM_CLOUD_SURF_LAST, laserCloudSurfLast_) ||
                 !e_->same(VLOAM_CLOUD_FULL_RES, laserCloudFullRes_);
    }
    if (upload) {
      e_->check(vloam_b200_laser_mapping_input(e_->ctx(), Engine::points(laserCloudCornerLast_), Engine::count(laserCloudCornerLast_),
                                               Engine::points(laserCloudSurfLast_), Engine::count(laserCloudSurfLast_), Engine::points(laserCloudFullRes_),
                                               Engine::count(laserCloudFullRes_), Engine::kStride, Engine::kWOffset, q, t, skip_frame ? 1 : 0));
      if (skip_frame) e_->check(vloam_b200_laser_mapping(e_->ctx(), q_, t_));  // consumes the input: the high-frequency pose
      return;
    }
    if ((e_->skip_from_device != 0) != skip_frame) throw AdapterError("input(): skip_frame differs from the one LaserOdometry::output returned");
    for (int k = 0; k < 4; ++k) if (q[k] != e_->q_wodom[k]) throw AdapterError("input(): q_wodom_curr is not the pose LaserOdometry::output returned");
    for (int k = 0; k < 3; ++k) if (t[k] != e_->t_wodom[k]) throw AdapterError("input(): t_wodom_curr is not the pose LaserOdometry::output returned");
    if (!skip_frame) {
      e_->expect(VLOAM_CLOUD_CORNER_LAST, laserCloudCornerLast_, "laserCloudCornerLast"); e_->expect(VLOAM_CLOUD_SURF_LAST, laserCloudSurfLast_, "laserCloudSurfLast");
      e_->expect(VLOAM_CLOUD_FULL_RES, laserCloudFullRes_, "laserCloudFullRes");
    } else {
      e_->check(vloam_b200_laser_mapping(e_->ctx(), q_, t_));  // propagates q_wmap_wodom * odometry only
    }
  }
  void solveMapping() { need(); e_->check(vloam_b200_laser_mapping(e_->ctx(), q_, t_)); frameCount++; }  // LM.cpp:212-814 (frameCount++ at its end)
  void publish() {  // the VloamTF write of LM.cpp:834-861 (mapped pose, or the high-frequency pose on a skipped frame)
    // LM.cpp:884-899: every map_pub_number mapped frames laserCloudMap (all 4851 cubes, corner then surf) is published -- queued
    // on the device here, read with laserCloudMap().  Parity unpinned: the reference is not in this checkout.  Before the first
    // mapped frame, and on skipped frames after a publication, the map is the one already published: nothing is queued again.
    if (e_ && map_pub_number > 0 && frameCount > 0 && frameCount % map_pub_number == 0 && frameCount != publishedAt_) {
      e_->check(vloam_b200_publish_map(e_->ctx()));
      publishedAt_ = frameCount;
    }
    if (!vloam_tf) return;
    vloam_tf->world_MOT_base_last.setOrigin(tf2::Vector3(t_[0], t_[1], t_[2]));
    vloam_tf->world_MOT_base_last.setRotation(tf2::Quaternion(q_[0], q_[1], q_[2], q_[3]));
  }
  // adapter-only accessor: the latest published laserCloudMap (blocks until its assembly is done); false before the first publication
  bool laserCloudMap(CloudPtr& out) {
    need();
    if (publishedAt_ == 0) return false;
    const int n = vloam_b200_get_map(e_->ctx(), nullptr, 0);
    e_->check(n);
    std::vector<float> buf((size_t)n * 4);
    if (n) e_->check(vloam_b200_get_map(e_->ctx(), buf.data(), n));
    if (!out) out = CloudPtr(new pcl::PointCloud<PointType>());
    out->points.resize(n);
    for (int i = 0; i < n; ++i) { PointType p; p.x = buf[i * 4]; p.y = buf[i * 4 + 1]; p.z = buf[i * 4 + 2]; p.intensity = buf[i * 4 + 3]; out->points[i] = p; }
    return true;
  }
  // adapter-only: the two kinds of the latest published laserCloudMap (vloam_b200_get_map_kind), in the form loadMap takes back;
  // false before the first publication
  bool laserCloudMap(CloudPtr& corner, CloudPtr& surf) {
    need();
    if (publishedAt_ == 0) return false;
    CloudPtr* outs[2] = {&corner, &surf};
    for (int k = 0; k < 2; ++k) {
      const int n = vloam_b200_get_map_kind(e_->ctx(), k, nullptr, 0);
      e_->check(n);
      std::vector<float> buf((size_t)n * 4);
      if (n) e_->check(vloam_b200_get_map_kind(e_->ctx(), k, buf.data(), n));
      CloudPtr& out = *outs[k];
      if (!out) out = CloudPtr(new pcl::PointCloud<PointType>());
      out->points.resize(n);
      for (int i = 0; i < n; ++i) { PointType p; p.x = buf[i * 4]; p.y = buf[i * 4 + 1]; p.z = buf[i * 4 + 2]; p.intensity = buf[i * 4 + 3]; out->points[i] = p; }
    }
    return true;
  }
  // adapter-only prior maps (no reference counterpart): replace the map with world-frame clouds (PCL memory passed as it is laid
  // out); returns the points dropped per kind (outside the cube grid or non-finite)
  std::pair<long long, long long> loadMap(const CloudPtr& corner, const CloudPtr& surf) {
    need();
    long long dropped[2] = {0, 0};
    e_->check(vloam_b200_load_map(e_->ctx(), Engine::points(corner), Engine::count(corner), Engine::points(surf), Engine::count(surf), Engine::kStride,
                                  Engine::kWOffset, dropped));
    return std::make_pair(dropped[0], dropped[1]);
  }
  // where the sensor starts in a loaded map: q_wmap_wodom / t_wmap_wodom (LM.cpp:147-151), used from the next solveMapping on
  void setMapPose(const Eigen::Quaterniond& q_wmap_wodom, const Eigen::Vector3d& t_wmap_wodom) {
    need();
    const double q[4] = {q_wmap_wodom.x(), q_wmap_wodom.y(), q_wmap_wodom.z(), q_wmap_wodom.w()}, t[3] = {t_wmap_wodom.x(), t_wmap_wodom.y(), t_wmap_wodom.z()};
    e_->check(vloam_b200_set_map_pose(e_->ctx(), q, t));
  }
  // false: localize against the map without changing it (LM.cpp:741-808 skipped); true (default) maps again
  void setMapUpdate(bool enabled) { need(); e_->check(vloam_b200_set_map_update(e_->ctx(), enabled ? 1 : 0)); }
  // adapter-only relocalization (vloam_b200_relocalize): find the last mapped sweep in the loaded map around the rough pose
  // T_map_sensor = (q_c, t_c) without needing it to be close; with options.apply and a found pose the next solveMapping starts there
  struct RelocOptions {
    double half_xy = 20.0, half_z = 1.0, half_yaw_deg = 180.0, resolution = 1.0, yaw_step_deg = 0.0, max_range = 60.0, min_score = 0.3;
    double exclusion_m = 3.0, exclusion_deg = 10.0;
    int max_points = 2048;
    bool apply = true;
  };
  vloam_b200_reloc_result relocalize(const Eigen::Quaterniond& q_c, const Eigen::Vector3d& t_c) { return relocalize(q_c, t_c, RelocOptions()); }
  vloam_b200_reloc_result relocalize(const Eigen::Quaterniond& q_c, const Eigen::Vector3d& t_c, const RelocOptions& o) {
    need();
    vloam_b200_reloc_params p;
    vloam_b200_default_reloc_params(&p);
    p.q_c[0] = q_c.x(); p.q_c[1] = q_c.y(); p.q_c[2] = q_c.z(); p.q_c[3] = q_c.w();
    p.t_c[0] = t_c.x(); p.t_c[1] = t_c.y(); p.t_c[2] = t_c.z();
    p.half_xy = o.half_xy; p.half_z = o.half_z; p.half_yaw_deg = o.half_yaw_deg; p.resolution = o.resolution; p.yaw_step_deg = o.yaw_step_deg;
    p.max_range = o.max_range; p.min_score = o.min_score; p.exclusion_m = o.exclusion_m; p.exclusion_deg = o.exclusion_deg;
    p.max_points = o.max_points; p.apply = o.apply ? 1 : 0;
    vloam_b200_reloc_result r;
    e_->check(vloam_b200_relocalize(e_->ctx(), &p, &r));
    return r;
  }
  int mappedFrames() const { return frameCount; }
  void output() {}                   // declared in LM.h:93, never defined in the reference
  void output(Eigen::Quaterniond& q_w_curr, Eigen::Vector3d& t_w_curr) const {  // adapter-only accessor of the mapped pose
    q_w_curr = Eigen::Quaterniond(q_[3], q_[0], q_[1], q_[2]); t_w_curr = Eigen::Vector3d(t_[0], t_[1], t_[2]);
  }
  void transformAssociateToMap() {}  // declared in LM.h:87, its definition is commented out in the reference (LM.cpp:138-143)
  void transformUpdate() {}          // LM.cpp:147-151: applied on the device at the end of solveMapping
  // LM.cpp:154-164 / 166-175 with the mapped pose of the last solveMapping
  void pointAssociateToMap(PointType const* const pi, PointType* const po) {
    const double v[3] = {pi->x, pi->y, pi->z};
    double r[3]; quat_rotate(q_, v, r);
    po->x = (float)(r[0] + t_[0]); po->y = (float)(r[1] + t_[1]); po->z = (float)(r[2] + t_[2]); po->intensity = pi->intensity;
  }
  void pointAssociateTobeMapped(PointType const* const pi, PointType* const po) {
    const double v[3] = {pi->x - t_[0], pi->y - t_[1], pi->z - t_[2]};
    double qi[4], r[3]; quat_inverse(q_, qi); quat_rotate(qi, v, r);
    po->x = (float)r[0]; po->y = (float)r[1]; po->z = (float)r[2]; po->intensity = pi->intensity;
  }
  // LM.cpp:901-905: the full-resolution cloud of this sweep in the map frame (computed on the device)
  void registeredFullCloud(CloudPtr& out) {
    need();
    const int n = vloam_b200_register_full_cloud(e_->ctx(), nullptr, 0);
    e_->check(n);
    std::vector<float> buf((size_t)n * 4);
    if (n) e_->check(vloam_b200_register_full_cloud(e_->ctx(), buf.data(), n));
    if (!out) out = CloudPtr(new pcl::PointCloud<PointType>());
    out->points.resize(n);
    for (int i = 0; i < n; ++i) { PointType p; p.x = buf[i * 4]; p.y = buf[i * 4 + 1]; p.z = buf[i * 4 + 2]; p.intensity = buf[i * 4 + 3]; out->points[i] = p; }
  }
  const std::shared_ptr<Engine>& engine() const { return e_; }
private:
  void need() const { if (!e_) throw AdapterError("LaserMapping used before init()"); }
  std::shared_ptr<Engine> e_;
  std::shared_ptr<VloamTF> vloam_tf;
  bool skip_frame = false;
  int map_pub_number = 20;
  int frameCount = 0;       // mapped frames (LM.cpp: incremented at the end of solveMapping)
  int publishedAt_ = 0;     // frameCount of the last queued laserCloudMap (0: none yet)
  double q_[4] = {0, 0, 0, 1}, t_[3] = {0, 0, 0};
};

// ---- lidar_odometry_mapping.h:45-86 / lidar_odometry_mapping.cpp:40-176 ---------------------------------------------------
class LidarOdometryMapping {
public:
  LidarOdometryMapping() {}
  void init(std::shared_ptr<VloamTF>& vloam_tf_) {  // LOM.cpp:40-63
    vloam_tf = vloam_tf_;
    verbose_level = (int)adapter_param("loam_verbose_level");
    std::shared_ptr<Engine> e = std::make_shared<Engine>();  // ONE context for the three stages
    scan_registration.attach(e); laser_odometry.attach(e); laser_mapping.attach(e);
    scan_registration.init();
    laser_odometry.init(vloam_tf);
    laser_mapping.init(vloam_tf);
  }
  void reset() { scan_registration.reset(); laser_mapping.reset(); }  // LOM.cpp:65-71
  void scanRegistrationIO(const pcl::PointCloud<pcl::PointXYZ>& laserCloudIn) {  // LOM.cpp:77-100
    scan_registration.input(laserCloudIn);
    scan_registration.output(laserCloud, cornerPointsSharp, cornerPointsLessSharp, surfPointsFlat, surfPointsLessFlat);
  }
  void laserOdometryIO() {  // LOM.cpp:110-141
    laser_odometry.input(laserCloud, cornerPointsSharp, cornerPointsLessSharp, surfPointsFlat, surfPointsLessFlat);
    laser_odometry.solveLO();
    laser_odometry.publish();
    laser_odometry.output(q_wodom_curr, t_wodom_curr, laserCloudCornerLast, laserCloudSurfLast, laserCloudFullRes, skip_frame);
  }
  void laserMappingIO() {  // LOM.cpp:144-176
    laser_mapping.input(laserCloudCornerLast, laserCloudSurfLast, laserCloudFullRes, q_wodom_curr, t_wodom_curr, skip_frame);
    if (!skip_frame) laser_mapping.solveMapping();
    laser_mapping.publish();
  }
  // adapter-only accessors (the reference keeps these private and publishes them over ROS instead)
  ScanRegistration& scanRegistration() { return scan_registration; }
  LaserOdometry& laserOdometry() { return laser_odometry; }
  LaserMapping& laserMapping() { return laser_mapping; }
private:
  std::shared_ptr<VloamTF> vloam_tf;
  int verbose_level = 0;
  ScanRegistration scan_registration;
  pcl::PointCloud<PointType>::Ptr laserCloud, cornerPointsSharp, cornerPointsLessSharp, surfPointsFlat, surfPointsLessFlat;
  LaserOdometry laser_odometry;
  Eigen::Quaterniond q_wodom_curr, q_w_curr;
  Eigen::Vector3d t_wodom_curr, t_w_curr;
  pcl::PointCloud<PointType>::Ptr laserCloudCornerLast, laserCloudSurfLast, laserCloudFullRes;
  bool skip_frame = false;
  LaserMapping laser_mapping;
};

}  // namespace vloam
