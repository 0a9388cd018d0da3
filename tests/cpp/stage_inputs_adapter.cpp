// stage_inputs_adapter.cpp -- stage objects of vloam_adapter.hpp that take their input from the caller, as the reference's
// LaserOdometry::input / LaserMapping::input (LO.cpp:137-148, LM.cpp:178-209) deep-copy it.  Three checks, on sweeps read from
// raw float files, each against the shared-engine pipeline or the C ABI, bit for bit:
//   1. a stand-alone LaserMapping (its own Engine from init()) fed from a LidarOdometryMapping's laserOdometry().output(...):
//      mapped poses and registeredFullCloud equal the pipeline's own;
//   2. adapter_options().caller_clouds = true: a point in the MIDDLE of each of the three clouds handed to LaserMapping::input is
//      moved; the input is uploaded, and the mapped pose and registeredFullCloud equal the same edit through the C ABI;
//   3. a stand-alone LaserOdometry fed from a stand-alone ScanRegistration on another Engine: odometry poses equal the pipeline's.
// usage: stage_inputs_adapter <scan0.bin> [scan1.bin ...]   (float32 x,y,z,r per point, KITTI layout)
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <lidar_odometry_mapping/lidar_odometry_mapping.h>

typedef pcl::PointCloud<vloam::PointType>::Ptr CloudPtr;
static int failures = 0;
#define EXPECT(cond, ...) do { if (!(cond)) { printf("FAIL: " __VA_ARGS__); printf("\n"); failures++; } } while (0)

static pcl::PointCloud<pcl::PointXYZ> read_bin(const char* path) {
  pcl::PointCloud<pcl::PointXYZ> c;
  FILE* f = fopen(path, "rb");
  if (!f) { perror(path); exit(2); }
  float v[4];
  while (fread(v, sizeof(float), 4, f) == 4) { pcl::PointXYZ p; p.x = v[0]; p.y = v[1]; p.z = v[2]; c.push_back(p); }
  fclose(f);
  return c;
}
static bool same_cloud(const CloudPtr& a, const CloudPtr& b) {
  return a->points.size() == b->points.size() && (a->points.empty() || memcmp(a->points.data(), b->points.data(), a->points.size() * sizeof(vloam::PointType)) == 0);
}
static bool same_pose(const Eigen::Quaterniond& qa, const Eigen::Vector3d& ta, const Eigen::Quaterniond& qb, const Eigen::Vector3d& tb) {
  const double a[7] = {qa.x(), qa.y(), qa.z(), qa.w(), ta.x(), ta.y(), ta.z()}, b[7] = {qb.x(), qb.y(), qb.z(), qb.w(), tb.x(), tb.y(), tb.z()};
  return memcmp(a, b, sizeof a) == 0;
}
static CloudPtr edited(const CloudPtr& c) {  // a copy with the middle point moved by 0.25 m in x
  CloudPtr e(new pcl::PointCloud<vloam::PointType>(*c));
  if (!e->points.empty()) e->points[e->points.size() / 2].x += 0.25f;
  return e;
}
static std::vector<float> xyzi(const CloudPtr& c) {
  std::vector<float> v;
  for (const auto& p : c->points) { v.push_back(p.x); v.push_back(p.y); v.push_back(p.z); v.push_back(p.intensity); }
  return v;
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  vloam::adapter_param_source().get = [](const std::string& k, double& v) -> bool {
    if (k == "scan_line") v = 16; else if (k == "minimum_range") v = 0.3; else if (k == "mapping_line_resolution") v = 0.2;
    else if (k == "mapping_plane_resolution") v = 0.4; else if (k == "mapping_skip_frame") v = 1; else if (k == "map_pub_number") v = 20;
    else if (k == "loam_verbose_level") v = 0; else if (k == "detach_VO_LO") v = 1; else return false;
    return true;
  };
  try {
    std::shared_ptr<vloam::VloamTF> tf = std::make_shared<vloam::VloamTF>();
    tf->init();
    // ---- 1 and 3: the pipeline, a stand-alone LaserMapping behind its odometry, a stand-alone ScanRegistration -> LaserOdometry
    vloam::LidarOdometryMapping lom;
    lom.init(tf);
    vloam::LaserMapping lmAlone;
    lmAlone.init(tf);
    vloam::ScanRegistration srAlone;
    srAlone.init();
    vloam::LaserOdometry loAlone;
    std::shared_ptr<vloam::VloamTF> noTf;
    loAlone.init(noTf);
    EXPECT(lmAlone.engine() != lom.laserMapping().engine() && loAlone.engine() != srAlone.engine(), "stand-alone stages share an Engine");
    for (int k = 1; k < argc; ++k) {
      const pcl::PointCloud<pcl::PointXYZ> scan = read_bin(argv[k]);
      lom.reset();
      lom.scanRegistrationIO(scan);
      lom.laserOdometryIO();
      Eigen::Quaterniond q; Eigen::Vector3d t; CloudPtr cl, sl, fr; bool skip = false;
      lom.laserOdometry().output(q, t, cl, sl, fr, skip);
      lom.laserMappingIO();
      lmAlone.reset();
      lmAlone.input(cl, sl, fr, q, t, skip);
      if (!skip) lmAlone.solveMapping();
      lmAlone.publish();
      Eigen::Quaterniond qa, qb; Eigen::Vector3d ta, tb;
      lom.laserMapping().output(qa, ta); lmAlone.output(qb, tb);
      EXPECT(same_pose(qa, ta, qb, tb), "frame %d: stand-alone LaserMapping pose differs", k - 1);
      CloudPtr ra, rb;
      lom.laserMapping().registeredFullCloud(ra); lmAlone.registeredFullCloud(rb);
      EXPECT(same_cloud(ra, rb), "frame %d: stand-alone LaserMapping registeredFullCloud differs", k - 1);
      // 3: ScanRegistration and LaserOdometry on two Engines of their own
      CloudPtr full, sharp, lessSharp, flat, lessFlat;
      srAlone.reset();
      srAlone.input(scan);
      srAlone.output(full, sharp, lessSharp, flat, lessFlat);
      loAlone.input(full, sharp, lessSharp, flat, lessFlat);
      loAlone.solveLO();
      Eigen::Quaterniond qo; Eigen::Vector3d to; CloudPtr c2, s2, f2; bool skip2 = false;
      loAlone.output(qo, to, c2, s2, f2, skip2);
      EXPECT(same_pose(q, t, qo, to) && skip == skip2, "frame %d: stand-alone LaserOdometry pose differs", k - 1);
      if (!skip) EXPECT(same_cloud(cl, c2) && same_cloud(sl, s2) && same_cloud(fr, f2), "frame %d: stand-alone LaserOdometry clouds differ", k - 1);
      printf("frame %d mapped %.17g %.17g %.17g\n", k - 1, ta.x(), ta.y(), ta.z());
    }
    // ---- 2: caller_clouds on the shared Engine against the same edit through the C ABI
    vloam::adapter_options().caller_clouds = true;
    {
      std::shared_ptr<vloam::Engine> e = std::make_shared<vloam::Engine>();
      vloam::ScanRegistration sr; vloam::LaserOdometry lo; vloam::LaserMapping lm;
      sr.attach(e); lo.attach(e); lm.attach(e);
      sr.init(); lo.init(tf); lm.init(tf);
      vloam_b200_params p;
      vloam_b200_default_params(&p);
      p.n_scans = 16; p.minimum_range = 0.3f; p.line_res = 0.2f; p.plane_res = 0.4f; p.mapping_skip_frame = 1;
      vloam_b200_ctx* c = nullptr;
      if (vloam_b200_create(&p, 0, &c) != VLOAM_OK) { printf("FAIL: create\n"); return 1; }
      for (int k = 1; k < argc; ++k) {
        const pcl::PointCloud<pcl::PointXYZ> scan = read_bin(argv[k]);
        sr.reset(); lm.reset();
        sr.input(scan);
        CloudPtr full, sharp, lessSharp, flat, lessFlat;
        sr.output(full, sharp, lessSharp, flat, lessFlat);
        lo.input(full, sharp, lessSharp, flat, lessFlat);  // unedited: the device copy is kept
        lo.solveLO();
        Eigen::Quaterniond q; Eigen::Vector3d t; CloudPtr cl, sl, fr; bool skip = false;
        lo.output(q, t, cl, sl, fr, skip);
        const bool edit = k % 2 == 0;
        CloudPtr ecl = edit ? edited(cl) : cl, esl = edit ? edited(sl) : sl, efr = edit ? edited(fr) : fr;
        lm.input(ecl, esl, efr, q, t, skip);
        if (!skip) lm.solveMapping();
        Eigen::Quaterniond qa; Eigen::Vector3d ta;
        lm.output(qa, ta);
        CloudPtr reg;
        lm.registeredFullCloud(reg);
        // the C ABI: own scan registration and odometry, the mapping fed the same (edited) clouds
        std::vector<float> xyz(scan.points.size() * 3);
        for (size_t i = 0; i < scan.points.size(); ++i) { xyz[i * 3] = scan.points[i].x; xyz[i * 3 + 1] = scan.points[i].y; xyz[i * 3 + 2] = scan.points[i].z; }
        double qw[4], tw[3], qm[4], tm[3]; int sk = 0;
        vloam_b200_begin_frame(c);
        vloam_b200_scan_registration(c, xyz.data(), (int)scan.points.size(), 3);
        vloam_b200_laser_odometry(c, nullptr, nullptr, 0, qw, tw, nullptr, nullptr, &sk);
        if (edit) {
          const std::vector<float> a = xyzi(ecl), b = xyzi(esl), f = xyzi(efr);
          vloam_b200_laser_mapping_input(c, a.data(), (int)a.size() / 4, b.data(), (int)b.size() / 4, f.data(), (int)f.size() / 4, 4, 3, qw, tw, sk);
        }
        vloam_b200_laser_mapping(c, qm, tm);
        const int n = vloam_b200_register_full_cloud(c, nullptr, 0);
        std::vector<float> regC((size_t)n * 4);
        if (n > 0) vloam_b200_register_full_cloud(c, regC.data(), n);
        EXPECT(same_pose(qa, ta, Eigen::Quaterniond(qm[3], qm[0], qm[1], qm[2]), Eigen::Vector3d(tm[0], tm[1], tm[2])),
               "frame %d: caller_clouds mapped pose differs from the C ABI", k - 1);
        EXPECT(xyzi(reg) == regC, "frame %d: caller_clouds registeredFullCloud differs from the C ABI", k - 1);
        if (edit && !fr->points.empty()) {  // the edit reached the device: the middle point of the registered cloud moved
          const size_t m = fr->points.size() / 2;
          EXPECT(memcmp(&reg->points[m], &regC[m * 4], 16) == 0, "frame %d: edited point", k - 1);
          vloam::PointType moved;
          lm.pointAssociateToMap(&efr->points[m], &moved);
          EXPECT(reg->points[m].x == moved.x && reg->points[m].y == moved.y && reg->points[m].z == moved.z, "frame %d: the edit was not uploaded", k - 1);
        }
      }
      vloam_b200_destroy(c);
    }
  } catch (const vloam::AdapterError& err) {
    printf("ERROR: %s\n", err.what());
    return 1;
  }
  if (failures) { printf("%d failures\n", failures); return 1; }
  printf("stage inputs ok\n");
  return 0;
}
