// transform_to_end_adapter.cpp -- the stage classes of vloam_adapter.hpp on one explicit-parameter Engine with
// VLOAM_FLAG_DISTORTION | VLOAM_FLAG_TRANSFORM_TO_END, driven in LidarOdometryMapping's call order (LOM.cpp:77-176).
// Per frame it prints the odometry and mapped poses and writes LaserOdometry::output's laserCloudFullRes -- the end-frame cloud
// that LaserMapping::input checks -- to <out_dir>/full_<frame>.bin (float32 x,y,z,i).
// usage: transform_to_end_adapter <out_dir> <scan0.bin> [scan1.bin ...]   (float32 x,y,z,r per point, KITTI layout)
#include <stdio.h>
#include <stdlib.h>
#include <string>
#include <vector>
#include <lidar_odometry_mapping/lidar_odometry_mapping.h>

static void read_bin(const char* path, pcl::PointCloud<pcl::PointXYZ>& c) {
  c.clear();
  FILE* f = fopen(path, "rb");
  if (!f) { perror(path); exit(2); }
  float v[4];
  while (fread(v, sizeof(float), 4, f) == 4) { pcl::PointXYZ p; p.x = v[0]; p.y = v[1]; p.z = v[2]; c.push_back(p); }
  fclose(f);
}

int main(int argc, char** argv) {
  if (argc < 3) return 2;
  // the ROS parameters the three init() functions read (loam_velodyne_VLP_16.launch); the context itself is created from `p` below
  vloam::adapter_param_source().get = [](const std::string& k, double& v) -> bool {
    if (k == "scan_line") v = 16; else if (k == "minimum_range") v = 0.3; else if (k == "mapping_line_resolution") v = 0.2;
    else if (k == "mapping_plane_resolution") v = 0.4; else if (k == "mapping_skip_frame") v = 1; else if (k == "map_pub_number") v = 20;
    else if (k == "loam_verbose_level") v = 0; else if (k == "detach_VO_LO") v = 1; else return false;
    return true;
  };
  try {
    vloam_b200_params p;  // loam_velodyne_VLP_16.launch, sweeps that are not motion-compensated
    vloam_b200_default_params(&p);
    p.n_scans = 16; p.minimum_range = 0.3f; p.line_res = 0.2f; p.plane_res = 0.4f; p.mapping_skip_frame = 1;
    p.reserved = VLOAM_FLAG_DISTORTION | VLOAM_FLAG_TRANSFORM_TO_END;
    std::shared_ptr<vloam::Engine> e = std::make_shared<vloam::Engine>(p);
    std::shared_ptr<vloam::VloamTF> tf = std::make_shared<vloam::VloamTF>();
    tf->init();
    vloam::ScanRegistration sr; vloam::LaserOdometry lo; vloam::LaserMapping lm;
    sr.attach(e); lo.attach(e); lm.attach(e);
    sr.init(); lo.init(tf); lm.init(tf);
    pcl::PointCloud<pcl::PointXYZ> cloud;
    pcl::PointCloud<vloam::PointType>::Ptr full, sharp, lessSharp, flat, lessFlat, cornerLast, surfLast, fullRes;
    Eigen::Quaterniond q_wodom, q_map; Eigen::Vector3d t_wodom, t_map;
    bool skip = false;
    for (int k = 2; k < argc; ++k) {
      read_bin(argv[k], cloud);
      sr.reset(); lm.reset();
      sr.input(cloud);
      sr.output(full, sharp, lessSharp, flat, lessFlat);
      lo.input(full, sharp, lessSharp, flat, lessFlat);
      lo.solveLO();
      lo.publish();
      lo.output(q_wodom, t_wodom, cornerLast, surfLast, fullRes, skip);
      lm.input(cornerLast, surfLast, fullRes, q_wodom, t_wodom, skip);
      if (!skip) lm.solveMapping();
      lm.publish();
      lm.output(q_map, t_map);
      printf("frame %d odom %.17g %.17g %.17g %.17g %.17g %.17g %.17g mapped %.17g %.17g %.17g %.17g %.17g %.17g %.17g\n", k - 2,
             q_wodom.x(), q_wodom.y(), q_wodom.z(), q_wodom.w(), t_wodom.x(), t_wodom.y(), t_wodom.z(),
             q_map.x(), q_map.y(), q_map.z(), q_map.w(), t_map.x(), t_map.y(), t_map.z());
      const std::string path = std::string(argv[1]) + "/full_" + std::to_string(k - 2) + ".bin";
      FILE* f = fopen(path.c_str(), "wb");
      if (!f) { perror(path.c_str()); return 2; }
      for (const auto& q : fullRes->points) { const float v[4] = {q.x, q.y, q.z, q.intensity}; fwrite(v, sizeof(float), 4, f); }
      fclose(f);
    }
  } catch (const vloam::AdapterError& err) {
    printf("ERROR: %s\n", err.what());
    return 1;
  }
  printf("transform to end ok\n");
  return 0;
}
