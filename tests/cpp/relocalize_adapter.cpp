// relocalize_adapter.cpp -- LidarOdometryMapping of vloam_adapter.hpp restarted inside a saved map: LaserMapping::loadMap from two
// KITTI-style .bin files (float32 x,y,z,i), setMapUpdate(false), one sweep, relocalize from a rough guess, then the per-frame IO calls
// of vloam_main_node.cpp.  Prints the search result and the mapped pose of every frame (%.17g).
// usage: relocalize_adapter <corner.bin> <surf.bin> qx qy qz qw tx ty tz <scan0.bin> [scan1.bin ...]
#include <stdio.h>
#include <stdlib.h>
#include <string>
#include <vector>
#include <lidar_odometry_mapping/lidar_odometry_mapping.h>

static std::vector<float> read_bin(const char* path) {
  std::vector<float> v;
  FILE* f = fopen(path, "rb");
  if (!f) { perror(path); exit(2); }
  float r[4];
  while (fread(r, sizeof(float), 4, f) == 4) v.insert(v.end(), r, r + 4);
  fclose(f);
  return v;
}
static void read_map(const char* path, pcl::PointCloud<vloam::PointType>& c) {
  const std::vector<float> v = read_bin(path);
  for (size_t i = 0; i < v.size(); i += 4) { vloam::PointType p; p.x = v[i]; p.y = v[i + 1]; p.z = v[i + 2]; p.intensity = v[i + 3]; c.push_back(p); }
}
static void read_scan(const char* path, pcl::PointCloud<pcl::PointXYZ>& c) {
  c.clear();
  const std::vector<float> v = read_bin(path);
  for (size_t i = 0; i < v.size(); i += 4) { pcl::PointXYZ p; p.x = v[i]; p.y = v[i + 1]; p.z = v[i + 2]; c.push_back(p); }
}

int main(int argc, char** argv) {
  if (argc < 11) return 2;
  vloam::adapter_param_source().get = [](const std::string& k, double& v) -> bool {
    if (k == "scan_line") v = 16; else if (k == "minimum_range") v = 0.3; else if (k == "mapping_line_resolution") v = 0.2;
    else if (k == "mapping_plane_resolution") v = 0.4; else if (k == "mapping_skip_frame") v = 1; else if (k == "map_pub_number") v = 20;
    else if (k == "loam_verbose_level") v = 0; else if (k == "detach_VO_LO") v = 1; else return false;
    return true;
  };
  try {
    std::shared_ptr<vloam::VloamTF> tf = std::make_shared<vloam::VloamTF>();
    tf->init();
    vloam::LidarOdometryMapping loam;
    loam.init(tf);
    pcl::PointCloud<vloam::PointType>::Ptr corner(new pcl::PointCloud<vloam::PointType>()), surf(new pcl::PointCloud<vloam::PointType>());
    read_map(argv[1], *corner);
    read_map(argv[2], *surf);
    loam.laserMapping().loadMap(corner, surf);
    loam.laserMapping().setMapUpdate(false);
    const Eigen::Quaterniond q_c(atof(argv[6]), atof(argv[3]), atof(argv[4]), atof(argv[5]));
    const Eigen::Vector3d t_c(atof(argv[7]), atof(argv[8]), atof(argv[9]));
    pcl::PointCloud<pcl::PointXYZ> cloud;
    for (int k = 10; k < argc; ++k) {
      read_scan(argv[k], cloud);
      loam.reset();
      loam.scanRegistrationIO(cloud);
      loam.laserOdometryIO();
      loam.laserMappingIO();
      Eigen::Quaterniond q; Eigen::Vector3d t;
      loam.laserMapping().output(q, t);
      printf("pose %.17g %.17g %.17g %.17g %.17g %.17g %.17g\n", q.x(), q.y(), q.z(), q.w(), t.x(), t.y(), t.z());
      if (k == 10) {  // the first sweep's mapped pose is meaningless: relocalize it, and localize from the next sweep on
        vloam::LaserMapping::RelocOptions o;
        o.half_xy = 30.0;
        const vloam_b200_reloc_result r = loam.laserMapping().relocalize(q_c, t_c, o);
        printf("reloc %lld %d %d %d\n", r.index, r.score, r.runner_score, r.found);
      }
    }
  } catch (const vloam::AdapterError& e) {
    printf("ERROR: %s\n", e.what());
    return 1;
  }
  printf("relocalize ok\n");
  return 0;
}
