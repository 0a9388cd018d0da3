// map_publish_adapter.cpp -- LidarOdometryMapping of vloam_adapter.hpp driven the way vloam_main_node.cpp drives it, with
// map_pub_number = 20: after every frame the latest published laserCloudMap (LM.cpp:884-899) is read through
// LaserMapping::laserCloudMap; a frame whose publication is new writes its cloud to <out_dir>/map_<frame>.bin (float32 x,y,z,i).
// usage: map_publish_adapter <out_dir> <scan0.bin> [scan1.bin ...]   (float32 x,y,z,r per point, KITTI layout)
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
  // loam_velodyne_VLP_16.launch through an injected parameter source, map_pub_number as shipped (20)
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
    pcl::PointCloud<pcl::PointXYZ> cloud;
    pcl::PointCloud<vloam::PointType>::Ptr map;
    int lastMapped = -1;
    for (int k = 2; k < argc; ++k) {
      read_bin(argv[k], cloud);
      loam.reset();
      loam.scanRegistrationIO(cloud);
      loam.laserOdometryIO();
      loam.laserMappingIO();
      const int mapped = loam.laserMapping().mappedFrames();
      const bool have = loam.laserMapping().laserCloudMap(map);
      const bool fresh = have && mapped % 20 == 0 && mapped != lastMapped;
      printf("frame %d mapped %d published %d points %zu\n", k - 2, mapped, fresh ? 1 : 0, have ? map->size() : (size_t)0);
      if (fresh) {
        lastMapped = mapped;
        const std::string path = std::string(argv[1]) + "/map_" + std::to_string(k - 2) + ".bin";
        FILE* f = fopen(path.c_str(), "wb");
        if (!f) { perror(path.c_str()); return 2; }
        for (const auto& p : map->points) { const float v[4] = {p.x, p.y, p.z, p.intensity}; fwrite(v, sizeof(float), 4, f); }
        fclose(f);
      }
    }
  } catch (const vloam::AdapterError& e) {
    printf("ERROR: %s\n", e.what());
    return 1;
  }
  printf("map publish ok\n");
  return 0;
}
