// Test aid for tests/test_gpu_stage_inputs.py: LaserOdometry::input (LO.cpp:137-148) on caller features for the CPU oracle.
// Built by the test into a temporary directory against oracle/vloam_oracle.h, and handed the Pipeline* that liboracle.so created:
// it replaces the five ScanRegistration clouds the oracle's next laser_odometry call deep-copies.
#include "vloam_oracle.h"

extern "C" int vloam_oracle_set_sr_features(void* h, const int* n, const float* pts) {
  vo::Pipeline* p = (vo::Pipeline*)h;
  vo::Cloud* dst[5] = {&p->sr.laserCloud, &p->sr.cornerSharp, &p->sr.cornerLessSharp, &p->sr.surfFlat, &p->sr.surfLessFlat};
  const vo::P4* q = (const vo::P4*)pts;
  for (int k = 0; k < 5; ++k) { dst[k]->assign(q, q + n[k]); q += n[k]; }
  return 0;
}
