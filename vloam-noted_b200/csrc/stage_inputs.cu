// stage_inputs.cu -- the odometry and mapping stages fed from the caller: LaserOdometry::input (LO.cpp:137-148) and
// LaserMapping::input (LM.cpp:178-209) deep-copy whatever clouds and pose they are handed.  The clouds come in as
// (stride, w_offset) float records (packed xyzi, pcl::PointXYZI as PCL lays it out, ...) and go to the float4 buffers the
// stages read; the copy moves bits only, so results computed from them are bit-identical to the same points produced on the
// device.  Nothing here runs unless the caller makes an input call.
#include "common.cuh"

struct VlPackJob {
  const float* src[VL_PACK_MAX];
  float4* dst[VL_PACK_MAX];
  int begin[VL_PACK_MAX + 1];  // exclusive prefix of the cloud sizes: record g belongs to cloud s when begin[s] <= g < begin[s + 1]
  int stride, w;
};

// x, y, z at floats 0..2 and the intensity at float w of every `stride`-float record, as 32-bit words (NaN payloads included)
__global__ void __launch_bounds__(256) vl_pack_xyzi(VlPackJob j) {
  VL_PDL_WAIT();
  const int total = j.begin[VL_PACK_MAX];
  for (int g = blockIdx.x * blockDim.x + threadIdx.x; g < total; g += gridDim.x * blockDim.x) {
    // (constant indices only: a dynamic index into the kernel parameters would copy them to a stack frame)
    const float* src = j.src[0]; float4* dst = j.dst[0]; int b = 0;
#pragma unroll
    for (int s = 1; s < VL_PACK_MAX; ++s)
      if (g >= j.begin[s]) { src = j.src[s]; dst = j.dst[s]; b = j.begin[s]; }
    const int i = g - b;
    const unsigned* p = reinterpret_cast<const unsigned*>(src) + (size_t)i * j.stride;
    reinterpret_cast<uint4*>(dst)[i] = make_uint4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + j.w));
  }
}

int vl_pack_clouds(vloam_b200_ctx* c, const VlCloudIn* cl, int k, int stride, int w, bool device) {
  const cudaMemcpyKind kind = device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  bool pinned = false;  // a page-locked host buffer is read by the copy engine after the call: wait for it before returning
  if (!device) {
    for (int s = 0; s < k; ++s) {
      cudaPointerAttributes a;
      if (cl[s].n > 0 && cudaPointerGetAttributes(&a, cl[s].src) == cudaSuccess && a.type == cudaMemoryTypeHost) pinned = true;
      (void)cudaGetLastError();
    }
  }
  if (stride == 4 && w == 3) {  // already float4 records: a plain copy
    for (int s = 0; s < k; ++s)
      if (cl[s].n > 0) VL_CUDA(cudaMemcpyAsync(cl[s].dst, cl[s].src, (size_t)cl[s].n * 16, kind, c->stream));
  } else {
    VlPackJob j = {};
    j.stride = stride; j.w = w;
    size_t floats = 0;
    for (int s = 0; s < k; ++s) floats += (size_t)cl[s].n * stride;
    if (!device) VL_TRY(vl_reserve(c, c->inStage, max(floats, (size_t)1)));
    size_t at = 0;
    for (int s = 0; s < VL_PACK_MAX; ++s) {
      const int n = s < k ? cl[s].n : 0;
      j.begin[s + 1] = j.begin[s] + n;
      if (n == 0) continue;
      j.dst[s] = cl[s].dst;
      if (device) j.src[s] = cl[s].src;
      else {
        j.src[s] = c->inStage.p + at;
        VL_CUDA(cudaMemcpyAsync(c->inStage.p + at, cl[s].src, (size_t)n * stride * sizeof(float), cudaMemcpyHostToDevice, c->stream));
        at += (size_t)n * stride;
      }
    }
    const int total = j.begin[VL_PACK_MAX];
    if (total > 0) {
      VL_BYTES((4.0 * stride + 16.0) * total);
      VL_LAUNCH(vl_pack_xyzi, min(vl_div_up(total, 256), c->num_sms * 4), 256, 0, j);
    }
  }
  VL_CUDA(cudaEventRecord(c->evIn, c->stream));
  if (pinned) VL_CUDA(cudaEventSynchronize(c->evIn));
  VL_CUDA(cudaGetLastError());
  return VLOAM_OK;
}
