// Stub of the capture boundary (reference camera.h:31-118). The RealSense pipeline is out of scope
// (BASELINE.json north_star: capture stubbed); a DepthFrame here is a view of either
//   - the W x H z16 depth image + depth-stream intrinsics, i.e. what the reference's Camera::DepthFrame wraps
//     (rs2::depth_frame; deprojection as in DepthFrame::deproject, camera.h:99-116, then runs on the GPU), or
//   - W x H packed {x,y,z} float vertices -- what rs2::pointcloud::calculate hands to the reference at
//     pointcloud.cpp:138 --
// in host or device memory.
#pragma once
#include "types.h"
#include "../../../include/ssd_gpu.h"
#include <cstddef>

namespace stairs
{

class Camera
{
public:
  struct DepthFrame
  {
    const float *vertices = nullptr; // width*height*3 floats, row-major pixel order, invalid pixel = (0,0,0)
    const uint16_t *z16 = nullptr;   // width*height depth counts, 0 = invalid
    ssd_gpu_intrinsics intrinsics{}; // of the depth stream (used with z16)
    ssd_gpu_distortion distortion{}; // lens of the depth stream (rs2_intrinsics.model / coeffs; used with z16); zero: pin-hole
    int w = 0, h = 0;
    bool onDevice = false;

    DepthFrame() = default;
    DepthFrame(const float *xyz, int width, int height, bool deviceMemory = false) : vertices(xyz), w(width), h(height), onDevice(deviceMemory) {}
    DepthFrame(const uint16_t *depth, const ssd_gpu_intrinsics &intr, int width, int height, bool deviceMemory = false)
    : z16(depth), intrinsics(intr), w(width), h(height), onDevice(deviceMemory)
    {
    }
    DepthFrame(const uint16_t *depth, const ssd_gpu_intrinsics &intr, const ssd_gpu_distortion &lens, int width, int height,
               bool deviceMemory = false)
    : z16(depth), intrinsics(intr), distortion(lens), w(width), h(height), onDevice(deviceMemory)
    {
    }
    int width() const { return w; }
    int height() const { return h; }
    size_t size() const { return size_t(w) * size_t(h); }
  };
};

} // namespace stairs
