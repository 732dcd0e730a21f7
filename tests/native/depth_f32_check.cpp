// depth_f32_check -- float depth frames through the C++ host classes: every frame is given once as z16 counts and once as
// float samples (float)count with the same intrinsics, and Pointcloud must print the same line for both. Plain calls (a pin-hole
// camera and a Brown-Conrady lens), one camera call and one group call over both cameras. tests/test_gpu_depth_f32.py compares
// the line pairs.
// Usage: depth_f32_check width height   -> 8 line pairs, each "z16 line" then "float line":
//   2 plain (pin-hole, BC lens), 4 camera call (frame f of camera f % 2), 2 group call (groups of 2 frames)
#include "../../stair_step_detector_b200/csrc/host/pointcloud.h"
#include "../../stair_step_detector_b200/csrc/host/transformation.h"
#include "../../stair_step_detector_b200/csrc/host/window.h"
#include "../../include/ssd_scene.h"
#include <cstdlib>
#include <iostream>
#include <vector>
using namespace stairs;

static GeometricTransformation *makeTransformation(const ssd_scene &s)
{
  double world[9], cam[9];
  ssd_scene_calibration_points(&s, world, cam);
  GeometricTransformation::RefPoints wp, cp;
  for(int i = 0; i < 3; i++)
  {
    wp[size_t(i)] = Point3(world[i * 3], world[i * 3 + 1], world[i * 3 + 2]);
    cp[size_t(i)] = Point3(cam[i * 3], cam[i * 3 + 1], cam[i * 3 + 2]);
  }
  return new GeometricTransformation(wp, cp);
}

static ssd_gpu_distortion lensOf(const ssd_scene &s)
{
  ssd_gpu_distortion d;
  d.model = s.distortion_model;
  for(int i = 0; i < 5; i++)
    d.coeffs[i] = s.coeffs[i];
  return d;
}

static void printPairs(const std::vector<Stairs> &a, const std::vector<Stairs> &b)
{
  for(size_t i = 0; i < a.size(); i++)
    std::cout << a[i].serialize() << "\n" << b[i].serialize() << std::endl;
}

int main(int argc, char **argv)
{
  const int w = argc > 2 ? std::atoi(argv[1]) : 640, h = argc > 2 ? std::atoi(argv[2]) : 480;
  Window app("depth_f32_check");
  ssd_scene base[2];
  for(int c = 0; c < 2; c++)
  {
    ssd_scene_default(&base[c], w, h);
    base[c].noise_sigma = 0.0025f;
  }
  // camera 1: pitched, longer focal length, a Brown-Conrady lens (tests/test_gpu_depth_f32.py: BC)
  static const float bc[5] = { 0.12f, -0.08f, 0.002f, -0.0015f, 0.03f };
  base[1].cam_pitch_deg += 4.f;
  base[1].fx *= 1.05f;
  base[1].distortion_model = SSD_DISTORTION_BROWN_CONRADY;
  for(int i = 0; i < 5; i++)
    base[1].coeffs[i] = bc[i];
  GeometricTransformation *trans[2] = { makeTransformation(base[0]), makeTransformation(base[1]) };
  const size_t N = size_t(w) * h;
  std::vector<uint16_t> depth(N * 4);
  for(int f = 0; f < 4; f++)
  {
    ssd_scene sc;
    ssd_scene_randomize(&sc, &base[f % 2], 77, f, 3, 8);
    ssd_synth_depth_host(&sc, depth.data() + N * size_t(f));
  }
  std::vector<float> depthF32(depth.begin(), depth.end()); // (float)count: exact
  Configuration config(w, h);
  ssd_gpu_intrinsics intr[2];
  ssd_gpu_distortion lens[2];
  for(int c = 0; c < 2; c++)
  {
    ssd_scene_intrinsics(&base[c], &intr[c]);
    lens[c] = lensOf(base[c]);
  }
  {
    // plain calls: one Pointcloud per camera, the lens comes with the frame; z16 and float frames alternate on one context
    for(int c = 0; c < 2; c++)
    {
      const Pointcloud pc(app, *trans[c], config, 0, 1);
      const Stairs a = pc.detect(Camera::DepthFrame(depth.data() + N * size_t(c), intr[c], lens[c], w, h));
      const Stairs b = pc.detect(Camera::DepthFrame(depthF32.data() + N * size_t(c), intr[c], lens[c], w, h));
      printPairs({ a }, { b });
    }
  }
  {
    // one camera call and one group call over both cameras
    const Pointcloud pc(app, *trans[0], config, 0, 4);
    for(int c = 0; c < 2; c++)
      pc.addCamera(*trans[c], intr[c], lens[c]);
    const std::vector<int32_t> cameraOfFrame = { 0, 1, 0, 1 }, groupFrames = { 2, 2 };
    printPairs(pc.processBatch(Camera::DepthFrame(depth.data(), ssd_gpu_intrinsics{}, w, h), 4, cameraOfFrame),
               pc.processBatch(Camera::DepthFrame(depthF32.data(), ssd_gpu_intrinsics{}, w, h), 4, cameraOfFrame));
    printPairs(pc.processGroups(Camera::DepthFrame(depth.data(), ssd_gpu_intrinsics{}, w, h), 4, cameraOfFrame, groupFrames),
               pc.processGroups(Camera::DepthFrame(depthF32.data(), ssd_gpu_intrinsics{}, w, h), 4, cameraOfFrame, groupFrames));
  }
  delete trans[0];
  delete trans[1];
  return 0;
}
