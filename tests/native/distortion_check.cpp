// distortion_check -- z16 frames of cameras with Brown-Conrady lenses through the C++ host classes: a plain Pointcloud fed
// Camera::DepthFrame(z16, intrinsics, distortion, w, h), then one batched call over cameras registered with
// Pointcloud::addCamera(trans, intrinsics, distortion). tests/test_gpu_distortion.py runs the same frames through the Python
// binding and compares the lines.
// Usage: distortion_check width height   -> 2 lines (plain: BC lens, IBC lens) then 4 lines (camera call, frame f of camera f % 2)
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

// the two lenses of the test (tests/test_gpu_distortion.py: BC, IBC)
static void setLens(ssd_scene &s, int model)
{
  static const float bc[5] = { 0.12f, -0.08f, 0.002f, -0.0015f, 0.03f }, ibc[5] = { -0.11f, 0.06f, -0.0012f, 0.0018f, -0.02f };
  s.distortion_model = model;
  for(int i = 0; i < 5; i++)
    s.coeffs[i] = model == SSD_DISTORTION_BROWN_CONRADY ? bc[i] : ibc[i];
}

int main(int argc, char **argv)
{
  const int w = argc > 2 ? std::atoi(argv[1]) : 640, h = argc > 2 ? std::atoi(argv[2]) : 480;
  Window app("distortion_check");
  ssd_scene base[2];
  for(int c = 0; c < 2; c++)
  {
    ssd_scene_default(&base[c], w, h);
    base[c].noise_sigma = 0.0025f;
    setLens(base[c], c == 0 ? SSD_DISTORTION_BROWN_CONRADY : SSD_DISTORTION_INVERSE_BROWN_CONRADY);
  }
  base[1].cam_pitch_deg += 4.f;
  base[1].fx *= 1.05f;
  GeometricTransformation *trans[2] = { makeTransformation(base[0]), makeTransformation(base[1]) };
  const size_t N = size_t(w) * h;
  std::vector<uint16_t> depth(N * 4);
  for(int f = 0; f < 4; f++)
  {
    ssd_scene sc;
    ssd_scene_randomize(&sc, &base[f % 2], 99, f, 3, 8);
    ssd_synth_depth_host(&sc, depth.data() + N * size_t(f));
  }
  Configuration config(w, h);
  {
    // plain calls: one Pointcloud per camera, the lens comes with the frame
    for(int c = 0; c < 2; c++)
    {
      const Pointcloud pc(app, *trans[c], config, 0, 1);
      ssd_gpu_intrinsics intr;
      const ssd_gpu_distortion lens = lensOf(base[c]);
      ssd_scene_intrinsics(&base[c], &intr);
      std::cout << pc.detect(Camera::DepthFrame(depth.data() + N * size_t(c), intr, lens, w, h)).serialize() << std::endl;
    }
  }
  {
    // one camera call over both cameras
    const Pointcloud pc(app, *trans[0], config, 0, 4);
    for(int c = 0; c < 2; c++)
    {
      ssd_gpu_intrinsics intr;
      const ssd_gpu_distortion lens = lensOf(base[c]);
      ssd_scene_intrinsics(&base[c], &intr);
      pc.addCamera(*trans[c], intr, lens);
    }
    const std::vector<int32_t> cameraOfFrame = { 0, 1, 0, 1 };
    for(const Stairs &s : pc.processBatch(Camera::DepthFrame(depth.data(), ssd_gpu_intrinsics{}, w, h), 4, cameraOfFrame))
      std::cout << s.serialize() << std::endl;
  }
  delete trans[0];
  delete trans[1];
  return 0;
}
