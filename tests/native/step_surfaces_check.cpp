// step_surfaces_check -- step surfaces through the C++ host classes: one z16 frame of the default scene through Pointcloud::detect with
// Pointcloud::enableStepSurfaces (which also enables the step labels), the records of Pointcloud::stepSurfaces written raw.
// tests/test_step_surfaces.py compares them with the C getter's for the same frame.
// Usage: step_surfaces_check width height out_path   -> the frame's line; n_steps * sizeof(ssd_gpu_step_surface) bytes into out_path
#include "../../stair_step_detector_b200/csrc/host/pointcloud.h"
#include "../../stair_step_detector_b200/csrc/host/transformation.h"
#include "../../stair_step_detector_b200/csrc/host/window.h"
#include "../../include/ssd_scene.h"
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <vector>
using namespace stairs;

int main(int argc, char **argv)
{
  if(argc < 4)
    return 2;
  const int w = std::atoi(argv[1]), h = std::atoi(argv[2]);
  Window app("step_surfaces_check");
  ssd_scene sc;
  ssd_scene_default(&sc, w, h);
  sc.noise_sigma = 0.0025f;
  double world[9], cam[9];
  ssd_scene_calibration_points(&sc, world, cam);
  GeometricTransformation::RefPoints wp, cp;
  for(int i = 0; i < 3; i++)
  {
    wp[size_t(i)] = Point3(world[i * 3], world[i * 3 + 1], world[i * 3 + 2]);
    cp[size_t(i)] = Point3(cam[i * 3], cam[i * 3 + 1], cam[i * 3 + 2]);
  }
  const GeometricTransformation trans(wp, cp);
  std::vector<uint16_t> depth(size_t(w) * h);
  ssd_synth_depth_host(&sc, depth.data());
  ssd_gpu_intrinsics intr;
  ssd_scene_intrinsics(&sc, &intr);
  Configuration config(w, h);
  const Pointcloud pc(app, trans, config);
  pc.enableStepSurfaces();
  std::cout << pc.detect(Camera::DepthFrame(depth.data(), intr, w, h)).serialize() << std::endl;
  const std::vector<ssd_gpu_step_surface> s = pc.stepSurfaces(0);
  FILE *f = std::fopen(argv[3], "wb");
  if(!f || std::fwrite(s.data(), sizeof(ssd_gpu_step_surface), s.size(), f) != s.size())
    return 1;
  std::fclose(f);
  return 0;
}
