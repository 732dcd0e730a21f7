// groups_check -- frame groups through the C++ host classes: two cameras registered with Pointcloud::addCamera, four z16 frames
// in groups of 1 and 3 through Pointcloud::processGroups. tests/test_gpu_groups.py runs the same frames through the Python binding
// and compares the lines.
// Usage: groups_check width height   -> 2 lines (one per group) and then the group sizes' status words, one line
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

int main(int argc, char **argv)
{
  const int w = argc > 2 ? std::atoi(argv[1]) : 640, h = argc > 2 ? std::atoi(argv[2]) : 480;
  Window app("groups_check");
  ssd_scene base[2];
  for(int c = 0; c < 2; c++)
  {
    ssd_scene_default(&base[c], w, h);
    base[c].noise_sigma = 0.0025f;
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
  const Pointcloud pc(app, *trans[0], config, 0, 4);
  for(int c = 0; c < 2; c++)
  {
    ssd_gpu_intrinsics intr;
    ssd_scene_intrinsics(&base[c], &intr);
    pc.addCamera(*trans[c], intr);
  }
  const std::vector<int32_t> cameraOfFrame = { 0, 1, 0, 1 }, groupFrames = { 1, 3 };
  std::vector<unsigned> status;
  for(const Stairs &s : pc.processGroups(Camera::DepthFrame(depth.data(), ssd_gpu_intrinsics{}, w, h), 4, cameraOfFrame, groupFrames, &status))
    std::cout << s.serialize() << std::endl;
  std::cout << status.size() << " " << status[0] << " " << status[1] << std::endl;
  delete trans[0];
  delete trans[1];
  return 0;
}
