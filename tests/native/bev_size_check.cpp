// bev_size_check -- a BEV size of its own through the C++ host classes: one z16 frame of the default scene through Pointcloud::detect,
// once with Configuration::binaryImage set to bev_width x bev_height and once with it left at 0 (the depth stream's size).
// tests/test_gpu_bev_size.py compares the lines with Detector(bev=(bev_width, bev_height)) and Detector() on the same frame.
// A half-set or negative binaryImage is refused: one line "refused" each for {bev_width, 0} and {-bev_width, -bev_height}.
// Usage: bev_size_check width height bev_width bev_height   -> four lines: with the BEV size, with the default, two refusals
#include "../../stair_step_detector_b200/csrc/host/pointcloud.h"
#include "../../stair_step_detector_b200/csrc/host/transformation.h"
#include "../../stair_step_detector_b200/csrc/host/window.h"
#include "../../include/ssd_scene.h"
#include <cstdlib>
#include <iostream>
#include <stdexcept>
#include <vector>
using namespace stairs;

int main(int argc, char **argv)
{
  if(argc < 5)
    return 2;
  const int w = std::atoi(argv[1]), h = std::atoi(argv[2]), bw = std::atoi(argv[3]), bh = std::atoi(argv[4]);
  Window app("bev_size_check");
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
  for(const bool own : { true, false })
  {
    Configuration config(w, h);
    if(own)
    {
      config.binaryImage.width = bw;
      config.binaryImage.height = bh;
    }
    const Pointcloud pc(app, trans, config);
    std::cout << pc.detect(Camera::DepthFrame(depth.data(), intr, w, h)).serialize() << std::endl;
  }
  for(const Configuration::BinaryImage bad : { Configuration::BinaryImage{ bw, 0 }, Configuration::BinaryImage{ -bw, -bh } })
  {
    Configuration config(w, h);
    config.binaryImage = bad;
    const Pointcloud pc(app, trans, config);
    try
    {
      pc.detect(Camera::DepthFrame(depth.data(), intr, w, h));
      std::cout << "accepted" << std::endl;
    }
    catch(const std::invalid_argument &)
    {
      std::cout << "refused" << std::endl;
    }
  }
  return 0;
}
