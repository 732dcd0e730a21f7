// detect_stairs_multicamera -- frames of several differently mounted cameras through ONE Pointcloud and one batched call per
// round: each camera is registered with its own GeometricTransformation and depth-stream intrinsics (Pointcloud::addCamera), and
// processBatch takes the camera of every frame. The reference would need one Pointcloud per camera, each fed its own frames.
// Synthetic cameras (the RealSense capture is out of scope): camera 0 the default mounting, camera 1 higher, pitched, rolled and
// yawed with other intrinsics, camera 2 mounted upside down with occluders in front of the stairs. Frame f comes from camera f % 3.
// Usage: detect_stairs_multicamera [width height n_frames]   -> one result line per frame on stdout, in frame order
#include "../stair_step_detector_b200/csrc/host/pointcloud.h"
#include "../stair_step_detector_b200/csrc/host/transformation.h"
#include "../stair_step_detector_b200/csrc/host/window.h"
#include "../include/ssd_scene.h" // synthetic input source (libssd_scene.so), in place of Camera::waitForFrames
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
  const int nFrames = argc > 3 ? std::atoi(argv[3]) : 6;
  const int nCameras = 3;
  Window app("stair-step-detector");

  ssd_scene base[nCameras];
  for(int c = 0; c < nCameras; c++)
  {
    ssd_scene_default(&base[c], w, h);
    base[c].noise_sigma = 0.0025f;
    base[c].dropout = 0.03f;
    base[c].n_holes = 3;
  }
  ssd_scene &b1 = base[1];
  b1.cam_height = (float)(b1.cam_height * 1.1);
  b1.cam_pitch_deg = (float)(b1.cam_pitch_deg + 4.0);
  b1.cam_roll_deg = 2.0f;
  b1.cam_yaw_deg = -3.0f;
  b1.fx = (float)(b1.fx * 1.08);
  b1.fy = (float)(b1.fy * 1.06);
  b1.ppx = (float)(b1.ppx + 7.0);
  b1.ppy = (float)(b1.ppy - 5.0);
  b1.n_occluders = 1;
  ssd_scene &b2 = base[2];
  b2.rotate180 = 1;
  b2.n_occluders = 2;
  b2.cam_roll_deg = -1.5f;
  b2.fx = (float)(b2.fx * 0.95);
  b2.fy = (float)(b2.fy * 0.97);
  b2.ppx = (float)(b2.ppx - 4.0);

  // the Pointcloud's own transformation is camera 0's; every camera, camera 0 included, is registered for the batched call
  std::vector<GeometricTransformation *> trans;
  for(int c = 0; c < nCameras; c++)
    trans.push_back(makeTransformation(base[c]));
  Configuration config(w, h);
  const Pointcloud pointcloud(app, *trans[0], config, 0, nFrames);
  for(int c = 0; c < nCameras; c++)
  {
    ssd_gpu_intrinsics intr;
    ssd_scene_intrinsics(&base[c], &intr);
    pointcloud.addCamera(*trans[size_t(c)], intr);
  }

  // one z16 depth image per frame, back to back, each from its own camera
  std::vector<uint16_t> depth(static_cast<size_t>(w) * h * nFrames);
  std::vector<int32_t> cameraOfFrame(static_cast<size_t>(nFrames));
  for(int f = 0; f < nFrames; f++)
  {
    const int c = f % nCameras;
    ssd_scene sc;
    ssd_scene_randomize(&sc, &base[c], 2027, f, 3, 8);
    sc.rotate180 = base[c].rotate180;
    sc.n_occluders = base[c].n_occluders;
    ssd_synth_depth_host(&sc, depth.data() + size_t(w) * h * size_t(f));
    cameraOfFrame[size_t(f)] = c;
  }
  ssd_gpu_intrinsics unused{}; // camera calls deproject every frame with its camera's intrinsics
  const std::vector<Stairs> stairs = pointcloud.processBatch(Camera::DepthFrame(depth.data(), unused, w, h), nFrames, cameraOfFrame);
  for(const Stairs &s : stairs)
    std::cout << s.serialize() << std::endl;
  for(GeometricTransformation *t : trans)
    delete t;
  return 0;
}
