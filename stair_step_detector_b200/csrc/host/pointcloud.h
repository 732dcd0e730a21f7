// Host mirror of the reference's pipeline driver (pointcloud.h:32-42, pointcloud.cpp:602-626): same
// constructor and process() signature. The per-frame chain runs as CUDA kernels behind the C ABI; process()
// prints the same result line the reference prints. Added on top (the reference only prints):
// detect() returns the Stairs value, processBatch() runs many independent frames in one call, also frames of several
// cameras (addCamera).
#pragma once
#include "camera.h"
#include "configuration.h"
#include "stairs.h"
#include <memory>
#include <string>
#include <vector>

struct ssd_gpu_ctx;

namespace stairs
{

class Window;
class GeometricTransformation;

class Pointcloud
{
public:
  Pointcloud(const Window &window, const GeometricTransformation &trans);
  // extended: explicit configuration, device ordinal and batch capacity
  Pointcloud(const Window &window, const GeometricTransformation &trans, const Configuration &config, int device = 0, int maxFrames = 1);
  ~Pointcloud();
  Pointcloud(const Pointcloud &) = delete;

  // reference behaviour: one frame, one line on stdout (pointcloud.cpp:625)
  void process(const Camera::DepthFrame &frame) const;

  Stairs detect(const Camera::DepthFrame &frame) const;
  // nFrames frames stored back to back at frames.vertices
  std::vector<Stairs> processBatch(const Camera::DepthFrame &frames, int nFrames, std::vector<unsigned> *status = nullptr) const;
  // Per-frame cameras (ssd_gpu_set_cameras): several Pointcloud instances, one per camera mounting, become one Pointcloud and
  // one call. addCamera registers a camera -- its GeometricTransformation (abi(), abiInverse()) and the intrinsics of its depth
  // stream (deprojection of z16 frames, overlay) -- and returns its index. processBatch with cameraOfFrame processes frame i as a
  // Pointcloud built with camera cameraOfFrame[i]'s transformation would (frames.intrinsics is then unused: every z16 frame is
  // deprojected with its camera's intrinsics).
  int addCamera(const GeometricTransformation &trans, const ssd_gpu_intrinsics &intrinsics) const;
  // the same for a camera with lens distortion (ssd_gpu_set_cameras_ex): its z16 frames and its overlay go through the lens
  int addCamera(const GeometricTransformation &trans, const ssd_gpu_intrinsics &intrinsics, const ssd_gpu_distortion &distortion) const;
  void clearCameras() const;
  int cameraCount() const { return static_cast<int>(_cameras.size()); }
  std::vector<Stairs> processBatch(const Camera::DepthFrame &frames, int nFrames, const std::vector<int32_t> &cameraOfFrame,
                                   std::vector<unsigned> *status = nullptr) const;
  // Frame groups (ssd_gpu_process_groups_*): groupFrames[g] consecutive frames form group g, and each group is detected once from
  // the union of its members' points, every frame through its camera cameraOfFrame[i]. Returns one Stairs per group (in the
  // external world of the group's first member's camera); status: one per group.
  std::vector<Stairs> processGroups(const Camera::DepthFrame &frames, int nFrames, const std::vector<int32_t> &cameraOfFrame,
                                    const std::vector<int32_t> &groupFrames, std::vector<unsigned> *status = nullptr) const;
  // per-pixel segment labels of frame `frame` of the last call (SSD_LABEL_* codes / plateau index)
  std::vector<uint8_t> labels(int frame = 0) const;
  // drawStairStep (reference pointcloud.cpp:583-597): project the corners of every detected step into the camera image
  // (WorldToCamera, then DepthFrame::project with these depth-stream intrinsics). The quadrilaterals the reference
  // hands to drawQuadrilateral are then available per frame after process()/processBatch().
  void enableOverlay(const ssd_gpu_intrinsics &intrinsics) const;
  // ... through a lens (ssd_gpu_set_distortion). The overlay of depth frames (z16 or float) uses the lens of the frame
  // (DepthFrame::distortion), the overlay of vertex frames this one.
  void enableOverlay(const ssd_gpu_intrinsics &intrinsics, const ssd_gpu_distortion &distortion) const;
  std::vector<Quadrilateralf_t> overlay(int frame = 0) const;
  // vertical faces (risers) from the remainder points -- the reference stops at "TODO use remainder to detect vertical faces"
  // (pointcloud.cpp:293); definition: include/ssd_gpu.h, ssd_gpu_riser. One more pass over the points when enabled.
  void enableVerticalFaces(bool enable = true) const;
  std::vector<ssd_gpu_riser> verticalFaces(int frame = 0) const;
  // step labels: per pixel the index of the step whose height its point is averaged into (getPointsInQuadrilateral,
  // pointcloud.cpp:560-572), SSD_STEP_LABEL_NONE elsewhere; definition: include/ssd_gpu.h, ssd_gpu_set_step_labels
  void enableStepLabels(bool enable = true) const;
  std::vector<uint8_t> stepLabels(int frame = 0) const;
  // step surfaces: least-squares plane, tilt, flatness and z extent of the points each step is measured from; definition:
  // include/ssd_gpu.h, ssd_gpu_set_step_surfaces. Enabling them also enables the step labels they are computed from.
  void enableStepSurfaces(bool enable = true) const;
  std::vector<ssd_gpu_step_surface> stepSurfaces(int frame = 0) const;
  ssd_gpu_ctx *context() const { return _ctx; }

private:
  void ensureContext(int width, int height) const;
  void applySettings() const;
  std::vector<Stairs> collect(int nFrames, std::vector<unsigned> *status) const;
  const Window &_window;
  const GeometricTransformation &_transformation;
  mutable Configuration _config;
  int _device = 0, _maxFrames = 1;
  mutable ssd_gpu_ctx *_ctx = nullptr;
  mutable bool _explicitConfig = false;
  mutable bool _overlay = false, _overlayApplied = false;
  mutable bool _risers = false, _risersApplied = false;
  mutable bool _stepLabels = false, _stepLabelsApplied = false;
  mutable bool _stepSurfaces = false, _stepSurfacesApplied = false;
  mutable ssd_gpu_intrinsics _overlayIntrinsics{};
  mutable ssd_gpu_distortion _overlayDistortion{}, _lensApplied{};
  mutable std::vector<ssd_gpu_camera> _cameras;
  mutable std::vector<ssd_gpu_distortion> _cameraDistortions;
  mutable bool _camerasApplied = true;
};

} // namespace stairs
