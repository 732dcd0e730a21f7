// Pointcloud: thin host driver over ssd_gpu_* (replaces reference pointcloud.cpp:602-626; the stage classes of
// its anonymous namespace are the CUDA kernels in ssd_kernels_points.cuh / ssd_kernels_outline.cuh).
#include "pointcloud.h"
#include "transformation.h"
#include "window.h"
#include <cstring>
#include <iostream>
#include <stdexcept>

namespace stairs
{

Pointcloud::Pointcloud(const Window &window, const GeometricTransformation &trans) : _window(window), _transformation(trans) {}

Pointcloud::Pointcloud(const Window &window, const GeometricTransformation &trans, const Configuration &config, int device, int maxFrames)
: _window(window), _transformation(trans), _config(config), _device(device), _maxFrames(maxFrames), _explicitConfig(true)
{
}

Pointcloud::~Pointcloud()
{
  ssd_gpu_destroy(_ctx);
}

void Pointcloud::ensureContext(int width, int height) const
{
  if(_ctx)
  {
    if(_config.streams.depth.width != width || _config.streams.depth.height != height)
      throw std::invalid_argument("Pointcloud: frame size differs from the configured depth stream");
    return;
  }
  if(!_explicitConfig)
    _config = Configuration(width, height); // the reference takes the size from its compile-time Configuration
  else if(_config.streams.depth.width != width || _config.streams.depth.height != height)
    throw std::invalid_argument("Pointcloud: frame size differs from the configured depth stream");
  if(_config.ownBinaryImage() && !(_config.binaryImage.width > 0 && _config.binaryImage.height > 0))
    throw std::invalid_argument("Pointcloud: Configuration::binaryImage needs a positive width and height, or both 0 (the depth stream's size)");
  const ssd_gpu_config cfg = _config.abi();
  const ssd_gpu_transform xf = _transformation.abi();
  if(ssd_gpu_create_bev(&cfg, _config.bevWidth(), _config.bevHeight(), &xf, _device, _maxFrames, &_ctx) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_create: ") + ssd_gpu_last_error(nullptr)); // no CPU fallback
}

void Pointcloud::enableOverlay(const ssd_gpu_intrinsics &intrinsics) const
{
  enableOverlay(intrinsics, ssd_gpu_distortion{});
}

void Pointcloud::enableOverlay(const ssd_gpu_intrinsics &intrinsics, const ssd_gpu_distortion &distortion) const
{
  _overlayIntrinsics = intrinsics;
  _overlayDistortion = distortion;
  _overlay = true;
  _overlayApplied = false;
  _risersApplied = false;
}

std::vector<Quadrilateralf_t> Pointcloud::overlay(int frame) const
{
  if(!_ctx)
    throw std::logic_error("Pointcloud::overlay before any frame was processed");
  ssd_gpu_overlay q[SSD_GPU_MAX_STEPS];
  int n = 0;
  if(ssd_gpu_get_overlay(_ctx, frame, q, SSD_GPU_MAX_STEPS, &n) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_get_overlay: ") + ssd_gpu_last_error(_ctx));
  std::vector<Quadrilateralf_t> out(static_cast<size_t>(n));
  for(int i = 0; i < n; i++)
    for(int c = 0; c < 4; c++)
      out[static_cast<size_t>(i)][static_cast<size_t>(c)] = Point2f{ q[i].px[c][0], q[i].px[c][1] };
  return out;
}

// overlay / vertical faces / step labels / step surfaces / camera table as last requested, once the context exists (the surfaces
// read the step labels: they go off before the labels and on after them)
void Pointcloud::applySettings() const
{
  if(_overlay && !_overlayApplied)
  {
    double aInv[9];
    _transformation.abiInverse(aInv);
    if(ssd_gpu_set_overlay(_ctx, aInv, &_overlayIntrinsics) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_overlay: ") + ssd_gpu_last_error(_ctx));
    _overlayApplied = true;
  }
  if(_risers != _risersApplied)
  {
    if(ssd_gpu_set_vertical_faces(_ctx, _risers ? 1 : 0) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_vertical_faces: ") + ssd_gpu_last_error(_ctx));
    _risersApplied = _risers;
  }
  if(!_stepSurfaces && _stepSurfacesApplied)
  {
    if(ssd_gpu_set_step_surfaces(_ctx, 0) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_step_surfaces: ") + ssd_gpu_last_error(_ctx));
    _stepSurfacesApplied = false;
  }
  if(_stepLabels != _stepLabelsApplied)
  {
    if(ssd_gpu_set_step_labels(_ctx, _stepLabels ? 1 : 0) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_step_labels: ") + ssd_gpu_last_error(_ctx));
    _stepLabelsApplied = _stepLabels;
  }
  if(_stepSurfaces && !_stepSurfacesApplied)
  {
    if(ssd_gpu_set_step_surfaces(_ctx, 1) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_step_surfaces: ") + ssd_gpu_last_error(_ctx));
    _stepSurfacesApplied = true;
  }
  if(!_camerasApplied)
  {
    if(ssd_gpu_set_cameras_ex(_ctx, _cameras.data(), _cameraDistortions.data(), static_cast<int>(_cameras.size())) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_cameras_ex: ") + ssd_gpu_last_error(_ctx));
    _camerasApplied = true;
  }
}

// The entry point for the frames' kind (z16, float or vertices) and memory (host or device): the plain call, the camera call when cam
// is given, the group call of nGroups groups when grp is given as well.
static int processFrames(ssd_gpu_ctx *c, const Camera::DepthFrame &f, int n, const int32_t *cam = nullptr, const int32_t *grp = nullptr, int ng = 0)
{
  const bool dev = f.onDevice;
  if(grp && f.z16)
    return dev ? ssd_gpu_process_depth_groups_device(c, f.z16, cam, grp, ng, 0) : ssd_gpu_process_depth_groups_host(c, f.z16, cam, grp, ng);
  if(grp && f.depthF32)
    return dev ? ssd_gpu_process_depth_f32_groups_device(c, f.depthF32, cam, grp, ng, 0) : ssd_gpu_process_depth_f32_groups_host(c, f.depthF32, cam, grp, ng);
  if(grp)
    return dev ? ssd_gpu_process_groups_device(c, f.vertices, cam, grp, ng, 0) : ssd_gpu_process_groups_host(c, f.vertices, cam, grp, ng);
  if(cam && f.z16)
    return dev ? ssd_gpu_process_depth_cameras_device(c, f.z16, cam, n) : ssd_gpu_process_depth_cameras_host(c, f.z16, cam, n);
  if(cam && f.depthF32)
    return dev ? ssd_gpu_process_depth_f32_cameras_device(c, f.depthF32, cam, n) : ssd_gpu_process_depth_f32_cameras_host(c, f.depthF32, cam, n);
  if(cam)
    return dev ? ssd_gpu_process_cameras_device(c, f.vertices, cam, n) : ssd_gpu_process_cameras_host(c, f.vertices, cam, n);
  if(f.z16)
    return dev ? ssd_gpu_process_depth_device(c, f.z16, &f.intrinsics, n) : ssd_gpu_process_depth_host(c, f.z16, &f.intrinsics, n);
  if(f.depthF32)
    return dev ? ssd_gpu_process_depth_f32_device(c, f.depthF32, &f.intrinsics, n) : ssd_gpu_process_depth_f32_host(c, f.depthF32, &f.intrinsics, n);
  return dev ? ssd_gpu_process_device(c, f.vertices, n) : ssd_gpu_process_host(c, f.vertices, n);
}

std::vector<Stairs> Pointcloud::processBatch(const Camera::DepthFrame &frames, int nFrames, std::vector<unsigned> *status) const
{
  ensureContext(frames.width(), frames.height());
  applySettings();
  // the lens of the plain call: the frame's for depth frames (z16 or float), the overlay's for vertex frames (set only when it
  // changes)
  const ssd_gpu_distortion &lens = frames.isDepth() ? frames.distortion : _overlayDistortion;
  if(memcmp(&lens, &_lensApplied, sizeof(lens)) != 0)
  {
    if(ssd_gpu_set_distortion(_ctx, &lens) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_distortion: ") + ssd_gpu_last_error(_ctx));
    _lensApplied = lens;
  }
  if(processFrames(_ctx, frames, nFrames) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_process: ") + ssd_gpu_last_error(_ctx));
  return collect(nFrames, status);
}

int Pointcloud::addCamera(const GeometricTransformation &trans, const ssd_gpu_intrinsics &intrinsics) const
{
  return addCamera(trans, intrinsics, ssd_gpu_distortion{});
}

int Pointcloud::addCamera(const GeometricTransformation &trans, const ssd_gpu_intrinsics &intrinsics, const ssd_gpu_distortion &distortion) const
{
  ssd_gpu_camera c{};
  c.xf = trans.abi();
  trans.abiInverse(c.a_inv);
  c.intr = intrinsics;
  _cameras.push_back(c);
  _cameraDistortions.push_back(distortion);
  _camerasApplied = false;
  return static_cast<int>(_cameras.size()) - 1;
}

void Pointcloud::clearCameras() const
{
  _cameras.clear();
  _cameraDistortions.clear();
  _camerasApplied = false;
}

std::vector<Stairs> Pointcloud::processBatch(const Camera::DepthFrame &frames, int nFrames, const std::vector<int32_t> &cameraOfFrame,
                                             std::vector<unsigned> *status) const
{
  if(nFrames < 0 || cameraOfFrame.size() != static_cast<size_t>(nFrames))
    throw std::invalid_argument("Pointcloud::processBatch: cameraOfFrame must hold one camera index per frame");
  ensureContext(frames.width(), frames.height());
  applySettings();
  if(processFrames(_ctx, frames, nFrames, cameraOfFrame.data()) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_process_cameras: ") + ssd_gpu_last_error(_ctx));
  return collect(nFrames, status);
}

std::vector<Stairs> Pointcloud::processGroups(const Camera::DepthFrame &frames, int nFrames, const std::vector<int32_t> &cameraOfFrame,
                                              const std::vector<int32_t> &groupFrames, std::vector<unsigned> *status) const
{
  if(nFrames < 0 || cameraOfFrame.size() != static_cast<size_t>(nFrames))
    throw std::invalid_argument("Pointcloud::processGroups: cameraOfFrame must hold one camera index per frame");
  long long total = 0;
  for(int32_t k : groupFrames)
    total += k;
  if(total != nFrames)
    throw std::invalid_argument("Pointcloud::processGroups: groupFrames must add up to nFrames");
  ensureContext(frames.width(), frames.height());
  applySettings();
  const int32_t *grp = groupFrames.data();
  const int nGroups = static_cast<int>(groupFrames.size());
  if(processFrames(_ctx, frames, nFrames, cameraOfFrame.data(), grp, nGroups) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_process_groups: ") + ssd_gpu_last_error(_ctx));
  // every member frame reads its group's result: keep the first member's
  const std::vector<Stairs> all = collect(nFrames, nullptr);
  std::vector<Stairs> out;
  if(status)
    status->clear();
  for(int g = 0, f = 0; g < nGroups; f += grp[g], g++)
  {
    out.push_back(all[static_cast<size_t>(f)]);
    if(status)
    {
      uint32_t st = 0;
      ssd_gpu_get_steps(_ctx, f, nullptr, 0, nullptr, &st);
      status->push_back(st);
    }
  }
  return out;
}

// the Stairs of every frame of the last call
std::vector<Stairs> Pointcloud::collect(int nFrames, std::vector<unsigned> *status) const
{
  std::vector<Stairs> out(static_cast<size_t>(nFrames));
  if(status)
    status->assign(static_cast<size_t>(nFrames), 0u);
  ssd_gpu_step steps[SSD_GPU_MAX_STEPS];
  for(int f = 0; f < nFrames; f++)
  {
    int n = 0;
    uint32_t st = 0;
    ssd_gpu_get_steps(_ctx, f, steps, SSD_GPU_MAX_STEPS, &n, &st);
    if(status)
      (*status)[static_cast<size_t>(f)] = st;
    Stairs &s = out[static_cast<size_t>(f)];
    s.stairSteps.resize(static_cast<size_t>(n));
    for(int i = 0; i < n; i++)
    {
      s.stairSteps[static_cast<size_t>(i)].height = steps[i].height;
      for(int c = 0; c < 4; c++)
        s.stairSteps[static_cast<size_t>(i)].quadrilateral[static_cast<size_t>(c)] = Point2(steps[i].quad[c][0], steps[i].quad[c][1]);
    }
  }
  return out;
}

Stairs Pointcloud::detect(const Camera::DepthFrame &frame) const
{
  return processBatch(frame, 1).front();
}

void Pointcloud::process(const Camera::DepthFrame &frame) const
{
  _window.setViewport(viewportId::depth);
  const Stairs stairs = detect(frame);
  _window.setViewport(viewportId::infrared);
  std::cout << stairs.serialize() << std::endl;
}

void Pointcloud::enableVerticalFaces(bool enable) const
{
  _risers = enable;
}

std::vector<ssd_gpu_riser> Pointcloud::verticalFaces(int frame) const
{
  if(!_ctx)
    throw std::logic_error("Pointcloud::verticalFaces before any frame was processed");
  ssd_gpu_riser r[SSD_GPU_MAX_PLATEAUS];
  int n = 0;
  if(ssd_gpu_get_vertical_faces(_ctx, frame, r, SSD_GPU_MAX_PLATEAUS, &n) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_get_vertical_faces: ") + ssd_gpu_last_error(_ctx));
  return std::vector<ssd_gpu_riser>(r, r + n);
}

void Pointcloud::enableStepLabels(bool enable) const
{
  _stepLabels = enable;
}

std::vector<uint8_t> Pointcloud::stepLabels(int frame) const
{
  if(!_ctx)
    throw std::logic_error("Pointcloud::stepLabels before any frame was processed");
  std::vector<uint8_t> l(static_cast<size_t>(_config.streams.depth.width) * _config.streams.depth.height);
  if(ssd_gpu_get_step_labels(_ctx, frame, l.data()) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_get_step_labels: ") + ssd_gpu_last_error(_ctx));
  return l;
}

void Pointcloud::enableStepSurfaces(bool enable) const
{
  _stepSurfaces = enable;
  if(enable)
    _stepLabels = true;
}

std::vector<ssd_gpu_step_surface> Pointcloud::stepSurfaces(int frame) const
{
  if(!_ctx)
    throw std::logic_error("Pointcloud::stepSurfaces before any frame was processed");
  ssd_gpu_step_surface s[SSD_GPU_MAX_STEPS];
  int n = 0;
  if(ssd_gpu_get_step_surfaces(_ctx, frame, s, SSD_GPU_MAX_STEPS, &n) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_get_step_surfaces: ") + ssd_gpu_last_error(_ctx));
  return std::vector<ssd_gpu_step_surface>(s, s + n);
}

std::vector<uint8_t> Pointcloud::labels(int frame) const
{
  if(!_ctx)
    throw std::logic_error("Pointcloud::labels before any frame was processed");
  std::vector<uint8_t> l(static_cast<size_t>(_config.streams.depth.width) * _config.streams.depth.height);
  if(ssd_gpu_get_labels(_ctx, frame, l.data()) != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_get_labels: ") + ssd_gpu_last_error(_ctx));
  return l;
}

} // namespace stairs
