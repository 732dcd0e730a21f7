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
  const ssd_gpu_config cfg = _config.abi();
  const ssd_gpu_transform xf = _transformation.abi();
  if(ssd_gpu_create(&cfg, &xf, _device, _maxFrames, &_ctx) != SSD_OK)
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

// overlay / vertical faces / camera table as last requested, once the context exists
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
  if(!_camerasApplied)
  {
    if(ssd_gpu_set_cameras_ex(_ctx, _cameras.data(), _cameraDistortions.data(), static_cast<int>(_cameras.size())) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_cameras_ex: ") + ssd_gpu_last_error(_ctx));
    _camerasApplied = true;
  }
}

std::vector<Stairs> Pointcloud::processBatch(const Camera::DepthFrame &frames, int nFrames, std::vector<unsigned> *status) const
{
  ensureContext(frames.width(), frames.height());
  applySettings();
  // the lens of the plain call: the frame's for z16 frames, the overlay's for vertex frames (set only when it changes)
  const ssd_gpu_distortion &lens = frames.z16 ? frames.distortion : _overlayDistortion;
  if(memcmp(&lens, &_lensApplied, sizeof(lens)) != 0)
  {
    if(ssd_gpu_set_distortion(_ctx, &lens) != SSD_OK)
      throw std::runtime_error(std::string("ssd_gpu_set_distortion: ") + ssd_gpu_last_error(_ctx));
    _lensApplied = lens;
  }
  int rc;
  if(frames.z16)
    rc = frames.onDevice ? ssd_gpu_process_depth_device(_ctx, frames.z16, &frames.intrinsics, nFrames)
                         : ssd_gpu_process_depth_host(_ctx, frames.z16, &frames.intrinsics, nFrames);
  else
    rc = frames.onDevice ? ssd_gpu_process_device(_ctx, frames.vertices, nFrames) : ssd_gpu_process_host(_ctx, frames.vertices, nFrames);
  if(rc != SSD_OK)
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
  const int32_t *cam = cameraOfFrame.data();
  int rc;
  if(frames.z16)
    rc = frames.onDevice ? ssd_gpu_process_depth_cameras_device(_ctx, frames.z16, cam, nFrames)
                         : ssd_gpu_process_depth_cameras_host(_ctx, frames.z16, cam, nFrames);
  else
    rc = frames.onDevice ? ssd_gpu_process_cameras_device(_ctx, frames.vertices, cam, nFrames)
                         : ssd_gpu_process_cameras_host(_ctx, frames.vertices, cam, nFrames);
  if(rc != SSD_OK)
    throw std::runtime_error(std::string("ssd_gpu_process_cameras: ") + ssd_gpu_last_error(_ctx));
  return collect(nFrames, status);
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
