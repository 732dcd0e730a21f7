// Runtime counterpart of the reference's compile-time struct Configuration (configuration.h:27-52).
// Same member names and default values; the depth stream size is a constructor parameter because the
// batched configurations run at 1024x768 and 4096x3072 as well as the reference's 640x480.
#pragma once
#include "../../../include/ssd_gpu.h"

namespace stairs
{

struct Configuration
{
  struct Streams
  {
    struct Stream
    {
      int width, height, bytesPerPixel;
      bool active;
    };
    Stream depth{ 640, 480, 2, true };
    Stream infrared{ 640, 480, 1, true };
    Stream grayscale{ 960, 540, 2, false };
  } streams;

  struct MeasuringRange
  {
    struct Range
    {
      double min, max;
    };
    Range x{ -0.6, 0.6 };
    Range y{ 0.1, 1.3 };
    Range z{ -0.1, 1.1 };
  } measuringRange;

  double heightInterval = 0.01;
  double minHeightAboveGround = 0.05;
  double minStepDepth = 0.1; // minimum extent in forward (y) direction
  unsigned minPeakPoints = 2000; // absolute histogram floor (reference pointcloud.cpp:251)
  // size of the bird's-eye image the detector works in (ssd_gpu_create_bev); {0, 0} means the depth stream's size, the reference's
  // coupling (Projection2D, pointcloud.cpp:71-76). The outline constants are in BEV pixels: a fixed BEV keeps one detector tuning
  // for depth frames of any resolution. Both sizes are set, or neither: Pointcloud refuses anything else (std::invalid_argument).
  struct BinaryImage
  {
    int width = 0, height = 0;
  } binaryImage;

  Configuration() = default;
  Configuration(int depthWidth, int depthHeight)
  {
    streams.depth.width = streams.infrared.width = depthWidth;
    streams.depth.height = streams.infrared.height = depthHeight;
  }

  bool ownBinaryImage() const { return binaryImage.width != 0 || binaryImage.height != 0; }
  int bevWidth() const { return ownBinaryImage() ? binaryImage.width : streams.depth.width; }
  int bevHeight() const { return ownBinaryImage() ? binaryImage.height : streams.depth.height; }

  ssd_gpu_config abi() const
  {
    ssd_gpu_config c{};
    c.width = streams.depth.width;
    c.height = streams.depth.height;
    c.x_min = measuringRange.x.min;
    c.x_max = measuringRange.x.max;
    c.y_min = measuringRange.y.min;
    c.y_max = measuringRange.y.max;
    c.z_min = measuringRange.z.min;
    c.z_max = measuringRange.z.max;
    c.height_interval = heightInterval;
    c.min_height_above_ground = minHeightAboveGround;
    c.min_step_depth = minStepDepth;
    c.min_peak_points = minPeakPoints;
    return c;
  }
};

} // namespace stairs
