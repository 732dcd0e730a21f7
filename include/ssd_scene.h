/*
 * ssd_scene.h -- synthetic input source for tests and benchmarks: procedurally generated staircases seen by a pin-hole
 * L515-like depth camera (optionally with a Brown-Conrady lens) (SURVEY.md 8(d) configs). It stands in for the stubbed RealSense capture
 * (Camera::waitForFrames, camera.cpp:27-60) and for rs2::pointcloud::calculate on the host (pointcloud.cpp:138).
 * NOT part of the product: it lives in its own library (stair_step_detector_b200/lib/libssd_scene.so) so that nothing
 * that only generates input or runs the CPU reference has to load the product library libssd_gpu.so.
 */
#ifndef SSD_SCENE_H_
#define SSD_SCENE_H_

#include "ssd_gpu.h" /* ssd_gpu_intrinsics, SSD_E_* */

#ifdef __cplusplus
extern "C" {
#endif

/* ---- synthetic input source (stands in for the stubbed RealSense capture) ---- */
typedef struct ssd_scene
{
  int32_t width, height;
  float fx, fy, ppx, ppy;      /* pin-hole intrinsics */
  float depth_unit;            /* metres per z16 count (L515: 0.00025) */
  float cam_height;            /* camera height above the calibration plane (m) */
  float cam_pitch_deg;         /* optical axis below horizontal */
  float cam_roll_deg;
  float cam_yaw_deg;
  float cam_x, cam_y;          /* camera foot point in scene coordinates */
  float ground_z;              /* ground plane height */
  int32_t n_steps;
  float riser, tread, width_m; /* step geometry (m) */
  float first_riser_y;         /* y of the first riser */
  float x_center;              /* lateral centre of the flight */
  float top_landing;           /* extra depth of the top tread (m) */
  float noise_sigma;           /* N(0,sigma) along the ray (m) */
  float dropout;               /* probability of a zero-depth pixel */
  int32_t n_holes;             /* rectangular zero-depth holes */
  int32_t n_occluders;         /* boxes floating between camera and stairs */
  int32_t rotate180;           /* camera mounted upside down (README "descending stairs") */
  int32_t randomize_camera;    /* ssd_scene_randomize also jitters the camera pose (needs a per-frame calibration) */
  uint64_t seed;
  int32_t distortion_model;    /* lens (ssd_gpu_distortion, include/ssd_gpu.h): SSD_DISTORTION_NONE = the pin-hole camera */
  float coeffs[5];             /* k1, k2, p1, p2, k3: pixel (u, v) is cast along its deprojected ray */
} ssd_scene;

void ssd_scene_default(ssd_scene *s, int32_t width, int32_t height);
/* Randomise the geometry of frame `index` of a batch (SURVEY.md 8(d) config 3/4/5 distributions). */
void ssd_scene_randomize(ssd_scene *s, const ssd_scene *base, uint64_t base_seed, int64_t index, int min_steps, int max_steps);
/* Three ground points seen by the scene's camera, for ssd_make_transform / the reference ctor. */
void ssd_scene_calibration_points(const ssd_scene *s, double world_pts[9], double camera_pts[9]);
/* z16 depth image of one scene, host. */
int ssd_synth_depth_host(const ssd_scene *s, uint16_t *depth_out);
/* z16 -> vertices (the stubbed rs2::pointcloud::calculate, pointcloud.cpp:138), host. */
int ssd_deproject_host(const ssd_scene *s, const uint16_t *depth, float *xyz_out);
/* intrinsics of a synthetic scene */
void ssd_scene_intrinsics(const ssd_scene *s, ssd_gpu_intrinsics *out);
/* Device version: generate n_frames randomised scenes straight into the memory of CUDA device `device`
 * (xyz_dev: n_frames*W*H*3 floats, depth_dev: n_frames*W*H uint16 or NULL; either may be NULL, not both). Synchronous.
 * Returns 0 or a negative SSD_E_* code. */
int ssd_scene_synth_frames_device(int device, const ssd_scene *base, uint64_t base_seed, int64_t first_index, int n_frames,
                                  int min_steps, int max_steps, float *xyz_dev, uint16_t *depth_dev);


#ifdef __cplusplus
}
#endif
#endif /* SSD_SCENE_H_ */
