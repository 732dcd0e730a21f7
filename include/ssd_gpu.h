/*
 * ssd_gpu.h -- C ABI of the B200-native per-frame geometry hot path of stair-step-detector.
 *
 * The reference has no FFI layer; its boundary for this path is the C++ class surface in namespace
 * `stairs` (reference files, relative to the upstream repo root):
 *   Pointcloud::process(const Camera::DepthFrame&)            pointcloud.h:35-36, pointcloud.cpp:608-626
 *   Transformation_<Dim>, CameraToWorld, ToExternalWorld,
 *   GeometricTransformation                                    transformation.h:42-126
 *   Segmentation::detectOutline / detectFrontEdge             segmentation.h:32-58
 *   QuadrilateralTest                                          quadrilateralTest.h:32-36
 *   Stairs, Stairs::StairStep, Stairs::serialize              stairs.h:30-39
 * Every entry point below names the reference interface it replaces. The C++ host classes in
 * stair_step_detector_b200/csrc/host/ keep the reference's names on top of these functions.
 *
 * Conventions: plain pointers and sizes only; every function returns SSD_OK (0) or a negative
 * SSD_E_* code and never throws; ssd_gpu_last_error() gives the text. One ctx per (device, host
 * thread); calls on one ctx are serialised by the caller. There is NO CPU fallback: without a CUDA
 * device ssd_gpu_create() fails with SSD_E_CUDA.
 */
#ifndef SSD_GPU_H_
#define SSD_GPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSD_GPU_ABI_VERSION 3

/* ---- limits ---- */
#define SSD_GPU_MAX_BINS 253      /* height-histogram bins; bin codes are u8, 253..255 reserved */
#define SSD_GPU_MAX_PLATEAUS 32   /* histogram peaks kept per frame */
#define SSD_GPU_MAX_STEPS 32      /* = MAX_PLATEAUS (ground + every valid plateau) */

/* ---- per-point segment label codes (u8), SURVEY.md section 8(d) ---- */
#define SSD_LABEL_REMAINDER 253u    /* inside the measuring range, in no plateau band (pointcloud.cpp:285-291) */
#define SSD_LABEL_OUT_OF_RANGE 254u /* z > 0 but outside the measuring range (pointcloud.cpp:150-165) */
#define SSD_LABEL_INVALID 255u      /* vertex.z <= 0 (pointcloud.cpp:143-146) */
/* 0 .. n_plateaus-1 : index of the plateau (ascending histogram peak) the point belongs to */

/* ---- error codes ---- */
#define SSD_OK 0
#define SSD_E_INVALID_ARG (-1)
#define SSD_E_CUDA (-2)
#define SSD_E_NOMEM (-3)
#define SSD_E_RANGE (-4)
#define SSD_E_STATE (-5)

/* ---- per-frame status bits ---- */
#define SSD_STATUS_NO_STEPS 0x1u             /* no valid plateau: Stairs has zero steps */
#define SSD_STATUS_DEGENERATE_QUAD 0x2u      /* QuadrilateralTest ctor would throw (quadrilateralTest.cpp:287-372);
                                                the reference terminates; here the step is dropped */
#define SSD_STATUS_INVALID_FRONT_EDGE 0x4u   /* ground front edge invalid: all-zero ground step emitted (pointcloud.cpp:546) */
#define SSD_STATUS_EMPTY_MEAN 0x8u           /* a step has no point inside its quadrilateral: height is NaN (pointcloud.cpp:580) */
#define SSD_STATUS_TOO_MANY_PLATEAUS 0x10u   /* more than SSD_GPU_MAX_PLATEAUS peaks; the extra ones were dropped */
#define SSD_STATUS_BEV_OOB 0x20u             /* a BEV pixel fell past the image end (pointcloud.cpp:81,468 has no bounds check) */
#define SSD_STATUS_HMIN_WRAP 0x40u           /* uint16 wrap of heightMin-1 (pointcloud.cpp:324): plateaus came out empty */

/*
 * Replaces struct Configuration (configuration.h:27-52) + ProcessingConfiguration (pointcloud.cpp:99-106).
 * Defaults (ssd_gpu_default_config) are the reference's values except width/height, which are parameters.
 */
typedef struct ssd_gpu_config
{
  int32_t width, height;          /* streams.depth width x height: the FRAME size (ssd_gpu_create_bev: the BEV size is separate) */
  double x_min, x_max;            /* measuringRange.x  (-0.6, 0.6) */
  double y_min, y_max;            /* measuringRange.y  ( 0.1, 1.3) */
  double z_min, z_max;            /* measuringRange.z  (-0.1, 1.1) */
  double height_interval;         /* 0.01 */
  double min_height_above_ground; /* 0.05 */
  double min_step_depth;          /* 0.1 */
  uint32_t min_peak_points;       /* 2000 (pointcloud.cpp:251) */
  uint32_t reserved;
} ssd_gpu_config;

/*
 * The doubles a GeometricTransformation holds (transformation.h:102-126):
 *   a, b        CameraToWorld:  w = a * p + b, row-major 3x3      (transformation.h:59-64)
 *   ext_a/b/z   ToExternalWorld: (x,y) -> ext_a*(x,y)+ext_b, z -> ext_z + z (transformation.cpp:190-194)
 */
typedef struct ssd_gpu_transform
{
  double a[9];
  double b[3];
  double ext_a[4];
  double ext_b[2];
  double ext_z;
} ssd_gpu_transform;

/* Replaces Stairs::StairStep (stairs.h:32-36): external-world height and corners
 * [frontLeft, frontRight, backLeft, backRight] (segmentation.h:44-53). */
typedef struct ssd_gpu_step
{
  double height;
  double quad[4][2];
} ssd_gpu_step;

/* Per-plateau intermediate record (struct Plateau, pointcloud.cpp:259-265) for parity checks. */
typedef struct ssd_gpu_plateau
{
  int32_t height;      /* histogram peak bin */
  int32_t hmin, hmax;  /* height band [hmin,hmax] (pointcloud.cpp:302-316) */
  uint32_t n_points;   /* plateauPoints.size() */
  int32_t valid;       /* Plateau::valid after detectStairSteps */
  int32_t outlined;    /* 1 if detectOutline ran on this plateau (height >= minHeight) */
  uint32_t n_in_quad;  /* points inside quadriWorld2D (getPointsInQuadrilateral) */
  int32_t quad_status; /* 0 ok, 1 QuadrilateralTest ctor would throw, -1 not evaluated */
  double quad_world[4][2]; /* Plateau::quadriWorld2D */
  double mean_z;       /* calcAverageZ over the points in the quadrilateral */
} ssd_gpu_plateau;

/* Per-frame summary. */
typedef struct ssd_gpu_frame_info
{
  uint32_t status;            /* SSD_STATUS_* */
  int32_t n_bins;
  int32_t n_plateaus;         /* K = filtered peaks */
  int32_t ground_index;       /* groundInd, -1 if none (pointcloud.cpp:403-418) */
  int32_t first_valid_index;  /* firstValidInd, -1 if none */
  int32_t n_steps;            /* Stairs::stairSteps.size() */
  uint32_t n_nonzero;         /* vertices with z > 0 */
  uint32_t n_in_range;        /* points inside the measuring range */
} ssd_gpu_frame_info;

typedef struct ssd_gpu_ctx ssd_gpu_ctx;

/* Timing of the last ssd_gpu_process_* call, CUDA events on the ctx stream (milliseconds). */
typedef struct ssd_gpu_timing
{
  float total_ms;    /* first copy / kernel to results resident in pinned host memory */
  float h2d_ms;      /* host-input calls: first to last host->device copy on the copy stream (the copies overlap the kernels
                        of earlier chunks, so this is a span inside total_ms, not a share of it); 0 for device input */
  float reserved0;
  float label_ms;    /* the dominant transform/histogram stage alone (calls made with SSD_FLAG_STAGE_TIMING), else 0 */
  int32_t n_launches;/* kernels launched by the call */
  int32_t reserved;
} ssd_gpu_timing;

/* ---- configuration / lifetime ---- */
void ssd_gpu_default_config(ssd_gpu_config *cfg, int32_t width, int32_t height);
int ssd_gpu_abi_version(void);
int ssd_gpu_device_count(void);

/* Replaces Pointcloud::Pointcloud(const Window&, const GeometricTransformation&) (pointcloud.cpp:602-606):
 * binds the constant transform and configuration, allocates device buffers for up to max_frames frames. */
int ssd_gpu_create(const ssd_gpu_config *cfg, const ssd_gpu_transform *xf, int device, int max_frames, ssd_gpu_ctx **out);
/*
 * A context has two sizes. The FRAME size, cfg->width x cfg->height, is the pixel grid of the input, of the segment labels and
 * step labels, and of the depth deprojection. The BEV size, bev_width x bev_height, is the bird's-eye image the detector works
 * in. The reference ties both to Configuration.streams.depth (pointcloud.cpp:71-76); ssd_gpu_create keeps that coupling and is
 * ssd_gpu_create_bev(cfg, cfg->width, cfg->height, ...). A BEV size of its own keeps one detector tuning (the outline constants
 * are in BEV pixels) for frames of any resolution, and any point grid (a LiDAR range image, an unorganised M x 1 cloud).
 * Everything the reference computes in image pixels uses the BEV size:
 *   x_to_image = bev_width / (x_max - x_min), y_to_image = bev_height / (y_max - y_min),
 *   min_img_y_extent = (int)(min_step_depth * bev_height / (y_max - y_min)),
 *   the column scans, front-edge columns and vertical probes of the outline, the SSD_STATUS_BEV_OOB test, and the images the
 *   single-stage entry points take (ssd_gpu_detect_outline, ssd_gpu_detect_front_edge).
 * What a frame produces: the reference chain run on that frame's points, in pixel order, with the configuration whose image is
 * the BEV size. Equivalently: pack the frame's points in pixel order into k = ceil(N_frame / N_bev) frames of BEV size, the rest
 * filled with invalid points (0,0,0); one frame (k = 1) goes through the plain call, more through one group. The labels of the
 * frame are the first N_frame labels of that packing; n_nonzero and n_in_range are the frame's own. min_peak_points stays
 * absolute (pointcloud.cpp:251). Camera tables, lenses, groups, overlay, risers, step labels and step surfaces all apply; every
 * camera of a context shares its frame size and its BEV size.
 * Limits (each a refusal that creates nothing):
 *   bev_width, bev_height <= 0: SSD_E_INVALID_ARG;
 *   BEV: bev_width / 25 + 4 <= 384 scans, bev_width / 50 + 6 <= 192 line points, bev_height / 10 + 2 <= 512 vertical probes
 *     (bev_width <= 9349, bev_height <= 5109), else SSD_E_RANGE;
 *   frame: N = width * height with N % 16 == 0 (SSD_E_INVALID_ARG) and N <= 9348 * 5108 (SSD_E_RANGE), the largest frame with
 *     the BEV of its own size: it keeps the 32-bit point counters of frame groups exact.
 * Depth input also needs width % 4 == 0 and N * width < 2^40 (the exact row division of the point kernels); a depth call on a
 * frame that breaks either returns SSD_E_INVALID_ARG and leaves the previous results readable.
 */
int ssd_gpu_create_bev(const ssd_gpu_config *cfg, int32_t bev_width, int32_t bev_height, const ssd_gpu_transform *xf, int device,
                       int max_frames, ssd_gpu_ctx **out);
void ssd_gpu_destroy(ssd_gpu_ctx *ctx);
const char *ssd_gpu_last_error(const ssd_gpu_ctx *ctx); /* ctx may be NULL: last create() error */

/* ---- the hot path: replaces Pointcloud::process (pointcloud.cpp:608-626), batched ---- */
/* xyz: n_frames * width*height (the frame size) packed {float x,y,z} vertices (rs2::vertex layout, qvmTraits.h:70-90),
 * row-major pixel order, invalid pixel = (0,0,0). Results stay in the ctx until the next call. */
int ssd_gpu_process_host(ssd_gpu_ctx *ctx, const float *xyz_host, int n_frames);
int ssd_gpu_process_device(ssd_gpu_ctx *ctx, const float *xyz_dev, int n_frames);
/*
 * The same call one step further upstream: the input is the z16 DEPTH FRAME the reference's process() receives
 * (Camera::DepthFrame, camera.h:58-118) and the library performs the deprojection the reference delegates to
 * rs2::pointcloud::calculate (pointcloud.cpp:138), pin-hole model as in rs2_deproject_pixel_to_point /
 * DepthFrame::deproject (camera.h:99-116) unless a lens is set (ssd_gpu_set_distortion, below):
 *     z = depth * depth_unit,  x = z * ((u - ppx) / fx),  y = z * ((v - ppy) / fy),   depth 0 -> invalid vertex (0,0,0)
 * single-rounded f32 operations in exactly this order. 2 bytes per pixel cross PCIe / HBM instead of 12.
 * depth: n_frames * width*height (the frame size) uint16, row-major.
 */
typedef struct ssd_gpu_intrinsics
{
  float fx, fy, ppx, ppy; /* rs2_intrinsics of the depth stream */
  float depth_unit;       /* metres per count (rs2::depth_sensor::get_depth_scale; L515: 0.00025) */
  int32_t reserved[3];
} ssd_gpu_intrinsics;
int ssd_gpu_process_depth_host(ssd_gpu_ctx *ctx, const uint16_t *z16_host, const ssd_gpu_intrinsics *intr, int n_frames);
int ssd_gpu_process_depth_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const ssd_gpu_intrinsics *intr, int n_frames);
/* Deprojection alone: n_frames depth frames (device) -> packed vertices (device), for parity checks; frame size. */
int ssd_gpu_deproject_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const ssd_gpu_intrinsics *intr, int n_frames, float *xyz_dev);

/* Record CUDA events around every kernel of the chain (on the launching streams); read with ssd_gpu_get_stage_times. */
#define SSD_FLAG_STAGE_TIMING 0x2
/* Run every chunk on one stream (no overlap between chunks): with STAGE_TIMING the event brackets are then the kernels' own durations. */
#define SSD_FLAG_SINGLE_STREAM 0x4
int ssd_gpu_process_device_ex(ssd_gpu_ctx *ctx, const float *xyz_dev, int n_frames, int flags);

/*
 * ---- per-frame cameras: frames of many camera mountings (or of a camera whose pose changes) in one batched call ----
 * A context binds one transform at ssd_gpu_create. A camera table adds any number of others: the camera calls below take the
 * camera of each frame, and frame i is processed exactly as a context created with camera camera_of_frame[i]'s transform
 * would process it (labels, histogram, plateaus, steps, overlay, risers: bit for bit). Replaces several Pointcloud instances,
 * one per camera (pointcloud.cpp:602-606), by one call. The configuration (frame size, measuring range) stays per context.
 *   xf     CameraToWorld + ToExternalWorld of the camera; checked as ssd_gpu_create checks its own.
 *   a_inv  WorldToCamera's _aInv (ssd_make_transform_ex): projects the overlay when ssd_gpu_set_overlay has switched it on
 *          (the a_inv / intrinsics given to ssd_gpu_set_overlay still apply to the plain calls only).
 *   intr   deprojection of depth-frame input (fx, fy non-zero, depth_unit > 0 for every camera a depth call uses) and the
 *          overlay's projection; may be all zero for cameras that only see vertex input without overlay.
 * ssd_gpu_set_cameras replaces the table (n_cameras >= 1, no upper limit; n_cameras == 0 frees it) and leaves the results of the last call
 * readable. It derives every camera's parameters and, for depth input, its deprojection tables once, on the host and with one
 * kernel: a call then only uploads camera_of_frame (4 bytes per frame).
 * camera_of_frame: host array of n_frames indices into the table. Checked before anything is launched: a camera call without a
 * table returns SSD_E_STATE, an index outside [0, n_cameras) SSD_E_RANGE, a depth call that uses a camera without valid
 * intrinsics SSD_E_INVALID_ARG; the results of the previous call stay readable.
 * Results are read with the getters above; ssd_gpu_get_stats counts the whole call and reports the largest filter bounds of
 * the cameras it used. A plain ssd_gpu_process_* call keeps using the context's own transform.
 */
typedef struct ssd_gpu_camera
{
  ssd_gpu_transform xf;
  double a_inv[9];
  ssd_gpu_intrinsics intr;
} ssd_gpu_camera;
int ssd_gpu_set_cameras(ssd_gpu_ctx *ctx, const ssd_gpu_camera *cams, int n_cameras);
int ssd_gpu_n_cameras(ssd_gpu_ctx *ctx);
int ssd_gpu_process_cameras_host(ssd_gpu_ctx *ctx, const float *xyz_host, const int32_t *camera_of_frame, int n_frames);
int ssd_gpu_process_cameras_device(ssd_gpu_ctx *ctx, const float *xyz_dev, const int32_t *camera_of_frame, int n_frames);
/* flags: SSD_FLAG_STAGE_TIMING / SSD_FLAG_SINGLE_STREAM as for ssd_gpu_process_device_ex */
int ssd_gpu_process_cameras_device_ex(ssd_gpu_ctx *ctx, const float *xyz_dev, const int32_t *camera_of_frame, int n_frames, int flags);
int ssd_gpu_process_depth_cameras_host(ssd_gpu_ctx *ctx, const uint16_t *z16_host, const int32_t *camera_of_frame, int n_frames);
int ssd_gpu_process_depth_cameras_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const int32_t *camera_of_frame, int n_frames);

/*
 * ---- lens distortion: the two Brown-Conrady models RealSense reports (rs2_distortion values, coeffs in rs2's order) ----
 * Two primitives on normalised coordinates, coefficients [k1, k2, p1, p2, k3]; every operation a single-rounded f32 operation
 * in C's left-to-right order of the expression as written, no FMA contraction:
 *   P(x, y):    r2 = x*x + y*y
 *               f  = 1 + k1*r2 + k2*r2*r2 + k3*r2*r2*r2
 *               x' = x*f + 2*p1*x*y + p2*(r2 + 2*x*x),   y' = y*f + 2*p2*x*y + p1*(r2 + 2*y*y)
 *   P^-1(x0, y0): exactly 10 fixed-point iterations from (x, y) = (x0, y0):
 *               r2 = x*x + y*y,  icd = 1 / (1 + ((k3*r2 + k2)*r2 + k1)*r2)
 *               dx = 2*p1*x*y + p2*(r2 + 2*x*x),  dy = 2*p2*x*y + p1*(r2 + 2*y*y)
 *               x = (x0 - dx)*icd,  y = (y0 - dy)*icd
 *   model                                    deprojection: x0 = (u - ppx)/fx,     overlay projection: x = X/Z, y = Y/Z,
 *                                            y0 = (v - ppy)/fy, then              then
 *   SSD_DISTORTION_NONE (0)                  identity (the pin-hole path)         identity
 *   SSD_DISTORTION_INVERSE_BROWN_CONRADY (2) (x, y) = P(x0, y0)                   (x, y) = P^-1(x, y)
 *   SSD_DISTORTION_BROWN_CONRADY (4)         (x, y) = P^-1(x0, y0)                (x, y) = P(x, y)
 * then z = depth * depth_unit, X = z*x, Y = z*y (deprojection) and u = x*fx + ppx, v = y*fy + ppy (overlay), as above.
 * This follows rsutil.h's rs2_deproject_pixel_to_point / rs2_project_point_to_pixel as published; agreement with a build of the
 * SDK is UNVERIFIED (the SDK is not part of this project's build or tests). A Brown-Conrady lens whose five coefficients are all
 * 0.0f is the pin-hole lens (P and P^-1 are then the identity in f32) and takes the pin-hole path.
 * The other rs2 models (MODIFIED_BROWN_CONRADY 1, FTHETA 3, KANNALA_BRANDT4 5) are rejected with SSD_E_INVALID_ARG; so are a
 * non-finite coefficient and a lens whose deprojection is non-finite at some pixel of the frame (P^-1 diverged).
 *
 * A distorted lens's ray depends on both u and v: the library builds one per-pixel ray table (W*H*8 bytes, 6.3 MB at 1024x768)
 * per distinct lens (intrinsics + distortion, compared bitwise) when the lens is set, and the z16 point kernels read the ray
 * of each pixel from it. Calls whose frames all have pin-hole lenses run exactly as before.
 *
 * ssd_gpu_set_distortion: the lens of the plain calls (ssd_gpu_process_depth_host/_device, ssd_gpu_deproject_device and the
 * plain overlay of ssd_gpu_set_overlay); NULL or SSD_DISTORTION_NONE switches it off. Vertex input is already deprojected:
 * there only the overlay uses it.
 * ssd_gpu_set_cameras_ex: ssd_gpu_set_cameras with one lens per camera (dist: n_cameras entries, NULL = all pin-hole); the lens
 * applies to the camera's depth frames and overlay. ssd_gpu_set_cameras(c, n) is ssd_gpu_set_cameras_ex(c, NULL, n). A rejected
 * lens or table leaves the previous one and the previous results in place.
 */
#define SSD_DISTORTION_NONE 0
#define SSD_DISTORTION_MODIFIED_BROWN_CONRADY 1 /* rejected */
#define SSD_DISTORTION_INVERSE_BROWN_CONRADY 2
#define SSD_DISTORTION_FTHETA 3                 /* rejected */
#define SSD_DISTORTION_BROWN_CONRADY 4
#define SSD_DISTORTION_KANNALA_BRANDT4 5        /* rejected */
typedef struct ssd_gpu_distortion
{
  int32_t model;    /* SSD_DISTORTION_*, rs2_intrinsics.model */
  float coeffs[5];  /* rs2_intrinsics.coeffs: k1, k2, p1, p2, k3 */
} ssd_gpu_distortion;
int ssd_gpu_set_distortion(ssd_gpu_ctx *ctx, const ssd_gpu_distortion *d);
int ssd_gpu_set_cameras_ex(ssd_gpu_ctx *ctx, const ssd_gpu_camera *cams, const ssd_gpu_distortion *dist, int n_cameras);
/* Ray tables the context holds (W*H*8 bytes each): one for the plain calls' distorted lens once a depth call has used it, and
 * one per distinct lens of a camera table with a distorted camera (its pin-hole cameras share one per intrinsics). 0 when every
 * lens is a pin-hole: then no call reads a ray table. */
int ssd_gpu_n_ray_tables(ssd_gpu_ctx *ctx);

/*
 * ---- frame groups: one stair detection from the combined points of several cameras or frames ----
 * A call takes n_groups groups of consecutive frames; group g has group_frames[g] members, 1 <= group_frames[g] <=
 * SSD_GPU_MAX_GROUP_FRAMES. Every frame has a camera index (camera_of_frame, as in the camera calls); a camera table is required.
 *  - Points: member i's vertices go through camera camera_of_frame[i]'s CameraToWorld, as given or deprojected from z16 with that
 *    camera's intrinsics and lens, with the per-point arithmetic of the camera calls. From there on the group is one point cloud:
 *    the union of its members' points.
 *  - Chain: range filter, height index, histogram, peaks, plateau bands, BEV images, outlines, ground / first-valid logic, ground
 *    quadrilateral, points in quadrilateral, mean z and the risers' remainder run once per group, over the union, with the
 *    context's configuration. min_peak_points stays absolute, as in the reference (pointcloud.cpp:251): a caller who fuses k views
 *    may raise it in the configuration; the library does not scale it.
 *  - External world: the group's steps go through the ToExternalWorld of the camera of the group's first member.
 *  - Overlay: when it is on, every member frame gets the group's steps projected into its own camera (a_inv, intrinsics, lens).
 *  - Labels: each member frame's pixels get labels as in the other calls; plateau indices are the group's.
 *  - Getters stay frame-indexed: for any member frame, ssd_gpu_get_steps, _get_frame_info, _get_plateaus, _get_histogram and
 *    _get_vertical_faces return its group's record (frame_info.n_nonzero and n_in_range are the group's totals); _get_labels and
 *    _get_overlay return the frame's own data. ssd_gpu_get_stats counts the whole call.
 *  - A group of one frame gives, bit for bit, what the camera call gives for that frame.
 * Every argument is checked before anything is launched; a rejected call leaves the previous results readable: no camera table
 * SSD_E_STATE; a camera index outside the table, or more frames in all than max_frames, SSD_E_RANGE; n_groups < 1, a NULL array or a
 * group size outside [1, SSD_GPU_MAX_GROUP_FRAMES] SSD_E_INVALID_ARG; a depth call that uses a camera without valid intrinsics
 * SSD_E_INVALID_ARG; misaligned input as in the other calls. flags: SSD_FLAG_STAGE_TIMING, SSD_FLAG_SINGLE_STREAM.
 */
#define SSD_GPU_MAX_GROUP_FRAMES 32
int ssd_gpu_process_groups_host(ssd_gpu_ctx *ctx, const float *xyz_host, const int32_t *camera_of_frame, const int32_t *group_frames,
                                int n_groups);
int ssd_gpu_process_groups_device(ssd_gpu_ctx *ctx, const float *xyz_dev, const int32_t *camera_of_frame, const int32_t *group_frames,
                                  int n_groups, int flags);
int ssd_gpu_process_depth_groups_host(ssd_gpu_ctx *ctx, const uint16_t *z16_host, const int32_t *camera_of_frame, const int32_t *group_frames,
                                      int n_groups);
int ssd_gpu_process_depth_groups_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const int32_t *camera_of_frame, const int32_t *group_frames,
                                        int n_groups, int flags);

/*
 * ---- float depth frames: 32-bit depth images (ROS 32FC1, simulators, stereo matchers, depth networks) ----
 * A float depth frame is width*height float samples, row-major, the layout of a z16 frame. A pixel is deprojected exactly as a
 * z16 pixel, with the sample in place of (float)count:
 *     z = depth * depth_unit,  then X = z * x, Y = z * y     (single-rounded f32 operations, no FMA; (x, y) from the pin-hole
 *                                                              tables or the lens's ray table, as for z16)
 * depth_unit is the same intrinsics field with the same check (> 0): 1.0f for depth in metres (exact), 0.001f for float
 * millimetres. There are no special cases; what follows comes from the z > 0 test and the range filter:
 *  - NaN, -inf, +-0 and negative samples are the invalid pixel (label SSD_LABEL_INVALID, not counted in n_nonzero);
 *  - +inf, and a finite sample whose product with depth_unit overflows, give a vertex with z > 0 and a non-finite world
 *    point: SSD_LABEL_OUT_OF_RANGE, counted in n_nonzero, as the same vertex given as vertex input would be;
 *  - subnormal samples are kept (the library is built without flush-to-zero).
 * So depth_f32[i] = (float)z16[i] with the same intrinsics gives, bit for bit, what the z16 call gives, and any float frame gives
 * what the vertex call gives on the vertices deprojected on the host by the f32 operations above.
 * Each entry point mirrors its z16 counterpart argument for argument, with every check, lens, option and getter of that call.
 * The input must be 16-byte aligned (SSD_E_INVALID_ARG otherwise): the point kernels read 4 pixels per 16-byte load. Host input
 * crosses PCIe at 4 bytes per pixel, through staging buffers of its own.
 */
int ssd_gpu_process_depth_f32_host(ssd_gpu_ctx *ctx, const float *depth_host, const ssd_gpu_intrinsics *intr, int n_frames);
int ssd_gpu_process_depth_f32_device(ssd_gpu_ctx *ctx, const float *depth_dev, const ssd_gpu_intrinsics *intr, int n_frames);
int ssd_gpu_process_depth_f32_cameras_host(ssd_gpu_ctx *ctx, const float *depth_host, const int32_t *camera_of_frame, int n_frames);
int ssd_gpu_process_depth_f32_cameras_device(ssd_gpu_ctx *ctx, const float *depth_dev, const int32_t *camera_of_frame, int n_frames);
int ssd_gpu_process_depth_f32_groups_host(ssd_gpu_ctx *ctx, const float *depth_host, const int32_t *camera_of_frame,
                                          const int32_t *group_frames, int n_groups);
int ssd_gpu_process_depth_f32_groups_device(ssd_gpu_ctx *ctx, const float *depth_dev, const int32_t *camera_of_frame,
                                            const int32_t *group_frames, int n_groups, int flags);

/* ---- results of the last process call ---- */
/* Stairs of one frame: out[0..*n) ; replaces the value printed at pointcloud.cpp:624-625. */
int ssd_gpu_get_steps(ssd_gpu_ctx *ctx, int frame, ssd_gpu_step *out, int cap, int *n, uint32_t *status);
int ssd_gpu_get_frame_info(ssd_gpu_ctx *ctx, int frame, ssd_gpu_frame_info *out);
int ssd_gpu_get_plateaus(ssd_gpu_ctx *ctx, int frame, ssd_gpu_plateau *out, int cap, int *n);
/*
 * Overlay of the detected steps in the camera image: replaces drawStairStep (pointcloud.cpp:583-597) up to the GL
 * call it ends in. Every corner {x, y, averageZ} of a step (the world quadrilateral BEFORE ToExternalWorld) goes
 * through WorldToCamera (transformation.h:90-94, transformation.cpp:185-188 = Transformation_::transformInv,
 * transformation.h:66-69: a_inv * (p - b), Boost.QVM mat*vec order, no FMA), is narrowed to f32 and projected by
 * DepthFrame::project (camera.h:80-97) = rs2_project_point_to_pixel without distortion:
 *     x = X / Z, y = Y / Z, u = x * fx + ppx, v = y * fy + ppy     (single-rounded f32 operations, this order);
 * with a distorted lens (ssd_gpu_set_distortion, or the camera's lens of ssd_gpu_set_cameras_ex) the model's projection is
 * applied to (x, y) before u, v.
 * The result is the Quadrilateralf_t handed to drawQuadrilateral (drawing.h:57), corners in the order of
 * ssd_gpu_step.quad. detectStairs draws every step twice (depth and infrared viewport, pointcloud.cpp:367-368,
 * 388-392) with the same corners; one record per step is kept. A rejected ground front edge ("return{}",
 * pointcloud.cpp:546) projects the all-zero quadrilateral like the reference does.
 * a_inv: the reference's Transformation_<3>::_aInv, row-major (GeometricTransformation::abiInverse() on the host
 * side). intr: depth_unit is not used. Off until set; a_inv == NULL switches it off again.
 */
typedef struct ssd_gpu_overlay
{
  float px[4][2];
} ssd_gpu_overlay;
int ssd_gpu_set_overlay(ssd_gpu_ctx *ctx, const double a_inv[9], const ssd_gpu_intrinsics *intr);
/* out[0..min(*n, cap)): one projected quadrilateral per step of ssd_gpu_get_steps, same order. */
int ssd_gpu_get_overlay(ssd_gpu_ctx *ctx, int frame, ssd_gpu_overlay *out, int cap, int *n);
/*
 * Vertical faces (risers) from the remainder. PlateausExtraction::extractPlateaus (pointcloud.cpp:280-297) collects the
 * remainder -- the in-range points that fall in no plateau band -- and then drops it: "TODO use remainder to detect vertical
 * faces" (:293). The reference therefore defines the point set but no result; this library's definition (restated in
 * oracle/ssd_oracle.c: ssd_oracle_vertical_faces, the checker of the parity tests) is:
 *   riser k (0 <= k < n_plateaus - 1) joins plateau k and plateau k + 1 (plateaus ascend in height). Its points are the
 *   remainder points (label SSD_LABEL_REMAINDER) whose height index h = (uint16)((z - z_min) * heightIntervalReciprocal)
 *   (calcHeights, pointcloud.cpp:175) lies strictly between the two bands: hmax[k] < h < hmin[k + 1].
 *   Footprint: with X = (int64)((x - x_min) * 65536), Y = (int64)((y - y_min) * 65536) of the exact double-precision world
 *   coordinates (CameraToWorld, transformation.h:59-64), x_min/x_max/y_min/y_max are the extremes of X, Y and x_mean/y_mean
 *   their integer sums divided by n_points, mapped back to metres (x = x_min_cfg + X / 65536). Integer sums: the result does
 *   not depend on the order the points are visited in. z_bottom / z_top: the top of the lower band and the bottom of the
 *   upper band, z_min + (hmax[k] + 1) * height_interval and z_min + hmin[k + 1] * height_interval.
 * A riser without points has n_points == 0 and a zero footprint. Off until enabled (one more pass over the remainder points,
 * about an eighth of a frame); enable != 0 switches it on for the following ssd_gpu_process_* calls.
 */
typedef struct ssd_gpu_riser
{
  int32_t lower_plateau, upper_plateau; /* k, k + 1 */
  uint32_t n_points;
  uint32_t pad;
  double x_min, x_max, y_min, y_max;    /* metres, world frame */
  double x_mean, y_mean;
  double z_bottom, z_top;
} ssd_gpu_riser;
int ssd_gpu_set_vertical_faces(ssd_gpu_ctx *ctx, int enable);
/* out[0..min(*n, cap)): *n = max(0, n_plateaus - 1) risers of the frame, ascending. */
int ssd_gpu_get_vertical_faces(ssd_gpu_ctx *ctx, int frame, ssd_gpu_riser *out, int cap, int *n);
/*
 * Step labels: which pixels each step stands on. For frame f of the last call, step_labels[f][i] (u8 per pixel, row-major
 * like the segment labels) is
 *   s (0 <= s < n_steps) when pixel i's point is one of the points whose z step s of ssd_gpu_get_steps(f) averages: the set
 *     StairsDetector::getPointsInQuadrilateral (pointcloud.cpp:560-572) returns for that step and calcAverageZ (:574-581)
 *     averages, decided on the exact double-precision world point (CameraToWorld, QuadrilateralTest::isPointWithin). For a
 *     plateau step (calcStairStep, :549-558) the points of that plateau inside its quadrilateral; for the ground step
 *     (calcGround, :528-547) the points of the ground plateau inside the ground quadrilateral (calcGroundQuadrilateral) --
 *     also when the front edge is invalid and the step is the all-zero one (SSD_STATUS_INVALID_FRONT_EDGE): the reference
 *     computes the set either way, and the status bit says that the step's corners are not usable;
 *   SSD_STEP_LABEL_NONE for every other pixel: frames without steps, plateaus dropped as SSD_STATUS_DEGENERATE_QUAD, the
 *     points of a plateau outside its quadrilateral, invalid, out-of-range and remainder pixels.
 * So count(step_labels == s) is n_in_quad of the step's plateau, step_labels == s implies that the pixel's segment label is
 * that plateau, and a step with SSD_STATUS_EMPTY_MEAN has no pixels. In group calls each member frame's step labels index its
 * group's steps, its pixels tested through its own camera (as its segment labels index the group's plateaus).
 * Off until enabled; enable != 0 applies to the following ssd_gpu_process_* calls (every entry point) and allocates
 * max_frames * width*height bytes (SSD_E_NOMEM, and the option stays off, when that fails); enable == 0 frees them. The
 * getters return SSD_E_STATE when the option is off or the last call ran without it, SSD_E_RANGE for a frame outside the
 * last call. With the option off nothing changes: the same kernels, launches and results.
 */
#define SSD_STEP_LABEL_NONE 255u
int ssd_gpu_set_step_labels(ssd_gpu_ctx *ctx, int enable);
/* device -> host copy of frame's width*height step labels (the frame size) */
int ssd_gpu_get_step_labels(ssd_gpu_ctx *ctx, int frame, uint8_t *out_host);
/* Device pointer to the step labels of the last call (n_frames * width*height bytes, the frame size). */
int ssd_gpu_step_labels_device_ptr(ssd_gpu_ctx *ctx, const uint8_t **out);
/*
 * Step surfaces: what the point set behind each step's height looks like -- a level tread, a ramp, a tread with something on
 * it, or a floor seen through a tilted calibration. For step s of frame f of the last call, the points are the pixels with
 * step_labels == s (in a group call: of every member frame of the group), each taken as its exact double-precision world
 * point (wx, wy, wz) through the frame's own camera (CameraToWorld, as ssd_gpu_camera_to_world). Definition (restated in
 * tests/native/oracle_step_surfaces.c: ssd_oracle_step_surfaces):
 *   fixed point: X = (int64)((wx - x_min) * 65536), Y = (int64)((wy - y_min) * 65536), Z = (int64)((wz - z_min) * 65536) with
 *     the configuration's range bounds (>= 0: the points are in range);
 *   exact integer moments n, Sx, Sy, Sz, Sxx, Sxy, Syy, Sxz, Syz, Szz (Sxy = sum X*Y, ...) and Zmin, Zmax: independent of the
 *     order the points are visited in;
 *   on the host, in double without FMA contraction, each integer below converted to double once:
 *     cxx = n*Sxx - Sx*Sx, cxy = n*Sxy - Sx*Sy, cyy = n*Syy - Sy*Sy, cxz = n*Sxz - Sx*Sz, cyz = n*Syz - Sy*Sz,
 *       czz = n*Szz - Sz*Sz (exact in signed 128-bit arithmetic, then converted);
 *     det = cxx*cyy - cxy*cxy; fit_valid = n >= 3 && det > 0;
 *     a = (cxz*cyy - cyz*cxy) / det, b = (cyz*cxx - cxz*cxy) / det: the least-squares plane z = a x + b y + c through the
 *       centroid;
 *     rms_dz = sqrt(max(czz - a*cxz - b*cyz, 0)) / n / 65536 metres (RMS vertical residual: flatness);
 *     tilt_deg = atan(sqrt(a*a + b*b)) * (180 / M_PI);
 *     a, b, tilt_deg and rms_dz are 0 when fit_valid is 0;
 *   reported in the external world of ssd_gpu_step, through the ToExternalWorld the step's corners went through (plain calls:
 *   the context's; camera calls: the frame's camera's; group calls: the group's first member's camera's), in k_finalize's
 *   operation order: xm = x_min + (double)Sx / (double)n / 65536 (ym, zm likewise),
 *     centroid = ((ext_a[0]*xm + ext_a[1]*ym) + ext_b[0], (ext_a[2]*xm + ext_a[3]*ym) + ext_b[1], ext_z + zm),
 *     gradient = (ext_a[0]*a + ext_a[1]*b, ext_a[2]*a + ext_a[3]*b) (for a rotation: dz/dx, dz/dy in the rotated axes),
 *     z_lo = ext_z + (z_min + (double)Zmin / 65536), z_hi likewise with Zmax.
 * n == 0 (a step with SSD_STATUS_EMPTY_MEAN) gives an all-zero record. The ground step with an invalid front edge still gets
 * the surface of the pixels its step labels mark. n_points = n_in_quad of the step's plateau.
 * The option only reports: it changes no step, label or other result. It reads the step labels, so enabling it while step
 * labels are off, and switching step labels off while it is on, return SSD_E_STATE. Enabling allocates
 * max_frames * SSD_GPU_MAX_STEPS moment records (SSD_E_NOMEM, and the option stays off, when that fails) and returns SSD_E_RANGE
 * for a configuration with a range (x_max - x_min, y_max - y_min or z_max - z_min) of 65536 m or more, for which X, Y or Z
 * could reach 2^32 (the bound under which the moments are exact); enable == 0 frees them. The pass runs after the chain of
 * every ssd_gpu_process_* call and is counted in timing.n_launches. The getter returns SSD_E_STATE when the option is off,
 * the last call ran without it or its results are no longer readable (a failed call, a single-stage entry point), SSD_E_RANGE
 * for a frame outside the last call. Results are fixed when the call runs: replacing the camera table afterwards changes none.
 */
typedef struct ssd_gpu_step_surface
{
  uint32_t n_points;    /* points of the step: count(step_labels == s) over the frame / group */
  int32_t fit_valid;    /* n >= 3 && det > 0 */
  double centroid[3];   /* metres, external world */
  double gradient[2];   /* dz/dx, dz/dy of the fitted plane, external axes */
  double tilt_deg;      /* angle of the plane from level, degrees */
  double rms_dz;        /* RMS vertical residual about the plane, metres */
  double z_lo, z_hi;    /* z extent of the points, metres, external world */
} ssd_gpu_step_surface; /* 80 bytes */
int ssd_gpu_set_step_surfaces(ssd_gpu_ctx *ctx, int enable);
/* out[0..min(*n, cap)): *n = n_steps of the frame, in the order of ssd_gpu_get_steps. */
int ssd_gpu_get_step_surfaces(ssd_gpu_ctx *ctx, int frame, ssd_gpu_step_surface *out, int cap, int *n);
/* Per-pixel segment labels (device -> host copy of width*height bytes, the frame size). */
int ssd_gpu_get_labels(ssd_gpu_ctx *ctx, int frame, uint8_t *out_host);
/* Height histogram, HeightsHistogram::calcHist (pointcloud.cpp:194-204). */
int ssd_gpu_get_histogram(ssd_gpu_ctx *ctx, int frame, uint32_t *out, int cap, int *n_bins);
int ssd_gpu_get_timing(ssd_gpu_ctx *ctx, ssd_gpu_timing *out);
/* Counters of the last call. n_exact_fallback: points whose single-precision, range-normalised transform
 * v = (w - range centre) / half range lay within the proven f32 error bound eps = filter_eps1 * max|x,y,z| + filter_eps0
 * of a range / height-bin threshold, so the decision was taken by the exact double-precision chain instead (results
 * are bit-identical either way). */
typedef struct ssd_gpu_stats
{
  uint64_t n_points;
  uint64_t n_exact_fallback;
  uint64_t n_quad_fast;   /* point-in-quadrilateral decisions taken in single precision (inner box / filtered test) */
  uint64_t n_quad_exact;  /* ... taken by the exact QuadrilateralTest evaluation (compacted exact pass) */
  double filter_eps0, filter_eps1;
  uint64_t n_bev_exact;   /* BEV pixels of outlined plateaus computed by the exact double chain */
} ssd_gpu_stats;
int ssd_gpu_get_stats(ssd_gpu_ctx *ctx, ssd_gpu_stats *out);
/* Per-stage device time of the last call made with SSD_FLAG_STAGE_TIMING: sum of per-launch durations (ms) and
 * launch counts. Stage order: 0 transform_bin, 1 peaks, 2 label_bev, 3 outline, 4 frame_logic, 5 quad_reduce, 6 finalize. */
#define SSD_GPU_N_STAGES 7
int ssd_gpu_get_stage_times(ssd_gpu_ctx *ctx, float ms[SSD_GPU_N_STAGES], int launches[SSD_GPU_N_STAGES]);
const char *ssd_gpu_stage_name(int stage);
/* Frames per launch chain (chunk) chosen for this context. */
int ssd_gpu_chunk_frames(ssd_gpu_ctx *ctx);
/* Device pointer to the label array of the last call (n_frames * width*height bytes, the frame size). */
int ssd_gpu_labels_device_ptr(ssd_gpu_ctx *ctx, const uint8_t **out);

/* Stairs::serialize (stairs.cpp:55-70): writes the NUL-terminated line into buf; returns the length
 * needed (excluding NUL) or a negative error. Host only. */
int ssd_stairs_serialize(const ssd_gpu_step *steps, int n, char *buf, size_t cap);

/* ---- single-stage entry points (same kernels, one image / one quadrilateral) ---- */
/* Segmentation::detectOutline (segmentation.cpp:919-971): image is a BEV image, bev_width*bev_height u8 (non-zero = set).
 * quad_px: 4 x (x,y) image points, valid: isConvex. */
int ssd_gpu_detect_outline(ssd_gpu_ctx *ctx, const uint8_t *image_host, int min_img_y_extent, double xy_ratio,
                           double quad_px[8], int *valid);
/* Segmentation::detectFrontEdge (segmentation.cpp:879-917); image as for ssd_gpu_detect_outline. */
int ssd_gpu_detect_front_edge(ssd_gpu_ctx *ctx, const uint8_t *image_host, double left_px[2], double right_px[2], int *valid);
/* QuadrilateralTest ctor + isPointWithin (quadrilateralTest.cpp:275-451) over n host points (x,y pairs).
 * *ctor_status = 0 ok, 1 the reference ctor would throw (then inside[] is all 0). */
int ssd_gpu_points_in_quad(ssd_gpu_ctx *ctx, const double quad[8], const double *xy_host, int n, uint8_t *inside_host,
                           int *ctor_status);
/* CameraToWorld over n host vertices -> n x 3 doubles (transformation.h:59-64). */
int ssd_gpu_camera_to_world(ssd_gpu_ctx *ctx, const float *xyz_host, int n, double *world_host);

/* ---- host-side transformation builders (transformation.cpp), no GPU needed ---- */
/* GeometricTransformation(worldPoints, cameraPoints) (transformation.cpp:196-215): 3 points each, xyz. */
int ssd_make_transform(const double world_pts[9], const double camera_pts[9], ssd_gpu_transform *out);
/* The same, and the camera transformation's _aInv (row-major) exactly as the reference holds it: the triangle ctor
 * (transformation.cpp:108-157) sets _aInv from the plane's base vectors and _a = transposed(_aInv). For ssd_gpu_set_overlay. */
int ssd_make_transform_ex(const double world_pts[9], const double camera_pts[9], ssd_gpu_transform *out, double a_inv[9]);
/* boost::qvm::inverse of a 3x3 as the (rp, rpMapping) ctor computes _aInv = inverse(_a) (transformation.cpp:175-178). */
int ssd_inverse3(const double a[9], double a_inv[9]);
/* GeometricCalibration::load() (geometricCalibration.cpp:185-203): reads "<directory>/calibration-triangle"
 * (CalibrationTriangle::load, calibrationTriangle.cpp:97-125; validity :148-168) and "<directory>/calibration-points"
 * (loadPoints, geometricCalibration.cpp:73-98: header + ten rows of three "x, y, z" float triples), averages the rows
 * (calcAverageRefPointSet, :127-141) and builds the transformation. directory NULL or "": current directory, as the
 * reference. Returns SSD_OK, or SSD_CAL_* > 0 when a file is missing / malformed -- then *out is the identity
 * transformation the reference silently falls back to (geometricCalibration.cpp:199-202); world_pts / camera_pts
 * (may be NULL) receive the six reference points. */
#define SSD_CAL_TRIANGLE_MISSING 1
#define SSD_CAL_TRIANGLE_INVALID 2
#define SSD_CAL_POINTS_MISSING 3
int ssd_load_calibration(const char *directory, ssd_gpu_transform *out, double world_pts[9], double camera_pts[9]);

/* ---- raw device memory helpers for callers without a CUDA runtime binding ---- */
int ssd_gpu_malloc(ssd_gpu_ctx *ctx, size_t bytes, void **dev_ptr);
int ssd_gpu_free(ssd_gpu_ctx *ctx, void *dev_ptr);
int ssd_gpu_memcpy_h2d(ssd_gpu_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes);
int ssd_gpu_memcpy_d2h(ssd_gpu_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes);
int ssd_gpu_malloc_host(size_t bytes, void **host_ptr); /* pinned */
int ssd_gpu_free_host(void *host_ptr);
/* Page-lock a buffer the caller already owns (cudaHostRegister) -- e.g. the frame buffer a capture SDK hands out, which is
 * ordinary pageable memory: the host-input entry points then copy at the PCIe rate instead of through the driver's staging
 * (measured on one B200: 34.8 k against 6.9 k frames/s of 1024 x 768 z16 frames). Unregister before the buffer is freed. */
int ssd_gpu_register_host(void *host_ptr, size_t bytes);
int ssd_gpu_unregister_host(void *host_ptr);

#ifdef __cplusplus
}
#endif
#endif /* SSD_GPU_H_ */
