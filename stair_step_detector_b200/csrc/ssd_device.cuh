// ssd_device.cuh -- device-side data layout and exact geometry primitives of the hot path.
//
// This translation unit is compiled with -fmad=false: the reference build never contracts a*b+c
// (CMakeLists.txt:23-28 sets no -march / -ffast-math), and bit-exact labels need the same roundings.
// Every formula cites the reference file:line whose arithmetic (operation order) it reproduces.
#pragma once
#include "../../include/ssd_gpu.h"
#include "ssd_lens.h"
#include <cstdint>
#include <cuda_runtime.h>

#define SSD_BINS_PAD 256            // histogram slots: bins 0..252, 254 = out of range, 255 = invalid
#define SSD_CODE_OUT_OF_RANGE 254u
#define SSD_CODE_INVALID 255u
#define SSD_MAX_LINE_PTS 192        // points per edge list (W/25 + 2 scans split in overlapping halves)
#define SSD_MAX_SCANS 384
#define SSD_MAX_VPTS 512            // vertical-edge probe rows (H/10 + 1)

// Constant per-context parameters, passed to every kernel by value (__grid_constant__).
struct DevParams
{
  int W, H, N;             // image size, points per frame
  int wpr;                 // 32-bit words per BEV bitmap row
  int n_bins;              // HeightsHistogram size (pointcloud.cpp:196)
  int min_height;          // ProcessingConfiguration::minHeight (pointcloud.cpp:102)
  int min_img_y_extent;    // (pointcloud.cpp:103)
  unsigned min_peak_points;
  int bev_slots;           // BEV bitmaps per frame
  int tiles_per_frame;
  int pad0, pad1;
  double a[9], b[3];       // CameraToWorld
  double ext_a[4], ext_b[2], ext_z;
  double x_min, x_max, y_min, y_max, z_min, z_max;
  double hir;              // heightIntervalReciprocal (pointcloud.cpp:101)
  double x_to_image, y_to_image, x_to_world, y_to_world, xy_ratio; // Projection2D (pointcloud.cpp:73-76,95)
  // single-precision world coordinates of a vertex: f32-rounded CameraToWorld rows and the coefficients of the rigorous
  // error bound eps = E1 * max|p| + E0 on them (derive_params); used through the packed pairs axy2 / bxy2 below
  float af[9], bf[3];
  float E0, E1;
  // single-precision BEV pixel (fast_pixel2): u = au . p + bu ~ (wx - x_min) * x_to_image, v = av . p + bv ~
  // (y_max - wy) * y_to_image, with the error bounds |u^ - u_ref| <= Eu1 * max|p| + Eu0 (same for v)
  float au[3], bu, av[3], bv;
  float Eu0, Eu1, Ev0, Ev1;
  float Tf;                // max |x|, |y| of an in-range world point (quadfilter margins)
  // the same bounds for ANY in-range point: max|p| <= Mmax (derive_params), so eps <= epsc etc. are constants
  float epsc, euc, evc;
  float hu, hv;            // fast_pixel2: 1/2 - euc - 2^-20, 1/2 - evc - 2^-20 (negative: never certain)
  // k_transform_bin (point_code_scaled): rows of the transform scaled to the measuring range, v_i = (w_i - c_i) / h_i,
  // so "in range" is max|v_i| < 1; height bin t = G * (v_z + 1) with G = h_z * hir; eps = E1s * max|p| + E0s bounds
  // |v^_i - v_i| (8u (S_i m + B_i), derive_params); bin certain iff |frac distance| < thr0 - Gup * eps
  float sa[9], sb[3];
  float E0s, E1s, Gf, Gm, Gup, thr0;
  // per-step z sum (z_fix_u): world z in single precision scaled by 2^zshift, rounded to an integer by the 1.5*2^23 add
  float azf[3], bzf;
  int zshift, pad2;
  // k_quad_reduce ground BEV column pre-filter: t = wx * gcol_a + gcol_b = ((wx - x_min) sx - (W/2 - 2)) / 50
  float gcol_a, gcol_b, gcol_lo, gcol_hi, gcol_tmax, pad3;
  // packed pairs for the f32x2 pipes: {af[j], af[3+j]}, {bf[0], bf[1]} (world x,y) and {au[j], av[j]}, {bu, bv} (BEV pixel)
  unsigned long long axy2[3], bxy2, auv2[3], buv2;
  // {sa[j], sa[3+j]}, {sb[0], sb[1]}: the x and y rows of the range-scaled transform (point_code_scaled)
  unsigned long long sxy2[3], sbxy2;
  // record chain / resident-frame path. Per-point record: ix | iy << rec_bx | (bin code & 1) << (rec_bx + rec_by) | d << (32 - rec_zbits), d = the point's
  // height offset from the centre of its bin in units of 2^-rec_zshift m (rec_mf = height_interval * 2^rec_zshift,
  // |d| <= rec_mf / 2 < 2^(rec_zbits - 1)); iy == H marks a pixel the f32 chain could not decide. rec_zbits == 0: the
  // frame size does not admit the path.
  int rec_bx, rec_by, rec_zbits, rec_zshift;
  float rec_mf;
  int gs_steps;            // 128-point steps per frame
  // k_quad_sum: world rectangle of a BEV pixel box in single precision (x = ix * gs_xw + gs_x0, y = gs_y0 - iy * gs_yw)
  float gs_xw, gs_x0, gs_yw, gs_y0, gs_margin, pad4;
};

struct SegmentDev
{
  double lo_x, hi_x, lo_y, hi_y; // bounding box
  double k, c;                   // flat: x*k + y + c ; steep: x + y*k + c
  int steep, left_is_pos;
};

// QuadrilateralTest flattened into data (quadrilateralTest.cpp:275-443): <=3 rows x <=3 cells,
// each cell a constant or 1-2 half-plane tests.
struct QuadTestDev
{
  double tb_lo_x, tb_hi_x, tb_lo_y, tb_hi_y;
  SegmentDev seg[4];
  double row_upper_y[3];
  double cell_upper_x[3][3];
  int nrow;
  int ncell[3];
  signed char cell_nseg[3][3]; // 0,1,2 segments; for 0: cell_seg[.][.][0] holds the constant result
  signed char cell_seg[3][3][2];
  int inside_is_left;
  int status; // 0 ok, 1 the reference ctor would throw
  // Axis-aligned box (centre / half width, metres) every point of which passes the test above -- verified
  // cell by cell in quadtest_inner_box(). ib_hx < 0: no box. Used as a single-precision fast accept.
  float ib_cx, ib_hx, ib_cy, ib_hy;
};

// Single-precision image of one QuadTestDev for the filtered point-in-quadrilateral decision (quadfilter_eval):
// the same bounding box / row / cell / half-plane structure evaluated in f32 with rigorous margins; a point
// whose f32 evaluation comes within a margin of any comparison is re-decided by the exact double test.
struct QuadFilterDev
{
  float4 ib;             // verified inner box (quadtest_inner_box): cx, hx, cy, hy; hx < 0: none
  float4 bb;             // bounding box: lo_x, hi_x, lo_y, hi_y
  float4 seg[6];         // kx, ky, c, margin; signed so that "passes" <=> kx*x + ky*y + c > 0. [4] always true, [5] always false
  float row_thr[2];      // y thresholds between rows (+inf when unused)
  float cell_thr[3][2];  // x thresholds between the cells of a row
  unsigned char cell_s[3][3][2]; // the two half-plane slots of each cell (indices into seg[])
  unsigned char ok, pad8;        // ok = 0: no filter for this quadrilateral (every point takes the exact test)
  float pad[3];
  float4 ibe;            // inner box for the constant-eps fast accept: cx, cy, hx - epsc, hy - epsc (negative: none)
  float4 rj;             // reject box around the same centre: |x - cx| > rj.x or |y - cy| > rj.y => certainly outside the bounding box
};

struct PlateauDev
{
  int height, hmin, hmax;
  unsigned n_points;
  int valid, outlined;
  unsigned n_in_quad;
  int quad_status;
  double quad_px[4][2];
  double quad_world[4][2];
  double mean_z;
  unsigned long long sum_fix; // sum of z_fix_u() over the points inside the quadrilateral that were tested one by one
  // ... and of the points taken in as whole 32-pixel summaries (k_quad_sum): height offsets, bin codes, how many
  long long sum_d;
  unsigned long long sum_c;
  unsigned n_sum, pad_s;
  int row_min, row_max;       // BEV rows touched by this plateau's bitmap
  int front_valid;
  int pad;
  QuadTestDev qt;
};

// accumulators of one riser (ssd_gpu_riser, include/ssd_gpu.h): X = (int64)((x - x_min) * 65536), Y likewise
struct RiserDev
{
  unsigned cnt;
  int xmin, xmax, ymin, ymax;
  int pad;
  unsigned long long sx, sy;
};

struct FrameDev
{
  unsigned hist[SSD_BINS_PAD];
  unsigned short lut16[SSD_BINS_PAD]; // bin code -> segment label | 0x100 if that label gets a BEV image (k_peaks)
  unsigned quad_amask;                // labels k_quad_reduce reduces: ground + valid plateaus with a usable test (k_frame_logic)
  unsigned ready;                     // k_frame_stream: plateau records and lut16 are written (the frame barrier's flag)
  unsigned tb_done, ol_done;          // fused small-batch chain: blocks of k_transform_bin / k_outline that have finished this frame
  QuadFilterDev qf[SSD_GPU_MAX_PLATEAUS]; // f32 image of each step's QuadrilateralTest (k_frame_logic)
  unsigned status;
  int n_plateaus;
  int ground_index, first_outlined, first_valid;
  int n_steps;
  unsigned n_nonzero, n_in_range;
  // counters of the filtered decisions (ssd_gpu_get_stats)
  unsigned n_exact_bin;  // k_transform_bin: points decided by the exact double chain
  unsigned n_quad_pts;   // k_quad_reduce: points tested against a quadrilateral
  unsigned n_def_quad;   // ... of which went to the compacted exact pass
  unsigned n_def_bev;    // k_label_bev: BEV pixels computed by the exact double chain
  PlateauDev plat[SSD_GPU_MAX_PLATEAUS];
  RiserDev ris[SSD_GPU_MAX_PLATEAUS]; // k_riser_reduce (only when vertical faces are enabled); zeroed by k_peaks
};

// compact per-frame result copied to the host after every call
struct FrameOut
{
  ssd_gpu_frame_info info;
  ssd_gpu_step steps[SSD_GPU_MAX_STEPS];
  unsigned n_exact_bin, n_quad_pts, n_def_quad, n_def_bev;
};

// drawStairStep's projection of the step corners into the camera image (pointcloud.cpp:583-597): WorldToCamera
// (transformation.h:66-69: a_inv * (p - b)) then rs2_project_point_to_pixel (camera.h:80-97). enabled = 0: off.
struct OverlayDev
{
  double a_inv[9];
  float fx, fy, ppx, ppy;
  int enabled, pad;
};

// Per-frame cameras (ssd_gpu_set_cameras). The kernels of the classic chain take a trailing CAM argument: NoCam (the default)
// processes every frame with the launch's DevParams, the context's own camera; CamTable takes each frame's parameters from the
// camera table, derived per camera by derive_params exactly as for a context created with that camera.
struct NoCam
{
};
struct CamTable
{
  const DevParams *params; // n_cameras
  const OverlayDev *ov;    // n_cameras: drawStairStep projection of each camera (a_inv, intrinsics; enabled = 1)
  const float *xn, *yn;    // n_cameras x W, n_cameras x H deprojection tables (depth input)
  const float *unit;       // n_cameras: metres per depth unit
  const int *cam;          // camera of each frame of the call
  int frame0;              // first frame of the launch within the call
};

__device__ __forceinline__ int frame_camera(const CamTable &c, int frame)
{
  return __ldg(c.cam + c.frame0 + frame);
}
__device__ __forceinline__ const DevParams &frame_params(const DevParams &p, const NoCam &, int)
{
  return p;
}
// The block copies its frame's table entry into shared memory once; every thread of the block must call this before any
// thread leaves the kernel.
__device__ __forceinline__ const DevParams &frame_params(const DevParams &, const CamTable &c, int frame)
{
  __shared__ DevParams s_cam_params;
  static_assert(sizeof(DevParams) % 8 == 0, "DevParams is copied in 8-byte words");
  const unsigned long long *src = reinterpret_cast<const unsigned long long *>(c.params + frame_camera(c, frame));
  unsigned long long *dst = reinterpret_cast<unsigned long long *>(&s_cam_params);
  for(int i = threadIdx.x; i < (int)(sizeof(DevParams) / 8); i += blockDim.x)
    dst[i] = __ldg(src + i);
  __syncthreads();
  return s_cam_params;
}
__device__ __forceinline__ const OverlayDev &frame_overlay(const OverlayDev &ov, const NoCam &, int)
{
  return ov;
}
__device__ __forceinline__ const OverlayDev &frame_overlay(const OverlayDev &ov, const CamTable &c, int frame)
{
  return ov.enabled ? c.ov[frame_camera(c, frame)] : ov;
}
// The overlay through a distorted lens (k_finalize only): LensCam<NoCam> / LensCam<CamTable> behave as their BASE and add the lens
// of the plain overlay (lens[0]) or of each camera (lens[camera]). NoCam and CamTable project through the pin-hole.
template<class BASE>
struct LensCam
{
  BASE base;
  const ssd_gpu_distortion *lens;
};
template<class BASE>
__device__ __forceinline__ const DevParams &frame_params(const DevParams &p, const LensCam<BASE> &c, int frame)
{
  return frame_params(p, c.base, frame);
}
template<class BASE>
__device__ __forceinline__ const OverlayDev &frame_overlay(const OverlayDev &ov, const LensCam<BASE> &c, int frame)
{
  return frame_overlay(ov, c.base, frame);
}
template<class CAM>
__device__ __forceinline__ void overlay_lens(const CAM &, int, float x, float y, float &xd, float &yd)
{
  xd = x;
  yd = y;
}
__device__ __forceinline__ void overlay_lens(const LensCam<NoCam> &c, int, float x, float y, float &xd, float &yd)
{
  const ssd_gpu_distortion d = c.lens[0];
  ssd_lens_project(&d, x, y, &xd, &yd);
}
__device__ __forceinline__ void overlay_lens(const LensCam<CamTable> &c, int frame, float x, float y, float &xd, float &yd)
{
  const ssd_gpu_distortion d = c.lens[frame_camera(c.base, frame)];
  ssd_lens_project(&d, x, y, &xd, &yd);
}

struct P2d
{
  double x, y;
};
struct P2id
{
  int x, y;
};
struct LineDd
{
  double a, b, c;
};
struct LineId
{
  int a, b, c;
};

// ---- CameraToWorld: ((a_i0*x + a_i1*y) + a_i2*z) + b_i  (transformation.h:59-64, Boost.QVM mat*vec, vec+vec) ----
__device__ __forceinline__ void camera_to_world(const DevParams &p, float fx, float fy, float fz, double &wx, double &wy, double &wz)
{
  const double x = fx, y = fy, z = fz;
  wx = ((p.a[0] * x + p.a[1] * y) + p.a[2] * z) + p.b[0];
  wy = ((p.a[3] * x + p.a[4] * y) + p.a[5] * z) + p.b[1];
  wz = ((p.a[6] * x + p.a[7] * y) + p.a[8] * z) + p.b[2];
}

// x,y rows only (BEV projection, point-in-quadrilateral) and the z row alone (height sum): same roundings
__device__ __forceinline__ void camera_to_world_xy(const DevParams &p, float fx, float fy, float fz, double &wx, double &wy)
{
  const double x = fx, y = fy, z = fz;
  wx = ((p.a[0] * x + p.a[1] * y) + p.a[2] * z) + p.b[0];
  wy = ((p.a[3] * x + p.a[4] * y) + p.a[5] * z) + p.b[1];
}
__device__ __forceinline__ double camera_to_world_z(const DevParams &p, float fx, float fy, float fz)
{
  const double x = fx, y = fy, z = fz;
  return ((p.a[6] * x + p.a[7] * y) + p.a[8] * z) + p.b[2];
}

// ---- packed f32x2 arithmetic (Blackwell FFMA2 / FADD2: two single-precision operations per instruction) ----
typedef unsigned long long f32x2_t;
__host__ __device__ __forceinline__ f32x2_t f2_pack_bits(float lo, float hi)
{
  union { float f[2]; unsigned long long u; } c;
  c.f[0] = lo;
  c.f[1] = hi;
  return c.u;
}
__device__ __forceinline__ f32x2_t f2_pack(float lo, float hi)
{
  f32x2_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(f32x2_t v, float &lo, float &hi)
{
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2_t f2_fma(f32x2_t a, f32x2_t b, f32x2_t c)
{
  f32x2_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ f32x2_t f2_add(f32x2_t a, f32x2_t b)
{
  f32x2_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// {c0.lo*x + ..., c0.hi*x + ...}: two rows of an affine map applied to one point, same fma order as the scalar chains
__device__ __forceinline__ f32x2_t f2_affine(const f32x2_t c[3], f32x2_t b, float x, float y, float z)
{
  return f2_fma(c[2], f2_pack(z, z), f2_fma(c[1], f2_pack(y, y), f2_fma(c[0], f2_pack(x, x), b)));
}

// z>0 (pointcloud.cpp:143-146), range (pointcloud.cpp:155-163), height index (pointcloud.cpp:175)
__device__ __forceinline__ unsigned point_code(const DevParams &p, float fx, float fy, float fz)
{
  if(!(fz > 0.f))
    return SSD_CODE_INVALID;
  double wx, wy, wz;
  camera_to_world(p, fx, fy, fz, wx, wy, wz);
  const bool in = wx > p.x_min && wx < p.x_max && wy > p.y_min && wy < p.y_max && wz > p.z_min && wz < p.z_max;
  if(!in)
    return SSD_CODE_OUT_OF_RANGE;
  return (unsigned)(unsigned short)((wz - p.z_min) * p.hir);
}

// out-of-line copy for the rare fallback of the filtered kernel (keeps its hot loop small)
__device__ __noinline__ unsigned point_code_slow(const DevParams &p, float fx, float fy, float fz)
{
  return point_code(p, fx, fy, fz);
}

// 3-input maximum of absolute values, NaN-propagating (one FMNMX3.NAN): a NaN coordinate must not be dropped
__device__ __forceinline__ float max3abs_nan(float a, float b, float c)
{
  float r;
  asm("max.NaN.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(fabsf(a)), "f"(fabsf(b)), "f"(fabsf(c)));
  return r;
}

// The decision of point_code() from single-precision arithmetic on range-scaled rows plus a rigorous error bound.
//   v^_i = fma chain with f32-rounded a_ij/h_i, (b_i-c_i)/h_i:  |v^_i - v_ref,i| <= 4.0001u (S_i m + B_i) + the
//   reference's own f64 roundings (2^-50 of the same magnitudes), u = 2^-24, m = max|p|; eps carries 8u: factor 2 slack.
//   in range  <=> max_i |v_i| < 1:   certain if |r - 1| > eps  (r - 1 is exact for r in [0.5, 2], elsewhere |r - 1| >> eps)
//   bin = floor(t), t = G (v_z + 1): u_f = fma(v^_z, G, G - 0.5) ~ t - 0.5 within Gup*eps + dbin; k = round(u_f) via the
//   1.5*2^23 trick (d = u_f - k is exact); floor(t) == k is certain iff |d| < 0.5 - (Gup*eps + dbin) = thr0 - Gup*eps.
// NaN anywhere makes r or eps NaN, every comparison false => uncertain => exact path. Inf likewise through eps.
// Returns the code when certain; `uncertain` asks for point_code().
__device__ __forceinline__ unsigned point_code_scaled(const DevParams &p, float x, float y, float z, bool &uncertain)
{
  const float m = max3abs_nan(x, y, z);
  const float eps = fmaf(p.E1s, m, p.E0s);
  // x and y rows as one packed chain (same fma order and roundings as the scalar chains)
  float vx, vy;
  f2_unpack(f2_affine(p.sxy2, p.sbxy2, x, y, z), vx, vy);
  const float vz = fmaf(p.sa[8], z, fmaf(p.sa[7], y, fmaf(p.sa[6], x, p.sb[2])));
  const float e1 = max3abs_nan(vx, vy, vz) - 1.0f;
  const float MAGIC = 12582912.0f;
  const float uf = fmaf(vz, p.Gf, p.Gm);
  const float s = uf + MAGIC;
  const float d = uf - (s - MAGIC);
  const float thr = fmaf(-p.Gup, eps, p.thr0);
  const bool out = e1 > eps;
  const bool in_bin = e1 < -eps && fabsf(d) < thr;
  const bool valid = z > 0.f;
  uncertain = valid && !(out || in_bin);
  const unsigned c = out ? SSD_CODE_OUT_OF_RANGE : ((unsigned)__float_as_int(s) & 0xffu);
  return valid ? c : SSD_CODE_INVALID;
}

// Single-precision BEV pixel of an in-range point with the constant error bounds euc / evc (packed arithmetic). Returns
// true when (ix, iy) is certainly the pixel the exact double chain (camera_to_world_xy + bev_pixel) produces.
//   s = RD(u^ + 1.5*2^23): the sum rounded towards -inf lands on the integer grid, so its mantissa holds floor(u^)
//   (no conversion instruction, no correction step); k = s - 1.5*2^23 and d = u^ - k in [0, 1) are exact.
//   floor(u_ref) == floor(u^) is certain when d is further than the error bound from both ends: |d - 1/2| < hu with
//   hu = 1/2 - euc - 2^-20 (the slack covers the rounding of d - 1/2). A certain pixel with 0 <= ix < W, 0 <= iy < H
//   lies inside the image, so neither the x == W wrap nor an out-of-image write (pointcloud.cpp:468) can occur.
__device__ __forceinline__ f32x2_t f2_sub(f32x2_t a, f32x2_t b)
{
  f32x2_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2_t f2_add_rm(f32x2_t a, f32x2_t b)
{
  f32x2_t r;
  asm("add.rm.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ bool fast_pixel2(const DevParams &p, float x, float y, float z, int &ix, int &iy)
{
  const float MAGIC = 12582912.0f;
  const f32x2_t uv = f2_affine(p.auv2, p.buv2, x, y, z);
  const f32x2_t s = f2_add_rm(uv, f2_pack(MAGIC, MAGIC));
  const f32x2_t k = f2_add(s, f2_pack(-MAGIC, -MAGIC));                 // exact
  const f32x2_t d = f2_sub(uv, k);                                      // exact, in [0, 1)
  const f32x2_t t = f2_add(d, f2_pack(-0.5f, -0.5f));
  float su, sv, tu, tv;
  f2_unpack(s, su, sv);
  f2_unpack(t, tu, tv);
  ix = __float_as_int(su) - 0x4B400000;
  iy = __float_as_int(sv) - 0x4B400000;
  return fabsf(tu) < p.hu && fabsf(tv) < p.hv && (unsigned)ix < (unsigned)p.W && (unsigned)iy < (unsigned)p.H;
}

// Projection2D::worldToImage (pointcloud.cpp:79-83)
__device__ __forceinline__ void world_to_image(const DevParams &p, double wx, double wy, int &ix, int &iy)
{
  ix = (int)((wx - p.x_min) * p.x_to_image);
  iy = (int)((p.y_max - wy) * p.y_to_image);
}

// BEV pixel of an in-range point the way the reference addresses it: *Mat::ptr(iy, ix) with no bounds check
// (pointcloud.cpp:468), i.e. linear offset iy*W + ix. In range means 0 <= ix <= W and 0 <= iy <= H (the upper
// ends only by rounding), so ix == W wraps to the next row and iy == H falls past the image.
__device__ __forceinline__ bool bev_pixel(const DevParams &p, double wx, double wy, int &x, int &y)
{
  world_to_image(p, wx, wy, x, y);
  if(x >= p.W)
  {
    x -= p.W;
    y += 1;
  }
  return x >= 0 && x < p.W && y >= 0 && y < p.H;
}

// Projection2D::imageToWorld (pointcloud.cpp:84-88)
__device__ __forceinline__ P2d image_to_world(const DevParams &p, P2d px)
{
  P2d w;
  w.x = p.x_min + px.x * p.x_to_world;
  w.y = p.y_max - px.y * p.y_to_world;
  return w;
}

// Correctly rounded hypot for the magnitudes that occur here (no overflow/underflow handling needed):
// x^2+y^2 in double-double via exact FMA residuals, one Newton correction of the square root.
// Stands in for std::hypot (segmentation.cpp:346-349); tests/test_hypot.py compiles this very function for the host and
// checks it against glibc's hypot on the operand ranges of the path (integer line coefficients, normalised lines).
#ifdef __CUDA_ARCH__
#define SSD_FMA_RN(a, b, c) __fma_rn(a, b, c)
#else
#define SSD_FMA_RN(a, b, c) fma(a, b, c)
#endif
__host__ __device__ __forceinline__ double hypot_cr(double x, double y)
{
  const double xx = x * x, yy = y * y;
  const double ex = SSD_FMA_RN(x, x, -xx), ey = SSD_FMA_RN(y, y, -yy);
  const double s = xx + yy;
  const double bb = s - xx;
  const double es = (xx - (s - bb)) + (yy - bb); // TwoSum error
  const double lo = es + (ex + ey);
  if(s == 0.0)
    return 0.0;
  const double h = sqrt(s);
  const double r = SSD_FMA_RN(-h, h, s) + lo;
  return h + r / (2.0 * h);
}

// ---- lines (types.h:117-163, segmentation.cpp:321-401) ----
__device__ __forceinline__ LineId linei_from(P2id p, P2id q)
{
  LineId l;
  l.a = q.y - p.y;
  l.b = p.x - q.x;
  l.c = q.x * p.y - p.x * q.y;
  return l;
}
__device__ __forceinline__ LineDd lined_from_pts(P2d p, P2d q)
{
  LineDd l;
  l.a = q.y - p.y;
  l.b = p.x - q.x;
  l.c = q.x * p.y - p.x * q.y;
  return l;
}
__device__ __forceinline__ LineDd lined_from_i(LineId l)
{
  LineDd d;
  d.a = l.a;
  d.b = l.b;
  d.c = l.c;
  return d;
}
__device__ __forceinline__ LineDd lined_normalized(LineDd l) // segmentation.cpp:381-385
{
  const double h = hypot_cr(l.a, l.b);
  LineDd r;
  r.a = l.a / h;
  r.b = l.b / h;
  r.c = l.c / h;
  return r;
}
__device__ __forceinline__ LineDd bisector(LineDd n, LineDd o) // :386-394, operands already normalized
{
  LineDd r;
  r.a = n.a + o.a;
  r.b = n.b + o.b;
  r.c = n.c + o.c;
  return r;
}
// Line::intersection with the 60 degree gate (segmentation.cpp:350-362)
__device__ __forceinline__ bool lined_intersection(LineDd t, LineDd o, P2d &out)
{
  const double tan60 = 1.7320508075688772935274463415059;
  const double numerator = t.a * o.b - o.a * t.b;
  const double denominator = t.a * o.a + t.b * o.b;
  if(fabs(numerator) > fabs(denominator) * tan60)
  {
    out.x = (t.b * o.c - o.b * t.c) / numerator;
    out.y = (o.a * t.c - t.a * o.c) / numerator;
    return true;
  }
  return false;
}
// nested Line::intersection without gate (pointcloud.cpp:514-526)
__device__ __forceinline__ P2d line_intersection_plain(LineDd t, LineDd o)
{
  const double d = t.a * o.b - o.a * t.b;
  P2d r;
  r.x = (t.b * o.c - o.b * t.c) / d;
  r.y = (o.a * t.c - t.a * o.c) / d;
  return r;
}

// Quadrilateral::isConvex (segmentation.cpp:755-787)
__device__ __forceinline__ bool quad_is_convex(const P2d q[4])
{
  const double vx[4] = { q[1].x - q[0].x, q[3].x - q[1].x, q[2].x - q[3].x, q[0].x - q[2].x };
  const double vy[4] = { q[1].y - q[0].y, q[3].y - q[1].y, q[2].y - q[3].y, q[0].y - q[2].y };
  const bool p01 = vx[0] * vy[1] - vx[1] * vy[0] > 0;
  const bool p12 = vx[1] * vy[2] - vx[2] * vy[1] > 0;
  const bool p23 = vx[2] * vy[3] - vx[3] * vy[2] > 0;
  const bool p30 = vx[3] * vy[0] - vx[0] * vy[3] > 0;
  return p01 == p12 && p01 == p23 && p01 == p30;
}

// ---- QuadrilateralTest (quadrilateralTest.cpp) ----
struct SectorD
{
  double lo, hi;
};
__device__ __forceinline__ SectorD sector_make(double a, double b) // :29-41
{
  SectorD s;
  s.lo = a;
  s.hi = a;
  if(s.lo > b)
    s.lo = b;
  else if(s.hi < b)
    s.hi = b;
  return s;
}
__device__ __forceinline__ void sector_expand(SectorD &s, double c)
{
  if(s.lo > c)
    s.lo = c;
  else if(s.hi < c)
    s.hi = c;
}
__device__ __forceinline__ bool sector_overlaps(SectorD a, SectorD b) { return a.lo < b.hi && a.hi > b.lo; }
__device__ __forceinline__ bool sector_is_above(SectorD a, SectorD b) { return (a.lo + a.hi) / 2 < b.lo; }
__device__ __forceinline__ bool sector_is_below(SectorD a, SectorD b) { return (a.lo + a.hi) / 2 > b.hi; }

__device__ __forceinline__ SegmentDev segment_create(P2d p, P2d q) // :240-259 with the line classes :133-231
{
  SegmentDev s;
  SectorD sx = sector_make(p.x, q.x), sy = sector_make(p.y, q.y);
  s.lo_x = sx.lo;
  s.hi_x = sx.hi;
  s.lo_y = sy.lo;
  s.hi_y = sy.hi;
  const double dx = q.x - p.x, dy = q.y - p.y;
  const LineDd l = lined_from_pts(p, q);
  if(fabs(dx) < fabs(dy))
  {
    s.steep = 1;
    s.k = l.b / l.a;
    s.c = l.c / l.a;
    s.left_is_pos = !(dy > 0);
  }
  else
  {
    s.steep = 0;
    s.k = l.a / l.b;
    s.c = l.c / l.b;
    s.left_is_pos = dx > 0;
  }
  return s;
}
__device__ __forceinline__ bool segment_is_left(const SegmentDev &s, double x, double y)
{
  const bool pos = s.steep ? (x + y * s.k + s.c > 0) : (x * s.k + y + s.c > 0);
  return s.left_is_pos ? pos : !pos;
}

// ctor (quadrilateralTest.cpp:275-443). status 1 where the reference throws std::invalid_argument.
__device__ inline void quadtest_init(QuadTestDev &t, const P2d q[4])
{
  t.status = 0;
  SectorD tx = sector_make(q[0].x, q[1].x), ty = sector_make(q[0].y, q[1].y);
  sector_expand(tx, q[2].x);
  sector_expand(ty, q[2].y);
  sector_expand(tx, q[3].x);
  sector_expand(ty, q[3].y);
  t.tb_lo_x = tx.lo;
  t.tb_hi_x = tx.hi;
  t.tb_lo_y = ty.lo;
  t.tb_hi_y = ty.hi;
  t.seg[0] = segment_create(q[0], q[1]);
  t.seg[1] = segment_create(q[1], q[3]);
  t.seg[2] = segment_create(q[3], q[2]);
  t.seg[3] = segment_create(q[2], q[0]);
  t.inside_is_left = segment_is_left(t.seg[0], q[3].x, q[3].y);
  t.nrow = 0;
  if(t.inside_is_left != (int)segment_is_left(t.seg[1], q[2].x, q[2].y) || t.inside_is_left != (int)segment_is_left(t.seg[2], q[0].x, q[0].y) ||
     t.inside_is_left != (int)segment_is_left(t.seg[3], q[1].x, q[1].y))
  {
    t.status = 1;
    return;
  }
  double xs[4] = { q[0].x, q[1].x, q[2].x, q[3].x }, ys[4] = { q[0].y, q[1].y, q[2].y, q[3].y };
#pragma unroll
  for(int i = 1; i < 4; i++)
    for(int j = i; j > 0; j--)
    {
      if(xs[j] < xs[j - 1])
      {
        const double tmp = xs[j];
        xs[j] = xs[j - 1];
        xs[j - 1] = tmp;
      }
      if(ys[j] < ys[j - 1])
      {
        const double tmp = ys[j];
        ys[j] = ys[j - 1];
        ys[j - 1] = tmp;
      }
    }
  // segment map: rows x cells (:314-345); neighbour flags only matter for empty cells
  int cellNb[3][3]; // bit r set: neighborExists[r]
  double lowerY = ys[0];
  for(int yi = 1; yi < 4; yi++)
  {
    if(!(lowerY < ys[yi]))
      continue;
    const int r = t.nrow++;
    t.row_upper_y[r] = ys[yi];
    t.ncell[r] = 0;
    double lowerX = xs[0];
    for(int xi = 1; xi < 4; xi++)
    {
      if(!(lowerX < xs[xi]))
        continue;
      const int c = t.ncell[r]++;
      t.cell_upper_x[r][c] = xs[xi];
      const SectorD cx = sector_make(lowerX, xs[xi]), cy = sector_make(lowerY, ys[yi]);
      int nseg = 0, nb = 0;
      int ids[4];
      for(int si = 0; si < 4; si++)
      {
        SectorD sx, sy;
        sx.lo = t.seg[si].lo_x;
        sx.hi = t.seg[si].hi_x;
        sy.lo = t.seg[si].lo_y;
        sy.hi = t.seg[si].hi_y;
        if(sector_overlaps(cx, sx) && sector_overlaps(cy, sy))
          ids[nseg++] = si;
        if(nseg == 0)
        {
          int rel = 0; // BBox::getRelativePosition (:96-113)
          if(sector_overlaps(cy, sy))
          {
            if(sector_is_above(cx, sx))
              rel = 1;
            else if(sector_is_below(cx, sx))
              rel = 2;
          }
          if(rel == 0 && sector_overlaps(cx, sx))
          {
            if(sector_is_above(cy, sy))
              rel = 3;
            else if(sector_is_below(cy, sy))
              rel = 4;
          }
          nb |= 1 << rel;
        }
      }
      if(nseg > 2)
        t.status = 1; // :357-358 (reported after the map is built; no side effects in between)
      t.cell_nseg[r][c] = (signed char)nseg;
      t.cell_seg[r][c][0] = (signed char)(nseg > 0 ? ids[0] : 0);
      t.cell_seg[r][c][1] = (signed char)(nseg > 1 ? ids[1] : 0);
      cellNb[r][c] = nb;
      lowerX = xs[xi];
    }
    lowerY = ys[yi];
  }
  if(t.nrow == 0)
  {
    t.status = 1; // :347-348
    return;
  }
  for(int r = 0; r < t.nrow; r++)
    if(t.ncell[r] == 0)
      t.status = 1; // :352-353
  if(t.status)
    return;
  // merge equal neighbours (:362-380)
  for(int r = 0; r < t.nrow; r++)
  {
    int ci = 0;
    while(ci != t.ncell[r] - 1)
    {
      const int n0 = t.cell_nseg[r][ci], n1 = t.cell_nseg[r][ci + 1];
      if((n0 == 0 && n1 == 0) || (n0 > 1 && n1 > 1))
      {
        t.status = 1;
        return;
      }
      bool same = n0 == n1;
      for(int s = 0; same && s < n0; s++)
        same = t.cell_seg[r][ci][s] == t.cell_seg[r][ci + 1][s];
      if(same)
      {
        for(int k = ci; k < t.ncell[r] - 1; k++)
        {
          t.cell_upper_x[r][k] = t.cell_upper_x[r][k + 1];
          t.cell_nseg[r][k] = t.cell_nseg[r][k + 1];
          t.cell_seg[r][k][0] = t.cell_seg[r][k + 1][0];
          t.cell_seg[r][k][1] = t.cell_seg[r][k + 1][1];
          cellNb[r][k] = cellNb[r][k + 1];
        }
        t.ncell[r]--;
      }
      else
        ci++;
    }
  }
  // set0Segments(...) constant (:387-392): all four neighbour directions seen
  for(int r = 0; r < t.nrow; r++)
    for(int c = 0; c < t.ncell[r]; c++)
      if(t.cell_nseg[r][c] == 0)
        t.cell_seg[r][c][0] = (signed char)((cellNb[r][c] & 0x1e) == 0x1e);
}

// isPointWithin (quadrilateralTest.cpp:445-451 and the selector/tester lambdas :453-598)
__device__ __forceinline__ bool quadtest_within(const QuadTestDev &t, double x, double y)
{
  if(!(t.tb_lo_x < x && x < t.tb_hi_x && t.tb_lo_y < y && y < t.tb_hi_y))
    return false;
  int r = 0;
  if(t.nrow == 2)
    r = y < t.row_upper_y[0] ? 0 : 1;
  else if(t.nrow == 3)
    r = y < t.row_upper_y[0] ? 0 : (y < t.row_upper_y[1] ? 1 : 2);
  int c = 0;
  if(t.ncell[r] == 2)
    c = x < t.cell_upper_x[r][0] ? 0 : 1;
  else if(t.ncell[r] == 3)
    c = x < t.cell_upper_x[r][0] ? 0 : (x < t.cell_upper_x[r][1] ? 1 : 2);
  const int n = t.cell_nseg[r][c];
  if(n == 0)
    return t.cell_seg[r][c][0] != 0;
  bool in = (int)segment_is_left(t.seg[t.cell_seg[r][c][0]], x, y) == t.inside_is_left;
  if(n == 2)
    in = in && (int)segment_is_left(t.seg[t.cell_seg[r][c][1]], x, y) == t.inside_is_left;
  return in;
}

// the predicate of one map cell at an arbitrary point (no bounding-box test, no cell selection)
__device__ __forceinline__ bool quadtest_cell_pred(const QuadTestDev &t, int r, int c, double x, double y)
{
  const int n = t.cell_nseg[r][c];
  if(n == 0)
    return t.cell_seg[r][c][0] != 0;
  bool in = (int)segment_is_left(t.seg[t.cell_seg[r][c][0]], x, y) == t.inside_is_left;
  if(n == 2)
    in = in && (int)segment_is_left(t.seg[t.cell_seg[r][c][1]], x, y) == t.inside_is_left;
  return in;
}

// Inner box for the fast accept. Candidate: the middle interval of the sorted corner coordinates, shrunk by
// 0.1 % .. 8 %. It is accepted only if, for every map cell it overlaps, the cell's predicate holds at the four corners
// of (box intersect cell): each half-plane value fl(fl(x*k)+y)+c is monotone in x and in y (IEEE operations
// are monotone), so its minimum over a rectangle is attained at a corner -- the predicate then holds on the
// whole intersection, hence isPointWithin() is true for every point of the box.
__device__ inline void quadtest_inner_box(QuadTestDev &t, const P2d q[4])
{
  t.ib_cx = t.ib_cy = 0.f;
  t.ib_hx = t.ib_hy = -1.f;
  if(t.status)
    return;
  double xs[4] = { q[0].x, q[1].x, q[2].x, q[3].x }, ys[4] = { q[0].y, q[1].y, q[2].y, q[3].y };
  for(int i = 1; i < 4; i++)
    for(int j = i; j > 0; j--)
    {
      if(xs[j] < xs[j - 1])
      {
        const double tmp = xs[j];
        xs[j] = xs[j - 1];
        xs[j - 1] = tmp;
      }
      if(ys[j] < ys[j - 1])
      {
        const double tmp = ys[j];
        ys[j] = ys[j - 1];
        ys[j - 1] = tmp;
      }
    }
  // the smallest shrink whose box verifies (a near-rectangle passes with the first; every percent of shrink sends
  // that share of the step's points to the slower filtered test)
  double bx0 = 0, bx1 = 0, by0 = 0, by1 = 0;
  bool found = false;
  for(int attempt = 0; attempt < 4 && !found; attempt++)
  {
    const double fr = attempt == 0 ? 0.001 : (attempt == 1 ? 0.005 : (attempt == 2 ? 0.02 : 0.08));
    const double sx = fr * (xs[2] - xs[1]) + 1e-6, sy = fr * (ys[2] - ys[1]) + 1e-6;
    bx0 = xs[1] + sx;
    bx1 = xs[2] - sx;
    by0 = ys[1] + sy;
    by1 = ys[2] - sy;
    if(!(bx0 < bx1 && by0 < by1))
      return;
    if(!(t.tb_lo_x < bx0 && bx1 < t.tb_hi_x && t.tb_lo_y < by0 && by1 < t.tb_hi_y))
      continue;
    bool ok = true;
    for(int r = 0; r < t.nrow && ok; r++)
    {
      const double ry0 = r == 0 ? t.tb_lo_y : t.row_upper_y[r - 1];
      const double ry1 = r == t.nrow - 1 ? t.tb_hi_y : t.row_upper_y[r];
      const double ay = by0 > ry0 ? by0 : ry0, cy = by1 < ry1 ? by1 : ry1;
      if(!(ay <= cy))
        continue;
      for(int c = 0; c < t.ncell[r] && ok; c++)
      {
        const double rx0 = c == 0 ? t.tb_lo_x : t.cell_upper_x[r][c - 1];
        const double rx1 = c == t.ncell[r] - 1 ? t.tb_hi_x : t.cell_upper_x[r][c];
        const double ax = bx0 > rx0 ? bx0 : rx0, cx = bx1 < rx1 ? bx1 : rx1;
        if(!(ax <= cx))
          continue;
        ok = quadtest_cell_pred(t, r, c, ax, ay) && quadtest_cell_pred(t, r, c, cx, ay) && quadtest_cell_pred(t, r, c, ax, cy) &&
             quadtest_cell_pred(t, r, c, cx, cy);
      }
    }
    found = ok;
  }
  if(!found)
    return;
  // single-precision centre / half width, rounded so the f32 box lies inside the verified box
  const double u = 1.0 / 16777216.0;
  const double mx = fmax(fabs(bx0), fabs(bx1)), my = fmax(fabs(by0), fabs(by1));
  const float cxf = (float)((bx0 + bx1) * 0.5), cyf = (float)((by0 + by1) * 0.5);
  const double hx = fmin((double)cxf - bx0, bx1 - (double)cxf) - 4.0 * u * mx;
  const double hy = fmin((double)cyf - by0, by1 - (double)cyf) - 4.0 * u * my;
  if(!(hx > 0 && hy > 0))
    return;
  t.ib_cx = cxf;
  t.ib_cy = cyf;
  t.ib_hx = __double2float_rd(hx);
  t.ib_hy = __double2float_rd(hy);
}

// ---- filtered point-in-quadrilateral -------------------------------------------------------------------
// f32 image of the test: called once per emitted step by k_frame_logic, after quadtest_init/inner_box.
// T bounds |x|, |y| of every point the filter will see (in-range world points).
__device__ inline void quadfilter_build(QuadFilterDev &f, const QuadTestDev &t, float T, float epsc)
{
  // |w^ - cx| < hx - epsc  =>  |w_ref - cx| < hx (the subtraction rounds down: the accept region only shrinks)
  {
    const bool box = t.ib_hx > 0.f && t.ib_hy > 0.f;
    const float cx = box ? t.ib_cx : (float)((t.tb_lo_x + t.tb_hi_x) * 0.5), cy = box ? t.ib_cy : (float)((t.tb_lo_y + t.tb_hi_y) * 0.5);
    f.ibe = make_float4(cx, cy, box ? __fadd_rd(t.ib_hx, -epsc) : -1.f, box ? __fadd_rd(t.ib_hy, -epsc) : -1.f);
    // |x^ - cx| > Rx with |x^ - x| <= epsc and the subtraction's own rounding (<= 2^-24 (|cx| + T)) implies x outside
    // [lo, hi]: Rx = max(cx - lo, hi - cx) + 2 epsc + 2^-22 (|cx| + T), rounded up. No usable test: infinite box.
    const float inf_ = __int_as_float(0x7f800000);
    const double rx = fmax((double)cx - t.tb_lo_x, t.tb_hi_x - (double)cx) + 2.0 * epsc + 2.4e-7 * (fabs((double)cx) + T);
    const double ry = fmax((double)cy - t.tb_lo_y, t.tb_hi_y - (double)cy) + 2.0 * epsc + 2.4e-7 * (fabs((double)cy) + T);
    f.rj = t.status == 0 ? make_float4(__double2float_ru(rx), __double2float_ru(ry), 0.f, 0.f) : make_float4(inf_, inf_, 0.f, 0.f);
  }
  const float u = 5.9604645e-08f; // 2^-24
  const float inf = __int_as_float(0x7f800000);
  f.ok = t.status == 0;
  f.pad8 = 0;
  f.ib = make_float4(t.ib_cx, t.ib_hx, t.ib_cy, t.ib_hy);
  for(int i = 0; i < 4; i++)
  {
    const SegmentDev &s = t.seg[i];
    // passes <=> isLeft == insideIsLeft <=> (val > 0) == (left_is_pos == inside_is_left)
    const double sg = (s.left_is_pos != 0) == (t.inside_is_left != 0) ? 1.0 : -1.0;
    const double kx = s.steep ? 1.0 : s.k, ky = s.steep ? s.k : 1.0;
    // |v^ - v_ref| <= 2 eps + 4u (T|kx| + T|ky| + |c|); stored with a factor 2 of slack (eps part added at run time)
    f.seg[i] = make_float4((float)(sg * kx), (float)(sg * ky), (float)(sg * s.c),
                           8.f * u * (float)(T * (fabs(kx) + fabs(ky)) + fabs(s.c)) * 1.001f + 1e-30f);
  }
  f.seg[4] = make_float4(0.f, 0.f, 1.f, 0.f);
  f.seg[5] = make_float4(0.f, 0.f, -1.f, 0.f);
  f.bb = make_float4((float)t.tb_lo_x, (float)t.tb_hi_x, (float)t.tb_lo_y, (float)t.tb_hi_y);
  f.row_thr[0] = f.row_thr[1] = inf;
  for(int r = 0; r < 3; r++)
  {
    f.cell_thr[r][0] = f.cell_thr[r][1] = inf;
    for(int c = 0; c < 3; c++)
      f.cell_s[r][c][0] = f.cell_s[r][c][1] = 5;
  }
  if(!f.ok)
    return;
  for(int r = 0; r < t.nrow; r++)
  {
    if(r < t.nrow - 1)
      f.row_thr[r] = (float)t.row_upper_y[r];
    for(int c = 0; c < t.ncell[r]; c++)
    {
      if(c < t.ncell[r] - 1)
        f.cell_thr[r][c] = (float)t.cell_upper_x[r][c];
      const int n = t.cell_nseg[r][c];
      if(n == 0)
        f.cell_s[r][c][0] = f.cell_s[r][c][1] = t.cell_seg[r][c][0] ? 4 : 5;
      else
      {
        f.cell_s[r][c][0] = (unsigned char)t.cell_seg[r][c][0];
        f.cell_s[r][c][1] = n == 2 ? (unsigned char)t.cell_seg[r][c][1] : 4;
      }
    }
  }
}

// f32 evaluation of isPointWithin at (x, y) = single-precision world position with |error| <= eps per coordinate.
// Returns the decision; `uncertain` is set when any comparison came within its margin (then the exact test decides).
// Margins: thresholds and the bounding box are f32-rounded doubles (<= u*T off) compared with x, y (<= eps off):
// 2*eps covers both because eps >= 16u*T (derive_params). Half planes: 3*eps + seg.w (quadfilter_build).
__device__ __forceinline__ bool quadfilter_eval(const QuadFilterDev &f, float x, float y, float eps, bool &uncertain)
{
  const float M = eps + eps;
  const float4 bb = f.bb;
  const float dbb = fminf(fminf(x - bb.x, bb.y - x), fminf(y - bb.z, bb.w - y));
  const float r0 = f.row_thr[0], r1 = f.row_thr[1];
  const int r = (y >= r0 ? 1 : 0) + (y >= r1 ? 1 : 0);
  const float c0 = f.cell_thr[r][0], c1 = f.cell_thr[r][1];
  const int c = (x >= c0 ? 1 : 0) + (x >= c1 ? 1 : 0);
  const float dthr = fminf(fminf(fabsf(y - r0), fabsf(y - r1)), fminf(fabsf(x - c0), fabsf(x - c1)));
  const float4 s0 = f.seg[f.cell_s[r][c][0]], s1 = f.seg[f.cell_s[r][c][1]];
  const float v0 = fmaf(x, s0.x, fmaf(y, s0.y, s0.z)), v1 = fmaf(x, s1.x, fmaf(y, s1.y, s1.z));
  const float m0 = fmaf(3.f, eps, s0.w), m1 = fmaf(3.f, eps, s1.w);
  const bool in = v0 > m0 && v1 > m1, out = v0 < -m0 || v1 < -m1;
  const bool sel = dthr > M; // row / cell selection is certain
  const bool cin = dbb > M && sel && in;
  const bool cout = dbb < -M || (sel && out);
  uncertain = !(cin || cout) || !f.ok;
  return cin;
}

// World z for the per-step mean (calcAverageZ, pointcloud.cpp:574-581) as an unsigned integer: single-precision
// fma chain on coefficients pre-scaled by 2^zshift (|error| <= 4u (S_z m + |b_z|) ~ 1e-6 m worst case, random sign),
// rounded to the nearest integer by adding 1.5*2^23; the 23 mantissa bits are k + 2^22 with k = round(wz * 2^zshift),
// |k| < 2^22 for every in-range point (derive_params picks zshift). Integer sums are order independent, so the
// mean is deterministic; total error of a mean << 1e-6 m against the 1e-4 m tolerance.
#define SSD_ZFIX_BIAS 4194304u
__device__ __forceinline__ unsigned z_fix_u(const DevParams &p, float x, float y, float z)
{
  const float zq = fmaf(p.azf[2], z, fmaf(p.azf[1], y, fmaf(p.azf[0], x, p.bzf)));
  return (unsigned)__float_as_int(zq + 12582912.0f) & 0x7fffffu;
}
