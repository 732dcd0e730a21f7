// ssd_gpu.cu -- context, launch chain and C ABI (include/ssd_gpu.h) of the B200 stair-step geometry path.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false (see build.py). No CPU fallback.
#include "ssd_device.cuh"
#include "ssd_kernels_points.cuh"
#include "ssd_kernels_outline.cuh"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <type_traits>
#include <vector>

#ifndef SSD_PT_ITERS
#define SSD_PT_ITERS 4 // k_transform_bin: 4096 points per block
#endif
#define SSD_TILE_POINTS (SSD_PT_THREADS * 4 * SSD_PT_ITERS)
#define SSD_MAX_STREAMS 4
#define SSD_FUSE_MAX_FRAMES 16 // batches up to this size take the fused (latency) variants of k_transform_bin / k_outline

static thread_local std::string g_create_error;

// ToExternalWorld of one result record (ssd_gpu_get_step_surfaces), taken when the call runs
struct SurfaceXf
{
  double ext_a[4], ext_b[2], ext_z;
};

struct ssd_gpu_ctx
{
  int device = 0;
  int max_frames = 0;
  int chunk_frames = 0;
  int host_chunk_frames = 0;  // chunk of the host-input entry points: small enough that PCIe copies and kernels pipeline
  ssd_gpu_config cfg{};
  ssd_gpu_transform xf{};
  DevParams dp{};
  size_t bm_words = 0;        // words per BEV bitmap
  size_t smem_cap_words = 0;  // dynamic shared memory available to the band (words)
  size_t ol_dyn_smem = 0;
  // blocks per frame of k_outline; they loop over the frame's outlined plateaus. Measured (tools/configs_bench.py): 12 against one
  // block per plateau slot (32): k_outline -7 % at 1024x768 (fewer empty blocks), unchanged at 4096x3072 with 13 outlined plateaus;
  // 8 and 6 lose there (1.15 -> 1.45 / 1.77 ms per 64 frames). SSD_GPU_OUTLINE_GRIDX overrides.
  int outline_gridx = 12;
  bool outline_small = false; // frame size admits the small work area of k_outline (OutlineSharedSmall)
  int n_streams = 2;
  cudaStream_t stream[SSD_MAX_STREAMS]{};
  cudaStream_t copy_stream{};
  // knobs, read once in ssd_gpu_create (DESIGN.md): blocks per frame of the point kernels, small-batch split
  int bpf_l_knob = 0, bpf_q_knob = 0;
  bool no_split_small = false;
  cudaEvent_t ev_start{}, ev_stop{}, ev_h2d0{}, ev_h2d1{};
  cudaEvent_t ev_in_ready[SSD_MAX_STREAMS]{}, ev_in_free[SSD_MAX_STREAMS]{}, ev_chunk_done[SSD_MAX_STREAMS]{};
  FrameDev *d_frames = nullptr;   // max_frames
  FrameOut *d_out = nullptr;      // max_frames
  FrameOut *h_out = nullptr;      // pinned
  OverlayDev ov{};                // drawStairStep projection (ssd_gpu_set_overlay); off by default
  ssd_gpu_overlay *d_ovl = nullptr, *h_ovl = nullptr; // max_frames * SSD_GPU_MAX_STEPS, allocated by ssd_gpu_set_overlay
  unsigned char *d_labels = nullptr; // max_frames * N
  unsigned *d_bev = nullptr; // 2 x chunk_frames * MAX_PLATEAUS * bm_words (per stream)
  void *d_stage[SSD_MAX_STREAMS]{};             // staging of the host-input calls: a chunk of vertices, z16 or float frames
  size_t stage_bytes = 0;                       // ... the bytes each holds: the largest chunk a call has needed
  float *d_xn = nullptr, *d_yn = nullptr;       // deprojection tables: (u - ppx) / fx per column, (v - ppy) / fy per row
  ssd_gpu_intrinsics intr{};                    // intrinsics the tables were built for
  bool risers = false;            // ssd_gpu_set_vertical_faces: k_riser_reduce after the chain
  unsigned char *d_step_labels = nullptr; // max_frames * N, allocated by ssd_gpu_set_step_labels
  bool step_labels = false;       // ssd_gpu_set_step_labels: k_quad_reduce's STEPS variant writes d_step_labels
  bool step_labels_last = false;  // the last accepted process call wrote them
  SurfaceDev *d_surf = nullptr;   // max_frames * SSD_GPU_MAX_STEPS, allocated by ssd_gpu_set_step_surfaces
  bool surfaces = false;          // ssd_gpu_set_step_surfaces: k_step_surface after the chain
  bool surfaces_last = false;     // the last accepted process call ran it
  std::vector<SurfaceXf> surf_xf; // per record of the last call: the ToExternalWorld its surfaces are reported through
  int pt_blocks_target = 0;       // blocks per launch of the tile-looping point kernels
  int n_frames_last = 0;
  int flags_last = 0;
  ssd_gpu_timing timing{};
  std::string err;
  // single-stage scratch
  unsigned char *d_img = nullptr; // a BEV image (W x H of the BEV)
  // optional per-kernel events (SSD_FLAG_STAGE_TIMING): (SSD_GPU_N_STAGES + 1) per chunk
  std::vector<cudaEvent_t> stage_ev;
  int stage_chunks = 0;
  float stage_ms[SSD_GPU_N_STAGES]{};
  int stage_launches[SSD_GPU_N_STAGES]{};
  // camera table (ssd_gpu_set_cameras): per camera the derived parameters, the overlay projection and the deprojection tables
  int n_cameras = 0;
  std::vector<DevParams> cam_dp;         // host copies (filter bounds for ssd_gpu_get_stats)
  std::vector<unsigned char> cam_depth_ok; // intrinsics admit depth input
  DevParams *d_cam_dp = nullptr;
  OverlayDev *d_cam_ov = nullptr;
  float *d_cam_xn = nullptr, *d_cam_yn = nullptr, *d_cam_unit = nullptr;
  int *d_cam_of_frame = nullptr;         // max_frames: camera of each frame of the current call
  // lenses (ssd_gpu_set_distortion / ssd_gpu_set_cameras_ex): one per-pixel ray table per distinct distorted lens
  ssd_gpu_distortion lens{};             // lens of the plain calls (model NONE: pin-hole)
  ssd_gpu_distortion *d_lens = nullptr;  // ... its device copy (overlay)
  float2 *d_ray = nullptr;               // ray table of the plain calls' lens, built for ray_intr
  ssd_gpu_intrinsics ray_intr{};
  bool ray_valid = false;
  std::vector<float2 *> cam_rays;        // distinct ray tables of the camera table (only when one of its cameras is distorted)
  std::vector<unsigned char> cam_distorted;
  bool cams_distorted = false;           // some camera of the table has a distorted lens
  const float2 **d_cam_ray = nullptr;    // n_cameras: ray table of each camera
  ssd_gpu_distortion *d_cam_lens = nullptr; // n_cameras
  double stats_eps0 = 0, stats_eps1 = 0; // filter bounds of the last call (largest over its cameras)
  // frame groups (ssd_gpu_process_groups_*): per frame its group, per group its first frame, member count and largest epsc
  int *d_grp_of_frame = nullptr;         // max_frames
  int2 *d_grp_members = nullptr;         // max_frames
  float *d_grp_epsc = nullptr;           // max_frames
  std::vector<int> grp_of_frame;         // host copy of the last call's (empty after a call without groups)
  std::vector<int2> grp_members;
  std::vector<float> grp_epsc;
};

// the result record (FrameDev / FrameOut) of a frame of the last call: its group's in a group call
static int frame_record(const ssd_gpu_ctx *ctx, int frame)
{
  return ctx->grp_of_frame.empty() ? frame : ctx->grp_of_frame[frame];
}
static int n_records_last(const ssd_gpu_ctx *ctx)
{
  return ctx->grp_of_frame.empty() || ctx->n_frames_last <= 0 ? ctx->n_frames_last : (int)ctx->grp_members.size();
}

#define CK(call)                                                                                         \
  do                                                                                                     \
  {                                                                                                      \
    cudaError_t e_ = (call);                                                                             \
    if(e_ != cudaSuccess)                                                                                \
    {                                                                                                    \
      ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                                     \
      return SSD_E_CUDA;                                                                                 \
    }                                                                                                    \
  } while(0)

static int fail(ssd_gpu_ctx *ctx, int code, const std::string &msg)
{
  if(ctx)
    ctx->err = msg;
  else
    g_create_error = msg;
  return code;
}

// The largest frame: N <= 9348 * 5108 points (the largest frame of a context whose BEV is its frame size), which keeps the
// 32-bit point counters of a frame group exact (DESIGN.md, frame groups)
#define SSD_MAX_FRAME_POINTS (9348LL * 5108LL)

// ProcessingConfiguration / Projection2D (pointcloud.cpp:60-106) for frames of c.width x c.height pixels and a BEV image of bw x bh
// pixels: the frame fields (N, FW, FH, tiles_per_frame) address the input, every image-pixel field is the BEV's
static int derive_params(const ssd_gpu_config &c, int bw, int bh, const ssd_gpu_transform &t, DevParams &d)
{
  memset(&d, 0, sizeof(d));
  if(c.width <= 0 || c.height <= 0 || bw <= 0 || bh <= 0 || !(c.x_max > c.x_min) || !(c.y_max > c.y_min) || !(c.z_max > c.z_min) ||
     !(c.height_interval > 0))
    return SSD_E_INVALID_ARG;
  const long long n_frame = (long long)c.width * c.height;
  d.W = bw;
  d.H = bh;
  d.N = (int)std::min<long long>(n_frame, INT32_MAX); // (refused below when it exceeds SSD_MAX_FRAME_POINTS)
  d.FW = c.width;
  d.FH = c.height;
  d.wpr = (int)(((long long)bw + 31) / 32); // (64-bit: a BEV past the limits is refused below, after these are derived)
  d.hir = 1.0 / c.height_interval;
  d.min_height = (uint16_t)((c.min_height_above_ground - c.z_min) * d.hir);
  d.min_img_y_extent = (int)(c.min_step_depth * bh / (c.y_max - c.y_min));
  d.x_to_image = bw / (c.x_max - c.x_min);
  d.y_to_image = bh / (c.y_max - c.y_min);
  d.x_to_world = 1 / d.x_to_image;
  d.y_to_world = 1 / d.y_to_image;
  d.xy_ratio = d.x_to_image / d.y_to_image;
  d.n_bins = (int)((size_t)((c.z_max - c.z_min) * d.hir) + 1);
  d.min_peak_points = c.min_peak_points;
  d.bev_slots = SSD_GPU_MAX_PLATEAUS;
  d.tiles_per_frame = (int)(((long long)d.N + SSD_TILE_POINTS - 1) / SSD_TILE_POINTS);
  memcpy(d.a, t.a, sizeof(d.a));
  memcpy(d.b, t.b, sizeof(d.b));
  memcpy(d.ext_a, t.ext_a, sizeof(d.ext_a));
  memcpy(d.ext_b, t.ext_b, sizeof(d.ext_b));
  d.ext_z = t.ext_z;
  d.x_min = c.x_min;
  d.x_max = c.x_max;
  d.y_min = c.y_min;
  d.y_max = c.y_max;
  d.z_min = c.z_min;
  d.z_max = c.z_max;
  // single-precision world coordinates (k_label_bev / k_quad_reduce): everything rounded so the bound stays an upper bound
  {
    const double u = 1.0 / 16777216.0; // 2^-24
    double e0 = 0, e1 = 0, T = 0;
    const double lo[3] = { c.x_min, c.y_min, c.z_min }, hi[3] = { c.x_max, c.y_max, c.z_max };
    for(int i = 0; i < 3; i++)
    {
      const double S = std::fabs(t.a[i * 3]) + std::fabs(t.a[i * 3 + 1]) + std::fabs(t.a[i * 3 + 2]);
      e0 = std::max(e0, std::fabs(t.b[i]));
      e1 = std::max(e1, S);
      T = std::max({ T, std::fabs(lo[i]), std::fabs(hi[i]) });
      for(int j = 0; j < 3; j++)
        d.af[i * 3 + j] = (float)t.a[i * 3 + j];
      d.bf[i] = (float)t.b[i];
    }
    // proven bound: 5u*(|b| + S*m) + 8u*T ; used: twice that, rounded up
    d.E0 = (float)((10.0 * u * e0 + 16.0 * u * T) * 1.001) + 1e-12f;
    d.E1 = (float)(10.0 * u * e1 * 1.001);
    // range-scaled rows for point_code_scaled: v_i = (w_i - c_i)/h_i
    {
      double S1 = 0, B1 = 0, X1 = 0;
      for(int i = 0; i < 3; i++)
      {
        const double ci = (lo[i] + hi[i]) * 0.5, hi_ = (hi[i] - lo[i]) * 0.5;
        double Si = 0;
        for(int j = 0; j < 3; j++)
        {
          d.sa[i * 3 + j] = (float)(t.a[i * 3 + j] / hi_);
          Si += std::fabs(t.a[i * 3 + j]) / hi_;
        }
        d.sb[i] = (float)((t.b[i] - ci) / hi_);
        S1 = std::max(S1, Si);
        B1 = std::max(B1, std::fabs(t.b[i] - ci) / hi_ + 1.0);
        X1 = std::max(X1, (std::fabs(t.b[i]) + std::fabs(ci)) / hi_);
      }
      d.E1s = (float)(8.0 * u * S1 * 1.001);
      d.E0s = (float)((8.0 * u * B1 + 1e-15 * X1) * 1.001);
      const double G = (c.z_max - c.z_min) * 0.5 * d.hir;
      d.Gf = (float)G;
      d.Gm = (float)(G - 0.5);
      d.Gup = (float)(G * 1.001);
      // |u_f - (t_ref - 0.5)| <= G eps + [f32 rounding of G, G - 0.5: 2u G (|v|+1)] + [fma rounding u (n_bins + 1)] + f64 roundings
      const double dbin = 8.0 * u * (2.0 * G + d.n_bins + 2.0) + 1e-9;
      d.thr0 = (float)((0.5 - dbin) * 0.9999);
    }
    // per-step z sum in 2^-zshift m units: |wz| * 2^zshift < 2^22 for every in-range point
    {
      const double zabs = std::max(std::fabs(c.z_min), std::fabs(c.z_max)) * 1.01 + 0.01;
      int sh = 0;
      while(sh < 30 && zabs * std::ldexp(1.0, sh + 1) < 4194304.0)
        sh++;
      d.zshift = sh;
      for(int j = 0; j < 3; j++)
        d.azf[j] = (float)std::ldexp((double)(float)t.a[6 + j], sh);
      d.bzf = (float)std::ldexp((double)(float)t.b[2], sh);
    }
    // BEV pixel in single precision (fast_pixel): u = sx*(wx - x_min), v = sy*(y_max - wy) folded into one fma chain.
    // |u^ - u_ref| <= 4u (S'm + |b'|) (coefficient rounding + three fma roundings; the reference's own f64
    // roundings are ~2^-50 of that); used: 6u, i.e. a factor 1.5 of slack, plus an absolute 1e-6 px. (Half of all
    // phase-B warp steps of k_label_bev see an uncertain pixel at 10u: the bound's slack is paid in divergence.)
    const double sx = d.x_to_image, sy = d.y_to_image;
    double Su = 0, Sv = 0;
    for(int j = 0; j < 3; j++)
    {
      d.au[j] = (float)(t.a[j] * sx);
      d.av[j] = (float)(-t.a[3 + j] * sy);
      Su += std::fabs(t.a[j] * sx);
      Sv += std::fabs(t.a[3 + j] * sy);
    }
    const double bu = (t.b[0] - c.x_min) * sx, bv = (c.y_max - t.b[1]) * sy;
    d.bu = (float)bu;
    d.bv = (float)bv;
    d.Eu1 = (float)(6.0 * u * Su * 1.001);
    d.Eu0 = (float)(6.0 * u * std::fabs(bu) * 1.001 + 1e-6);
    d.Ev1 = (float)(6.0 * u * Sv * 1.001);
    d.Ev0 = (float)(6.0 * u * std::fabs(bv) * 1.001 + 1e-6);
    d.Tf = (float)(std::max({ std::fabs(c.x_min), std::fabs(c.x_max), std::fabs(c.y_min), std::fabs(c.y_max) }) * 1.001 + 1e-3);
    // Constant bounds for points that are known to be in range (everything k_label_bev / k_quad_reduce touch):
    // p = A^-1 (w - b), so max|p| <= max_i sum_j |A^-1_ij| (T_j + |b_j|) =: Mmax (1 % slack). A singular A gives
    // infinite bounds: every decision then goes to the exact pass.
    {
      const double *a = t.a;
      const double det = a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) + a[2] * (a[3] * a[7] - a[4] * a[6]);
      double Mmax = INFINITY;
      if(std::fabs(det) > 1e-12)
      {
        const double inv[9] = { (a[4] * a[8] - a[5] * a[7]) / det, (a[2] * a[7] - a[1] * a[8]) / det, (a[1] * a[5] - a[2] * a[4]) / det,
                                (a[5] * a[6] - a[3] * a[8]) / det, (a[0] * a[8] - a[2] * a[6]) / det, (a[2] * a[3] - a[0] * a[5]) / det,
                                (a[3] * a[7] - a[4] * a[6]) / det, (a[1] * a[6] - a[0] * a[7]) / det, (a[0] * a[4] - a[1] * a[3]) / det };
        Mmax = 0;
        for(int i = 0; i < 3; i++)
        {
          double r = 0;
          for(int j = 0; j < 3; j++)
            r += std::fabs(inv[i * 3 + j]) * (std::max(std::fabs(lo[j]), std::fabs(hi[j])) + std::fabs(t.b[j]));
          Mmax = std::max(Mmax, r);
        }
        Mmax *= 1.01;
      }
      d.epsc = (float)((double)d.E1 * Mmax * 1.0001) + d.E0;
      d.euc = (float)((double)d.Eu1 * Mmax * 1.0001) + d.Eu0;
      d.evc = (float)((double)d.Ev1 * Mmax * 1.0001) + d.Ev0;
      d.hu = 0.5f - d.euc - 9.5367431640625e-07f; // infinite / NaN bounds make every comparison false: exact pass
      d.hv = 0.5f - d.evc - 9.5367431640625e-07f;
    }
    {
      // ground BEV columns W/2 - 2 + 50 j + {0..4}: f32 pre-filter with a conservative margin (pixel error of the f32
      // world x: epsc * sx, plus the rounding of the filter's own arithmetic)
      const double gd = ((double)d.epsc * sx * 1.0001 + 8.0 * bw / 16777216.0 + 1e-3) / 50.0;
      d.gcol_a = (float)(sx / 50.0);
      d.gcol_b = (float)((-c.x_min * sx - (bw / 2 - 2)) / 50.0);
      d.gcol_lo = (float)(0.1 + gd);
      d.gcol_hi = (float)(1.0 - gd);
      d.gcol_tmax = (float)((bw - 2 - (bw / 2 - 2)) / 50.0 - gd);
    }
    for(int j = 0; j < 3; j++)
    {
      d.axy2[j] = f2_pack_bits(d.af[j], d.af[3 + j]);
      d.sxy2[j] = f2_pack_bits(d.sa[j], d.sa[3 + j]);
      d.auv2[j] = f2_pack_bits(d.au[j], d.av[j]);
    }
    d.bxy2 = f2_pack_bits(d.bf[0], d.bf[1]);
    d.sbxy2 = f2_pack_bits(d.sb[0], d.sb[1]);
    d.buv2 = f2_pack_bits(d.bu, d.bv);
  }
  if(d.n_bins < 3 || d.n_bins > SSD_GPU_MAX_BINS)
    return SSD_E_RANGE;
  if(n_frame % 16 != 0)
    return SSD_E_INVALID_ARG; // vertices are loaded four at a time (three 16-byte loads), labels sixteen at a time
  // the BEV: column scans, front-edge line points and vertical probes of the outline (ssd_kernels_outline.cuh)
  if(bw / 25 + 4 > SSD_MAX_SCANS || bw / 50 + 6 > SSD_MAX_LINE_PTS || bh / 10 + 2 > SSD_MAX_VPTS)
    return SSD_E_RANGE;
  if(n_frame > SSD_MAX_FRAME_POINTS)
    return SSD_E_RANGE;
  return SSD_OK;
}

// ---------------------------------------------------------------------------------------------
// depth frame -> vertices: the deprojection the reference delegates to rs2::pointcloud::calculate
// (pointcloud.cpp:138; pin-hole model of rs2_deproject_pixel_to_point / camera.h:99-116). Single-rounded f32
// operations in the order of ssd_deproject_pixel (scene_model.h), so the vertices are bit-identical to the host's.
// ---------------------------------------------------------------------------------------------
__global__ void k_deproject_tables(int W, int H, ssd_gpu_intrinsics in, float *__restrict__ xn, float *__restrict__ yn)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if(i < W)
    xn[i] = __fdiv_rn(__fsub_rn((float)i, in.ppx), in.fx);
  if(i < H)
    yn[i] = __fdiv_rn(__fsub_rn((float)i, in.ppy), in.fy);
}

// the same tables for every camera of a camera table: grid = (ceil(max(W, H) / 256), min(n_cameras, 65535)), cameras grid-strided
__global__ void k_deproject_tables_cams(int W, int H, const ssd_gpu_camera *__restrict__ cams, int n_cameras, float *__restrict__ xn,
                                        float *__restrict__ yn)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  for(int c = blockIdx.y; c < n_cameras; c += gridDim.y)
  {
    const ssd_gpu_intrinsics in = cams[c].intr;
    if(i < W)
      xn[(size_t)c * W + i] = __fdiv_rn(__fsub_rn((float)i, in.ppx), in.fx);
    if(i < H)
      yn[(size_t)c * H + i] = __fdiv_rn(__fsub_rn((float)i, in.ppy), in.fy);
  }
}

// 4 consecutive pixels per thread: one 8-byte load, three 16-byte stores. grid = (ceil(N/4/256), frames). W % 4 == 0.
__global__ void __launch_bounds__(256) k_deproject(int W, int N, float depth_unit, const float *__restrict__ xn, const float *__restrict__ yn,
                                                   const uint16_t *__restrict__ depth, float *__restrict__ xyz)
{
  const int q = blockIdx.x * blockDim.x + threadIdx.x; // quad of pixels within the frame
  if(q * 4 >= N)
    return;
  const size_t fbase = (size_t)blockIdx.y * N;
  const uint2 d = __ldg(reinterpret_cast<const uint2 *>(depth + fbase) + q);
  const int i0 = q * 4, v = i0 / W, u = i0 - v * W;
  const float4 x4 = __ldg(reinterpret_cast<const float4 *>(xn + u));
  const float y = __ldg(yn + v);
  const float z0 = __fmul_rn((float)(d.x & 0xffffu), depth_unit), z1 = __fmul_rn((float)(d.x >> 16), depth_unit);
  const float z2 = __fmul_rn((float)(d.y & 0xffffu), depth_unit), z3 = __fmul_rn((float)(d.y >> 16), depth_unit);
  float4 *dst = reinterpret_cast<float4 *>(xyz + (fbase + (size_t)i0) * 3);
  dst[0] = make_float4(__fmul_rn(z0, x4.x), __fmul_rn(z0, y), z0, __fmul_rn(z1, x4.y));
  dst[1] = make_float4(__fmul_rn(z1, y), z1, __fmul_rn(z2, x4.z), __fmul_rn(z2, y));
  dst[2] = make_float4(z2, __fmul_rn(z3, x4.w), __fmul_rn(z3, y), z3);
}

// Ray table of a lens (include/ssd_gpu.h, ssd_gpu_distortion): pixel (u, v) -> (x, y) of its ray at z = 1, x0 and y0 computed as
// k_deproject_tables computes xn[u], yn[v] (so a pin-hole lens's table holds exactly those values), then the model's deprojection.
// *bad is set when a ray is not finite (P^-1 diverged). grid-stride over the W*H pixels.
__global__ void k_lens_rays(int W, int H, ssd_gpu_intrinsics in, ssd_gpu_distortion d, float2 *__restrict__ ray, unsigned *__restrict__ bad)
{
  const size_t N = (size_t)W * H;
  for(size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < N; i += (size_t)gridDim.x * blockDim.x)
  {
    const int v = (int)(i / W), u = (int)(i - (size_t)v * W);
    const float x0 = __fdiv_rn(__fsub_rn((float)u, in.ppx), in.fx), y0 = __fdiv_rn(__fsub_rn((float)v, in.ppy), in.fy);
    float x, y;
    ssd_lens_deproject(&d, x0, y0, &x, &y);
    ray[i] = make_float2(x, y);
    if(!isfinite(x) || !isfinite(y))
      *bad = 1u;
  }
}

// k_deproject with a ray table: 4 consecutive pixels per thread. grid = (ceil(N/4/256), frames).
__global__ void __launch_bounds__(256) k_deproject_lens(int N, float depth_unit, const float2 *__restrict__ ray, const uint16_t *__restrict__ depth,
                                                        float *__restrict__ xyz)
{
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if(q * 4 >= N)
    return;
  const size_t fbase = (size_t)blockIdx.y * N;
  const uint2 d = __ldg(reinterpret_cast<const uint2 *>(depth + fbase) + q);
  const float4 r01 = __ldg(reinterpret_cast<const float4 *>(ray) + (size_t)q * 2), r23 = __ldg(reinterpret_cast<const float4 *>(ray) + (size_t)q * 2 + 1);
  const float z0 = __fmul_rn((float)(d.x & 0xffffu), depth_unit), z1 = __fmul_rn((float)(d.x >> 16), depth_unit);
  const float z2 = __fmul_rn((float)(d.y & 0xffffu), depth_unit), z3 = __fmul_rn((float)(d.y >> 16), depth_unit);
  float4 *dst = reinterpret_cast<float4 *>(xyz + (fbase + (size_t)q * 4) * 3);
  dst[0] = make_float4(__fmul_rn(z0, r01.x), __fmul_rn(z0, r01.y), z0, __fmul_rn(z1, r01.z));
  dst[1] = make_float4(__fmul_rn(z1, r01.w), z1, __fmul_rn(z2, r23.x), __fmul_rn(z2, r23.y));
  dst[2] = make_float4(z2, __fmul_rn(z3, r23.z), __fmul_rn(z3, r23.w), z3);
}

// ---------------------------------------------------------------------------------------------
// single-stage kernels behind ssd_gpu_detect_outline / _front_edge / _points_in_quad / _camera_to_world: the host classes
// Segmentation, QuadrilateralTest and CameraToWorld call them (same device functions as the chain)
// ---------------------------------------------------------------------------------------------
__global__ void k_pack_bitmap(const __grid_constant__ DevParams p, const unsigned char *__restrict__ img, unsigned *__restrict__ bm)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x; // word index
  if(i >= p.H * p.wpr)
    return;
  const int y = i / p.wpr, w = i - y * p.wpr;
  unsigned v = 0;
  for(int b = 0; b < 32; b++)
  {
    const int x = w * 32 + b;
    if(x < p.W && img[(size_t)y * p.W + x])
      v |= 1u << b;
  }
  bm[i] = v;
}

__global__ void k_single_setup_plateau(FrameDev *frames, int H)
{
  FrameDev &F = frames[0];
  F.n_plateaus = 1;
  F.first_outlined = 0;
  F.ground_index = -1;
  F.first_valid = -1;
  F.status = 0;
  PlateauDev &P = F.plat[0];
  P.outlined = 1;
  P.valid = 0;
  P.row_min = 0;
  P.row_max = H - 1;
}

__global__ void __launch_bounds__(SSD_OL_THREADS) k_single_front_edge(const __grid_constant__ DevParams p, unsigned *__restrict__ bev,
                                                                     size_t smem_cap_words, double *out)
{
  extern __shared__ __align__(16) unsigned s_words[];
  __shared__ OutlineShared S;
  __shared__ Band bd;
  __shared__ int s_smem_path;
  const int tid = threadIdx.x;
  if(tid == 0)
    s_smem_path = band_setup(p, bd, 0, p.H - 1, s_words, smem_cap_words, bev);
  __syncthreads();
  if(s_smem_path)
    band_stage(p, s_words, bd, bev, tid, SSD_OL_THREADS);
  P2d l, r;
  int valid;
  detect_front_edge_block(p, bd, S, l, r, valid, tid, SSD_OL_THREADS);
  if(!s_smem_path)
  {
    __syncthreads();
    band_clear_global(p, bd, bev, tid, SSD_OL_THREADS);
  }
  if(tid == 0)
  {
    out[0] = l.x;
    out[1] = l.y;
    out[2] = r.x;
    out[3] = r.y;
    out[4] = valid;
  }
}

__global__ void k_single_points_in_quad(const double *__restrict__ quad, const double *__restrict__ xy, int n, unsigned char *__restrict__ inside,
                                      int *ctor_status)
{
  __shared__ QuadTestDev qt;
  if(threadIdx.x == 0)
  {
    P2d q[4];
    for(int i = 0; i < 4; i++)
    {
      q[i].x = quad[i * 2];
      q[i].y = quad[i * 2 + 1];
    }
    quadtest_init(qt, q);
    if(blockIdx.x == 0)
      *ctor_status = qt.status;
  }
  __syncthreads();
  for(int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    inside[i] = qt.status ? 0 : (unsigned char)quadtest_within(qt, xy[i * 2], xy[i * 2 + 1]);
}

__global__ void k_single_camera_to_world(const __grid_constant__ DevParams p, const float *__restrict__ xyz, int n, double *__restrict__ world)
{
  for(int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
  {
    double x, y, z;
    camera_to_world(p, xyz[i * 3], xyz[i * 3 + 1], xyz[i * 3 + 2], x, y, z);
    world[i * 3] = x;
    world[i * 3 + 1] = y;
    world[i * 3 + 2] = z;
  }
}

// Pass 1 (k_transform_bin): packed vertices through the kernel's bulk-copy staging, depth frames (SrcDepthT, SrcLensT) from registers
template<bool FUSE, class CAM>
static void launch_transform_bin(const dim3 &grid, cudaStream_t st, const DevParams &p, const SrcVertices &src, unsigned char *labels,
                                 FrameDev *frames, const CAM &cam)
{
  k_transform_bin<SSD_PT_ITERS, FUSE, CAM><<<grid, SSD_PT_THREADS, SSD_PT_ITERS * SSD_TB_STAGE_BYTES, st>>>(p, src.xyz, labels, frames, cam);
}
template<bool FUSE, class SRC, class CAM>
static void launch_transform_bin(const dim3 &grid, cudaStream_t st, const DevParams &p, const SRC &src, unsigned char *labels, FrameDev *frames,
                                 const CAM &cam)
{
  k_transform_bin_z16<SSD_PT_ITERS, FUSE, SRC, CAM><<<grid, SSD_PT_THREADS, 0, st>>>(p, src, labels, frames, cam);
}

// The classic chain: k_transform_bin -> k_peaks -> k_label_bev -> k_outline -> k_frame_logic -> k_quad_reduce -> k_finalize
// (+ k_riser_reduce), for one chunk of frames on stream s. SRC: where the points come from (SrcVertices, SrcDepthT, SrcLensT), its
// input pointer the chunk's. CAM = NoCam: every frame with the context's own camera; CamTable: each frame with its camera's
// parameters (camera calls); GroupTable: as CamTable, with the frames of each group accumulated into one record (group calls).
// OL: the outline work area of the frame size (OutlineSharedSmall, OutlineShared).
// Records (FrameDev, FrameOut, BEV slots): rec0 is the launch's first within the call, nr their number (frames, or groups).
// ov_lens: the lenses the overlay projects through (k_finalize), else nullptr: the pin-hole.
template<class OL, class SRC, class CAM>
static int launch_classic(ssd_gpu_ctx *ctx, int s, const SRC &src, int frame0, int nf, int rec0, int nr, int *launches, cudaEvent_t *ev,
                          const CAM &cam, const ssd_gpu_distortion *ov_lens)
{
#define STAGE_EV(i)                         \
  do                                        \
  {                                         \
    if(ev)                                  \
      CK(cudaEventRecord(ev[i], st));       \
  } while(0)
  const DevParams &p = ctx->dp;
  cudaStream_t st = ctx->stream[s];
  FrameDev *frames = ctx->d_frames + rec0;
  unsigned char *labels = ctx->d_labels + (size_t)frame0 * p.N;
  unsigned *bev = ctx->d_bev + (size_t)s * ctx->chunk_frames * SSD_GPU_MAX_PLATEAUS * ctx->bm_words;
  const dim3 gpt(p.tiles_per_frame, nf);
  // k_label_bev / k_quad_reduce: each block loops over tiles of its frame; enough blocks for ~6 waves of the GPU
  const int tiles2 = (p.N + SSD_WT_PX * SSD_PT_WARPS - 1) / (SSD_WT_PX * SSD_PT_WARPS); // at least one warp-tile per warp
  const int bpf = std::max(1, std::min(tiles2, (ctx->pt_blocks_target + nf - 1) / nf));
  const int bpf_l = ctx->bpf_l_knob > 0 ? std::min(tiles2, ctx->bpf_l_knob) : bpf, bpf_q = ctx->bpf_q_knob > 0 ? std::min(tiles2, ctx->bpf_q_knob) : bpf;
  const dim3 gpt2l(bpf_l, nf), gpt2q(bpf_q, nf);
  ssd_gpu_overlay *ovl = ctx->d_ovl ? ctx->d_ovl + (size_t)frame0 * SSD_GPU_MAX_STEPS : nullptr;
  // small batches (the reference's real use is one frame per call): the last block of a frame in k_transform_bin evaluates the
  // peaks and the last block in k_outline the frame logic -- five launches instead of seven. Group calls take the seven
  // (their blocks do not count a frame's completion).
  constexpr bool FUSABLE = !std::is_same<CAM, GroupTable>::value;
  const bool fused = FUSABLE && nf <= SSD_FUSE_MAX_FRAMES && !ev;
  STAGE_EV(0);
  if(!fused)
    launch_transform_bin<false>(gpt, st, p, src, labels, frames, cam);
  else if constexpr(FUSABLE)
    launch_transform_bin<true>(gpt, st, p, src, labels, frames, cam);
  STAGE_EV(1);
  if(!fused)
    k_peaks<<<nr, 32, 0, st>>>(p, frames, nr);
  STAGE_EV(2);
  k_label_bev<SRC, CAM><<<gpt2l, SSD_PT_THREADS, 0, st>>>(p, src, labels, frames, bev, ctx->bm_words, cam);
  STAGE_EV(3);
  // the unfused k_outline reads configuration fields only: one kernel for every camera type
  if(!fused)
    k_outline<OL><<<dim3(ctx->outline_gridx, nr), OL::THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words);
  else if constexpr(FUSABLE)
    k_outline<OL, true, CAM><<<dim3(ctx->outline_gridx, nf), OL::THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words, cam);
  STAGE_EV(4);
  if(!fused)
    k_frame_logic<CAM><<<nr, 32, 0, st>>>(p, frames, nr, cam);
  STAGE_EV(5);
  const auto quad_reduce = [&](auto so) {
    constexpr bool STEPS = std::is_same<decltype(so), StepLabelsOut<true>>::value;
    k_quad_reduce<SRC, CAM, STEPS><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, src, labels, frames, bev, ctx->bm_words, cam, so);
  };
  if(ctx->step_labels)
  {
    // step labels: the chunk's slice starts as SSD_STEP_LABEL_NONE (words without counted points, labels outside quad_amask and
    // frames without steps are never written by k_quad_reduce). The memset is part of the quad_reduce stage's time and is not
    // counted in timing.n_launches (a copy-engine / driver fill, not one of the chain's kernels).
    unsigned char *steps = ctx->d_step_labels + (size_t)frame0 * p.N;
    CK(cudaMemsetAsync(steps, SSD_STEP_LABEL_NONE, (size_t)nf * p.N, st));
    quad_reduce(StepLabelsOut<true>{ steps });
  }
  else
    quad_reduce(StepLabelsOut<false>());
  STAGE_EV(6);
  // k_finalize runs SSD_OL_THREADS on either work area
  k_finalize<OL, CAM><<<nr, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + rec0, bev, ctx->bm_words, ctx->smem_cap_words, ctx->ov,
                                                                   ovl, ov_lens, cam);
  STAGE_EV(7);
#undef STAGE_EV
  *launches += fused ? SSD_GPU_N_STAGES - 2 : SSD_GPU_N_STAGES;
  if(ctx->risers)
  {
    // optional fourth pass: vertical faces from the remainder (labels are final once the chain's label kernel has run)
    k_riser_reduce<SRC, CAM><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, src, labels, frames, cam);
    *launches += 1;
  }
  if(ctx->surfaces)
  {
    // optional pass: step surfaces from the step labels k_quad_reduce wrote. The memset clears the chunk's records (not counted in
    // timing.n_launches, like the step labels' memset).
    SurfaceDev *surf = ctx->d_surf + (size_t)rec0 * SSD_GPU_MAX_STEPS;
    CK(cudaMemsetAsync(surf, 0, sizeof(SurfaceDev) * SSD_GPU_MAX_STEPS * (size_t)nr, st));
    k_step_surface<SRC, CAM><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, src, ctx->d_step_labels + (size_t)frame0 * p.N, frames, surf, cam);
    *launches += 1;
  }
  CK(cudaGetLastError());
  return SSD_OK;
}

// A chunk's source and camera: the call's, with the chunk's input (the caller's frames or the staging buffer they were copied to)
// and, in camera and group calls, its first frame and first group.
static SrcVertices chunk_src(SrcVertices s, const void *in)
{
  s.xyz = static_cast<const float *>(in);
  return s;
}
template<class SRC>
static SRC chunk_src(SRC s, const void *in)
{
  s.depth = static_cast<decltype(s.depth)>(in);
  return s;
}
static NoCam chunk_cam(NoCam c, int, int)
{
  return c;
}
static CamTable chunk_cam(CamTable c, int frame0, int)
{
  c.frame0 = frame0;
  return c;
}
static GroupTable chunk_cam(GroupTable g, int frame0, int rec0)
{
  g.cams.frame0 = frame0;
  g.group0 = rec0;
  return g;
}

// The dynamic work area of the outline kernels a chain of camera type CAM launches with a dynamic band (launch_classic): the fused
// k_outline (not in group calls) and k_finalize, on both work areas.
template<class CAM>
static void allow_outline_smem(int dyn)
{
  const auto allow = [dyn](auto kernel) { cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, dyn); };
  if constexpr(!std::is_same<CAM, GroupTable>::value)
  {
    allow(k_outline<OutlineSharedSmall, true, CAM>);
    allow(k_outline<OutlineShared, true, CAM>);
  }
  allow(k_finalize<OutlineSharedSmall, CAM>);
  allow(k_finalize<OutlineShared, CAM>);
}

extern "C"
{

int ssd_gpu_device_count(void)
{
  int n = 0;
  if(cudaGetDeviceCount(&n) != cudaSuccess)
    return 0;
  return n;
}

const char *ssd_gpu_last_error(const ssd_gpu_ctx *ctx)
{
  return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

void ssd_gpu_destroy(ssd_gpu_ctx *ctx)
{
  if(!ctx)
    return;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  cudaFree(ctx->d_frames);
  cudaFree(ctx->d_out);
  cudaFreeHost(ctx->h_out);
  cudaFree(ctx->d_ovl);
  cudaFreeHost(ctx->h_ovl);
  cudaFree(ctx->d_labels);
  cudaFree(ctx->d_step_labels);
  cudaFree(ctx->d_surf);
  cudaFree(ctx->d_bev);
  cudaFree(ctx->d_img);
  cudaFree(ctx->d_xn);
  cudaFree(ctx->d_yn);
  cudaFree(ctx->d_cam_dp);
  cudaFree(ctx->d_cam_ov);
  cudaFree(ctx->d_cam_xn);
  cudaFree(ctx->d_cam_yn);
  cudaFree(ctx->d_cam_unit);
  cudaFree(ctx->d_cam_of_frame);
  cudaFree(ctx->d_grp_of_frame);
  cudaFree(ctx->d_grp_members);
  cudaFree(ctx->d_grp_epsc);
  for(float2 *t : ctx->cam_rays)
    cudaFree(t);
  cudaFree(ctx->d_cam_ray);
  cudaFree(ctx->d_cam_lens);
  cudaFree(ctx->d_ray);
  cudaFree(ctx->d_lens);
  for(int i = 0; i < SSD_MAX_STREAMS; i++)
  {
    cudaFree(ctx->d_stage[i]);
    if(ctx->stream[i])
      cudaStreamDestroy(ctx->stream[i]);
    if(ctx->ev_in_ready[i])
      cudaEventDestroy(ctx->ev_in_ready[i]);
    if(ctx->ev_in_free[i])
      cudaEventDestroy(ctx->ev_in_free[i]);
    if(ctx->ev_chunk_done[i])
      cudaEventDestroy(ctx->ev_chunk_done[i]);
  }
  if(ctx->copy_stream)
    cudaStreamDestroy(ctx->copy_stream);
  for(cudaEvent_t e : { ctx->ev_start, ctx->ev_stop, ctx->ev_h2d0, ctx->ev_h2d1 })
    if(e)
      cudaEventDestroy(e);
  for(cudaEvent_t e : ctx->stage_ev)
    cudaEventDestroy(e);
  delete ctx;
}

int ssd_gpu_create(const ssd_gpu_config *cfg, const ssd_gpu_transform *xf, int device, int max_frames, ssd_gpu_ctx **out)
{
  if(!cfg)
    return fail(nullptr, SSD_E_INVALID_ARG, "ssd_gpu_create: bad argument");
  return ssd_gpu_create_bev(cfg, cfg->width, cfg->height, xf, device, max_frames, out);
}

int ssd_gpu_create_bev(const ssd_gpu_config *cfg, int32_t bev_width, int32_t bev_height, const ssd_gpu_transform *xf, int device, int max_frames,
                       ssd_gpu_ctx **out)
{
  if(!cfg || !xf || !out || max_frames <= 0)
    return fail(nullptr, SSD_E_INVALID_ARG, "ssd_gpu_create: bad argument");
  *out = nullptr;
  int ndev = 0;
  if(cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, SSD_E_CUDA, "ssd_gpu_create: no CUDA device (this library has no CPU fallback)");
  if(device < 0 || device >= ndev)
    return fail(nullptr, SSD_E_INVALID_ARG, "ssd_gpu_create: bad device index");
  DevParams dp;
  const int rc = derive_params(*cfg, bev_width, bev_height, *xf, dp);
  if(rc)
    return fail(nullptr, rc, "ssd_gpu_create: configuration out of range (3 <= height bins <= 253, frame width*height % 16 == 0 and at most "
                             "9348*5108, BEV width <= 9349, BEV height <= 5109)");

  ssd_gpu_ctx *ctx = new ssd_gpu_ctx();
  ctx->device = device;
  ctx->max_frames = max_frames;
  ctx->cfg = *cfg;
  ctx->xf = *xf;
  ctx->dp = dp;
  ctx->bm_words = (size_t)dp.H * dp.wpr;

  auto bail = [&](const std::string &m, int code)
  {
    g_create_error = m + (ctx->err.empty() ? "" : (": " + ctx->err));
    ssd_gpu_destroy(ctx);
    return code;
  };
  if(cudaSetDevice(device) != cudaSuccess)
    return bail("cudaSetDevice failed", SSD_E_CUDA);

  // frames per launch chain (chunk). Two chains are in flight on two streams, so one chain's latency-bound
  // per-plateau kernels overlap the other's HBM-bound point kernels. Measured on B200 (tools/sweep.py):
  // throughput grows with the chunk size up to ~256 frames. SSD_GPU_CHUNK_FRAMES overrides.
  {
    int cf = 1024;
    if(const char *e = getenv("SSD_GPU_CHUNK_FRAMES"))
      cf = atoi(e);
    if(const char *e = getenv("SSD_GPU_OUTLINE_GRIDX"))
      ctx->outline_gridx = std::max(1, std::min(SSD_GPU_MAX_PLATEAUS, atoi(e)));
    if(const char *e = getenv("SSD_GPU_STREAMS"))
      ctx->n_streams = std::max(1, std::min(SSD_MAX_STREAMS, atoi(e)));
    // the BEV bitmaps (2 streams x chunk x 32 slots) must stay a small part of HBM
    const size_t per_frame = (size_t)ctx->n_streams * SSD_GPU_MAX_PLATEAUS * ctx->bm_words * 4;
    const size_t budget = (size_t)8 << 30;
    if((size_t)cf * per_frame > budget)
      cf = (int)(budget / per_frame);
    cf = std::max(1, std::min({ cf, max_frames, 65535 })); // (a chunk is gridDim.y of the point kernels)
    ctx->chunk_frames = cf;
    int hc = 32; // measured on B200 (tools/e2e_sweep.py): 16..64 frames reach 54.4 GB/s of H2D, 512 only 49.5
    if(const char *e = getenv("SSD_GPU_HOST_CHUNK_FRAMES"))
      hc = atoi(e);
    ctx->host_chunk_frames = std::max(1, std::min(hc, cf));
  }

  {
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    int bt = sms * 4 * 5;
    if(const char *e = getenv("SSD_GPU_PT_BLOCKS"))
      bt = atoi(e);
    ctx->pt_blocks_target = std::max(1, bt);
  }
  int max_optin = 0;
  cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
  cudaFuncAttributes fa{};
  ctx->outline_small = dp.W / 25 + 4 <= 64 && dp.W / 50 + 6 <= 32 && dp.H / 10 + 2 <= 112;
  if(cudaFuncGetAttributes(&fa, k_outline<OutlineShared>) != cudaSuccess)
    return bail("cudaFuncGetAttributes(k_outline) failed: was the library built for this GPU (sm_100a)?", SSD_E_CUDA);
  cudaFuncAttributes fb{}, fc{};
  cudaFuncGetAttributes(&fb, k_finalize<OutlineShared>);
  cudaFuncGetAttributes(&fc, k_single_front_edge);
  const size_t stat = std::max({ fa.sharedSizeBytes, fb.sharedSizeBytes, fc.sharedSizeBytes });
  size_t dyn = (size_t)max_optin > stat + 1024 ? (size_t)max_optin - stat - 1024 : 0;
  // raw band only (the close is evaluated on the fly); no more than the full image needs, and by default
  // small enough for three resident blocks per SM (larger bands fall back to probing global memory)
  const size_t full = (size_t)dp.H * (dp.wpr + 1) * 4;
  size_t want = 32 * 1024; // measured on B200 (tools/knobs.sh): 32 KB beats 24 / 40 / 48 KB at 1024x768
  if(const char *e = getenv("SSD_GPU_OUTLINE_SMEM_KB"))
    want = (size_t)atoi(e) * 1024;
  dyn = std::min(dyn, std::min(full, want));
  dyn &= ~(size_t)15;
  ctx->ol_dyn_smem = dyn;
  ctx->smem_cap_words = dyn / 4;
  cudaFuncSetAttribute(k_transform_bin<SSD_PT_ITERS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SSD_PT_ITERS * SSD_TB_STAGE_BYTES);
  cudaFuncSetAttribute(k_transform_bin<SSD_PT_ITERS, true, CamTable>, cudaFuncAttributeMaxDynamicSharedMemorySize, SSD_PT_ITERS * SSD_TB_STAGE_BYTES);
  cudaFuncSetAttribute(k_transform_bin<SSD_PT_ITERS, false, CamTable>, cudaFuncAttributeMaxDynamicSharedMemorySize, SSD_PT_ITERS * SSD_TB_STAGE_BYTES);
  cudaFuncSetAttribute(k_transform_bin<SSD_PT_ITERS, false, GroupTable>, cudaFuncAttributeMaxDynamicSharedMemorySize, SSD_PT_ITERS * SSD_TB_STAGE_BYTES);
  if(cudaFuncSetAttribute(k_transform_bin<SSD_PT_ITERS>, cudaFuncAttributeMaxDynamicSharedMemorySize, SSD_PT_ITERS * SSD_TB_STAGE_BYTES) != cudaSuccess)
    return bail("cudaFuncSetAttribute(k_transform_bin) failed", SSD_E_CUDA);
  {
    // The attribute is per function and process-wide: never lower it (another context of a larger frame size may be alive).
    static std::mutex mtx;
    static size_t granted = 0;
    std::lock_guard<std::mutex> lock(mtx);
    if(dyn > granted)
    {
      cudaFuncSetAttribute(k_outline<OutlineShared>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_outline<OutlineSharedSmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      allow_outline_smem<NoCam>((int)dyn);
      allow_outline_smem<CamTable>((int)dyn);
      allow_outline_smem<GroupTable>((int)dyn);
      cudaFuncSetAttribute(k_single_front_edge, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      granted = dyn;
    }
  }

#define CKC(call)                                                            \
  do                                                                         \
  {                                                                          \
    cudaError_t e_ = (call);                                                 \
    if(e_ != cudaSuccess)                                                    \
    {                                                                        \
      ctx->err = cudaGetErrorString(e_);                                     \
      return bail(#call, e_ == cudaErrorMemoryAllocation ? SSD_E_NOMEM : SSD_E_CUDA); \
    }                                                                        \
  } while(0)
  if(const char *e = getenv("SSD_GPU_L_BPF"))
    ctx->bpf_l_knob = std::max(0, atoi(e));
  if(const char *e = getenv("SSD_GPU_Q_BPF"))
    ctx->bpf_q_knob = std::max(0, atoi(e));
  if(const char *e = getenv("SSD_GPU_NO_SPLIT_SMALL"))
    ctx->no_split_small = atoi(e) != 0;
  for(int i = 0; i < ctx->n_streams; i++)
  {
    CKC(cudaStreamCreateWithFlags(&ctx->stream[i], cudaStreamNonBlocking));
    CKC(cudaEventCreateWithFlags(&ctx->ev_in_ready[i], cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&ctx->ev_in_free[i], cudaEventDisableTiming));
    CKC(cudaEventCreateWithFlags(&ctx->ev_chunk_done[i], cudaEventDisableTiming));
  }
  CKC(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  CKC(cudaEventCreate(&ctx->ev_start));
  CKC(cudaEventCreate(&ctx->ev_stop));
  CKC(cudaEventCreate(&ctx->ev_h2d0));
  CKC(cudaEventCreate(&ctx->ev_h2d1));
  CKC(cudaMalloc(&ctx->d_frames, sizeof(FrameDev) * (size_t)max_frames));
  CKC(cudaMalloc(&ctx->d_out, sizeof(FrameOut) * (size_t)max_frames));
  CKC(cudaMallocHost(&ctx->h_out, sizeof(FrameOut) * (size_t)max_frames));
  CKC(cudaMalloc(&ctx->d_labels, (size_t)max_frames * dp.N));
  const size_t bev_bytes = (size_t)ctx->n_streams * ctx->chunk_frames * SSD_GPU_MAX_PLATEAUS * ctx->bm_words * 4;
  CKC(cudaMalloc(&ctx->d_bev, bev_bytes));
  CKC(cudaMemset(ctx->d_bev, 0, bev_bytes)); // bitmaps are self-cleaning afterwards
  CKC(cudaMemset(ctx->d_frames, 0, sizeof(FrameDev) * (size_t)max_frames));
  CKC(cudaMemset(ctx->d_out, 0, sizeof(FrameOut) * (size_t)max_frames));
  memset(ctx->h_out, 0, sizeof(FrameOut) * (size_t)max_frames);
  CKC(cudaDeviceSynchronize());
#undef CKC
  *out = ctx;
  return SSD_OK;
}

// The ray table of lens d with intrinsics in into ray (N entries), on stream 0, synchronously. SSD_E_INVALID_ARG when a ray is
// not finite: the lens does not admit this frame.
static int build_ray_table(ssd_gpu_ctx *ctx, const ssd_gpu_intrinsics &in, const ssd_gpu_distortion &d, float2 *ray)
{
  const DevParams &p = ctx->dp;
  unsigned *d_bad = nullptr;
  CK(cudaMalloc(&d_bad, sizeof(unsigned)));
  unsigned bad = 0;
  cudaStream_t st = ctx->stream[0];
  cudaError_t e = cudaMemsetAsync(d_bad, 0, sizeof(unsigned), st);
  if(e == cudaSuccess)
  {
    k_lens_rays<<<(int)std::min<size_t>(((size_t)p.N + 255) / 256, 4096), 256, 0, st>>>(p.FW, p.FH, in, d, ray, d_bad);
    e = cudaGetLastError();
  }
  if(e == cudaSuccess)
    e = cudaMemcpyAsync(&bad, d_bad, sizeof(unsigned), cudaMemcpyDeviceToHost, st);
  if(e == cudaSuccess)
    e = cudaStreamSynchronize(st); // every stream reads the table
  cudaFree(d_bad);
  CK(e);
  if(bad)
    return fail(ctx, SSD_E_INVALID_ARG, "lens distortion: the deprojection is not finite at some pixel of the frame (the lens model diverges there)");
  return SSD_OK;
}

static int check_distortion(ssd_gpu_ctx *ctx, const ssd_gpu_distortion &d, const std::string &who)
{
  static const char *const names[] = { "NONE", "MODIFIED_BROWN_CONRADY", "INVERSE_BROWN_CONRADY", "FTHETA", "BROWN_CONRADY", "KANNALA_BRANDT4" };
  if(d.model != SSD_DISTORTION_NONE && d.model != SSD_DISTORTION_INVERSE_BROWN_CONRADY && d.model != SSD_DISTORTION_BROWN_CONRADY)
    return fail(ctx, SSD_E_INVALID_ARG, who + ": distortion model " + std::to_string(d.model) +
                                            (d.model >= 0 && d.model <= 5 ? std::string(" (") + names[d.model] + ")" : std::string()) +
                                            " is not supported (NONE, INVERSE_BROWN_CONRADY and BROWN_CONRADY are)");
  for(int i = 0; i < 5; i++)
    if(!std::isfinite(d.coeffs[i]))
      return fail(ctx, SSD_E_INVALID_ARG, who + ": distortion coefficient " + std::to_string(i) + " is not finite");
  return SSD_OK;
}

// (re)build the deprojection tables when the intrinsics change
static int ensure_deproject_tables(ssd_gpu_ctx *ctx, const ssd_gpu_intrinsics &in)
{
  const DevParams &p = ctx->dp;
  if(!(in.fx != 0.f) || !(in.fy != 0.f) || !(in.depth_unit > 0.f))
    return fail(ctx, SSD_E_INVALID_ARG, "depth input: fx, fy must be non-zero and depth_unit positive");
  if(p.FW % 4 != 0)
    return fail(ctx, SSD_E_INVALID_ARG, "depth input: the frame width must be a multiple of 4");
  if(!ctx->d_xn)
  {
    CK(cudaMalloc(&ctx->d_xn, sizeof(float) * (size_t)p.FW));
    CK(cudaMalloc(&ctx->d_yn, sizeof(float) * (size_t)p.FH));
    memset(&ctx->intr, 0, sizeof(ctx->intr));
  }
  if(memcmp(&ctx->intr, &in, sizeof(float) * 5) != 0)
  {
    const int n = std::max(p.FW, p.FH);
    k_deproject_tables<<<(n + 255) / 256, 256, 0, ctx->stream[0]>>>(p.FW, p.FH, in, ctx->d_xn, ctx->d_yn);
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream[0])); // every stream reads the tables
    ctx->intr = in;
  }
  if(ssd_lens_is_pinhole(&ctx->lens))
    return SSD_OK;
  // a distorted lens: its ray table, rebuilt when the intrinsics change (ssd_gpu_set_distortion invalidates it)
  if(!ctx->ray_valid || memcmp(&ctx->ray_intr, &in, sizeof(float) * 4) != 0)
  {
    if(!ctx->d_ray)
      CK(cudaMalloc(&ctx->d_ray, sizeof(float2) * (size_t)p.N));
    ctx->ray_valid = false;
    const int rc = build_ray_table(ctx, in, ctx->lens, ctx->d_ray);
    if(rc)
      return rc;
    ctx->ray_intr = in;
    ctx->ray_valid = true;
  }
  return SSD_OK;
}

} // extern "C": the call description and its driver follow

// One process call, as every entry point describes it
enum CallMode
{
  CALL_PLAIN,   // every frame with the context's own camera
  CALL_CAMERAS, // each frame with the camera camera_of_frame names
  CALL_GROUPS,  // as CALL_CAMERAS, the frames of each group detected as one point cloud
};
enum InputKind
{
  IN_VERTICES, // packed {x, y, z} floats
  IN_Z16,      // z16 depth counts, deprojected inside the point kernels
  IN_F32,      // float depth samples, likewise
};
struct ProcessCall
{
  CallMode mode;
  InputKind kind;
  const void *input; // n_frames x N pixels of the kind
  bool host;         // input in host memory: staged through d_stage
  int n_frames;      // group calls: set by check_call from group_frames
  int flags;
  const ssd_gpu_intrinsics *intr = nullptr; // plain depth calls
  const int32_t *camera_of_frame = nullptr; // camera and group calls
  const int32_t *group_frames = nullptr;    // group calls: frames of each of the n_groups groups
  int n_groups = 0;
};

// Everything a call can be refused for. Steps 1-7 change nothing; step 8 comes last because it builds the plain depth path's tables.
// Only the RANGE / STATE checks sit between INVALID_ARG checks, so the code a call with several faults gets does not depend on which
// INVALID_ARG fault is found first.
static int check_call(ssd_gpu_ctx *ctx, ProcessCall &c)
{
  static const char *const family[] = { "process", "camera call", "group call" };
  const std::string who = family[c.mode];
  const bool depth = c.kind != IN_VERTICES;
  // 1. null and count arguments
  if(c.mode == CALL_PLAIN && depth && (!c.input || !c.intr))
    return fail(ctx, SSD_E_INVALID_ARG, c.kind == IN_Z16 ? "process_depth: bad argument" : "process_depth_f32: bad argument");
  if(!ctx || !c.input || (c.mode != CALL_PLAIN && !c.camera_of_frame) ||
     (c.mode == CALL_GROUPS ? !c.group_frames || c.n_groups < 1 : c.n_frames <= 0))
    return fail(ctx, SSD_E_INVALID_ARG, who + ": bad argument");
  // 2. group sizes
  long long n_frames = c.n_frames;
  if(c.mode == CALL_GROUPS)
  {
    n_frames = 0;
    for(int g = 0; g < c.n_groups; g++)
    {
      if(c.group_frames[g] < 1 || c.group_frames[g] > SSD_GPU_MAX_GROUP_FRAMES)
        return fail(ctx, SSD_E_INVALID_ARG, "group call: group " + std::to_string(g) + " has " + std::to_string(c.group_frames[g]) +
                                                " frames, outside [1, " + std::to_string(SSD_GPU_MAX_GROUP_FRAMES) + "]");
      n_frames += c.group_frames[g];
    }
  }
  // 3. the camera table
  if(c.mode != CALL_PLAIN && ctx->n_cameras <= 0)
    return fail(ctx, SSD_E_STATE, who + ": no camera table (ssd_gpu_set_cameras)");
  // 4. frames
  if(n_frames > ctx->max_frames)
    return fail(ctx, SSD_E_RANGE, c.mode == CALL_GROUPS ? "group call: the groups hold " + std::to_string(n_frames) +
                                                            " frames, more than max_frames of the context"
                                                      : "process: n_frames exceeds max_frames of the context");
  c.n_frames = (int)n_frames;
  // 5. the frame width of depth input: one load per 4-pixel word; the point kernels divide a pixel index by the width with a 40-bit
  // reciprocal (wmagic), exact for every index of the frame when N * W < 2^40
  if(depth && ctx->dp.FW % 4 != 0)
    return fail(ctx, SSD_E_INVALID_ARG, "depth input: the frame width must be a multiple of 4");
  if(depth && (unsigned long long)ctx->dp.N * (unsigned long long)ctx->dp.FW >= (1ull << 40))
    return fail(ctx, SSD_E_INVALID_ARG, "depth input: the frame's points times its width must stay below 2^40 (row division)");
  // 6. each frame's camera
  for(int f = 0; f < c.n_frames && c.mode != CALL_PLAIN; f++)
  {
    const int32_t cam = c.camera_of_frame[f];
    if(cam < 0 || cam >= ctx->n_cameras)
      return fail(ctx, SSD_E_RANGE, "camera call: frame " + std::to_string(f) + " names camera " + std::to_string(cam) + ", outside [0, " +
                                      std::to_string(ctx->n_cameras) + ")");
    if(depth && !ctx->cam_depth_ok[cam])
      return fail(ctx, SSD_E_INVALID_ARG, "depth camera call: camera " + std::to_string(cam) + " has no depth intrinsics (fx, fy must be non-zero and "
                                                                                              "depth_unit positive)");
  }
  // 7. alignment: the point kernels use 16-byte vector loads / bulk copies (vertices), one load per 4-pixel word of depth (8 bytes of
  // z16, 16 bytes of float)
  if((uintptr_t)c.input & (c.kind == IN_Z16 ? 7u : 15u))
    return fail(ctx, SSD_E_INVALID_ARG, c.kind == IN_F32 ? "process: float depth input must be 16-byte aligned"
                                                         : "process: the input buffer must be 16-byte aligned (vertices) / 8-byte aligned (depth)");
  // 8. the plain depth path's intrinsics, and its deprojection and ray tables
  if(c.mode == CALL_PLAIN && depth)
  {
    CK(cudaSetDevice(ctx->device));
    return ensure_deproject_tables(ctx, *c.intr);
  }
  return SSD_OK;
}

// Runs an accepted call: its frames in chunks through launch_classic, for the call's one source and camera type.
static int process(ssd_gpu_ctx *ctx, ProcessCall c)
{
  int rc = check_call(ctx, c);
  if(rc == SSD_OK)
    rc = [&]() -> int {
      CK(cudaSetDevice(ctx->device));
      const DevParams &p = ctx->dp;
      const bool depth_input = c.kind != IN_VERTICES;
      const size_t frame_bytes = (size_t)p.N * (c.kind == IN_VERTICES ? 12 : c.kind == IN_Z16 ? 2 : 4);
      const int32_t *cam_of_frame = c.camera_of_frame, *group_frames = c.group_frames;
      const int n_frames = c.n_frames, n_groups = c.n_groups, flags = c.flags;
      // host input: every byte crosses PCIe, the copy of chunk i+1 overlaps the kernels of chunk i and only the last
      // chunk's kernels stay exposed -- small chunks. Device input: large chunks (the per-frame kernels need the parallelism).
      int cf = c.host ? ctx->host_chunk_frames : ctx->chunk_frames;
      // a device-resident batch that fits one chunk is still split over the streams, so that one half's latency-bound
      // per-plateau kernels overlap the other half's point kernels (measured: 64 frames of 4096x3072 as 2 x 32: +5 %;
      // below ~32 frames per chain the per-frame kernels lose more parallelism than the overlap returns)
      if(!c.host && !(flags & SSD_FLAG_SINGLE_STREAM) && ctx->n_streams > 1 && n_frames <= cf && !ctx->no_split_small)
      {
        const int half = (n_frames + ctx->n_streams - 1) / ctx->n_streams;
        if(half >= 32)
          cf = half;
      }
      // a distorted lens: depth frames read their rays from ray tables (SrcLens), the overlay projects through the lens
      bool use_lens = false;
      const ssd_gpu_distortion *ov_lens = nullptr;
      if(cam_of_frame)
      {
        for(int f = 0; f < n_frames && depth_input && ctx->cams_distorted && !use_lens; f++)
          use_lens = ctx->cam_distorted[cam_of_frame[f]] != 0;
        if(ctx->cams_distorted && ctx->ov.enabled)
          ov_lens = ctx->d_cam_lens;
      }
      else if(!ssd_lens_is_pinhole(&ctx->lens))
      {
        use_lens = depth_input;
        if(ctx->ov.enabled)
          ov_lens = ctx->d_lens;
      }
      // chunks {first frame, frames, first record, records}: cf frames each, or in a group call whole groups up to cf frames (a group
      // larger than cf is a chunk of its own)
      struct Chunk
      {
        int f0, nf, r0, nr;
      };
      std::vector<Chunk> chunks;
      int max_nf = 0;
      if(group_frames)
      {
        for(int g = 0, f = 0; g < n_groups; f += group_frames[g], g++)
        {
          if(chunks.empty() || chunks.back().nf + group_frames[g] > cf)
            chunks.push_back({ f, 0, g, 0 });
          chunks.back().nf += group_frames[g];
          chunks.back().nr++;
          max_nf = std::max(max_nf, chunks.back().nf);
        }
      }
      else
        for(int f0 = 0; f0 < n_frames; f0 += cf)
        {
          const int nf = std::min(cf, n_frames - f0);
          chunks.push_back({ f0, nf, f0, nf });
          max_nf = std::max(max_nf, nf);
        }
      const int n_records = group_frames ? n_groups : n_frames;
      // host input: the staging buffers grow to the largest chunk any call has needed (no call is in flight between calls)
      if(c.host && (size_t)max_nf * frame_bytes > ctx->stage_bytes)
      {
        ctx->stage_bytes = 0;
        for(int i = 0; i < ctx->n_streams; i++)
        {
          CK(cudaFree(ctx->d_stage[i]));
          ctx->d_stage[i] = nullptr;
          CK(cudaMalloc(&ctx->d_stage[i], (size_t)max_nf * frame_bytes));
        }
        ctx->stage_bytes = (size_t)max_nf * frame_bytes;
      }

      int launches = 0;
      const bool stage_timing = (flags & SSD_FLAG_STAGE_TIMING) != 0;
      const int n_chunks = (int)chunks.size();
      if(stage_timing && ctx->stage_chunks < n_chunks)
      {
        const size_t want = (size_t)n_chunks * (SSD_GPU_N_STAGES + 1);
        while(ctx->stage_ev.size() < want)
        {
          cudaEvent_t e;
          CK(cudaEventCreate(&e));
          ctx->stage_ev.push_back(e);
        }
        ctx->stage_chunks = n_chunks;
      }
      ctx->n_frames_last = n_frames;
      ctx->flags_last = flags;
      ctx->step_labels_last = ctx->step_labels;
      ctx->surfaces_last = ctx->surfaces;
      ctx->grp_of_frame.clear();
      ctx->grp_members.clear();
      ctx->grp_epsc.clear();
      ctx->stats_eps0 = ctx->dp.E0s;
      ctx->stats_eps1 = ctx->dp.E1s;
      CamTable cams{};
      if(cam_of_frame)
      {
        cams.params = ctx->d_cam_dp;
        cams.ov = ctx->d_cam_ov;
        cams.xn = ctx->d_cam_xn;
        cams.yn = ctx->d_cam_yn;
        cams.unit = ctx->d_cam_unit;
        cams.cam = ctx->d_cam_of_frame;
        ctx->stats_eps0 = ctx->stats_eps1 = 0;
        for(int f = 0; f < n_frames; f++)
        {
          const DevParams &d = ctx->cam_dp[cam_of_frame[f]];
          ctx->stats_eps0 = std::max(ctx->stats_eps0, (double)d.E0s);
          ctx->stats_eps1 = std::max(ctx->stats_eps1, (double)d.E1s);
        }
      }
      GroupTable grp{};
      if(group_frames)
      {
        if(!ctx->d_grp_of_frame)
        {
          CK(cudaMalloc(&ctx->d_grp_of_frame, sizeof(int) * (size_t)ctx->max_frames));
          CK(cudaMalloc(&ctx->d_grp_members, sizeof(int2) * (size_t)ctx->max_frames));
          CK(cudaMalloc(&ctx->d_grp_epsc, sizeof(float) * (size_t)ctx->max_frames));
        }
        // the quadrilateral filters of a group decide the points of all its cameras: the largest of their bounds
        for(int g = 0, f = 0; g < n_groups; f += group_frames[g], g++)
        {
          float e = 0.f;
          for(int i = 0; i < group_frames[g]; i++)
          {
            ctx->grp_of_frame.push_back(g);
            e = std::max(e, ctx->cam_dp[cam_of_frame[f + i]].epsc); // (an infinite bound stays infinite: every decision is exact)
          }
          ctx->grp_members.push_back(make_int2(f, group_frames[g]));
          ctx->grp_epsc.push_back(e);
        }
        grp.cams = cams;
        grp.group = ctx->d_grp_of_frame;
        grp.members = ctx->d_grp_members;
        grp.epsc = ctx->d_grp_epsc;
      }
      if(ctx->surfaces)
      {
        // each record's ToExternalWorld as k_finalize uses it: the context's, the frame's camera's, the group's first member's
        ctx->surf_xf.resize((size_t)n_records);
        for(int r = 0; r < n_records; r++)
        {
          const DevParams &d = !cam_of_frame ? ctx->dp : ctx->cam_dp[cam_of_frame[group_frames ? ctx->grp_members[r].x : r]];
          SurfaceXf &x = ctx->surf_xf[r];
          memcpy(x.ext_a, d.ext_a, sizeof(x.ext_a));
          memcpy(x.ext_b, d.ext_b, sizeof(x.ext_b));
          x.ext_z = d.ext_z;
        }
      }
      // the whole call is ordered after ev_start on stream 0; stream 1 joins via events
      CK(cudaEventRecord(ctx->ev_start, ctx->stream[0]));
      for(int i = 1; i < ctx->n_streams; i++)
        CK(cudaStreamWaitEvent(ctx->stream[i], ctx->ev_start, 0));
      CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_start, 0));
      if(c.host)
        CK(cudaEventRecord(ctx->ev_h2d0, ctx->copy_stream));
      // per-frame state: histogram must start at zero
      CK(cudaMemsetAsync(ctx->d_frames, 0, sizeof(FrameDev) * (size_t)n_records, ctx->stream[0]));
      if(cam_of_frame)
        CK(cudaMemcpyAsync(ctx->d_cam_of_frame, cam_of_frame, sizeof(int32_t) * (size_t)n_frames, cudaMemcpyHostToDevice, ctx->stream[0]));
      if(group_frames)
      {
        CK(cudaMemcpyAsync(ctx->d_grp_of_frame, ctx->grp_of_frame.data(), sizeof(int) * (size_t)n_frames, cudaMemcpyHostToDevice, ctx->stream[0]));
        CK(cudaMemcpyAsync(ctx->d_grp_members, ctx->grp_members.data(), sizeof(int2) * (size_t)n_groups, cudaMemcpyHostToDevice, ctx->stream[0]));
        CK(cudaMemcpyAsync(ctx->d_grp_epsc, ctx->grp_epsc.data(), sizeof(float) * (size_t)n_groups, cudaMemcpyHostToDevice, ctx->stream[0]));
      }
      CK(cudaEventRecord(ctx->ev_chunk_done[0], ctx->stream[0]));
      for(int i = 1; i < ctx->n_streams; i++)
        CK(cudaStreamWaitEvent(ctx->stream[i], ctx->ev_chunk_done[0], 0));

      // the chunk loop for the call's one source and camera type
      const auto run_chunks = [&](const auto &src, const auto &cam) -> int {
        for(int chunk = 0; chunk < n_chunks; chunk++)
        {
          const int f0 = chunks[chunk].f0, nf = chunks[chunk].nf;
          const int s = (flags & SSD_FLAG_SINGLE_STREAM) ? 0 : chunk % ctx->n_streams;
          const void *in = static_cast<const char *>(c.input) + (size_t)f0 * frame_bytes;
          if(c.host)
          {
            // staging buffer s may be overwritten once the chunk that last used it has consumed it
            if(chunk >= ((flags & SSD_FLAG_SINGLE_STREAM) ? 1 : ctx->n_streams))
              CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_in_free[s], 0));
            CK(cudaMemcpyAsync(ctx->d_stage[s], in, (size_t)nf * frame_bytes, cudaMemcpyHostToDevice, ctx->copy_stream));
            in = ctx->d_stage[s];
            CK(cudaEventRecord(ctx->ev_in_ready[s], ctx->copy_stream));
            CK(cudaStreamWaitEvent(ctx->stream[s], ctx->ev_in_ready[s], 0));
          }
          const auto csrc = chunk_src(src, in);
          const auto ccam = chunk_cam(cam, f0, chunks[chunk].r0);
          cudaEvent_t *ev = stage_timing ? &ctx->stage_ev[(size_t)chunk * (SSD_GPU_N_STAGES + 1)] : nullptr;
          const int rc = ctx->outline_small
                           ? launch_classic<OutlineSharedSmall>(ctx, s, csrc, f0, nf, chunks[chunk].r0, chunks[chunk].nr, &launches, ev, ccam, ov_lens)
                           : launch_classic<OutlineShared>(ctx, s, csrc, f0, nf, chunks[chunk].r0, chunks[chunk].nr, &launches, ev, ccam, ov_lens);
          if(rc)
            return rc;
          if(c.host)
            CK(cudaEventRecord(ctx->ev_in_free[s], ctx->stream[s])); // all three passes have read the staging
        }
        return SSD_OK;
      };
      // The call's one source: vertices, or depth frames deprojected inside the point kernels, with the pin-hole tables (a camera
      // call's per camera) or the rays of a distorted lens. Each chunk sets the input pointer.
      const float unit = c.intr ? c.intr->depth_unit : 0.f;
      const unsigned long long wmagic = (((unsigned long long)1 << 40) + (unsigned long long)p.FW - 1) / (unsigned long long)p.FW;
      const auto run_depth = [&](auto sample, const auto &cam) -> int {
        typedef decltype(sample) T;
        if(use_lens)
          return run_chunks(SrcLensT<T>{ nullptr, ctx->d_ray, ctx->d_cam_ray, unit }, cam);
        return run_chunks(SrcDepthT<T>{ nullptr, ctx->d_xn, ctx->d_yn, unit, wmagic }, cam);
      };
      const auto run_source = [&](const auto &cam) -> int {
        switch(c.kind)
        {
        case IN_VERTICES:
          return run_chunks(SrcVertices{}, cam);
        case IN_Z16:
          return run_depth(uint16_t(), cam);
        case IN_F32:
          return run_depth(float(), cam);
        }
        return SSD_E_INVALID_ARG;
      };
      const int rs = group_frames ? run_source(grp) : cam_of_frame ? run_source(cams) : run_source(NoCam());
      if(rs)
        return rs;
      if(c.host)
        CK(cudaEventRecord(ctx->ev_h2d1, ctx->copy_stream));
      // join stream 1 into stream 0, then bring the compact results home
      for(int i = 1; i < ctx->n_streams; i++)
      {
        CK(cudaEventRecord(ctx->ev_chunk_done[i], ctx->stream[i]));
        CK(cudaStreamWaitEvent(ctx->stream[0], ctx->ev_chunk_done[i], 0));
      }
      CK(cudaMemcpyAsync(ctx->h_out, ctx->d_out, sizeof(FrameOut) * (size_t)n_records, cudaMemcpyDeviceToHost, ctx->stream[0]));
      if(ctx->ov.enabled)
        CK(cudaMemcpyAsync(ctx->h_ovl, ctx->d_ovl, sizeof(ssd_gpu_overlay) * SSD_GPU_MAX_STEPS * (size_t)n_frames, cudaMemcpyDeviceToHost, ctx->stream[0]));
      CK(cudaEventRecord(ctx->ev_stop, ctx->stream[0]));
      CK(cudaEventSynchronize(ctx->ev_stop));
      CK(cudaGetLastError());
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
      ctx->timing.total_ms = ms;
      ctx->timing.h2d_ms = 0;
      if(c.host)
      {
        float h = 0;
        CK(cudaEventElapsedTime(&h, ctx->ev_h2d0, ctx->ev_h2d1));
        ctx->timing.h2d_ms = h;
      }
      ctx->timing.label_ms = 0;
      ctx->timing.n_launches = launches;
      for(int i = 0; i < SSD_GPU_N_STAGES; i++)
      {
        ctx->stage_ms[i] = 0;
        ctx->stage_launches[i] = 0;
      }
      if(stage_timing)
      {
        for(int ch = 0; ch < n_chunks; ch++)
          for(int i = 0; i < SSD_GPU_N_STAGES; i++)
          {
            float t = 0;
            const cudaEvent_t *ev = &ctx->stage_ev[(size_t)ch * (SSD_GPU_N_STAGES + 1)];
            CK(cudaEventElapsedTime(&t, ev[i], ev[i + 1]));
            ctx->stage_ms[i] += t;
            ctx->stage_launches[i]++;
          }
        ctx->timing.label_ms = ctx->stage_ms[0];
      }
      return SSD_OK;
    }();
  // A refused call (INVALID_ARG, RANGE or STATE from check_call) has changed no result: the previous ones stay readable. Every other
  // failure is a device error (SSD_E_CUDA) in step 8's table build or in the chain: a launch error, a bad user pointer, out of memory
  // while growing a staging buffer. It may leave streams unsynchronised and BEV bitmaps half written (the bitmaps are
  // "self-cleaning" only along a complete chain): bring the context back to a clean state so that the next call starts from zeroed
  // bitmaps and no stale results can be read.
  if(rc == SSD_E_CUDA)
  {
    const std::string keep = ctx->err;
    cudaDeviceSynchronize();
    cudaGetLastError();
    cudaMemset(ctx->d_bev, 0, (size_t)ctx->n_streams * ctx->chunk_frames * SSD_GPU_MAX_PLATEAUS * ctx->bm_words * 4);
    ctx->n_frames_last = 0;
    ctx->step_labels_last = false;
    ctx->surfaces_last = false;
    ctx->err = keep;
  }
  return rc;
}

extern "C"
{

int ssd_gpu_process_host(ssd_gpu_ctx *ctx, const float *xyz_host, int n_frames)
{
  return process(ctx, { CALL_PLAIN, IN_VERTICES, xyz_host, true, n_frames, 0 });
}

int ssd_gpu_process_device(ssd_gpu_ctx *ctx, const float *xyz_dev, int n_frames)
{
  return process(ctx, { CALL_PLAIN, IN_VERTICES, xyz_dev, false, n_frames, 0 });
}

int ssd_gpu_process_device_ex(ssd_gpu_ctx *ctx, const float *xyz_dev, int n_frames, int flags)
{
  return process(ctx, { CALL_PLAIN, IN_VERTICES, xyz_dev, false, n_frames, flags });
}

int ssd_gpu_process_depth_host(ssd_gpu_ctx *ctx, const uint16_t *z16_host, const ssd_gpu_intrinsics *intr, int n_frames)
{
  return process(ctx, { CALL_PLAIN, IN_Z16, z16_host, true, n_frames, 0, intr });
}

int ssd_gpu_process_depth_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const ssd_gpu_intrinsics *intr, int n_frames)
{
  return process(ctx, { CALL_PLAIN, IN_Z16, z16_dev, false, n_frames, 0, intr });
}

int ssd_gpu_process_depth_f32_host(ssd_gpu_ctx *ctx, const float *depth_host, const ssd_gpu_intrinsics *intr, int n_frames)
{
  return process(ctx, { CALL_PLAIN, IN_F32, depth_host, true, n_frames, 0, intr });
}

int ssd_gpu_process_depth_f32_device(ssd_gpu_ctx *ctx, const float *depth_dev, const ssd_gpu_intrinsics *intr, int n_frames)
{
  return process(ctx, { CALL_PLAIN, IN_F32, depth_dev, false, n_frames, 0, intr });
}

// ---- per-frame cameras ----
static void free_cameras(ssd_gpu_ctx *ctx)
{
  for(void *p : { (void *)ctx->d_cam_dp, (void *)ctx->d_cam_ov, (void *)ctx->d_cam_xn, (void *)ctx->d_cam_yn, (void *)ctx->d_cam_unit,
                  (void *)ctx->d_cam_ray, (void *)ctx->d_cam_lens })
    cudaFree(p);
  for(float2 *t : ctx->cam_rays)
    cudaFree(t);
  ctx->cam_rays.clear();
  ctx->cam_distorted.clear();
  ctx->cams_distorted = false;
  ctx->d_cam_ray = nullptr;
  ctx->d_cam_lens = nullptr;
  ctx->d_cam_dp = nullptr;
  ctx->d_cam_ov = nullptr;
  ctx->d_cam_xn = ctx->d_cam_yn = ctx->d_cam_unit = nullptr;
  ctx->cam_dp.clear();
  ctx->cam_depth_ok.clear();
  ctx->n_cameras = 0;
}

// The ray tables of a camera table with at least one distorted lens: one per distinct lens (the intrinsics' fx, fy, ppx, ppy and the
// distortion, compared bitwise; a pin-hole camera's lens is model NONE), built and checked before the table is replaced. Cameras
// without depth intrinsics get none. On failure every table built here is freed.
struct CamLensKey
{
  float in[4];
  ssd_gpu_distortion d;
};
static int build_camera_rays(ssd_gpu_ctx *ctx, const ssd_gpu_camera *cams, const std::vector<ssd_gpu_distortion> &lens,
                             const std::vector<unsigned char> &depth_ok, std::vector<float2 *> &tables, std::vector<const float2 *> &of_camera)
{
  std::vector<CamLensKey> keys;
  of_camera.assign(lens.size(), nullptr);
  for(size_t c = 0; c < lens.size(); c++)
  {
    if(!depth_ok[c])
      continue;
    CamLensKey k;
    memset(&k, 0, sizeof(k));
    memcpy(k.in, &cams[c].intr, sizeof(k.in));
    if(!ssd_lens_is_pinhole(&lens[c]))
      k.d = lens[c];
    size_t t = 0;
    while(t < keys.size() && memcmp(&keys[t], &k, sizeof(k)) != 0)
      t++;
    if(t == keys.size())
    {
      float2 *ray = nullptr;
      cudaError_t e = cudaMalloc(&ray, sizeof(float2) * (size_t)ctx->dp.N);
      if(e != cudaSuccess)
      {
        ctx->err = std::string("cudaMalloc (ray table): ") + cudaGetErrorString(e);
        return SSD_E_CUDA;
      }
      tables.push_back(ray);
      keys.push_back(k);
      const int rc = build_ray_table(ctx, cams[c].intr, k.d, ray);
      if(rc)
      {
        if(rc == SSD_E_INVALID_ARG)
          ctx->err = "ssd_gpu_set_cameras_ex: camera " + std::to_string(c) + ": " + ctx->err;
        return rc;
      }
    }
    of_camera[c] = tables[t];
  }
  return SSD_OK;
}

int ssd_gpu_set_cameras(ssd_gpu_ctx *ctx, const ssd_gpu_camera *cams, int n_cameras)
{
  return ssd_gpu_set_cameras_ex(ctx, cams, nullptr, n_cameras);
}

int ssd_gpu_set_cameras_ex(ssd_gpu_ctx *ctx, const ssd_gpu_camera *cams, const ssd_gpu_distortion *dist, int n_cameras)
{
  if(!ctx || n_cameras < 0 || (n_cameras > 0 && !cams))
    return fail(ctx, SSD_E_INVALID_ARG, "ssd_gpu_set_cameras: bad argument");
  std::vector<ssd_gpu_distortion> lens((size_t)n_cameras);
  std::vector<unsigned char> distorted((size_t)n_cameras, 0);
  bool any_distorted = false;
  for(int c = 0; c < n_cameras && dist; c++)
  {
    const int rc = check_distortion(ctx, dist[c], "ssd_gpu_set_cameras_ex: camera " + std::to_string(c));
    if(rc)
      return rc;
    lens[c] = dist[c];
    distorted[c] = !ssd_lens_is_pinhole(&dist[c]);
    any_distorted = any_distorted || distorted[c];
  }
  // every camera is checked before the table is touched: a rejected table leaves the previous one in place
  std::vector<DevParams> dp((size_t)n_cameras);
  std::vector<OverlayDev> ov((size_t)n_cameras);
  std::vector<float> unit((size_t)n_cameras);
  std::vector<unsigned char> depth_ok((size_t)n_cameras);
  for(int c = 0; c < n_cameras; c++)
  {
    if(derive_params(ctx->cfg, ctx->dp.W, ctx->dp.H, cams[c].xf, dp[c]))
      return fail(ctx, SSD_E_INVALID_ARG, "ssd_gpu_set_cameras: camera " + std::to_string(c) + ": transform out of range");
    const ssd_gpu_intrinsics &in = cams[c].intr;
    OverlayDev &o = ov[c];
    memset(&o, 0, sizeof(o));
    for(int i = 0; i < 9; i++)
      o.a_inv[i] = cams[c].a_inv[i];
    o.fx = in.fx;
    o.fy = in.fy;
    o.ppx = in.ppx;
    o.ppy = in.ppy;
    o.enabled = 1;
    unit[c] = in.depth_unit;
    depth_ok[c] = in.fx != 0.f && in.fy != 0.f && in.depth_unit > 0.f; // as ensure_deproject_tables
  }
  CK(cudaSetDevice(ctx->device));
  CK(cudaDeviceSynchronize());
  // the ray tables are built (and the lenses checked) before the previous table is freed
  std::vector<float2 *> rays;
  std::vector<const float2 *> ray_of_camera;
  if(any_distorted)
  {
    const int rc = build_camera_rays(ctx, cams, lens, depth_ok, rays, ray_of_camera);
    if(rc)
    {
      for(float2 *t : rays)
        cudaFree(t);
      return rc;
    }
  }
  free_cameras(ctx);
  ctx->cam_rays.swap(rays);
  if(n_cameras == 0)
    return SSD_OK;
  const DevParams &p = ctx->dp;
  if(!ctx->d_cam_of_frame)
    CK(cudaMalloc(&ctx->d_cam_of_frame, sizeof(int32_t) * (size_t)ctx->max_frames));
  ssd_gpu_camera *d_in = nullptr;
  CK(cudaMalloc(&ctx->d_cam_dp, sizeof(DevParams) * (size_t)n_cameras));
  CK(cudaMalloc(&ctx->d_cam_ov, sizeof(OverlayDev) * (size_t)n_cameras));
  CK(cudaMalloc(&ctx->d_cam_unit, sizeof(float) * (size_t)n_cameras));
  CK(cudaMalloc(&ctx->d_cam_xn, sizeof(float) * (size_t)n_cameras * p.FW));
  CK(cudaMalloc(&ctx->d_cam_yn, sizeof(float) * (size_t)n_cameras * p.FH));
  CK(cudaMalloc(&d_in, sizeof(ssd_gpu_camera) * (size_t)n_cameras));
  CK(cudaMalloc(&ctx->d_cam_lens, sizeof(ssd_gpu_distortion) * (size_t)n_cameras));
  CK(cudaMalloc(&ctx->d_cam_ray, sizeof(float2 *) * (size_t)n_cameras));
  cudaStream_t st = ctx->stream[0];
  cudaError_t e = cudaMemcpyAsync(ctx->d_cam_dp, dp.data(), sizeof(DevParams) * (size_t)n_cameras, cudaMemcpyHostToDevice, st);
  if(e == cudaSuccess)
    e = cudaMemcpyAsync(ctx->d_cam_ov, ov.data(), sizeof(OverlayDev) * (size_t)n_cameras, cudaMemcpyHostToDevice, st);
  if(e == cudaSuccess)
    e = cudaMemcpyAsync(ctx->d_cam_unit, unit.data(), sizeof(float) * (size_t)n_cameras, cudaMemcpyHostToDevice, st);
  if(e == cudaSuccess)
    e = cudaMemcpyAsync(d_in, cams, sizeof(ssd_gpu_camera) * (size_t)n_cameras, cudaMemcpyHostToDevice, st);
  if(e == cudaSuccess)
    e = cudaMemcpyAsync(ctx->d_cam_lens, lens.data(), sizeof(ssd_gpu_distortion) * (size_t)n_cameras, cudaMemcpyHostToDevice, st);
  if(e == cudaSuccess && any_distorted)
    e = cudaMemcpyAsync(ctx->d_cam_ray, ray_of_camera.data(), sizeof(float2 *) * (size_t)n_cameras, cudaMemcpyHostToDevice, st);
  if(e == cudaSuccess)
  {
    // (cameras without depth intrinsics get meaningless tables: depth calls never use them)
    const int n = std::max(p.FW, p.FH);
    k_deproject_tables_cams<<<dim3((n + 255) / 256, std::min(n_cameras, 65535)), 256, 0, st>>>(p.FW, p.FH, d_in, n_cameras, ctx->d_cam_xn, ctx->d_cam_yn);
    e = cudaGetLastError();
  }
  if(e == cudaSuccess)
    e = cudaStreamSynchronize(st);
  cudaFree(d_in);
  if(e != cudaSuccess)
  {
    free_cameras(ctx);
    CK(e);
  }
  ctx->cam_dp.swap(dp);
  ctx->cam_depth_ok.swap(depth_ok);
  ctx->cam_distorted.swap(distorted);
  ctx->cams_distorted = any_distorted;
  ctx->n_cameras = n_cameras;
  return SSD_OK;
}

int ssd_gpu_set_distortion(ssd_gpu_ctx *ctx, const ssd_gpu_distortion *d)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  ssd_gpu_distortion nd{};
  if(d)
  {
    const int rc = check_distortion(ctx, *d, "ssd_gpu_set_distortion");
    if(rc)
      return rc;
    nd = *d;
  }
  if(!ssd_lens_is_pinhole(&nd))
  {
    CK(cudaSetDevice(ctx->device));
    if(!ctx->d_lens)
      CK(cudaMalloc(&ctx->d_lens, sizeof(ssd_gpu_distortion)));
    CK(cudaDeviceSynchronize()); // no call in flight reads the lens or the ray table
    CK(cudaMemcpy(ctx->d_lens, &nd, sizeof(nd), cudaMemcpyHostToDevice));
  }
  if(memcmp(&nd, &ctx->lens, sizeof(nd)) != 0)
    ctx->ray_valid = false; // rebuilt for the next depth call's intrinsics
  ctx->lens = nd;
  return SSD_OK;
}

int ssd_gpu_n_ray_tables(ssd_gpu_ctx *ctx)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  return (int)ctx->cam_rays.size() + (ctx->ray_valid && !ssd_lens_is_pinhole(&ctx->lens) ? 1 : 0);
}

int ssd_gpu_n_cameras(ssd_gpu_ctx *ctx)
{
  return ctx ? ctx->n_cameras : SSD_E_INVALID_ARG;
}

int ssd_gpu_process_cameras_host(ssd_gpu_ctx *ctx, const float *xyz_host, const int32_t *camera_of_frame, int n_frames)
{
  return process(ctx, { CALL_CAMERAS, IN_VERTICES, xyz_host, true, n_frames, 0, nullptr, camera_of_frame });
}

int ssd_gpu_process_cameras_device(ssd_gpu_ctx *ctx, const float *xyz_dev, const int32_t *camera_of_frame, int n_frames)
{
  return process(ctx, { CALL_CAMERAS, IN_VERTICES, xyz_dev, false, n_frames, 0, nullptr, camera_of_frame });
}

int ssd_gpu_process_cameras_device_ex(ssd_gpu_ctx *ctx, const float *xyz_dev, const int32_t *camera_of_frame, int n_frames, int flags)
{
  return process(ctx, { CALL_CAMERAS, IN_VERTICES, xyz_dev, false, n_frames, flags, nullptr, camera_of_frame });
}

int ssd_gpu_process_depth_cameras_host(ssd_gpu_ctx *ctx, const uint16_t *z16_host, const int32_t *camera_of_frame, int n_frames)
{
  return process(ctx, { CALL_CAMERAS, IN_Z16, z16_host, true, n_frames, 0, nullptr, camera_of_frame });
}

int ssd_gpu_process_depth_cameras_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const int32_t *camera_of_frame, int n_frames)
{
  return process(ctx, { CALL_CAMERAS, IN_Z16, z16_dev, false, n_frames, 0, nullptr, camera_of_frame });
}

int ssd_gpu_process_depth_f32_cameras_host(ssd_gpu_ctx *ctx, const float *depth_host, const int32_t *camera_of_frame, int n_frames)
{
  return process(ctx, { CALL_CAMERAS, IN_F32, depth_host, true, n_frames, 0, nullptr, camera_of_frame });
}

int ssd_gpu_process_depth_f32_cameras_device(ssd_gpu_ctx *ctx, const float *depth_dev, const int32_t *camera_of_frame, int n_frames)
{
  return process(ctx, { CALL_CAMERAS, IN_F32, depth_dev, false, n_frames, 0, nullptr, camera_of_frame });
}

int ssd_gpu_process_groups_host(ssd_gpu_ctx *ctx, const float *xyz_host, const int32_t *camera_of_frame, const int32_t *group_frames, int n_groups)
{
  return process(ctx, { CALL_GROUPS, IN_VERTICES, xyz_host, true, 0, 0, nullptr, camera_of_frame, group_frames, n_groups });
}

int ssd_gpu_process_groups_device(ssd_gpu_ctx *ctx, const float *xyz_dev, const int32_t *camera_of_frame, const int32_t *group_frames, int n_groups,
                                  int flags)
{
  return process(ctx, { CALL_GROUPS, IN_VERTICES, xyz_dev, false, 0, flags, nullptr, camera_of_frame, group_frames, n_groups });
}

int ssd_gpu_process_depth_groups_host(ssd_gpu_ctx *ctx, const uint16_t *z16_host, const int32_t *camera_of_frame, const int32_t *group_frames,
                                      int n_groups)
{
  return process(ctx, { CALL_GROUPS, IN_Z16, z16_host, true, 0, 0, nullptr, camera_of_frame, group_frames, n_groups });
}

int ssd_gpu_process_depth_groups_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const int32_t *camera_of_frame, const int32_t *group_frames,
                                        int n_groups, int flags)
{
  return process(ctx, { CALL_GROUPS, IN_Z16, z16_dev, false, 0, flags, nullptr, camera_of_frame, group_frames, n_groups });
}

int ssd_gpu_process_depth_f32_groups_host(ssd_gpu_ctx *ctx, const float *depth_host, const int32_t *camera_of_frame, const int32_t *group_frames,
                                          int n_groups)
{
  return process(ctx, { CALL_GROUPS, IN_F32, depth_host, true, 0, 0, nullptr, camera_of_frame, group_frames, n_groups });
}

int ssd_gpu_process_depth_f32_groups_device(ssd_gpu_ctx *ctx, const float *depth_dev, const int32_t *camera_of_frame, const int32_t *group_frames,
                                            int n_groups, int flags)
{
  return process(ctx, { CALL_GROUPS, IN_F32, depth_dev, false, 0, flags, nullptr, camera_of_frame, group_frames, n_groups });
}

int ssd_gpu_deproject_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const ssd_gpu_intrinsics *intr, int n_frames, float *xyz_dev)
{
  if(!ctx || !z16_dev || !intr || !xyz_dev || n_frames <= 0)
    return fail(ctx, SSD_E_INVALID_ARG, "deproject: bad argument");
  CK(cudaSetDevice(ctx->device));
  const int rc = ensure_deproject_tables(ctx, *intr);
  if(rc)
    return rc;
  const DevParams &p = ctx->dp;
  const bool lens = !ssd_lens_is_pinhole(&ctx->lens);
  for(int f0 = 0; f0 < n_frames; f0 += 32768)
  {
    const int nf = std::min(32768, n_frames - f0);
    if(lens)
    {
      k_deproject_lens<<<dim3((p.N / 4 + 255) / 256, nf), 256, 0, ctx->stream[0]>>>(p.N, intr->depth_unit, ctx->d_ray, z16_dev + (size_t)f0 * p.N,
                                                                                  xyz_dev + (size_t)f0 * p.N * 3);
      continue;
    }
    k_deproject<<<dim3((p.N / 4 + 255) / 256, nf), 256, 0, ctx->stream[0]>>>(p.FW, p.N, intr->depth_unit, ctx->d_xn, ctx->d_yn, z16_dev + (size_t)f0 * p.N,
                                                                            xyz_dev + (size_t)f0 * p.N * 3);
  }
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(ctx->stream[0]));
  return SSD_OK;
}

static int check_frame(ssd_gpu_ctx *ctx, int frame)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  if(ctx->n_frames_last <= 0)
    return fail(ctx, SSD_E_STATE, "no processed batch in this context");
  if(frame < 0 || frame >= ctx->n_frames_last)
    return fail(ctx, SSD_E_RANGE, "frame index out of range");
  return SSD_OK;
}

int ssd_gpu_get_steps(ssd_gpu_ctx *ctx, int frame, ssd_gpu_step *out, int cap, int *n, uint32_t *status)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  const FrameOut &o = ctx->h_out[frame_record(ctx, frame)];
  if(n)
    *n = o.info.n_steps;
  if(status)
    *status = o.info.status;
  if(out)
    for(int i = 0; i < o.info.n_steps && i < cap; i++)
      out[i] = o.steps[i];
  return SSD_OK;
}

int ssd_gpu_set_overlay(ssd_gpu_ctx *ctx, const double a_inv[9], const ssd_gpu_intrinsics *intr)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  if(!a_inv)
  {
    ctx->ov.enabled = 0;
    return SSD_OK;
  }
  if(!intr)
    return fail(ctx, SSD_E_INVALID_ARG, "ssd_gpu_set_overlay: intrinsics missing");
  CK(cudaSetDevice(ctx->device));
  if(!ctx->d_ovl)
  {
    const size_t bytes = sizeof(ssd_gpu_overlay) * SSD_GPU_MAX_STEPS * (size_t)ctx->max_frames;
    CK(cudaMalloc(&ctx->d_ovl, bytes));
    CK(cudaMallocHost(&ctx->h_ovl, bytes));
    CK(cudaMemset(ctx->d_ovl, 0, bytes));
    memset(ctx->h_ovl, 0, bytes);
  }
  for(int i = 0; i < 9; i++)
    ctx->ov.a_inv[i] = a_inv[i];
  ctx->ov.fx = intr->fx;
  ctx->ov.fy = intr->fy;
  ctx->ov.ppx = intr->ppx;
  ctx->ov.ppy = intr->ppy;
  ctx->ov.enabled = 1;
  ctx->n_frames_last = 0; // results of an earlier call carry no overlay
  return SSD_OK;
}

int ssd_gpu_get_overlay(ssd_gpu_ctx *ctx, int frame, ssd_gpu_overlay *out, int cap, int *n)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  if(!ctx->ov.enabled || !ctx->h_ovl)
    return fail(ctx, SSD_E_STATE, "ssd_gpu_get_overlay: overlay not enabled (ssd_gpu_set_overlay)");
  const int ns = ctx->h_out[frame_record(ctx, frame)].info.n_steps;
  if(n)
    *n = ns;
  if(out)
    for(int i = 0; i < ns && i < cap; i++)
      out[i] = ctx->h_ovl[(size_t)frame * SSD_GPU_MAX_STEPS + i];
  return SSD_OK;
}

int ssd_gpu_set_vertical_faces(ssd_gpu_ctx *ctx, int enable)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  ctx->risers = enable != 0;
  ctx->n_frames_last = 0; // results of an earlier call carry no risers
  return SSD_OK;
}

int ssd_gpu_get_vertical_faces(ssd_gpu_ctx *ctx, int frame, ssd_gpu_riser *out, int cap, int *n)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  if(!ctx->risers)
    return fail(ctx, SSD_E_STATE, "ssd_gpu_get_vertical_faces: not enabled (ssd_gpu_set_vertical_faces)");
  CK(cudaSetDevice(ctx->device));
  const int r = frame_record(ctx, frame);
  std::vector<PlateauDev> pl(SSD_GPU_MAX_PLATEAUS);
  std::vector<RiserDev> rs(SSD_GPU_MAX_PLATEAUS);
  CK(cudaMemcpy(pl.data(), ctx->d_frames[r].plat, sizeof(PlateauDev) * SSD_GPU_MAX_PLATEAUS, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(rs.data(), ctx->d_frames[r].ris, sizeof(RiserDev) * SSD_GPU_MAX_PLATEAUS, cudaMemcpyDeviceToHost));
  const int K = ctx->h_out[r].info.n_plateaus;
  const int R = K > 1 ? K - 1 : 0;
  if(n)
    *n = R;
  const ssd_gpu_config &c = ctx->cfg;
  for(int k = 0; k < R && k < cap && out; k++)
  {
    ssd_gpu_riser o{};
    o.lower_plateau = k;
    o.upper_plateau = k + 1;
    o.n_points = rs[k].cnt;
    o.z_bottom = c.z_min + (double)(pl[k].hmax + 1) * c.height_interval;
    o.z_top = c.z_min + (double)pl[k + 1].hmin * c.height_interval;
    if(rs[k].cnt)
    {
      o.x_min = c.x_min + (double)rs[k].xmin / 65536.0;
      o.x_max = c.x_min + (double)rs[k].xmax / 65536.0;
      o.y_min = c.y_min + (double)rs[k].ymin / 65536.0;
      o.y_max = c.y_min + (double)rs[k].ymax / 65536.0;
      o.x_mean = c.x_min + (double)rs[k].sx / (double)rs[k].cnt / 65536.0;
      o.y_mean = c.y_min + (double)rs[k].sy / (double)rs[k].cnt / 65536.0;
    }
    out[k] = o;
  }
  return SSD_OK;
}

int ssd_gpu_set_step_labels(ssd_gpu_ctx *ctx, int enable)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  if(!enable && ctx->surfaces)
    return fail(ctx, SSD_E_STATE, "ssd_gpu_set_step_labels: step surfaces are on and read the step labels (ssd_gpu_set_step_surfaces)");
  CK(cudaSetDevice(ctx->device));
  if((enable != 0) != ctx->step_labels)
    ctx->step_labels_last = false; // the map of an earlier call is not kept across a switch
  if(!enable)
  {
    // the pointer and the flag are cleared whatever the free returns: a failed free must not leave a pointer to free again
    const cudaError_t e = cudaFree(ctx->d_step_labels);
    ctx->d_step_labels = nullptr;
    ctx->step_labels = false;
    if(e != cudaSuccess)
      return fail(ctx, SSD_E_CUDA, std::string("ssd_gpu_set_step_labels: ") + cudaGetErrorString(e));
    return SSD_OK;
  }
  if(!ctx->d_step_labels)
  {
    const cudaError_t e = cudaMalloc(&ctx->d_step_labels, (size_t)ctx->max_frames * ctx->dp.N);
    if(e != cudaSuccess)
    {
      cudaGetLastError(); // clear the sticky allocation error: the context stays usable
      ctx->d_step_labels = nullptr;
      ctx->step_labels = false;
      return fail(ctx, SSD_E_NOMEM, std::string("ssd_gpu_set_step_labels: ") + cudaGetErrorString(e));
    }
  }
  ctx->step_labels = true;
  return SSD_OK;
}

// the step labels of the last call: SSD_E_STATE unless that call ran with them, they are still enabled and the call's results are
// readable (a failed call, or a setting that invalidates earlier results, sets n_frames_last to 0)
static int check_step_labels(ssd_gpu_ctx *ctx, const char *fn)
{
  if(!ctx->step_labels || !ctx->step_labels_last || ctx->n_frames_last <= 0)
    return fail(ctx, SSD_E_STATE, std::string(fn) + ": not enabled for the last call (ssd_gpu_set_step_labels)");
  return SSD_OK;
}

int ssd_gpu_get_step_labels(ssd_gpu_ctx *ctx, int frame, uint8_t *out_host)
{
  int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  if(!out_host)
    return SSD_E_INVALID_ARG;
  if((rc = check_step_labels(ctx, "ssd_gpu_get_step_labels")))
    return rc;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy(out_host, ctx->d_step_labels + (size_t)frame * ctx->dp.N, (size_t)ctx->dp.N, cudaMemcpyDeviceToHost));
  return SSD_OK;
}

int ssd_gpu_step_labels_device_ptr(ssd_gpu_ctx *ctx, const uint8_t **out)
{
  if(!ctx || !out)
    return SSD_E_INVALID_ARG;
  const int rc = check_step_labels(ctx, "ssd_gpu_step_labels_device_ptr");
  if(rc)
    return rc;
  *out = ctx->d_step_labels;
  return SSD_OK;
}

int ssd_gpu_set_step_surfaces(ssd_gpu_ctx *ctx, int enable)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  if(enable && !ctx->step_labels)
    return fail(ctx, SSD_E_STATE, "ssd_gpu_set_step_surfaces: the pass reads the step labels, which are off (ssd_gpu_set_step_labels)");
  const ssd_gpu_config &c = ctx->cfg;
  // fixed-point coordinates below 2^32 (k_step_surface): every range shorter than 65536 m
  if(enable && !(c.x_max - c.x_min < 65536.0 && c.y_max - c.y_min < 65536.0 && c.z_max - c.z_min < 65536.0))
    return fail(ctx, SSD_E_RANGE, "ssd_gpu_set_step_surfaces: a measuring range of 65536 m or more (the moments are exact below it)");
  CK(cudaSetDevice(ctx->device));
  if((enable != 0) != ctx->surfaces)
    ctx->surfaces_last = false; // the surfaces of an earlier call are not kept across a switch
  if(!enable)
  {
    // the pointer and the flag are cleared whatever the free returns: a failed free must not leave a pointer to free again
    const cudaError_t e = cudaFree(ctx->d_surf);
    ctx->d_surf = nullptr;
    ctx->surfaces = false;
    if(e != cudaSuccess)
      return fail(ctx, SSD_E_CUDA, std::string("ssd_gpu_set_step_surfaces: ") + cudaGetErrorString(e));
    return SSD_OK;
  }
  if(!ctx->d_surf)
  {
    const cudaError_t e = cudaMalloc(&ctx->d_surf, sizeof(SurfaceDev) * SSD_GPU_MAX_STEPS * (size_t)ctx->max_frames);
    if(e != cudaSuccess)
    {
      cudaGetLastError(); // clear the sticky allocation error: the context stays usable
      ctx->d_surf = nullptr;
      ctx->surfaces = false;
      return fail(ctx, SSD_E_NOMEM, std::string("ssd_gpu_set_step_surfaces: ") + cudaGetErrorString(e));
    }
  }
  ctx->surfaces = true;
  return SSD_OK;
}

// 128-bit moments of one step (SurfaceDev) as signed 128-bit integers
static __int128 u128_of(const unsigned long long m[2])
{
  return (__int128)(((unsigned __int128)m[1] << 64) | m[0]);
}

// The fields of include/ssd_gpu.h (ssd_gpu_step_surface) from the moments of one step and its record's ToExternalWorld.
// Double arithmetic in the stated order; the host build passes -ffp-contract=off.
static ssd_gpu_step_surface derive_surface(const SurfaceDev &m, const SurfaceXf &x, const ssd_gpu_config &c)
{
  ssd_gpu_step_surface o;
  memset(&o, 0, sizeof(o));
  if(m.n == 0)
    return o;
  const __int128 n = m.n, Sx = m.sx, Sy = m.sy, Sz = m.sz;
  const __int128 Sxx = u128_of(m.m2[0]), Sxy = u128_of(m.m2[1]), Syy = u128_of(m.m2[2]), Sxz = u128_of(m.m2[3]), Syz = u128_of(m.m2[4]),
                 Szz = u128_of(m.m2[5]);
  const double cxx = (double)(n * Sxx - Sx * Sx), cxy = (double)(n * Sxy - Sx * Sy), cyy = (double)(n * Syy - Sy * Sy);
  const double cxz = (double)(n * Sxz - Sx * Sz), cyz = (double)(n * Syz - Sy * Sz), czz = (double)(n * Szz - Sz * Sz);
  const double det = cxx * cyy - cxy * cxy;
  const double dn = (double)m.n;
  o.n_points = m.n;
  o.fit_valid = m.n >= 3 && det > 0;
  double a = 0, b = 0;
  if(o.fit_valid)
  {
    a = (cxz * cyy - cyz * cxy) / det;
    b = (cyz * cxx - cxz * cxy) / det;
    const double r = czz - a * cxz - b * cyz;
    o.rms_dz = std::sqrt(r > 0 ? r : 0.0) / dn / 65536.0;
    o.tilt_deg = std::atan(std::sqrt(a * a + b * b)) * (180.0 / M_PI);
  }
  const double xm = c.x_min + (double)m.sx / dn / 65536.0, ym = c.y_min + (double)m.sy / dn / 65536.0, zm = c.z_min + (double)m.sz / dn / 65536.0;
  o.centroid[0] = (x.ext_a[0] * xm + x.ext_a[1] * ym) + x.ext_b[0];
  o.centroid[1] = (x.ext_a[2] * xm + x.ext_a[3] * ym) + x.ext_b[1];
  o.centroid[2] = x.ext_z + zm;
  o.gradient[0] = x.ext_a[0] * a + x.ext_a[1] * b;
  o.gradient[1] = x.ext_a[2] * a + x.ext_a[3] * b;
  o.z_lo = x.ext_z + (c.z_min + (double)~m.zmin_inv / 65536.0);
  o.z_hi = x.ext_z + (c.z_min + (double)m.zmax / 65536.0);
  return o;
}

int ssd_gpu_get_step_surfaces(ssd_gpu_ctx *ctx, int frame, ssd_gpu_step_surface *out, int cap, int *n)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  if(!ctx->surfaces || !ctx->surfaces_last)
    return fail(ctx, SSD_E_STATE, "ssd_gpu_get_step_surfaces: not enabled for the last call (ssd_gpu_set_step_surfaces)");
  const int r = frame_record(ctx, frame);
  const int ns = ctx->h_out[r].info.n_steps;
  if(n)
    *n = ns;
  const int k = out ? std::min(ns, cap) : 0;
  if(k <= 0)
    return SSD_OK;
  CK(cudaSetDevice(ctx->device));
  std::vector<SurfaceDev> m((size_t)k);
  CK(cudaMemcpy(m.data(), ctx->d_surf + (size_t)r * SSD_GPU_MAX_STEPS, sizeof(SurfaceDev) * (size_t)k, cudaMemcpyDeviceToHost));
  for(int s = 0; s < k; s++)
    out[s] = derive_surface(m[s], ctx->surf_xf[r], ctx->cfg);
  return SSD_OK;
}

int ssd_gpu_get_frame_info(ssd_gpu_ctx *ctx, int frame, ssd_gpu_frame_info *out)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  if(!out)
    return SSD_E_INVALID_ARG;
  *out = ctx->h_out[frame_record(ctx, frame)].info;
  return SSD_OK;
}

int ssd_gpu_get_plateaus(ssd_gpu_ctx *ctx, int frame, ssd_gpu_plateau *out, int cap, int *n)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  CK(cudaSetDevice(ctx->device));
  const int r = frame_record(ctx, frame);
  std::vector<PlateauDev> tmp(SSD_GPU_MAX_PLATEAUS);
  CK(cudaMemcpy(tmp.data(), ctx->d_frames[r].plat, sizeof(PlateauDev) * SSD_GPU_MAX_PLATEAUS, cudaMemcpyDeviceToHost));
  const int K = ctx->h_out[r].info.n_plateaus;
  if(n)
    *n = K;
  for(int k = 0; k < K && k < cap && out; k++)
  {
    const PlateauDev &P = tmp[k];
    ssd_gpu_plateau &o = out[k];
    o.height = P.height;
    o.hmin = P.hmin;
    o.hmax = P.hmax;
    o.n_points = P.n_points;
    o.valid = P.valid;
    o.outlined = P.outlined;
    o.n_in_quad = P.n_in_quad;
    o.quad_status = P.quad_status;
    memcpy(o.quad_world, P.quad_world, sizeof(o.quad_world));
    o.mean_z = P.mean_z;
  }
  return SSD_OK;
}

int ssd_gpu_get_labels(ssd_gpu_ctx *ctx, int frame, uint8_t *out_host)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  if(!out_host)
    return SSD_E_INVALID_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy(out_host, ctx->d_labels + (size_t)frame * ctx->dp.N, (size_t)ctx->dp.N, cudaMemcpyDeviceToHost));
  return SSD_OK;
}

int ssd_gpu_get_histogram(ssd_gpu_ctx *ctx, int frame, uint32_t *out, int cap, int *n_bins)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  CK(cudaSetDevice(ctx->device));
  uint32_t tmp[SSD_BINS_PAD];
  CK(cudaMemcpy(tmp, ctx->d_frames[frame_record(ctx, frame)].hist, sizeof(tmp), cudaMemcpyDeviceToHost));
  if(n_bins)
    *n_bins = ctx->dp.n_bins;
  for(int i = 0; i < ctx->dp.n_bins && i < cap && out; i++)
    out[i] = tmp[i];
  return SSD_OK;
}

int ssd_gpu_get_timing(ssd_gpu_ctx *ctx, ssd_gpu_timing *out)
{
  if(!ctx || !out)
    return SSD_E_INVALID_ARG;
  *out = ctx->timing;
  return SSD_OK;
}

int ssd_gpu_get_stats(ssd_gpu_ctx *ctx, ssd_gpu_stats *out)
{
  if(!ctx || !out)
    return SSD_E_INVALID_ARG;
  uint64_t c[4] = { 0, 0, 0, 0 };
  for(int f = 0; f < n_records_last(ctx); f++)
  {
    const FrameOut &o = ctx->h_out[f];
    c[0] += o.n_exact_bin;
    c[1] += o.n_quad_pts;
    c[2] += o.n_def_quad;
    c[3] += o.n_def_bev;
  }
  out->n_points = (uint64_t)ctx->n_frames_last * (uint64_t)ctx->dp.N;
  out->n_exact_fallback = c[0];
  out->n_quad_fast = c[1] - c[2];
  out->n_quad_exact = c[2];
  out->n_bev_exact = c[3];
  out->filter_eps0 = ctx->n_frames_last > 0 ? ctx->stats_eps0 : ctx->dp.E0s;
  out->filter_eps1 = ctx->n_frames_last > 0 ? ctx->stats_eps1 : ctx->dp.E1s;
  return SSD_OK;
}

int ssd_gpu_get_stage_times(ssd_gpu_ctx *ctx, float ms[SSD_GPU_N_STAGES], int launches[SSD_GPU_N_STAGES])
{
  if(!ctx || !ms || !launches)
    return SSD_E_INVALID_ARG;
  for(int i = 0; i < SSD_GPU_N_STAGES; i++)
  {
    ms[i] = ctx->stage_ms[i];
    launches[i] = ctx->stage_launches[i];
  }
  return SSD_OK;
}

const char *ssd_gpu_stage_name(int stage)
{
  static const char *names[SSD_GPU_N_STAGES] = { "transform_bin", "peaks", "label_bev", "outline", "frame_logic", "quad_reduce", "finalize" };
  return stage >= 0 && stage < SSD_GPU_N_STAGES ? names[stage] : "";
}

int ssd_gpu_chunk_frames(ssd_gpu_ctx *ctx)
{
  return ctx ? ctx->chunk_frames : SSD_E_INVALID_ARG;
}

int ssd_gpu_labels_device_ptr(ssd_gpu_ctx *ctx, const uint8_t **out)
{
  if(!ctx || !out)
    return SSD_E_INVALID_ARG;
  *out = ctx->d_labels;
  return SSD_OK;
}

// ---- single-stage entry points ----
static int upload_image(ssd_gpu_ctx *ctx, const uint8_t *image_host)
{
  const DevParams &p = ctx->dp;
  const size_t bev_pixels = (size_t)p.W * p.H;
  CK(cudaSetDevice(ctx->device));
  if(!ctx->d_img)
    CK(cudaMalloc(&ctx->d_img, bev_pixels));
  CK(cudaMemcpyAsync(ctx->d_img, image_host, bev_pixels, cudaMemcpyHostToDevice, ctx->stream[0]));
  const int words = p.H * p.wpr;
  k_pack_bitmap<<<(words + 255) / 256, 256, 0, ctx->stream[0]>>>(p, ctx->d_img, ctx->d_bev);
  CK(cudaGetLastError());
  return SSD_OK;
}

int ssd_gpu_detect_outline(ssd_gpu_ctx *ctx, const uint8_t *image_host, int min_img_y_extent, double xy_ratio, double quad_px[8], int *valid)
{
  if(!ctx || !image_host || !quad_px || !valid)
    return SSD_E_INVALID_ARG;
  int rc = upload_image(ctx, image_host);
  if(rc)
    return rc;
  DevParams p = ctx->dp;
  p.min_img_y_extent = min_img_y_extent;
  p.xy_ratio = xy_ratio;
  cudaStream_t st = ctx->stream[0];
  k_single_setup_plateau<<<1, 1, 0, st>>>(ctx->d_frames, p.H);
  if(ctx->outline_small)
    k_outline<OutlineSharedSmall><<<dim3(1, 1), SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, ctx->d_frames, ctx->d_bev, ctx->bm_words, ctx->smem_cap_words);
  else
    k_outline<OutlineShared><<<dim3(1, 1), OutlineShared::THREADS, ctx->ol_dyn_smem, st>>>(p, ctx->d_frames, ctx->d_bev, ctx->bm_words, ctx->smem_cap_words);
  CK(cudaGetLastError());
  PlateauDev P;
  CK(cudaMemcpyAsync(&P, &ctx->d_frames[0].plat[0], sizeof(P), cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  memcpy(quad_px, P.quad_px, sizeof(double) * 8);
  *valid = P.valid;
  ctx->n_frames_last = 0;
  return SSD_OK;
}

int ssd_gpu_detect_front_edge(ssd_gpu_ctx *ctx, const uint8_t *image_host, double left_px[2], double right_px[2], int *valid)
{
  if(!ctx || !image_host || !left_px || !right_px || !valid)
    return SSD_E_INVALID_ARG;
  int rc = upload_image(ctx, image_host);
  if(rc)
    return rc;
  cudaStream_t st = ctx->stream[0];
  double *d_out = nullptr;
  CK(cudaMalloc(&d_out, sizeof(double) * 8));
  k_single_front_edge<<<1, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(ctx->dp, ctx->d_bev, ctx->smem_cap_words, d_out);
  double h[8];
  cudaError_t e = cudaMemcpyAsync(h, d_out, sizeof(double) * 5, cudaMemcpyDeviceToHost, st);
  if(e == cudaSuccess)
    e = cudaStreamSynchronize(st);
  cudaFree(d_out);
  CK(e);
  left_px[0] = h[0];
  left_px[1] = h[1];
  right_px[0] = h[2];
  right_px[1] = h[3];
  *valid = (int)h[4];
  ctx->n_frames_last = 0;
  return SSD_OK;
}

int ssd_gpu_points_in_quad(ssd_gpu_ctx *ctx, const double quad[8], const double *xy_host, int n, uint8_t *inside_host, int *ctor_status)
{
  if(!ctx || !quad || !xy_host || !inside_host || !ctor_status || n <= 0)
    return SSD_E_INVALID_ARG;
  CK(cudaSetDevice(ctx->device));
  double *d_q = nullptr, *d_xy = nullptr;
  unsigned char *d_in = nullptr;
  int *d_st = nullptr;
  cudaStream_t st = ctx->stream[0];
  CK(cudaMalloc(&d_q, sizeof(double) * 8));
  CK(cudaMalloc(&d_xy, sizeof(double) * 2 * (size_t)n));
  CK(cudaMalloc(&d_in, (size_t)n));
  CK(cudaMalloc(&d_st, sizeof(int)));
  cudaMemcpyAsync(d_q, quad, sizeof(double) * 8, cudaMemcpyHostToDevice, st);
  cudaMemcpyAsync(d_xy, xy_host, sizeof(double) * 2 * (size_t)n, cudaMemcpyHostToDevice, st);
  k_single_points_in_quad<<<std::min(1024, (n + 255) / 256), 256, 0, st>>>(d_q, d_xy, n, d_in, d_st);
  cudaMemcpyAsync(inside_host, d_in, (size_t)n, cudaMemcpyDeviceToHost, st);
  cudaMemcpyAsync(ctor_status, d_st, sizeof(int), cudaMemcpyDeviceToHost, st);
  const cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(d_q);
  cudaFree(d_xy);
  cudaFree(d_in);
  cudaFree(d_st);
  CK(e);
  return SSD_OK;
}

int ssd_gpu_camera_to_world(ssd_gpu_ctx *ctx, const float *xyz_host, int n, double *world_host)
{
  if(!ctx || !xyz_host || !world_host || n <= 0)
    return SSD_E_INVALID_ARG;
  CK(cudaSetDevice(ctx->device));
  float *d_in = nullptr;
  double *d_out = nullptr;
  cudaStream_t st = ctx->stream[0];
  CK(cudaMalloc(&d_in, sizeof(float) * 3 * (size_t)n));
  CK(cudaMalloc(&d_out, sizeof(double) * 3 * (size_t)n));
  cudaMemcpyAsync(d_in, xyz_host, sizeof(float) * 3 * (size_t)n, cudaMemcpyHostToDevice, st);
  k_single_camera_to_world<<<std::min(1024, (n + 255) / 256), 256, 0, st>>>(ctx->dp, d_in, n, d_out);
  cudaMemcpyAsync(world_host, d_out, sizeof(double) * 3 * (size_t)n, cudaMemcpyDeviceToHost, st);
  const cudaError_t e = cudaStreamSynchronize(st);
  cudaFree(d_in);
  cudaFree(d_out);
  CK(e);
  return SSD_OK;
}

// ---- raw memory helpers ----
int ssd_gpu_malloc(ssd_gpu_ctx *ctx, size_t bytes, void **dev_ptr)
{
  if(!ctx || !dev_ptr)
    return SSD_E_INVALID_ARG;
  CK(cudaSetDevice(ctx->device));
  const cudaError_t e = cudaMalloc(dev_ptr, bytes);
  if(e == cudaErrorMemoryAllocation)
  {
    cudaGetLastError();
    return fail(ctx, SSD_E_NOMEM, "cudaMalloc: out of memory");
  }
  CK(e);
  return SSD_OK;
}

int ssd_gpu_free(ssd_gpu_ctx *ctx, void *dev_ptr)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaFree(dev_ptr));
  return SSD_OK;
}

int ssd_gpu_memcpy_h2d(ssd_gpu_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy(dst_dev, src_host, bytes, cudaMemcpyHostToDevice));
  return SSD_OK;
}

int ssd_gpu_memcpy_d2h(ssd_gpu_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes)
{
  if(!ctx)
    return SSD_E_INVALID_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost));
  return SSD_OK;
}

int ssd_gpu_malloc_host(size_t bytes, void **host_ptr)
{
  if(!host_ptr)
    return SSD_E_INVALID_ARG;
  return cudaMallocHost(host_ptr, bytes) == cudaSuccess ? SSD_OK : SSD_E_NOMEM;
}

int ssd_gpu_free_host(void *host_ptr)
{
  return cudaFreeHost(host_ptr) == cudaSuccess ? SSD_OK : SSD_E_CUDA;
}

int ssd_gpu_register_host(void *host_ptr, size_t bytes)
{
  if(!host_ptr || !bytes)
    return SSD_E_INVALID_ARG;
  const cudaError_t e = cudaHostRegister(host_ptr, bytes, cudaHostRegisterPortable);
  if(e != cudaSuccess)
    cudaGetLastError(); // (not sticky: clear it for the next call)
  return e == cudaSuccess ? SSD_OK : (e == cudaErrorMemoryAllocation ? SSD_E_NOMEM : SSD_E_CUDA);
}

int ssd_gpu_unregister_host(void *host_ptr)
{
  if(!host_ptr)
    return SSD_E_INVALID_ARG;
  const cudaError_t e = cudaHostUnregister(host_ptr);
  if(e != cudaSuccess)
    cudaGetLastError();
  return e == cudaSuccess ? SSD_OK : SSD_E_CUDA;
}

} // extern "C"
