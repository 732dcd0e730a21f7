// ssd_gpu.cu -- context, launch chain and C ABI (include/ssd_gpu.h) of the B200 stair-step geometry path.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -fmad=false (see build.py). No CPU fallback.
#include "ssd_device.cuh"
#include "ssd_kernels_points.cuh"
#include "ssd_kernels_outline.cuh"
#include "ssd_kernels_stream.cuh"
#include "ssd_kernels_records.cuh"

#include <algorithm>
#include <cmath>
#include <cstdio>
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
  // knobs, read once in ssd_gpu_create (DESIGN.md): blocks per frame of the point kernels, small-batch split, depth A/B path
  int bpf_l_knob = 0, bpf_q_knob = 0;
  bool no_split_small = false, depth_unfused = false;
  cudaEvent_t ev_start{}, ev_stop{}, ev_h2d0{}, ev_h2d1{};
  cudaEvent_t ev_in_ready[SSD_MAX_STREAMS]{}, ev_in_free[SSD_MAX_STREAMS]{}, ev_chunk_done[SSD_MAX_STREAMS]{};
  FrameDev *d_frames = nullptr;   // max_frames
  FrameOut *d_out = nullptr;      // max_frames
  FrameOut *h_out = nullptr;      // pinned
  OverlayDev ov{};                // drawStairStep projection (ssd_gpu_set_overlay); off by default
  ssd_gpu_overlay *d_ovl = nullptr, *h_ovl = nullptr; // max_frames * SSD_GPU_MAX_STEPS, allocated by ssd_gpu_set_overlay
  unsigned char *d_labels = nullptr; // max_frames * N
  unsigned *d_bev = nullptr; // 2 x chunk_frames * MAX_PLATEAUS * bm_words (per stream)
  float *d_stage[SSD_MAX_STREAMS]{};            // vertex staging (host input / deprojected depth)
  int stage_frames[SSD_MAX_STREAMS]{};          // ... and its capacity in frames
  uint16_t *d_depth[SSD_MAX_STREAMS]{};         // z16 staging of the host depth-frame path
  float *d_xn = nullptr, *d_yn = nullptr;       // deprojection tables: (u - ppx) / fx per column, (v - ppy) / fy per row
  ssd_gpu_intrinsics intr{};                    // intrinsics the tables were built for
  // resident-frame path (ssd_kernels_stream.cuh): one persistent kernel per chunk instead of the three point passes
  bool resident = false;
  bool records = false;           // record chain (ssd_kernels_records.cuh): the default where the frame size admits it
  uint4 *d_rec4 = nullptr;        // n_streams x chunk_frames x N/4 x {4 records}
  // word-record chain (SSD_GPU_PATH=wordrec, experimental): k_label_bev<SRC, true> leaves 8 bytes per 4-pixel word of the
  // outlined plateaus, k_quad_reduce_rec takes the words that lie inside their step's quadrilateral from those
  bool wordrec = false;
  bool risers = false;            // ssd_gpu_set_vertical_faces: k_riser_reduce after the chain
  uint2 *d_wrec = nullptr;        // n_streams x chunk_frames x N/4
  int fs_grid = 0, fs_d_raw = 4, fs_d_rec = 0, fs_lag_frames = 8;
  GroupSum *d_sums = nullptr;     // n_streams x chunk_frames x N/32 summaries
  unsigned *d_done = nullptr;     // n_streams x chunk_frames frame counters (self-resetting)
  unsigned char *d_recs = nullptr; // record ring of k_frame_stream (one kernel at a time uses it): grid x 16 warps x fs_d_rec slots, L2-resident
  unsigned long long *d_prof = nullptr; // SSD_GPU_FS_PROF=1: cycle counters of k_frame_stream
  cudaEvent_t ev_fs{};            // the persistent kernels of consecutive chunks never overlap (each wants every SM)
  bool fs_pending = false;
  int pt_blocks_target = 0;       // blocks per launch of the tile-looping point kernels
  int n_frames_last = 0;
  int flags_last = 0;
  ssd_gpu_timing timing{};
  std::string err;
  // single-stage scratch
  unsigned char *d_img = nullptr;
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
};

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

// ProcessingConfiguration / Projection2D (pointcloud.cpp:60-106)
static int derive_params(const ssd_gpu_config &c, const ssd_gpu_transform &t, DevParams &d)
{
  memset(&d, 0, sizeof(d));
  if(c.width <= 0 || c.height <= 0 || !(c.x_max > c.x_min) || !(c.y_max > c.y_min) || !(c.z_max > c.z_min) || !(c.height_interval > 0))
    return SSD_E_INVALID_ARG;
  d.W = c.width;
  d.H = c.height;
  d.N = c.width * c.height;
  d.wpr = (c.width + 31) / 32;
  d.hir = 1.0 / c.height_interval;
  d.min_height = (uint16_t)((c.min_height_above_ground - c.z_min) * d.hir);
  d.min_img_y_extent = (int)(c.min_step_depth * c.height / (c.y_max - c.y_min));
  d.x_to_image = c.width / (c.x_max - c.x_min);
  d.y_to_image = c.height / (c.y_max - c.y_min);
  d.x_to_world = 1 / d.x_to_image;
  d.y_to_world = 1 / d.y_to_image;
  d.xy_ratio = d.x_to_image / d.y_to_image;
  d.n_bins = (int)((size_t)((c.z_max - c.z_min) * d.hir) + 1);
  d.min_peak_points = c.min_peak_points;
  d.bev_slots = SSD_GPU_MAX_PLATEAUS;
  d.tiles_per_frame = (d.N + SSD_TILE_POINTS - 1) / SSD_TILE_POINTS;
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
      const double gd = ((double)d.epsc * sx * 1.0001 + 8.0 * c.width / 16777216.0 + 1e-3) / 50.0;
      d.gcol_a = (float)(sx / 50.0);
      d.gcol_b = (float)((-c.x_min * sx - (c.width / 2 - 2)) / 50.0);
      d.gcol_lo = (float)(0.1 + gd);
      d.gcol_hi = (float)(1.0 - gd);
      d.gcol_tmax = (float)((c.width - 2 - (c.width / 2 - 2)) / 50.0 - gd);
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
  {
    // resident-frame path: record layout and the summary -> world-rectangle map (ssd_kernels_stream.cuh)
    int bx = 1, by = 1;
    while((1 << bx) < c.width)
      bx++;
    while((1 << by) < c.height + 1)
      by++;
    const int zbits = std::min(12, 32 - bx - by - 1); // (one bit: parity of the bin code)
    d.rec_bx = bx;
    d.rec_by = by;
    d.rec_zbits = 0;
    d.gs_steps = d.N / SSD_FS_STEP_PX;
    if(zbits >= 10 && d.N % SSD_FS_STEP_PX == 0 && c.width <= 0xfffe && c.height <= 0xfffe)
    {
      int sh = 0;
      while(sh < 24 && 0.5 * std::ldexp(c.height_interval, sh + 1) + 1.0 < std::ldexp(1.0, zbits - 1) - 1.0)
        sh++;
      d.rec_zbits = zbits;
      d.rec_zshift = sh;
      d.rec_mf = (float)std::ldexp(1.0 / d.hir, sh);
    }
    d.gs_xw = (float)d.x_to_world;
    d.gs_x0 = (float)c.x_min;
    d.gs_yw = (float)d.y_to_world;
    d.gs_y0 = (float)c.y_max;
    d.gs_margin = (float)(16.0 / 16777216.0 * (std::fabs(c.x_min) + std::fabs(c.x_max) + std::fabs(c.y_min) + std::fabs(c.y_max) + 1.0) + 1e-7);
  }
  if(d.n_bins < 3 || d.n_bins > SSD_GPU_MAX_BINS)
    return SSD_E_RANGE;
  if(d.N % 16 != 0)
    return SSD_E_INVALID_ARG; // vertices are loaded four at a time (three 16-byte loads), labels sixteen at a time
  if(c.width / 25 + 4 > SSD_MAX_SCANS || c.width / 50 + 6 > SSD_MAX_LINE_PTS || c.height / 10 + 2 > SSD_MAX_VPTS)
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

// The classic chain: k_transform_bin -> k_peaks -> k_label_bev -> k_outline -> k_frame_logic -> k_quad_reduce -> k_finalize
// (+ k_riser_reduce). CAM = NoCam: every frame with the context's own camera; CamTable: each frame with its camera's parameters
// (camera calls; the word-record variant is never taken there).
// sl: the chunk's z16 frames through ray tables (a call with a distorted lens), else nullptr. ov_lens: the lenses the overlay
// projects through (LensCam), else nullptr.
template<class CAM>
static int launch_classic(ssd_gpu_ctx *ctx, int s, const SrcVertices &sv, const SrcDepth &sd, const SrcLens *sl, int frame0, int nf, int *launches,
                          cudaEvent_t *ev, const CAM cam, const ssd_gpu_distortion *ov_lens)
{
#define STAGE_EV(i)                         \
  do                                        \
  {                                         \
    if(ev)                                  \
      CK(cudaEventRecord(ev[i], st));       \
  } while(0)
  const DevParams &p = ctx->dp;
  cudaStream_t st = ctx->stream[s];
  FrameDev *frames = ctx->d_frames + frame0;
  unsigned char *labels = ctx->d_labels + (size_t)frame0 * p.N;
  unsigned *bev = ctx->d_bev + (size_t)s * ctx->chunk_frames * SSD_GPU_MAX_PLATEAUS * ctx->bm_words;
  const dim3 gpt(p.tiles_per_frame, nf);
  const int tiles2 = (p.N + SSD_WT_PX * SSD_PT_WARPS - 1) / (SSD_WT_PX * SSD_PT_WARPS);
  const int bpf = std::max(1, std::min(tiles2, (ctx->pt_blocks_target + nf - 1) / nf));
  const int bpf_l = ctx->bpf_l_knob > 0 ? std::min(tiles2, ctx->bpf_l_knob) : bpf, bpf_q = ctx->bpf_q_knob > 0 ? std::min(tiles2, ctx->bpf_q_knob) : bpf;
  const dim3 gpt2l(bpf_l, nf), gpt2q(bpf_q, nf);
  const bool depth = sv.xyz == nullptr;
  const float *xyz_dev = sv.xyz;
  ssd_gpu_overlay *ovl = ctx->d_ovl ? ctx->d_ovl + (size_t)frame0 * SSD_GPU_MAX_STEPS : nullptr;
  // small batches (the reference's real use is one frame per call): the last block of a frame in k_transform_bin evaluates the
  // peaks and the last block in k_outline the frame logic -- five launches instead of seven
  const bool fused = nf <= SSD_FUSE_MAX_FRAMES && !ev;
  STAGE_EV(0);
  if(fused)
  {
    if(sl)
      k_transform_bin_lens<SSD_PT_ITERS, true, CAM><<<gpt, SSD_PT_THREADS, 0, st>>>(p, *sl, labels, frames, cam);
    else if(depth)
      k_transform_bin_depth<SSD_PT_ITERS, true, CAM><<<gpt, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, cam);
    else
      k_transform_bin<SSD_PT_ITERS, true, CAM><<<gpt, SSD_PT_THREADS, SSD_PT_ITERS * SSD_TB_STAGE_BYTES, st>>>(p, xyz_dev, labels, frames, cam);
  }
  else
  {
    if(sl)
      k_transform_bin_lens<SSD_PT_ITERS, false, CAM><<<gpt, SSD_PT_THREADS, 0, st>>>(p, *sl, labels, frames, cam);
    else if(depth)
      k_transform_bin_depth<SSD_PT_ITERS, false, CAM><<<gpt, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, cam);
    else
      k_transform_bin<SSD_PT_ITERS, false, CAM><<<gpt, SSD_PT_THREADS, SSD_PT_ITERS * SSD_TB_STAGE_BYTES, st>>>(p, xyz_dev, labels, frames, cam);
  }
  STAGE_EV(1);
  if(!fused)
    k_peaks<<<nf, 32, 0, st>>>(p, frames, nf);
  STAGE_EV(2);
  constexpr bool plain = std::is_same<CAM, NoCam>::value;
  uint2 *wrec = plain && ctx->wordrec ? ctx->d_wrec + (size_t)s * ctx->chunk_frames * (size_t)(p.N / 4) : nullptr;
  if constexpr(plain)
  {
    if(wrec)
    {
      if(depth)
        k_label_bev<SrcDepth, true><<<gpt2l, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, bev, ctx->bm_words, wrec);
      else
        k_label_bev<SrcVertices, true><<<gpt2l, SSD_PT_THREADS, 0, st>>>(p, sv, labels, frames, bev, ctx->bm_words, wrec);
    }
  }
  if(!wrec)
  {
    if(sl)
      k_label_bev<SrcLens, false, CAM><<<gpt2l, SSD_PT_THREADS, 0, st>>>(p, *sl, labels, frames, bev, ctx->bm_words, nullptr, cam);
    else if(depth)
      k_label_bev<SrcDepth, false, CAM><<<gpt2l, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, bev, ctx->bm_words, nullptr, cam);
    else
      k_label_bev<SrcVertices, false, CAM><<<gpt2l, SSD_PT_THREADS, 0, st>>>(p, sv, labels, frames, bev, ctx->bm_words, nullptr, cam);
  }
  STAGE_EV(3);
  if(fused)
  {
    if(ctx->outline_small)
      k_outline<OutlineSharedSmall, true, CAM><<<dim3(ctx->outline_gridx, nf), SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words, cam);
    else
      k_outline<OutlineShared, true, CAM><<<dim3(ctx->outline_gridx, nf), OutlineShared::THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words, cam);
  }
  else
  {
    if(ctx->outline_small)
      k_outline<OutlineSharedSmall><<<dim3(ctx->outline_gridx, nf), SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words);
    else
      k_outline<OutlineShared><<<dim3(ctx->outline_gridx, nf), OutlineShared::THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words);
  }
  STAGE_EV(4);
  if(!fused)
    k_frame_logic<CAM><<<nf, 32, 0, st>>>(p, frames, nf, cam);
  STAGE_EV(5);
  if constexpr(plain)
  {
    if(wrec)
    {
      if(depth)
        k_quad_reduce_rec<SrcDepth><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, bev, ctx->bm_words, wrec);
      else
        k_quad_reduce_rec<SrcVertices><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sv, labels, frames, bev, ctx->bm_words, wrec);
    }
  }
  if(!wrec)
  {
    if(sl)
      k_quad_reduce<SrcLens, CAM><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, *sl, labels, frames, bev, ctx->bm_words, cam);
    else if(depth)
      k_quad_reduce<SrcDepth, CAM><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, bev, ctx->bm_words, cam);
    else
      k_quad_reduce<SrcVertices, CAM><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sv, labels, frames, bev, ctx->bm_words, cam);
  }
  STAGE_EV(6);
  if(ov_lens)
  {
    const LensCam<CAM> lc = { cam, ov_lens };
    if(ctx->outline_small)
      k_finalize<OutlineSharedSmall, LensCam<CAM>><<<nf, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + frame0, bev, ctx->bm_words,
                                                                                             ctx->smem_cap_words, ctx->ov, ovl, lc);
    else
      k_finalize<OutlineShared, LensCam<CAM>><<<nf, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + frame0, bev, ctx->bm_words,
                                                                                        ctx->smem_cap_words, ctx->ov, ovl, lc);
  }
  else if(ctx->outline_small)
    k_finalize<OutlineSharedSmall, CAM><<<nf, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + frame0, bev, ctx->bm_words, ctx->smem_cap_words,
                                                                               ctx->ov, ovl, cam);
  else
    k_finalize<OutlineShared, CAM><<<nf, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + frame0, bev, ctx->bm_words, ctx->smem_cap_words,
                                                                          ctx->ov, ovl, cam);
  STAGE_EV(7);
#undef STAGE_EV
  *launches += fused ? SSD_GPU_N_STAGES - 2 : SSD_GPU_N_STAGES;
  if(ctx->risers)
  {
    // optional fourth pass: vertical faces from the remainder (labels are final once the chain's label kernel has run)
    if(sl)
      k_riser_reduce<SrcLens, CAM><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, *sl, labels, frames, cam);
    else if(depth)
      k_riser_reduce<SrcDepth, CAM><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, cam);
    else
      k_riser_reduce<SrcVertices, CAM><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sv, labels, frames, cam);
    *launches += 1;
  }
  CK(cudaGetLastError());
  return SSD_OK;
}


// ---------------------------------------------------------------------------------------------
// the launch chain for one chunk of frames on one stream
// ---------------------------------------------------------------------------------------------
// xyz_dev: packed vertices of the chunk, or nullptr with z16_dev: the chunk's depth frames, deprojected inside the
// three point kernels (SrcDepth). cam: the camera table of a camera call (classic chain only), else nullptr.
// sl: the call's lens source (its z16 member is set here), else nullptr; ov_lens: see launch_classic.
static int launch_chunk(ssd_gpu_ctx *ctx, int s, const float *xyz_dev, const uint16_t *z16_dev, float depth_unit, int frame0, int nf, int *launches,
                        cudaEvent_t *ev, const CamTable *cam, const SrcLens *sl, const ssd_gpu_distortion *ov_lens)
{
#define STAGE_EV(i)                         \
  do                                        \
  {                                         \
    if(ev)                                  \
      CK(cudaEventRecord(ev[i], st));       \
  } while(0)
  const DevParams &p = ctx->dp;
  cudaStream_t st = ctx->stream[s];
  FrameDev *frames = ctx->d_frames + frame0;
  unsigned char *labels = ctx->d_labels + (size_t)frame0 * p.N;
  unsigned *bev = ctx->d_bev + (size_t)s * ctx->chunk_frames * SSD_GPU_MAX_PLATEAUS * ctx->bm_words;
  const dim3 gpt(p.tiles_per_frame, nf);
  // k_label_bev / k_quad_reduce: each block loops over tiles of its frame; enough blocks for ~6 waves of the GPU
  const int tiles2 = (p.N + SSD_WT_PX * SSD_PT_WARPS - 1) / (SSD_WT_PX * SSD_PT_WARPS); // at least one warp-tile per warp
  const int bpf = std::max(1, std::min(tiles2, (ctx->pt_blocks_target + nf - 1) / nf));
  const int bpf_l = ctx->bpf_l_knob > 0 ? std::min(tiles2, ctx->bpf_l_knob) : bpf, bpf_q = ctx->bpf_q_knob > 0 ? std::min(tiles2, ctx->bpf_q_knob) : bpf;
  const dim3 gpt2l(bpf_l, nf), gpt2q(bpf_q, nf);
  const bool depth = xyz_dev == nullptr;
  SrcVertices sv;
  sv.xyz = xyz_dev;
  SrcDepth sd;
  sd.z16 = z16_dev;
  sd.xn = ctx->d_xn;
  sd.yn = ctx->d_yn;
  sd.unit = depth_unit;
  sd.wmagic = (((unsigned long long)1 << 40) + (unsigned long long)p.W - 1) / (unsigned long long)p.W;
  // optional fourth pass: vertical faces from the remainder (labels are final once the chain's label kernel has run)
  auto launch_risers = [&]()
  {
    if(!ctx->risers)
      return;
    if(depth)
      k_riser_reduce<SrcDepth><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames);
    else
      k_riser_reduce<SrcVertices><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sv, labels, frames);
    *launches += 1;
  };

  SrcLens sll;
  if(sl)
  {
    sll = *sl;
    sll.z16 = z16_dev;
  }
  if(cam)
  {
    CamTable c = *cam;
    c.frame0 = frame0;
    return launch_classic(ctx, s, sv, sd, sl ? &sll : nullptr, frame0, nf, launches, ev, c, ov_lens);
  }
  if(ctx->records)
  {
    // ---- record chain: k_transform_rec -> k_peaks -> k_label_sum -> k_outline -> k_frame_logic -> k_quad_sum -> k_finalize ----
    uint4 *recs = ctx->d_rec4 + (size_t)s * ctx->chunk_frames * (size_t)(p.N / 4);
    STAGE_EV(0);
    if(depth)
      k_transform_rec_depth<SSD_PT_ITERS><<<gpt, SSD_PT_THREADS, 0, st>>>(p, sd, labels, recs, frames);
    else
      k_transform_rec<SSD_PT_ITERS><<<gpt, SSD_PT_THREADS, SSD_PT_ITERS * SSD_TB_STAGE_BYTES, st>>>(p, xyz_dev, labels, recs, frames);
    STAGE_EV(1);
    k_peaks<<<nf, 32, 0, st>>>(p, frames, nf);
    STAGE_EV(2);
    if(depth)
      k_label_rec<SrcDepth><<<gpt2l, SSD_PT_THREADS, 0, st>>>(p, sd, labels, recs, frames, bev, ctx->bm_words);
    else
      k_label_rec<SrcVertices><<<gpt2l, SSD_PT_THREADS, 0, st>>>(p, sv, labels, recs, frames, bev, ctx->bm_words);
    STAGE_EV(3);
    if(ctx->outline_small)
      k_outline<OutlineSharedSmall><<<dim3(ctx->outline_gridx, nf), SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words);
    else
      k_outline<OutlineShared><<<dim3(ctx->outline_gridx, nf), OutlineShared::THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words);
    STAGE_EV(4);
    k_frame_logic<<<nf, 32, 0, st>>>(p, frames, nf);
    STAGE_EV(5);
    if(depth)
      k_quad_rec<SrcDepth><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, bev, ctx->bm_words, recs);
    else
      k_quad_rec<SrcVertices><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sv, labels, frames, bev, ctx->bm_words, recs);
    STAGE_EV(6);
    if(ctx->outline_small)
      k_finalize<OutlineSharedSmall><<<nf, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + frame0, bev, ctx->bm_words, ctx->smem_cap_words, ctx->ov,
                                                                            ctx->d_ovl ? ctx->d_ovl + (size_t)frame0 * SSD_GPU_MAX_STEPS : nullptr);
    else
      k_finalize<OutlineShared><<<nf, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + frame0, bev, ctx->bm_words, ctx->smem_cap_words, ctx->ov,
                                                                            ctx->d_ovl ? ctx->d_ovl + (size_t)frame0 * SSD_GPU_MAX_STEPS : nullptr);
    STAGE_EV(7);
    *launches += SSD_GPU_N_STAGES;
    launch_risers();
    CK(cudaGetLastError());
    return SSD_OK;
  }
  if(ctx->resident)
  {
    // ---- resident-frame chain: k_frame_stream -> k_outline -> k_frame_logic -> k_quad_sum -> k_finalize ----
    FsParams a;
    a.n_frames = nf;
    a.d_raw = ctx->fs_d_raw;
    a.d_rec = ctx->fs_d_rec;
    a.flags = 0;
    a.done = ctx->d_done + (size_t)s * ctx->chunk_frames;
    a.sums = ctx->d_sums + (size_t)s * ctx->chunk_frames * (size_t)(p.N / 32);
    a.recs = ctx->d_recs;
    a.prof = ctx->d_prof;
    a.prof_warp_off = FS_PROF_HDR + (size_t)FS_PROF_PER_FRAME * ctx->chunk_frames;
    if(ctx->d_prof)
    {
      std::vector<unsigned long long> init(FS_PROF_HDR + (size_t)FS_PROF_PER_FRAME * ctx->chunk_frames + (size_t)8 * ctx->fs_grid * SSD_FS_WARPS, 0ull);
      for(int f = 0; f < ctx->chunk_frames; f++)
        init[FS_PROF_HDR + (size_t)f * FS_PROF_PER_FRAME + 0] = init[FS_PROF_HDR + (size_t)f * FS_PROF_PER_FRAME + 3] = ~0ull;
      CK(cudaStreamSynchronize(st));
      CK(cudaMemcpy(ctx->d_prof, init.data(), init.size() * 8, cudaMemcpyHostToDevice));
    }
    size_t bmw = ctx->bm_words;
    DevParams pp = p;
    if(ctx->fs_pending)
      CK(cudaStreamWaitEvent(st, ctx->ev_fs, 0));
    STAGE_EV(0);
    if(depth)
    {
      void *args[] = { &pp, &sd, &a, &labels, &frames, &bev, &bmw };
      CK(cudaLaunchCooperativeKernel((const void *)k_frame_stream<SrcDepth>, dim3(ctx->fs_grid), dim3(SSD_FS_THREADS), args,
                                     fs_smem_bytes(FsSrc<SrcDepth>::STEP_BYTES, a.d_raw, a.d_rec), st));
    }
    else
    {
      void *args[] = { &pp, &sv, &a, &labels, &frames, &bev, &bmw };
      CK(cudaLaunchCooperativeKernel((const void *)k_frame_stream<SrcVertices>, dim3(ctx->fs_grid), dim3(SSD_FS_THREADS), args,
                                     fs_smem_bytes(FsSrc<SrcVertices>::STEP_BYTES, a.d_raw, a.d_rec), st));
    }
    CK(cudaEventRecord(ctx->ev_fs, st));
    ctx->fs_pending = true;
    STAGE_EV(1);
    STAGE_EV(2);
    STAGE_EV(3);
    if(ctx->outline_small)
      k_outline<OutlineSharedSmall><<<dim3(ctx->outline_gridx, nf), SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words);
    else
      k_outline<OutlineShared><<<dim3(ctx->outline_gridx, nf), OutlineShared::THREADS, ctx->ol_dyn_smem, st>>>(p, frames, bev, ctx->bm_words, ctx->smem_cap_words);
    STAGE_EV(4);
    k_frame_logic<<<nf, 32, 0, st>>>(p, frames, nf);
    STAGE_EV(5);
    if(depth)
      k_quad_sum<SrcDepth><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sd, labels, frames, bev, ctx->bm_words, a.sums, nullptr);
    else
      k_quad_sum<SrcVertices><<<gpt2q, SSD_PT_THREADS, 0, st>>>(p, sv, labels, frames, bev, ctx->bm_words, a.sums, nullptr);
    STAGE_EV(6);
    if(ctx->outline_small)
      k_finalize<OutlineSharedSmall><<<nf, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + frame0, bev, ctx->bm_words, ctx->smem_cap_words, ctx->ov,
                                                                            ctx->d_ovl ? ctx->d_ovl + (size_t)frame0 * SSD_GPU_MAX_STEPS : nullptr);
    else
      k_finalize<OutlineShared><<<nf, SSD_OL_THREADS, ctx->ol_dyn_smem, st>>>(p, frames, ctx->d_out + frame0, bev, ctx->bm_words, ctx->smem_cap_words, ctx->ov,
                                                                            ctx->d_ovl ? ctx->d_ovl + (size_t)frame0 * SSD_GPU_MAX_STEPS : nullptr);
    STAGE_EV(7);
    *launches += 5;
    launch_risers();
    CK(cudaGetLastError());
    return SSD_OK;
  }
  return launch_classic(ctx, s, sv, sd, sl ? &sll : nullptr, frame0, nf, launches, ev, NoCam(), ov_lens);
#undef STAGE_EV
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
  cudaFree(ctx->d_bev);
  cudaFree(ctx->d_sums);
  cudaFree(ctx->d_done);
  cudaFree(ctx->d_recs);
  cudaFree(ctx->d_rec4);
  cudaFree(ctx->d_wrec);
  cudaFree(ctx->d_prof);
  if(ctx->ev_fs)
    cudaEventDestroy(ctx->ev_fs);
  cudaFree(ctx->d_img);
  cudaFree(ctx->d_xn);
  cudaFree(ctx->d_yn);
  cudaFree(ctx->d_cam_dp);
  cudaFree(ctx->d_cam_ov);
  cudaFree(ctx->d_cam_xn);
  cudaFree(ctx->d_cam_yn);
  cudaFree(ctx->d_cam_unit);
  cudaFree(ctx->d_cam_of_frame);
  for(float2 *t : ctx->cam_rays)
    cudaFree(t);
  cudaFree(ctx->d_cam_ray);
  cudaFree(ctx->d_cam_lens);
  cudaFree(ctx->d_ray);
  cudaFree(ctx->d_lens);
  for(int i = 0; i < SSD_MAX_STREAMS; i++)
  {
    cudaFree(ctx->d_stage[i]);
    cudaFree(ctx->d_depth[i]);
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
  if(!cfg || !xf || !out || max_frames <= 0)
    return fail(nullptr, SSD_E_INVALID_ARG, "ssd_gpu_create: bad argument");
  *out = nullptr;
  int ndev = 0;
  if(cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, SSD_E_CUDA, "ssd_gpu_create: no CUDA device (this library has no CPU fallback)");
  if(device < 0 || device >= ndev)
    return fail(nullptr, SSD_E_INVALID_ARG, "ssd_gpu_create: bad device index");
  DevParams dp;
  const int rc = derive_params(*cfg, *xf, dp);
  if(rc)
    return fail(nullptr, rc, "ssd_gpu_create: configuration out of range (3 <= height bins <= 253, width*height % 16 == 0, width <= 4700, height <= 5100)");

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
      cudaFuncSetAttribute(k_outline<OutlineShared, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_outline<OutlineSharedSmall, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_finalize<OutlineShared>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_finalize<OutlineSharedSmall>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      // the camera-table variants (ssd_gpu_set_cameras) of the kernels with a dynamic work area
      cudaFuncSetAttribute(k_outline<OutlineShared, true, CamTable>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_outline<OutlineSharedSmall, true, CamTable>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_finalize<OutlineShared, CamTable>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_finalize<OutlineSharedSmall, CamTable>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      // the overlay through a distorted lens (ssd_gpu_set_distortion / ssd_gpu_set_cameras_ex)
      cudaFuncSetAttribute(k_finalize<OutlineShared, LensCam<NoCam>>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_finalize<OutlineSharedSmall, LensCam<NoCam>>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_finalize<OutlineShared, LensCam<CamTable>>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
      cudaFuncSetAttribute(k_finalize<OutlineSharedSmall, LensCam<CamTable>>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn);
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
  if(const char *e = getenv("SSD_GPU_DEPTH_UNFUSED"))
    ctx->depth_unfused = atoi(e) != 0;
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
  {
    // Resident-frame path: used when a frame's records fit the shared memory of the GPU with room for the frame barrier's
    // latency (every warp must hold all its steps of one frame, plus what it works ahead). SSD_GPU_PATH=classic|resident.
    const char *pe = getenv("SSD_GPU_PATH");
    const bool want = pe && !strcmp(pe, "resident"); // experimental: measured slower than the record chain (DESIGN.md)
    // word-record chain (experimental: measured slower than the classic chain, DESIGN.md): box coordinates are 12 bits each
    if(pe && !strcmp(pe, "wordrec") && dp.W <= 4096 && dp.H <= 4096)
    {
      ctx->wordrec = true;
      CKC(cudaMalloc(&ctx->d_wrec, (size_t)ctx->n_streams * ctx->chunk_frames * (size_t)(dp.N / 4) * sizeof(uint2)));
    }
    if(pe && !strcmp(pe, "wordrec") && !ctx->wordrec)
      return bail("SSD_GPU_PATH=wordrec: the frame size does not admit the word-record chain", SSD_E_RANGE);
    if(pe && !strcmp(pe, "records") && dp.rec_zbits > 0) // experimental: measured slower than the classic chain (DESIGN.md)
    {
      ctx->records = true;
      CKC(cudaMalloc(&ctx->d_rec4, (size_t)ctx->n_streams * ctx->chunk_frames * (size_t)(dp.N / 4) * sizeof(uint4)));
      if(cudaFuncSetAttribute(k_transform_rec<SSD_PT_ITERS>, cudaFuncAttributeMaxDynamicSharedMemorySize, SSD_PT_ITERS * SSD_TB_STAGE_BYTES) != cudaSuccess)
        return bail("cudaFuncSetAttribute(k_transform_rec) failed", SSD_E_CUDA);
    }
    if(pe && !strcmp(pe, "records") && !ctx->records)
      return bail("SSD_GPU_PATH=records: the frame size does not admit the record chain", SSD_E_RANGE);
    int sms = 148, coop = 0;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
    if(const char *e = getenv("SSD_GPU_FS_RAW"))
      ctx->fs_d_raw = std::max(2, atoi(e));
    if(const char *e = getenv("SSD_GPU_FS_REC"))
      ctx->fs_d_rec = std::max(2, atoi(e));
    int grid = sms;
    if(const char *e = getenv("SSD_GPU_FS_CTAS"))
      grid = std::max(1, std::min(sms, atoi(e)));
    if(want && coop && dp.rec_zbits > 0 && dp.gs_steps % SSD_FS_SUB == 0 && dp.gs_steps / SSD_FS_SUB >= 64)
    {
      // record ring: fs_lag_frames frames of a warp's steps (phase 2 may trail phase 1 by that much: the frame barrier's
      // latency and the skew between the CTAs disappear in it); ~3.9 MB per frame at 1024x768, re-used before L2 evicts it
      if(const char *e = getenv("SSD_GPU_FS_LAG"))
        ctx->fs_lag_frames = std::max(1, std::min(SSD_FS_NB - 3, atoi(e)));
      const long long S = dp.gs_steps / SSD_FS_SUB, TW = (long long)grid * SSD_FS_WARPS;
      const int per_warp = (int)((S + TW - 1) / TW);
      if(!ctx->fs_d_rec)
        ctx->fs_d_rec = (int)((ctx->fs_lag_frames * S + TW - 1) / TW) + 2;
      ctx->fs_d_rec = std::max(ctx->fs_d_rec, per_warp + 2);
      const size_t sm_v = fs_smem_bytes(FsSrc<SrcVertices>::STEP_BYTES, ctx->fs_d_raw, ctx->fs_d_rec);
      const size_t sm_d = fs_smem_bytes(FsSrc<SrcDepth>::STEP_BYTES, ctx->fs_d_raw, ctx->fs_d_rec);
      int occ = 0;
      if(sm_v <= (size_t)max_optin &&
         cudaFuncSetAttribute(k_frame_stream<SrcVertices>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_v) == cudaSuccess &&
         cudaFuncSetAttribute(k_frame_stream<SrcDepth>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm_d) == cudaSuccess &&
         cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_frame_stream<SrcVertices>, SSD_FS_THREADS, sm_v) == cudaSuccess && occ >= 1)
      {
        ctx->resident = true;
        ctx->fs_grid = grid;
        const size_t n_sums = (size_t)ctx->n_streams * ctx->chunk_frames * (size_t)(dp.N / 32);
        CKC(cudaMalloc(&ctx->d_sums, n_sums * sizeof(GroupSum)));
        CKC(cudaMalloc(&ctx->d_done, (size_t)ctx->n_streams * ctx->chunk_frames * sizeof(unsigned)));
        CKC(cudaMalloc(&ctx->d_recs, (size_t)grid * SSD_FS_WARPS * ctx->fs_d_rec * SSD_FS_REC_BYTES * SSD_FS_SUB));
        CKC(cudaMemset(ctx->d_done, 0, (size_t)ctx->n_streams * ctx->chunk_frames * sizeof(unsigned)));
        CKC(cudaEventCreateWithFlags(&ctx->ev_fs, cudaEventDisableTiming));
        if(getenv("SSD_GPU_FS_PROF"))
        {
          CKC(cudaMalloc(&ctx->d_prof, 8 * (FS_PROF_HDR + (size_t)FS_PROF_PER_FRAME * ctx->chunk_frames + (size_t)8 * grid * SSD_FS_WARPS)));
        }
      }
      cudaGetLastError();
    }
    if(pe && !strcmp(pe, "resident") && !ctx->resident)
      return bail("SSD_GPU_PATH=resident: the frame size does not admit the resident-frame path", SSD_E_RANGE);
  }
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
    k_lens_rays<<<(int)std::min<size_t>(((size_t)p.N + 255) / 256, 4096), 256, 0, st>>>(p.W, p.H, in, d, ray, d_bad);
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
  if(p.W % 4 != 0)
    return fail(ctx, SSD_E_INVALID_ARG, "depth input: the frame width must be a multiple of 4");
  if(!ctx->d_xn)
  {
    CK(cudaMalloc(&ctx->d_xn, sizeof(float) * (size_t)p.W));
    CK(cudaMalloc(&ctx->d_yn, sizeof(float) * (size_t)p.H));
    memset(&ctx->intr, 0, sizeof(ctx->intr));
  }
  if(memcmp(&ctx->intr, &in, sizeof(float) * 5) != 0)
  {
    const int n = std::max(p.W, p.H);
    k_deproject_tables<<<(n + 255) / 256, 256, 0, ctx->stream[0]>>>(p.W, p.H, in, ctx->d_xn, ctx->d_yn);
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

// xyz != nullptr: packed vertices; else z16 depth frames + intrinsics (deprojected chunk by chunk into the vertex staging)
// cam_of_frame != nullptr: a camera call (validated by check_cameras; the depth tables are the camera table's, intr is unused)
static int process_impl(ssd_gpu_ctx *ctx, const float *xyz, const uint16_t *z16, const ssd_gpu_intrinsics *intr, bool host_input, int n_frames,
                        int flags, const int32_t *cam_of_frame)
{
  if(!ctx || (!xyz && !(z16 && (intr || cam_of_frame))) || n_frames <= 0)
    return fail(ctx, SSD_E_INVALID_ARG, "process: bad argument");
  if(n_frames > ctx->max_frames)
    return fail(ctx, SSD_E_RANGE, "process: n_frames exceeds max_frames of the context");
  // the point kernels use 16-byte vector loads / bulk copies (vertices) and 8-byte loads (depth)
  if((xyz && ((uintptr_t)xyz & 15u)) || (z16 && ((uintptr_t)z16 & 7u)))
    return fail(ctx, SSD_E_INVALID_ARG, "process: the input buffer must be 16-byte aligned (vertices) / 8-byte aligned (depth)");
  CK(cudaSetDevice(ctx->device));
  const DevParams &p = ctx->dp;
  const size_t frame_floats = (size_t)p.N * 3;
  // host input: every byte crosses PCIe, the copy of chunk i+1 overlaps the kernels of chunk i and only the last
  // chunk's kernels stay exposed -- small chunks. Device input: large chunks (the per-frame kernels need the parallelism).
  int cf = host_input ? ctx->host_chunk_frames : ctx->chunk_frames;
  // a device-resident batch that fits one chunk is still split over the streams, so that one half's latency-bound
  // per-plateau kernels overlap the other half's point kernels (measured: 64 frames of 4096x3072 as 2 x 32: +5 %;
  // below ~32 frames per chain the per-frame kernels lose more parallelism than the overlap returns)
  if(!host_input && !(flags & SSD_FLAG_SINGLE_STREAM) && ctx->n_streams > 1 && n_frames <= cf && !ctx->no_split_small)
  {
    const int half = (n_frames + ctx->n_streams - 1) / ctx->n_streams;
    if(half >= 32)
      cf = half;
  }
  const bool depth_input = xyz == nullptr;
  // a distorted lens: depth frames read their rays from ray tables (SrcLens), the overlay projects through the lens (LensCam)
  const bool plain_lens = !cam_of_frame && !ssd_lens_is_pinhole(&ctx->lens);
  SrcLens sl{};
  bool use_lens = false;
  const ssd_gpu_distortion *ov_lens = nullptr;
  if(cam_of_frame)
  {
    for(int f = 0; f < n_frames && depth_input && ctx->cams_distorted && !use_lens; f++)
      use_lens = ctx->cam_distorted[cam_of_frame[f]] != 0;
    sl.cam_ray = ctx->d_cam_ray;
    if(ctx->cams_distorted && ctx->ov.enabled)
      ov_lens = ctx->d_cam_lens;
  }
  else if(plain_lens)
  {
    use_lens = depth_input;
    if(ctx->ov.enabled)
      ov_lens = ctx->d_lens;
  }
  if(depth_input && !cam_of_frame)
  {
    const int rc = ensure_deproject_tables(ctx, *intr);
    if(rc)
      return rc;
    sl.ray = ctx->d_ray;
    sl.unit = intr->depth_unit;
  }
  // depth frames are deprojected inside the point kernels (SrcDepth): no vertex array is ever written.
  const bool unfused = ctx->depth_unfused; // A/B switch (SSD_GPU_DEPTH_UNFUSED, read in ssd_gpu_create)
  if(host_input || depth_input)
    for(int i = 0; i < ctx->n_streams; i++)
    {
      if(depth_input && !unfused)
      {
        if(host_input && !ctx->d_depth[i])
          CK(cudaMalloc(&ctx->d_depth[i], (size_t)ctx->host_chunk_frames * p.N * sizeof(uint16_t)));
        continue;
      }
      if(ctx->stage_frames[i] < cf) // grows once when a device-depth call follows host-input calls
      {
        CK(cudaDeviceSynchronize());
        if(ctx->d_stage[i])
          CK(cudaFree(ctx->d_stage[i]));
        ctx->d_stage[i] = nullptr;
        CK(cudaMalloc(&ctx->d_stage[i], (size_t)cf * frame_floats * sizeof(float)));
        ctx->stage_frames[i] = cf;
      }
      if(depth_input && host_input && !ctx->d_depth[i])
        CK(cudaMalloc(&ctx->d_depth[i], (size_t)ctx->host_chunk_frames * p.N * sizeof(uint16_t)));
    }

  int launches = 0;
  const bool stage_timing = (flags & SSD_FLAG_STAGE_TIMING) != 0;
  const int n_chunks = (n_frames + cf - 1) / cf;
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
  // the whole call is ordered after ev_start on stream 0; stream 1 joins via events
  CK(cudaEventRecord(ctx->ev_start, ctx->stream[0]));
  for(int i = 1; i < ctx->n_streams; i++)
    CK(cudaStreamWaitEvent(ctx->stream[i], ctx->ev_start, 0));
  CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_start, 0));
  if(host_input)
    CK(cudaEventRecord(ctx->ev_h2d0, ctx->copy_stream));
  // per-frame state: histogram must start at zero
  CK(cudaMemsetAsync(ctx->d_frames, 0, sizeof(FrameDev) * (size_t)n_frames, ctx->stream[0]));
  if(cam_of_frame)
    CK(cudaMemcpyAsync(ctx->d_cam_of_frame, cam_of_frame, sizeof(int32_t) * (size_t)n_frames, cudaMemcpyHostToDevice, ctx->stream[0]));
  CK(cudaEventRecord(ctx->ev_chunk_done[0], ctx->stream[0]));
  for(int i = 1; i < ctx->n_streams; i++)
    CK(cudaStreamWaitEvent(ctx->stream[i], ctx->ev_chunk_done[0], 0));

  int chunk = 0;
  for(int f0 = 0; f0 < n_frames; f0 += cf, chunk++)
  {
    const int nf = std::min(cf, n_frames - f0);
    const int s = (flags & SSD_FLAG_SINGLE_STREAM) ? 0 : chunk % ctx->n_streams;
    const float *src = depth_input ? nullptr : xyz + (size_t)f0 * frame_floats;
    const uint16_t *dsrc = depth_input ? z16 + (size_t)f0 * p.N : nullptr;
    if(host_input)
    {
      // staging buffer s may be overwritten once the chunk that last used it has consumed it
      if(chunk >= ((flags & SSD_FLAG_SINGLE_STREAM) ? 1 : ctx->n_streams))
        CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_in_free[s], 0));
      if(depth_input)
      {
        CK(cudaMemcpyAsync(ctx->d_depth[s], dsrc, (size_t)nf * p.N * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->copy_stream));
        dsrc = ctx->d_depth[s];
      }
      else
      {
        CK(cudaMemcpyAsync(ctx->d_stage[s], src, (size_t)nf * frame_floats * sizeof(float), cudaMemcpyHostToDevice, ctx->copy_stream));
        src = ctx->d_stage[s];
      }
      CK(cudaEventRecord(ctx->ev_in_ready[s], ctx->copy_stream));
      CK(cudaStreamWaitEvent(ctx->stream[s], ctx->ev_in_ready[s], 0));
    }
    if(depth_input && unfused)
    {
      // A/B path (SSD_GPU_DEPTH_UNFUSED=1): materialise the vertices, then the vertex kernels
      // (the vertex staging of stream s is free: the chunk that used it last ran on this very stream)
      if(use_lens)
        k_deproject_lens<<<dim3((p.N / 4 + 255) / 256, nf), 256, 0, ctx->stream[s]>>>(p.N, intr->depth_unit, ctx->d_ray, dsrc, ctx->d_stage[s]);
      else
        k_deproject<<<dim3((p.N / 4 + 255) / 256, nf), 256, 0, ctx->stream[s]>>>(p.W, p.N, intr->depth_unit, ctx->d_xn, ctx->d_yn, dsrc, ctx->d_stage[s]);
      launches++;
      src = ctx->d_stage[s];
      if(host_input)
        CK(cudaEventRecord(ctx->ev_in_free[s], ctx->stream[s])); // the z16 staging is consumed
    }
    const bool fused = depth_input && !unfused;
    const int rc = launch_chunk(ctx, s, fused ? nullptr : src, fused ? dsrc : nullptr, fused && intr ? intr->depth_unit : 0.f, f0, nf, &launches,
                                stage_timing ? &ctx->stage_ev[(size_t)chunk * (SSD_GPU_N_STAGES + 1)] : nullptr, cam_of_frame ? &cams : nullptr,
                                fused && use_lens ? &sl : nullptr, ov_lens);
    if(rc)
      return rc;
    if(host_input && (!depth_input || fused))
      CK(cudaEventRecord(ctx->ev_in_free[s], ctx->stream[s])); // all three passes have read the staging
  }
  if(host_input)
    CK(cudaEventRecord(ctx->ev_h2d1, ctx->copy_stream));
  // join stream 1 into stream 0, then bring the compact results home
  for(int i = 1; i < ctx->n_streams; i++)
  {
    CK(cudaEventRecord(ctx->ev_chunk_done[i], ctx->stream[i]));
    CK(cudaStreamWaitEvent(ctx->stream[0], ctx->ev_chunk_done[i], 0));
  }
  CK(cudaMemcpyAsync(ctx->h_out, ctx->d_out, sizeof(FrameOut) * (size_t)n_frames, cudaMemcpyDeviceToHost, ctx->stream[0]));
  if(ctx->ov.enabled)
    CK(cudaMemcpyAsync(ctx->h_ovl, ctx->d_ovl, sizeof(ssd_gpu_overlay) * SSD_GPU_MAX_STEPS * (size_t)n_frames, cudaMemcpyDeviceToHost, ctx->stream[0]));
  CK(cudaEventRecord(ctx->ev_stop, ctx->stream[0]));
  CK(cudaEventSynchronize(ctx->ev_stop));
  CK(cudaGetLastError());
  if(ctx->d_prof)
  {
    // (profiling runs use one chunk per call: the buffer is reset before every launch)
    const int nf = std::min(n_frames, ctx->chunk_frames);
    const size_t woff = FS_PROF_HDR + (size_t)FS_PROF_PER_FRAME * ctx->chunk_frames;
    std::vector<unsigned long long> h(woff + (size_t)8 * ctx->fs_grid * SSD_FS_WARPS);
    CK(cudaMemcpy(h.data(), ctx->d_prof, h.size() * 8, cudaMemcpyDeviceToHost));
    const double w = h[5] ? (double)h[5] : 1.0;
    fprintf(stderr, "[fs prof] warps %llu  per warp: total %.0f cyc, phase1 %.0f, phase2 %.0f, TMA wait %.0f, idle loops %.1f (input done %.1f, ring full %.1f, other %.1f; mean lag %.2f frames), polls %.1f\n",
            h[5], h[2] / w, h[0] / w, h[1] / w, h[6] / w, h[3] / w, h[7] / w, h[8] / w, h[9] / w, h[3] ? (double)h[10] / (double)h[3] : 0.0, h[4] / w);
    fprintf(stderr, "[fs prof] per warp: busy iterations %.0f cyc, idle iterations %.0f cyc; section TMA issue %.0f, sections prefetch+poll issue %.0f\n", h[11] / w, h[12] / w, h[13] / w, h[14] / w);
    double skew = 0, own = 0, peaks = 0, detect = 0, p2span = 0, period = 0;
    int cnt = 0;
    for(int f = 16; f + 16 < nf; f++)
    {
      const unsigned long long *q = &h[FS_PROF_HDR + (size_t)f * FS_PROF_PER_FRAME];
      skew += (double)(q[5] - q[0]);
      own += (double)q[1] - (double)q[5];
      peaks += (double)(q[2] - q[1]);
      detect += (double)q[3] - (double)q[2];
      p2span += (double)(q[4] - q[3]);
      period += (double)(q[5 + FS_PROF_PER_FRAME] - q[5]);
      cnt++;
    }
    if(n_frames >= 64)
    {
      // per CTA: sums over its warps
      double best_idle = 1e30, worst_idle = -1;
      int bi = -1, wi = -1;
      std::vector<double> ci(ctx->fs_grid, 0.0);
      for(int c = 0; c < ctx->fs_grid; c++)
      {
        for(int q = 0; q < SSD_FS_WARPS; q++)
          ci[c] += (double)h[woff + ((size_t)c * SSD_FS_WARPS + q) * 8 + 3];
        if(ci[c] < best_idle)
          best_idle = ci[c], bi = c;
        if(ci[c] > worst_idle)
          worst_idle = ci[c], wi = c;
      }
      for(int c : { bi, wi })
      {
        double s8[8] = { 0 };
        for(int q = 0; q < SSD_FS_WARPS; q++)
          for(int i = 0; i < 8; i++)
            s8[i] += (double)h[woff + ((size_t)c * SSD_FS_WARPS + q) * 8 + i] / SSD_FS_WARPS;
        fprintf(stderr, "[fs prof] CTA %d (%s idle): per warp p1 %.0f p2 %.0f tma %.0f idle loops %.0f (ring %.0f) total %.0f leave %.0f peaks %.0f\n", c,
                c == bi ? "least" : "most", s8[0], s8[1], s8[2], s8[3], s8[5], s8[4], s8[6], s8[7]);
      }
      {
        double mn = 1e30, mx = 0, sm = 0;
        const int nw = ctx->fs_grid * SSD_FS_WARPS;
        for(int q = 0; q < nw; q++)
        {
          const double v = (double)h[woff + (size_t)q * 8 + 0] + (double)h[woff + (size_t)q * 8 + 1];
          mn = std::min(mn, v), mx = std::max(mx, v), sm += v;
        }
        fprintf(stderr, "[fs prof] phase1+phase2 cycles per warp: min %.0f mean %.0f max %.0f\n", mn, sm / nw, mx);
      }
      int n_low = 0;
      for(int c = 0; c < ctx->fs_grid; c++)
        n_low += ci[c] < 0.25 * worst_idle;
      fprintf(stderr, "[fs prof] CTAs with less than a quarter of the worst CTA's idle loops: %d of %d\n", n_low, ctx->fs_grid);
    }
    if(cnt)
      fprintf(stderr, "[fs prof] per frame (ns): first -> last CTA delivered %.0f, -> owner saw it complete %.0f, -> LUT published %.0f, -> first phase-2 step %.0f, phase-2 span %.0f, period %.0f\n",
              skew / cnt, own / cnt, peaks / cnt, detect / cnt, p2span / cnt, period / cnt);
  }
  float ms = 0;
  CK(cudaEventElapsedTime(&ms, ctx->ev_start, ctx->ev_stop));
  ctx->timing.total_ms = ms;
  ctx->timing.h2d_ms = 0;
  if(host_input)
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
    for(int c = 0; c < n_chunks; c++)
      for(int i = 0; i < SSD_GPU_N_STAGES; i++)
      {
        float t = 0;
        const cudaEvent_t *ev = &ctx->stage_ev[(size_t)c * (SSD_GPU_N_STAGES + 1)];
        CK(cudaEventElapsedTime(&t, ev[i], ev[i + 1]));
        ctx->stage_ms[i] += t;
        ctx->stage_launches[i]++;
      }
    ctx->timing.label_ms = ctx->stage_ms[0];
  }
  return SSD_OK;
}

// A failure inside the chain (launch error, bad user pointer, out of memory while growing a staging buffer) may leave streams
// unsynchronised and BEV bitmaps half written: the bitmaps are "self-cleaning" only along a complete chain. Bring the context
// back to a clean state so that the next call starts from zeroed bitmaps and no stale results can be read.
static int process_common(ssd_gpu_ctx *ctx, const float *xyz, const uint16_t *z16, const ssd_gpu_intrinsics *intr, bool host_input, int n_frames,
                          int flags, const int32_t *cam_of_frame = nullptr)
{
  // refused before anything is launched: the results of the previous call stay readable
  if(ctx && !cam_of_frame && !ssd_lens_is_pinhole(&ctx->lens) && (ctx->records || ctx->wordrec || ctx->resident) && (!xyz || ctx->ov.enabled))
    return fail(ctx, SSD_E_STATE, "lens distortion runs on the default (classic) chain only; this context was created with "
                                  "SSD_GPU_PATH=records|wordrec|resident");
  const int rc = process_impl(ctx, xyz, z16, intr, host_input, n_frames, flags, cam_of_frame);
  if(rc != SSD_OK && rc != SSD_E_INVALID_ARG && rc != SSD_E_RANGE && ctx)
  {
    const std::string keep = ctx->err;
    cudaDeviceSynchronize();
    cudaGetLastError();
    if(ctx->d_bev)
      cudaMemset(ctx->d_bev, 0, (size_t)ctx->n_streams * ctx->chunk_frames * SSD_GPU_MAX_PLATEAUS * ctx->bm_words * 4);
    ctx->fs_pending = false;
    ctx->n_frames_last = 0;
    ctx->err = keep;
  }
  return rc;
}

int ssd_gpu_process_host(ssd_gpu_ctx *ctx, const float *xyz_host, int n_frames)
{
  return process_common(ctx, xyz_host, nullptr, nullptr, true, n_frames, 0);
}

int ssd_gpu_process_device(ssd_gpu_ctx *ctx, const float *xyz_dev, int n_frames)
{
  return process_common(ctx, xyz_dev, nullptr, nullptr, false, n_frames, 0);
}

int ssd_gpu_process_device_ex(ssd_gpu_ctx *ctx, const float *xyz_dev, int n_frames, int flags)
{
  return process_common(ctx, xyz_dev, nullptr, nullptr, false, n_frames, flags);
}

int ssd_gpu_process_depth_host(ssd_gpu_ctx *ctx, const uint16_t *z16_host, const ssd_gpu_intrinsics *intr, int n_frames)
{
  if(!z16_host || !intr)
    return fail(ctx, SSD_E_INVALID_ARG, "process_depth: bad argument");
  return process_common(ctx, nullptr, z16_host, intr, true, n_frames, 0);
}

int ssd_gpu_process_depth_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const ssd_gpu_intrinsics *intr, int n_frames)
{
  if(!z16_dev || !intr)
    return fail(ctx, SSD_E_INVALID_ARG, "process_depth: bad argument");
  return process_common(ctx, nullptr, z16_dev, intr, false, n_frames, 0);
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
    if(derive_params(ctx->cfg, cams[c].xf, dp[c]))
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
  CK(cudaMalloc(&ctx->d_cam_xn, sizeof(float) * (size_t)n_cameras * p.W));
  CK(cudaMalloc(&ctx->d_cam_yn, sizeof(float) * (size_t)n_cameras * p.H));
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
    const int n = std::max(p.W, p.H);
    k_deproject_tables_cams<<<dim3((n + 255) / 256, std::min(n_cameras, 65535)), 256, 0, st>>>(p.W, p.H, d_in, n_cameras, ctx->d_cam_xn, ctx->d_cam_yn);
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

// Everything a camera call can be refused for, before anything is launched (the previous results stay readable).
static int check_cameras(ssd_gpu_ctx *ctx, const void *input, const int32_t *cam_of_frame, int n_frames, bool depth)
{
  if(!ctx || !input || !cam_of_frame || n_frames <= 0)
    return fail(ctx, SSD_E_INVALID_ARG, "camera call: bad argument");
  if(ctx->records || ctx->wordrec || ctx->resident)
    return fail(ctx, SSD_E_STATE, "camera call: camera tables run on the default (classic) chain only; this context was created with "
                                  "SSD_GPU_PATH=records|wordrec|resident");
  if(depth && ctx->depth_unfused)
    return fail(ctx, SSD_E_STATE, "depth camera call: not available with SSD_GPU_DEPTH_UNFUSED=1 (the fused depth path only)");
  if(ctx->n_cameras <= 0)
    return fail(ctx, SSD_E_STATE, "camera call: no camera table (ssd_gpu_set_cameras)");
  if(n_frames > ctx->max_frames)
    return fail(ctx, SSD_E_RANGE, "process: n_frames exceeds max_frames of the context");
  if(depth && ctx->dp.W % 4 != 0)
    return fail(ctx, SSD_E_INVALID_ARG, "depth input: the frame width must be a multiple of 4");
  for(int f = 0; f < n_frames; f++)
  {
    const int32_t c = cam_of_frame[f];
    if(c < 0 || c >= ctx->n_cameras)
      return fail(ctx, SSD_E_RANGE, "camera call: frame " + std::to_string(f) + " names camera " + std::to_string(c) + ", outside [0, " +
                                      std::to_string(ctx->n_cameras) + ")");
    if(depth && !ctx->cam_depth_ok[c])
      return fail(ctx, SSD_E_INVALID_ARG, "depth camera call: camera " + std::to_string(c) + " has no depth intrinsics (fx, fy must be non-zero and "
                                                                                            "depth_unit positive)");
  }
  return SSD_OK;
}

int ssd_gpu_process_cameras_host(ssd_gpu_ctx *ctx, const float *xyz_host, const int32_t *camera_of_frame, int n_frames)
{
  const int rc = check_cameras(ctx, xyz_host, camera_of_frame, n_frames, false);
  return rc ? rc : process_common(ctx, xyz_host, nullptr, nullptr, true, n_frames, 0, camera_of_frame);
}

int ssd_gpu_process_cameras_device(ssd_gpu_ctx *ctx, const float *xyz_dev, const int32_t *camera_of_frame, int n_frames)
{
  const int rc = check_cameras(ctx, xyz_dev, camera_of_frame, n_frames, false);
  return rc ? rc : process_common(ctx, xyz_dev, nullptr, nullptr, false, n_frames, 0, camera_of_frame);
}

int ssd_gpu_process_cameras_device_ex(ssd_gpu_ctx *ctx, const float *xyz_dev, const int32_t *camera_of_frame, int n_frames, int flags)
{
  const int rc = check_cameras(ctx, xyz_dev, camera_of_frame, n_frames, false);
  return rc ? rc : process_common(ctx, xyz_dev, nullptr, nullptr, false, n_frames, flags, camera_of_frame);
}

int ssd_gpu_process_depth_cameras_host(ssd_gpu_ctx *ctx, const uint16_t *z16_host, const int32_t *camera_of_frame, int n_frames)
{
  const int rc = check_cameras(ctx, z16_host, camera_of_frame, n_frames, true);
  return rc ? rc : process_common(ctx, nullptr, z16_host, nullptr, true, n_frames, 0, camera_of_frame);
}

int ssd_gpu_process_depth_cameras_device(ssd_gpu_ctx *ctx, const uint16_t *z16_dev, const int32_t *camera_of_frame, int n_frames)
{
  const int rc = check_cameras(ctx, z16_dev, camera_of_frame, n_frames, true);
  return rc ? rc : process_common(ctx, nullptr, z16_dev, nullptr, false, n_frames, 0, camera_of_frame);
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
    k_deproject<<<dim3((p.N / 4 + 255) / 256, nf), 256, 0, ctx->stream[0]>>>(p.W, p.N, intr->depth_unit, ctx->d_xn, ctx->d_yn, z16_dev + (size_t)f0 * p.N,
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
  const FrameOut &o = ctx->h_out[frame];
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
  const int ns = ctx->h_out[frame].info.n_steps;
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
  std::vector<PlateauDev> pl(SSD_GPU_MAX_PLATEAUS);
  std::vector<RiserDev> rs(SSD_GPU_MAX_PLATEAUS);
  CK(cudaMemcpy(pl.data(), ctx->d_frames[frame].plat, sizeof(PlateauDev) * SSD_GPU_MAX_PLATEAUS, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(rs.data(), ctx->d_frames[frame].ris, sizeof(RiserDev) * SSD_GPU_MAX_PLATEAUS, cudaMemcpyDeviceToHost));
  const int K = ctx->h_out[frame].info.n_plateaus;
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

int ssd_gpu_get_frame_info(ssd_gpu_ctx *ctx, int frame, ssd_gpu_frame_info *out)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  if(!out)
    return SSD_E_INVALID_ARG;
  *out = ctx->h_out[frame].info;
  return SSD_OK;
}

int ssd_gpu_get_plateaus(ssd_gpu_ctx *ctx, int frame, ssd_gpu_plateau *out, int cap, int *n)
{
  const int rc = check_frame(ctx, frame);
  if(rc)
    return rc;
  CK(cudaSetDevice(ctx->device));
  std::vector<PlateauDev> tmp(SSD_GPU_MAX_PLATEAUS);
  CK(cudaMemcpy(tmp.data(), ctx->d_frames[frame].plat, sizeof(PlateauDev) * SSD_GPU_MAX_PLATEAUS, cudaMemcpyDeviceToHost));
  const int K = ctx->h_out[frame].info.n_plateaus;
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
  CK(cudaMemcpy(tmp, ctx->d_frames[frame].hist, sizeof(tmp), cudaMemcpyDeviceToHost));
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
  for(int f = 0; f < ctx->n_frames_last; f++)
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
  CK(cudaSetDevice(ctx->device));
  if(!ctx->d_img)
    CK(cudaMalloc(&ctx->d_img, (size_t)p.N));
  CK(cudaMemcpyAsync(ctx->d_img, image_host, (size_t)p.N, cudaMemcpyHostToDevice, ctx->stream[0]));
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
