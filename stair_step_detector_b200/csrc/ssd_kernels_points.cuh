// ssd_kernels_points.cuh -- the per-point (HBM-bound) kernels of the chain:
//   k_transform_bin : z>0 filter, camera->world transform, range filter, height bin, height histogram
//   k_peaks         : histogram peaks -> plateau bands -> bin->label LUT, ground selection
//   k_label_bev     : per-point segment label + top-down (BEV) occupancy bitmaps of the outlined plateaus
//   k_quad_reduce   : point-in-quadrilateral filter, per-step z sum / count, ground BEV bitmap
// Algorithmic traffic: 12 B read + 1 B written per point (SURVEY.md 8(d)); the bin codes are written once by
// k_transform_bin and rewritten in place as labels by k_label_bev.
#pragma once
#include "ssd_device.cuh"

#define SSD_PT_THREADS 256
#define SSD_PT_WARPS (SSD_PT_THREADS / 32)

// ---- TMA bulk staging (cp.async.bulk + mbarrier): one elected thread streams a whole tile of vertices into
// shared memory; the loads in flight no longer cost registers or depend on occupancy ----
__device__ __forceinline__ void mbar_init(unsigned bar, unsigned count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init()
{
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, unsigned bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
// wait for phase `parity` of the barrier; a copy that never lands traps instead of hanging the GPU
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity)
{
  for(int spin = 0; spin < (1 << 24); spin++)
  {
    unsigned ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
    if(ok)
      return;
  }
  __trap();
}

// ---------------------------------------------------------------------------------------------
// Where the point kernels read their vertices from. Two sources, chosen at launch (template parameter):
//   SrcVertices : the packed rs2::vertex array (12 B/point) -- what rs2::pointcloud::calculate returns
//                 (pointcloud.cpp:138-147);
//   SrcDepth    : the z16 depth frame itself (2 B/point) -- what Pointcloud::process receives (pointcloud.cpp:608).
//                 The deprojection the reference delegates to rs2::pointcloud::calculate (pin-hole model of
//                 rs2_deproject_pixel_to_point / camera.h:99-116) is evaluated in registers, with the single-rounded f32
//                 operations of ssd_deproject_pixel (scene_model.h) / k_deproject: the vertices never exist in memory
//                 and all three passes move 2 bytes per point instead of 12.
// A kernel derives a frame cursor once (src_frame), then loads 4-point words (word_load: where a kernel issues it ahead of use, the
// registers of a word in flight are the raw loads) and unpacks them where they are consumed (word_unpack).
// ---------------------------------------------------------------------------------------------
struct SrcVertices
{
  const float *xyz; // n_frames x N x {x, y, z}
};
struct SrcDepth
{
  const uint16_t *z16;         // n_frames x N
  const float *xn, *yn;        // (u - ppx) / fx per column, (v - ppy) / fy per row (k_deproject_tables)
  float unit;                  // metres per depth unit
  unsigned long long wmagic;   // ceil(2^40 / W): row of pixel i = (i * wmagic) >> 40, exact for i * W < 2^40
};
// SrcLens: z16 frames of a camera with a distorted lens (ssd_gpu_set_distortion). Its ray (x, y) depends on u and v, so it is
// read per pixel from the lens's ray table (k_lens_rays): 2 B of depth + 8 B of ray per point, the table shared by every frame
// of the lens and L2-resident at the usual frame sizes. Then X = z * x, Y = z * y as for SrcDepth.
struct SrcLens
{
  const uint16_t *z16;              // n_frames x N
  const float2 *ray;                // N rays of the lens (plain calls)
  const float2 *const *cam_ray;     // camera calls: the ray table of each camera (a pin-hole camera's holds (xn[u], yn[v]))
  float unit;
};
struct FrameV
{
  const float4 *f4;
};
struct FrameL
{
  const uint2 *d2;    // four z16 pixels per element
  const float4 *r4;   // two rays per element
  float unit;
};
struct WordL
{
  uint2 d;
  float4 r01, r23;
};
struct FrameD
{
  const uint2 *d2; // four z16 pixels per element
  const float *xn, *yn;
  float unit;
  unsigned long long wmagic;
  unsigned W;
};
struct WordV
{
  float4 a, b, c;
};
struct WordD
{
  uint2 d;
  float4 x4;
  float y;
};
template<class SRC>
struct SrcTraits;
template<>
struct SrcTraits<SrcVertices>
{
  typedef FrameV Frame;
  typedef WordV Word;
};
template<>
struct SrcTraits<SrcDepth>
{
  typedef FrameD Frame;
  typedef WordD Word;
};
template<>
struct SrcTraits<SrcLens>
{
  typedef FrameL Frame;
  typedef WordL Word;
};
__device__ __forceinline__ FrameL src_frame(const SrcLens &s, const DevParams &, size_t fbase)
{
  FrameL f;
  f.d2 = reinterpret_cast<const uint2 *>(s.z16 + fbase);
  f.r4 = reinterpret_cast<const float4 *>(s.ray);
  f.unit = s.unit;
  return f;
}
__device__ __forceinline__ SrcLens frame_src(const SrcLens &s, const CamTable &c, const DevParams &, int frame)
{
  const int cam = frame_camera(c, frame);
  SrcLens d = s;
  d.ray = s.cam_ray[cam];
  d.unit = __ldg(c.unit + cam);
  return d;
}
__device__ __forceinline__ void word_zero(WordL &r)
{
  r.d = make_uint2(0u, 0u);
  r.r01 = r.r23 = make_float4(0.f, 0.f, 0.f, 0.f);
}
__device__ __forceinline__ void word_load(const FrameL &f, unsigned w, WordL &r)
{
  r.d = __ldg(f.d2 + w);
  r.r01 = __ldg(f.r4 + (size_t)w * 2);
  r.r23 = __ldg(f.r4 + (size_t)w * 2 + 1);
}
__device__ __forceinline__ void word_unpack(const FrameL &f, const WordL &r, float vx[4], float vy[4], float vz[4])
{
  vz[0] = __fmul_rn((float)(r.d.x & 0xffffu), f.unit);
  vz[1] = __fmul_rn((float)(r.d.x >> 16), f.unit);
  vz[2] = __fmul_rn((float)(r.d.y & 0xffffu), f.unit);
  vz[3] = __fmul_rn((float)(r.d.y >> 16), f.unit);
  const float rx[4] = { r.r01.x, r.r01.z, r.r23.x, r.r23.z }, ry[4] = { r.r01.y, r.r01.w, r.r23.y, r.r23.w };
#pragma unroll
  for(int j = 0; j < 4; j++)
  {
    vx[j] = __fmul_rn(vz[j], rx[j]);
    vy[j] = __fmul_rn(vz[j], ry[j]);
  }
}
__device__ __forceinline__ void word_prefetch_l2(const FrameL &f, unsigned w)
{
  asm volatile("prefetch.global.L2 [%0];" ::"l"(f.d2 + w));
  asm volatile("prefetch.global.L2 [%0];" ::"l"(f.r4 + (size_t)w * 2)); // the word's 32 bytes of rays: one sector
}
__device__ __forceinline__ void point_load(const FrameL &f, unsigned pt, float &x, float &y, float &z)
{
  const unsigned d = __ldg(reinterpret_cast<const unsigned short *>(f.d2) + pt);
  const float2 r = __ldg(reinterpret_cast<const float2 *>(f.r4) + pt);
  z = __fmul_rn((float)d, f.unit);
  x = __fmul_rn(z, r.x);
  y = __fmul_rn(z, r.y);
}
__device__ __forceinline__ FrameV src_frame(const SrcVertices &s, const DevParams &p, size_t fbase)
{
  FrameV f;
  f.f4 = reinterpret_cast<const float4 *>(s.xyz + fbase * 3);
  return f;
}
__device__ __forceinline__ FrameD src_frame(const SrcDepth &s, const DevParams &p, size_t fbase)
{
  FrameD f;
  f.d2 = reinterpret_cast<const uint2 *>(s.z16 + fbase);
  f.xn = s.xn;
  f.yn = s.yn;
  f.unit = s.unit;
  f.wmagic = s.wmagic;
  f.W = (unsigned)p.W;
  return f;
}
// The source of one frame: in camera mode a depth frame is deprojected with its own camera's tables and depth unit.
template<class SRC>
__device__ __forceinline__ const SRC &frame_src(const SRC &s, const NoCam &, const DevParams &, int)
{
  return s;
}
__device__ __forceinline__ SrcVertices frame_src(const SrcVertices &s, const CamTable &, const DevParams &, int)
{
  return s;
}
__device__ __forceinline__ SrcDepth frame_src(const SrcDepth &s, const CamTable &c, const DevParams &p, int frame)
{
  const int cam = frame_camera(c, frame);
  SrcDepth d = s;
  d.xn = c.xn + (size_t)cam * p.W;
  d.yn = c.yn + (size_t)cam * p.H;
  d.unit = __ldg(c.unit + cam);
  return d;
}
__device__ __forceinline__ void word_zero(WordV &r)
{
  r.a = r.b = r.c = make_float4(0.f, 0.f, 0.f, 0.f);
}
__device__ __forceinline__ void word_zero(WordD &r)
{
  r.d = make_uint2(0u, 0u);
  r.x4 = make_float4(0.f, 0.f, 0.f, 0.f);
  r.y = 0.f;
}
// w: index of the 4-point word within the frame
__device__ __forceinline__ void word_load(const FrameV &f, unsigned w, WordV &r)
{
  const float4 *src = f.f4 + (size_t)w * 3;
  r.a = __ldg(src);
  r.b = __ldg(src + 1);
  r.c = __ldg(src + 2);
}
__device__ __forceinline__ void word_load(const FrameD &f, unsigned w, WordD &r)
{
  r.d = __ldg(f.d2 + w);
  const unsigned i0 = w * 4u;
  const unsigned v = (unsigned)(((unsigned long long)i0 * f.wmagic) >> 40), u = i0 - v * f.W; // W % 4 == 0: one row per word
  r.x4 = __ldg(reinterpret_cast<const float4 *>(f.xn + u));
  r.y = __ldg(f.yn + v);
}
__device__ __forceinline__ void word_unpack(const FrameV &, const WordV &r, float vx[4], float vy[4], float vz[4])
{
  vx[0] = r.a.x, vy[0] = r.a.y, vz[0] = r.a.z;
  vx[1] = r.a.w, vy[1] = r.b.x, vz[1] = r.b.y;
  vx[2] = r.b.z, vy[2] = r.b.w, vz[2] = r.c.x;
  vx[3] = r.c.y, vy[3] = r.c.z, vz[3] = r.c.w;
}
__device__ __forceinline__ void word_unpack(const FrameD &f, const WordD &r, float vx[4], float vy[4], float vz[4])
{
  vz[0] = __fmul_rn((float)(r.d.x & 0xffffu), f.unit);
  vz[1] = __fmul_rn((float)(r.d.x >> 16), f.unit);
  vz[2] = __fmul_rn((float)(r.d.y & 0xffffu), f.unit);
  vz[3] = __fmul_rn((float)(r.d.y >> 16), f.unit);
  const float xn[4] = { r.x4.x, r.x4.y, r.x4.z, r.x4.w };
#pragma unroll
  for(int j = 0; j < 4; j++)
  {
    vx[j] = __fmul_rn(vz[j], xn[j]);
    vy[j] = __fmul_rn(vz[j], r.y);
  }
}
// request a word into L2 (issued as soon as it is known to matter, a phase ahead of its use)
__device__ __forceinline__ void word_prefetch_l2(const FrameV &f, unsigned w)
{
  const float4 *src = f.f4 + (size_t)w * 3;
  asm volatile("prefetch.global.L2 [%0];" ::"l"(src));     // both 32-byte sectors the 48 bytes can touch
  asm volatile("prefetch.global.L2 [%0];" ::"l"(src + 2));
}
__device__ __forceinline__ void word_prefetch_l2(const FrameD &f, unsigned w)
{
  asm volatile("prefetch.global.L2 [%0];" ::"l"(f.d2 + w));
}
// one point by its index within the frame (the compacted exact passes)
__device__ __forceinline__ void point_load(const FrameV &f, unsigned pt, float &x, float &y, float &z)
{
  const float *v = reinterpret_cast<const float *>(f.f4) + (size_t)pt * 3;
  x = __ldg(v);
  y = __ldg(v + 1);
  z = __ldg(v + 2);
}
__device__ __forceinline__ void point_load(const FrameD &f, unsigned pt, float &x, float &y, float &z)
{
  const unsigned d = __ldg(reinterpret_cast<const unsigned short *>(f.d2) + pt);
  const unsigned v = (unsigned)(((unsigned long long)pt * f.wmagic) >> 40), u = pt - v * f.W;
  z = __fmul_rn((float)d, f.unit);
  x = __fmul_rn(z, __ldg(f.xn + u));
  y = __fmul_rn(z, __ldg(f.yn + v));
}

// ---------------------------------------------------------------------------------------------
// Peaks of one frame, one warp: HeightsHistogram::findPeaks / filterPeaks (pointcloud.cpp:214-256), the plateau bands of
// extractPlateauPoints (:300-335) as a bin -> label LUT, ground / first-outlined bookkeeping (:402-418). Evaluated bin-parallel:
//   rise(i) = hist[i] < hist[i+1], fall(i) = hist[i] > hist[i+1]   (i < n_bins - 1)
//   ascending before i  <=>  the nearest j < i with rise(j) or fall(j) is a rise      (equal neighbours keep the flag)
//   peak(i) = fall(i) && ascending && hist[i] >= min_peak_points && (2 hist[i] - hist[i-1] - hist[i+1]) * 2 > hist[i]
//   band(i) = [i-1, i] if hist[i-1] > hist[i+1] else [i, i+1]; a bin claimed by two bands goes to the lower peak
//   (peaks are at least two bins apart, so only the bands of the peaks at b-1, b, b+1 can hold bin b).
// ---------------------------------------------------------------------------------------------
struct __align__(16) PeaksScratch // per-warp scratch of peaks_warp (16-byte vector stores into hist)
{
  unsigned hist[SSD_BINS_PAD + 8]; // bin b at [4 + b]; zeros either side
  unsigned short lut[SSD_BINS_PAD];
  int height[SSD_GPU_MAX_PLATEAUS], hmin[SSD_GPU_MAX_PLATEAUS], hmax[SSD_GPU_MAX_PLATEAUS];
  unsigned np[SSD_GPU_MAX_PLATEAUS];
};

#define SSD_LUT_OUTLINED 0x100u  // lut16 flags: the label gets a BEV image
#define SSD_LUT_GROUND 0x200u    //              the label is the ground plateau
#define SSD_LUT_VALID 0x8000u    //              entry written (a zero entry means "frame not ready")

// bit (32 r + lane + D) of a 256-bit string held as eight warp-uniform words (zeros outside), D in {-2, -1, 0, +1}
template<int D>
__device__ __forceinline__ unsigned peaks_bit_at(const unsigned (&w)[8], int r, int lane)
{
  const unsigned cur = w[r];
  if(D == 0)
    return (cur >> lane) & 1u;
  if(D < 0)
  {
    const unsigned prev = r > 0 ? w[r - 1] : 0u;
    return (__funnelshift_l(prev, cur, -D) >> lane) & 1u; // bit i of the result = bit (i + D) of the string
  }
  const unsigned next = r < 7 ? w[r + 1] : 0u;
  return (__funnelshift_r(cur, next, D) >> lane) & 1u;
}

// K: scratch in shared memory, private to the calling warp for the duration of the call. h0, h1: bins 8 lane .. 8 lane + 7.
// lut_flags: OR-ed into every lut16 entry (SSD_LUT_VALID for the resident-frame path's polling).
__device__ inline void peaks_warp(const DevParams &p, FrameDev &F, PeaksScratch &K, const uint4 h0, const uint4 h1, int lane)
{
  {
    // the frame's complete histogram (bins 8 lane .. 8 lane + 7), as the owner's poll read it
    uint4 *dst = reinterpret_cast<uint4 *>(K.hist + 4 + lane * 8);
    dst[0] = h0;
    dst[1] = h1;
    if(lane < 4)
    {
      K.hist[lane] = 0;
      K.hist[4 + SSD_BINS_PAD + lane] = 0;
    }
  }
  __syncwarp();
  const unsigned *H = K.hist + 4;
  const int last = p.n_bins - 1;
  const unsigned lt = (1u << lane) - 1u;
  unsigned R[8], Fm[8], Pw[8], BL[8], hc[8], hm[8], hp[8];
#pragma unroll
  for(int r = 0; r < 8; r++)
  {
    const int b = 32 * r + lane;
    hc[r] = H[b];
    hm[r] = H[b - 1];
    hp[r] = H[b + 1];
    const bool v = b < last;
    R[r] = __ballot_sync(0xffffffffu, v && hc[r] < hp[r]);
    Fm[r] = __ballot_sync(0xffffffffu, v && hc[r] > hp[r]);
    BL[r] = __ballot_sync(0xffffffffu, hm[r] > hp[r]);
  }
  {
    bool carry = false; // ascending at the start of word r
#pragma unroll
    for(int r = 0; r < 8; r++)
    {
      const unsigned c = hc[r];
      const unsigned E = R[r] | Fm[r];
      const unsigned m = E & lt;
      const bool asc = m ? ((R[r] >> (31 - __clz(m))) & 1u) != 0u : carry;
      const bool fall = (Fm[r] >> lane) & 1u;
      const bool peak = fall && asc && !(c < p.min_peak_points) && (unsigned)((c * 2u - hm[r] - hp[r]) * 2u) > c;
      Pw[r] = __ballot_sync(0xffffffffu, peak);
      if(E)
        carry = ((R[r] >> (31 - __clz(E))) & 1u) != 0u;
    }
  }
  int n_all = 0;
#pragma unroll
  for(int r = 0; r < 8; r++)
    n_all += __popc(Pw[r]);
  const int Kn = min(n_all, SSD_GPU_MAX_PLATEAUS);
  unsigned status = n_all > SSD_GPU_MAX_PLATEAUS ? SSD_STATUS_TOO_MANY_PLATEAUS : 0u;
  // uint16 wrap of heightMin - 1 (pointcloud.cpp:324): a peak at bin 1 with band [0, 1] -- necessarily the first peak --
  // sends every point to the remainder; that plateau and all later ones stay empty
  const bool wrapped = ((Pw[0] >> 1) & 1u) && ((BL[0] >> 1) & 1u);
  if(wrapped)
    status |= SSD_STATUS_HMIN_WRAP;
  {
    int base = 0;
#pragma unroll
    for(int r = 0; r < 8; r++)
    {
      const int b = 32 * r + lane;
      const int cntlt = base + __popc(Pw[r] & lt); // peaks at bins < b
      const bool pk = (Pw[r] >> lane) & 1u;
      unsigned l = SSD_LABEL_REMAINDER;
      if(!wrapped)
      {
        int k = -1;
        if(peaks_bit_at<-1>(Pw, r, lane) && !peaks_bit_at<-1>(BL, r, lane))
          k = cntlt - 1;
        else if(pk)
          k = cntlt;
        else if(peaks_bit_at<1>(Pw, r, lane) && peaks_bit_at<1>(BL, r, lane))
          k = cntlt;
        if(k >= 0 && k < SSD_GPU_MAX_PLATEAUS)
          l = (unsigned)k;
      }
      if(b == (int)SSD_CODE_OUT_OF_RANGE)
        l = SSD_LABEL_OUT_OF_RANGE;
      if(b == (int)SSD_CODE_INVALID)
        l = SSD_LABEL_INVALID;
      K.lut[b] = (unsigned short)l;
      if(pk && cntlt < SSD_GPU_MAX_PLATEAUS)
      {
        const bool lo = (BL[r] >> lane) & 1u;
        unsigned np = hc[r];
        if(lo)
          np += (peaks_bit_at<-2>(Pw, r, lane) && !peaks_bit_at<-2>(BL, r, lane)) ? 0u : hm[r];
        else
          np += hp[r];
        K.height[cntlt] = b;
        K.hmin[cntlt] = lo ? b - 1 : b;
        K.hmax[cntlt] = lo ? b : b + 1;
        K.np[cntlt] = wrapped ? 0u : np;
      }
      base += __popc(Pw[r]);
    }
  }
  __syncwarp();
  // ground = the largest of the leading plateaus below minHeight (first maximum), outlines from the first plateau at or above it
  const bool mine = lane < Kn;
  const int height = mine ? K.height[lane] : 0;
  const unsigned np = mine ? K.np[lane] : 0u;
  const unsigned hi = __ballot_sync(0xffffffffu, mine && height >= p.min_height);
  const int fo = hi ? __ffs(hi) - 1 : Kn;
  const unsigned gnp = (mine && lane < fo) ? np : 0u;
  const unsigned gmax = __reduce_max_sync(0xffffffffu, gnp);
  const unsigned gb = __ballot_sync(0xffffffffu, lane < fo && mine && gnp == gmax);
  const int ground = gmax > 0u ? __ffs(gb) - 1 : -1;
  if(lane == 0)
  {
    F.n_nonzero = (unsigned)p.N - H[SSD_CODE_INVALID];
    F.n_in_range = (unsigned)p.N - H[SSD_CODE_INVALID] - H[SSD_CODE_OUT_OF_RANGE];
    F.n_plateaus = Kn;
    F.ground_index = ground;
    F.first_outlined = fo;
    F.first_valid = -1;
    F.n_steps = 0;
    F.status = status;
  }
  {
    RiserDev &R = F.ris[lane]; // SSD_GPU_MAX_PLATEAUS == 32: one per lane
    R.cnt = 0;
    R.xmin = R.ymin = 0x7fffffff;
    R.xmax = R.ymax = -1;
    R.sx = R.sy = 0;
  }
  if(mine)
  {
    PlateauDev &P = F.plat[lane];
    P.height = height;
    P.hmin = K.hmin[lane];
    P.hmax = K.hmax[lane];
    P.n_points = np;
    P.valid = 0;
    P.outlined = lane >= fo;
    P.n_in_quad = 0;
    P.quad_status = -1;
    P.mean_z = 0;
    P.sum_fix = 0;
    P.sum_d = 0;
    P.sum_c = 0;
    P.n_sum = 0;
    P.row_min = 0x7fffffff;
    P.row_max = -1;
    P.front_valid = 0;
    for(int c4 = 0; c4 < 4; c4++)
      P.quad_px[c4][0] = P.quad_px[c4][1] = P.quad_world[c4][0] = P.quad_world[c4][1] = 0;
  }
  {
    unsigned w[4];
#pragma unroll
    for(int i = 0; i < 4; i++)
    {
      unsigned e2[2];
#pragma unroll
      for(int h = 0; h < 2; h++)
      {
        const unsigned l = K.lut[lane * 8 + i * 2 + h];
        unsigned e = l | SSD_LUT_VALID;
        if((int)l >= fo && (int)l < Kn)
          e |= SSD_LUT_OUTLINED;
        if((int)l == ground)
          e |= SSD_LUT_GROUND;
        e2[h] = e;
      }
      w[i] = e2[0] | (e2[1] << 16);
    }
    *(reinterpret_cast<uint4 *>(F.lut16) + lane) = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// ---------------------------------------------------------------------------------------------
// k_transform_bin: PointsExtraction::extract + HeightsHistogram::calcHist
// (pointcloud.cpp:122-178, 194-204). grid = (tiles_per_frame, frames), block = 256.
// Each thread handles 4 consecutive points per iteration: three 16 B loads, one 4 B store.
// The camera->world transform, range filter and height bin are decided in single precision with a rigorous
// error bound (point_code_filtered); the exact double-precision chain runs only for the few points whose
// f32 value lies within that bound of a threshold, so the result is bit-identical to the all-double chain.
// Histogram: one shared-memory increment per point into one histogram per block (the hardware aggregates the lanes
// of a warp that hit the same bin); one global atomic per non-empty bin per block.
// ---------------------------------------------------------------------------------------------
// One 4-point word of k_transform_bin: codes (filtered decision, exact fallback), the 4-byte code store, the block
// histogram update. Shared by the vertex and the depth-frame variant of the kernel.
__device__ __forceinline__ void tb_word(const DevParams &p, const float vx[4], const float vy[4], const float vz[4], unsigned *__restrict__ dst_word,
                                        unsigned *s_hist, unsigned &exact)
{
  // Two speeds. When every point of the warp's 128 is invalid or certainly outside the measuring range in x or y (the image
  // rows that look past the staircase: about four words in ten) only the packed x/y rows of the transform are evaluated:
  // max(|v_x|, |v_y|) - 1 > eps implies max_i |v_i| - 1 > eps, which is point_code_scaled's own "certainly out of range".
  float eps[4], sx[4], sy[4];
  bool skip = true;
#pragma unroll
  for(int j = 0; j < 4; j++)
  {
    const float m = max3abs_nan(vx[j], vy[j], vz[j]);
    eps[j] = fmaf(p.E1s, m, p.E0s);
    f2_unpack(f2_affine(p.sxy2, p.sbxy2, vx[j], vy[j], vz[j]), sx[j], sy[j]);
    const bool far = fmaxf(fabsf(sx[j]), fabsf(sy[j])) - 1.0f > eps[j];
    skip = skip && (far || !(vz[j] > 0.f));
  }
  unsigned c[4];
  if(__all_sync(__activemask(), skip)) // (the lanes of a frame's last, partial warp that have no word are not here)
  {
#pragma unroll
    for(int j = 0; j < 4; j++)
    {
      c[j] = vz[j] > 0.f ? SSD_CODE_OUT_OF_RANGE : SSD_CODE_INVALID;
      atomicAdd(s_hist + c[j], 1u);
    }
    *dst_word = c[0] | (c[1] << 8) | (c[2] << 16) | (c[3] << 24);
    return;
  }
  bool unc[4];
  const float MAGIC = 12582912.0f;
#pragma unroll
  for(int j = 0; j < 4; j++)
  {
    // the rest of point_code_scaled (ssd_device.cuh): z row, range test on all three rows, height bin with its certainty
    const float sz = fmaf(p.sa[8], vz[j], fmaf(p.sa[7], vy[j], fmaf(p.sa[6], vx[j], p.sb[2])));
    const float e1 = max3abs_nan(sx[j], sy[j], sz) - 1.0f;
    const float uf = fmaf(sz, p.Gf, p.Gm);
    const float s = uf + MAGIC;
    const float d = uf - (s - MAGIC);
    const float thr = fmaf(-p.Gup, eps[j], p.thr0);
    const bool out = e1 > eps[j];
    const bool in_bin = e1 < -eps[j] && fabsf(d) < thr;
    const bool valid = vz[j] > 0.f;
    unc[j] = valid && !(out || in_bin);
    const unsigned cc = out ? SSD_CODE_OUT_OF_RANGE : ((unsigned)__float_as_int(s) & 0xffu);
    c[j] = valid ? cc : SSD_CODE_INVALID;
  }
  if(unc[0] || unc[1] || unc[2] || unc[3])
  {
    // rare: one out-of-line exact evaluation per uncertain point
#pragma unroll
    for(int j = 0; j < 4; j++)
      if(unc[j])
      {
        c[j] = point_code_slow(p, vx[j], vy[j], vz[j]);
        exact++;
      }
  }
  const unsigned cw = c[0] | (c[1] << 8) | (c[2] << 16) | (c[3] << 24);
  *dst_word = cw;
  // Histogram: one shared-memory increment per point. The lanes of a warp mostly hit the same two or three bins
  // (image rows are iso-height); the hardware aggregates the lanes that address the same word (ATOMS.POPC.INC: one
  // update per distinct bin and instruction), which measured faster than any software aggregation tried here
  // (per-lane run-length merging: 43 instructions per word against 8; k_transform_bin 3.22 -> 2.93 ms per 2048 frames).
#pragma unroll
  for(int j = 0; j < 4; j++)
    atomicAdd(s_hist + c[j], 1u);
}

#define SSD_TB_STAGE_BYTES (SSD_PT_THREADS * 48) // one iteration of the block: 256 threads x 4 vertices x 12 B
// FUSE_PEAKS (small batches): the last block of a frame to deliver its histogram evaluates the peaks (k_peaks) itself.
__device__ __forceinline__ void tb_fused_peaks(const DevParams &p, FrameDev &F, PeaksScratch &K, unsigned &s_last, int tid)
{
  __threadfence();
  __syncthreads();
  if(tid == 0)
    s_last = atomicAdd(&F.tb_done, 1u) == gridDim.x - 1 ? 1u : 0u;
  __syncthreads();
  if(s_last && tid < 32)
  {
    __threadfence();
    const uint4 *src = reinterpret_cast<const uint4 *>(F.hist) + tid * 2;
    const uint4 h0 = __ldcg(src), h1 = __ldcg(src + 1);
    peaks_warp(p, F, K, h0, h1, tid);
  }
}

template<int ITERS, bool FUSE_PEAKS = false, class CAM = NoCam>
__global__ void __launch_bounds__(SSD_PT_THREADS) k_transform_bin(const __grid_constant__ DevParams p0, const float *__restrict__ xyz,
                                                                   unsigned char *__restrict__ codes, FrameDev *__restrict__ frames,
                                                                   const CAM cam = CAM())
{
  extern __shared__ __align__(128) unsigned char s_dyn[]; // ITERS stages of SSD_TB_STAGE_BYTES
  __shared__ __align__(8) unsigned long long s_bar[ITERS];
  __shared__ unsigned s_hist[SSD_BINS_PAD];
  __shared__ unsigned s_exact;
  const int tid = threadIdx.x;
  const int frame = blockIdx.y;
  const size_t fbase = (size_t)frame * p0.N; // (configuration fields: equal in every camera's parameters)
  const int nquads = p0.N >> 2;
  const int qb = blockIdx.x * (ITERS * SSD_PT_THREADS); // first quad (4 vertices) of the block
  const unsigned stage_sa = (unsigned)__cvta_generic_to_shared(s_dyn);
  const unsigned bar_sa = (unsigned)__cvta_generic_to_shared(s_bar);
  if(tid == 0)
  {
#pragma unroll
    for(int it = 0; it < ITERS; it++)
      mbar_init(bar_sa + it * 8, 1);
    mbar_fence_init();
    // the whole tile is requested at once: ITERS bulk copies of up to 12 KB, each signalling its own barrier
    const unsigned char *gsrc = reinterpret_cast<const unsigned char *>(xyz + fbase * 3) + (size_t)qb * 48;
#pragma unroll
    for(int it = 0; it < ITERS; it++)
    {
      const int nq = min(SSD_PT_THREADS, nquads - (qb + it * SSD_PT_THREADS));
      if(nq > 0)
      {
        mbar_expect_tx(bar_sa + it * 8, (unsigned)nq * 48u);
        bulk_g2s(stage_sa + it * SSD_TB_STAGE_BYTES, gsrc + (size_t)it * SSD_TB_STAGE_BYTES, (unsigned)nq * 48u, bar_sa + it * 8);
      }
    }
    s_exact = 0;
  }
  // camera mode: the frame's parameters are staged while the bulk copies are in flight
  const DevParams &p = frame_params(p0, cam, frame);
  s_hist[tid] = 0; // SSD_PT_THREADS == SSD_BINS_PAD
  __syncthreads();

  const int q0 = qb + tid;
  unsigned *dst = reinterpret_cast<unsigned *>(codes + fbase) + q0;
  unsigned exact = 0;

#pragma unroll
  for(int it = 0; it < ITERS; it++)
  {
    if(qb + it * SSD_PT_THREADS < nquads) // block-uniform: the stage was requested
      mbar_wait(bar_sa + it * 8, 0);
    if(q0 + it * SSD_PT_THREADS < nquads)
    {
      const float4 *s4 = reinterpret_cast<const float4 *>(s_dyn + it * SSD_TB_STAGE_BYTES) + tid * 3;
      const float4 v0 = s4[0], v1 = s4[1], v2 = s4[2];
      const float vx[4] = { v0.x, v0.w, v1.z, v2.y }, vy[4] = { v0.y, v1.x, v1.w, v2.z }, vz[4] = { v0.z, v1.y, v2.x, v2.w };
      tb_word(p, vx, vy, vz, dst + it * SSD_PT_THREADS, s_hist, exact);
    }
  }
  if(exact)
    atomicAdd(&s_exact, exact);
  __syncthreads();
  const unsigned sum = s_hist[tid];
  if(sum)
    atomicAdd(&frames[frame].hist[tid], sum);
  if(tid == 0 && s_exact)
    atomicAdd(&frames[frame].n_exact_bin, s_exact);
  if(FUSE_PEAKS)
  {
    __shared__ PeaksScratch K;
    __shared__ unsigned s_last;
    tb_fused_peaks(p, frames[frame], K, s_last, tid);
  }
}

// ---------------------------------------------------------------------------------------------
// k_transform_bin_depth: the same pass on a z16 depth frame (SrcDepth): 2 bytes per point come in, 1 goes out, the
// deprojected vertices live in registers only. No staging: the loads are 8 bytes per lane (256 B per warp, coalesced) and
// all ITERS words of a thread are requested before the first is consumed. Not HBM-bound (3 B/point): issue-bound.
// ---------------------------------------------------------------------------------------------
template<int ITERS, bool FUSE_PEAKS = false, class CAM = NoCam>
__global__ void __launch_bounds__(SSD_PT_THREADS) k_transform_bin_depth(const __grid_constant__ DevParams p0, const SrcDepth src0,
                                                                         unsigned char *__restrict__ codes, FrameDev *__restrict__ frames,
                                                                         const CAM cam = CAM())
{
  __shared__ unsigned s_hist[SSD_BINS_PAD];
  __shared__ unsigned s_exact;
  const int tid = threadIdx.x;
  const int frame = blockIdx.y;
  const DevParams &p = frame_params(p0, cam, frame);
  const auto &src = frame_src(src0, cam, p, frame);
  const size_t fbase = (size_t)frame * p.N;
  const int nquads = p.N >> 2;
  const int q0 = blockIdx.x * (ITERS * SSD_PT_THREADS) + tid;
  const FrameD F = src_frame(src, p, fbase);
  WordD w[ITERS];
#pragma unroll
  for(int it = 0; it < ITERS; it++)
  {
    word_zero(w[it]);
    if(q0 + it * SSD_PT_THREADS < nquads)
      word_load(F, (unsigned)(q0 + it * SSD_PT_THREADS), w[it]);
  }
  s_hist[tid] = 0; // SSD_PT_THREADS == SSD_BINS_PAD
  if(tid == 0)
    s_exact = 0;
  __syncthreads();
  unsigned *dst = reinterpret_cast<unsigned *>(codes + fbase) + q0;
  unsigned exact = 0;
#pragma unroll
  for(int it = 0; it < ITERS; it++)
    if(q0 + it * SSD_PT_THREADS < nquads)
    {
      float vx[4], vy[4], vz[4];
      word_unpack(F, w[it], vx, vy, vz);
      tb_word(p, vx, vy, vz, dst + it * SSD_PT_THREADS, s_hist, exact);
    }
  if(exact)
    atomicAdd(&s_exact, exact);
  __syncthreads();
  const unsigned sum = s_hist[tid];
  if(sum)
    atomicAdd(&frames[frame].hist[tid], sum);
  if(tid == 0 && s_exact)
    atomicAdd(&frames[frame].n_exact_bin, s_exact);
  if(FUSE_PEAKS)
  {
    __shared__ PeaksScratch K;
    __shared__ unsigned s_last;
    tb_fused_peaks(p, frames[frame], K, s_last, tid);
  }
}
// k_transform_bin_lens: the same pass on z16 frames of a distorted lens (SrcLens), 10 bytes per point in (2 of depth, 8 of ray
// from the L2-resident table). A copy of k_transform_bin_depth's body: that kernel's code stays as it was.
template<int ITERS, bool FUSE_PEAKS = false, class CAM = NoCam>
__global__ void __launch_bounds__(SSD_PT_THREADS) k_transform_bin_lens(const __grid_constant__ DevParams p0, const SrcLens src0,
                                                                        unsigned char *__restrict__ codes, FrameDev *__restrict__ frames,
                                                                        const CAM cam = CAM())
{
  __shared__ unsigned s_hist[SSD_BINS_PAD];
  __shared__ unsigned s_exact;
  const int tid = threadIdx.x;
  const int frame = blockIdx.y;
  const DevParams &p = frame_params(p0, cam, frame);
  const auto &src = frame_src(src0, cam, p, frame);
  const size_t fbase = (size_t)frame * p.N;
  const int nquads = p.N >> 2;
  const int q0 = blockIdx.x * (ITERS * SSD_PT_THREADS) + tid;
  const FrameL F = src_frame(src, p, fbase);
  WordL w[ITERS];
#pragma unroll
  for(int it = 0; it < ITERS; it++)
  {
    word_zero(w[it]);
    if(q0 + it * SSD_PT_THREADS < nquads)
      word_load(F, (unsigned)(q0 + it * SSD_PT_THREADS), w[it]);
  }
  s_hist[tid] = 0; // SSD_PT_THREADS == SSD_BINS_PAD
  if(tid == 0)
    s_exact = 0;
  __syncthreads();
  unsigned *dst = reinterpret_cast<unsigned *>(codes + fbase) + q0;
  unsigned exact = 0;
#pragma unroll
  for(int it = 0; it < ITERS; it++)
    if(q0 + it * SSD_PT_THREADS < nquads)
    {
      float vx[4], vy[4], vz[4];
      word_unpack(F, w[it], vx, vy, vz);
      tb_word(p, vx, vy, vz, dst + it * SSD_PT_THREADS, s_hist, exact);
    }
  if(exact)
    atomicAdd(&s_exact, exact);
  __syncthreads();
  const unsigned sum = s_hist[tid];
  if(sum)
    atomicAdd(&frames[frame].hist[tid], sum);
  if(tid == 0 && s_exact)
    atomicAdd(&frames[frame].n_exact_bin, s_exact);
  if(FUSE_PEAKS)
  {
    __shared__ PeaksScratch K;
    __shared__ unsigned s_last;
    tb_fused_peaks(p, frames[frame], K, s_last, tid);
  }
}

// ---------------------------------------------------------------------------------------------
// k_peaks: HeightsHistogram::findPeaks/filterPeaks (pointcloud.cpp:214-256), the plateau bands of
// PlateausExtraction::extractPlateauPoints (:300-335) folded into a bin->label LUT, and the ground /
// first-outlined bookkeeping of StairsDetector::detectStairSteps (:402-418).
// One warp per frame (peaks_warp above: bin-parallel).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_peaks(const __grid_constant__ DevParams p, FrameDev *__restrict__ frames, int n_frames)
{
  __shared__ PeaksScratch K;
  const int f = blockIdx.x, lane = threadIdx.x;
  if(f >= n_frames)
    return;
  const uint4 *src = reinterpret_cast<const uint4 *>(frames[f].hist) + lane * 2;
  const uint4 h0 = src[0], h1 = src[1];
  peaks_warp(p, frames[f], K, h0, h1, lane);
}

// ---------------------------------------------------------------------------------------------
// Shared machinery of k_label_bev and k_quad_reduce: warp-level stream compaction per segment.
// Both walk a frame in pixel order. grid = (blocks per frame, frames): a block loads the frame's small tables
// once; each of its warps then works through its own contiguous run of warp-tiles (1024 consecutive pixels,
// i.e. eight coalesced 128 B label loads per warp), with no block-level barrier until the very end.
//   Phase A (all pixels, a handful of instructions per 4-pixel word): label word -> which of its pixels matter
//     -> the warp compacts the words with at least one such pixel into its private list in shared memory
//     (ballot + popc prefix, no atomics). The next warp-tile's line of label words is requested into L2 as soon as the
//     current one has been read (keeping it in registers across phase B cost more in occupancy than it hid).
//   Phase B (dense): the warp walks the compacted list 32 words = 128 pixels at a time: three aligned 16 B
//     vertex loads per lane (or 8 B of depth); only words that matter are ever fetched. k_quad_reduce requests
//     them into L2 during phase A and loads them where they are consumed; k_label_bev issues the loads one step ahead.
// Every per-point decision in phase B is first taken in single precision with a rigorous error bound
// (fast_pixel, quadfilter_eval). The few points that come within the bound of a threshold are appended to a
// second compacted list and re-decided by the exact double-precision chain in a dense pass at the end of the
// warp-tile, instead of diverging the warp in line. Both lists have one slot per word / pixel: no overflow.
// ---------------------------------------------------------------------------------------------
#define SSD_WT_PX 1024   // pixels per warp-tile = 32 lanes x 8 label words x 4 pixels
#define SSD_WT_WORDS 8
#define SSD_DEF_BEVONLY 0x8000u

struct WarpLists
{
  unsigned lab[SSD_PT_WARPS][SSD_WT_PX / 4];        // the warp-tile's label words
  unsigned short act[SSD_PT_WARPS][SSD_WT_PX / 4];  // word index << 4 | mask of the pixels that matter
  unsigned short def[SSD_PT_WARPS][SSD_WT_PX];      // flag | word index << 2 | pixel of the word
  unsigned ndef[SSD_PT_WARPS];
  unsigned short gb[SSD_PT_WARPS][SSD_WT_PX / 4];   // k_quad_reduce: words with ground points whose BEV pixel is wanted (index << 4 | mask)
  unsigned ngb[SSD_PT_WARPS];
};

// Append word (it*32+lane) with pixel mask am4 to the warp's list (length n, warp-uniform); returns the new
// length. All 32 lanes call.
__device__ __forceinline__ unsigned compact_append(unsigned short *list, unsigned n, unsigned am4, int it, int lane)
{
  const unsigned b = __ballot_sync(0xffffffffu, am4 != 0u);
  if(am4)
    list[n + __popc(b & ((1u << lane) - 1u))] = (unsigned short)(((unsigned)(it * 32 + lane) << 4) | am4);
  return n + __popc(b);
}

__device__ __forceinline__ void defer_push(WarpLists &L, int warp, unsigned e)
{
  const unsigned slot = atomicAdd(&L.ndef[warp], 1u);
  L.def[warp][slot] = (unsigned short)e;
}

// warp-tiles of this warp: first, first + stride, ... < n_wt. Interleaved over all warps of the frame's blocks:
// neighbouring image rows carry similar amounts of work, so every warp (and block) gets an even share and the
// final block barrier does not wait for a straggler.
__device__ __forceinline__ void warp_tile_range(int n_wt, int warp, int &first, int &end, int &stride)
{
  first = blockIdx.x * SSD_PT_WARPS + warp;
  stride = gridDim.x * SSD_PT_WARPS;
  end = n_wt;
}

// ---------------------------------------------------------------------------------------------
// k_label_bev: the per-point segment label (PlateausExtraction::extractPlateaus, pointcloud.cpp:280-343,
// as a LUT lookup) and StairsDetector::projectToBinaryImage (:458-471) for every outlined plateau.
// Rewrites the bin codes in place as labels (a word is stored only if it changes: invalid / out-of-range
// codes equal their labels).
// ---------------------------------------------------------------------------------------------
struct LabelBevShared
{
  // bin code -> {label << 8 j, (label gets a BEV image) << j}, one table per byte position j of a 4-pixel code word: the label
  // word and the pixel mask of a code word are the OR of four 8-byte lookups, no shifting / masking of the looked-up values
  // (measured against one 16-bit table: k_label_bev 2.03 -> 1.96 ms per 2048 frames)
  uint2 lut64[4][SSD_BINS_PAD];
  int rmin[SSD_GPU_MAX_PLATEAUS], rmax[SSD_GPU_MAX_PLATEAUS];
  unsigned oob, n_def;
  WarpLists L;
};

__device__ __forceinline__ void label_bev_exact_point(const DevParams &p, float fx, float fy, float fz, unsigned l, unsigned *__restrict__ fbev,
                                                      size_t bm_words, LabelBevShared &S)
{
  double wx, wy;
  camera_to_world_xy(p, fx, fy, fz, wx, wy);
  int x, y;
  if(bev_pixel(p, wx, wy, x, y))
  {
    atomicOr(fbev + (size_t)l * bm_words + (size_t)y * p.wpr + (x >> 5), 1u << (x & 31));
    atomicMin(&S.rmin[l], y);
    atomicMax(&S.rmax[l], y);
  }
  else
    S.oob = 1;
}

#ifndef SSD_LB_MINB
#define SSD_LB_MINB 4
#endif
// REC: every 4-pixel word with points of outlined plateaus also leaves an 8-byte word record for k_quad_reduce_rec (word_rec_*):
// the box of its BEV pixels and the fixed-point z sum of those points, so that pass 3 takes a word that lies inside its step's
// quadrilateral without reading its vertices again.
#define SSD_WREC_ELIGIBLE 0x40000000u // one label, every pixel certain, box at most 8 x 8 pixels
__device__ __forceinline__ uint2 word_rec_pack(bool eligible, int xlo, int ylo, int xhi, int yhi, unsigned zsum, unsigned count)
{
  const unsigned lo = eligible ? ((unsigned)xlo | ((unsigned)ylo << 12) | ((unsigned)(xhi - xlo) << 24) | ((unsigned)(yhi - ylo) << 27) | SSD_WREC_ELIGIBLE) : 0u;
  return make_uint2(lo, zsum | (count << 25));
}

template<class SRC, bool REC = false, class CAM = NoCam>
__global__ void __launch_bounds__(SSD_PT_THREADS, SSD_LB_MINB) k_label_bev(const __grid_constant__ DevParams p0, const SRC src0,
                                                               unsigned char *__restrict__ labels, FrameDev *__restrict__ frames,
                                                               unsigned *__restrict__ bev, size_t bm_words, uint2 *__restrict__ wrec = nullptr,
                                                               const CAM cam = CAM())
{
  __shared__ LabelBevShared S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int frame = blockIdx.y;
  const DevParams &p = frame_params(p0, cam, frame);
  const auto &src = frame_src(src0, cam, p, frame);
  FrameDev &F = frames[frame];
  const size_t fbase = (size_t)frame * p.N;
  unsigned *lab32 = reinterpret_cast<unsigned *>(labels + fbase);
  unsigned *fbev = bev + (size_t)frame * SSD_GPU_MAX_PLATEAUS * bm_words;
  const typename SrcTraits<SRC>::Frame FR = src_frame(src, p, fbase);
  const int nquads = p.N >> 2;
  int wt, wt_end, wt_stride;
  warp_tile_range((p.N + SSD_WT_PX - 1) / SSD_WT_PX, warp, wt, wt_end, wt_stride);

  {
    const unsigned e = F.lut16[tid]; // SSD_PT_THREADS == SSD_BINS_PAD
#pragma unroll
    for(int j = 0; j < 4; j++)
      S.lut64[j][tid] = make_uint2((e & 0xffu) << (8 * j), ((e >> 8) & 1u) << j);
  }
  if(tid < SSD_GPU_MAX_PLATEAUS)
  {
    S.rmin[tid] = 0x7fffffff;
    S.rmax[tid] = -1;
  }
  if(tid < SSD_PT_WARPS)
    S.L.ndef[tid] = 0;
  if(tid == 0)
  {
    S.oob = 0;
    S.n_def = 0;
  }
  __syncthreads();

  unsigned short *act = S.L.act[warp];
  unsigned *labs = S.L.lab[warp];
  const unsigned bmw = (unsigned)bm_words, wpr = (unsigned)p.wpr;
  unsigned rl = 0xffu; // label of the lane's current row-range run
  int rlo = 0x7fffffff, rhi = -1;
  unsigned n_def = 0;

  for(; wt < wt_end; wt += wt_stride)
  {
    // ---- phase A: codes -> labels, compaction of the words with pixels of outlined plateaus ----
    unsigned n = 0;
    // the tile's eight code words per lane, live in registers during phase A only; the next tile's 1 KB line is requested
    // into L2 now (keeping it in registers across phase B cost more in occupancy than it hid in latency)
    unsigned labw[SSD_WT_WORDS];
#pragma unroll
    for(int it = 0; it < SSD_WT_WORDS; it++)
    {
      const int q = wt * (SSD_WT_PX / 4) + it * 32 + lane;
      labw[it] = q < nquads ? lab32[q] : 0xffffffffu;
    }
    if(wt + wt_stride < wt_end)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(lab32 + (size_t)(wt + wt_stride) * (SSD_WT_PX / 4) + lane * 8));
#pragma unroll
    for(int it = 0; it < SSD_WT_WORDS; it++)
    {
      const unsigned cw = labw[it];
      unsigned am4 = 0;
      // codes 254 / 255 (out of range / invalid) are their own labels and never matter: skip such words outright
      if((cw & 0xfefefefeu) != 0xfefefefeu)
      {
        const uint2 a0 = S.lut64[0][cw & 0xffu], a1 = S.lut64[1][(cw >> 8) & 0xffu], a2 = S.lut64[2][(cw >> 16) & 0xffu], a3 = S.lut64[3][cw >> 24];
        const unsigned lab = a0.x | a1.x | a2.x | a3.x;
        am4 = a0.y | a1.y | a2.y | a3.y;
        lab32[wt * (SSD_WT_PX / 4) + it * 32 + lane] = lab; // (cw is never the all-ones padding here)
        labs[it * 32 + lane] = lab;
      }
      if(__any_sync(0xffffffffu, am4 != 0u))
        n = compact_append(act, n, am4, it, lane);
    }
    if(n == 0)
      continue;
    __syncwarp();

    // ---- phase B: dense walk over the compacted words ----
    const unsigned wbase = (unsigned)wt * (SSD_WT_PX / 4); // first word of the warp-tile within the frame
    unsigned e = lane < n ? act[lane] : 0u;
    typename SrcTraits<SRC>::Word wc, wn;
    word_zero(wc);
    word_zero(wn);
    if(e)
      word_load(FR, wbase + (e >> 4), wc);
    for(unsigned s0 = 0; s0 < n; s0 += 32)
    {
      const unsigned i1 = s0 + 32 + lane;
      const unsigned e1 = i1 < n ? act[i1] : 0u;
      if(e1)
        word_load(FR, wbase + (e1 >> 4), wn);
      const unsigned lab = labs[e >> 4];
      const unsigned m4 = e & 15u;
      float vx[4], vy[4], vz[4];
      word_unpack(FR, wc, vx, vy, vz);
      // the four pixels in straight-line code (the chains of the four points interleave); inactive lanes (e == 0) and
      // inactive points compute on whatever the registers hold and are masked out by m4
      int ix[4], iy[4];
      unsigned okm = 0;
#pragma unroll
      for(int j = 0; j < 4; j++)
        okm |= fast_pixel2(p, vx[j], vy[j], vz[j], ix[j], iy[j]) ? (1u << j) : 0u;
      const unsigned good = okm & m4, bad = ~okm & m4;
      // label of the word's first point of an outlined plateau; the word is "uniform" when all such points carry it
      // (image rows are iso-height: almost every word is)
      const unsigned l0 = (lab >> (8 * (__ffs(m4 | 16u) - 1) & 31)) & 0xffu;
      const unsigned bytes = ((m4 * 0x00204081u) & 0x01010101u) * 0xffu;
      const bool uniform = ((lab ^ (l0 * 0x01010101u)) & bytes) == 0u;
      int ylo = 0x7fffffff, yhi = -1, xlo = 0x7fffffff, xhi = -1;
      if(uniform)
      {
        // word index of the plateau's bitmap within the stream's BEV buffer: 32-bit (the buffer holds < 2^32 words, see
        // ssd_gpu_create), so a reduction's address is one widening multiply-add on the kernel's base pointer
        unsigned lidx = ((unsigned)frame * SSD_GPU_MAX_PLATEAUS + l0) * bmw;
        asm volatile("" : "+r"(lidx)); // keep it in a register: the compiler otherwise recomputes it inside every predicated reduction
#pragma unroll
        for(int j = 0; j < 4; j++)
          if((good >> j) & 1u)
          {
            atomicOr(bev + (lidx + (unsigned)iy[j] * wpr + ((unsigned)ix[j] >> 5)), 1u << (ix[j] & 31));
            ylo = min(ylo, iy[j]);
            yhi = max(yhi, iy[j]);
            if(REC)
            {
              xlo = min(xlo, ix[j]);
              xhi = max(xhi, ix[j]);
            }
          }
        if(yhi >= 0)
        {
          if(l0 != rl)
          {
            if(rhi >= 0)
            {
              atomicMin(&S.rmin[rl], rlo);
              atomicMax(&S.rmax[rl], rhi);
            }
            rl = l0;
            rlo = 0x7fffffff;
            rhi = -1;
          }
          rlo = min(rlo, ylo);
          rhi = max(rhi, yhi);
        }
      }
      else
      {
        // two plateaus meet inside the word: per point
#pragma unroll
        for(int j = 0; j < 4; j++)
          if((good >> j) & 1u)
          {
            const unsigned l = (lab >> (8 * j)) & 0xffu;
            atomicOr(fbev + (l * bmw + (unsigned)iy[j] * wpr + ((unsigned)ix[j] >> 5)), 1u << (ix[j] & 31));
            atomicMin(&S.rmin[l], iy[j]);
            atomicMax(&S.rmax[l], iy[j]);
          }
      }
      if(bad)
      {
#pragma unroll
        for(int j = 0; j < 4; j++)
          if((bad >> j) & 1u)
            defer_push(S.L, warp, ((e >> 4) << 2) | (unsigned)j);
      }
      if(REC && e)
      {
        unsigned zs = 0;
#pragma unroll
        for(int j = 0; j < 4; j++)
          zs += z_fix_u(p, vx[j], vy[j], vz[j]) & (0u - ((m4 >> j) & 1u));
        const bool eligible = uniform && bad == 0u && yhi >= 0 && xhi - xlo < 8 && yhi - ylo < 8;
        wrec[(size_t)frame * (size_t)nquads + wbase + (e >> 4)] = word_rec_pack(eligible, xlo, ylo, xhi, yhi, zs, (unsigned)__popc(m4));
      }
      e = e1;
      wc = wn;
    }
    // ---- dense exact pass over the warp's compacted uncertain points ----
    __syncwarp();
    const unsigned nd = S.L.ndef[warp];
    if(nd)
    {
      for(unsigned i = lane; i < nd; i += 32)
      {
        const unsigned d = S.L.def[warp][i];
        const unsigned w = (d >> 2) & 0xffu, j = d & 3u;
        float fx, fy, fz;
        point_load(FR, (wbase + w) * 4u + j, fx, fy, fz);
        label_bev_exact_point(p, fx, fy, fz, (labs[w] >> (8 * j)) & 0xffu, fbev, bm_words, S);
      }
      __syncwarp();
      n_def += nd;
      if(lane == 0)
        S.L.ndef[warp] = 0;
    }
    __syncwarp();
  }
  if(rhi >= 0)
  {
    atomicMin(&S.rmin[rl], rlo);
    atomicMax(&S.rmax[rl], rhi);
  }
  if(lane == 0 && n_def)
    atomicAdd(&S.n_def, n_def);
  __syncthreads();
  if(tid < SSD_GPU_MAX_PLATEAUS && S.rmax[tid] >= 0)
  {
    atomicMin(&F.plat[tid].row_min, S.rmin[tid]);
    atomicMax(&F.plat[tid].row_max, S.rmax[tid]);
  }
  if(tid == 0)
  {
    if(S.oob)
      atomicOr(&F.status, SSD_STATUS_BEV_OOB);
    if(S.n_def)
      atomicAdd(&F.n_def_bev, S.n_def);
  }
}

// ---------------------------------------------------------------------------------------------
// k_quad_reduce: StairsDetector::getPointsInQuadrilateral + calcAverageZ (pointcloud.cpp:560-581) for the
// ground and every valid plateau, and the ground's BEV image (calcGround, :530-531).
// Point-in-quadrilateral: single-precision fast accept against the verified inner box; the warp steps that
// still have undecided points evaluate the f32 image of the reference's own test structure
// (quadfilter_eval); what stays uncertain goes to the compacted exact pass.
// z is accumulated in 2^-36 m fixed point: integer sums are order independent, so the result is deterministic;
// the error (<= 2^-37 m per point) is seven orders below the 0.1 mm tolerance. Each lane keeps a running
// (label, sum, count) segment in registers -- consecutive words of a lane mostly share a label -- and
// adds it to the block's shared-memory accumulators when the label changes; at the end the warp combines its
// 32 open segments with one match.any + redux pass (single-pass segmented reduce): one shared-memory add per
// distinct label and warp, one global atomic per step and block.
// Ground BEV: only the pixel columns Segmentation::detectFrontEdge can see (BottomScanner probes columns
// W/2 + 50 j; the 3x3 close reaches two columns to either side) are written.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ bool ground_col_needed(const DevParams &p, int x)
{
  const unsigned v = (unsigned)(x - (p.W / 2 - 2) + 50 * 128); // non-negative for W <= 12800
  return v % 50u < 5u;
}

struct QuadFast
{
  float4 ibe; // cx, cy, inner half widths minus epsc (negative: no inner box)
  float2 rj;  // reject half widths
  float2 pad;
};

struct QuadReduceShared
{
  QuadFilterDev qf[SSD_GPU_MAX_PLATEAUS];
  QuadFast fast[SSD_GPU_MAX_PLATEAUS];
  unsigned slo[SSD_GPU_MAX_PLATEAUS], shi[SSD_GPU_MAX_PLATEAUS]; // per-step z sum: low 16 bits / the rest (native 32-bit shared atomics)
  unsigned cnt[SSD_GPU_MAX_PLATEAUS];
  int rmin, rmax;
  unsigned oob, n_def, pad, pad1;
  WarpLists L;
};

// add a (sum, count) segment of label l to the block's accumulators. sum < 2^23 * points of a block: fits 16 + 32 bits
__device__ __forceinline__ void seg_flush(QuadReduceShared &S, unsigned l, unsigned long long sum, unsigned n)
{
  atomicAdd(&S.slo[l], (unsigned)sum & 0xffffu);
  atomicAdd(&S.shi[l], (unsigned)(sum >> 16));
  atomicAdd(&S.cnt[l], n);
}

// one point of the compacted exact pass: the reference's own double-precision test
__device__ __forceinline__ void quad_reduce_exact_point(const DevParams &p, float fx, float fy, float fz, unsigned l, bool bevonly, const FrameDev &F,
                                                        unsigned amask, int ground, unsigned *__restrict__ gbev, QuadReduceShared &S)
{
  if(l >= SSD_GPU_MAX_PLATEAUS || !((amask >> l) & 1u))
    return;
  double wx, wy;
  camera_to_world_xy(p, fx, fy, fz, wx, wy);
  if(!bevonly)
  {
    if(!quadtest_within(F.plat[l].qt, wx, wy))
      return;
    seg_flush(S, l, z_fix_u(p, fx, fy, fz), 1u);
  }
  if((int)l == ground)
  {
    int x, y;
    if(!bev_pixel(p, wx, wy, x, y))
      S.oob = 1;
    else if(ground_col_needed(p, x))
    {
      atomicOr(gbev + (size_t)y * p.wpr + (x >> 5), 1u << (x & 31));
      atomicMin(&S.rmin, y);
      atomicMax(&S.rmax, y);
    }
  }
}

#define SSD_DEF_MID 0x2000u     // deferred point between inner and reject box: f32 image of the test first
#define SSD_DEF_GENERIC 0x4000u // deferred point of a word with mixed labels: not yet checked against amask

// state a warp of k_quad_reduce / k_quad_sum carries across its warp-tiles
struct QrWarp
{
  unsigned seg_l, seg_n, n_def, n_mid;
  unsigned long long seg_sum;
  int rmin, rmax;
};

// end of a warp-tile: combine the warp's 32 open segments (single-pass segmented reduce: lanes grouped by label, 64-bit sums
// as 21 low bits + the rest), one set of shared-memory adds per distinct label
__device__ __forceinline__ void qr_seg_combine(QuadReduceShared &S, QrWarp &W, int lane)
{
  const unsigned key = W.seg_n ? W.seg_l : 0xffu;
  const unsigned grp = __match_any_sync(0xffffffffu, key);
  const unsigned lo = __reduce_add_sync(grp, (unsigned)W.seg_sum & 0x1fffffu);
  const unsigned hi = __reduce_add_sync(grp, (unsigned)(W.seg_sum >> 21)); // a lane's sum < 2^23 * 2^10 points per tile
  const unsigned cn = __reduce_add_sync(grp, W.seg_n);
  if(key != 0xffu && lane == __ffs(grp) - 1)
    seg_flush(S, key, ((unsigned long long)hi << 21) + (unsigned long long)lo, cn);
  W.seg_l = 0xffu;
  W.seg_sum = 0;
  W.seg_n = 0;
}

// The dense part of one warp-tile: phase B over the n compacted words of the warp's list (S.L.act / S.L.lab), the exact
// pass over the deferred points, the queued ground BEV pixels, and the warp's segmented reduce. wbase: first 4-point word
// of the warp-tile within the frame.
template<class SRC, class FRAME>
__device__ __forceinline__ void qr_dense(const DevParams &p, const FRAME &FR, QuadReduceShared &S, QrWarp &W, const FrameDev &F, unsigned amask, int ground,
                                         unsigned *__restrict__ gbev, unsigned wbase, unsigned n, int warp, int lane)
{
  unsigned short *act = S.L.act[warp];
  unsigned *labs = S.L.lab[warp];
  unsigned &seg_l = W.seg_l, &seg_n = W.seg_n, &n_def = W.n_def, &n_mid = W.n_mid;
  unsigned long long &seg_sum = W.seg_sum;
  int &rmin = W.rmin, &rmax = W.rmax;
  // ---- phase B: dense walk over the compacted words ----
  unsigned e = lane < n ? act[lane] : 0u;
  typename SrcTraits<SRC>::Word wc;
  word_zero(wc);
  if(e)
    word_load(FR, wbase + (e >> 4), wc);
  for(unsigned s0 = 0; s0 < n; s0 += 32)
  {
    // (no software prefetch of the next step's words: the L2 prefetch of phase A and four resident blocks per SM hide the
    //  latency better than twelve more registers per thread did -- measured 2.51 -> 2.28 ms per 2048 frames)
    if(s0)
    {
      const unsigned i0 = s0 + lane;
      e = i0 < n ? act[i0] : 0u;
      if(e)
        word_load(FR, wbase + (e >> 4), wc);
    }
    const unsigned m4 = e & 15u;
    const unsigned lw = labs[e >> 4];
    // label of the word's first plateau point; the word is "uniform" when all its plateau points carry it
    const unsigned l0 = (lw >> (8 * (__ffs(m4 | 16u) - 1) & 31)) & 0x1fu;
    const unsigned bytes = ((m4 * 0x00204081u) & 0x01010101u) * 0xffu;
    const bool uniform = ((lw ^ (l0 * 0x01010101u)) & bytes) == 0u;
    float vx[4], vy[4], vz[4];
    word_unpack(FR, wc, vx, vy, vz);
    if(uniform)
    {
      // Branch-free on sign bits (every operand is finite here: plateau points are valid and in range, the tables
      // hold finite numbers or +inf). Labels outside amask have an empty inner box and an empty reject box.
      //   in  <=> active && |wx - cx| < hx && |wy - cy| < hy      (sign of |d| - h, both set)
      //   rej <=> |wx - cx| > Rx || |wy - cy| > Ry                 (sign of R - |d|, either set)
      //   mid <=> active && !in && !rej  -> deferred
      const float4 ib = S.fast[l0].ibe;
      const float2 rj = S.fast[l0].rj;
      float wxs[4];
      int inm[4], midm[4];
      int cnt = 0;
      unsigned zs = 0;
#pragma unroll
      for(int j = 0; j < 4; j++)
      {
        float wy;
        f2_unpack(f2_affine(p.axy2, p.bxy2, vx[j], vy[j], vz[j]), wxs[j], wy);
        const float dx = fabsf(wxs[j] - ib.x), dy = fabsf(wy - ib.y);
        const int act = (int)(m4 << (31 - j));
        const int ins = __float_as_int(dx - ib.z) & __float_as_int(dy - ib.w) & act;
        const int rej = __float_as_int(rj.x - dx) | __float_as_int(rj.y - dy);
        midm[j] = act & ~ins & ~rej;
        inm[j] = ins >> 31; // all ones when inside
        zs += z_fix_u(p, vx[j], vy[j], vz[j]) & (unsigned)inm[j];
        cnt -= inm[j];
      }
      // between the inner box and the reject box (a few percent of the points, but in most warp steps): deferred to
      // the dense pass at the end of the warp-tile, which evaluates the f32 image of the full test one point per lane
      if((midm[0] | midm[1] | midm[2] | midm[3]) < 0)
      {
#pragma unroll
        for(int j = 0; j < 4; j++)
          if(midm[j] < 0)
            defer_push(S.L, warp, SSD_DEF_MID | ((e >> 4) << 2) | (unsigned)j);
      }
      if(cnt)
      {
        if(l0 != seg_l)
        {
          if(seg_n)
            seg_flush(S, seg_l, seg_sum, seg_n);
          seg_l = l0;
          seg_sum = 0;
          seg_n = 0;
        }
        seg_sum += zs;
        seg_n += (unsigned)cnt;
        if((int)l0 == ground)
        {
          // Ground BEV image: only the pixel columns detectFrontEdge can see are written. Cheap column pre-filter
          // (f32, conservative margin): t = ((wx - x_min) sx - (W/2 - 2)) / 50, the column is needed iff frac(t) in
          // [0, 0.1). The few points that pass are queued per word; their pixels are computed densely at the end of
          // the warp-tile (one point per lane) instead of diverging every step here.
          unsigned gm = 0;
#pragma unroll
          for(int j = 0; j < 4; j++)
          {
            const float t = fmaf(wxs[j], p.gcol_a, p.gcol_b);
            const float fr = t - floorf(t);
            gm |= (fr < p.gcol_lo || fr > p.gcol_hi || t > p.gcol_tmax) ? (1u << j) : 0u;
          }
          gm &= (unsigned)(inm[0] & 1) | (unsigned)(inm[1] & 2) | (unsigned)(inm[2] & 4) | (unsigned)(inm[3] & 8);
          if(gm)
            S.L.gb[warp][atomicAdd(&S.L.ngb[warp], 1u)] = (unsigned short)((e & 0xff0u) | gm);
        }
      }
    }
    else
    {
      // mixed labels in one word (plateau boundaries in the image): every point goes to the exact pass
#pragma unroll
      for(int j = 0; j < 4; j++)
        if((m4 >> j) & 1u)
          defer_push(S.L, warp, SSD_DEF_GENERIC | ((e >> 4) << 2) | (unsigned)j);
    }
  }
  // ---- dense exact pass over the warp's compacted uncertain points ----
  __syncwarp();
  const unsigned nd = S.L.ndef[warp];
  if(nd)
  {
    for(unsigned i = lane; i < nd; i += 32)
    {
      const unsigned d = S.L.def[warp][i];
      const unsigned w = (d >> 2) & 0xffu, j = d & 3u;
      const unsigned l = (labs[w] >> (8 * j)) & 0xffu;
      float fx, fy, fz;
      point_load(FR, (wbase + w) * 4u + j, fx, fy, fz);
      bool exact = true, bevonly = (d & SSD_DEF_BEVONLY) != 0u;
      if(d & SSD_DEF_MID)
      {
        float wxf, wyf;
        f2_unpack(f2_affine(p.axy2, p.bxy2, fx, fy, fz), wxf, wyf);
        bool unc;
        const bool in = quadfilter_eval(S.qf[l & 31u], wxf, wyf, p.epsc, unc);
        if(!unc)
        {
          n_mid++;
          exact = in && (int)l == ground; // certain: count it here; an inside ground point still needs its BEV pixel
          bevonly = true;
          if(in)
          {
            // into the lane's running segment (no shared-memory atomics: 64-bit ones are CAS loops)
            if(l != seg_l)
            {
              if(seg_n)
                seg_flush(S, seg_l, seg_sum, seg_n);
              seg_l = l;
              seg_sum = 0;
              seg_n = 0;
            }
            seg_sum += z_fix_u(p, fx, fy, fz);
            seg_n++;
          }
        }
      }
      if(exact)
        quad_reduce_exact_point(p, fx, fy, fz, l, bevonly, F, amask, ground, gbev, S);
    }
    __syncwarp();
    n_def += nd;
    if(lane == 0)
      S.L.ndef[warp] = 0;
  }
  {
    // ---- dense pass over the queued ground points: BEV pixel, one queued word per lane ----
    const unsigned ng = S.L.ngb[warp];
    if(ng)
    {
      for(unsigned i = lane; i < ng; i += 32)
      {
        const unsigned d = S.L.gb[warp][i];
        const unsigned w = (d >> 4) & 0xffu;
        unsigned mask = d & 15u;
#pragma unroll 1
        while(mask)
        {
          const unsigned j = __ffs(mask) - 1;
          mask &= mask - 1u;
          float fx, fy, fz;
          point_load(FR, (wbase + w) * 4u + j, fx, fy, fz);
          int ix, iy;
          if(fast_pixel2(p, fx, fy, fz, ix, iy))
          {
            if(ground_col_needed(p, ix))
            {
              atomicOr(gbev + (unsigned)iy * (unsigned)p.wpr + (unsigned)(ix >> 5), 1u << (ix & 31));
              rmin = min(rmin, iy);
              rmax = max(rmax, iy);
            }
          }
          else
            quad_reduce_exact_point(p, fx, fy, fz, (unsigned)ground, true, F, amask, ground, gbev, S);
        }
      }
      __syncwarp();
      if(lane == 0)
        S.L.ngb[warp] = 0;
    }
  }
  qr_seg_combine(S, W, lane);
}

// the frame's filter tables and the block's accumulators (k_quad_reduce / k_quad_sum)
__device__ __forceinline__ void qr_init(QuadReduceShared &S, const FrameDev &F, unsigned amask, int tid)
{
    // the frame's filter tables: one coalesced copy, independent of anything else
    const unsigned *src = reinterpret_cast<const unsigned *>(F.qf);
    unsigned *dst = reinterpret_cast<unsigned *>(S.qf);
    for(int i = tid; i < (int)(sizeof(S.qf) / 4); i += SSD_PT_THREADS)
      dst[i] = src[i];
    if(tid < SSD_GPU_MAX_PLATEAUS)
    {
      S.slo[tid] = 0;
      S.shi[tid] = 0;
      S.cnt[tid] = 0;
      const bool live = (amask >> tid) & 1u;
      // labels outside amask: never inside, always rejected
      S.fast[tid].ibe = live ? F.qf[tid].ibe : make_float4(0.f, 0.f, -1.f, -1.f);
      const float4 rj = F.qf[tid].rj;
      S.fast[tid].rj = live ? make_float2(rj.x, rj.y) : make_float2(-1.f, -1.f);
    }
    if(tid < SSD_PT_WARPS)
    {
      S.L.ndef[tid] = 0;
      S.L.ngb[tid] = 0;
    }
    if(tid == 0)
    {
      S.rmin = 0x7fffffff;
      S.rmax = -1;
      S.oob = 0;
      S.n_def = 0;
    }
}

// end of k_quad_reduce / k_quad_sum: the warps' leftovers into the block's accumulators, the block's into the frame's
__device__ __forceinline__ void qr_epilogue(QuadReduceShared &S, QrWarp &W, FrameDev &F, int ground, int tid, int lane)
{
  unsigned n_def = W.n_def;
  int rmin = W.rmin, rmax = W.rmax;
  n_def -= __reduce_add_sync(0xffffffffu, W.n_mid); // deferred points settled by the f32 image of the test are not exact decisions
  rmin = __reduce_min_sync(0xffffffffu, rmin);
  rmax = __reduce_max_sync(0xffffffffu, rmax);
  if(lane == 0)
  {
    if(rmax >= 0)
    {
      atomicMin(&S.rmin, rmin);
      atomicMax(&S.rmax, rmax);
    }
    if(n_def)
      atomicAdd(&S.n_def, n_def);
  }
  __syncthreads();
  if(tid < SSD_GPU_MAX_PLATEAUS && S.cnt[tid])
  {
    atomicAdd(&F.plat[tid].sum_fix, ((unsigned long long)S.shi[tid] << 16) + (unsigned long long)S.slo[tid]);
    atomicAdd(&F.plat[tid].n_in_quad, S.cnt[tid]);
  }
  if(tid == 0)
  {
    if(S.rmax >= 0)
    {
      atomicMin(&F.plat[ground].row_min, S.rmin);
      atomicMax(&F.plat[ground].row_max, S.rmax);
    }
    if(S.oob)
      atomicOr(&F.status, SSD_STATUS_BEV_OOB);
    if(S.n_def)
      atomicAdd(&F.n_def_quad, S.n_def);
  }
}

#ifndef SSD_QR_MINB
#define SSD_QR_MINB 4
#endif
template<class SRC, class CAM = NoCam>
__global__ void __launch_bounds__(SSD_PT_THREADS, SSD_QR_MINB) k_quad_reduce(const __grid_constant__ DevParams p0, const SRC src0,
                                                                 const unsigned char *__restrict__ labels, FrameDev *__restrict__ frames,
                                                                 unsigned *__restrict__ bev, size_t bm_words, const CAM cam = CAM())
{
  __shared__ QuadReduceShared S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int frame = blockIdx.y;
  const DevParams &p = frame_params(p0, cam, frame);
  const auto &src = frame_src(src0, cam, p, frame);
  FrameDev &F = frames[frame];
  const unsigned amask = F.quad_amask;
  if(amask == 0u)
    return; // no valid plateau: nothing is emitted (pointcloud.cpp:434)
  const int ground = F.ground_index;
  const size_t fbase = (size_t)frame * p.N;
  const unsigned *lab32 = reinterpret_cast<const unsigned *>(labels + fbase);
  unsigned *gbev = ground >= 0 ? bev + ((size_t)frame * SSD_GPU_MAX_PLATEAUS + ground) * bm_words : nullptr;
  const int nquads = p.N >> 2;
  int wt, wt_end, wt_stride;
  warp_tile_range((p.N + SSD_WT_PX - 1) / SSD_WT_PX, warp, wt, wt_end, wt_stride);

  qr_init(S, F, amask, tid);
  __syncthreads();

  unsigned short *act = S.L.act[warp];
  unsigned *labs = S.L.lab[warp];
  QrWarp W = { 0xffu, 0u, 0u, 0u, 0ull, 0x7fffffff, -1 };
  const typename SrcTraits<SRC>::Frame FR = src_frame(src, p, fbase);

  for(; wt < wt_end; wt += wt_stride)
  {
    const unsigned wbase = (unsigned)wt * (SSD_WT_PX / 4); // first word of the warp-tile within the frame
    // ---- phase A: compaction of the words holding plateau labels (bit 7 of a label byte clear <=> label < 128) ----
    unsigned n = 0;
    unsigned labw[SSD_WT_WORDS];
#pragma unroll
    for(int it = 0; it < SSD_WT_WORDS; it++)
    {
      const int q = wt * (SSD_WT_PX / 4) + it * 32 + lane;
      labw[it] = q < nquads ? __ldg(lab32 + q) : 0xffffffffu;
    }
    if(wt + wt_stride < wt_end)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(lab32 + (size_t)(wt + wt_stride) * (SSD_WT_PX / 4) + lane * 8));
#pragma unroll
    for(int it = 0; it < SSD_WT_WORDS; it++)
    {
      const unsigned lw = labw[it];
      const unsigned am4 = (((~lw >> 7) & 0x01010101u) * 0x10204080u) >> 28; // bit j <-> byte j < 128
      if(__any_sync(0xffffffffu, am4 != 0u))
      {
        if(am4)
        {
          labs[it * 32 + lane] = lw;
          word_prefetch_l2(FR, wbase + (unsigned)(it * 32 + lane));
        }
        n = compact_append(act, n, am4, it, lane);
      }
    }
    if(n == 0)
      continue;
    __syncwarp();

    qr_dense<SRC>(p, FR, S, W, F, amask, ground, gbev, wbase, n, warp, lane);
    __syncwarp();
  }
  qr_epilogue(S, W, F, ground, tid, lane);
}


// ---------------------------------------------------------------------------------------------
// k_quad_reduce_rec: k_quad_reduce for the chain whose k_label_bev<SRC, true> left word records. A 4-pixel word whose plateau
// points share one label of a valid (non-ground) step and whose record is eligible is decided as a whole: the world
// rectangle that every point with a BEV pixel in the record's box lies in -- centre (cx, cy), half extents widened by the
// rounding margins -- goes through the step's verified inner box and, failing that, through the f32 image of the reference's
// test (quadfilter_eval with the half extent as the position uncertainty: "certainly inside" then holds for every point of the
// rectangle). Such a word adds the record's z sum and count; its 48 bytes of vertices are not read. Everything else -- ground
// words (they also feed the ground's BEV image), words with mixed labels or an uncertain pixel, words the quadrilateral's
// edges come near -- is re-compacted and takes the dense pass of k_quad_reduce (qr_dense) unchanged, so both chains produce
// the same integer sums and counts.
// ---------------------------------------------------------------------------------------------
template<class SRC>
__global__ void __launch_bounds__(SSD_PT_THREADS, SSD_QR_MINB) k_quad_reduce_rec(const __grid_constant__ DevParams p, const SRC src,
                                                                     const unsigned char *__restrict__ labels, FrameDev *__restrict__ frames,
                                                                     unsigned *__restrict__ bev, size_t bm_words, const uint2 *__restrict__ wrec)
{
  __shared__ QuadReduceShared S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int frame = blockIdx.y;
  FrameDev &F = frames[frame];
  const unsigned amask = F.quad_amask;
  if(amask == 0u)
    return; // no valid plateau: nothing is emitted (pointcloud.cpp:434)
  const int ground = F.ground_index;
  const unsigned wmask = ground >= 0 ? amask & ~(1u << ground) : amask; // steps whose words can be taken whole
  const size_t fbase = (size_t)frame * p.N;
  const unsigned *lab32 = reinterpret_cast<const unsigned *>(labels + fbase);
  unsigned *gbev = ground >= 0 ? bev + ((size_t)frame * SSD_GPU_MAX_PLATEAUS + ground) * bm_words : nullptr;
  const int nquads = p.N >> 2;
  const uint2 *frec = wrec + (size_t)frame * (size_t)nquads;
  int wt, wt_end, wt_stride;
  warp_tile_range((p.N + SSD_WT_PX - 1) / SSD_WT_PX, warp, wt, wt_end, wt_stride);

  qr_init(S, F, amask, tid);
  __syncthreads();

  unsigned short *act = S.L.act[warp];
  unsigned *labs = S.L.lab[warp];
  QrWarp W = { 0xffu, 0u, 0u, 0u, 0ull, 0x7fffffff, -1 };
  const typename SrcTraits<SRC>::Frame FR = src_frame(src, p, fbase);
  const unsigned lt = (1u << lane) - 1u;

  for(; wt < wt_end; wt += wt_stride)
  {
    const unsigned wbase = (unsigned)wt * (SSD_WT_PX / 4); // first word of the warp-tile within the frame
    // ---- phase A: compaction of the words holding plateau labels (bit 7 of a label byte clear <=> label < 128) ----
    unsigned n = 0;
    unsigned labw[SSD_WT_WORDS];
#pragma unroll
    for(int it = 0; it < SSD_WT_WORDS; it++)
    {
      const int q = wt * (SSD_WT_PX / 4) + it * 32 + lane;
      labw[it] = q < nquads ? __ldg(lab32 + q) : 0xffffffffu;
    }
    if(wt + wt_stride < wt_end)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(lab32 + (size_t)(wt + wt_stride) * (SSD_WT_PX / 4) + lane * 8));
#pragma unroll
    for(int it = 0; it < SSD_WT_WORDS; it++)
    {
      const unsigned lw = labw[it];
      const unsigned am4 = (((~lw >> 7) & 0x01010101u) * 0x10204080u) >> 28; // bit j <-> byte j < 128
      if(__any_sync(0xffffffffu, am4 != 0u))
      {
        if(am4)
          labs[it * 32 + lane] = lw;
        n = compact_append(act, n, am4, it, lane);
      }
    }
    if(n == 0)
      continue;
    __syncwarp();

    // ---- phase B': whole words from their records; the rest is re-compacted in place (writes trail the reads) ----
    unsigned n2 = 0;
    for(unsigned s0 = 0; s0 < n; s0 += 32)
    {
      const unsigned i0 = s0 + lane;
      const unsigned e = i0 < n ? act[i0] : 0u;
      bool dense = false;
      if(e)
      {
        const unsigned m4 = e & 15u;
        const unsigned lw = labs[e >> 4];
        const unsigned l0 = (lw >> (8 * (__ffs(m4) - 1))) & 0xffu;
        const unsigned bytes = ((m4 * 0x00204081u) & 0x01010101u) * 0xffu;
        const bool uniform = ((lw ^ (l0 * 0x01010101u)) & bytes) == 0u;
        if(!uniform)
          dense = true;
        else if(l0 < SSD_GPU_MAX_PLATEAUS && ((amask >> l0) & 1u))
        {
          dense = true;
          if((wmask >> l0) & 1u)
          {
            const uint2 r = __ldg(frec + wbase + (e >> 4));
            if(r.x & SSD_WREC_ELIGIBLE)
            {
              // centre and half extents of the pixel box [x0, x0 + w] x [y0, y0 + h] in pixels, then in metres
              const float hw = 0.5f * (float)(((r.x >> 24) & 7u) + 1u), hh = 0.5f * (float)(((r.x >> 27) & 7u) + 1u);
              const float cx = fmaf((float)(r.x & 0xfffu) + hw, p.gs_xw, p.gs_x0);
              const float cy = fmaf(-((float)((r.x >> 12) & 0xfffu) + hh), p.gs_yw, p.gs_y0);
              const float eb = fmaxf(hw * p.gs_xw, hh * p.gs_yw) + p.gs_margin;
              const float4 ib = S.fast[l0].ibe;
              bool whole = fabsf(cx - ib.x) < ib.z - eb && fabsf(cy - ib.y) < ib.w - eb;
              if(!whole)
              {
                bool unc;
                const bool in = quadfilter_eval(S.qf[l0], cx, cy, eb + p.epsc, unc);
                whole = in && !unc;
              }
              if(whole)
              {
                dense = false;
                if(l0 != W.seg_l)
                {
                  if(W.seg_n)
                    seg_flush(S, W.seg_l, W.seg_sum, W.seg_n);
                  W.seg_l = l0;
                  W.seg_sum = 0;
                  W.seg_n = 0;
                }
                W.seg_sum += r.y & 0x1ffffffu;
                W.seg_n += r.y >> 25;
              }
            }
          }
        }
      }
      const unsigned b = __ballot_sync(0xffffffffu, dense);
      __syncwarp();
#ifdef SSD_WREC_DEBUG
      {
        // debug build: words taken whole / words sent to the dense pass, in the counters the stats call reports as n_bev_exact / n_quad_exact
        const unsigned bw = __ballot_sync(0xffffffffu, e != 0u && !dense);
        if(lane == 0)
        {
          atomicAdd(&F.n_def_bev, (unsigned)__popc(bw));
          atomicAdd(&F.n_def_quad, (unsigned)__popc(b));
        }
      }
#endif
      if(dense)
      {
        act[n2 + __popc(b & lt)] = (unsigned short)e;
        word_prefetch_l2(FR, wbase + (e >> 4));
      }
      n2 += __popc(b);
    }
    __syncwarp();
    if(n2)
      qr_dense<SRC>(p, FR, S, W, F, amask, ground, gbev, wbase, n2, warp, lane);
    __syncwarp();
  }
  qr_seg_combine(S, W, lane);
  qr_epilogue(S, W, F, ground, tid, lane);
}


// ---------------------------------------------------------------------------------------------
// k_riser_reduce: vertical faces from the remainder (include/ssd_gpu.h: ssd_gpu_riser; the reference only leaves
// "TODO use remainder to detect vertical faces", pointcloud.cpp:293). Optional fourth pass over the points, launched only
// when ssd_gpu_set_vertical_faces is on: the words that hold remainder labels are compacted like in the other passes, their
// vertices re-read, and every remainder point goes through the exact double-precision CameraToWorld (these are an eighth of
// the points and the footprint wants the exact coordinates): height index -> riser through a per-frame bin table, footprint
// as integer extremes and sums (order independent). Per-lane running segment, shared-memory accumulators per block, one set
// of global atomics per riser and block.
// ---------------------------------------------------------------------------------------------
struct RiserShared
{
  signed char riser_of_bin[SSD_BINS_PAD];
  unsigned cnt[SSD_GPU_MAX_PLATEAUS];
  int xmin[SSD_GPU_MAX_PLATEAUS], xmax[SSD_GPU_MAX_PLATEAUS], ymin[SSD_GPU_MAX_PLATEAUS], ymax[SSD_GPU_MAX_PLATEAUS];
  unsigned long long sx[SSD_GPU_MAX_PLATEAUS], sy[SSD_GPU_MAX_PLATEAUS];
  unsigned short act[SSD_PT_WARPS][SSD_WT_PX / 4];
};

struct RiserSeg
{
  int r;
  unsigned cnt;
  int xmin, xmax, ymin, ymax;
  unsigned long long sx, sy;
};

__device__ __forceinline__ void riser_flush(RiserShared &S, RiserSeg &g)
{
  if(g.cnt)
  {
    atomicAdd(&S.cnt[g.r], g.cnt);
    atomicAdd(&S.sx[g.r], g.sx);
    atomicAdd(&S.sy[g.r], g.sy);
    atomicMin(&S.xmin[g.r], g.xmin);
    atomicMax(&S.xmax[g.r], g.xmax);
    atomicMin(&S.ymin[g.r], g.ymin);
    atomicMax(&S.ymax[g.r], g.ymax);
  }
  g.cnt = 0;
  g.sx = g.sy = 0;
  g.xmin = g.ymin = 0x7fffffff;
  g.xmax = g.ymax = -1;
}

template<class SRC, class CAM = NoCam>
__global__ void __launch_bounds__(SSD_PT_THREADS) k_riser_reduce(const __grid_constant__ DevParams p0, const SRC src0,
                                                                 const unsigned char *__restrict__ labels, FrameDev *__restrict__ frames,
                                                                 const CAM cam = CAM())
{
  __shared__ RiserShared S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int frame = blockIdx.y;
  const DevParams &p = frame_params(p0, cam, frame);
  const auto &src = frame_src(src0, cam, p, frame);
  FrameDev &F = frames[frame];
  const int K = F.n_plateaus;
  if(K < 2)
    return;
  const size_t fbase = (size_t)frame * p.N;
  const unsigned *lab32 = reinterpret_cast<const unsigned *>(labels + fbase);
  const int nquads = p.N >> 2;
  int wt, wt_end, wt_stride;
  warp_tile_range((p.N + SSD_WT_PX - 1) / SSD_WT_PX, warp, wt, wt_end, wt_stride);
  {
    // bin -> riser: k where hmax[k] < bin < hmin[k + 1], else -1 (SSD_PT_THREADS == SSD_BINS_PAD: one bin per thread)
    int r = -1;
    for(int k = 0; k + 1 < K; k++)
      if(tid > F.plat[k].hmax && tid < F.plat[k + 1].hmin)
        r = k;
    S.riser_of_bin[tid] = (signed char)r;
    if(tid < SSD_GPU_MAX_PLATEAUS)
    {
      S.cnt[tid] = 0;
      S.sx[tid] = S.sy[tid] = 0;
      S.xmin[tid] = S.ymin[tid] = 0x7fffffff;
      S.xmax[tid] = S.ymax[tid] = -1;
    }
  }
  __syncthreads();
  unsigned short *act = S.act[warp];
  const typename SrcTraits<SRC>::Frame FR = src_frame(src, p, fbase);
  RiserSeg g;
  g.r = 0;
  g.cnt = 0;
  g.sx = g.sy = 0;
  g.xmin = g.ymin = 0x7fffffff;
  g.xmax = g.ymax = -1;

  for(; wt < wt_end; wt += wt_stride)
  {
    const unsigned wbase = (unsigned)wt * (SSD_WT_PX / 4);
    // ---- phase A: words with remainder labels ----
    unsigned n = 0;
#pragma unroll
    for(int it = 0; it < SSD_WT_WORDS; it++)
    {
      const int q = wt * (SSD_WT_PX / 4) + it * 32 + lane;
      const unsigned lw = q < nquads ? __ldg(lab32 + q) : 0xffffffffu;
      const unsigned x = lw ^ (SSD_LABEL_REMAINDER * 0x01010101u);                 // zero byte <=> remainder label
      const unsigned z = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;     // bit 7 of every zero byte (exact, no borrow)
      const unsigned am4 = ((z >> 7) * 0x10204080u) >> 28;
      if(__any_sync(0xffffffffu, am4 != 0u))
        n = compact_append(act, n, am4, it, lane);
    }
    if(n == 0)
      continue;
    __syncwarp();
    // ---- phase B: the remainder points of the compacted words ----
    for(unsigned s0 = 0; s0 < n; s0 += 32)
    {
      const unsigned i0 = s0 + lane;
      const unsigned e = i0 < n ? act[i0] : 0u;
      if(e)
      {
        typename SrcTraits<SRC>::Word w;
        word_load(FR, wbase + (e >> 4), w);
        float vx[4], vy[4], vz[4];
        word_unpack(FR, w, vx, vy, vz);
#pragma unroll
        for(int j = 0; j < 4; j++)
          if((e >> j) & 1u)
          {
            double wx, wy, wz;
            camera_to_world(p, vx[j], vy[j], vz[j], wx, wy, wz);
            const unsigned h = (unsigned)(unsigned short)((wz - p.z_min) * p.hir); // calcHeights (pointcloud.cpp:175)
            const int r = h < SSD_BINS_PAD ? (int)S.riser_of_bin[h] : -1;
            if(r >= 0)
            {
              const long long X = (long long)((wx - p.x_min) * 65536.0), Y = (long long)((wy - p.y_min) * 65536.0);
              if(r != g.r)
              {
                riser_flush(S, g);
                g.r = r;
              }
              g.cnt++;
              g.sx += (unsigned long long)X;
              g.sy += (unsigned long long)Y;
              g.xmin = min(g.xmin, (int)X);
              g.xmax = max(g.xmax, (int)X);
              g.ymin = min(g.ymin, (int)Y);
              g.ymax = max(g.ymax, (int)Y);
            }
          }
      }
    }
    __syncwarp();
  }
  riser_flush(S, g);
  __syncthreads();
  if(tid < SSD_GPU_MAX_PLATEAUS && S.cnt[tid])
  {
    RiserDev &R = F.ris[tid];
    atomicAdd(&R.cnt, S.cnt[tid]);
    atomicAdd(&R.sx, S.sx[tid]);
    atomicAdd(&R.sy, S.sy[tid]);
    atomicMin(&R.xmin, S.xmin[tid]);
    atomicMax(&R.xmax, S.xmax[tid]);
    atomicMin(&R.ymin, S.ymin[tid]);
    atomicMax(&R.ymax, S.ymax[tid]);
  }
}
