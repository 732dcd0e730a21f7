// scene_model.h -- synthetic L515-style input source (stands in for the stubbed RealSense capture,
// reference camera.cpp:27-50 and rs2::pointcloud::calculate at pointcloud.cpp:138).
//
// A scene is a solid straight flight of stairs on a ground plane, seen by a pin-hole depth camera. The
// generator ray-casts a z16 depth image (depth_unit metres per count, like the L515's 0.25 mm), and the
// deprojection turns it into the packed {x,y,z} float vertices the hot path consumes. Every function is
// __host__ __device__ so the same model runs on the host (tests) and in a CUDA kernel (bench).
//
// Deprojection uses only single IEEE f32 operations in a fixed order (no contraction), so host, device
// and numpy produce identical vertices from the same depth image.
#ifndef SSD_SCENE_MODEL_H_
#define SSD_SCENE_MODEL_H_

#include "../../../include/ssd_scene.h"
#include "../ssd_lens.h"
#include <math.h>

#ifdef __CUDACC__
#define SSD_HD __host__ __device__ __forceinline__
#else
#define SSD_HD static inline
#endif

#define SSD_SCENE_MAX_STEPS 16
#define SSD_SCENE_MAX_BOXES 4

struct ssd_scene_rt
{
  // camera pose in scene coordinates: origin + axes (columns of R)
  float ox, oy, oz;
  float xc[3], yc[3], zc[3];
  int n_holes;
  int hole[SSD_SCENE_MAX_BOXES][4]; // u0,v0,u1,v1
  int n_boxes;
  float box[SSD_SCENE_MAX_BOXES][6]; // xmin,xmax,ymin,ymax,zmin,zmax
};

SSD_HD uint64_t ssd_mix64(uint64_t z)
{
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// uniform in [0,1) from a 64-bit hash
SSD_HD float ssd_u01(uint64_t h)
{
  return (float)(h >> 40) * (1.0f / 16777216.0f);
}

struct ssd_rng
{
  uint64_t s;
};
SSD_HD float ssd_rng_next(ssd_rng *r)
{
  r->s = ssd_mix64(r->s);
  return ssd_u01(r->s);
}
SSD_HD float ssd_rng_range(ssd_rng *r, float lo, float hi)
{
  return lo + (hi - lo) * ssd_rng_next(r);
}

SSD_HD void ssd_scene_default_hd(ssd_scene *s, int32_t width, int32_t height)
{
  s->width = width;
  s->height = height;
  // L515 depth FOV 70 x 55 degrees (SURVEY.md 8(d) config 1)
  s->fx = (float)(width / (2.0 * 0.70020753820970971)); // tan(35 deg)
  s->fy = (float)(height / (2.0 * 0.52056705055174624)); // tan(27.5 deg)
  s->ppx = width * 0.5f;
  s->ppy = height * 0.5f;
  s->depth_unit = 0.00025f;
  s->cam_height = 1.25f;
  s->cam_pitch_deg = 50.f;
  s->cam_roll_deg = 0.f;
  s->cam_yaw_deg = 0.f;
  s->cam_x = 0.f;
  s->cam_y = 0.f;
  s->ground_z = 0.004f;
  s->n_steps = 3;
  s->riser = 0.173f;
  s->tread = 0.28f;
  s->width_m = 0.9f;
  s->first_riser_y = 0.45f;
  s->x_center = 0.f;
  s->top_landing = 0.f;
  s->noise_sigma = 0.f;
  s->dropout = 0.f;
  s->n_holes = 0;
  s->n_occluders = 0;
  s->rotate180 = 0;
  s->randomize_camera = 0;
  s->seed = 12345;
  s->distortion_model = SSD_DISTORTION_NONE;
  for(int i = 0; i < 5; i++)
    s->coeffs[i] = 0.f;
}

SSD_HD ssd_gpu_distortion ssd_scene_lens(const ssd_scene *s)
{
  ssd_gpu_distortion d;
  d.model = s->distortion_model;
  for(int i = 0; i < 5; i++)
    d.coeffs[i] = s->coeffs[i];
  return d;
}

// frame `index` of a batch: geometry drawn from the distributions of SURVEY.md 8(d) config 3
SSD_HD void ssd_scene_randomize_hd(ssd_scene *s, const ssd_scene *base, uint64_t base_seed, int64_t index, int min_steps, int max_steps)
{
  *s = *base;
  ssd_rng r;
  r.s = ssd_mix64(base_seed ^ ssd_mix64((uint64_t)index + 0x5851F42D4C957F2Dull));
  int span = max_steps - min_steps + 1;
  if(span < 1)
    span = 1;
  int n = min_steps + (int)(ssd_rng_next(&r) * span);
  if(n > max_steps)
    n = max_steps;
  if(n > SSD_SCENE_MAX_STEPS)
    n = SSD_SCENE_MAX_STEPS;
  s->n_steps = n;
  s->riser = ssd_rng_range(&r, 0.12f, 0.20f);
  s->tread = ssd_rng_range(&r, 0.25f, 0.32f);
  s->width_m = ssd_rng_range(&r, 0.7f, 1.1f);
  s->x_center = base->x_center + ssd_rng_range(&r, -0.05f, 0.05f);
  // a context binds ONE calibration (one camera mounting): the pose only varies when asked to
  const float dp = ssd_rng_range(&r, -5.f, 5.f), dh = ssd_rng_range(&r, -0.15f, 0.15f), dy = ssd_rng_range(&r, -2.f, 2.f),
              dr = ssd_rng_range(&r, -1.5f, 1.5f);
  if(base->randomize_camera)
  {
    s->cam_pitch_deg = base->cam_pitch_deg + dp;
    s->cam_height = base->cam_height + dh;
    s->cam_yaw_deg = base->cam_yaw_deg + dy;
    s->cam_roll_deg = base->cam_roll_deg + dr;
  }
  // the flight itself is yawed / shifted instead (same relative geometry as a yawed camera)
  s->x_center += 0.f;
  s->first_riser_y = base->first_riser_y + ssd_rng_range(&r, -0.05f, 0.08f);
  s->seed = ssd_mix64(r.s);
}

SSD_HD void ssd_scene_prepare(const ssd_scene *s, ssd_scene_rt *rt)
{
  const float d2r = 0.017453292519943295f;
  const float th = s->cam_pitch_deg * d2r;
  const float ro = (s->cam_roll_deg + (s->rotate180 ? 180.f : 0.f)) * d2r;
  const float ya = s->cam_yaw_deg * d2r;
  const float st = sinf(th), ct = cosf(th), sr = sinf(ro), cr = cosf(ro), sy = sinf(ya), cy = cosf(ya);
  // zero roll/yaw: x_c=(1,0,0), optical z_c=(0,ct,-st), image-down y_c=(0,-st,-ct)
  const float x0[3] = { 1.f, 0.f, 0.f }, y0[3] = { 0.f, -st, -ct }, z0[3] = { 0.f, ct, -st };
  float xr[3], yr[3];
  for(int i = 0; i < 3; i++)
  {
    xr[i] = cr * x0[i] + sr * y0[i];
    yr[i] = -sr * x0[i] + cr * y0[i];
  }
  // yaw about scene Z
  const float *src[3] = { xr, yr, z0 };
  float *dst[3] = { rt->xc, rt->yc, rt->zc };
  for(int a = 0; a < 3; a++)
  {
    dst[a][0] = cy * src[a][0] - sy * src[a][1];
    dst[a][1] = sy * src[a][0] + cy * src[a][1];
    dst[a][2] = src[a][2];
  }
  rt->ox = s->cam_x;
  rt->oy = s->cam_y;
  rt->oz = s->cam_height;

  ssd_rng r;
  r.s = ssd_mix64(s->seed ^ 0xA5A5A5A55A5A5A5Aull);
  rt->n_holes = s->n_holes > SSD_SCENE_MAX_BOXES ? SSD_SCENE_MAX_BOXES : s->n_holes;
  for(int h = 0; h < rt->n_holes; h++)
  {
    const int hw = (int)(s->width * ssd_rng_range(&r, 0.02f, 0.06f));
    const int hh = (int)(s->height * ssd_rng_range(&r, 0.02f, 0.06f));
    const int u0 = (int)(ssd_rng_next(&r) * (s->width - hw));
    const int v0 = (int)(ssd_rng_next(&r) * (s->height - hh));
    rt->hole[h][0] = u0;
    rt->hole[h][1] = v0;
    rt->hole[h][2] = u0 + hw;
    rt->hole[h][3] = v0 + hh;
  }
  rt->n_boxes = s->n_occluders > SSD_SCENE_MAX_BOXES ? SSD_SCENE_MAX_BOXES : s->n_occluders;
  for(int b = 0; b < rt->n_boxes; b++)
  {
    // boxes floating above the measuring range (z > 1.1): their own points are out of range, their
    // shadows remove 10-40 % of one or two treads
    const float bw = ssd_rng_range(&r, 0.10f, 0.30f), bd = ssd_rng_range(&r, 0.06f, 0.16f);
    const float cx = s->x_center + ssd_rng_range(&r, -0.3f, 0.3f);
    const float cyy = s->first_riser_y + ssd_rng_range(&r, 0.0f, 0.5f);
    const float zc = s->cam_height - ssd_rng_range(&r, 0.08f, 0.12f);
    rt->box[b][0] = cx - bw * 0.5f;
    rt->box[b][1] = cx + bw * 0.5f;
    rt->box[b][2] = cyy - bd * 0.5f;
    rt->box[b][3] = cyy + bd * 0.5f;
    rt->box[b][4] = zc - 0.02f;
    rt->box[b][5] = zc;
  }
}

// camera coordinates of a scene point (for calibration marks)
SSD_HD void ssd_scene_to_camera(const ssd_scene_rt *rt, const double p[3], double c[3])
{
  const double d[3] = { p[0] - rt->ox, p[1] - rt->oy, p[2] - rt->oz };
  c[0] = d[0] * rt->xc[0] + d[1] * rt->xc[1] + d[2] * rt->xc[2];
  c[1] = d[0] * rt->yc[0] + d[1] * rt->yc[1] + d[2] * rt->yc[2];
  c[2] = d[0] * rt->zc[0] + d[1] * rt->zc[1] + d[2] * rt->zc[2];
}

// z16 depth count of pixel (u,v)
SSD_HD uint16_t ssd_scene_depth(const ssd_scene *s, const ssd_scene_rt *rt, int u, int v)
{
  for(int h = 0; h < rt->n_holes; h++)
    if(u >= rt->hole[h][0] && u < rt->hole[h][2] && v >= rt->hole[h][1] && v < rt->hole[h][3])
      return 0;

  const uint64_t ph = ssd_mix64(s->seed ^ ssd_mix64((uint64_t)v * (uint64_t)s->width + (uint64_t)u));
  if(s->dropout > 0.f && ssd_u01(ph) < s->dropout)
    return 0;

  float dx = ((float)u - s->ppx) / s->fx, dy = ((float)v - s->ppy) / s->fy;
  const ssd_gpu_distortion lens = ssd_scene_lens(s);
  ssd_lens_deproject(&lens, dx, dy, &dx, &dy); // the ray of pixel (u, v) at z = 1 (the identity for the pin-hole)
  const float D[3] = { dx * rt->xc[0] + dy * rt->yc[0] + rt->zc[0], dx * rt->xc[1] + dy * rt->yc[1] + rt->zc[1],
                       dx * rt->xc[2] + dy * rt->yc[2] + rt->zc[2] };
  const float O[3] = { rt->ox, rt->oy, rt->oz };
  const float big = 1e30f;
  float tbest = big;

  const float xl = s->x_center - 0.5f * s->width_m, xr = s->x_center + 0.5f * s->width_m;
  const float g = s->ground_z;
  const int n = s->n_steps;
  const float y0 = s->first_riser_y;
  const float yend = y0 + n * s->tread + s->top_landing;
  const float eps = 1e-6f;

  // ground
  if(D[2] < 0.f)
  {
    const float t = (g - O[2]) / D[2];
    if(t > 0.f && t < tbest)
      tbest = t;
  }
  for(int i = 1; i <= n; i++)
  {
    const float zi = g + i * s->riser, zim = g + (i - 1) * s->riser;
    const float ya = y0 + (i - 1) * s->tread;
    const float yb = (i == n) ? yend : y0 + i * s->tread;
    // tread top
    if(D[2] != 0.f)
    {
      const float t = (zi - O[2]) / D[2];
      if(t > 0.f && t < tbest)
      {
        const float x = O[0] + t * D[0], y = O[1] + t * D[1];
        if(x >= xl && x <= xr && y >= ya && y <= yb)
          tbest = t;
      }
    }
    // riser
    if(D[1] != 0.f)
    {
      const float t = (ya - O[1]) / D[1];
      if(t > 0.f && t < tbest)
      {
        const float x = O[0] + t * D[0], z = O[2] + t * D[2];
        if(x >= xl && x <= xr && z >= zim - eps && z <= zi + eps)
          tbest = t;
      }
    }
    // side faces of the solid under tread i
    if(D[0] != 0.f)
    {
      for(int sgn = 0; sgn < 2; sgn++)
      {
        const float xs = sgn ? xr : xl;
        const float t = (xs - O[0]) / D[0];
        if(t > 0.f && t < tbest)
        {
          const float y = O[1] + t * D[1], z = O[2] + t * D[2];
          if(y >= ya && y <= yb && z >= g && z <= zi)
            tbest = t;
        }
      }
    }
  }
  // back face
  if(n > 0 && D[1] != 0.f)
  {
    const float t = (yend - O[1]) / D[1];
    if(t > 0.f && t < tbest)
    {
      const float x = O[0] + t * D[0], z = O[2] + t * D[2];
      if(x >= xl && x <= xr && z >= g && z <= g + n * s->riser)
        tbest = t;
    }
  }
  // occluder boxes (slab test)
  for(int b = 0; b < rt->n_boxes; b++)
  {
    float t0 = 0.f, t1 = big;
    bool ok = true;
    for(int a = 0; a < 3 && ok; a++)
    {
      const float lo = rt->box[b][2 * a], hi = rt->box[b][2 * a + 1];
      if(D[a] == 0.f)
      {
        ok = O[a] >= lo && O[a] <= hi;
        continue;
      }
      float ta = (lo - O[a]) / D[a], tb = (hi - O[a]) / D[a];
      if(ta > tb)
      {
        const float tmp = ta;
        ta = tb;
        tb = tmp;
      }
      t0 = ta > t0 ? ta : t0;
      t1 = tb < t1 ? tb : t1;
      ok = t0 <= t1;
    }
    if(ok && t0 > 0.f && t0 < tbest)
      tbest = t0;
  }
  if(tbest >= big)
    return 0;

  // camera depth z_c = t (d_c.z == 1); noise along the ray
  float zc = tbest;
  if(s->noise_sigma > 0.f)
  {
    const uint64_t h1 = ssd_mix64(ph), h2 = ssd_mix64(h1);
    const float u1 = ssd_u01(h1) + (1.0f / 33554432.0f), u2 = ssd_u01(h2);
    const float nrm = sqrtf(-2.f * logf(u1)) * cosf(6.2831853071795864f * u2);
    const float len = sqrtf(dx * dx + dy * dy + 1.f);
    zc += s->noise_sigma * nrm / len;
  }
  const float counts = zc / s->depth_unit + 0.5f;
  if(!(counts >= 1.f) || counts >= 65535.f)
    return 0;
  return (uint16_t)counts;
}

// z16 count -> vertex; single-rounded f32 operations in this order (the stubbed SDK deprojection), the scene's lens applied to
// the normalised coordinates (include/ssd_gpu.h, ssd_gpu_distortion)
SSD_HD void ssd_deproject_pixel(const ssd_scene *s, int u, int v, uint16_t d, float out[3])
{
  const ssd_gpu_distortion lens = ssd_scene_lens(s);
#ifdef __CUDA_ARCH__
  float xn = __fdiv_rn(__fsub_rn((float)u, s->ppx), s->fx);
  float yn = __fdiv_rn(__fsub_rn((float)v, s->ppy), s->fy);
  ssd_lens_deproject(&lens, xn, yn, &xn, &yn);
  const float z = __fmul_rn((float)d, s->depth_unit);
  out[0] = __fmul_rn(z, xn);
  out[1] = __fmul_rn(z, yn);
  out[2] = z;
#else
  float xn = ((float)u - s->ppx) / s->fx;
  float yn = ((float)v - s->ppy) / s->fy;
  ssd_lens_deproject(&lens, xn, yn, &xn, &yn);
  const float z = (float)d * s->depth_unit;
  out[0] = z * xn;
  out[1] = z * yn;
  out[2] = z;
#endif
}

#endif // SSD_SCENE_MODEL_H_
