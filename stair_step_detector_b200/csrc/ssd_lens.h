// ssd_lens.h -- the lens primitives P and P^-1 of include/ssd_gpu.h (ssd_gpu_distortion): Brown-Conrady distortion of
// normalised image coordinates as rsutil.h's rs2_deproject_pixel_to_point / rs2_project_point_to_pixel evaluate it.
// __host__ __device__: the product's ray tables and overlay (device) and the synthetic scene's deprojection (host and device)
// share this one statement. Every operation is a single-rounded f32 operation in the order the header writes it: explicit
// __f*_rn on the device, plain operators on the host (built with -ffp-contract=off), so host and device agree bit for bit.
#ifndef SSD_LENS_H_
#define SSD_LENS_H_

#include "../../include/ssd_gpu.h"

#ifdef __CUDACC__
#define SSD_LENS_HD __host__ __device__ __forceinline__
#else
#define SSD_LENS_HD static inline
#endif

#ifdef __CUDA_ARCH__
#define SSD_LENS_ADD(a, b) __fadd_rn(a, b)
#define SSD_LENS_SUB(a, b) __fsub_rn(a, b)
#define SSD_LENS_MUL(a, b) __fmul_rn(a, b)
#define SSD_LENS_DIV(a, b) __fdiv_rn(a, b)
#else
#define SSD_LENS_ADD(a, b) ((a) + (b))
#define SSD_LENS_SUB(a, b) ((a) - (b))
#define SSD_LENS_MUL(a, b) ((a) * (b))
#define SSD_LENS_DIV(a, b) ((a) / (b))
#endif

// the lens changes nothing: no model, or a Brown-Conrady model whose coefficients are all zero
SSD_LENS_HD int ssd_lens_is_pinhole(const ssd_gpu_distortion *d)
{
  if(!d || d->model == SSD_DISTORTION_NONE)
    return 1;
  for(int i = 0; i < 5; i++)
    if(d->coeffs[i] != 0.f)
      return 0;
  return 1;
}

// P(x, y): r2 = x*x + y*y, f = 1 + k1*r2 + k2*r2*r2 + k3*r2*r2*r2, x' = x*f + 2*p1*x*y + p2*(r2 + 2*x*x), y' likewise
SSD_LENS_HD void ssd_lens_P(const float k[5], float x, float y, float *xo, float *yo)
{
  const float r2 = SSD_LENS_ADD(SSD_LENS_MUL(x, x), SSD_LENS_MUL(y, y));
  const float f = SSD_LENS_ADD(SSD_LENS_ADD(SSD_LENS_ADD(1.f, SSD_LENS_MUL(k[0], r2)), SSD_LENS_MUL(SSD_LENS_MUL(k[1], r2), r2)),
                               SSD_LENS_MUL(SSD_LENS_MUL(SSD_LENS_MUL(k[4], r2), r2), r2));
  *xo = SSD_LENS_ADD(SSD_LENS_ADD(SSD_LENS_MUL(x, f), SSD_LENS_MUL(SSD_LENS_MUL(SSD_LENS_MUL(2.f, k[2]), x), y)),
                     SSD_LENS_MUL(k[3], SSD_LENS_ADD(r2, SSD_LENS_MUL(SSD_LENS_MUL(2.f, x), x))));
  *yo = SSD_LENS_ADD(SSD_LENS_ADD(SSD_LENS_MUL(y, f), SSD_LENS_MUL(SSD_LENS_MUL(SSD_LENS_MUL(2.f, k[3]), x), y)),
                     SSD_LENS_MUL(k[2], SSD_LENS_ADD(r2, SSD_LENS_MUL(SSD_LENS_MUL(2.f, y), y))));
}

// P^-1(x0, y0): exactly 10 fixed-point iterations from (x0, y0)
SSD_LENS_HD void ssd_lens_Pinv(const float k[5], float x0, float y0, float *xo, float *yo)
{
  float x = x0, y = y0;
  for(int i = 0; i < 10; i++)
  {
    const float r2 = SSD_LENS_ADD(SSD_LENS_MUL(x, x), SSD_LENS_MUL(y, y));
    const float icd = SSD_LENS_DIV(1.f, SSD_LENS_ADD(1.f, SSD_LENS_MUL(SSD_LENS_ADD(SSD_LENS_MUL(SSD_LENS_ADD(SSD_LENS_MUL(k[4], r2), k[1]), r2), k[0]), r2)));
    const float dx = SSD_LENS_ADD(SSD_LENS_MUL(SSD_LENS_MUL(SSD_LENS_MUL(2.f, k[2]), x), y), SSD_LENS_MUL(k[3], SSD_LENS_ADD(r2, SSD_LENS_MUL(SSD_LENS_MUL(2.f, x), x))));
    const float dy = SSD_LENS_ADD(SSD_LENS_MUL(SSD_LENS_MUL(SSD_LENS_MUL(2.f, k[3]), x), y), SSD_LENS_MUL(k[2], SSD_LENS_ADD(r2, SSD_LENS_MUL(SSD_LENS_MUL(2.f, y), y))));
    x = SSD_LENS_MUL(SSD_LENS_SUB(x0, dx), icd);
    y = SSD_LENS_MUL(SSD_LENS_SUB(y0, dy), icd);
  }
  *xo = x;
  *yo = y;
}

// deprojection: (x0, y0) = ((u - ppx)/fx, (v - ppy)/fy) -> the ray (x, y) with z = 1
SSD_LENS_HD void ssd_lens_deproject(const ssd_gpu_distortion *d, float x0, float y0, float *x, float *y)
{
  if(ssd_lens_is_pinhole(d))
    *x = x0, *y = y0;
  else if(d->model == SSD_DISTORTION_INVERSE_BROWN_CONRADY)
    ssd_lens_P(d->coeffs, x0, y0, x, y);
  else
    ssd_lens_Pinv(d->coeffs, x0, y0, x, y);
}

// overlay projection: (X/Z, Y/Z) -> the normalised image point
SSD_LENS_HD void ssd_lens_project(const ssd_gpu_distortion *d, float x0, float y0, float *x, float *y)
{
  if(ssd_lens_is_pinhole(d))
    *x = x0, *y = y0;
  else if(d->model == SSD_DISTORTION_INVERSE_BROWN_CONRADY)
    ssd_lens_Pinv(d->coeffs, x0, y0, x, y);
  else
    ssd_lens_P(d->coeffs, x0, y0, x, y);
}

#endif // SSD_LENS_H_
