/*
 * oracle_step_surfaces.c -- TEST INFRASTRUCTURE. CPU restatement of step surfaces (include/ssd_gpu.h, ssd_gpu_set_step_surfaces):
 * the least-squares plane, tilt, flatness and z extent of the points each step's height averages (the pixels its step labels
 * mark). The reference discards that point set after calcAverageZ (pointcloud.cpp:574-581), so this restates the library's
 * DEFINITION: moments in exact integers (fixed point of the exact double world point), the plane and the external-world fields in
 * double in the stated order. It compiles the single-frame oracle (oracle/ssd_oracle.c) into the same translation unit, for its
 * CameraToWorld and for the chain that builds the step labels it is fed. It takes the points and a step map, so one function
 * serves single frames (n_members = 1) and groups.
 * Build: gcc -std=c11 -O2 -ffp-contract=off -fPIC -shared (the flags of oracle/Makefile) -o libssd_oracle_surfaces.so
 *        oracle_step_surfaces.c -lm
 */
#include "../../oracle/ssd_oracle.c"

#include <limits.h>

/* n_members frames back to back in xyz (W*H*3 floats each) with their step labels (n_members*W*H), member m through xfs[m];
 * ext_xf: the transform whose ToExternalWorld the steps are reported in. out: n_steps records. */
int ssd_oracle_step_surfaces(const ssd_gpu_config *cfg, int n_members, const ssd_gpu_transform *xfs, const float *xyz, const uint8_t *step_labels,
                             int n_steps, const ssd_gpu_transform *ext_xf, ssd_gpu_step_surface *out)
{
  if(n_members < 1 || n_steps < 0 || n_steps > SSD_GPU_MAX_STEPS)
    return SSD_E_INVALID_ARG;
  typedef __int128 i128;
  i128 n[SSD_GPU_MAX_STEPS], sx[SSD_GPU_MAX_STEPS], sy[SSD_GPU_MAX_STEPS], sz[SSD_GPU_MAX_STEPS], sxx[SSD_GPU_MAX_STEPS],
    sxy[SSD_GPU_MAX_STEPS], syy[SSD_GPU_MAX_STEPS], sxz[SSD_GPU_MAX_STEPS], syz[SSD_GPU_MAX_STEPS], szz[SSD_GPU_MAX_STEPS];
  long long zmin[SSD_GPU_MAX_STEPS], zmax[SSD_GPU_MAX_STEPS];
  for(int s = 0; s < SSD_GPU_MAX_STEPS; s++)
  {
    n[s] = sx[s] = sy[s] = sz[s] = sxx[s] = sxy[s] = syy[s] = sxz[s] = syz[s] = szz[s] = 0;
    zmin[s] = LLONG_MAX;
    zmax[s] = LLONG_MIN;
  }
  const size_t N = (size_t)cfg->width * cfg->height;
  for(size_t i = 0; i < N * (size_t)n_members; i++)
  {
    const int s = step_labels[i];
    if(s >= n_steps)
      continue;
    double w[3];
    camera_to_world(&xfs[i / N], xyz + i * 3, w);
    const long long X = (long long)((w[0] - cfg->x_min) * 65536.0), Y = (long long)((w[1] - cfg->y_min) * 65536.0),
                    Z = (long long)((w[2] - cfg->z_min) * 65536.0);
    n[s]++;
    sx[s] += X;
    sy[s] += Y;
    sz[s] += Z;
    sxx[s] += (i128)X * X;
    sxy[s] += (i128)X * Y;
    syy[s] += (i128)Y * Y;
    sxz[s] += (i128)X * Z;
    syz[s] += (i128)Y * Z;
    szz[s] += (i128)Z * Z;
    if(Z < zmin[s]) zmin[s] = Z;
    if(Z > zmax[s]) zmax[s] = Z;
  }
  const ssd_gpu_transform *e = ext_xf;
  for(int s = 0; s < n_steps; s++)
  {
    ssd_gpu_step_surface o;
    memset(&o, 0, sizeof o);
    if(n[s] > 0)
    {
      const double cxx = (double)(n[s] * sxx[s] - sx[s] * sx[s]), cxy = (double)(n[s] * sxy[s] - sx[s] * sy[s]),
                   cyy = (double)(n[s] * syy[s] - sy[s] * sy[s]), cxz = (double)(n[s] * sxz[s] - sx[s] * sz[s]),
                   cyz = (double)(n[s] * syz[s] - sy[s] * sz[s]), czz = (double)(n[s] * szz[s] - sz[s] * sz[s]);
      const double det = cxx * cyy - cxy * cxy, dn = (double)n[s];
      double a = 0, b = 0;
      o.n_points = (uint32_t)n[s];
      o.fit_valid = n[s] >= 3 && det > 0;
      if(o.fit_valid)
      {
        a = (cxz * cyy - cyz * cxy) / det;
        b = (cyz * cxx - cxz * cxy) / det;
        const double r = czz - a * cxz - b * cyz;
        o.rms_dz = sqrt(r > 0 ? r : 0.0) / dn / 65536.0;
        o.tilt_deg = atan(sqrt(a * a + b * b)) * (180.0 / 3.14159265358979323846); /* M_PI, which strict C11 does not declare */
      }
      const double xm = cfg->x_min + (double)sx[s] / dn / 65536.0, ym = cfg->y_min + (double)sy[s] / dn / 65536.0,
                   zm = cfg->z_min + (double)sz[s] / dn / 65536.0;
      o.centroid[0] = (e->ext_a[0] * xm + e->ext_a[1] * ym) + e->ext_b[0];
      o.centroid[1] = (e->ext_a[2] * xm + e->ext_a[3] * ym) + e->ext_b[1];
      o.centroid[2] = e->ext_z + zm;
      o.gradient[0] = e->ext_a[0] * a + e->ext_a[1] * b;
      o.gradient[1] = e->ext_a[2] * a + e->ext_a[3] * b;
      o.z_lo = e->ext_z + (cfg->z_min + (double)zmin[s] / 65536.0);
      o.z_hi = e->ext_z + (cfg->z_min + (double)zmax[s] / 65536.0);
    }
    out[s] = o;
  }
  return SSD_OK;
}
