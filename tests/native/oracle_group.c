/*
 * oracle_group.c -- TEST INFRASTRUCTURE. CPU restatement of frame groups (include/ssd_gpu.h, ssd_gpu_process_groups_*): the
 * reference's Pointcloud::process chain run once on the union of the world points of several frames, each member through its own
 * CameraToWorld. It compiles the single-frame oracle (oracle/ssd_oracle.c) into the same translation unit and reuses its chain;
 * ssd_oracle_process_group is ssd_oracle_process with the extraction loop taken over the members' frames, so a group of one frame
 * is ssd_oracle_process bit for bit. ssd_oracle_last_overlay then projects the last group's steps for any member's camera.
 * Build: gcc -std=c11 -O2 -ffp-contract=off -fPIC -shared (the flags of oracle/Makefile) -o libssd_oracle_group.so oracle_group.c -lm
 */
#include "../../oracle/ssd_oracle.c"

/* n_members frames back to back in xyz (W*H*3 floats each), member m with transform xfs[m]. labels: n_members*W*H (may be NULL);
 * the rest as ssd_oracle_process. */
int ssd_oracle_process_group(const ssd_gpu_config *cfg, const ssd_gpu_transform *xfs, const float *xyz, int n_members, uint8_t *labels,
                             uint32_t *hist_out, int hist_cap, ssd_gpu_frame_info *info, ssd_gpu_plateau *plats, ssd_gpu_step *steps)
{
  if(n_members < 1)
    return SSD_E_INVALID_ARG;
  const ssd_gpu_transform *xf = &xfs[0]; /* ToExternalWorld of the first member */
  Frame f;
  memset(&f, 0, sizeof(f));
  f.cfg = cfg;
  int rc = ssd_oracle_derive(cfg, &f.d);
  if(rc)
    return rc;
  const int W = cfg->width, H = cfg->height;
  const size_t N = (size_t)W * H * (size_t)n_members; /* the union of the members' points; pixel i of member m is m * W * H + i */
  memset(info, 0, sizeof(*info));
  info->ground_index = info->first_valid_index = -1;
  info->n_bins = f.d.n_bins;

  f.world = (double *)malloc(sizeof(double) * 3 * N);
  f.pixel = (uint32_t *)malloc(sizeof(uint32_t) * N);
  f.height = (uint16_t *)malloc(sizeof(uint16_t) * N);
  uint32_t *cur = (uint32_t *)malloc(sizeof(uint32_t) * N);   /* pointsHt (indices into f.world) */
  uint32_t *upper = (uint32_t *)malloc(sizeof(uint32_t) * N);
  uint32_t *store = (uint32_t *)malloc(sizeof(uint32_t) * N); /* plateau point lists, concatenated */
  uint32_t *sel = (uint32_t *)malloc(sizeof(uint32_t) * N);
  uint8_t *img = (uint8_t *)malloc(N);
  if(!f.world || !f.pixel || !f.height || !cur || !upper || !store || !sel || !img)
  {
    rc = SSD_E_NOMEM;
    goto done;
  }

  /* PointsExtraction::extract (pointcloud.cpp:122-178): z>0, transform, range, height index */
  uint32_t n = 0, nNonZero = 0;
  for(size_t i = 0; i < N; i++)
  {
    const float *v = xyz + i * 3;
    if(!(v[2] > 0))
    {
      if(labels)
        labels[i] = SSD_LABEL_INVALID;
      continue;
    }
    nNonZero++;
    double w[3];
    camera_to_world(&xfs[i / ((size_t)W * H)], v, w);
    const int in = w[0] > cfg->x_min && w[0] < cfg->x_max && w[1] > cfg->y_min && w[1] < cfg->y_max && w[2] > cfg->z_min &&
                   w[2] < cfg->z_max;
    if(labels)
      labels[i] = in ? SSD_LABEL_REMAINDER : SSD_LABEL_OUT_OF_RANGE;
    if(!in)
      continue;
    f.world[(size_t)n * 3] = w[0];
    f.world[(size_t)n * 3 + 1] = w[1];
    f.world[(size_t)n * 3 + 2] = w[2];
    f.pixel[n] = (uint32_t)i;
    f.height[n] = (uint16_t)((w[2] - cfg->z_min) * f.d.height_interval_reciprocal); /* :175 */
    n++;
  }
  f.n_points = n;
  info->n_nonzero = nNonZero;
  info->n_in_range = n;

  /* HeightsHistogram::calcHist (:194-204) */
  uint32_t hist[SSD_GPU_MAX_BINS + 2];
  memset(hist, 0, sizeof(hist));
  for(uint32_t i = 0; i < n; i++)
    ++hist[f.height[i]];
  if(hist_out)
    for(int i = 0; i < hist_cap && i < f.d.n_bins; i++)
      hist_out[i] = hist[i];

  /* findPeaks (:214-241) + filterPeaks (:243-256) */
  uint16_t peaks[SSD_GPU_MAX_BINS];
  int nPeaks = 0;
  {
    const size_t last = (size_t)f.d.n_bins - 1;
    int ascending = 0;
    for(uint16_t i = 0; i < last; i++)
    {
      const uint32_t c = hist[i], s = hist[i + 1];
      if(c < s)
      {
        ascending = 1;
        continue;
      }
      if(c > s)
      {
        if(ascending)
        {
          const uint32_t np = hist[i];
          if(!(np < cfg->min_peak_points) && (uint32_t)((np * 2 - hist[i - 1] - hist[i + 1]) * 2) > np)
            peaks[nPeaks++] = i;
        }
        ascending = 0;
      }
    }
  }
  if(nPeaks > SSD_GPU_MAX_PLATEAUS)
  {
    info->status |= SSD_STATUS_TOO_MANY_PLATEAUS;
    nPeaks = SSD_GPU_MAX_PLATEAUS;
  }
  info->n_plateaus = nPeaks;

  /* PlateausExtraction::extractPlateaus (:280-343), literally: two stable splits per peak */
  uint32_t nCur = n;
  for(uint32_t i = 0; i < n; i++)
    cur[i] = i;
  uint32_t *pStart[SSD_GPU_MAX_PLATEAUS];
  uint32_t pCount[SSD_GPU_MAX_PLATEAUS];
  uint32_t stored = 0;
  for(int k = 0; k < nPeaks; k++)
  {
    const uint16_t h = peaks[k];
    const uint16_t pred = (uint16_t)(h - 1), succ = (uint16_t)(h + 1);
    uint16_t hmin, hmax;
    if(hist[pred] > hist[succ])
    {
      hmin = pred;
      hmax = h;
    }
    else
    {
      hmin = h;
      hmax = succ;
    }
    const uint16_t thr = (uint16_t)(hmin - 1); /* wraps to 65535 when hmin == 0 (:324,337) */
    if(hmin == 0)
      info->status |= SSD_STATUS_HMIN_WRAP;
    uint32_t nUpper = 0;
    for(uint32_t i = 0; i < nCur; i++)
      if(thr < f.height[cur[i]])
        upper[nUpper++] = cur[i];
    pStart[k] = store + stored;
    uint32_t np = 0;
    nCur = 0;
    for(uint32_t i = 0; i < nUpper; i++)
    {
      if(hmax < f.height[upper[i]])
        cur[nCur++] = upper[i];
      else
        pStart[k][np++] = upper[i];
    }
    pCount[k] = np;
    stored += np;
    ssd_gpu_plateau *o = &plats[k];
    memset(o, 0, sizeof(*o));
    o->height = h;
    o->hmin = hmin;
    o->hmax = hmax;
    o->n_points = np;
    o->quad_status = -1;
    if(labels)
      for(uint32_t i = 0; i < np; i++)
        labels[f.pixel[pStart[k][i]]] = (uint8_t)k;
  }

  /* StairsDetector::detectStairSteps (:399-456) */
  P2 quadW[SSD_GPU_MAX_PLATEAUS][4];
  memset(quadW, 0, sizeof(quadW));
  int groundInd = -1, firstValid = -1;
  {
    size_t maxGround = 0;
    int i = 0;
    for(; i < nPeaks; i++)
    {
      if(plats[i].height >= f.d.min_height)
        break;
      if(maxGround < pCount[i])
      {
        maxGround = pCount[i];
        groundInd = i;
      }
    }
    for(; i < nPeaks; i++)
    {
      if(project_to_binary_image(&f, pStart[i], pCount[i], img))
        info->status |= SSD_STATUS_BEV_OOB;
      ssd_oracle_close(img, W, H);
      P2 qpx[4];
      int valid;
      detect_outline_closed(img, W, H, f.d.min_img_y_extent, f.d.xy_ratio, qpx, &valid);
      for(int c = 0; c < 4; c++)
        quadW[i][c] = image_to_world(&f, qpx[c]); /* imgPointsToWorld :476-487 */
      plats[i].valid = valid;
      plats[i].outlined = 1;
      if(valid && firstValid < 0)
        firstValid = i;
    }
  }
  info->ground_index = groundInd;
  info->first_valid_index = firstValid;

  typedef struct { double x, y, z; } P3;
  P3 stepQuads[SSD_GPU_MAX_STEPS][4];
  int nSteps = 0;
  if(firstValid >= 0)
  {
    if(groundInd >= 0)
    {
      /* ground (:436-443) + calcGround (:528-547) */
      calc_ground_quadrilateral(&f, quadW[firstValid], quadW[groundInd]);
      plats[groundInd].valid = 1;
      const P2 *gq = quadW[groundInd];
      uint32_t nSel;
      double mean;
      const int st = points_in_quad_mean(&f, pStart[groundInd], pCount[groundInd], gq, sel, &nSel, &mean);
      plats[groundInd].quad_status = st;
      if(st)
        info->status |= SSD_STATUS_DEGENERATE_QUAD; /* the reference terminates here */
      else
      {
        plats[groundInd].n_in_quad = nSel;
        plats[groundInd].mean_z = mean;
        if(project_to_binary_image(&f, sel, nSel, img))
          info->status |= SSD_STATUS_BEV_OOB;
        ssd_oracle_close(img, W, H);
        P2 l, r;
        int valid;
        detect_front_edge_closed(img, W, H, &l, &r, &valid);
        P3 *sq = stepQuads[nSteps++];
        if(valid)
        {
          const P2 fl = image_to_world(&f, l), fr = image_to_world(&f, r);
          const LineD frontLine = lined_from_pts(fl, fr);
          const P2 frontLeft = line_intersection_plain(frontLine, lined_from_pts(gq[0], gq[2]));
          const P2 frontRight = line_intersection_plain(frontLine, lined_from_pts(gq[1], gq[3]));
          const P3 a = { frontLeft.x, frontLeft.y, mean }, b = { frontRight.x, frontRight.y, mean }, c = { gq[2].x, gq[2].y, mean },
                   d = { gq[3].x, gq[3].y, mean };
          sq[0] = a;
          sq[1] = b;
          sq[2] = c;
          sq[3] = d;
          if(nSel == 0)
            info->status |= SSD_STATUS_EMPTY_MEAN;
        }
        else
        {
          memset(sq, 0, sizeof(P3) * 4); /* return{} (:546) */
          info->status |= SSD_STATUS_INVALID_FRONT_EDGE;
        }
      }
    }
    for(int i = firstValid; i < nPeaks; i++) /* :445-452, calcStairStep :549-558 */
    {
      if(!plats[i].valid)
        continue;
      uint32_t nSel;
      double mean;
      const int st = points_in_quad_mean(&f, pStart[i], pCount[i], quadW[i], NULL, &nSel, &mean);
      plats[i].quad_status = st;
      if(st)
      {
        info->status |= SSD_STATUS_DEGENERATE_QUAD;
        continue;
      }
      plats[i].n_in_quad = nSel;
      plats[i].mean_z = mean;
      if(nSel == 0)
        info->status |= SSD_STATUS_EMPTY_MEAN;
      P3 *sq = stepQuads[nSteps++];
      for(int c = 0; c < 4; c++)
      {
        sq[c].x = quadW[i][c].x;
        sq[c].y = quadW[i][c].y;
        sq[c].z = mean;
      }
    }
  }
  for(int k = 0; k < nPeaks; k++)
    for(int c = 0; c < 4; c++)
    {
      plats[k].quad_world[c][0] = quadW[k][c].x;
      plats[k].quad_world[c][1] = quadW[k][c].y;
    }

  /* detectStairs result assembly (:370-383) with ToExternalWorld (transformation.cpp:190-194) */
  info->n_steps = nSteps;
  for(int s = 0; s < nSteps; s++)
  {
    for(int c = 0; c < 4; c++)
    {
      g_last_step_quads[s][c][0] = stepQuads[s][c].x;
      g_last_step_quads[s][c][1] = stepQuads[s][c].y;
      g_last_step_quads[s][c][2] = stepQuads[s][c].z;
    }
    for(int c = 0; c < 4; c++)
    {
      const double x = stepQuads[s][c].x, y = stepQuads[s][c].y;
      steps[s].quad[c][0] = (xf->ext_a[0] * x + xf->ext_a[1] * y) + xf->ext_b[0];
      steps[s].quad[c][1] = (xf->ext_a[2] * x + xf->ext_a[3] * y) + xf->ext_b[1];
    }
    steps[s].height = xf->ext_z + stepQuads[s][0].z;
  }
  g_last_n_steps = nSteps;
  if(nSteps == 0)
    info->status |= SSD_STATUS_NO_STEPS;

done:
  free(f.world);
  free(f.pixel);
  free(f.height);
  free(cur);
  free(upper);
  free(store);
  free(sel);
  free(img);
  return rc;
}

/* ssd_oracle_vertical_faces on a group: every member's remainder points through its own CameraToWorld, into one set of risers.
 * labels: n_members*W*H as ssd_oracle_process_group wrote them; plateaus: the group's. */
int ssd_oracle_vertical_faces_group(const ssd_gpu_config *cfg, const ssd_gpu_transform *xfs, const float *xyz, int n_members,
                                    const uint8_t *labels, const ssd_gpu_plateau *plateaus, int n_plateaus, ssd_gpu_riser *out, int cap, int *n)
{
  ssd_oracle_derived d;
  const int rc = ssd_oracle_derive(cfg, &d);
  if(rc)
    return rc;
  if(n_members < 1)
    return SSD_E_INVALID_ARG;
  const int R = n_plateaus > 1 ? n_plateaus - 1 : 0;
  if(n)
    *n = R;
  if(R > SSD_GPU_MAX_PLATEAUS)
    return SSD_E_RANGE;
  uint32_t cnt[SSD_GPU_MAX_PLATEAUS];
  long long sx[SSD_GPU_MAX_PLATEAUS], sy[SSD_GPU_MAX_PLATEAUS], xmin[SSD_GPU_MAX_PLATEAUS], xmax[SSD_GPU_MAX_PLATEAUS], ymin[SSD_GPU_MAX_PLATEAUS],
    ymax[SSD_GPU_MAX_PLATEAUS];
  for(int k = 0; k < SSD_GPU_MAX_PLATEAUS; k++)
  {
    cnt[k] = 0;
    sx[k] = sy[k] = 0;
    xmin[k] = ymin[k] = 0x7fffffff;
    xmax[k] = ymax[k] = -1;
  }
  const size_t N = (size_t)cfg->width * cfg->height;
  for(size_t i = 0; i < N * (size_t)n_members; i++)
  {
    if(labels[i] != SSD_LABEL_REMAINDER)
      continue;
    double w[3];
    camera_to_world(&xfs[i / N], xyz + i * 3, w);
    const int h = (uint16_t)((w[2] - cfg->z_min) * d.height_interval_reciprocal); /* calcHeights (pointcloud.cpp:175) */
    int r = -1;
    for(int k = 0; k + 1 < n_plateaus; k++)
      if(h > plateaus[k].hmax && h < plateaus[k + 1].hmin)
        r = k;
    if(r < 0)
      continue;
    const long long X = (long long)((w[0] - cfg->x_min) * 65536.0), Y = (long long)((w[1] - cfg->y_min) * 65536.0);
    cnt[r]++;
    sx[r] += X;
    sy[r] += Y;
    if(X < xmin[r]) xmin[r] = X;
    if(X > xmax[r]) xmax[r] = X;
    if(Y < ymin[r]) ymin[r] = Y;
    if(Y > ymax[r]) ymax[r] = Y;
  }
  for(int k = 0; k < R && k < cap && out; k++)
  {
    ssd_gpu_riser o;
    memset(&o, 0, sizeof o);
    o.lower_plateau = k;
    o.upper_plateau = k + 1;
    o.n_points = cnt[k];
    o.z_bottom = cfg->z_min + (double)(plateaus[k].hmax + 1) * cfg->height_interval;
    o.z_top = cfg->z_min + (double)plateaus[k + 1].hmin * cfg->height_interval;
    if(cnt[k])
    {
      o.x_min = cfg->x_min + (double)xmin[k] / 65536.0;
      o.x_max = cfg->x_min + (double)xmax[k] / 65536.0;
      o.y_min = cfg->y_min + (double)ymin[k] / 65536.0;
      o.y_max = cfg->y_min + (double)ymax[k] / 65536.0;
      o.x_mean = cfg->x_min + (double)(unsigned long long)sx[k] / (double)cnt[k] / 65536.0;
      o.y_mean = cfg->y_min + (double)(unsigned long long)sy[k] / (double)cnt[k] / 65536.0;
    }
    out[k] = o;
  }
  return SSD_OK;
}
