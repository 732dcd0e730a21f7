/*
 * oracle_outline.c -- TEST INFRASTRUCTURE. Inspection of the outline and front-edge line fits of the oracle (oracle/ssd_oracle.c,
 * compiled into this translation unit): the scan-point lists a closed image yields, and per list the statistics of the brute-force
 * fit that decide which line wins -- so that tests can construct lists with a designed residual path, tie or hypot dependence.
 *
 * Every hypot of the oracle goes through oo_hypot. Mode 0 (default) is glibc's hypot, i.e. the reference. Mode 1 takes the IEEE
 * square root of a*a + b*b for integer operands (the correctly rounded hypot) and glibc's hypot otherwise: with it the oracle
 * computes what a line fit with a correctly rounded denominator selects, so a test can show what a hypot-dependent tie changes.
 * Build: gcc -std=c11 -O2 -ffp-contract=off -fPIC -shared (the flags of oracle/Makefile) -o libssd_oracle_outline.so oracle_outline.c -lm
 */
#include <math.h>

static double oo_hypot(double x, double y);
#define hypot oo_hypot
#include "../../oracle/ssd_oracle.c"
#undef hypot

static int g_hypot_mode;

static int oo_small_int(double v) { return v == floor(v) && fabs(v) < 67108864.0; }

static double oo_hypot(double x, double y)
{
  if(g_hypot_mode == 1 && oo_small_int(x) && oo_small_int(y))
    return sqrt(x * x + y * y);
  return hypot(x, y);
}

void oo_set_hypot_mode(int mode) { g_hypot_mode = mode; }

/* the closed image's scans and the four edge lists of detectOutline (segmentation.cpp:607-620, :129-156).
 * scans: (x, yFirst, ySecond) of the right scans then the left scans (cap 3 * (W / 25 + 2) ints), *nr / *nl their counts.
 * lists: four blocks of cap2 = W / 25 + 4 points (x, y) in the order frontLeft, frontRight, backLeft, backRight; n[4] their lengths
 * (all 0 when the outline is rejected before the fit: no right scan or fewer than three scans). Returns 1 if the fit runs. */
int oo_outline_lists(const uint8_t *image, int W, int H, int min_img_y_extent, int *scans, int *nr, int *nl, int *lists, int n[4])
{
  uint8_t *img = (uint8_t *)malloc((size_t)W * H);
  memcpy(img, image, (size_t)W * H);
  ssd_oracle_close(img, W, H);
  const int cap = W / 25 + 2, cap2 = W / 25 + 4;
  Scan *sr = (Scan *)malloc(sizeof(Scan) * (size_t)cap), *sl = (Scan *)malloc(sizeof(Scan) * (size_t)cap);
  *nr = scanner_scan(img, W, H, min_img_y_extent, W / 2, 25, sr);
  *nl = *nr > 0 ? scanner_scan(img, W, H, min_img_y_extent, W / 2 - 25, -25, sl) : 0;
  for(int i = 0; i < *nr; i++)
  {
    scans[3 * i] = sr[i].x;
    scans[3 * i + 1] = sr[i].yFirst;
    scans[3 * i + 2] = sr[i].ySecond;
  }
  for(int i = 0; i < *nl; i++)
  {
    scans[3 * (*nr + i)] = sl[i].x;
    scans[3 * (*nr + i) + 1] = sl[i].yFirst;
    scans[3 * (*nr + i) + 2] = sl[i].ySecond;
  }
  for(int e = 0; e < 4; e++)
    n[e] = 0;
  const int ok = *nr > 0 && *nl + *nr >= 3;
  if(ok)
  {
    P2i *buf = (P2i *)malloc(sizeof(P2i) * (size_t)(4 * cap2));
    LinePts left = { buf, buf + cap2, 0 }, right = { buf + 2 * cap2, buf + 3 * cap2, 0 };
    obtain_line_points(sl, *nl, sr, *nr, &left, &right);
    const P2i *src[4] = { left.front, right.front, left.back, right.back };
    const int ns[4] = { left.n, right.n, left.n, right.n };
    for(int e = 0; e < 4; e++)
    {
      n[e] = ns[e];
      for(int i = 0; i < ns[e]; i++)
      {
        lists[2 * (e * cap2 + i)] = src[e][i].x;
        lists[2 * (e * cap2 + i) + 1] = src[e][i].y;
      }
    }
    free(buf);
  }
  free(sr);
  free(sl);
  free(img);
  return ok;
}

/* the closed image's front-edge list (BottomScanner, segmentation.cpp:169-222): up to W / 50 + 3 points (x, y); returns n */
int oo_front_list(const uint8_t *image, int W, int H, int *pts)
{
  uint8_t *img = (uint8_t *)malloc((size_t)W * H);
  memcpy(img, image, (size_t)W * H);
  ssd_oracle_close(img, W, H);
  P2i *p = (P2i *)malloc(sizeof(P2i) * (size_t)(W / 50 + 3));
  const int n = bottom_scan(img, W, H, W / 2, 50, p);
  for(int i = 0; i < n; i++)
  {
    pts[2 * i] = p[i].x;
    pts[2 * i + 1] = p[i].y;
  }
  free(p);
  free(img);
  return n;
}

/* Statistics of BestLine on one list (segmentation.cpp:409-478), with the residual's denominator cnt * hypot(a, b) taken from
 * glibc's hypot (use_sqrt = 0, the reference) or the IEEE sqrt(a*a + b*b) (use_sqrt = 1).
 * out: [0] cnt  [1] minimal residual  [2] pairs at the minimum  [3] distinct lines at the minimum (FlatLine m, n; exact up to 2, more means at least 3)
 *      [4] index of the winning pair (first minimum in (p, q) order)  [5] its integer distance sum (as the reference's int)
 *      [6] largest (int64) distance sum over all pairs  [7..9] a, b, c of the winner  [10..12] a, b, c of the first line at the
 *      minimum that differs from the winner (0, 0, 0 if none) */
void oo_fit_stats(const int *xy, int n, int use_sqrt, double out[13])
{
  P2i *pts = (P2i *)malloc(sizeof(P2i) * (size_t)(n > 0 ? n : 1));
  int *d = (int *)malloc(sizeof(int) * (size_t)(n > 2 ? n : 2));
  for(int i = 0; i < n; i++)
  {
    pts[i].x = xy[2 * i];
    pts[i].y = xy[2 * i + 1];
  }
  for(int k = 0; k < 13; k++)
    out[k] = 0;
  const int m0 = n - 2;
  const size_t cnt = m0 > 4 ? (size_t)(m0 - 1) / 2 : 1;
  out[0] = (double)cnt;
  double best = 0;
  int have = 0, idx = 0, at_min = 0, distinct = 0;
  LineI bl = { 0, 0, 0 }, other = { 0, 0, 0 };
  long long maxsum = 0;
  for(int p = 0; p < n - 1; p++)
    for(int q = p + 1; q < n; q++, idx++)
    {
      const LineI l = linei_from(pts[p], pts[q]);
      double r = 0;
      long long lsum = 0;
      if(n > 2)
      {
        int m = 0;
        for(int i = 0; i < n; i++)
          if(i != p && i != q)
            d[m++] = abs(pts[i].x * l.a + pts[i].y * l.b + l.c);
        for(size_t k = cnt; k > 0; k--)
        {
          int mi = 0;
          for(int j = 1; j < m; j++)
            if(d[j] < d[mi])
              mi = j;
          lsum += d[mi];
          d[mi] = d[--m];
        }
        const int isum = (int)(unsigned)(long long)lsum; /* the reference's int sum: wraps modulo 2^32 */
        const double h = use_sqrt ? sqrt((double)l.a * l.a + (double)l.b * l.b) : hypot(l.a, l.b);
        r = isum / (cnt * h);
      }
      if(lsum > maxsum)
        maxsum = lsum;
      if(!have || r < best)
      {
        have = 1;
        best = r;
        bl = l;
        out[4] = idx;
        out[5] = (double)(int)(unsigned)(long long)lsum;
        at_min = 1;
        distinct = 1;
        other.a = other.b = other.c = 0;
      }
      else if(r == best)
      {
        at_min++;
        const FlatLine f = flat_from(l), g = flat_from(bl);
        if(f.m != g.m || f.n != g.n)
        {
          if(!other.a && !other.b && !other.c)
          {
            other = l;
            distinct++;
          }
          else
          {
            const FlatLine o = flat_from(other);
            if(f.m != o.m || f.n != o.n)
              distinct++;
          }
        }
      }
    }
  out[1] = best;
  out[2] = at_min;
  out[3] = distinct;
  out[6] = (double)maxsum;
  out[7] = bl.a;
  out[8] = bl.b;
  out[9] = bl.c;
  out[10] = other.a;
  out[11] = other.b;
  out[12] = other.c;
  free(pts);
  free(d);
}
