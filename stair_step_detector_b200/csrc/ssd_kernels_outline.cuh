// ssd_kernels_outline.cuh -- the per-plateau geometry kernels:
//   k_outline     : Segmentation::detectOutline (segmentation.cpp:919-971) on each plateau's BEV bitmap
//   k_frame_logic : first-valid / ground quadrilateral / QuadrilateralTest construction
//   k_finalize    : Segmentation::detectFrontEdge for the ground (segmentation.cpp:879-917), step assembly,
//                   ToExternalWorld, result records
// A BEV image is a bit-packed W x H occupancy bitmap (1 bit/pixel). Only the band of rows a plateau touched
// is staged into shared memory (coalesced), closed there with word-parallel 3x3 dilate/erode, and probed;
// the global bitmap is zeroed behind the read so it is clean for the next batch.
#pragma once
#include "ssd_device.cuh"
#include <type_traits>
#ifdef SSD_OL_PROF
#include <cstdio>
#endif

#define SSD_OL_THREADS 256
// columns a warp probes at once (probe_columns). Measured on B200 (r2): 1 -> k_outline 0.49 ms per 2048 frames, 35 us for one
// frame; 2 -> 0.55 ms / 37 us; 3 -> 0.57 ms / 40 us: the kernel lives under a 40-register cap and the extra chains spill
#ifndef SSD_OL_PROBE_G
#define SSD_OL_PROBE_G 1
#endif

// Band of a raw BEV bitmap: rows [b0, b0+nb) with row stride rs words, staged in shared memory (or left
// in global memory for images too large); rows outside the band are all zero. The 3x3 close is evaluated
// on the fly, word-parallel, wherever a probe needs it.
struct Band
{
  const unsigned *A;
  int b0, nb, rs;
};

__device__ __forceinline__ unsigned raw_word(const Band &bd, int r, int w, int wpr)
{
  // r is band-relative; caller guarantees 0 <= r < nb
  return (w >= 0 && w < wpr) ? bd.A[(unsigned)(r * bd.rs + w)] : 0u;
}

// 64-bit window of raw row r: bit p <-> image column 32*w - 16 + p
__device__ __forceinline__ unsigned long long raw_win(const Band &bd, int r, int w, int wpr)
{
  const unsigned long long l = raw_word(bd, r, w - 1, wpr), c = raw_word(bd, r, w, wpr), n = raw_word(bd, r, w + 1, wpr);
  return (l >> 16) | (c << 16) | (n << 48);
}

// One 32-pixel word of cv::morphologyEx(MORPH_CLOSE, 3x3) (call sites segmentation.cpp:888,928) at image
// row y, word w: dilate (out-of-image = 0) then erode (out-of-image ignored = 1), OpenCV's default borders.
__device__ inline unsigned closed_word(const DevParams &p, const Band &bd, int y, int w)
{
  const int wpr = p.wpr, H = p.H, W = p.W;
  // horizontally dilated raw rows y-2 .. y+2 (zero outside the band / image)
  unsigned long long hd[5];
#pragma unroll
  for(int k = 0; k < 5; k++)
  {
    const int r = y - 2 + k - bd.b0;
    unsigned long long v = 0;
    if(r >= 0 && r < bd.nb)
    {
      const unsigned long long R = raw_win(bd, r, w, wpr);
      v = R | (R << 1) | (R >> 1);
    }
    hd[k] = v;
  }
  // columns outside the image count as set for the erosion
  unsigned long long outside = 0;
  {
    const long long x0 = (long long)32 * w - 16; // image column of bit 0
    if(x0 < 0)
      outside |= (1ull << (-x0)) - 1ull;
    const long long over = x0 + 64 - W; // number of window bits at columns >= W
    if(over > 0)
      outside |= over >= 64 ? ~0ull : ~((1ull << (64 - over)) - 1ull);
  }
  unsigned long long acc = ~0ull;
#pragma unroll
  for(int k = 1; k <= 3; k++) // dilated rows y-1, y, y+1
  {
    const int yy = y - 2 + k;
    if(yy < 0 || yy >= H)
      continue; // row outside the image: ignored by the erosion
    unsigned long long D = hd[k];
    if(yy - 1 >= 0)
      D |= hd[k - 1];
    if(yy + 1 < H)
      D |= hd[k + 1];
    D |= outside;
    acc &= D & (D << 1 | 1ull) & (D >> 1 | (1ull << 63));
  }
  unsigned out = (unsigned)(acc >> 16);
  if(w == wpr - 1 && (W & 31))
    out &= (1u << (W & 31)) - 1u;
  return out;
}

// stage the raw rows of a band into shared memory (coalesced) and clear the global bitmap behind the read. The band is one
// contiguous run of words in the bitmap; eight independent loads per thread are in flight before the first is consumed (the
// plain loop -- load, conditional store to the same array, next load -- ran as a chain of dependent L2 round trips).
__device__ inline void band_stage(const DevParams &p, unsigned *sm, const Band &bd, unsigned *__restrict__ g, int tid, int nthreads)
{
  const unsigned wpr = (unsigned)p.wpr;
  const unsigned total = (unsigned)bd.nb * wpr;
  // row = (i * magic) >> 32, exact for i * wpr < 2^32. One word per row (W <= 32) would need magic = 2^32, which wraps
  // to 0 in 32 bits: there the row is i itself.
  const unsigned magic = 0xffffffffu / wpr + 1u;
  unsigned *src = g + (size_t)bd.b0 * wpr;
  for(unsigned base = (unsigned)tid; base < total; base += (unsigned)nthreads * 8u)
  {
    unsigned v[8];
#pragma unroll
    for(int k = 0; k < 8; k++)
    {
      const unsigned i = base + (unsigned)(k * nthreads);
      v[k] = i < total ? __ldcg(src + i) : 0u;
    }
#pragma unroll
    for(int k = 0; k < 8; k++)
    {
      const unsigned i = base + (unsigned)(k * nthreads);
      if(i < total)
      {
        if(v[k])
          src[i] = 0u;
        const unsigned r = wpr == 1u ? i : __umulhi(i, magic);
        sm[i + r * (unsigned)(bd.rs - (int)wpr)] = v[k]; // row stride rs: r * rs + (i - r * wpr)
      }
    }
  }
  __syncthreads();
}

// first / last set row of column x of the closed image within rows [ylo, yhi]
// (Scanner::probeVertical, segmentation.cpp:85-111; BottomScanner::probeBottomUp :225-240); one warp per column.
// Only ONE bit per row is wanted, so the 3x3 close is evaluated for that column alone, one image row per lane:
//   f   = raw bits of columns x-2 .. x+2 of the lane's row (0 outside the image / band)
//   hd  = horizontal dilation at columns x-1, x, x+1              (3 bits, from f)
//   D   = hd of rows y-1, y, y+1 OR-ed (warp shuffles)            = dilated image at (x-1..x+1, y)
//   E   = D with out-of-image columns forced to 1; rows outside the image count as all ones (erosion ignores them)
//   closed(x, y) = E(y-1) == E(y) == E(y+1) == 111b
// A warp pass covers 28 rows (lanes 2..29) plus a two-row halo on either side.
// rows base .. base + 27 of column x as a ballot mask (bit = lane = row base - 2 + lane), restricted to rows [lo, hi]
__device__ __forceinline__ unsigned probe_chunk(const DevParams &p, const Band &bd, int x, int base, int lo, int hi, int lane)
{
  const int xl = x - 2;
  const int wA = xl >> 5, sh = xl & 31; // arithmetic shift: xl < 0 -> word -1 (reads as 0)
  // columns x-1, x, x+1 that lie outside the image
  const unsigned colout = (x - 1 < 0 ? 1u : 0u) | (x + 1 >= p.W ? 4u : 0u);
  const int y = base - 2 + lane;
  const int r = y - bd.b0;
  unsigned hd = 0;
  if(r >= 0 && r < bd.nb) // (band rows are image rows)
  {
    const unsigned w0 = raw_word(bd, r, wA, p.wpr), w1 = raw_word(bd, r, wA + 1, p.wpr);
    const unsigned f = __funnelshift_r(w0, w1, sh) & 31u;
    hd = (f | (f >> 1) | (f >> 2)) & 7u;
  }
  const unsigned up = __shfl_up_sync(0xffffffffu, hd, 1), dn = __shfl_down_sync(0xffffffffu, hd, 1);
  const bool inimg = y >= 0 && y < p.H;
  // lanes 0 and 31 lack one neighbour: their E is never used for a reported row (lanes 2..29 read lanes 1..30)
  const unsigned E = inimg ? (hd | up | dn | colout) : 7u;
  const unsigned full = E == 7u ? 1u : 0u;
  const unsigned fu = __shfl_up_sync(0xffffffffu, full, 1), fd = __shfl_down_sync(0xffffffffu, full, 1);
  const bool set = (full & fu & fd) != 0u && lane >= 2 && lane < 30 && y >= lo && y <= hi;
  return __ballot_sync(0xffffffffu, set);
}

__device__ __forceinline__ bool probe_column(const DevParams &p, const Band &bd, int x, int ylo, int yhi, int lane, int &yFirst, int &ySecond)
{
  int first = 0x7fffffff, last = -1;
  // the closed image can only be set within one row of the raw band
  const int lo = max(ylo, bd.b0), hi = min(yhi, bd.b0 + bd.nb - 1);
  // top-down to the first set row, then bottom-up to the last one: a plateau's column is set near both ends of its band,
  // so two passes usually do where a full scan of the band took nine
  int bf = lo;
  for(; bf <= hi; bf += 28)
  {
    const unsigned m = probe_chunk(p, bd, x, bf, lo, hi, lane);
    if(m)
    {
      first = bf - 2 + __ffs(m) - 1;
      last = bf - 2 + 31 - __clz(m);
      break;
    }
  }
  if(last >= 0)
    for(int b2 = hi - 27; b2 > bf; b2 -= 28)
    {
      const unsigned m = probe_chunk(p, bd, x, b2, lo, hi, lane);
      if(m)
      {
        last = max(last, b2 - 2 + 31 - __clz(m));
        break;
      }
    }
  yFirst = first;
  ySecond = last;
  return last >= 0;
}

// G columns at once (one warp): the top and the bottom chunk of every column are evaluated first -- independent chains of
// shared-memory loads and shuffles that overlap -- and decide the column when both hold a set row (they nearly always do: the
// band hugs the plateau); any other column takes probe_column. Same result: first / last set row of the column in [ylo, yhi].
template<int G>
__device__ __forceinline__ void probe_columns(const DevParams &p, const Band &bd, const int (&x)[G], int nvalid, int ylo, int yhi, int lane,
                                              int (&yFirst)[G], int (&ySecond)[G], bool (&found)[G])
{
  const int lo = max(ylo, bd.b0), hi = min(yhi, bd.b0 + bd.nb - 1);
  const bool two = hi - 27 > lo;
  unsigned mt[G], mb[G];
#pragma unroll
  for(int g = 0; g < G; g++)
    mt[g] = (g < nvalid && lo <= hi) ? probe_chunk(p, bd, x[g], lo, lo, hi, lane) : 0u;
#pragma unroll
  for(int g = 0; g < G; g++)
    mb[g] = (g < nvalid && two) ? probe_chunk(p, bd, x[g], hi - 27, lo, hi, lane) : 0u;
#pragma unroll
  for(int g = 0; g < G; g++)
  {
    if(g >= nvalid)
      continue;
    if(mt[g] && (!two || mb[g]))
    {
      yFirst[g] = lo - 2 + __ffs(mt[g]) - 1;
      int last = lo - 2 + 31 - __clz(mt[g]);
      if(two)
        last = max(last, hi - 27 - 2 + 31 - __clz(mb[g]));
      ySecond[g] = last;
      found[g] = true;
    }
    else
      found[g] = probe_column(p, bd, x[g], ylo, yhi, lane, yFirst[g], ySecond[g]);
  }
}

// ---- BestLine (segmentation.cpp:409-487): every pair (p,q), residual = mean of the n smallest integer
// distances of the other points / hypot(a,b); winner = first minimal residual in (p,q) order.
// Up to four point lists are fitted in one pass: one (list, pair) task per thread, warp-shuffle arg-min on
// (residual, pair index) per list, one shared-memory round across the warps.
#define SSD_BL_CHUNK 2048 // line-fit candidates probed per round (large frame-size class)
template<int NWARPS>
struct BestLineWorkT
{
  double res[NWARPS][4];
  int idx[NWARPS][4];
  unsigned long long best[4]; // large frame-size class: bits of the smallest residual any thread has computed so far, per list
  // ... and the queue of the candidates that survive the pruning probe (best_lines_block): the few survivors are evaluated
  // densely, one per thread, instead of dragging the 31 pruned lanes of their warps through the bisection
  int nq;
  int queue[NWARPS > 8 ? SSD_BL_CHUNK : 1];
};

// Sum of the cnt (<= S) smallest distances of the other points to line l: insertion into a sorted register array
// (one min / max pair per slot, no branches). Ties need no order: only the sum of the values is used.
template<int S>
__device__ __forceinline__ long long sum_smallest(const P2id *pts, int n, int pi, int qi, LineId l, int cnt)
{
  int a[S];
#pragma unroll
  for(int k = 0; k < S; k++)
    a[k] = 0x7fffffff;
  for(int i = 0; i < n; i++)
  {
    if(i == pi || i == qi)
      continue;
    int d = abs(pts[i].x * l.a + pts[i].y * l.b + l.c);
#pragma unroll
    for(int k = 0; k < S; k++)
    {
      const int lo = min(a[k], d);
      d = max(a[k], d);
      a[k] = lo;
    }
  }
  long long sum = 0;
#pragma unroll
  for(int k = 0; k < S; k++)
    sum += k < cnt ? a[k] : 0;
  return sum;
}

// The pruning probe of pair_residual alone (large frame-size class): true when the line through points pi, qi is certainly worse
// than `bound` (see pair_residual for the argument). No per-thread array: one pass over the list.
__device__ inline bool pair_abandoned(const P2id *pts, int n, int pi, int qi, LineId l, double bound)
{
  if(n <= 2 || !(bound < 1e300))
    return false;
  const int m = n - 2;
  const int cnt = m > 4 ? (m - 1) / 2 : 1;
  const double Bf = bound * ((double)(size_t)cnt * hypot_glibc_int(l.a, l.b)) * (1.0 + 1e-12);
  if(!(Bf < 4e18))
    return false;
  const long long B = (long long)Bf + 1;
  const long long th = 2 * B / cnt;
  const int mid = th < 0x7fffffffll ? (int)th : 0x7fffffff;
  int c = 0, mx = 0;
  long long sb = 0;
  for(int i = 0; i < n; i++)
    if(i != pi && i != qi)
    {
      const int v = abs(pts[i].x * l.a + pts[i].y * l.b + l.c);
      mx = max(mx, v);
      if(v <= mid)
      {
        c++;
        sb += v;
      }
    }
  return (long long)cnt * mx < (1ll << 31) && th < mx && c < cnt && sb + (long long)(cnt - c) * ((long long)mid + 1) >= B;
}

// bound: a residual some line of this list is already known to reach (+inf: none). Only the large frame-size class
// uses it: a line whose residual is certainly LARGER than bound is abandoned after one probe and reported as +inf
// (it can neither be the minimum nor tie with it, so the winner -- first minimal residual in pair order -- is unchanged).
template<int MAXPTS>
__device__ inline double pair_residual(const P2id *pts, int n, int pi, int qi, LineId l, double bound)
{
  if(n <= 2)
    return 0.0;
  const int m = n - 2;
  const int cnt = m > 4 ? (m - 1) / 2 : 1;
  long long sum = 0;
  if(cnt <= 4)
    sum = sum_smallest<4>(pts, n, pi, qi, l, cnt);
  else if(cnt <= 8)
    sum = sum_smallest<8>(pts, n, pi, qi, l, cnt);
  else if(cnt <= 12)
    sum = sum_smallest<12>(pts, n, pi, qi, l, cnt);
  else if(cnt <= 24 && MAXPTS <= 64)
  {
    // repeated minimum extraction without materialising the list: extract in (value, index) order
    int lastv = -1, lasti = -1;
    for(int t = 0; t < cnt; t++)
    {
      int bestv = 0x7fffffff, besti = -1;
      for(int i = 0; i < n; i++)
      {
        if(i == pi || i == qi)
          continue;
        const int d = abs(pts[i].x * l.a + pts[i].y * l.b + l.c);
        if((d > lastv || (d == lastv && i > lasti)) && d < bestv)
        {
          bestv = d;
          besti = i;
        }
      }
      sum += bestv;
      lastv = bestv;
      lasti = besti;
    }
  }
  else if(MAXPTS > 64)
  {
    // many points per list (high-resolution frames): value bisection for T = the cnt-th smallest distance, i.e. the
    // smallest T with count(d <= T) >= cnt; sum = sum(d < T) + (cnt - count(d < T)) * T. The distances are computed once
    // into a per-thread array (local memory: interleaved per thread, so a warp's accesses coalesce and stay in L1) and
    // each of the ~22 bisection passes is a load, a compare and an add per point.
    // (measured, r2: recomputing the distances from the list in shared memory in every pass instead of keeping them in this
    //  local-memory array is 2.8x slower for k_outline at 4096x3072 -- 3.43 against 1.21 ms per 64 frames -- although the
    //  array's L1 hit rate is poor)
    // Pruning probe FIRST, without the array (r2: the array made every candidate write and re-read 81 values of local memory, ~9 MB
    // per plateau through L2; all but a few candidates end here). residual = isum / D with D = cnt * hypot (below). If
    // isum >= B := floor(bound * D * (1 + 1e-12)) + 1 then isum / D exceeds bound by a relative 0.9e-12 >> 1 ulp, so the rounded
    // residual is strictly larger than bound. With c = count(d <= mid) < cnt every one of the cnt smallest beyond those c is
    // >= mid + 1, so sum >= sum(d <= mid) + (cnt - c) * (mid + 1): at mid = 2 B / cnt (twice the admissible mean) a line with
    // fewer than cnt / 2 points that close is out after this single pass; otherwise the probe narrows the bisection interval.
    // Only when the reference's int sum cannot wrap (cnt * hi < 2^31), so that isum == sum.
    int hi = -1, lo = 0;
    if(bound < 1e300)
    {
      const double Bf = bound * ((double)(size_t)cnt * hypot_glibc_int(l.a, l.b)) * (1.0 + 1e-12);
      if(Bf < 4e18)
      {
        const long long B = (long long)Bf + 1;
        const long long th = 2 * B / cnt;
        const int mid = th < 0x7fffffffll ? (int)th : 0x7fffffff;
        int c = 0, mx = 0;
        long long sb = 0;
        for(int i = 0; i < n; i++)
          if(i != pi && i != qi)
          {
            const int v = abs(pts[i].x * l.a + pts[i].y * l.b + l.c);
            mx = max(mx, v);
            if(v <= mid)
            {
              c++;
              sb += v;
            }
          }
        hi = mx;
        if((long long)cnt * mx < (1ll << 31) && th < mx)
        {
          if(c >= cnt)
            hi = mid;
          else
          {
            if(sb + (long long)(cnt - c) * ((long long)mid + 1) >= B)
              return __longlong_as_double(0x7ff0000000000000ll);
            lo = mid + 1;
          }
        }
      }
    }
    // survivors (and the first candidates, which have no bound yet): value bisection on the distances, computed once into a
    // per-thread array (local memory: interleaved per thread, so a warp's accesses coalesce)
    int d[MAXPTS]; // the list capacity of the frame-size class
    int k = 0, mx2 = 0;
    for(int i = 0; i < n; i++)
      if(i != pi && i != qi)
      {
        const int v = abs(pts[i].x * l.a + pts[i].y * l.b + l.c);
        d[k++] = v;
        mx2 = max(mx2, v);
      }
    if(hi < 0)
      hi = mx2;
    while(lo < hi)
    {
      const int mid = lo + ((hi - lo) >> 1);
      int c = 0;
      for(int i = 0; i < k; i++)
        c += d[i] <= mid;
      if(c >= cnt)
        hi = mid;
      else
        lo = mid + 1;
    }
    int below = 0;
    for(int i = 0; i < k; i++)
      if(d[i] < lo)
      {
        sum += d[i];
        below++;
      }
    sum += (long long)(cnt - below) * lo;
  }
  else
  {
    // the same value bisection for the few such fits of a small frame (n <= 32 points): distances recomputed per pass,
    // no per-thread array (it would cost every thread of the kernel its local-memory frame)
    int lo = 0, hi = 0;
    for(int i = 0; i < n; i++)
      if(i != pi && i != qi)
        hi = max(hi, abs(pts[i].x * l.a + pts[i].y * l.b + l.c));
    while(lo < hi)
    {
      const int mid = lo + ((hi - lo) >> 1);
      int c = 0;
      for(int i = 0; i < n; i++)
        if(i != pi && i != qi)
          c += abs(pts[i].x * l.a + pts[i].y * l.b + l.c) <= mid;
      if(c >= cnt)
        hi = mid;
      else
        lo = mid + 1;
    }
    int below = 0;
    for(int i = 0; i < n; i++)
      if(i != pi && i != qi)
      {
        const int v = abs(pts[i].x * l.a + pts[i].y * l.b + l.c);
        if(v < lo)
        {
          sum += v;
          below++;
        }
      }
    sum += (long long)(cnt - below) * lo;
  }
  // the reference sums into int (segmentation.cpp:434); keep its wrap-around semantics.
  // glibc's hypot, not the correctly rounded one: equal a*a+b*b with different glibc roundings must not tie (hypot_glibc_int)
  const int isum = (int)sum;
  const double h = hypot_glibc_int(l.a, l.b);
  return isum / ((double)(size_t)cnt * h); // :442
}

// all threads of the block must call. lists[e] with n[e] points (n[e] < 2: skipped); out[e] = winning line.
template<int MAXPTS, class BestLineWork>
__device__ inline void best_lines_block(const P2id *const lists[4], const int n[4], BestLineWork &wk, LineId *out, int tid, int nthreads)
{
  int off[5];
  off[0] = 0;
  for(int e = 0; e < 4; e++)
    off[e + 1] = off[e] + (n[e] >= 2 ? n[e] * (n[e] - 1) / 2 : 0);
  double bres[4];
  int bidx[4];
#pragma unroll
  for(int e = 0; e < 4; e++)
  {
    bres[e] = 0;
    bidx[e] = 0x7fffffff;
  }
  if(MAXPTS > 64)
  {
    if(tid < 4)
      wk.best[tid] = 0x7ff0000000000000ull; // +inf
    __syncthreads();
  }
  // one candidate: task index -> (list, pair), residual (with the list's current bound), the thread's running minimum
  auto decode = [&](int t, int &e, int &local, int &pI, int &qI)
  {
    e = 0;
    while(t >= off[e + 1])
      e++;
    local = t - off[e];
    const int ne = n[e];
    // local = pI*ne - pI*(pI+1)/2 + (qI - pI - 1), pairs in (p,q) lexicographic order: pI is the largest p whose row starts at
    // or before local, from the root of the quadratic (single precision: exact to within one, then corrected)
    const int bq = 2 * ne - 1;
    pI = (int)(((float)bq - sqrtf((float)(bq * bq - 8 * local))) * 0.5f);
    pI = max(0, min(pI, ne - 2));
    while(pI + 1 <= ne - 2 && (pI + 1) * ne - (pI + 1) * (pI + 2) / 2 <= local)
      pI++;
    while(pI * ne - pI * (pI + 1) / 2 > local)
      pI--;
    const int rowStart = pI * ne - pI * (pI + 1) / 2;
    qI = local - rowStart + pI + 1;
  };
  auto evaluate = [&](int t)
  {
    int e, local, pI, qI;
    decode(t, e, local, pI, qI);
    const P2id *pts = lists[e];
    const LineId l = linei_from(pts[pI], pts[qI]);
    double bound = __longlong_as_double(0x7ff0000000000000ll);
    if(MAXPTS > 64)
      bound = __longlong_as_double((long long)atomicMin(&wk.best[e], ~0ull)); // atomic read (other threads lower it concurrently)
    const double r = pair_residual<MAXPTS>(pts, n[e], pI, qI, l, bound);
    if(MAXPTS > 64 && r >= 0.0 && r < bound) // (false for NaN; non-negative doubles order like their bit patterns)
      atomicMin(&wk.best[e], (unsigned long long)__double_as_longlong(r));
#pragma unroll
    for(int k = 0; k < 4; k++)
      if(k == e && (bidx[k] == 0x7fffffff || r < bres[k] || (r == bres[k] && local < bidx[k]))) // first of equals in pair order
      {
        bres[k] = r;
        bidx[k] = local;
      }
  };
  if(MAXPTS > 64 && sizeof(wk.queue) >= sizeof(int) * SSD_BL_CHUNK)
  {
    // Large frame-size class (n ~ 40-80 points per list, thousands of candidate lines): almost every candidate is pruned by
    // one probe against the best residual known so far, but a warp that holds one survivor used to take all its lanes through
    // the array fill and ~25 bisection passes (a third of the warps did: 32 % of the kernel's instructions). Instead:
    //   seeds   one candidate per thread evaluated in full: the pairs (i, i + n/2) of each list give every list a tight bound
    //   rounds  SSD_BL_CHUNK candidates at a time: every thread probes its share (no array), survivors go to a queue in shared
    //           memory; then the queue is evaluated densely, one survivor per thread (the probe is repeated there against the
    //           bound as it stands then). Abandoned candidates are provably worse than a residual that some line reaches, so
    //           the minimum and its first index are unchanged.
    // seeds: the pairs (i, i + n/2) of every list -- long baselines, i.e. lines close to the best -- one per thread
    {
      const int e = tid & 3, i = tid >> 2, ne = n[e], h = ne >> 1;
      if(ne >= 2 && i < ne - h)
        evaluate(off[e] + i * ne - i * (i + 1) / 2 + (h - 1)); // local index of the pair (i, i + h)
    }
    if(tid == 0)
      wk.nq = 0;
    __syncthreads();
    for(int base = 0; base < off[4]; base += SSD_BL_CHUNK)
    {
      const int end = min(off[4], base + SSD_BL_CHUNK);
      for(int t = base + tid; t < end; t += nthreads)
      {
        int e, local, pI, qI;
        decode(t, e, local, pI, qI);
        if(qI - pI == (n[e] >> 1) && pI < (nthreads >> 2))
          continue; // evaluated as a seed
        const P2id *pts = lists[e];
        const double bound = __longlong_as_double((long long)atomicMin(&wk.best[e], ~0ull));
        if(!pair_abandoned(pts, n[e], pI, qI, linei_from(pts[pI], pts[qI]), bound))
          wk.queue[atomicAdd(&wk.nq, 1)] = t;
      }
      __syncthreads();
      const int nq = wk.nq;
      for(int i = tid; i < nq; i += nthreads)
        evaluate(wk.queue[i]);
      __syncthreads();
      if(tid == 0)
        wk.nq = 0;
      __syncthreads();
    }
  }
  else
  {
    for(int t = tid; t < off[4]; t += nthreads)
      evaluate(t);
  }
  const int lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
#pragma unroll
  for(int e = 0; e < 4; e++)
  {
    double r1 = bres[e];
    int i1 = bidx[e];
#pragma unroll
    for(int s = 16; s > 0; s >>= 1)
    {
      const double r2 = __shfl_xor_sync(0xffffffffu, r1, s);
      const int i2 = __shfl_xor_sync(0xffffffffu, i1, s);
      // lowest pair index among the minimal residuals (min_element, segmentation.cpp:473-477)
      if(i2 != 0x7fffffff && (i1 == 0x7fffffff || r2 < r1 || (r2 == r1 && i2 < i1)))
      {
        r1 = r2;
        i1 = i2;
      }
    }
    if(lane == 0)
    {
      wk.res[warp][e] = r1;
      wk.idx[warp][e] = i1;
    }
  }
  __syncthreads();
  if(tid < 4)
  {
    const int e = tid;
    double r1 = wk.res[0][e];
    int i1 = wk.idx[0][e];
    for(int w = 1; w < nwarps; w++)
    {
      const double r2 = wk.res[w][e];
      const int i2 = wk.idx[w][e];
      if(i2 != 0x7fffffff && (i1 == 0x7fffffff || r2 < r1 || (r2 == r1 && i2 < i1)))
      {
        r1 = r2;
        i1 = i2;
      }
    }
    if(i1 != 0x7fffffff)
    {
      const int ne = n[e];
      int pI = 0, rowStart = 0;
      while(rowStart + (ne - 1 - pI) <= i1)
      {
        rowStart += ne - 1 - pI;
        pI++;
      }
      const int qI = i1 - rowStart + pI + 1;
      out[e] = linei_from(lists[e][pI], lists[e][qI]);
    }
  }
  __syncthreads();
}

// FlatLine (segmentation.cpp:490-519)
struct FlatLineD
{
  double m, n;
};
__device__ __forceinline__ FlatLineD flat_from(LineId l)
{
  FlatLineD f;
  f.m = (double)(-l.a) / l.b;
  f.n = (double)(-l.c) / l.b;
  return f;
}
__device__ __forceinline__ P2d flat_point(FlatLineD f, double x)
{
  P2d r;
  r.x = x;
  r.y = x * f.m + f.n;
  return r;
}
// BoundaryPoints::outer (segmentation.cpp:545-547): last list point within 10 px of the line, snapped onto it
__device__ inline P2d boundary_outer(const P2id *pts, int n, FlatLineD line)
{
  P2d r;
  r.x = -1;
  r.y = -1;
  for(int i = n - 1; i >= 0; i--)
  {
    const P2d pd = flat_point(line, pts[i].x);
    if(fabs(pd.y - pts[i].y) < 10)
    {
      r = pd;
      break;
    }
  }
  return r;
}

// Work area of one outline block. Sized per frame-size class (the launch picks it from W x H): the small class keeps
// the block under 40 KB of shared memory with a 32 KB band, so five to six blocks are resident per SM -- the kernel is a
// chain of short latency-bound phases and lives on resident blocks, not on issue slots.
template<int MAX_SCANS, int MAX_LINE_PTS, int MAX_VPTS_, int THREADS_ = SSD_OL_THREADS, int MINB_ = 0>
struct OutlineSharedT
{
  // block size / minimum resident blocks of k_outline for this class (MINB_ = 0: SSD_OL_MINB)
  static constexpr int THREADS = THREADS_;
  static constexpr int MINB = MINB_;
  static constexpr int MAX_VPTS = MAX_VPTS_;
  static constexpr int MAX_LPTS = MAX_LINE_PTS;
  // column scans
  int scan_found[MAX_SCANS];
  int scan_yf[MAX_SCANS];
  int scan_ys[MAX_SCANS];
  // the four edge point lists (segmentation.cpp:557-567)
  P2id frontLeft[MAX_LINE_PTS], backLeft[MAX_LINE_PTS], frontRight[MAX_LINE_PTS], backRight[MAX_LINE_PTS];
  int nLeft, nRight, ok;
  LineId line[4]; // frontLeft, frontRight, backLeft, backRight
  BestLineWorkT<(THREADS_ > SSD_OL_THREADS ? THREADS_ : SSD_OL_THREADS) / 32> wk; // (k_finalize runs SSD_OL_THREADS on either class)
  // vertical edge probing
  P2id vpts[MAX_VPTS_];
  int vfound[MAX_VPTS_];
  double vdist[MAX_VPTS_];
  int vn;
  int ve_left, ve_right, ve_ystart, ve_yend, ve_go;
  LineDd base;
  LineDd nl[4], nl2[2]; // base line: the four normalised edge lines, then the two normalised bisectors (one thread each)
  P2d outer[4];
  int best_pt;
};
// any supported frame size. 512 threads: the O(n^4) line fits are ~14 k tasks per block of long-latency (local-memory) work;
// the larger block halves a block's run time (fewer, longer blocks left a 30 % tail on 148 SMs) and raises the resident
// warps from 32 to 48 per SM (shared memory admits 4 blocks either way; registers admit 3 x 512 threads)
typedef OutlineSharedT<SSD_MAX_SCANS, SSD_MAX_LINE_PTS, SSD_MAX_VPTS, 512, 3> OutlineShared;
typedef OutlineSharedT<64, 32, 112> OutlineSharedSmall;                              // W <= 1280, H <= 1100

// Segmentation::detectOutline after the close (segmentation.cpp:930-946). Block-cooperative.
// Thread 0 ends up with the quadrilateral (image pixels) and the valid flag.
#ifdef SSD_OL_PROF
// debug variant: cycle stamps of thread 0 at the phase boundaries of one plateau (printed by k_outline for frame 0)
__device__ long long g_olp[16];
#define OLP(i)                     \
  do                               \
  {                                \
    if(tid == 0 && blockIdx.y == 0 && blockIdx.x == 0) \
      g_olp[i] = clock64();        \
  } while(0)
#else
#define OLP(i)
#endif
template<class OutlineShared>
__device__ inline void detect_outline_block(const DevParams &p, const Band &bd, OutlineShared &S, int min_img_y_extent, double xy_ratio,
                                            P2d quad[4], int &valid, int tid, int nthreads)
{
  OLP(1);
  const int W = p.W, H = p.H;
  const int lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
  const int xStep = 25, xCenter = W / 2; // HorizontalEdgesDetector (segmentation.cpp:605-611)
  // candidate columns: right = xCenter + j*25 (< W); left = xCenter - 25 - j*25 (>= 0)
  const int nRc = (W - 1 - xCenter) / xStep + 1;
  const int nLc = xCenter - xStep >= 0 ? (xCenter - xStep) / xStep + 1 : 0;
  {
    constexpr int G = SSD_OL_PROBE_G; // columns a warp probes at once
    for(int c0 = warp * G; c0 < nRc + nLc; c0 += nwarps * G)
    {
      int x[G], yf[G], ys[G];
      bool f[G];
      const int nv = min(G, nRc + nLc - c0);
#pragma unroll
      for(int g = 0; g < G; g++)
      {
        const int c = c0 + g;
        x[g] = c < nRc ? xCenter + c * xStep : xCenter - xStep - (c - nRc) * xStep;
      }
      probe_columns<G>(p, bd, x, nv, 0, H - 1, lane, yf, ys, f);
      if(lane < nv)
      {
#pragma unroll
        for(int g = 0; g < G; g++)
          if(lane == g)
          {
            S.scan_found[c0 + g] = f[g];
            S.scan_yf[c0 + g] = yf[g];
            S.scan_ys[c0 + g] = ys[g];
          }
      }
    }
  }
  __syncthreads();
  OLP(2);
  {
    // Scanner::scan stop rule (segmentation.cpp:68-80): stop at the first empty or too short column. Every warp counts the
    // leading good columns itself (ballots over the scan results), then all threads fill the four point lists.
    auto good = [&](int c) { return S.scan_found[c] && S.scan_ys[c] - S.scan_yf[c] >= min_img_y_extent; };
    int nr = 0, nl = 0;
    for(int b = 0; b < nRc; b += 32)
    {
      const int c = b + lane;
      const unsigned bad = ~__ballot_sync(0xffffffffu, c < nRc && good(c));
      if(bad)
      {
        nr = b + __ffs(bad) - 1;
        break;
      }
      nr = b + 32;
    }
    if(nr > 0)
      for(int b = 0; b < nLc; b += 32)
      {
        const int c = b + lane;
        const unsigned bad = ~__ballot_sync(0xffffffffu, c < nLc && good(nRc + c));
        if(bad)
        {
          nl = b + __ffs(bad) - 1;
          break;
        }
        nl = b + 32;
      }
    const bool ok = nr > 0 && nl + nr >= 3; // :612-616
    // Scanner::obtainLinePoints (:129-156) in closed form; scansRight[i] = column i, scansLeft[i] = column nRc+i.
    //   half = total / 2 + 1
    //   nl >= half:  right list = left columns iL .. 0 (iL = nl - half), then right columns 0 .. nr-1;  left list = left columns iL .. nl-1
    //   else:        left list = right columns iR .. 0 (iR = nr - half if nr > half, else 0), then left columns 0 .. nl-1;
    //                right list = right columns iR .. nr-1
    int nLeft = 0, nRight = 0;
    if(ok)
    {
      const int half = (nl + nr) / 2 + 1;
      const bool caseA = nl >= half;
      const int iL = caseA ? nl - half : 0, iR = (!caseA && nr > half) ? nr - half : 0;
      nLeft = caseA ? nl - iL : iR + 1 + nl;
      nRight = caseA ? iL + 1 + nr : nr - iR;
      for(int j = tid; j < nLeft || j < nRight; j += nthreads)
      {
        if(j < nLeft)
        {
          const int c = caseA ? nRc + iL + j : (j <= iR ? iR - j : nRc + (j - iR - 1));
          const int x = c < nRc ? xCenter + c * xStep : xCenter - xStep - (c - nRc) * xStep;
          S.frontLeft[j].x = x;
          S.frontLeft[j].y = S.scan_ys[c];
          S.backLeft[j].x = x;
          S.backLeft[j].y = S.scan_yf[c];
        }
        if(j < nRight)
        {
          const int c = caseA ? (j <= iL ? nRc + (iL - j) : j - iL - 1) : iR + j;
          const int x = c < nRc ? xCenter + c * xStep : xCenter - xStep - (c - nRc) * xStep;
          S.frontRight[j].x = x;
          S.frontRight[j].y = S.scan_ys[c];
          S.backRight[j].x = x;
          S.backRight[j].y = S.scan_yf[c];
        }
      }
    }
    if(tid == 0)
    {
      S.ok = ok;
      S.nLeft = nLeft;
      S.nRight = nRight;
    }
  }
  __syncthreads();
  valid = 0;
  if(tid == 0)
    for(int i = 0; i < 4; i++)
      quad[i].x = quad[i].y = 0; // Outline{} value-initialised
  if(!S.ok)
    return;

  OLP(3);
  // HorizontalEdges (:592-599): four best lines
  {
    const P2id *const lists[4] = { S.frontLeft, S.frontRight, S.backLeft, S.backRight };
    const int ns[4] = { S.nLeft, S.nRight, S.nLeft, S.nRight };
    best_lines_block<OutlineShared::MAX_LPTS>(lists, ns, S.wk, S.line, tid, nthreads);
  }
  OLP(4);

  // The boundary points of the four edges and the base line (VerticalEdgesDetector::calcBaseLine, :672-679) are chains of
  // double-precision divisions and square roots; the independent ones run on one thread each (first lanes of eight warps),
  // the same operations on the same operands as the serial order.
  if((tid & 31) == 0 && tid < 256)
  {
    const int j = tid >> 5;
    if(j < 4)
    {
      const P2id *lst = j == 0 ? S.frontLeft : (j == 1 ? S.frontRight : (j == 2 ? S.backLeft : S.backRight));
      S.outer[j] = boundary_outer(lst, (j & 1) ? S.nRight : S.nLeft, flat_from(S.line[j]));
    }
    else
    {
      // nl[0] = normalised reversed front-left, nl[1] = front-right, nl[2] = reversed back-left, nl[3] = back-right
      const int e = j - 4;
      LineId l = S.line[e];
      if(!(e & 1))
      {
        l.a = -l.a;
        l.b = -l.b;
        l.c = -l.c;
      }
      S.nl[e] = lined_normalized(lined_from_i(l));
    }
  }
  __syncthreads();
  if(tid == 0 || tid == 32)
  {
    const int h = tid >> 5; // 0: front, 1: back
    S.nl2[h] = lined_normalized(bisector(S.nl[2 * h], S.nl[2 * h + 1]));
  }
  __syncthreads();
  if(tid == 0)
  {
    const LineDd center = bisector(S.nl2[0], S.nl2[1]);
    const double cf = xy_ratio * xy_ratio;
    LineDd corr;
    corr.a = center.a * cf; // slopeCorrection (:377-380)
    corr.b = center.b;
    corr.c = center.c;
    const P2id p0 = S.frontLeft[0];
    S.base.a = -corr.b; // perpendicular (:372-376)
    S.base.b = corr.a;
    S.base.c = corr.b * p0.x - corr.a * p0.y;
    for(int i = 0; i < 4; i++)
      quad[i] = S.outer[i]; // value_or fall-backs (:939-945)
  }
  __syncthreads();

  // VerticalEdgesDetector::detect (:653-669): left edge (probe to the right), right edge (probe to the left)
  for(int e = 0; e < 2; e++)
  {
    OLP(5 + 4 * e);
    if(tid == 0)
    {
      const P2d front = S.outer[e], back = S.outer[2 + e];
      const int yStep = 10;
      int left = (int)((front.x < back.x ? front.x : back.x) - xStep); // detectEdge (:681-697)
      int right = (int)((front.x < back.x ? back.x : front.x) + xStep);
      int yStart = (int)(front.y - yStep);
      int yEnd = (int)(back.y + yStep);
      if(left < 0)
        left = 0;
      if(right >= W)
        right = W - 1;
      if(yStart >= H)
        yStart = H - 1;
      if(yEnd < 0)
        yEnd = 0;
      S.ve_go = !(yStart < yEnd) && right > left && left < W && yStart >= 0;
      S.ve_left = left;
      S.ve_right = right;
      S.ve_ystart = yStart;
      S.ve_yend = yEnd;
      S.vn = 0;
    }
    __syncthreads();
    if(S.ve_go)
    {
      const int left = S.ve_left, right = S.ve_right, yStart = S.ve_ystart, yEnd = S.ve_yend;
      const int nrows = (yStart - yEnd) / 10 + 1;
      // window: left edge scans x in [left, right-1] ascending; right edge scans x in [left+1, right] descending
      // (VerticalEdgePointsDetector, :243-312)
      const int x0 = e == 0 ? left : left + 1, x1 = e == 0 ? right - 1 : right;
      const int w0 = x0 >> 5, w1 = x1 >> 5;
      for(int r = warp; r < nrows && r < OutlineShared::MAX_VPTS; r += nwarps)
      {
        const int y = yStart - r * 10;
        int fx = -1;
        if(e == 0)
        {
          for(int wb = w0; wb <= w1 && fx < 0; wb += 32)
          {
            const int w = wb + lane;
            unsigned v = w <= w1 ? closed_word(p, bd, y, w) : 0u;
            if(w == w0)
              v &= 0xffffffffu << (x0 & 31);
            if(w == w1 && (x1 & 31) != 31)
              v &= (1u << ((x1 & 31) + 1)) - 1u;
            const unsigned m = __ballot_sync(0xffffffffu, v != 0u);
            if(m)
            {
              const int src = __ffs(m) - 1;
              const unsigned vv = __shfl_sync(0xffffffffu, v, src);
              fx = ((wb + src) << 5) + __ffs(vv) - 1;
            }
          }
        }
        else
        {
          for(int wb = w1; wb >= w0 && fx < 0; wb -= 32)
          {
            const int w = wb - lane;
            unsigned v = w >= w0 ? closed_word(p, bd, y, w) : 0u;
            if(w == w0)
              v &= 0xffffffffu << (x0 & 31);
            if(w == w1 && (x1 & 31) != 31)
              v &= (1u << ((x1 & 31) + 1)) - 1u;
            const unsigned m = __ballot_sync(0xffffffffu, v != 0u);
            if(m)
            {
              const int src = __ffs(m) - 1; // lowest lane = highest word
              const unsigned vv = __shfl_sync(0xffffffffu, v, src);
              fx = ((wb - src) << 5) + 31 - __clz(vv);
            }
          }
        }
        if(lane == 0)
        {
          S.vfound[r] = fx >= 0;
          S.vpts[r].x = fx;
          S.vpts[r].y = y;
        }
      }
      __syncthreads();
      OLP(6 + 4 * e);
      if(tid == 0)
      {
        // compact in probing order (top of the list = yStart)
        int n = 0;
        const int lim = nrows < OutlineShared::MAX_VPTS ? nrows : OutlineShared::MAX_VPTS;
        for(int r = 0; r < lim; r++)
          if(S.vfound[r])
          {
            S.vpts[n] = S.vpts[r];
            n++;
          }
        S.vn = n;
        for(int i = 0; i < n; i++)
          S.vdist[i] = fabs(S.vpts[i].x * S.base.a + S.vpts[i].y * S.base.b + S.base.c); // comparableDistance (:397-400)
        S.best_pt = -1;
      }
      __syncthreads();
      OLP(7 + 4 * e);
      // findBestPoint (:708-728): element of rank 2n/3 by distance (ties: list order)
      const int n = S.vn;
      if(n > 0)
      {
        const int want = 2 * n / 3;
        for(int i = tid; i < n; i += nthreads)
        {
          const double di = S.vdist[i];
          int rank = 0;
          for(int j = 0; j < n; j++)
          {
            const double dj = S.vdist[j];
            rank += (dj < di) || (dj == di && j < i);
          }
          if(rank == want)
            S.best_pt = i;
        }
      }
      __syncthreads();
      OLP(8 + 4 * e);
      if(tid == 0 && S.vn > 0 && S.best_pt >= 0)
      {
        const P2id bp = S.vpts[S.best_pt];
        LineDd edge; // Line::parallel (:367-371)
        edge.a = S.base.a;
        edge.b = S.base.b;
        edge.c = -S.base.a * bp.x - S.base.b * bp.y;
        P2d c;
        // Corners (:738-750): front with lines 0/1, back with lines 2/3
        if(lined_intersection(edge, lined_from_i(S.line[e]), c))
          quad[e] = c;
        if(lined_intersection(edge, lined_from_i(S.line[2 + e]), c))
          quad[2 + e] = c;
      }
    }
    __syncthreads();
  }
  OLP(13);
  if(tid == 0)
    valid = quad_is_convex(quad);
}

// BottomScanner::scan + detectFrontEdge after the close (segmentation.cpp:169-241, 890-904). Block-cooperative;
// thread 0 gets the result.
template<class OutlineShared>
__device__ inline void detect_front_edge_block(const DevParams &p, const Band &bd, OutlineShared &S, P2d &left, P2d &right, int &valid, int tid,
                                               int nthreads)
{
  const int W = p.W, H = p.H;
  const int lane = tid & 31, warp = tid >> 5, nwarps = nthreads >> 5;
  const int xStep = 50, xCenter = W / 2;
  // all candidate columns x = xCenter + j*50 for j in [-jl, jr]
  const int jr = (W - 1 - xCenter) / xStep, jl = xCenter / xStep;
  const int ncols = jl + jr + 1;
  {
    constexpr int G = SSD_OL_PROBE_G; // columns a warp probes at once
    for(int c0 = warp * G; c0 < ncols; c0 += nwarps * G)
    {
      int x[G], yf[G], ys[G];
      bool f[G];
      const int nv = min(G, ncols - c0);
#pragma unroll
      for(int g = 0; g < G; g++)
        x[g] = xCenter + (c0 + g - jl) * xStep;
      // probeBottomUp (:225-240): lowest set pixel with y > H/2
      probe_columns<G>(p, bd, x, nv, H / 2 + 1, H - 1, lane, yf, ys, f);
      if(lane < nv)
      {
#pragma unroll
        for(int g = 0; g < G; g++)
          if(lane == g)
          {
            S.scan_found[c0 + g] = f[g];
            S.scan_ys[c0 + g] = ys[g];
          }
      }
    }
  }
  __syncthreads();
  if(tid == 0)
  {
    // scan order (:177-221): first hit to the right of the centre (incl.), else to the left; then the
    // contiguous run right of it, then the contiguous run left of it
    int n = 0, start = -1;
    for(int c = jl; c < ncols; c++)
      if(S.scan_found[c])
      {
        start = c;
        break;
      }
    if(start < 0)
      for(int c = jl - 1; c >= 0; c--)
        if(S.scan_found[c])
        {
          start = c;
          break;
        }
    if(start >= 0)
    {
      auto push = [&](int c)
      {
        S.frontLeft[n].x = xCenter + (c - jl) * xStep;
        S.frontLeft[n].y = S.scan_ys[c];
        n++;
      };
      push(start);
      for(int c = start + 1; c < ncols && S.scan_found[c]; c++)
        push(c);
      for(int c = start - 1; c >= 0 && S.scan_found[c]; c--)
        push(c);
    }
    S.nLeft = n;
  }
  __syncthreads();
  valid = 0;
  left.x = left.y = right.x = right.y = 0;
  const int n = S.nLeft;
  if(n < 2)
    return;
  {
    const P2id *const lists[4] = { S.frontLeft, S.frontLeft, S.frontLeft, S.frontLeft };
    const int ns[4] = { n, 0, 0, 0 };
    best_lines_block<OutlineShared::MAX_LPTS>(lists, ns, S.wk, S.line, tid, nthreads);
  }
  if(tid == 0)
  {
    const FlatLineD edge = flat_from(S.line[0]);
    int lo = 0, hi = 0; // ranges::minmax by x (:897-900)
    for(int i = 1; i < n; i++)
    {
      if(S.frontLeft[i].x < S.frontLeft[lo].x)
        lo = i;
      if(!(S.frontLeft[i].x < S.frontLeft[hi].x))
        hi = i;
    }
    left = flat_point(edge, S.frontLeft[lo].x);
    right = flat_point(edge, S.frontLeft[hi].x);
    valid = 1;
  }
}

// Band descriptor of one bitmap: shared memory if the touched rows fit, else the global bitmap itself.
__device__ inline bool band_setup(const DevParams &p, Band &bd, int row_min, int row_max, unsigned *smem_words, size_t smem_cap_words,
                                  const unsigned *gbitmap)
{
  bd.b0 = max(0, row_min - 2);
  const int b1 = min(p.H - 1, row_max + 2);
  bd.nb = b1 - bd.b0 + 1;
  const int rs = p.wpr + 1; // +1 word: conflict-free column probing
  if((size_t)bd.nb * rs <= smem_cap_words)
  {
    bd.rs = rs;
    bd.A = smem_words;
    return true;
  }
  bd.rs = p.wpr;
  bd.A = gbitmap + (size_t)bd.b0 * p.wpr;
  return false;
}

__device__ inline void band_clear_global(const DevParams &p, const Band &bd, unsigned *g, int tid, int nthreads)
{
  unsigned *base = g + (size_t)bd.b0 * p.wpr;
  for(int i = tid; i < bd.nb * p.wpr; i += nthreads)
    base[i] = 0u;
}

// the rest of detectStairSteps after the outlines (k_frame_logic below; also the tail of k_outline's fused variant)
struct FrameLogicScratch
{
  QuadTestDev qt[SSD_GPU_MAX_PLATEAUS];
  double gq[4][2];
};

// one warp, one lane per plateau; Sc: the warp's scratch in shared memory
__device__ inline void frame_logic_warp(const DevParams &p, FrameDev &F, FrameLogicScratch &Sc, int lane)
{
  QuadTestDev *s_qt = Sc.qt;
  double(*s_gq)[2] = Sc.gq;
  const int K = F.n_plateaus, ground = F.ground_index;
  const bool myValid = lane < K && lane >= F.first_outlined && F.plat[lane].valid;
  const unsigned vm = __ballot_sync(0xffffffffu, myValid);
  const int firstValid = vm ? __ffs(vm) - 1 : -1;
  if(lane == 0)
    F.first_valid = firstValid;
  if(firstValid < 0)
    return;
  if(lane == 0 && ground >= 0)
  {
    const double(*q)[2] = F.plat[firstValid].quad_world;
    const double yMin = p.y_min;
    if(q[0][1] < q[1][1])
    {
      s_gq[0][0] = q[0][0];
      s_gq[1][0] = q[1][0] + (q[1][1] - yMin) * (q[1][1] - q[0][1]) / (q[1][0] - q[0][0]); // calcDx(q0,q1)
    }
    else
    {
      s_gq[0][0] = q[0][0] + (q[0][1] - yMin) * (q[0][1] - q[1][1]) / (q[0][0] - q[1][0]); // calcDx(q1,q0)
      s_gq[1][0] = q[1][0];
    }
    s_gq[0][1] = yMin;
    s_gq[1][1] = yMin;
    s_gq[2][0] = q[0][0];
    s_gq[2][1] = q[0][1];
    s_gq[3][0] = q[1][0];
    s_gq[3][1] = q[1][1];
  }
  __syncwarp();
  const bool emit = myValid || (lane == ground && ground >= 0);
  if(emit)
  {
    PlateauDev &P = F.plat[lane];
    P2d q[4];
    for(int c = 0; c < 4; c++)
    {
      if(lane == ground)
      {
        q[c].x = s_gq[c][0];
        q[c].y = s_gq[c][1];
        P.quad_world[c][0] = q[c].x;
        P.quad_world[c][1] = q[c].y;
      }
      else
      {
        q[c].x = P.quad_world[c][0];
        q[c].y = P.quad_world[c][1];
      }
    }
    quadtest_init(s_qt[lane], q);
    quadtest_inner_box(s_qt[lane], q);
    quadfilter_build(F.qf[lane], s_qt[lane], p.Tf, p.epsc);
    P.valid = 1;
    P.quad_status = s_qt[lane].status;
  }
  const unsigned em = __ballot_sync(0xffffffffu, emit);
  const unsigned bad = __ballot_sync(0xffffffffu, emit && s_qt[lane].status != 0);
  if(lane == 0)
    F.quad_amask = em & ~bad;
  __syncwarp();
  // coalesced copy of the emitted tests to global memory
  for(int k = 0; k < K; k++)
    if(em >> k & 1u)
    {
      const unsigned *src = reinterpret_cast<const unsigned *>(&s_qt[k]);
      unsigned *dst = reinterpret_cast<unsigned *>(&F.plat[k].qt);
      for(int i = lane; i < (int)(sizeof(QuadTestDev) / 4); i += 32)
        dst[i] = src[i];
    }
  if(lane == 0 && bad)
    F.status |= SSD_STATUS_DEGENERATE_QUAD;
}

// ---------------------------------------------------------------------------------------------
// k_outline: grid = (SSD_GPU_MAX_PLATEAUS, frames); one block per outlined plateau
// (loop B of detectStairSteps, pointcloud.cpp:419-429, incl. imgPointsToWorld :476-487)
// ---------------------------------------------------------------------------------------------
#ifndef SSD_OL_MINB
#define SSD_OL_MINB 6
#endif
// FUSE_LOGIC (small batches: latency matters, not occupancy): the last block of a frame to finish runs the frame logic
// (k_frame_logic) itself -- one launch and one kernel boundary less on the single-frame path.
template<class OutlineShared, bool FUSE_LOGIC = false, class CAM = NoCam>
__global__ void __launch_bounds__(OutlineShared::THREADS, FUSE_LOGIC ? 1 : (OutlineShared::MINB ? OutlineShared::MINB : SSD_OL_MINB)) k_outline(const __grid_constant__ DevParams p0, FrameDev *__restrict__ frames,
                                                             unsigned *__restrict__ bev, size_t bm_words, size_t smem_cap_words,
                                                             const CAM cam = CAM())
{
  extern __shared__ __align__(16) unsigned s_words[];
  __shared__ OutlineShared S;
  __shared__ Band bd;
  __shared__ int s_smem_path;
  const int frame = blockIdx.y, tid = threadIdx.x;
  const DevParams &p = frame_params(p0, cam, frame);
  FrameDev &F = frames[frame];
  // grid.x blocks per frame walk the frame's outlined plateaus (first_outlined .. n_plateaus-1, k_peaks); grid.x is
  // smaller than SSD_GPU_MAX_PLATEAUS because a frame rarely has more than a handful (ssd_gpu.cu, launch_chain)
  const int n_plat = F.n_plateaus;
  for(int k = max(F.first_outlined, 0) + (int)blockIdx.x; k < n_plat; k += (int)gridDim.x)
  {
  if(!F.plat[k].outlined)
    continue;
  PlateauDev &P = F.plat[k];
  P2d quad[4];
  int valid = 0;
  if(P.row_max >= 0)
  {
    unsigned *gb = bev + ((size_t)frame * SSD_GPU_MAX_PLATEAUS + k) * bm_words;
    OLP(0);
    if(tid == 0)
      s_smem_path = band_setup(p, bd, P.row_min, P.row_max, s_words, smem_cap_words, gb);
    __syncthreads();
    if(s_smem_path)
      band_stage(p, s_words, bd, gb, tid, OutlineShared::THREADS);
    detect_outline_block(p, bd, S, p.min_img_y_extent, p.xy_ratio, quad, valid, tid, OutlineShared::THREADS);
    if(!s_smem_path)
    {
      __syncthreads();
      band_clear_global(p, bd, gb, tid, OutlineShared::THREADS);
    }
  }
  else if(tid == 0)
  {
    for(int i = 0; i < 4; i++)
      quad[i].x = quad[i].y = 0;
  }
  if(tid == 0)
  {
    for(int c = 0; c < 4; c++)
    {
      P.quad_px[c][0] = quad[c].x;
      P.quad_px[c][1] = quad[c].y;
      const P2d w = image_to_world(p, quad[c]);
      P.quad_world[c][0] = w.x;
      P.quad_world[c][1] = w.y;
    }
    P.valid = valid;
  }
#ifdef SSD_OL_PROF
  if(tid == 0 && blockIdx.y == 0 && blockIdx.x == 0)
  {
    g_olp[14] = clock64();
    printf("[ol prof] plateau %d band rows %d:", k, bd.nb);
    for(int i = 1; i <= 14; i++)
      printf(" %lld", g_olp[i] - g_olp[i - 1]);
    printf("\n");
  }
#endif
  __syncthreads(); // the shared band / work area is reused by the next plateau of this block
  }
  if(FUSE_LOGIC)
  {
    __shared__ FrameLogicScratch Sc;
    __shared__ unsigned s_last;
    __threadfence();
    __syncthreads();
    if(tid == 0)
      s_last = atomicAdd(&F.ol_done, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if(s_last && tid < 32)
    {
      __threadfence();
      frame_logic_warp(p, F, Sc, tid);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// k_frame_logic: the rest of detectStairSteps (pointcloud.cpp:427-443): first valid plateau, the ground
// quadrilateral (calcGroundQuadrilateral, :489-512) and one QuadrilateralTest per emitted step.
// One warp per frame, one lane per plateau.
// ---------------------------------------------------------------------------------------------
template<class CAM = NoCam>
__global__ void __launch_bounds__(32) k_frame_logic(const __grid_constant__ DevParams p0, FrameDev *__restrict__ frames, int n_frames,
                                                    const CAM cam = CAM())
{
  __shared__ FrameLogicScratch Sc;
  const int f = blockIdx.x;
  if(f >= n_frames)
    return;
  const DevParams &p = group_params(p0, cam, f);
  frame_logic_warp(p, frames[f], Sc, threadIdx.x);
}

// drawStairStep (pointcloud.cpp:588-597) of one step corner q: quadriWorld -> worldToCamera (b, a_inv) -> the lens, if any (nullptr:
// the pin-hole) -> DepthFrame::project (intrinsics)
__device__ __forceinline__ void overlay_corner(const double *q, const double *b, const OverlayDev &ov, const ssd_gpu_distortion *lens, float *px)
{
  const double dx = q[0] - b[0], dy = q[1] - b[1], dz = q[2] - b[2];
  const float X = (float)((ov.a_inv[0] * dx + ov.a_inv[1] * dy) + ov.a_inv[2] * dz);
  const float Y = (float)((ov.a_inv[3] * dx + ov.a_inv[4] * dy) + ov.a_inv[5] * dz);
  const float Z = (float)((ov.a_inv[6] * dx + ov.a_inv[7] * dy) + ov.a_inv[8] * dz);
  float x = __fdiv_rn(X, Z), y = __fdiv_rn(Y, Z);
  if(lens)
  {
    const ssd_gpu_distortion d = *lens;
    float xd, yd;
    ssd_lens_project(&d, x, y, &xd, &yd);
    x = xd;
    y = yd;
  }
  px[0] = __fadd_rn(__fmul_rn(x, ov.fx), ov.ppx);
  px[1] = __fadd_rn(__fmul_rn(y, ov.fy), ov.ppy);
}
// A group's steps into the overlay of every member frame, each through its own camera (b, a_inv, intrinsics, lens[camera]).
__device__ __forceinline__ void group_overlay(const GroupTable &g, const ssd_gpu_distortion *lens, int slot, const double (*sq)[4][3], int nSteps,
                                              ssd_gpu_overlay *__restrict__ overlay)
{
  const int2 m = group_members(g, slot);
  for(int i = 0; i < m.y; i++)
  {
    const int frame = m.x + i - g.cams.frame0; // within the launch
    const int c = frame_camera(g.cams, frame);
    double b[3];
    for(int j = 0; j < 3; j++)
      b[j] = g.cams.params[c].b[j];
    const OverlayDev &ov = g.cams.ov[c];
    ssd_gpu_overlay *Q = overlay + (size_t)frame * SSD_GPU_MAX_STEPS;
    for(int s = 0; s < nSteps; s++)
      for(int k = 0; k < 4; k++)
        overlay_corner(sq[s][k], b, ov, lens ? lens + c : nullptr, Q[s].px[k]);
  }
}
__device__ __forceinline__ const ssd_gpu_distortion *frame_lens(const ssd_gpu_distortion *lens, const NoCam &, int)
{
  return lens;
}
__device__ __forceinline__ const ssd_gpu_distortion *frame_lens(const ssd_gpu_distortion *lens, const CamTable &c, int frame)
{
  return lens ? lens + frame_camera(c, frame) : nullptr;
}

// ---------------------------------------------------------------------------------------------
// k_finalize: calcGround's front edge (pointcloud.cpp:531-547), calcStairStep (:549-558), the result
// assembly of detectStairs with ToExternalWorld (:370-383, transformation.cpp:190-194).
// grid = frames, one block per frame. ov_lens: the lenses the overlay projects through (plain calls: [0], camera and group calls: per
// camera), or nullptr: the pin-hole.
// ---------------------------------------------------------------------------------------------
template<class OutlineShared, class CAM = NoCam>
__global__ void __launch_bounds__(SSD_OL_THREADS, SSD_OL_MINB) k_finalize(const __grid_constant__ DevParams p0, FrameDev *__restrict__ frames,
                                                              FrameOut *__restrict__ out, unsigned *__restrict__ bev, size_t bm_words,
                                                              size_t smem_cap_words, const __grid_constant__ OverlayDev ov0,
                                                              ssd_gpu_overlay *__restrict__ overlay, const ssd_gpu_distortion *ov_lens,
                                                              const CAM cam = CAM())
{
  extern __shared__ __align__(16) unsigned s_words[];
  __shared__ OutlineShared S;
  __shared__ Band bd;
  __shared__ int s_smem_path;
  const int frame = blockIdx.x, tid = threadIdx.x;
  const DevParams &p = group_params(p0, cam, frame);
  const OverlayDev &ov = frame_overlay(ov0, cam, frame);
  FrameDev &F = frames[frame];
  FrameOut &O = out[frame];
  const int K = F.n_plateaus, ground = F.ground_index, firstValid = F.first_valid;

  P2d fl, fr;
  int frontValid = 0;
  const bool groundStep = firstValid >= 0 && ground >= 0 && F.plat[ground].quad_status == 0;
  if(groundStep)
  {
    PlateauDev &G = F.plat[ground];
    if(G.row_max >= 0)
    {
      unsigned *gb = bev + ((size_t)frame * SSD_GPU_MAX_PLATEAUS + ground) * bm_words;
      if(tid == 0)
        s_smem_path = band_setup(p, bd, G.row_min, G.row_max, s_words, smem_cap_words, gb);
      __syncthreads();
      if(s_smem_path)
        band_stage(p, s_words, bd, gb, tid, SSD_OL_THREADS);
      detect_front_edge_block(p, bd, S, fl, fr, frontValid, tid, SSD_OL_THREADS);
      if(!s_smem_path)
      {
        __syncthreads();
        band_clear_global(p, bd, gb, tid, SSD_OL_THREADS);
      }
    }
  }
  if(tid != 0)
    return;

  unsigned status = F.status;
  int nSteps = 0;
  double sq[SSD_GPU_MAX_STEPS][4][3];
  if(firstValid >= 0)
  {
    for(int i = 0; i < K; i++)
    {
      PlateauDev &P = F.plat[i];
      if(P.valid && P.quad_status == 0)
      {
        // calcAverageZ (:574-581) from the z_fix_u sum, which is order independent
        const double n_pp = (double)P.n_in_quad;
        const double zs = ((double)P.sum_fix - n_pp * (double)SSD_ZFIX_BIAS) / (double)(1u << p.zshift);
        P.mean_z = zs / n_pp;
      }
    }
    if(groundStep)
    {
      PlateauDev &G = F.plat[ground];
      G.front_valid = frontValid;
      double(*s)[3] = sq[nSteps++];
      if(frontValid)
      {
        const P2d wl = image_to_world(p, fl), wr = image_to_world(p, fr);
        const LineDd frontLine = lined_from_pts(wl, wr);
        P2d g0, g1, g2, g3;
        g0.x = G.quad_world[0][0];
        g0.y = G.quad_world[0][1];
        g1.x = G.quad_world[1][0];
        g1.y = G.quad_world[1][1];
        g2.x = G.quad_world[2][0];
        g2.y = G.quad_world[2][1];
        g3.x = G.quad_world[3][0];
        g3.y = G.quad_world[3][1];
        const P2d frontLeft = line_intersection_plain(frontLine, lined_from_pts(g0, g2));
        const P2d frontRight = line_intersection_plain(frontLine, lined_from_pts(g1, g3));
        s[0][0] = frontLeft.x;
        s[0][1] = frontLeft.y;
        s[1][0] = frontRight.x;
        s[1][1] = frontRight.y;
        s[2][0] = g2.x;
        s[2][1] = g2.y;
        s[3][0] = g3.x;
        s[3][1] = g3.y;
        for(int c = 0; c < 4; c++)
          s[c][2] = G.mean_z;
        if(G.n_in_quad == 0)
          status |= SSD_STATUS_EMPTY_MEAN;
      }
      else
      {
        for(int c = 0; c < 4; c++)
          s[c][0] = s[c][1] = s[c][2] = 0; // return{} (:546)
        status |= SSD_STATUS_INVALID_FRONT_EDGE;
      }
    }
    for(int i = firstValid; i < K; i++)
    {
      const PlateauDev &P = F.plat[i];
      if(!P.valid || P.quad_status != 0)
        continue;
      double(*s)[3] = sq[nSteps++];
      for(int c = 0; c < 4; c++)
      {
        s[c][0] = P.quad_world[c][0];
        s[c][1] = P.quad_world[c][1];
        s[c][2] = P.mean_z;
      }
      if(P.n_in_quad == 0)
        status |= SSD_STATUS_EMPTY_MEAN;
    }
  }
  if(nSteps == 0)
    status |= SSD_STATUS_NO_STEPS;
  for(int s = 0; s < nSteps; s++)
  {
    for(int c = 0; c < 4; c++)
    {
      const double x = sq[s][c][0], y = sq[s][c][1];
      O.steps[s].quad[c][0] = (p.ext_a[0] * x + p.ext_a[1] * y) + p.ext_b[0];
      O.steps[s].quad[c][1] = (p.ext_a[2] * x + p.ext_a[3] * y) + p.ext_b[1];
    }
    O.steps[s].height = p.ext_z + sq[s][0][2];
  }
  if constexpr(std::is_same<CAM, GroupTable>::value)
  {
    if(ov.enabled)
      group_overlay(cam, ov_lens, frame, sq, nSteps, overlay);
  }
  else if(ov.enabled)
  {
    ssd_gpu_overlay *Q = overlay + (size_t)frame * SSD_GPU_MAX_STEPS;
    const ssd_gpu_distortion *lens = frame_lens(ov_lens, cam, frame);
    for(int s = 0; s < nSteps; s++)
      for(int c = 0; c < 4; c++)
        overlay_corner(sq[s][c], p.b, ov, lens, Q[s].px[c]);
  }
  F.n_steps = nSteps;
  F.status = status;
  O.info.status = status;
  O.info.n_bins = p.n_bins;
  O.info.n_plateaus = K;
  O.info.ground_index = ground;
  O.info.first_valid_index = firstValid;
  O.info.n_steps = nSteps;
  O.info.n_nonzero = F.n_nonzero + group_extra_points(cam, frame, (unsigned)p.N);
  O.info.n_in_range = F.n_in_range + group_extra_points(cam, frame, (unsigned)p.N);
  O.n_exact_bin = F.n_exact_bin;
  {
    // points tested against a quadrilateral: every point of the ground and of the valid plateaus (k_quad_reduce)
    unsigned nq = 0;
    if(firstValid >= 0)
      for(int i = 0; i < K; i++)
        if((F.quad_amask >> i) & 1u)
          nq += F.plat[i].n_points;
    O.n_quad_pts = nq;
  }
  O.n_def_quad = F.n_def_quad;
  O.n_def_bev = F.n_def_bev;
}
