// nq_gilbert.h -- the generalized Hilbert visiting order (GilbertCurve.java:282-334, 356-365) as a function of the curve
// position: no stack and no walk, so every position of every image can be computed by its own thread (k_gilbert_order in
// nq_api.cu), and the host entry nq_gilbert_order computes the same table.
#pragma once
#include "nq_math.h"   // NQ_HD

namespace nq {

NQ_HD int gsgn(int v) { return (v > 0) - (v < 0); }
NQ_HD int gabs(int v) { return v < 0 ? -v : v; }

// (x, y) of the n-th pixel (0 <= n < w*h) that the reference's generate2d visits on a w x h image. Descends the recursion
// of generate2d: a node's children cover |a| x |b| pixel rectangles in the order the reference visits them, so the child
// that holds n is the first whose pixel count exceeds what is left of n. The odd-size adjustments of ax2 / bx2 are the
// reference's. Depth: about 2 log2(max(w, h)).
NQ_HD void gilbert_xy(int w, int h, unsigned long long n, int* px, int* py) {
  typedef unsigned long long u64;
  int x = 0, y = 0, ax, ay, bx, by;
  if (w >= h) { ax = w; ay = 0; bx = 0; by = h; }
  else { ax = 0; ay = h; bx = w; by = 0; }
  for (;;) {
    const int W = gabs(ax + ay), H = gabs(bx + by);
    const int dax = gsgn(ax), day = gsgn(ay), dbx = gsgn(bx), dby = gsgn(by);
    if (H == 1) { x += dax * (int)n; y += day * (int)n; break; }
    if (W == 1) { x += dbx * (int)n; y += dby * (int)n; break; }
    int ax2 = ax / 2, ay2 = ay / 2, bx2 = bx / 2, by2 = by / 2;
    const int w2 = gabs(ax2 + ay2), h2 = gabs(bx2 + by2);
    if (2 * W > 3 * H) {
      if ((w2 % 2) != 0 && W > 2) { ax2 += dax; ay2 += day; }
      const u64 c1 = (u64)gabs(ax2 + ay2) * (u64)H;                   // generate2d(x, y, ax2, ay2, bx, by)
      if (n < c1) { ax = ax2; ay = ay2; continue; }
      n -= c1;                                                         // generate2d(x + ax2, y + ay2, ax - ax2, ay - ay2, bx, by)
      x += ax2; y += ay2; ax -= ax2; ay -= ay2;
      continue;
    }
    if ((h2 % 2) != 0 && H > 2) { bx2 += dbx; by2 += dby; }
    const u64 c1 = (u64)gabs(bx2 + by2) * (u64)gabs(ax2 + ay2);       // generate2d(x, y, bx2, by2, ax2, ay2)
    if (n < c1) { const int tx = ax2, ty = ay2; ax = bx2; ay = by2; bx = tx; by = ty; continue; }
    n -= c1;
    const u64 c2 = (u64)W * (u64)gabs((bx - bx2) + (by - by2));      // generate2d(x + bx2, y + by2, ax, ay, bx - bx2, by - by2)
    if (n < c2) { x += bx2; y += by2; bx -= bx2; by -= by2; continue; }
    n -= c2;   // generate2d(x + (ax - dax) + (bx2 - dbx), y + (ay - day) + (by2 - dby), -bx2, -by2, -(ax - ax2), -(ay - ay2))
    x += (ax - dax) + (bx2 - dbx); y += (ay - day) + (by2 - dby);
    const int nbx = -(ax - ax2), nby = -(ay - ay2);
    ax = -bx2; ay = -by2; bx = nbx; by = nby;
  }
  *px = x; *py = y;
}

}  // namespace nq
