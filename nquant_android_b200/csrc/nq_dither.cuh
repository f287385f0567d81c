// nq_dither.cuh -- palette lookup + error-diffusion along the generalized Hilbert curve, and the
// blue-noise second pass.
// Reference: GilbertCurve (GC:50-373), BlueNoise.diffuse/dither (BN:180-222), nearestColorIndex /
// closestColorIndex (PQ:269-375, PL:329-474), dither() drivers (PQ:393-407, PL:492-522).
//
// The dither is a strictly serial chain along the curve: every pixel needs the quantization error
// of the previous one, the lookups share a first-seen memo when the key is the reduced 16-bit
// colour (PQ:271-274, PL:332-335) and the LAB lookup consumes a java.util.Random stream in visiting
// order (PL:467). One CTA per image: k_dither_fifo pairs a producer warp (pixel gather, and the palette
// lookups whenever they do not depend on the running error) with a consumer warp that owns the error
// recurrence; k_dither_sorted is the PriorityQueue mode. The cooperative per-pixel routines below
// (nearest_* / closest_* / dither_pixel) split a single lookup across the 32 lanes and are what the
// consumer falls back to when a lookup does read the diffused colour.
#pragma once
#include "nq_types.h"
#include "nq_color.h"
#include "nq_hist.cuh"
#include "nq_pnn.cuh"

namespace nq {

#define FULL 0xffffffffu

struct WarpShared {
  uint32_t pal[NQ_MAXK];
  float4 palLab[NQ_MAXK];     // alpha, L, A, B of palette[i] (getLab(c2), PL:352)
  double lut[256];            // gammaToLinear(v) (CL:71-75), copy of g_gammaLut
  signed char bn[4096];       // TELL_BLUE_NOISE (BN:13-178), copy of g_blueNoise
  // PnnLABQuantizer.closestColorIndex cost split per channel: T?[v] = cost of a channel difference of
  // |v| (see closest_lab); Ta only when the image is semi-transparent
  double Tr[256], Tg[256], Tb[256], Ta[256];
  // java.util.Random jump-ahead: seed after k more steps = jmpA[k] * seed + jmpC[k] (mod 2^48), k = 0..32
  unsigned long long jmpA[33], jmpC[33];
};
// java.util.PriorityQueue state of the sortedByYDiff mode (GC:87-94)
struct SortedShared {
  float q[16][4];             // backing array of ErrorBoxes
  double qy[16];              // their yDiff
  float w[8];                 // current weights[] (length 1, 3 or 7)
};

struct Env {
  WarpShared* sh;
  int plen, margin, thresold, DM, ditherMax;
  bool lab, dither, semi, hasTrans, isNano, sorted, useSal, gHasAlpha;
  uint32_t transColor;
  double PR, PG, PB, PA, ratio, gWeight, exp15;
  float beta;
  unsigned short* memo;
  unsigned short* mcache;     // optional shared-memory cache of memo (consumer warp of k_dither_fifo only)
  unsigned int* bits;         // pixelMap as a bit set (see NqSlot::bits), with its size counter
  unsigned int* distinct;
  const uint4* cells;         // candidate lists of the closest-colour scan, 32 B per 5-5-5 RGB cell (k_build_cells)
  JRandom rng;
  unsigned long long draws;
  int width;
};

__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(FULL, v, src); }

// (dist, idx) argmin across the warp, ties -> larger idx ("last minimal index wins", PQ:291-307)
__device__ __forceinline__ void warp_min_last(double& d, int& i) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    double d2 = __shfl_xor_sync(FULL, d, o);
    int i2 = __shfl_xor_sync(FULL, i, o);
    if (d2 < d || (d2 == d && i2 > i)) { d = d2; i = i2; }
  }
}

// nearestMap for reduced keys (PQ:271-274, PL:332-335): 65 536 x u16 in global memory, 0xFFFF = absent. An
// entry never changes once written, so the serial consumer may keep copies in a direct-mapped shared-memory
// cache (E.mcache: bits 0-8 = value + 1, bits 9-10 = key >> 14): a hit costs a shared load instead of a trip to L2.
__device__ __forceinline__ int memo_get(const Env& E, int key) {
  if (E.mcache) {
    const unsigned e = E.mcache[key & 0x3FFF];
    if ((e & 0x1FFu) != 0u && (e >> 9) == (unsigned)(key >> 14)) return (int)(e & 0x1FFu) - 1;
  }
  unsigned short got = 0;
  if (lane_id() == 0) got = E.memo[key];
  got = __shfl_sync(FULL, got, 0);
  if (got == 0xFFFF) return -1;
  if (E.mcache && lane_id() == 0) E.mcache[key & 0x3FFF] = (unsigned short)(((unsigned)(key >> 14) << 9) | ((unsigned)got + 1u));
  __syncwarp();
  return got;
}
__device__ __forceinline__ void memo_put(const Env& E, int key, int value) {
  if (lane_id() == 0) {
    E.memo[key] = (unsigned short)value;
    if (E.mcache) E.mcache[key & 0x3FFF] = (unsigned short)(((unsigned)(key >> 14) << 9) | ((unsigned)value + 1u));
  }
  __syncwarp();
}

// PnnQuantizer.nearestColorIndex (PQ:269-311)
__device__ int nearest_rgb(Env& E, uint32_t c) {
  const unsigned lane = lane_id();
  int offset = 0;
  if (E.isNano) {
    offset = color_index(c, E.semi, E.hasTrans);
    const int got = memo_get(E, offset);
    if (got >= 0) return got;
  }
  int k = 0;
  if (c_alpha(c) <= 0xF) c = E.transColor;
  if (E.plen > 2 && E.hasTrans && c_alpha(c) > 0xF) k = 1;
  double pr = E.PR, pg = E.PG, pb = E.PB, pa = E.PA;
  if (E.plen < 3) pr = pg = pb = pa = 1;
  const int ca = c_alpha(c), cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  double best = 1e300;
  int bi = -1;
  for (int i = k + lane; i < E.plen; i += 32) {
    const uint32_t c2 = E.sh->pal[i];
    double da = (double)(c_alpha(c2) - ca), dr = (double)(c_red(c2) - cr), dg = (double)(c_green(c2) - cg), db = (double)(c_blue(c2) - cb);
    double cur = pa * (da * da);
    cur += pr * (dr * dr);
    cur += pg * (dg * dg);
    cur += pb * (db * db);
    if (cur <= best) { best = cur; bi = i; }
  }
  warp_min_last(best, bi);
  if (!(best <= 2147483647.0) || bi < 0) bi = k;   // mindist starts at Integer.MAX_VALUE (PQ:286)
  if (E.isNano) memo_put(E, offset, bi);
  return bi;
}

// the two smallest (floor(err), index) pairs across the warp; the sequential top-2 scan of
// PQ:329-357 / PL:418-458 keeps exactly these (its comparisons are against truncated ints)
struct Top2 { int i0, i1, d0, d1; };
__device__ __forceinline__ bool t2_less(int da, int ia, int db, int ib) { return da < db || (da == db && ia < ib); }
__device__ __forceinline__ void t2_insert(Top2& t, int d, int i) {
  if (t2_less(d, i, t.d0, t.i0)) { t.d1 = t.d0; t.i1 = t.i0; t.d0 = d; t.i0 = i; }
  else if (t2_less(d, i, t.d1, t.i1)) { t.d1 = d; t.i1 = i; }
}
__device__ __forceinline__ void t2_reduce(Top2& t) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    int d0 = __shfl_xor_sync(FULL, t.d0, o), i0 = __shfl_xor_sync(FULL, t.i0, o);
    int d1 = __shfl_xor_sync(FULL, t.d1, o), i1 = __shfl_xor_sync(FULL, t.i1, o);
    t2_insert(t, d0, i0);
    t2_insert(t, d1, i1);
  }
}
// entries whose err truncates to Integer.MAX_VALUE are never stored (err < closest[] fails)
#define T2_NONE 0x7fffffff

// PnnQuantizer.closestColorIndex (PQ:313-375)
__device__ int closest_rgb(Env& E, uint32_t c, int pos) {
  if (c_alpha(c) <= 0xF) return nearest_rgb(E, c);
  const unsigned lane = lane_id();
  double pr = E.PR, pg = E.PG, pb = E.PB, pa = E.PA;
  if (E.plen < 3) pr = pg = pb = pa = 1;
  const int ca = c_alpha(c), cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  Top2 t = {1 << 30, 1 << 30, T2_NONE, T2_NONE};
  for (int k = lane; k < E.plen; k += 32) {
    const uint32_t c2 = E.sh->pal[k];
    double dr = (double)(c_red(c2) - cr), dg = (double)(c_green(c2) - cg), db = (double)(c_blue(c2) - cb);
    double err = pr * (dr * dr);
    err += pg * (dg * dg);
    err += pb * (db * db);
    if (E.semi) { double da = (double)(c_alpha(c2) - ca); err += pa * (da * da); }
    int d = j2i(err);
    if (d != T2_NONE) t2_insert(t, d, k);
  }
  t2_reduce(t);
  int c0 = t.d0 == T2_NONE ? 0 : t.i0, e0 = t.d0;
  int c1 = t.d1 == T2_NONE ? c0 : t.i1, e1 = t.d1;     // PQ:359-360
  int MAX_ERR = E.plen << 2;
  int idx = (pos + 1) % 2;
  if ((double)e1 * .67 < (double)(e1 - e0)) idx = 0;
  else if (c0 > c1) idx = pos % 2;
  const int ci = idx ? c1 : c0, ei = idx ? e1 : e0;
  if (ei >= MAX_ERR || (E.hasTrans && ci == 0)) return nearest_rgb(E, c);
  return ci;
}

// PnnLABQuantizer.nearestColorIndex (PL:329-404)
__device__ int nearest_lab(Env& E, uint32_t c) {
  const unsigned lane = lane_id();
  int offset = 0;
  if (E.isNano) {
    offset = color_index(c, E.semi, E.hasTrans);
    const int got = memo_get(E, offset);
    if (got >= 0) return got;
  }
  int k = 0;
  if (c_alpha(c) <= 0xF) c = E.transColor;
  if (E.plen > 2 && E.hasTrans && c_alpha(c) > 0xF) k = 1;
  const int ca = c_alpha(c), cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  const Lab4 l1 = lab_of(c);
  if (E.bits) {   // getLab(c) and, without semi-transparency, getLab(palette[i]) for every i >= k (PL:345-352)
    pixelmap_add(E.bits, E.distinct, c, lane == 0);
    for (int i0 = k; i0 < E.plen; i0 += 32) pixelmap_add(E.bits, E.distinct, i0 + (int)lane < E.plen ? E.sh->pal[i0 + lane] : 0u, i0 + (int)lane < E.plen);
  }
  int bi;
  if (E.plen > 4 && !(E.semi || E.plen < 16) && E.plen <= 32) {
    // CIEDE2000 branch (PL:376-395): R_T can be negative, so acceptance depends on the running
    // mindist; one palette entry per lane, resolved in index order
    const int i = k + lane;
    double g = 1e300, f = 1e300;
    if (i < E.plen) {
      const float4 l2 = E.sh->palLab[i];
      double cur = 0;   // hasSemiTransparency is false on this branch
      float tL = ciede_L(l1.L, l2.y);
      cur += (double)tL * (double)tL;
      g = cur;
      CiedeC cc;
      float tC = ciede_C(l1.A, l1.B, l2.z, l2.w, &cc);
      cur += (double)tC * (double)tC;
      g = cur > g ? cur : g;
      double barC, barh;
      float tH = ciede_H(l1.B, l2.w, cc, &barC, &barh);
      cur += (double)tH * (double)tH;
      g = cur > g ? cur : g;
      cur += (double)ciede_RT(barC, barh, tC, tH);
      g = cur > g ? cur : g;
      f = cur;
    }
    double mind = 2147483647.0;
    bi = k;
    unsigned remaining = FULL;
    for (;;) {
      unsigned m = __ballot_sync(FULL, g <= mind) & remaining;
      if (!m) break;
      int L = __ffs(m) - 1;
      mind = shfl_d(f, L);
      bi = k + L;
      remaining = (L == 31) ? 0u : ~((2u << L) - 1u);
    }
  } else {
    const double exp15 = E.exp15;
    double best = 1e300;
    bi = -1;
    for (int i = k + lane; i < E.plen; i += 32) {
      const uint32_t c2 = E.sh->pal[i];
      double cur = 0;
      if (E.semi) { double da = (double)(c_alpha(c2) - ca); cur = (da * da) / exp15; }
      if (E.plen <= 4) {
        double dr = (double)(c_red(c2) - cr), dg = (double)(c_green(c2) - cg), db = (double)(c_blue(c2) - cb);
        cur = (dr * dr) + (dg * dg) + (db * db);
        if (E.semi) { double da = (double)(c_alpha(c2) - ca); cur += da * da; }
      } else {
        const float4 l2 = E.sh->palLab[i];
        if (E.semi || E.plen < 16) {
          double d = (double)(l2.y - l1.L); cur += d * d;
          d = (double)(l2.z - l1.A); cur += d * d;
          d = (double)(l2.w - l1.B); cur += d * d;
        } else {
          cur += (double)fabsf(l2.y - l1.L);
          double da = (double)(l2.z - l1.A), db = (double)(l2.w - l1.B);
          cur += nqm::sqrt_((da * da) + (db * db));
        }
      }
      if (cur <= best) { best = cur; bi = i; }
    }
    warp_min_last(best, bi);
    if (!(best <= 2147483647.0) || bi < 0) bi = k;
  }
  if (E.isNano) memo_put(E, offset, bi);
  return bi;
}

// exact cost of palette entry c2 for colour c, in the reference's operation order (PL:421-446)
__device__ __forceinline__ double closest_lab_err(const Env& E, uint32_t c2, int ca, int cr, int cg, int cb) {
  const int ir = c_red(c2) - cr, ig = c_green(c2) - cg, ib = c_blue(c2) - cb;
  double dr = (double)ir, dg = (double)ig, db = (double)ib;
  double err = E.PR * (1 - E.ratio) * (dr * dr);
  err += E.PG * (1 - E.ratio) * (dg * dg);
  err += E.PB * (1 - E.ratio) * (db * db);
  if (E.semi) { double da = (double)(c_alpha(c2) - ca); err += E.PA * (da * da); }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    double t0 = (double)(c_coeffs[i][0] * (float)ir);   // float * int -> float (PL:437)
    err += E.ratio * (t0 * t0);
    double t1 = (double)(c_coeffs[i][1] * (float)ig);
    err += E.ratio * (t1 * t1);
    double t2 = (double)(c_coeffs[i][2] * (float)ib);
    err += E.ratio * (t2 * t2);
  }
  return err;
}
// per-channel cost tables for the fast scan: every term of closest_lab_err depends on ONE channel
// difference, and all terms are >= 0, so the reference's 12/13-term sequential double sum S and the
// regrouped sum A = Tr[|dr|] + Tg[|dg|] + Tb[|db|] (+ Ta[|da|]) agree to a few ulp:
// |S - A| <= 2e-14 * A. Only floor(S) enters the top-2 decision (see Top2), so A decides it unless A
// lies within 1e-6 (>> 2e-14 * 2^31) of an integer, in which case the exact S is evaluated.
__device__ __forceinline__ void closest_lab_table_entry(double PR, double PG, double PB, double PA, double ratio, bool semi, int v,
                                                        double* tr, double* tg, double* tb, double* ta) {
  const double dv = (double)v;
  double r = PR * (1 - ratio) * (dv * dv), g = PG * (1 - ratio) * (dv * dv), b = PB * (1 - ratio) * (dv * dv);
  for (int i = 0; i < 3; ++i) {
    double t0 = (double)(c_coeffs[i][0] * (float)v), t1 = (double)(c_coeffs[i][1] * (float)v), t2 = (double)(c_coeffs[i][2] * (float)v);
    r += ratio * (t0 * t0); g += ratio * (t1 * t1); b += ratio * (t2 * t2);
  }
  *tr = r; *tg = g; *tb = b;
  *ta = semi ? PA * (dv * dv) : 0.0;
}
__device__ void closest_lab_tables(const Env& E) {
  for (int v = lane_id(); v < 256; v += 32)
    closest_lab_table_entry(E.PR, E.PG, E.PB, E.PA, E.ratio, E.semi, v, &E.sh->Tr[v], &E.sh->Tg[v], &E.sh->Tb[v], &E.sh->Ta[v]);
  __syncwarp();
}

// PnnLABQuantizer.closestColorIndex (PL:406-474)
__device__ int closest_lab(Env& E, uint32_t c, int pos) {
  if (c_alpha(c) <= 0xF) return nearest_lab(E, c);
  const unsigned lane = lane_id();
  const int ca = c_alpha(c), cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  Top2 t = {1 << 30, 1 << 30, T2_NONE, T2_NONE};
  for (int k = lane; k < E.plen; k += 32) {
    const uint32_t c2 = E.sh->pal[k];
    double a = E.sh->Tr[abs(c_red(c2) - cr)] + E.sh->Tg[abs(c_green(c2) - cg)] + E.sh->Tb[abs(c_blue(c2) - cb)];
    if (E.semi) a += E.sh->Ta[abs(c_alpha(c2) - ca)];
    int d = j2i(a);
    const double fr = a - (double)d;
    if (fr < 1e-6 || fr > 1.0 - 1e-6) d = j2i(closest_lab_err(E, c2, ca, cr, cg, cb));
    if (d != T2_NONE) t2_insert(t, d, k);
  }
  t2_reduce(t);
  const int c0 = t.d0 == T2_NONE ? 0 : t.i0, e0 = t.d0;
  const int c1 = t.d1 == T2_NONE ? c0 : t.i1, e1 = t.d1;     // PL:460-461
  int idx = 1;
  if (e0 == 0) idx = 0;                                       // short-circuit: no draw (PL:467)
  else {
    int r = E.rng.next_int(32767);
    ++E.draws;
    int sum = (int)((unsigned)e1 + (unsigned)e0);
    if ((r % sum) <= e1) idx = 0;
  }
  const int ci = idx ? c1 : c0, ei = idx ? e1 : e0;
  int MAX_ERR = E.plen;
  if (ei >= MAX_ERR || ci == 0 || c_alpha(E.sh->pal[ci]) < ca) return nearest_lab(E, c);
  return ci;
}

// Ditherable.nearestColorIndex as bound by getDitherFn (PQ:377-391, PL:476-490)
__device__ __forceinline__ int lookup(Env& E, uint32_t c, int pos) {
  if (E.lab) return E.plen <= 4 ? nearest_lab(E, c) : closest_lab(E, c, pos);
  return E.dither ? nearest_rgb(E, c) : closest_rgb(E, c, pos);
}

// GilbertCurve.normalDistribution (GC:114-123)
__device__ float normal_distribution(float x, float peak) {
  const float mean = .5f, stdDev = .1f;
  double d = (double)(x - mean);
  double sd = (double)stdDev;
  double exponent = -(d * d) / (2 * (sd * sd));
  double pdf = (1 / (sd * nqm::sqrt_(2 * 3.141592653589793))) * nqm::nq_exp(exponent);
  double maxPdf = 1 / (sd * nqm::sqrt_(2 * 3.141592653589793));
  double scaledPdf = (pdf / maxPdf) * (double)peak;
  return (float)dmax(0.0, dmin((double)peak, scaledPdf));
}

// Y_Diff(pixel, c) with color2Y(pixel) already known (CL:215-227)
__device__ __forceinline__ double y_diff_pre(double ypix, uint32_t c, const double* lut) {
  return nqm::fabs_(color_y(c, lut) - ypix) * 100;
}

// GilbertCurve.ditherPixel (GC:125-185). qcur = qPixels[bidx] at the time of the call; sal =
// saliencies[bidx]; ypix = color2Y(pixel).
__device__ int dither_pixel(Env& E, int x, int y, int bidx, uint32_t pixel, float sal, double ypix, uint32_t c2, float beta, int qcur) {
  const int plen = E.plen, margin = E.margin;
  const double weight = E.gWeight;
  const uint32_t qcol = E.sh->pal[qcur];
  const signed char* bn = E.sh->bn;
  const double* lut = E.sh->lut;
  const int r_pix = c_red(c2), g_pix = c_green(c2), b_pix = c_blue(c2), a_pix = c_alpha(c2);
  const float strength = 1 / 3.f;
  const int acceptedDiff = max(2, plen - margin);
  if (plen <= 4 && sal > .2f && sal < .25f)
    c2 = bn_diffuse(pixel, qcol, beta * 2 / sal, strength, x, y, bn);
  else if (plen <= 4 || y_diff_pre(ypix, c2, lut) < (double)(2 * acceptedDiff)) {
    if (plen > 64) {
      float kappa = sal < .6f ? beta * .15f / sal : beta * .4f / sal;
      c2 = bn_diffuse(pixel, qcol, kappa, strength, x, y, bn);
    } else if (plen > 16 && weight < .005)
      c2 = bn_diffuse(pixel, qcol, beta * normal_distribution(sal, .5f) + beta, strength, x, y, bn);
    else
      c2 = bn_diffuse(pixel, qcol, beta * .5f / sal, strength, x, y, bn);
  }

  double gamma = (plen <= 32 && weight < .01 && weight > .007) ? (double)(1 - beta) : (double)beta;
  if (plen > 4 && y_diff_pre(ypix, c2, lut) > (gamma * acceptedDiff)) {
    if (margin > 6 || gamma > (double)beta) {
      float kappa = sal < .4f ? beta * .4f * sal : beta * .4f / sal;
      uint32_t c1 = c_argb(a_pix, r_pix, g_pix, b_pix);
      if (plen > 32 && (double)sal < .9)
        kappa = beta * normal_distribution(sal, 2.f);
      else {
        if (weight >= .0015 && (double)sal < .6) c1 = pixel;
        if (weight >= .005 && (double)sal < .6)
          kappa = beta * normal_distribution(sal, weight < .0008 ? 2.5f : 1.75f);
        else if (plen >= 32 || y_diff(c1, c2, lut) > (gamma * 3.141592653589793 * acceptedDiff)) {
          double ub = 1 - plen / 320.0;
          if ((double)sal > .15 && (double)sal < ub)
            kappa = beta * (!E.sorted && weight < .0025 ? .55f : .5f) / sal;
          else
            kappa = beta * normal_distribution(sal, weight < .0025 ? 1.82f : 2.f);
        }
      }
      c2 = bn_diffuse(c1, qcol, kappa, strength, x, y, bn);
    } else if (plen <= 32 && weight >= .004)
      c2 = bn_diffuse(c2, qcol, beta * normal_distribution(sal, .25f), strength, x, y, bn);
    else
      c2 = c_argb(a_pix, r_pix, g_pix, b_pix);
  }

  if (E.DM < 16 && plen > 4 && sal < .6f && y_diff_pre(ypix, c2, lut) > (double)(margin - 1))
    c2 = c_argb(a_pix, r_pix, g_pix, b_pix);
  if (plen > 32 && (double)sal > .95) {
    float kappa = beta * fmaxf(.05f, .75f - plen / 128.f) * sal;
    c2 = bn_diffuse(pixel, qcol, kappa, strength, x, y, bn);
  }
  return lookup(E, c2, bidx);
}

// (float) Math.tanh(x) for the error shaping (GC:255). The double result is only used after narrowing
// to float, so a plain-double evaluation t with relative error < 1e-13 decides the float whenever
// (float)(t(1-d)) == (float)(t(1+d)), d = 1e-12 (rounding is monotone); otherwise, and for |x| < 1
// where 1 - 2/(e^2x + 1) cancels, the double-double kernel runs. Same float as (float)nq_tanh(x).
__device__ __forceinline__ float tanh_to_float(double x) {
  const double ax = nqm::fabs_(x);
  if (ax >= 1.0 && ax < 22.0) {
    const double y = 2.0 * ax;
    const double fk = nqm::rint_(y * nqm::INV_LN2_32);
    const int kk = (int)fk;
    const double r = (y - fk * nqm::LN2_32_HI) - fk * nqm::LN2_32_LO;
    double p = 1.0 / 720.0;
    p = p * r + 1.0 / 120.0;
    p = p * r + 1.0 / 24.0;
    p = p * r + 1.0 / 6.0;
    p = p * r + 0.5;
    p = p * r + 1.0;
    p = p * r;                                     // expm1(r), |r| <= 0.011
    const double T = nqm::exp2_32_tab(kk & 31, 0);
    const double Ee = (T + T * p) * nqm::pow2i(kk >> 5);
    const double t = 1.0 - 2.0 / (Ee + 1.0);
    const float lo = (float)(t * (1.0 - 1e-12)), hi = (float)(t * (1.0 + 1e-12));
    if (lo == hi) return x < 0 ? -lo : lo;
  }
  return (float)nqm::nq_tanh(x);
}

// Straight-line variant for the serial chain: explicit fma, Estrin evaluation and a reciprocal instead of the
// division (the chain is latency bound; the decision logic is the same interval test, so the float it
// returns with `true` is again exactly (float)nq_tanh(x)). (float)tanh(x) == 1.0f for x >= 9.0109.
__device__ __forceinline__ bool tanh_fast(double x, float* out) {
  const double ax = nqm::fabs_(x);
  const double y = 2.0 * (ax < 9.5 ? ax : 9.5);
  const double fk = nqm::rint_(y * nqm::INV_LN2_32);
  const int kk = (int)fk;
  double r = __fma_rn(-fk, nqm::LN2_32_HI, y);
  r = __fma_rn(-fk, nqm::LN2_32_LO, r);
  const double r2 = r * r;
  const double u0 = __fma_rn(r, 1.0 / 6.0, 0.5), u1 = __fma_rn(r, 1.0 / 120.0, 1.0 / 24.0);
  const double u2 = __fma_rn(r2, 1.0 / 720.0, u1);
  const double q = __fma_rn(r2, u2, u0);
  const double p = __fma_rn(r2, q, r);                    // expm1(r), |r| <= 0.011
  const double T = nqm::exp2_32_tab(kk & 31, 0);
  const double Ee = __fma_rn(T, p, T) * nqm::pow2i(kk >> 5);
  // 1 / (Ee + 1) by two Newton steps from the hardware estimate: no special-case branch (Ee + 1 is in [8, 2^28]),
  // relative error ~2e-16, far inside the 1e-12 interval below
  const double d = Ee + 1.0;
  double rc;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(rc) : "d"(d));
  rc = __fma_rn(rc, __fma_rn(-d, rc, 1.0), rc);
  rc = __fma_rn(rc, __fma_rn(-d, rc, 1.0), rc);
  const double t = __fma_rn(-2.0, rc, 1.0);
  const float lo = (float)(t * (1.0 - 1e-12)), hi = (float)(t * (1.0 + 1e-12));
  const bool sat = ax >= 9.02;
  const float v = sat ? 1.0f : lo;
  *out = x < 0 ? -v : v;
  return sat || (ax >= 1.0 && lo == hi);
}

// -------------------------------------------------------------------------------------------------
// GilbertCurve constructor constants + initWeights (GC:50-112, 336-354), one thread per image
// -------------------------------------------------------------------------------------------------
__device__ void init_weights(float* weights, int size) {
  const float weightRatio = (float)nqm::nq_pow((double)(343.f + 1.f), (double)(1.f / ((float)size - 1.f)));
  float weight = 1.f, sumweight = 0.f;
  for (int c = 0; c < size; ++c) {
    sumweight += (weights[size - c - 1] = weight);
    weight /= weightRatio;
  }
  weight = 0.f;
  for (int c = 0; c < size; ++c) weight += (weights[c] /= sumweight);
  weights[0] += 1.f - weight;
}

__global__ void k_dither_setup(NqImage* imgs, const NqSlot* slots, int nimg) {
  int img = blockIdx.x * blockDim.x + threadIdx.x;
  if (img >= nimg) return;
  NqImage& I = imgs[img];
  if (I.nmax <= 2) {   // fixed palette (PQ:441-452)
    I.weight = 1;
    I.paletteLen = I.nmax;
    if (I.transIdx >= 0) { I.palette[0] = I.transColor; I.palette[1] = 0xFF000000u; }
    else { I.palette[0] = 0xFF000000u; I.palette[1] = 0xFFFFFFFFu; }
    if (I.nmax < 2) I.paletteLen = I.nmax < 0 ? 0 : I.nmax;
  }
  const int plen = I.paletteLen;
  const bool lab = I.kind == NQ_KIND_LAB;
  const double weight = I.hasSemi ? -I.weight : I.weight;   // PQ:396-397, PL:496-497
  // PnnQuantizer.nearestColorIndex tests the FIELD `weight > .015` while it carries the sign flip
  // (PQ:271 after PQ:396-397): a semi-transparent image always uses the reduced memo key there.
  // PnnLABQuantizer latched isNano inside pnnquan, before the flip (PL:180).
  if (!lab) I.isNano = !(weight > .015);
  // which saliency map exists (PL:135, PL:499-508)
  const bool salFromPnn = lab && I.nmax > 2 && I.nmax < 128;
  const bool salFromDither = lab && I.dither && !salFromPnn && (plen <= 256 || weight > .99);
  const bool sal = salFromPnn || salFromDither;
  I.gUseSal = sal;
  const bool hasAlpha = weight < 0;
  I.gHasAlpha = hasAlpha;
  I.gWeight = nqm::fabs_(weight);
  I.gMargin = weight < .0025 ? 12 : weight < .004 ? 8 : 6;
  const bool sorted = plen > 128 && weight >= .02 && (!hasAlpha || weight < .18);
  I.gSorted = sorted;
  float beta = plen > 4 ? (float)(.6f - .00625f * (float)plen) : 1.f;
  if (plen > 4) {
    double boundary = .005 - .0000625 * plen;
    beta = (float)(weight > boundary ? .25 : dmin(1.5, (double)beta + plen * weight));
    if (plen > 16 && plen <= 32 && weight < .003) beta += .075f;
    else if (weight < .0015 || (plen > 32 && plen < 256)) beta += .1f;
    if ((plen >= 64 && (weight > .012 && weight < .0125)) || (weight > .025 && weight < .03)) beta += .05f;
    else if (plen > 32 && plen < 64 && weight < .015) beta = .55f;
    else if (plen > 16 && plen <= 32 && weight <= .005) beta += (float)(.05 + weight * plen);
  } else
    beta *= .95f;
  if (plen > 64 || (plen > 4 && weight > .02)) beta *= .4f;
  if (plen > 64 && weight < .02) beta = .18f;
  int DM = weight < .015 ? ((weight > .0025) ? 25 : 16) : 9;
  if (weight > .99) { beta = (float)weight; DM = 25; }
  double edge = hasAlpha ? 1 : nqm::nq_exp(weight) - .25;
  double deviation = weight > .002 ? -.25 : 1;
  double sq = nqm::sqrt_((double)DM) + edge * deviation;
  int ditherMax = (hasAlpha || DM > 9) ? j2b(sq * sq) : j2b(DM * (sal ? 2.0 : 2.718281828459045));
  const int density = plen > 16 ? 3200 : 1500;
  if (plen / weight > 5000 && (weight > .045 || (weight > .01 && plen < 64))) ditherMax = j2b((5 + edge) * (5 + edge));
  else if (weight < .03 && plen / weight < density && plen >= 16 && plen < 256) ditherMax = j2b((5 + edge) * (5 + edge));
  I.gBeta = beta; I.gDitherMaxQ = DM; I.gDitherMax = ditherMax;
  I.gThresold = DM > 9 ? -112 : -64;
  init_weights(I.gWeights, DM);
  init_weights(I.gW1, 1);
  init_weights(I.gW3, 3);
  init_weights(I.gW7, 7);
  I.bnWeight = 1.0f;
  // PnnQuantizer: BlueNoise.dither's lookups (closestColorIndex, PQ:313-375) are pure per pixel except for the first-seen memo
  // of the nearestColorIndex fall-back: done by the per-pixel kernels k_bn_rgb_* after the Gilbert pass
  I.bnParallel = (!lab && !I.dither && plen > 32 && slots[img].idx != nullptr) ? 1 : 0;
  // pixelMap.size() is only tracked exactly when getLab's call pattern does not depend on the scan order (PL:347-349)
  if (lab && !I.dither && plen > 32 && I.hasSemi && !I.error) I.error = 4;
}

// -------------------------------------------------------------------------------------------------
// The serial pass: Gilbert-order error diffusion (GC:187-280), then BlueNoise.dither (BN:207-222)
// when dither == false and the palette has more than 32 entries. One warp per image.
//
// The warp walks the curve in blocks of 32 pixels. Everything that does not depend on the running
// error is gathered for a whole block at once, one pixel per lane, a block ahead of its use: the
// visiting order, the source pixel, its saliency (from the Lab table) and its luminance.
//
// Two kernels share the code below: k_dither_fifo for the ArrayDeque queue (sortedByYDiff == false)
// and k_dither_sorted for the PriorityQueue queue (GC:87-94). Each returns at once for images of the
// other mode.
// -------------------------------------------------------------------------------------------------
struct PixBlock { uint32_t xy, px; float sal; double ypix; };

__device__ __forceinline__ int chan(uint32_t c, int ch) {   // ErrorBox channel order r, g, b, a (GC:24-31)
  return (int)((c >> (ch == 3 ? 24 : 16 - 8 * ch)) & 0xFF);
}

struct DitherCtx {
  Env E;
  const uint32_t* in;
  uint32_t* out;
  int npix, width, fixA0;
  bool salReplaced;
};

// common prologue, register part: the constants of the GilbertCurve object
__device__ __forceinline__ void dither_prologue_regs(NqImage& I, const NqSlot& S, WarpShared& sh, DitherCtx& D) {
  Env& E = D.E;
  const int plen = I.paletteLen;
  E.sh = &sh;
  E.plen = plen; E.margin = I.gMargin; E.thresold = I.gThresold; E.DM = I.gDitherMaxQ; E.ditherMax = I.gDitherMax;
  E.lab = I.kind == NQ_KIND_LAB; E.dither = I.dither != 0; E.semi = I.hasSemi != 0; E.hasTrans = I.transIdx >= 0;
  E.isNano = I.isNano != 0; E.sorted = I.gSorted != 0; E.useSal = I.gUseSal != 0; E.gHasAlpha = I.gHasAlpha != 0;
  E.transColor = I.transColor;
  E.PR = I.PR; E.PG = I.PG; E.PB = I.PB; E.PA = I.PA; E.ratio = I.ratioMerge; E.gWeight = I.gWeight;
  E.exp15 = E.semi ? nqm::nq_exp(1.5) : 1.0;
  E.beta = I.gBeta;
  E.memo = S.memo;
  E.mcache = nullptr;
  E.cells = reinterpret_cast<const uint4*>(S.cells);
  E.bits = S.bits; E.distinct = &I.distinctColors;
  E.rng.set_seed(I.seed);
  E.draws = 0;
  E.width = I.width;
  D.in = S.in; D.out = S.out; D.npix = I.npix; D.width = I.width; D.fixA0 = I.fixA0;
  D.salReplaced = I.nmax < 128 && I.nmax > 2;   // which pixel feeds getLab for the saliency (PL:141-156 vs PL:503-506)
}
// ... and the shared tables (one warp)
__device__ __forceinline__ void dither_prologue(NqImage& I, const NqSlot& S, WarpShared& sh, DitherCtx& D) {
  dither_prologue_regs(I, S, sh, D);
  const unsigned lane = lane_id();
  Env& E = D.E;
  const int plen = I.paletteLen;
  for (int i = lane; i < 256; i += 32) sh.lut[i] = g_gammaLut[i];
  for (int i = lane; i < 4096; i += 32) sh.bn[i] = g_blueNoise[i];
  for (int i = lane; i < plen; i += 32) {
    uint32_t pc = I.palette[i];
    sh.pal[i] = pc;
    if (E.lab) { Lab4 l = lab_of(pc); sh.palLab[i] = make_float4(l.alpha, l.L, l.A, l.B); }
  }
  if (lane == 0) {
    unsigned long long a = 1ULL, c = 0ULL;
    const unsigned long long MASK = (1ULL << 48) - 1;
    for (int k = 0; k <= 32; ++k) {
      sh.jmpA[k] = a; sh.jmpC[k] = c;
      a = (a * 0x5DEECE66DULL) & MASK;
      c = (c * 0x5DEECE66DULL + 0xBULL) & MASK;
    }
  }
  __syncwarp();
  if (E.lab && plen > 4) closest_lab_tables(E);
}

// one pixel per lane: visiting order, source pixel, saliency, luminance of pixels [n0, n0 + 32)
__device__ __forceinline__ PixBlock fetch_block(const DitherCtx& D, const uint32_t* order, int n0) {
  PixBlock b;
  b.xy = 0; b.px = 0; b.sal = 0.f; b.ypix = 0.0;
  const int n = n0 + (int)lane_id();
  if (n < D.npix) {
    b.xy = order[n];
    const int bidx = (int)(b.xy & 0xFFFF) + (int)(b.xy >> 16) * D.width;
    b.px = eff_pixel(D.in[bidx], D.fixA0);
    if (D.E.useSal) {
      uint32_t sp = b.px;
      if (D.salReplaced && (sp >> 24) <= 0xF) sp = D.E.transColor;
      const Lab4 l = lab_of(sp);
      const float saliencyBase = .1f;
      b.sal = saliencyBase + (1 - saliencyBase) * l.L / 100.f * l.alpha / 255.f;
    }
    b.ypix = color_y(b.px, D.E.sh->lut);
  }
  return b;
}

// the quantization branch of diffusePixel (GC:211-229), warp-cooperative: every lane holds the same
// arguments. c2 = the error-diffused colour.
__device__ int quantize_pixel(Env& E, int x, int y, int bidx, uint32_t pixel, float sal, double ypix, uint32_t c2) {
  const int plen = E.plen, margin = E.margin;
  const int a_pix = c_alpha(c2);
  int qi;
  if (E.useSal && E.dither && !E.sorted && (!E.gHasAlpha || c_alpha(pixel) < a_pix)) {
    if ((plen >= 256 && sal > .99f) || (E.gHasAlpha && (double)(c_alpha(pixel) - a_pix) < (.5 * margin)))
      qi = lookup(E, c2, bidx);
    else
      qi = dither_pixel(E, x, y, bidx, pixel, sal, ypix, c2, E.beta, 0);    // qPixels[bidx] is still 0 here (GC:136,216)
  } else if (plen <= 32 && a_pix > 0xF0) {
    qi = lookup(E, c2, bidx);
    const int acceptedDiff = max(2, plen - margin);
    if (E.useSal && (y_diff_pre(ypix, c2, E.sh->lut) > (double)acceptedDiff || u_diff(pixel, c2) > (double)(2 * acceptedDiff))) {
      const float strength = 1 / 3.f;
      c2 = bn_diffuse(pixel, E.sh->pal[qi], 1 / sal, strength, x, y, E.sh->bn);
      qi = lookup(E, c2, bidx);
    }
  } else
    qi = lookup(E, c2, bidx);
  return qi;
}

// BlueNoise.dither second pass (PQ:400-401, PL:511-515, BN:207-222); memo and RNG carry over
__device__ void bluenoise_pass(NqImage& I, DitherCtx& D) {
  Env& E = D.E;
  const unsigned lane = lane_id();
  const int npix = D.npix, width = D.width;
  __syncwarp();
  __threadfence_block();
  float weight = 1.0f;
  const float strength = 1 / 3.f;
  if (E.lab) {   // PL:511-513: depends on how many colours getLab has seen by now
    __threadfence();
    const double size = (double)*(volatile unsigned int*)E.distinct;
    const double delta = ((double)E.plen * (double)E.plen) / size;
    weight = delta > 0.023 ? 1.0f : (float)(37.013 * delta + 0.906);
  }
  if (lane == 0) I.bnWeight = weight;
  for (int n0 = 0; n0 < npix; n0 += 32) {
    const int n = n0 + (int)lane;
    uint32_t px = 0, qv = 0;
    if (n < npix) { px = eff_pixel(D.in[n], D.fixA0); qv = D.out[n]; }
    uint32_t myOut = 0;
    const int cnt = min(32, npix - n0);
    for (int j = 0; j < cnt; ++j) {
      const int bidx = n0 + j, x = bidx % width, y = bidx / width;
      const uint32_t pixel = __shfl_sync(FULL, px, j);
      const uint32_t q0 = __shfl_sync(FULL, qv, j);
      const uint32_t c1 = bn_diffuse(pixel, E.sh->pal[q0], weight, strength, x, y, E.sh->bn);
      const int qi = lookup(E, c1, bidx);
      if ((int)lane == j) myOut = E.sh->pal[qi];
    }
    if (n < npix) D.out[n] = myOut;
  }
}

// -------------------------------------------------------------------------------------------------
// FIFO queue mode. The ArrayDeque always holds DITHER_MAX boxes (initWeights pushes DITHER_MAX
// empty ones before the first pixel, GC:345,358-359; afterwards every pixel polls one and adds one),
// so the sum of GC:193-204 for pixel n is
//     ((pixel_n + e[n-DM] w[0]) + e[n-DM+1] w[1]) + ... + e[n-1] w[DM-1]        (e[t] = 0 for t < 0)
// in exactly that float order. Only the LAST term depends on the previous pixel. The partial sums are
// kept in registers as a systolic pipeline: at step n lane k holds the sum of pixel n + DM-1-k through
// tap k, every lane adds e[n-1] w[k] to what its left neighbour held one step earlier, and the sum of
// pixel n through tap DM-2 is broadcast before e[n-1] is known. maxErr (max over all partial sums,
// GC:192,200-201) travels with the sums. Every lane redundantly finishes the four channels of pixel n,
// so nothing is shuffled on the dependency chain.
//
// CIELAB images with a saliency map mostly take GilbertCurve.ditherPixel (GC:125-185), which for
// palettes with palette.length - margin > 50 replaces the error-diffused colour by
// BlueNoise.diffuse(pixel, palette[0], kappa) BEFORE the palette lookup: Y_Diff <= 100 < 2 acceptedDiff
// makes GC:137 always true. The looked-up index then does not depend on the running error at all, so
// the lookups of a whole block are done one pixel per lane ("pre-lookup"), consuming the
// java.util.Random stream and the first-seen memo in curve order, and only the error arithmetic
// stays on the serial chain. Blocks containing a pixel whose lookup does consume the diffused colour
// fall back to the cooperative per-pixel path.
// -------------------------------------------------------------------------------------------------

// ditherPixel (GC:125-185) with qPixels[bidx] == 0, evaluated without the error-diffused colour.
// Returns false when the reference's result would read it. The caller guarantees
// plen <= 4 || 2 * acceptedDiff > 101 (so GC:137 holds for any c2).
__device__ bool dither_pixel_pre(const Env& E, int x, int y, uint32_t pixel, float sal, double ypix, uint32_t* out) {
  const int plen = E.plen, margin = E.margin;
  const double weight = E.gWeight;
  const float beta = E.beta;
  const uint32_t qcol = E.sh->pal[0];
  const signed char* bn = E.sh->bn;
  const double* lut = E.sh->lut;
  const float strength = 1 / 3.f;
  const int acceptedDiff = max(2, plen - margin);
  uint32_t c2;
  if (plen <= 4 && sal > .2f && sal < .25f)
    c2 = bn_diffuse(pixel, qcol, beta * 2 / sal, strength, x, y, bn);
  else if (plen > 64) {
    float kappa = sal < .6f ? beta * .15f / sal : beta * .4f / sal;
    c2 = bn_diffuse(pixel, qcol, kappa, strength, x, y, bn);
  } else if (plen > 16 && weight < .005)
    c2 = bn_diffuse(pixel, qcol, beta * normal_distribution(sal, .5f) + beta, strength, x, y, bn);
  else
    c2 = bn_diffuse(pixel, qcol, beta * .5f / sal, strength, x, y, bn);

  const double gamma = (plen <= 32 && weight < .01 && weight > .007) ? (double)(1 - beta) : (double)beta;
  if (plen > 4 && y_diff_pre(ypix, c2, lut) > (gamma * acceptedDiff)) return false;   // GC:149-172 reads r_pix..a_pix
  if (E.DM < 16 && plen > 4 && sal < .6f && y_diff_pre(ypix, c2, lut) > (double)(margin - 1)) return false;   // GC:175
  if (plen > 32 && (double)sal > .95) {
    float kappa = beta * fmaxf(.05f, .75f - plen / 128.f) * sal;
    c2 = bn_diffuse(pixel, qcol, kappa, strength, x, y, bn);
  }
  *out = c2;
  return true;
}

// PnnLABQuantizer.closestColorIndex top-2 scan (PL:418-458), one colour per lane over the whole palette.
// Keys are floor(err) << 8 | index: the two smallest keys are the reference's closest[0..3].
#define K2_NONE 0xFFFFFFFFu
__device__ __forceinline__ void closest_scan_lane(const Env& E, uint32_t c, unsigned& k0, unsigned& k1) {
  const WarpShared& sh = *E.sh;
  const int ca = c_alpha(c), cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  k0 = K2_NONE; k1 = K2_NONE;
  // a + 1.5 * 2^32 has an ulp of 2^-20: its mantissa is a in 2^-20 fixed point (rounded to nearest)
  const double MAGIC = 6442450944.0;
#pragma unroll 4
  for (int k = 0; k < E.plen; ++k) {
    const uint32_t c2 = sh.pal[k];
    double a = sh.Tr[abs(c_red(c2) - cr)] + sh.Tg[abs(c_green(c2) - cg)] + sh.Tb[abs(c_blue(c2) - cb)];
    if (E.semi) a += sh.Ta[abs(c_alpha(c2) - ca)];
    const long long bits = __double_as_longlong(a + MAGIC);
    const unsigned lo = (unsigned)bits, hi = (unsigned)(bits >> 32) & 0x7FFFFu;
    int d = (int)__funnelshift_r(lo, hi, 20);
    const unsigned fr = lo & 0xFFFFFu;
    // the table sum is within 2e-14 relative of the reference's 12/13-term sum (see closest_lab_tables):
    // only within 2^-19 of an integer can the floors differ
    if (((fr + 2u) & 0xFFFFFu) < 4u) d = j2i(closest_lab_err(E, c2, ca, cr, cg, cb));
    const unsigned key = ((unsigned)d << 8) | (unsigned)k;
    const unsigned t = max(key, k0);
    k0 = min(key, k0);
    k1 = min(k1, t);
  }
}

// -------------------------------------------------------------------------------------------------
// Candidate lists for the closest-colour scan. The cost of palette entry p for colour c is separable,
// S_p(c) = Tr[|dr|] + Tg[|dg|] + Tb[|db|] with every table increasing, so over a cell of 8x8x8 colours
// (5-5-5 bits of r, g, b) it lies in [lo_p, hi_p] with lo/hi taken at the nearest/farthest corner. With
// D2 = the second smallest floor(hi_p), an entry with floor(lo_p) > D2 can never be one of the two smallest
// (floor(err), index) pairs the scan keeps (PL:418-458). Each cell stores up to 31 candidates (byte 0 =
// count, 255 = too many: scan the whole palette). Only used for images without semi-transparency.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_build_cells(const NqImage* imgs, const NqSlot* slots) {
  __shared__ double Tr[256], Tg[256], Tb[256];
  __shared__ uint32_t pal[NQ_MAXK];
  const int img = blockIdx.y;
  const NqImage& I = imgs[img];
  const int plen = I.paletteLen;
  if (I.kind != NQ_KIND_LAB || !I.gUseSal || !I.dither || I.gSorted || I.gHasAlpha || plen <= 4 || I.error || !slots[img].cells) return;
  const int t = threadIdx.x;
  {
    double ta;
    closest_lab_table_entry(I.PR, I.PG, I.PB, I.PA, I.ratioMerge, false, t, &Tr[t], &Tg[t], &Tb[t], &ta);
    if (t < plen) pal[t] = I.palette[t];
  }
  __syncthreads();
  unsigned char* out = slots[img].cells;
  for (int cell = blockIdx.x * blockDim.x + t; cell < 32768; cell += gridDim.x * blockDim.x) {
    const int r0 = (cell >> 10) << 3, g0 = ((cell >> 5) & 31) << 3, b0 = (cell & 31) << 3;
    // pass 1: the two smallest floor(hi)
    int h0 = 0x7fffffff, h1 = 0x7fffffff;
    for (int k = 0; k < plen; ++k) {
      const uint32_t pc = pal[k];
      const int pr = c_red(pc), pg = c_green(pc), pb = c_blue(pc);
      const double hi = Tr[max(abs(pr - r0), abs(pr - r0 - 7))] + Tg[max(abs(pg - g0), abs(pg - g0 - 7))] + Tb[max(abs(pb - b0), abs(pb - b0 - 7))];
      const int d = j2i(hi * (1.0 + 1e-12) + 1e-9);
      if (d < h0) { h1 = h0; h0 = d; } else if (d < h1) h1 = d;
    }
    // pass 2: everything that can still reach the top two
    unsigned words[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    int cnt = 0;
    for (int k = 0; k < plen; ++k) {
      const uint32_t pc = pal[k];
      const int pr = c_red(pc), pg = c_green(pc), pb = c_blue(pc);
      const double lo = Tr[max(0, max(r0 - pr, pr - r0 - 7))] + Tg[max(0, max(g0 - pg, pg - g0 - 7))] + Tb[max(0, max(b0 - pb, pb - b0 - 7))];
      const int d = j2i(lo * (1.0 - 1e-12) - 1e-9);
      if (d <= h1) {
        ++cnt;
        if (cnt <= 31) words[cnt >> 2] |= (unsigned)k << (8 * (cnt & 3));
      }
    }
    words[0] |= cnt > 31 ? 255u : (unsigned)cnt;
    uint4* o = reinterpret_cast<uint4*>(out + (size_t)cell * 32);
    o[0] = make_uint4(words[0], words[1], words[2], words[3]);
    o[1] = make_uint4(words[4], words[5], words[6], words[7]);
  }
}

// top-2 scan of one colour per lane over its cell's candidate list (see k_build_cells); false if any
// lane's cell overflowed (the caller then scans the whole palette)
__device__ __forceinline__ bool closest_scan_cells(const Env& E, uint32_t c, bool active, unsigned& k0, unsigned& k1) {
  const WarpShared& sh = *E.sh;
  const int ca = c_alpha(c), cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  k0 = K2_NONE; k1 = K2_NONE;
  unsigned w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (active) {
    const uint4* p = E.cells + 2 * (size_t)(((cr >> 3) << 10) | ((cg >> 3) << 5) | (cb >> 3));
    const uint4 a = __ldg(p), b = __ldg(p + 1);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
  }
  const int cnt = (int)(w[0] & 255u);
  if (__any_sync(FULL, cnt == 255)) return false;
  const int maxCnt = __reduce_max_sync(FULL, cnt);
  const double MAGIC = 6442450944.0;
#pragma unroll
  for (int j = 1; j < 32; ++j) {
    if (j > maxCnt) break;
    const int k = (int)((w[j >> 2] >> (8 * (j & 3))) & 255u);
    const uint32_t c2 = sh.pal[k];
    double a = sh.Tr[abs(c_red(c2) - cr)] + sh.Tg[abs(c_green(c2) - cg)] + sh.Tb[abs(c_blue(c2) - cb)];
    const long long bits = __double_as_longlong(a + MAGIC);
    const unsigned lo = (unsigned)bits, hi = (unsigned)(bits >> 32) & 0x7FFFFu;
    int d = (int)__funnelshift_r(lo, hi, 20);
    const unsigned fr = lo & 0xFFFFFu;
    if (((fr + 2u) & 0xFFFFFu) < 4u) d = j2i(closest_lab_err(E, c2, ca, cr, cg, cb));
    const unsigned key = j <= cnt ? (((unsigned)d << 8) | (unsigned)k) : K2_NONE;
    const unsigned t = max(key, k0);
    k0 = min(key, k0);
    k1 = min(k1, t);
  }
  return true;
}

// Ring between the producer warp (gathers pixels, does the pre-lookups) and the consumer warp (the
// serial error recurrence). Block b lives in slot b & 3. Counters only grow: `fetched` blocks have their
// pixels in the ring, `looked` blocks their pre-lookup result (or the note that there is none),
// `consumed` blocks are finished. The java.util.Random state and the draw counter travel through the
// ring too: whoever does lookups (producer for pre-lookup blocks, consumer for the others) owns them,
// and the producer never commits a block before every earlier non-pre block has been consumed.
#define NQ_RING 4
struct DitherRing {
  uint32_t px[NQ_RING][32], xy[NQ_RING][32], pre[NQ_RING][32];
  float sal[NQ_RING][32];
  double ypix[NQ_RING][32];
  unsigned diffMask[NQ_RING];
  int blockPre[NQ_RING];
  int fetched, looked, consumed;
  unsigned long long rngSeed, draws;
};
// `ns`: how long to sleep between polls. The producer runs blocks ahead and idles most of the time, so it polls
// rarely (its polling instructions would otherwise take a fifth of the SM's issue slots from the consumers).
template <int NS = 40>
__device__ __forceinline__ void ring_wait(const int* p, int v, long long* waited = nullptr) {
  const volatile int* vp = p;
  if (*vp < v) {
    const long long t0 = clock64();
    while (*vp < v) __nanosleep(NS);
    if (waited) *waited += clock64() - t0;
  }
  __syncwarp();
  __threadfence_block();
}
__device__ __forceinline__ void ring_signal(int* p, int v) {
  __syncwarp();
  __threadfence_block();
  if (lane_id() == 0) *(volatile int*)p = v;
}

// pre-lookup of one block: colour c per lane (dither_pixel_pre), top-2 scan, java.util.Random draws and
// nearest fallbacks in curve order. Returns the palette colour chosen for this lane's pixel.
__device__ uint32_t prelookup_commit(Env& E, uint32_t c, bool mine) {
  WarpShared& sh = *E.sh;
  const unsigned lane = lane_id();
  const int plen = E.plen;
  const int ca = c_alpha(c);
  const bool viaClosest = mine && plen > 4 && ca > 0xF;    // PL:484-487, PL:407-408
  unsigned k0 = K2_NONE, k1 = K2_NONE;
  if (__any_sync(FULL, viaClosest)) {
    if (!E.cells || E.semi || !closest_scan_cells(E, c, viaClosest, k0, k1)) closest_scan_lane(E, c, k0, k1);
  }
  const int c0 = k0 == K2_NONE ? 0 : (int)(k0 & 255u), d0 = k0 == K2_NONE ? T2_NONE : (int)(k0 >> 8);
  const int c1 = k1 == K2_NONE ? c0 : (int)(k1 & 255u), d1 = k1 == K2_NONE ? T2_NONE : (int)(k1 >> 8);
  const bool draw = viaClosest && d0 != 0;                  // short-circuit: no draw when closest[2] == 0 (PL:467)
  const unsigned dm = __ballot_sync(FULL, draw);
  const int myDraw = __popc(dm & ((1u << lane) - 1u)), total = __popc(dm);
  int r = 0;
  if (total) {
    // jump ahead: this lane's draw is step myDraw + 1 from the current seed, unless a nextInt in the block
    // rejected its first value (probability 1.5e-5 per draw), in which case the block is replayed in order
    const unsigned long long MASK = (1ULL << 48) - 1;
    const unsigned long long sd = (sh.jmpA[myDraw + 1] * E.rng.seed + sh.jmpC[myDraw + 1]) & MASK;
    const int u = (int)(sd >> 17);
    r = u % 32767;
    const bool rejected = draw && (int)((unsigned)(u - r) + 32766u) < 0;
    if (__any_sync(FULL, rejected)) {
      for (int t = 0; t < total; ++t) {
        const int v = E.rng.next_int(32767);
        if (myDraw == t) r = v;
      }
    } else
      E.rng.seed = (sh.jmpA[total] * E.rng.seed + sh.jmpC[total]) & MASK;
  }
  E.draws += (unsigned long long)total;
  int idx = 1;
  if (d0 == 0) idx = 0;
  else {
    const int sum = (int)((unsigned)d1 + (unsigned)d0);
    if ((r % sum) <= d1) idx = 0;
  }
  const int ci = idx ? c1 : c0, ei = idx ? d1 : d0;
  int qi = ci;
  bool needNear = mine && (!viaClosest || ei >= plen || ci == 0 || c_alpha(sh.pal[ci]) < ca);   // PL:470-472
  if (E.isNano && needNear) {   // memo entries never change once written: hits can be read out of order
    const unsigned short got = *(volatile unsigned short*)&E.memo[color_index(c, E.semi, E.hasTrans)];
    if (got != 0xFFFF) { qi = got; needNear = false; }
  }
  unsigned nm = __ballot_sync(FULL, needNear);
  while (nm) {                  // misses in curve order (first-seen colour fixes a bucket, PL:332-335,402)
    const int L = __ffs(nm) - 1;
    nm &= nm - 1;
    const int res = nearest_lab(E, __shfl_sync(FULL, c, L));
    if ((int)lane == L) qi = res;
  }
  return sh.pal[qi];
}

// `want`: which images this launch takes by NqImage::specDone: 0 = not the speculative path's, 3 = handed back by it
__global__ void __launch_bounds__(64) k_dither_fifo(NqImage* imgs, const NqSlot* slots, int cacheBytes, int want) {
  __shared__ WarpShared sh;
  __shared__ DitherRing ring;
  extern __shared__ unsigned short dynCache[];     // 16 384 entries when launched with cacheBytes, else nothing
  const int img = blockIdx.x;
  NqImage& I = imgs[img];
  const NqSlot& S = slots[img];
  const uint32_t* order = S.order;
  const unsigned lane = lane_id();
  const int plen = I.paletteLen;
  if (plen <= 0 || I.error || I.gSorted || I.specDone != want) return;
  DitherCtx D;
  const bool producer = threadIdx.x >= 32;
  if (cacheBytes) for (int i = threadIdx.x; i < 16384; i += 64) dynCache[i] = 0;
  if (!producer) {
    dither_prologue(I, S, sh, D);
    if (lane == 0) { ring.fetched = 0; ring.looked = 0; ring.consumed = 0; ring.rngSeed = D.E.rng.seed; ring.draws = 0; }
  }
  __syncthreads();
  if (producer) dither_prologue_regs(I, S, sh, D);      // same registers, shared tables already filled
  Env& E = D.E;
  const int npix = D.npix, width = D.width;
  const int nblocks = (npix + 31) >> 5;

  const int DM = E.DM;
  const bool useSal = E.useSal, dither = E.dither;
  const int thresold = E.thresold, margin = E.margin;
  const signed char* bn = sh.bn;
  const int acceptedDiff = max(2, plen - margin);
  // images whose ditherPixel lookups do not read the diffused colour (see above)
  const bool preImg = E.lab && useSal && dither && !E.gHasAlpha && (plen <= 4 || 2 * acceptedDiff > 101);

  if (producer) {
    // =========================== producer warp ===========================
    int lastSlow = -1;                           // last block left to the consumer's own lookups
    long long pwait = 0;
    for (int b = 0; b < nblocks; ++b) {
      const int slot = b & (NQ_RING - 1);
      ring_wait<500>(&ring.consumed, b - (NQ_RING - 1), &pwait);
      const PixBlock cur = fetch_block(D, order, b << 5);
      const int cnt = min(32, npix - (b << 5));
      const bool mine = (int)lane < cnt;
      const int myX = cur.xy & 0xFFFF, myY = cur.xy >> 16, myBidx = myX + myY * width;
      const unsigned diffMask = __ballot_sync(FULL, mine && bn[myBidx & 4095] > thresold);
      ring.px[slot][lane] = cur.px; ring.xy[slot][lane] = cur.xy; ring.sal[slot][lane] = cur.sal; ring.ypix[slot][lane] = cur.ypix;
      if (lane == 0) ring.diffMask[slot] = diffMask;
      ring_signal(&ring.fetched, b + 1);

      bool blockPre = false;
      uint32_t preCol = 0;
      if (preImg) {
        uint32_t c = 0;
        bool ok = true;
        if (mine) {
          if (plen >= 256 && cur.sal > .99f) ok = false;          // GC:214-215: looks up the diffused colour
          else ok = dither_pixel_pre(E, myX, myY, cur.px, cur.sal, cur.ypix, &c);
        }
        blockPre = __all_sync(FULL, ok);
        if (blockPre) {
          ring_wait<200>(&ring.consumed, lastSlow + 1);   // the consumer is done drawing for every earlier block
          E.rng.seed = ring.rngSeed; E.draws = ring.draws;
          preCol = prelookup_commit(E, c, mine);
          if (lane == 0) { ring.rngSeed = E.rng.seed; ring.draws = E.draws; }
        }
      }
      if (!blockPre) lastSlow = b;
      ring.pre[slot][lane] = preCol;
      if (lane == 0) ring.blockPre[slot] = blockPre ? 1 : 0;
      ring_signal(&ring.looked, b + 1);
    }
    if (lane == 0) I.statDither[2] = (unsigned long long)pwait;
    return;
  }

  // =========================== consumer warp ===========================
  if (cacheBytes) E.mcache = dynCache;             // the producer's lookups (pre-lookup blocks) go to global memory
  uint32_t* out = D.out;
  const int ditherMax = E.ditherMax;
  const float wk = lane < (unsigned)DM ? I.gWeights[lane] : 0.f;   // this lane's tap
  const float wLast = I.gWeights[DM - 1];
  const float fDitherMax = (float)ditherMax, fDitherMax1 = (float)(ditherMax - 1);
  const float divisor = (float)(1 + nqm::sqrt_((double)ditherMax));
  const bool denoise = plen > 2;
  const bool illusion0 = bn[0] > thresold;          // yDiff == 1: bn[(int)(4096.0) & 4095] (GC:251-252)
  const bool rgbMemo = !E.lab && dither && E.isNano;

  // systolic state: lane k carries the sum of some pixel through tap k, and its running maximum
  float P0 = 0.f, P1 = 0.f, P2 = 0.f, P3 = 0.f, M = (float)(DM - 1);
  float e0 = 0.f, e1 = 0.f, e2 = 0.f, e3 = 0.f;    // shaped error of the previous pixel (r, g, b, a)

  // one systolic step: inject `px` at lane 0, every lane adds e * w[k]
  auto advance = [&](uint32_t injectPx) {
    float q0 = __shfl_up_sync(FULL, P0, 1), q1 = __shfl_up_sync(FULL, P1, 1), q2 = __shfl_up_sync(FULL, P2, 1), q3 = __shfl_up_sync(FULL, P3, 1);
    float qm = __shfl_up_sync(FULL, M, 1);
    if (lane == 0) {
      q0 = (float)c_red(injectPx); q1 = (float)c_green(injectPx); q2 = (float)c_blue(injectPx); q3 = (float)c_alpha(injectPx);
      qm = (float)(DM - 1);
    }
    P0 = q0 + e0 * wk; P1 = q1 + e1 * wk; P2 = q2 + e2 * wk; P3 = q3 + e3 * wk;
    M = fmaxf(fmaxf(fmaxf(qm, P0), fmaxf(P1, P2)), P3);
  };

  long long cwait = 0;
  const long long cstart = clock64();
  ring_wait(&ring.fetched, 1);
  uint32_t nxtPx = ring.px[0][lane];
  // fill the pipeline: pixels 0 .. DM-2 enter with zero errors behind them
  for (int s = 0; s < DM - 1; ++s) advance(__shfl_sync(FULL, nxtPx, s));

  for (int b = 0; b < nblocks; ++b) {
    const int slot = b & (NQ_RING - 1), n0 = b << 5;
    ring_wait(&ring.looked, b + 1, &cwait);
    ring_wait(&ring.fetched, min(b + 2, nblocks), &cwait);
    const uint32_t curPx = nxtPx;
    nxtPx = b + 1 < nblocks ? ring.px[(b + 1) & (NQ_RING - 1)][lane] : 0u;
    const uint32_t curXy = ring.xy[slot][lane];
    const uint32_t preCol = ring.pre[slot][lane];
    const bool blockPre = ring.blockPre[slot] != 0;
    const unsigned diffMask = ring.diffMask[slot];
    float curSal = 0.f;
    double curY = 0.0;
    if (!blockPre) {
      curSal = ring.sal[slot][lane]; curY = ring.ypix[slot][lane];
      E.rng.seed = ring.rngSeed; E.draws = ring.draws;
    }
    const int cnt = min(32, npix - n0);
    const bool mine = (int)lane < cnt;
    const int myBidx = (int)(curXy & 0xFFFF) + (int)(curXy >> 16) * width;

    uint32_t myOut = preCol;
    for (int j = 0; j < cnt; ++j) {
      // ---- independent of the previous pixel's error: sum of this pixel through tap DM-2
      const float b0 = __shfl_sync(FULL, P0, DM - 2), b1 = __shfl_sync(FULL, P1, DM - 2), b2 = __shfl_sync(FULL, P2, DM - 2), b3 = __shfl_sync(FULL, P3, DM - 2);
      const float bm = __shfl_sync(FULL, M, DM - 2);
      const uint32_t pixel = __shfl_sync(FULL, curPx, j);
      const uint32_t pcPre = __shfl_sync(FULL, preCol, j);
      const int jn = j + DM - 1;
      const uint32_t injA = __shfl_sync(FULL, curPx, jn & 31), injB = __shfl_sync(FULL, nxtPx, jn & 31);
      const uint32_t inject = jn < 32 ? injA : injB;

      // ---- last tap, clamp (GC:199-211)
      const float a0 = b0 + e0 * wLast, a1 = b1 + e1 * wLast, a2 = b2 + e2 * wLast, a3 = b3 + e3 * wLast;
      const float maxErr = fmaxf(fmaxf(fmaxf(bm, a0), fmaxf(a1, a2)), a3);
      // (int) Math.min(BYTE_MAX, Math.max(error.p[j], 0.0)): widening the float is exact, so the clamp can stay in float
      const int r_pix = __float2int_rz(fminf(255.f, fmaxf(a0, 0.f))), g_pix = __float2int_rz(fminf(255.f, fmaxf(a1, 0.f)));
      const int b_pix = __float2int_rz(fminf(255.f, fmaxf(a2, 0.f))), a_pix = __float2int_rz(fminf(255.f, fmaxf(a3, 0.f)));
      advance(inject);     // uses e0..e3 of the previous pixel; must precede their update below

      // ---- quantize (GC:211-229)
      uint32_t pc;
      if (blockPre) pc = pcPre;
      else {
        const uint32_t c2 = c_argb(a_pix, r_pix, g_pix, b_pix);
        // PnnQuantizer with dither: the branch of GC:211-229 is nearestColorIndex(c2), and with the reduced memo key
        // (PQ:271) it is nearly always a hit: answer it inline, without the call into the general path
        int qi = -1;
        if (rgbMemo) qi = memo_get(E, color_index(c2, E.semi, E.hasTrans));
        if (qi < 0) {
          const uint32_t xy = __shfl_sync(FULL, curXy, j);
          const int x = xy & 0xFFFF, y = xy >> 16;
          qi = quantize_pixel(E, x, y, x + y * width, pixel, __shfl_sync(FULL, curSal, j), shfl_d(curY, j), c2);
        }
        pc = sh.pal[qi];
        const uint32_t res = (dither || plen <= 32) ? pc : (uint32_t)qi;   // GC:278-279
        if ((int)lane == j) myOut = res;
      }

      // ---- error of this pixel and its shaping (GC:236-264); yDiff == 1 in this mode
      e0 = (float)(r_pix - c_red(pc)); e1 = (float)(g_pix - c_green(pc)); e2 = (float)(b_pix - c_blue(pc)); e3 = (float)(a_pix - c_alpha(pc));
      if (denoise) {
        const bool s0 = fabsf(e0) >= fDitherMax, s1 = fabsf(e1) >= fDitherMax, s2 = fabsf(e2) >= fDitherMax;
        if (s0 || s1 || s2) {
          if ((diffMask >> j) & 1u) {
            // lanes 0, 1, 2 shape r, g, b at the same time (the other lanes mirror b); the exact kernel only if undecided
            const float eL = lane == 0 ? e0 : (lane == 1 ? e1 : e2);
            const bool sL = lane == 0 ? s0 : (lane == 1 ? s1 : s2);
            const double xL = (double)(eL / maxErr * 20.f);
            float vL;
            const bool kL = tanh_fast(xL, &vL);
            if (__any_sync(FULL, sL && !kL)) {
              if (sL && !kL) vL = (float)nqm::nq_tanh(xL);
            }
            const float rL = vL * fDitherMax1;
            const float r0 = __shfl_sync(FULL, rL, 0), r1 = __shfl_sync(FULL, rL, 1), r2 = __shfl_sync(FULL, rL, 2);
            if (s0) e0 = r0;
            if (s1) e1 = r1;
            if (s2) e2 = r2;
          } else if (illusion0) {
            if (s0) e0 = (float)((double)(e0 / maxErr) * 1.0) * fDitherMax1;
            if (s1) e1 = (float)((double)(e1 / maxErr) * 1.0) * fDitherMax1;
            if (s2) e2 = (float)((double)(e2 / maxErr) * 1.0) * fDitherMax1;
          } else {
            if (s0) e0 /= divisor;
            if (s1) e1 /= divisor;
            if (s2) e2 /= divisor;
          }
        }
      }
    }
    if (mine) out[myBidx] = myOut;
    if (!blockPre && lane == 0) { ring.rngSeed = E.rng.seed; ring.draws = E.draws; }
    ring_signal(&ring.consumed, b + 1);
  }

  if (lane == 0) { I.statDither[0] = (unsigned long long)(clock64() - cstart); I.statDither[1] = (unsigned long long)cwait; }
  E.rng.seed = ring.rngSeed; E.draws = ring.draws;
  if (!dither && plen > 32 && !I.bnParallel) bluenoise_pass(I, D);
  if (lane == 0) I.rngDraws = E.draws;
}

// -------------------------------------------------------------------------------------------------
// PriorityQueue mode (sortedByYDiff, GC:87-94): the queue is a binary heap ordered by yDiff; the sum
// of GC:193-204 walks its backing array, so the order of the float additions changes with every
// sift. The recurrence stays in shared memory and the warp splits only the four channels.
// Steady state: 15 boxes, weights of length 7 (initWeights is re-run with sizes 1, 3, 7 on pixels
// 2, 3, 4, each time pushing `size` empty boxes, GC:233-234,345).
// -------------------------------------------------------------------------------------------------
struct PQ {
  SortedShared* sh;
  int n;
  __device__ __forceinline__ void put(int k, const float* p, double yd) {
    if (lane_id() == 0) { sh->q[k][0] = p[0]; sh->q[k][1] = p[1]; sh->q[k][2] = p[2]; sh->q[k][3] = p[3]; sh->qy[k] = yd; }
  }
  __device__ __forceinline__ void move(int dst, int src) {
    float p[4] = {sh->q[src][0], sh->q[src][1], sh->q[src][2], sh->q[src][3]};
    double yd = sh->qy[src];
    __syncwarp();
    put(dst, p, yd);
    __syncwarp();
  }
  __device__ void offer(const float* p, double yd) {   // siftUp; "x before e" <=> x.yDiff > e.yDiff
    int k = n++;
    while (k > 0) {
      int parent = (k - 1) >> 1;
      double pe = sh->qy[parent];
      if (!(yd > pe)) break;            // cmp(x, e) >= 0
      move(k, parent);
      k = parent;
    }
    __syncwarp();
    put(k, p, yd);
    __syncwarp();
  }
  __device__ void poll() {              // remove head, siftDown the last element
    int last = --n;
    if (last == 0) return;
    float p[4] = {sh->q[last][0], sh->q[last][1], sh->q[last][2], sh->q[last][3]};
    double yd = sh->qy[last];
    __syncwarp();
    int k = 0, half = last >> 1;
    while (k < half) {
      int child = (k << 1) + 1, right = child + 1;
      double cy = sh->qy[child];
      if (right < last) { double ry = sh->qy[right]; if (ry > cy) { child = right; cy = ry; } }   // cmp(c, right) > 0
      if (!(cy > yd)) break;            // cmp(x, c) <= 0
      move(k, child);
      k = child;
    }
    put(k, p, yd);
    __syncwarp();
  }
};

__global__ void __launch_bounds__(32) k_dither_sorted(NqImage* imgs, const NqSlot* slots) {
  __shared__ WarpShared sh;
  __shared__ SortedShared qs;
  const int img = blockIdx.x;
  NqImage& I = imgs[img];
  const NqSlot& S = slots[img];
  const uint32_t* order = S.order;
  const unsigned lane = lane_id();
  const int plen = I.paletteLen;
  if (plen <= 0 || I.error || !I.gSorted) return;
  DitherCtx D;
  dither_prologue(I, S, sh, D);
  Env& E = D.E;
  const int npix = D.npix, width = D.width;
  uint32_t* out = D.out;

  const int DM = E.DM;
  for (int i = lane; i < 16 * 4; i += 32) qs.q[i >> 2][i & 3] = 0.f;
  if (lane < 16) qs.qy[lane] = 0;
  if (lane < 8) qs.w[lane] = 0.f;
  __syncwarp();

  const bool useSal = E.useSal, dither = E.dither;
  const int ch = lane & 3;
  const int thresold = E.thresold, ditherMax = E.ditherMax;
  const float beta = E.beta;
  const double* lut = sh.lut;
  const signed char* bn = sh.bn;
  PQ pq{&qs, 0};
  int wlen = 0;            // weights.length (0, 1, 3, 7)

  PixBlock nxt = fetch_block(D, order, 0);
  for (int n0 = 0; n0 < npix; n0 += 32) {
    const PixBlock cur = nxt;
    if (n0 + 32 < npix) nxt = fetch_block(D, order, n0 + 32);
    uint32_t myOut = 0;
    const int cnt = min(32, npix - n0);
    for (int j = 0; j < cnt; ++j) {
      const uint32_t xy = __shfl_sync(FULL, cur.xy, j);
      const uint32_t pixel = __shfl_sync(FULL, cur.px, j);
      const float sal = __shfl_sync(FULL, cur.sal, j);
      const double ypix = shfl_d(cur.ypix, j);
      const int x = xy & 0xFFFF, y = xy >> 16, bidx = x + y * width;

      // ---- error.p = pixel + sum(queue[i].p * weights[i]), backing-array order, weights from the top
      //      down (GC:190-204); lane&3 = channel
      float acc = (float)chan(pixel, ch);
      float mx = (float)(DM - 1);
      {
        int i = wlen - 1;
        for (int qi = 0; qi < pq.n && i >= 0; ++qi, --i) {
          acc += qs.q[qi][ch] * qs.w[i];
          if (acc > mx) mx = acc;
        }
      }
      mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 2));
      const float maxErr = mx;
      const int mine = j2i(dmin(255.0, dmax((double)acc, 0.0)));
      const int r_pix = __shfl_sync(FULL, mine, 0), g_pix = __shfl_sync(FULL, mine, 1), b_pix = __shfl_sync(FULL, mine, 2), a_pix = __shfl_sync(FULL, mine, 3);

      // ---- quantize (GC:211-229)
      uint32_t c2 = c_argb(a_pix, r_pix, g_pix, b_pix);
      int qi = quantize_pixel(E, x, y, bidx, pixel, sal, ypix, c2);

      // ---- queue maintenance (GC:231-234)
      if (pq.n >= DM) pq.poll();
      else if (pq.n != 0) {
        const int size = pq.n;                      // initWeights(size): size empty boxes + new weights
        const float zero[4] = {0.f, 0.f, 0.f, 0.f};
        for (int k = 0; k < size; ++k) pq.offer(zero, 0.0);
        const float* src = size == 1 ? I.gW1 : (size == 3 ? I.gW3 : I.gW7);
        if (lane < (unsigned)size) qs.w[lane] = src[lane];
        wlen = size;
        __syncwarp();
      }

      // ---- error of this pixel and its shaping (GC:236-264); lanes 0..2 shape r, g, b
      c2 = sh.pal[qi];
      const int pixch = ch == 0 ? r_pix : (ch == 1 ? g_pix : (ch == 2 ? b_pix : a_pix));
      float e = (float)(pixch - chan(c2, ch));
      const bool denoise = plen > 2;
      const bool diffuse = bn[bidx & 4095] > thresold;
      const double yDiff = y_diff_pre(ypix, c2, lut);
      const bool illusion = !diffuse && bn[j2i(yDiff * 4096) & 4095] > thresold;
      bool unacc = false;
      if (denoise && ch < 3) {
        if (fabsf(e) >= (float)ditherMax) {
          if (useSal) unacc = true;
          if (diffuse) e = tanh_to_float((double)(e / maxErr * 20.f)) * (float)(ditherMax - 1);
          else if (illusion) e = (float)((double)(e / maxErr) * yDiff) * (float)(ditherMax - 1);
          else e /= (float)(1 + nqm::sqrt_((double)ditherMax));
        }
        if (!useSal && fabsf(e) >= (float)DM) unacc = true;
      }
      const bool unaccepted = (__ballot_sync(FULL, unacc) & 7u) != 0;

      if (unaccepted) {   // GC:266-274
        if (useSal) qi = dither_pixel(E, x, y, bidx, pixel, sal, ypix, c2, beta, qi);
        else if (y_diff_pre(ypix, c2, lut) > 3 && u_diff(pixel, c2) > 3) {
          const float strength = 1 / 3.f;
          c2 = bn_diffuse(pixel, sh.pal[qi], strength, strength, x, y, bn);
          qi = lookup(E, c2, bidx);
        }
      }

      // ---- errorq.add(error) (GC:276)
      float p[4];
      p[0] = __shfl_sync(FULL, e, 0); p[1] = __shfl_sync(FULL, e, 1); p[2] = __shfl_sync(FULL, e, 2); p[3] = __shfl_sync(FULL, e, 3);
      pq.offer(p, yDiff);

      const uint32_t res = (dither || plen <= 32) ? sh.pal[qi] : (uint32_t)qi;   // GC:278-279
      if ((int)lane == j) myOut = res;
    }
    if ((int)lane < cnt) {
      const int bidx = (int)(cur.xy & 0xFFFF) + (int)(cur.xy >> 16) * width;
      out[bidx] = myOut;
    }
  }

  if (!dither && plen > 32 && !I.bnParallel) bluenoise_pass(I, D);
  if (lane == 0) I.rngDraws = E.draws;
}


// -------------------------------------------------------------------------------------------------
// BlueNoise.dither (BN:207-222) for PnnQuantizer, one THREAD per pixel. The second pass perturbs every original pixel
// away from its first-pass colour and looks the result up again with closestColorIndex (PQ:313-375), which is a pure
// function of (colour, position) -- its cache is written under another key than it is read with (PQ:320 vs 362) -- except
// where it falls back to nearestColorIndex (PQ:372), whose memo under the reduced key keeps the FIRST colour seen in a
// bucket (PQ:271-274), in raster order here (BN:212-219), after whatever the Gilbert pass left in it (PQ:398-404).
//   a: every pixel; fall-backs that miss the memo of the first pass post (raster position, colour) to their bucket with
//      a 64-bit atomicMin and mark the pixel (bit 15 of the index plane)
//   b: one thread per bucket that was posted to: the entry its first colour creates
//   c: the marked pixels read their bucket
// -------------------------------------------------------------------------------------------------
struct BnRgb {
  int plen, hasTrans, semi, isNano, fixA0, width, npix;
  uint32_t transColor;
  double PR, PG, PB, PA;
};
__device__ __forceinline__ BnRgb bn_rgb_consts(const NqImage& I) {
  BnRgb B;
  B.plen = I.paletteLen; B.hasTrans = I.transIdx >= 0; B.semi = I.hasSemi != 0; B.isNano = I.isNano != 0; B.fixA0 = I.fixA0;
  B.width = I.width; B.npix = I.npix; B.transColor = I.transColor;
  B.PR = I.PR; B.PG = I.PG; B.PB = I.PB; B.PA = I.PA;
  if (B.plen < 3) B.PR = B.PG = B.PB = B.PA = 1;
  return B;
}
// PnnQuantizer.nearestColorIndex without its memo (PQ:276-310), one thread
__device__ int nearest_rgb_thread(const BnRgb& B, const uint32_t* pal, uint32_t c) {
  int k = 0;
  if (c_alpha(c) <= 0xF) c = B.transColor;
  if (B.plen > 2 && B.hasTrans && c_alpha(c) > 0xF) k = 1;
  const int ca = c_alpha(c), cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  double best = 1e300;
  int bi = -1;
  for (int i = k; i < B.plen; ++i) {
    const uint32_t c2 = pal[i];
    const double da = (double)(c_alpha(c2) - ca), dr = (double)(c_red(c2) - cr), dg = (double)(c_green(c2) - cg), db = (double)(c_blue(c2) - cb);
    double cur = B.PA * (da * da);
    cur += B.PR * (dr * dr);
    cur += B.PG * (dg * dg);
    cur += B.PB * (db * db);
    if (cur <= best) { best = cur; bi = i; }            // strict > pruning: the last minimal index wins (PQ:291-307)
  }
  if (!(best <= 2147483647.0) || bi < 0) bi = k;         // mindist starts at Integer.MAX_VALUE (PQ:286)
  return bi;
}
// PnnQuantizer.closestColorIndex (PQ:313-375), one thread; -1 = falls back to nearestColorIndex(c)
__device__ int closest_rgb_thread(const BnRgb& B, const uint32_t* pal, uint32_t c, int pos) {
  if (c_alpha(c) <= 0xF) return -1;
  const int ca = c_alpha(c), cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  Top2 t = {1 << 30, 1 << 30, T2_NONE, T2_NONE};
  for (int k = 0; k < B.plen; ++k) {
    const uint32_t c2 = pal[k];
    const double dr = (double)(c_red(c2) - cr), dg = (double)(c_green(c2) - cg), db = (double)(c_blue(c2) - cb);
    double err = B.PR * (dr * dr);
    err += B.PG * (dg * dg);
    err += B.PB * (db * db);
    if (B.semi) { const double da = (double)(c_alpha(c2) - ca); err += B.PA * (da * da); }
    const int d = j2i(err);
    if (d != T2_NONE) t2_insert(t, d, k);
  }
  const int c0 = t.d0 == T2_NONE ? 0 : t.i0, e0 = t.d0;
  const int c1 = t.d1 == T2_NONE ? c0 : t.i1, e1 = t.d1;     // PQ:359-360
  const int MAX_ERR = B.plen << 2;
  int idx = (pos + 1) % 2;
  if ((double)e1 * .67 < (double)(e1 - e0)) idx = 0;
  else if (c0 > c1) idx = pos % 2;
  const int ci = idx ? c1 : c0, ei = idx ? e1 : e0;
  if (ei >= MAX_ERR || (B.hasTrans && ci == 0)) return -1;
  return ci;
}
#define NQ_BN_PENDING 0x8000u
__global__ void __launch_bounds__(256) k_bn_rgb_init(const NqImage* imgs, const NqSlot* slots) {
  const NqImage& I = imgs[blockIdx.y];
  if (!I.bnParallel || I.error || I.paletteLen <= 0) return;
  unsigned long long* first = slots[blockIdx.y].hSum;       // 65 536 buckets; the histogram sums are long dead
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < NQ_NBINS; k += gridDim.x * blockDim.x) first[k] = ~0ULL;
}
__global__ void __launch_bounds__(256) k_bn_rgb_a(NqImage* imgs, const NqSlot* slots) {
  __shared__ uint32_t pal[NQ_MAXK];
  NqImage& I = imgs[blockIdx.y];
  if (!I.bnParallel || I.error || I.paletteLen <= 0) return;
  const NqSlot& S = slots[blockIdx.y];
  const BnRgb B = bn_rgb_consts(I);
  for (int k = threadIdx.x; k < NQ_MAXK; k += blockDim.x) pal[k] = k < B.plen ? I.palette[k] : 0u;
  __syncthreads();
  unsigned long long* first = S.hSum;
  const float strength = 1 / 3.f;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < B.npix; n += gridDim.x * blockDim.x) {
    const uint32_t px = eff_pixel(S.in[n], B.fixA0);
    const unsigned q0 = S.out[n] & 0xFFFFu;                  // the Gilbert pass stored indices (GC:278-279)
    const int x = n % B.width, y = n / B.width;
    const uint32_t c1 = bn_diffuse(px, pal[q0 < (unsigned)B.plen ? q0 : 0], 1.0f, strength, x, y, g_blueNoise);
    int qi = closest_rgb_thread(B, pal, c1, n);
    unsigned mark = q0;
    if (qi < 0) {
      if (!B.isNano) qi = nearest_rgb_thread(B, pal, c1);    // full-colour key: the memo is a pure cache (PQ:271)
      else {
        const int key = color_index(c1, B.semi, B.hasTrans);
        const unsigned short got = S.memo[key];
        if (got != 0xFFFF) qi = got;
        else { atomicMin(&first[key], ((unsigned long long)(unsigned)n << 32) | (unsigned long long)c1); mark |= NQ_BN_PENDING; }
      }
    }
    S.idx[n] = (unsigned short)mark;
    if (qi >= 0) S.out[n] = pal[qi];
  }
}
__global__ void __launch_bounds__(256) k_bn_rgb_b(const NqImage* imgs, const NqSlot* slots) {
  __shared__ uint32_t pal[NQ_MAXK];
  const NqImage& I = imgs[blockIdx.y];
  if (!I.bnParallel || I.error || I.paletteLen <= 0 || !I.isNano) return;
  const NqSlot& S = slots[blockIdx.y];
  const BnRgb B = bn_rgb_consts(I);
  for (int k = threadIdx.x; k < NQ_MAXK; k += blockDim.x) pal[k] = k < B.plen ? I.palette[k] : 0u;
  __syncthreads();
  const unsigned long long* first = S.hSum;
  for (int key = blockIdx.x * blockDim.x + threadIdx.x; key < NQ_NBINS; key += gridDim.x * blockDim.x) {
    const unsigned long long f = first[key];
    if (f != ~0ULL) S.memo[key] = (unsigned short)nearest_rgb_thread(B, pal, (uint32_t)f);
  }
}
__global__ void __launch_bounds__(256) k_bn_rgb_c(const NqImage* imgs, const NqSlot* slots) {
  __shared__ uint32_t pal[NQ_MAXK];
  const NqImage& I = imgs[blockIdx.y];
  if (!I.bnParallel || I.error || I.paletteLen <= 0 || !I.isNano) return;
  const NqSlot& S = slots[blockIdx.y];
  const BnRgb B = bn_rgb_consts(I);
  for (int k = threadIdx.x; k < NQ_MAXK; k += blockDim.x) pal[k] = k < B.plen ? I.palette[k] : 0u;
  __syncthreads();
  const float strength = 1 / 3.f;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < B.npix; n += gridDim.x * blockDim.x) {
    const unsigned m = S.idx[n];
    if (!(m & NQ_BN_PENDING)) continue;
    const unsigned q0 = m & 0x7FFFu;
    const uint32_t px = eff_pixel(S.in[n], B.fixA0);
    const int x = n % B.width, y = n / B.width;
    const uint32_t c1 = bn_diffuse(px, pal[q0 < (unsigned)B.plen ? q0 : 0], 1.0f, strength, x, y, g_blueNoise);
    S.out[n] = pal[S.memo[color_index(c1, B.semi, B.hasTrans)]];
  }
}

}  // namespace nq
