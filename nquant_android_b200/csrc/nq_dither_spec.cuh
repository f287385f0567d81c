// nq_dither_spec.cuh -- speculative segment-parallel Gilbert dither (SURVEY.md section 8f rank 1) for the images
// whose palette lookups do not read the error-diffused colour: PnnLABQuantizer, dither on, ArrayDeque queue,
// no semi-transparency, more than 64 colours (GilbertCurve.ditherPixel replaces the colour by
// BlueNoise.diffuse(pixel, palette[0], kappa) before the lookup, GC:137-141; see nq_dither.cuh).
//
// Reference: GilbertCurve.diffusePixel / ditherPixel (GC:125-280), PnnLABQuantizer.closestColorIndex /
// nearestColorIndex (PL:329-474), java.util.Random (PL:22,467).
//
// The sequential chain carries three states (profiles/r1_spec_dither_study.md): the error queue Q, the number D
// of java.util.Random draws, and the first-seen memo nearestMap. For these images D and the memo are decided by
// per-pixel passes (stages 1-5 below) because 99.8 % of the lookups never see the running error; Q re-synchronises
// within a few hundred pixels of a restart from an empty queue. Stage 6 runs one THREAD per segment of the curve
// (warm-up from an empty queue, then the owned pixels); stage 7 validates the segments in curve order: the queue
// a segment warmed up to must equal, bit for bit, the queue its predecessor ended with, the draws it made must
// equal the prediction, and a memo entry created by one of its error-dependent lookups must not contradict an
// earlier one. A segment that fails re-runs from its predecessor's exact state in the next round. A memo entry that
// an error-dependent lookup created before the first pre-lookup of its key is patched into the later pixels
// (stage_patch); a draw that goes against its prediction moves every later draw index, so the pixel's flag is
// corrected and stages 2-5 are redone behind it (stage_rekey, k_spec_redo_*). Images that would thrash (stage_gate)
// or exhaust a cap are left to the serial kernel (k_dither_fifo) -- one such image costs the batch the whole serial
// chain, so the gates sit before any segment runs. The result is bit-identical to the sequential run by
// construction: a segment is only accepted from an exact input state.
//
// Every stage body is a scalar NQ_HD function so that the very same code is compiled by g++ and checked
// against the CPU oracle (tests/test_spec_dither_host.py); the kernels at the end of the file only index.
#pragma once
#include "nq_types.h"
#include "nq_color.h"

namespace nq {
namespace spec {

#define NQS_NOTES 256           // memo entries a segment may create through error-dependent lookups
#define NQS_READS 64            // memo entries of the pre-lookups its error-dependent lookups may read
#define NQS_NOPOS 0x7fffffff
#define NQS_MAXREJ 8             // generator steps whose value nextInt(32767) rejects, per image (expected: 0.008 for a 4K image)
#define NQS_NONE 0xFFFFFFFFu    // absent top-2 key

// per-pixel flags (curve order)
#define NQS_F_PRE 1u            // lookup does not read the diffused colour
#define NQS_F_DRAW 2u           // the lookup is predicted to call Random.nextInt (PL:467)
#define NQS_F_RISK 8u           // error-dependent lookup predicted NOT to draw: the pixel is (nearly) a palette colour, any diffused
                                // error makes it draw (PL:467) and every later draw index moves
#define NQS_MAXRISK 0x3fffffff  // (no limit: a run from the exact state handles any number of them, stage 7)
#define NQS_MAXREDO 256         // rounds with a draw misprediction per image before giving up
#define NQS_F_NEAR 4u           // resolved through nearestColorIndex's memo (PL:470-472), key = memo_key(ccol)
// What stage 6 saw an error-dependent lookup do. NQS_F_DRAW stays the prediction the CURRENT prefix sums, pre-lookups and
// packed records were made with; the next re-resolve adopts the observation as the prediction (stage_adopt) before its prefix sum.
#define NQS_F_SEEN 32u          // an outcome has been recorded since the last re-resolve
#define NQS_F_ACT 16u           // ... and it was a draw

// Constants of one image: what GilbertCurve's constructor and the quantizer hold while dithering.
struct SpecConst {
  int plen, margin, thresold, DM, ditherMax, width, npix;
  int isNano, hasTrans, salReplaced;
  int opaque;                            // every pixel has alpha 255 and every palette entry 254 or 255: stage 6 keeps the alpha errors as bits
  int seg, warm, nseg;
  uint32_t transColor;
  double gWeight, PR, PG, PB, ratio;
  float beta;
  unsigned long long seed0;              // java.util.Random state after setSeed
  float w[NQ_MAXQ];                      // initWeights(DITHER_MAX)
  uint32_t pal[NQ_MAXK];
  Lab4 palLab[NQ_MAXK];                  // getLab(palette[i]) (PL:352)
  double Tr[256], Tg[256], Tb[256];      // closestColorIndex cost of one channel difference (see nq_dither.cuh)
  unsigned long long jmpA[40], jmpC[40]; // java.util.Random: state after 2^i more steps = jmpA[i] * state + jmpC[i] (mod 2^48)
  // Random.nextInt(32767) draws AGAIN when next(31) is one of the two top values (2 in 2^31 per draw: a few images of every
  // large batch). Which steps of the generator do that depends on the seed alone: they are listed here (1-based step
  // indices, ascending; k_spec_rejects), and draw d is the d-th step that is not in the list (lcg_step_of).
  int nrej;
  unsigned rej[NQS_MAXREJ];
};

// Per-image work arrays (curve order, npix entries unless noted) and segment records.
struct SpecSeg {
  float qwarm[NQ_MAXQ][4];               // queue when the owned pixels begin (oldest box first)
  float qout[NQ_MAXQ][4];                // queue after the last owned pixel
  float qstart[NQ_MAXQ][4];              // exact start state (when exact != 0)
  int exact, dirty, done;
  int qok;                               // stage 6b: start queue == predecessor's final queue, bit for bit
  int warmMul;                           // warm-up length in units of SpecConst::warm (grows when the warm-up proved too short)
  int draws;                             // draws made by the owned pixels
  int mispos;                            // first owned error-dependent lookup whose draw differs from its prediction, or -1
  int nnotes;                            // > NQS_NOTES: overflow
  int noteKey[NQS_NOTES], notePos[NQS_NOTES], noteVal[NQS_NOTES];
  int nreads;                            // > NQS_READS: overflow (treated as "may have read any key")
  int readKey[NQS_READS];
  int nslow;                             // error-dependent lookups among the owned pixels (last run)
  int chain;                             // exact segment: how many segments (this one included) its thread runs in a row
  int chained;                           // run by the thread of an earlier segment (its chain): the own thread stands aside
  int dev;                               // sequential run: curve position of the chain's first draw against its prediction, or NQS_NOPOS
  unsigned idx0;                         // sequential run: draws made in front of the segment (the index its first draw continues from)
};
#define NQS_MAXCHAIN 4            // segments one thread runs in a row: bounds the time a round waits for its slowest thread
#define NQS_MAXPATCH 24          // memo entries corrected per round and image
// What stage 6 reads per pixel, packed by stage 5b and stored SEGMENT-INTERLEAVED: record of curve position n lives at
// (n % seg) * nseg + n / seg, so the threads of a warp (consecutive segments, same offset inside the segment) read
// consecutive 16-byte records.
struct alignas(16) SpecRec {
  uint32_t px;                           // source pixel
  uint32_t xy;                           // x | y << 16
  uint32_t qf;                           // palette index | flags << 16 | (TELL_BLUE_NOISE[bidx & 4095] > thresold) << 24
  float sal;                             // saliency of the pixel, for error-dependent lookups only (0 otherwise)
};
struct SpecWork {
  const uint32_t* order;                 // x | y << 16 per curve position
  const uint32_t* in;                    // source pixels, row-major
  uint32_t* out;
  uint32_t* cpx;                         // pixel per curve position
  uint32_t* ccol;                        // colour the pre-lookup asks for
  uint32_t* ck0;                         // smallest top-2 key (floor(err) << 8 | index)
  uint32_t* ck1;                         // second smallest
  unsigned short* cq;                    // resolved palette index (or memo key while NQS_F_NEAR)
  unsigned char* cflag;
  SpecRec* rec;                          // [nseg * seg] packed view for stage 6 (stage_pack)
  uint32_t* cdraw;                       // [npix + 1] draws predicted before this pixel (exclusive prefix of NQS_F_DRAW)
  int* firstPos;                         // [65536] first curve position whose pre-lookup needs memo key k
  unsigned short* memo;                  // [65536] nearestMap for reduced keys (0xFFFF = absent)
  int* slowPos;                          // [65536] entries created by error-dependent lookups of validated segments
  unsigned short* slowVal;               // [65536]
  const unsigned char* cells;            // candidate lists of k_build_cells, or nullptr
  const double* lut;                     // gammaToLinear table
  const signed char* bn;                 // TELL_BLUE_NOISE
  unsigned* chunkSum;                    // [npix / NQS_CHUNK + 1] draws predicted in front of each block of NQS_CHUNK pixels (stage 2)
  int* patch;                            // [2 * NQS_MAXPATCH] (key, position) pairs of the pending patches, count in state[2]
  SpecSeg* segs;
  int* state;                            // [16]: firstOpen, anomaly, patch key + 1 (0 = none), patch position, failed validations,
                                         //      re-resolve position + 1 (0 = none), re-resolves so far, pixels flagged NQS_F_RISK, error-dependent lookups
};

// ---- java.util.Random: state after j more steps of the LCG ------------------------------------------------
NQ_HD void lcg_tables(unsigned long long* A, unsigned long long* Cc, int n) {
  const unsigned long long MASK = (1ULL << 48) - 1;
  unsigned long long a = 0x5DEECE66DULL, c = 0xBULL;
  for (int i = 0; i < n; ++i) {
    A[i] = a; Cc[i] = c;
    c = ((a + 1ULL) * c) & MASK;
    a = (a * a) & MASK;
  }
}
NQ_HD unsigned long long lcg_jump(const unsigned long long* A, const unsigned long long* Cc, unsigned long long seed, unsigned long long j) {
  const unsigned long long MASK = (1ULL << 48) - 1;
  for (int i = 0; j; ++i, j >>= 1)
    if (j & 1ULL) seed = (A[i] * seed + Cc[i]) & MASK;
  return seed;
}
// value of Random.nextInt(32767) taken from state `s` (the state AFTER the step); rejected = the reference would draw again
NQ_HD int next_int_from(unsigned long long s, bool* rejected) {
  const int u = (int)(s >> 17), r = u % 32767;
  *rejected = (int)((unsigned)(u - r) + 32766u) < 0;
  return r;
}

NQ_HD bool lcg_rejects(unsigned long long s) { return (unsigned)(s >> 17) >= 0x7FFFFFFEu; }   // next(31) in {2^31 - 2, 2^31 - 1}: u - u % 32767 + 32766 overflows
// generator step that delivers draw d (1-based): the d-th step nextInt does not reject
template <class SC>
NQ_HD unsigned long long lcg_step_of(const SC& C, unsigned long long d) {
  unsigned long long j = 0;
  while (j < (unsigned long long)C.nrej && (unsigned long long)C.rej[j] <= d + j) ++j;
  return d + j;
}
NQ_HD Lab4 lab_at(uint32_t c, const double* lut) {
#if defined(__CUDA_ARCH__)
  return lab_of(c);                      // 2^24-entry table (nq_hist.cuh)
#else
  Lab4 l = rgb2lab(0xFF000000u | c, lut);
  l.alpha = (float)(c >> 24);
  return l;
#endif
}
NQ_HD float tanh_f(double x) {            // (float) Math.tanh(x) (GC:255)
#if defined(__CUDA_ARCH__)
  float v;
  if (tanh_fast(x, &v)) return v;        // nq_dither.cuh: same float whenever it answers
#endif
  return (float)nqm::nq_tanh(x);
}
NQ_HD float coeff(int i, int j) {         // PQ:26-30
  constexpr float k[3][3] = {{0.299f, 0.587f, 0.114f}, {-0.14713f, -0.28886f, 0.436f}, {0.615f, -0.51499f, -0.10001f}};
  return k[i][j];
}

// ---- tables --------------------------------------------------------------------------------------------------
NQ_HD void fill_tables(SpecConst& C, const double* lut) {
  for (int v = 0; v < 256; ++v) {
    const double dv = (double)v;
    double r = C.PR * (1 - C.ratio) * (dv * dv), g = C.PG * (1 - C.ratio) * (dv * dv), b = C.PB * (1 - C.ratio) * (dv * dv);
    for (int i = 0; i < 3; ++i) {
      double t0 = (double)(coeff(i, 0) * (float)v), t1 = (double)(coeff(i, 1) * (float)v), t2 = (double)(coeff(i, 2) * (float)v);
      r += C.ratio * (t0 * t0); g += C.ratio * (t1 * t1); b += C.ratio * (t2 * t2);
    }
    C.Tr[v] = r; C.Tg[v] = g; C.Tb[v] = b;
  }
  for (int i = 0; i < C.plen; ++i) C.palLab[i] = lab_at(C.pal[i], lut);
  lcg_tables(C.jmpA, C.jmpC, 40);
}

// exact cost of palette entry c2 for colour c in the reference's operation order (PL:421-446), no semi-transparency
NQ_HD double closest_err(const SpecConst& C, uint32_t c2, int cr, int cg, int cb) {
  const int ir = c_red(c2) - cr, ig = c_green(c2) - cg, ib = c_blue(c2) - cb;
  const double dr = (double)ir, dg = (double)ig, db = (double)ib;
  double err = C.PR * (1 - C.ratio) * (dr * dr);
  err += C.PG * (1 - C.ratio) * (dg * dg);
  err += C.PB * (1 - C.ratio) * (db * db);
  for (int i = 0; i < 3; ++i) {
    double t0 = (double)(coeff(i, 0) * (float)ir);
    err += C.ratio * (t0 * t0);
    double t1 = (double)(coeff(i, 1) * (float)ig);
    err += C.ratio * (t1 * t1);
    double t2 = (double)(coeff(i, 2) * (float)ib);
    err += C.ratio * (t2 * t2);
  }
  return err;
}
// where the top-2 scan reads the palette and the per-channel cost tables from (global memory: SpecConst; stage 6 keeps
// copies in shared memory)
struct ScanTabs { const uint32_t* pal; const double *Tr, *Tg, *Tb; int plen; };
NQ_HD ScanTabs scan_tabs(const SpecConst& C) { ScanTabs T; T.pal = C.pal; T.Tr = C.Tr; T.Tg = C.Tg; T.Tb = C.Tb; T.plen = C.plen; return T; }
NQ_HD unsigned top2_key(const SpecConst& C, const ScanTabs& T, int k, int cr, int cg, int cb) {
  const uint32_t c2 = T.pal[k];
  const int ar = c_red(c2) - cr, ag = c_green(c2) - cg, ab = c_blue(c2) - cb;
  const double a = T.Tr[ar < 0 ? -ar : ar] + T.Tg[ag < 0 ? -ag : ag] + T.Tb[ab < 0 ? -ab : ab];
  int d = j2i(a);
  const double fr = a - (double)d;
  if (fr < 1e-6 || fr > 1.0 - 1e-6) d = j2i(closest_err(C, c2, cr, cg, cb));   // only floor(err) is compared (PL:448-456)
  return ((unsigned)d << 8) | (unsigned)k;
}
// the two smallest (floor(err), index) pairs = closest[0..3] of PL:418-458
NQ_HD void top2(const SpecConst& C, const ScanTabs& T, const unsigned char* cells, uint32_t c, unsigned* k0, unsigned* k1) {
  const int cr = c_red(c), cg = c_green(c), cb = c_blue(c);
  unsigned a0 = NQS_NONE, a1 = NQS_NONE;
  int cnt = 255;
  unsigned w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (cells) {
    const unsigned* cell = reinterpret_cast<const unsigned*>(cells + 32 * (size_t)(((cr >> 3) << 10) | ((cg >> 3) << 5) | (cb >> 3)));
#if defined(__CUDA_ARCH__)
    const uint4 lo = __ldg(reinterpret_cast<const uint4*>(cell)), hi = __ldg(reinterpret_cast<const uint4*>(cell) + 1);
    w[0] = lo.x; w[1] = lo.y; w[2] = lo.z; w[3] = lo.w; w[4] = hi.x; w[5] = hi.y; w[6] = hi.z; w[7] = hi.w;
#else
    for (int q = 0; q < 8; ++q) w[q] = cell[q];
#endif
    cnt = (int)(w[0] & 255u);
  }
  if (cnt != 255) {
    for (int j = 1; j <= cnt; ++j) {
      const unsigned key = top2_key(C, T, (int)((w[j >> 2] >> (8 * (j & 3))) & 255u), cr, cg, cb);
      const unsigned t = key > a0 ? key : a0;
      a0 = key < a0 ? key : a0;
      a1 = a1 < t ? a1 : t;
    }
  } else {
    for (int k = 0; k < T.plen; ++k) {
      const unsigned key = top2_key(C, T, k, cr, cg, cb);
      const unsigned t = key > a0 ? key : a0;
      a0 = key < a0 ? key : a0;
      a1 = a1 < t ? a1 : t;
    }
  }
  *k0 = a0; *k1 = a1;
}
NQ_HD void top2(const SpecConst& C, const unsigned char* cells, uint32_t c, unsigned* k0, unsigned* k1) { top2(C, scan_tabs(C), cells, c, k0, k1); }

// PnnLABQuantizer.nearestColorIndex without its memo (PL:337-401), palettes of more than 32 colours, no semi-transparency
NQ_HD int nearest_nomemo(const SpecConst& C, uint32_t c, const double* lut) {
  int k = 0;
  if (c_alpha(c) <= 0xF) c = C.transColor;
  if (C.plen > 2 && C.hasTrans && c_alpha(c) > 0xF) k = 1;
  const Lab4 l1 = lab_at(c, lut);
  double best = 1e300;
  int bi = -1;
  for (int i = k; i < C.plen; ++i) {
    const Lab4 l2 = C.palLab[i];
    float dl = l2.L - l1.L;
    double cur = (double)(dl < 0.f ? -dl : dl);
    const double da = (double)(l2.A - l1.A), db = (double)(l2.B - l1.B);
    cur += nqm::sqrt_((da * da) + (db * db));
    if (cur <= best) { best = cur; bi = i; }            // strict > pruning: the last minimal index wins (PL:397-400)
  }
  if (!(best <= 2147483647.0) || bi < 0) bi = k;         // mindist starts at Integer.MAX_VALUE
  return bi;
}

// GilbertCurve.normalDistribution (GC:114-123)
NQ_HD float normal_dist(float x, float peak) {
  const float mean = .5f, stdDev = .1f;
  const double d = (double)(x - mean), sd = (double)stdDev;
  const double exponent = -(d * d) / (2 * (sd * sd));
  const double pdf = (1 / (sd * nqm::sqrt_(2 * 3.141592653589793))) * nqm::nq_exp(exponent);
  const double maxPdf = 1 / (sd * nqm::sqrt_(2 * 3.141592653589793));
  const double scaledPdf = (pdf / maxPdf) * (double)peak;
  return (float)dmax(0.0, dmin((double)peak, scaledPdf));
}
NQ_HD double ydiff_pre(double ypix, uint32_t c, const double* lut) { return nqm::fabs_(color_y(c, lut) - ypix) * 100; }

// ditherPixel (GC:125-185) with qPixels[bidx] == 0, evaluated without the diffused colour; false when the reference's
// result would read it. Requires plen > 64 and 2 * (plen - margin) > 101 (GC:137 then holds for any colour).
NQ_HD bool pre_colour(const SpecConst& C, const SpecWork& W, int x, int y, uint32_t pixel, float sal, double ypix, uint32_t* out) {
  const int plen = C.plen, margin = C.margin;
  const float beta = C.beta;
  const uint32_t qcol = C.pal[0];
  const float strength = 1 / 3.f;
  const int acceptedDiff = plen - margin > 2 ? plen - margin : 2;
  const float kappa = sal < .6f ? beta * .15f / sal : beta * .4f / sal;
  uint32_t c2 = bn_diffuse(pixel, qcol, kappa, strength, x, y, W.bn);
  const double gamma = (double)beta;                      // plen > 32
  if (ydiff_pre(ypix, c2, W.lut) > (gamma * acceptedDiff)) return false;   // GC:149-172 reads r_pix..a_pix
  if (C.DM < 16 && sal < .6f && ydiff_pre(ypix, c2, W.lut) > (double)(margin - 1)) return false;   // GC:175
  if ((double)sal > .95) {
    const float k2 = beta * fmaxf(.05f, .75f - plen / 128.f) * sal;
    c2 = bn_diffuse(pixel, qcol, k2, strength, x, y, W.bn);
  }
  *out = c2;
  return true;
}

// ditherPixel (GC:125-185) in full for plen > 64, qPixels[bidx] == 0: the colour that is looked up
NQ_HD uint32_t slow_colour(const SpecConst& C, const SpecWork& W, int x, int y, uint32_t pixel, float sal, double ypix, uint32_t c2) {
  const int plen = C.plen, margin = C.margin;
  const double weight = C.gWeight;
  const float beta = C.beta;
  const uint32_t qcol = C.pal[0];
  const int r_pix = c_red(c2), g_pix = c_green(c2), b_pix = c_blue(c2), a_pix = c_alpha(c2);
  const float strength = 1 / 3.f;
  const int acceptedDiff = plen - margin > 2 ? plen - margin : 2;
  if (ydiff_pre(ypix, c2, W.lut) < (double)(2 * acceptedDiff)) {
    const float kappa = sal < .6f ? beta * .15f / sal : beta * .4f / sal;
    c2 = bn_diffuse(pixel, qcol, kappa, strength, x, y, W.bn);
  }
  const double gamma = (double)beta;
  if (ydiff_pre(ypix, c2, W.lut) > (gamma * acceptedDiff)) {
    if (margin > 6) {                                      // gamma > beta cannot hold for plen > 32
      float kappa = sal < .4f ? beta * .4f * sal : beta * .4f / sal;
      uint32_t c1 = c_argb(a_pix, r_pix, g_pix, b_pix);
      if ((double)sal < .9)
        kappa = beta * normal_dist(sal, 2.f);
      else {
        if (weight >= .0015 && (double)sal < .6) c1 = pixel;
        if (weight >= .005 && (double)sal < .6)
          kappa = beta * normal_dist(sal, weight < .0008 ? 2.5f : 1.75f);
        else {                                             // plen >= 32
          const double ub = 1 - plen / 320.0;
          if ((double)sal > .15 && (double)sal < ub)
            kappa = beta * (weight < .0025 ? .55f : .5f) / sal;   // !sortedByYDiff in this mode
          else
            kappa = beta * normal_dist(sal, weight < .0025 ? 1.82f : 2.f);
        }
      }
      c2 = bn_diffuse(c1, qcol, kappa, strength, x, y, W.bn);
    } else
      c2 = c_argb(a_pix, r_pix, g_pix, b_pix);
  }
  if (C.DM < 16 && sal < .6f && ydiff_pre(ypix, c2, W.lut) > (double)(margin - 1))
    c2 = c_argb(a_pix, r_pix, g_pix, b_pix);
  if ((double)sal > .95) {
    const float kappa = beta * fmaxf(.05f, .75f - plen / 128.f) * sal;
    c2 = bn_diffuse(pixel, qcol, kappa, strength, x, y, W.bn);
  }
  return c2;
}

NQ_HD float saliency_of(const SpecConst& C, const SpecWork& W, uint32_t px) {     // PL:155-156, 503-506
  uint32_t sp = px;
  if (C.salReplaced && (sp >> 24) <= 0xF) sp = C.transColor;
  const Lab4 l = lab_at(sp, W.lut);
  const float saliencyBase = .1f;
  return saliencyBase + (1 - saliencyBase) * l.L / 100.f * l.alpha / 255.f;
}

// closestColorIndex (PL:406-474) after the top-2 scan: which entry, and whether nearestColorIndex takes over
NQ_HD int closest_pick(const SpecConst& C, uint32_t c, unsigned k0, unsigned k1, int r, bool* needNear) {
  const int c0 = k0 == NQS_NONE ? 0 : (int)(k0 & 255u), d0 = k0 == NQS_NONE ? 0x7fffffff : (int)(k0 >> 8);
  const int c1 = k1 == NQS_NONE ? c0 : (int)(k1 & 255u), d1 = k1 == NQS_NONE ? 0x7fffffff : (int)(k1 >> 8);
  int idx = 1;
  if (d0 == 0) idx = 0;
  else {
    const int sum = (int)((unsigned)d1 + (unsigned)d0);
    if ((r % sum) <= d1) idx = 0;
  }
  const int ci = idx ? c1 : c0, ei = idx ? d1 : d0;
  *needNear = ei >= C.plen || ci == 0 || c_alpha(C.pal[ci]) < c_alpha(c);        // PL:470-472
  return ci;
}

// ---- stage 1: one pixel of the curve ------------------------------------------------------------------------
NQ_HD void stage_pre(const SpecConst& C, const ScanTabs& T, const SpecWork& W, int n) {
  const uint32_t xy = W.order[n];
  const int x = (int)(xy & 0xFFFF), y = (int)(xy >> 16);
  const uint32_t px = W.in[x + y * C.width];
  W.cpx[n] = px;
  const float sal = saliency_of(C, W, px);
  const double ypix = color_y(px, W.lut);
  uint32_t c = px;                                         // error-dependent lookups: predict the draw with the undiffused pixel
  unsigned flag = 0;
  if (!(C.plen >= 256 && sal > .99f) && pre_colour(C, W, x, y, px, sal, ypix, &c)) flag |= NQS_F_PRE;   // GC:214-215
  else c = px;
  unsigned k0 = NQS_NONE, k1 = NQS_NONE;
  const bool viaClosest = c_alpha(c) > 0xF;                // PL:407-408
  if (viaClosest) {
    top2(C, T, W.cells, c, &k0, &k1);
    if ((k0 >> 8) != 0u) flag |= NQS_F_DRAW;               // short-circuit: no draw when closest[2] == 0 (PL:467)
    else if (!(flag & NQS_F_PRE)) {
      // The pixel itself costs 0 (it is a palette colour): the reference draws unless the DIFFUSED colour is that colour
      // too, i.e. unless the errors around it are zero. Guess from the previous pixel of the curve: if that one is not a
      // zero-cost colour either, its error is not zero and this lookup will draw; in a flat run of palette colours it
      // will not. Only a prediction -- stage 7 corrects what it gets wrong.
      bool flat = n == 0;
      if (n > 0) {
        const uint32_t pxy = W.order[n - 1];
        const uint32_t ppx = W.in[(int)(pxy & 0xFFFF) + (int)(pxy >> 16) * C.width];
        unsigned p0 = NQS_NONE, p1 = NQS_NONE;
        if (c_alpha(ppx) > 0xF) top2(C, T, W.cells, ppx, &p0, &p1);
        flat = (p0 >> 8) == 0u;
      }
      if (flat) flag |= NQS_F_RISK; else flag |= NQS_F_DRAW;
    }
  }
  W.ccol[n] = c; W.ck0[n] = k0; W.ck1[n] = k1;
  W.cflag[n] = (unsigned char)flag;
}

NQ_HD void stage_pre(const SpecConst& C, const SpecWork& W, int n) { stage_pre(C, scan_tabs(C), W, n); }

// ---- stage 3: the draw, the choice between the two candidates, first-seen positions of the memo keys -------
// (stage 2 = exclusive prefix sum of NQS_F_DRAW into cdraw). Returns false when a nextInt would have rejected.
NQ_HD int memo_key(const SpecConst& C, uint32_t c) { return color_index(c, false, C.hasTrans != 0); }   // PL:332
NQ_HD bool stage_resolve(const SpecConst& C, const SpecWork& W, int n, int* firstPosOut /* key or -1 */, const unsigned long long* state = nullptr) {
  *firstPosOut = -1;
  const unsigned flag = W.cflag[n] & ~NQS_F_NEAR;          // (a re-resolve after a draw misprediction starts over)
  W.cflag[n] = (unsigned char)flag;
  if (!(flag & NQS_F_PRE)) return true;
  const uint32_t c = W.ccol[n];
  bool needNear = true;
  int qi = 0;
  bool ok = true;
  if (c_alpha(c) > 0xF) {
    int r = 0;
    if (flag & NQS_F_DRAW) {
      bool rej;
      r = next_int_from(state ? *state : lcg_jump(C.jmpA, C.jmpC, C.seed0, lcg_step_of(C, (unsigned long long)W.cdraw[n] + 1ULL)), &rej);
      ok = !rej;
    }
    qi = closest_pick(C, c, W.ck0[n], W.ck1[n], r, &needNear);
  }
  if (needNear) {
    if (C.isNano) {
      W.cflag[n] = (unsigned char)(flag | NQS_F_NEAR);
      *firstPosOut = memo_key(C, c);                       // caller: firstPos[key] = min(firstPos[key], n)
    } else
      W.cq[n] = (unsigned short)nearest_nomemo(C, c, W.lut);   // full-colour key: the memo is a pure cache (PL:332)
  } else
    W.cq[n] = (unsigned short)qi;
  return ok;
}
// ---- gate after stage 3 (state[7] = pixels flagged NQS_F_RISK): too many likely mispredictions, do not start
NQ_HD void stage_gate(const SpecConst& C, const SpecWork& W) {
  if (W.state[7] > NQS_MAXRISK) { W.state[1] = 1; W.state[11] = 1; }
  if (W.state[8] > (C.npix >> 4)) { W.state[1] = 1; W.state[11] = 2; }           // state[8] = error-dependent lookups: past 6 % of the image the sequential runs (and their notes) outgrow this scheme
}
// ---- stage 4: one memo key ------------------------------------------------------------------------------------
// `after`: only entries first seen behind that curve position (-1 = all); the others are settled
NQ_HD void stage_memo(const SpecConst& C, const SpecWork& W, int key, int after) {
  const int n = W.firstPos[key];
  if (n != NQS_NOPOS && n <= after) return;
  // an entry that an error-dependent lookup of a validated segment created in front of the first pre-lookup stands (PL:402)
  if (W.slowPos[key] != NQS_NOPOS && (n == NQS_NOPOS || W.slowPos[key] < n)) { W.memo[key] = W.slowVal[key]; return; }
  W.memo[key] = n == NQS_NOPOS ? (unsigned short)0xFFFF : (unsigned short)nearest_nomemo(C, W.ccol[n], W.lut);
}
// ---- stage 5 ------------------------------------------------------------------------------------------------------
NQ_HD void stage_fill(const SpecConst& C, const SpecWork& W, int n) {
  if (W.cflag[n] & NQS_F_NEAR) W.cq[n] = W.memo[memo_key(C, W.ccol[n])];
}
// ---- stage 5b: the packed record of one pixel (again after a patch or a re-resolve) -------------------------------
NQ_HD size_t rec_index(const SpecConst& C, int n) { return (size_t)(n % C.seg) * (size_t)C.nseg + (size_t)(n / C.seg); }
NQ_HD void stage_pack(const SpecConst& C, const SpecWork& W, int n) {
  const uint32_t xy = W.order[n];
  const int bidx = (int)(xy & 0xFFFF) + (int)(xy >> 16) * C.width;
  SpecRec r;
  r.px = W.cpx[n];
  r.xy = xy;
  r.qf = (uint32_t)W.cq[n] | ((uint32_t)W.cflag[n] << 16) | (W.bn[bidx & 4095] > C.thresold ? 1u << 24 : 0u);
  r.sal = (W.cflag[n] & NQS_F_PRE) ? 0.f : saliency_of(C, W, r.px);
  W.rec[rec_index(C, n)] = r;
}
// ---- first step of a re-resolve: what stage 6 saw the error-dependent lookups do becomes the prediction
NQ_HD void stage_adopt(const SpecWork& W, int n) {
  const unsigned f = W.cflag[n];
  if (f & NQS_F_SEEN) W.cflag[n] = (unsigned char)((f & (15u & ~NQS_F_DRAW)) | ((f & NQS_F_ACT) ? NQS_F_DRAW : 0u));
}
// ---- re-resolve after a draw misprediction at curve position `from` = state[5] - 1 (stage_validate has corrected the
//      pixel's flag): stage 2 again, then per memo key this reset, then stages 3-5 for the pixels behind `from`
// (entries first seen at or behind curve position state[10] <= from + 1 are dropped: behind a draw that went against its
//  prediction inside a sequential run the pre-lookups were decided again by that run, and what they created are its notes)
NQ_HD void stage_rekey(const SpecWork& W, int key, int from) {
  const int rk = W.state[10] > 0 && W.state[10] <= from ? W.state[10] - 1 : from;
  if (W.firstPos[key] != NQS_NOPOS && W.firstPos[key] > rk) { W.firstPos[key] = NQS_NOPOS; W.memo[key] = 0xFFFF; }
}
// ---- patch: an error-dependent lookup at curve position state[3] created memo entry state[2] - 1 BEFORE the first
//      pre-lookup that needs it, with another value than stage 4 gave it (PL:402: the first colour of a bucket fixes
//      it). stage_validate has already corrected memo/firstPos; every later pre-lookup of that key is redirected and
//      its segment re-runs. One call per pixel.
NQ_HD void stage_patch(const SpecConst& C, const SpecWork& W, int n) {
  const int cnt = W.state[2];
  if (cnt <= 0 || n <= W.state[3] || !(W.cflag[n] & NQS_F_NEAR)) return;
  const int mine = memo_key(C, W.ccol[n]);
  for (int i = 0; i < cnt; ++i) {
    if (W.patch[2 * i] == mine && n > W.patch[2 * i + 1]) {
      W.cq[n] = W.memo[mine];
      W.segs[n / C.seg].dirty = 1;                           // benign race on the device: every writer stores 1
    }
  }
}

// ---- stage 6: one segment ---------------------------------------------------------------------------------------
// An error-dependent lookup (GC:214-216 with the diffused colour c2): closestColorIndex with the draw this pixel
// was predicted to make, nearestColorIndex through the memo. `owned` = the pixel belongs to the segment (notes kept).
// java.util.Random addressed by draw index, for a caller that asks for (mostly) increasing indices: the state of the last
// index is kept and stepped forward; only a long way ahead (or back) takes the O(log) jump from the seed.
struct LcgCursor { unsigned long long state; unsigned idx; int valid; };
NQ_HD unsigned long long lcg_state_at(const SpecConst& C, LcgCursor& L, unsigned draw) {   // state that delivers draw `draw` (1-based)
  const unsigned long long MASK = (1ULL << 48) - 1;
  const unsigned idx = (unsigned)lcg_step_of(C, (unsigned long long)draw);                 // generator steps from the seed
  if (L.valid && idx >= L.idx && idx - L.idx <= 24u) {
    for (unsigned k = L.idx; k < idx; ++k) L.state = (L.state * 0x5DEECE66DULL + 0xBULL) & MASK;
  } else
    L.state = lcg_jump(C.jmpA, C.jmpC, C.seed0, (unsigned long long)idx);
  L.idx = idx; L.valid = 1;
  return L.state;
}
// nearestColorIndex through the first-seen memo for a lookup made inside stage 6 (PL:332-335, 402). `trust` = pre-lookup
// entries (firstPos / memo) first seen before that curve position are the sequential run's too. Entries created by
// stage-6 lookups are notes: of this segment, of the earlier segments of the same chain (chainFirst .. S - 1), and of
// validated segments (slowPos / slowVal).
NQ_HD int near_lookup(const SpecConst& C, const SpecWork& W, SpecSeg& S, int chainFirst, int n, int trust, uint32_t c, bool owned) {
  if (!C.isNano) return nearest_nomemo(C, c, W.lut);
  const int key = color_index(c, false, C.hasTrans != 0);
  if (owned) {
    for (int i = 0; i < S.nnotes && i < NQS_NOTES; ++i) if (S.noteKey[i] == key) return S.noteVal[i];
    for (const SpecSeg* P = &S - 1; P >= W.segs + chainFirst; --P)
      for (int i = 0; i < P->nnotes && i < NQS_NOTES; ++i) if (P->noteKey[i] == key) return P->noteVal[i];
  }
  if (W.slowPos[key] < n) return W.slowVal[key];           // created by an error-dependent lookup of a validated segment
  if (W.firstPos[key] < trust || (!owned && W.firstPos[key] != NQS_NOPOS)) {
    if (owned) {                                           // remembered: a later patch of this key invalidates the segment
      if (S.nreads < NQS_READS) S.readKey[S.nreads] = key;
      ++S.nreads;
    }
    return W.memo[key];
  }
  const int v = nearest_nomemo(C, c, W.lut);               // first colour of the bucket: this lookup fixes the entry (PL:402)
  if (owned) {
    if (S.nnotes < NQS_NOTES) { S.noteKey[S.nnotes] = key; S.notePos[S.nnotes] = n; S.noteVal[S.nnotes] = v; }
    ++S.nnotes;
  }
  return v;
}
// closestColorIndex (PL:406-474) for colour c whose top-2 keys are known, with the draw of index drawIdx + 1
NQ_HD int pick_lookup(const SpecConst& C, const SpecWork& W, SpecSeg& S, LcgCursor& L, int chainFirst, int n, int trust, unsigned drawIdx,
                      uint32_t c, unsigned k0, unsigned k1, bool owned, bool* drew) {
  *drew = false;
  bool needNear = true;
  int qi = 0;
  if (c_alpha(c) > 0xF) {
    int r = 0;
    if ((k0 >> 8) != 0u) {
      bool rej;
      r = next_int_from(lcg_state_at(C, L, drawIdx + 1u), &rej);
      if (rej) S.nnotes = NQS_NOTES + 1;                   // never seen; handled as an overflow = not validated
      *drew = true;
    }
    qi = closest_pick(C, c, k0, k1, r, &needNear);
  }
  if (!needNear) return qi;
  return near_lookup(C, W, S, chainFirst, n, trust, c, owned);
}

// ---- stage 6 proper -----------------------------------------------------------------------------------------------------
// DM is a template constant (DITHER_MAX is 9, 16 or 25, GC:96): the queue lives in registers as a window of DM + NQS_U boxes
// that slides one box per pixel and is moved back every NQS_U pixels, the weights are compile-time-indexed operands (constant
// bank on the device). For images whose pixels all have alpha 255 and whose palette alphas are 254 or 255 (NCH == 3) the
// alpha channel shrinks to one bit per box: the alpha sum 255 + (errors >= 0) never drops below 255, so a_pix is always 255
// and the error of a box is 255 - palette alpha = 0 or 1 (a palette alpha of 254 is the reference's float mean of 255s,
// PL:301-305); the sum itself still feeds maxErr (GC:192-201).
#define NQS_U 4                 // pixels per group: one slide of the register window per NQS_U pixels

#if defined(__CUDACC__)
__constant__ float c_specW[3][NQ_MAXQ + 3];   // initWeights(9 | 16 | 25), written once per context (k_spec_tables + cudaMemcpyToSymbol)
#endif
#if defined(__CUDA_ARCH__)
#define NQS_W(C, DMI, k) c_specW[DMI][k]
NQ_HD float max3f(float a, float b, float c) { float d; asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c)); return d; }
#define NQS_NOINLINE __noinline__
#else
#define NQS_W(C, DMI, k) (C).w[k]
NQ_HD float max3f(float a, float b, float c) { const float m = a > b ? a : b; return m > c ? m : c; }
#define NQS_NOINLINE
#endif

// (float) Math.tanh(e / maxErr * 20) (GC:255). e is an integer in [-255, 255] and maxErr is exactly 255 nearly always, so
// the value comes from a 511-entry table of exactly this expression (tab, nullptr = compute); otherwise it is evaluated.
#if defined(__CUDA_ARCH__)
__device__ NQS_NOINLINE float shape_tanh_eval(float e, float maxErr) { return tanh_f((double)(e / maxErr * 20.f)); }
#else
inline float shape_tanh_eval(float e, float maxErr) { return tanh_f((double)(e / maxErr * 20.f)); }
#endif
NQ_HD float shape_tanh(float e, float maxErr, const float* tab) {
  if (tab && maxErr == 255.f) return tab[(int)e + 255];
  return shape_tanh_eval(e, maxErr);
}

struct WarpRing;                // the staged record stream of a warp (device only, below)
struct RunEnv {                 // what the pixel step needs besides the queue
  const SpecConst* C;
  const SpecWork* W;
  SpecSeg* S;
  ScanTabs T;                   // palette and cost tables (shared memory copies on the device)
  const float* tanhTab;         // shape_tanh
  float fDitherMax, fDitherMax1, divisor;
  bool illusion0;
  int draws;                    // draws made by the pixels of the current span
  int nslow;                    // error-dependent lookups of the current span
  bool seq;                     // sequential truth: the run started from an exact state and addresses java.util.Random by the
                                // draws it has really made (actIdx), re-deciding the pre-lookups behind a deviation
  int chainFirst;               // first segment of the chain this thread runs
  int devPos;                   // seq: curve position of the first draw that went against its prediction (NQS_NOPOS: none yet)
  unsigned actIdx;              // seq: draws really made in front of the current pixel
  unsigned drawIdx;             // draws PREDICTED in front of the current pixel = cdraw[n], kept up from the records' flags
  unsigned amask;               // three-channel variant: alpha error (0 or 1) of queue box k in bit k, oldest box first
  WarpRing* ring;               // device: this warp's staged record stream (nullptr: per-thread loads)
  unsigned ringPhase;           // parity of the next phase of the ring's two mbarriers
  LcgCursor lcg;
};

// the quantization of an error-dependent lookup (GC:211-229 with the diffused colour), kept out of the hot loop
NQ_HD int run_slow_pixel_body(RunEnv& X, int n, uint32_t px, uint32_t xy, unsigned flag, int a_pix, int r_pix, int g_pix, int b_pix, bool owned,
                              int* drawn) {
  const SpecConst& C = *X.C;
  const SpecWork& W = *X.W;
  const float sal = W.rec[rec_index(C, n)].sal;            // (kept out of the registers of the hot loop)
  const int x = (int)(xy & 0xFFFFu), y = (int)(xy >> 16);
  const uint32_t c2 = c_argb(a_pix, r_pix, g_pix, b_pix);
  uint32_t c = c2;
  if (!(C.plen >= 256 && sal > .99f)) c = slow_colour(C, W, x, y, px, sal, color_y(px, W.lut), c2);
  unsigned k0 = NQS_NONE, k1 = NQS_NONE;
  if (c_alpha(c) > 0xF) top2(C, X.T, W.cells, c, &k0, &k1);
  bool drew;
  const int trust = X.seq && X.devPos < n ? X.devPos : n;
  const int qi = pick_lookup(C, W, *X.S, X.lcg, X.chainFirst, n, trust, X.seq ? X.actIdx : X.drawIdx, c, k0, k1, owned, &drew);
  *drawn = drew ? 1 : 0;
  if (owned) {
    // What this lookup did is the prediction from now on (the flag in the packed record is the one this run was resolved with).
    W.cflag[n] = (unsigned char)((flag & 15u) | NQS_F_SEEN | (drew ? NQS_F_ACT : 0u));
    if (drew != ((flag & NQS_F_DRAW) != 0)) {
      // A draw against the prediction (PL:467): every later draw index of the image is off by one. A speculative segment
      // reports the first such pixel and is run again, from its predecessor's exact state, as sequential truth (stage 7);
      // a sequential run just goes on with the index it has really reached.
      if (!X.seq) { if (X.S->mispos < 0) X.S->mispos = n; }
      else if (X.devPos == NQS_NOPOS) X.devPos = n;
    }
  }
  return qi;
}
// sequential truth behind a deviation: the pre-lookup of pixel n decided again with the draw it really gets
NQ_HD int run_seq_pre_body(RunEnv& X, int n, bool owned) {
  const SpecWork& W = *X.W;
  bool drew;
  const int trust = X.devPos < n ? X.devPos : n;
  return pick_lookup(*X.C, W, *X.S, X.lcg, X.chainFirst, n, trust, X.actIdx, W.ccol[n], W.ck0[n], W.ck1[n], owned, &drew);
}
#if defined(__CUDA_ARCH__)
__device__ NQS_NOINLINE int run_slow_pixel(RunEnv& X, int n, uint32_t px, uint32_t xy, unsigned flag, int a_pix, int r_pix, int g_pix, int b_pix, bool owned, int* drawn) {
  return run_slow_pixel_body(X, n, px, xy, flag, a_pix, r_pix, g_pix, b_pix, owned, drawn);
}
__device__ NQS_NOINLINE int run_seq_pre(RunEnv& X, int n, bool owned) { return run_seq_pre_body(X, n, owned); }
#else
inline int run_slow_pixel(RunEnv& X, int n, uint32_t px, uint32_t xy, unsigned flag, int a_pix, int r_pix, int g_pix, int b_pix, bool owned, int* drawn) {
  return run_slow_pixel_body(X, n, px, xy, flag, a_pix, r_pix, g_pix, b_pix, owned, drawn);
}
inline int run_seq_pre(RunEnv& X, int n, bool owned) { return run_seq_pre_body(X, n, owned); }
#endif

// One pixel at window offset u: the queue is e[u .. u + DM - 1] (oldest first), the new box goes to e[u + DM].
template <int DM, int DMI, int NCH, int u, bool OWNED>
NQ_HD void run_pixel(RunEnv& X, float (&e)[DM + NQS_U][NCH], const SpecRec& rc, int n) {
  const SpecConst& C = *X.C;
  const uint32_t px = rc.px;
  // ---- error.p = pixel + sum(queue[i].p * weights[i]), oldest box first (GC:190-204)
  float a0 = (float)c_red(px), a1 = (float)c_green(px), a2 = (float)c_blue(px), a3 = (float)c_alpha(px);
  float maxErr = (float)(DM - 1);
#pragma unroll
  for (int k = 0; k < DM; ++k) {
    const float wk = NQS_W(C, DMI, k);
    a0 = a0 + e[u + k][0] * wk;
    a1 = a1 + e[u + k][1] * wk;
    a2 = a2 + e[u + k][2] * wk;
    maxErr = max3f(maxErr, a0, a1);
    if (NCH == 4) { a3 = a3 + e[u + k][NCH - 1] * wk; maxErr = max3f(maxErr, a2, a3); }
    else {
      // alpha error of box k is 0 or 1 (bit k of amask): 1.0f * w == w and a3 + 0.0f == a3, so this is the reference's sum
      a3 = a3 + (((X.amask >> k) & 1u) ? wk : 0.f);
      maxErr = fmaxf(maxErr, a2);
    }
  }
  if (NCH == 3) maxErr = fmaxf(maxErr, a3);                 // alpha partial sums never decrease: their maximum is the last one
  const int r_pix = (int)fminf(255.f, fmaxf(a0, 0.f)), g_pix = (int)fminf(255.f, fmaxf(a1, 0.f));
  const int b_pix = (int)fminf(255.f, fmaxf(a2, 0.f)), a_pix = NCH == 4 ? (int)fminf(255.f, fmaxf(a3, 0.f)) : 255;
  const unsigned flag = (rc.qf >> 16) & 0xFFu;
  // ---- quantize (GC:211-229)
  int qi, drawn;
  if (flag & NQS_F_PRE) {
    drawn = (flag & NQS_F_DRAW) ? 1 : 0;                    // whether a pre-lookup draws depends on its colour alone (PL:467)
    if (X.seq && X.actIdx != X.drawIdx) qi = run_seq_pre(X, n, OWNED);
    else qi = (int)(rc.qf & 0xFFFFu);
  } else {
    qi = run_slow_pixel(X, n, px, rc.xy, flag, a_pix, r_pix, g_pix, b_pix, OWNED, &drawn);
    ++X.nslow;
  }
  X.draws += drawn;
  X.actIdx += (unsigned)drawn;
  X.drawIdx += (flag & NQS_F_DRAW) ? 1u : 0u;               // the prefix every pre-lookup behind this pixel was resolved with
  const uint32_t pc = X.T.pal[qi];
  if (OWNED) X.W->out[(rc.xy & 0xFFFFu) + (rc.xy >> 16) * (uint32_t)C.width] = pc;   // dither == true: the palette colour (GC:278-279)
  // ---- error of this pixel and its shaping (GC:236-264)
  float e0 = (float)(r_pix - c_red(pc)), e1 = (float)(g_pix - c_green(pc)), e2 = (float)(b_pix - c_blue(pc));
  const bool s0 = fabsf_(e0) >= X.fDitherMax, s1 = fabsf_(e1) >= X.fDitherMax, s2 = fabsf_(e2) >= X.fDitherMax;
  if (s0 || s1 || s2) {
    if ((rc.qf >> 24) & 1u) {                              // diffuse = TELL_BLUE_NOISE[bidx & 4095] > thresold (GC:250)
      if (s0) e0 = shape_tanh(e0, maxErr, X.tanhTab) * X.fDitherMax1;
      if (s1) e1 = shape_tanh(e1, maxErr, X.tanhTab) * X.fDitherMax1;
      if (s2) e2 = shape_tanh(e2, maxErr, X.tanhTab) * X.fDitherMax1;
    } else if (X.illusion0) {
      if (s0) e0 = (float)((double)(e0 / maxErr) * 1.0) * X.fDitherMax1;
      if (s1) e1 = (float)((double)(e1 / maxErr) * 1.0) * X.fDitherMax1;
      if (s2) e2 = (float)((double)(e2 / maxErr) * 1.0) * X.fDitherMax1;
    } else {
      if (s0) e0 /= X.divisor;
      if (s1) e1 /= X.divisor;
      if (s2) e2 /= X.divisor;
    }
  }
  // ---- errorq.poll(); errorq.add(error) (GC:231, 276): the window slides
  e[u + DM][0] = e0; e[u + DM][1] = e1; e[u + DM][2] = e2;
  if (NCH == 4) e[u + DM][NCH - 1] = (float)(a_pix - c_alpha(pc));
  else X.amask = (X.amask >> 1) | ((unsigned)(255 - c_alpha(pc)) << (DM - 1));   // a_pix is 255, palette alphas are 254 or 255
}
template <int DM, int NCH, int BY>
NQ_HD void run_slide(float (&e)[DM + NQS_U][NCH]) {
#pragma unroll
  for (int k = 0; k < DM; ++k)
#pragma unroll
    for (int j = 0; j < NCH; ++j) e[k][j] = e[k + BY][j];
}
NQ_HD SpecRec run_fetch(const SpecRec* recs, int segLen, int nsegs, int n) {
  return recs[(size_t)(n % segLen) * (size_t)nsegs + (size_t)(n / segLen)];
}
// pixels [n0, n1) from the queue in e[0 .. DM - 1]; groups of NQS_U with the records of the next group in flight
#if defined(__CUDACC__)
// ---- the record stream of a warp through shared memory (sm_90+ bulk copies completing on an mbarrier) -------------------
// When the 32 lanes of a warp run 32 consecutive segments in step (the first launch of an image: same warm-up, same length),
// pixel k of the span needs ONE row of the segment-interleaved record matrix per warp: 32 x 16 = 512 contiguous bytes.
// Lane 0 fetches NQS_TROWS rows per stage with cp.async.bulk into a two-stage ring; the copies complete on the stage's
// mbarrier (complete_tx), every lane waits for its phase and reads its own 16-byte record with one LDS.128. Against the
// register prefetch (four records ahead per thread) this takes 24 registers out of the loop and puts a whole tile of loads
// in flight per instruction.
#define NQS_TROWS 8
__device__ int g_specBulk;       // 1: stage 6 streams its records through shared memory with bulk copies (nq_create: NQ_SPEC_BULK)
struct WarpRing {
  uint4 rec[2][NQS_TROWS][32];
  unsigned long long bar[2];
};
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_load(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src), "r"(bytes),
               "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  unsigned done;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  } while (!done);
}
#endif

template <int DM, int DMI, int NCH, bool OWNED>
NQ_HD void run_span(RunEnv& X, float (&e)[DM + NQS_U][NCH], int n0, int n1) {
  const SpecConst& C = *X.C;
  const SpecRec* const recs = X.W->rec;
  const int segLen = C.seg, nsegs = C.nseg;
  int n = n0;
  if (n0 < n1) X.drawIdx = X.W->cdraw[n0];
#if defined(__CUDA_ARCH__)
  if (X.ring) {
    // all 32 lanes here, consecutive segments, same offset and length, no wrap into the next column: the staged stream
    const unsigned lane = threadIdx.x & 31;
    const int len = n1 - n0, base = n0 - (int)lane * segLen;
    bool uni = __activemask() == 0xffffffffu;
    if (uni) uni = __all_sync(0xffffffffu, len >= 2 * NQS_TROWS && base == __shfl_sync(0xffffffffu, base, 0) && len == __shfl_sync(0xffffffffu, len, 0) &&
                                               (n0 % segLen) + len <= segLen && !X.seq);
    if (uni) {
      WarpRing& R = *X.ring;
      const int row0 = n0 % segLen, col0 = __shfl_sync(0xffffffffu, n0 / segLen, 0);
      const int ntile = (len + NQS_TROWS - 1) / NQS_TROWS;
      auto issue = [&](int t) {                              // lane 0: rows of tile t into stage t & 1
        const int st = t & 1, r0 = t * NQS_TROWS, nr = len - r0 < NQS_TROWS ? len - r0 : NQS_TROWS;
        mbar_expect_tx(&R.bar[st], (unsigned)nr * 512u);
        for (int r = 0; r < nr; ++r) bulk_load(&R.rec[st][r][0], recs + ((size_t)(row0 + r0 + r) * (size_t)nsegs + (size_t)col0), 512u, &R.bar[st]);
      };
      if (lane == 0) { issue(0); if (ntile > 1) issue(1); }
      for (int t = 0; t < ntile; ++t) {
        const int st = t & 1, r0 = t * NQS_TROWS, nr = len - r0 < NQS_TROWS ? len - r0 : NQS_TROWS;
        mbar_wait(&R.bar[st], (X.ringPhase >> st) & 1u);
        X.ringPhase ^= 1u << st;
        int r = 0;
        for (; r + NQS_U <= nr; r += NQS_U) {
          SpecRec rc[NQS_U];
#pragma unroll
          for (int u = 0; u < NQS_U; ++u) { const uint4 v = R.rec[st][r + u][lane]; rc[u].px = v.x; rc[u].xy = v.y; rc[u].qf = v.z; rc[u].sal = __uint_as_float(v.w); }
          run_pixel<DM, DMI, NCH, 0, OWNED>(X, e, rc[0], n);
          run_pixel<DM, DMI, NCH, 1, OWNED>(X, e, rc[1], n + 1);
          run_pixel<DM, DMI, NCH, 2, OWNED>(X, e, rc[2], n + 2);
          run_pixel<DM, DMI, NCH, 3, OWNED>(X, e, rc[3], n + 3);
          run_slide<DM, NCH, NQS_U>(e);
          n += NQS_U;
        }
        for (; r < nr; ++r, ++n) {
          const uint4 v = R.rec[st][r][lane];
          SpecRec rc; rc.px = v.x; rc.xy = v.y; rc.qf = v.z; rc.sal = __uint_as_float(v.w);
          run_pixel<DM, DMI, NCH, 0, OWNED>(X, e, rc, n);
          run_slide<DM, NCH, 1>(e);
        }
        __syncwarp();                                        // every lane has read the stage before it is refilled
        if (lane == 0 && t + 2 < ntile) issue(t + 2);
      }
      return;
    }
  }
#endif
  if (n + NQS_U <= n1) {
    // record (row, col) of pixel n in the segment-interleaved layout, advanced without a division per pixel
    int row = n % segLen, col = n / segLen;
    SpecRec cur[NQS_U], nxt[NQS_U];
#pragma unroll
    for (int u = 0; u < NQS_U; ++u) {
      cur[u] = recs[(size_t)row * (size_t)nsegs + (size_t)col];
      if (++row == segLen) { row = 0; ++col; }
    }
    for (; n + NQS_U <= n1; n += NQS_U) {
      const bool more = n + 2 * NQS_U <= n1;
      if (more) {
#pragma unroll
        for (int u = 0; u < NQS_U; ++u) {
          nxt[u] = recs[(size_t)row * (size_t)nsegs + (size_t)col];
          if (++row == segLen) { row = 0; ++col; }
        }
      }
      run_pixel<DM, DMI, NCH, 0, OWNED>(X, e, cur[0], n);
      run_pixel<DM, DMI, NCH, 1, OWNED>(X, e, cur[1], n + 1);
      run_pixel<DM, DMI, NCH, 2, OWNED>(X, e, cur[2], n + 2);
      run_pixel<DM, DMI, NCH, 3, OWNED>(X, e, cur[3], n + 3);
      run_slide<DM, NCH, NQS_U>(e);
      if (more) {
#pragma unroll
        for (int u = 0; u < NQS_U; ++u) cur[u] = nxt[u];
      }
    }
  }
  for (; n < n1; ++n) {                                     // fewer than NQS_U pixels left
    const SpecRec rc = run_fetch(recs, segLen, nsegs, n);
    run_pixel<DM, DMI, NCH, 0, OWNED>(X, e, rc, n);
    run_slide<DM, NCH, 1>(e);
  }
}
static_assert(NQS_U == 4, "run_span spells out the NQS_U pixel steps");

template <int DM, int DMI, int NCH>
NQ_HD void stage_run_t(const SpecConst& C, const SpecWork& W, int s, const ScanTabs& T, const float* tanhTab, WarpRing* ring = nullptr) {
  SpecSeg& S0 = W.segs[s];
  if (S0.done || !S0.dirty || S0.chained) return;
  const int p0 = s * C.seg;
  float e[DM + NQS_U][NCH];                                // the queue window, e[0] = oldest box
  unsigned amask0 = 0u;
  int from = p0;
  const bool seq = S0.exact != 0;                          // started from the exact state: this run IS the sequential algorithm
  if (S0.exact && p0 > 0) {
#pragma unroll
    for (int k = 0; k < DM; ++k)
#pragma unroll
      for (int j = 0; j < NCH; ++j) e[k][j] = S0.qstart[k][j];
    if (NCH == 3) for (int k = 0; k < DM; ++k) amask0 |= (S0.qstart[k][3] != 0.f ? 1u : 0u) << k;
  } else {
#pragma unroll
    for (int k = 0; k < DM; ++k)
#pragma unroll
      for (int j = 0; j < NCH; ++j) e[k][j] = 0.f;
    if (!S0.exact) { const long long w = (long long)C.warm * (long long)S0.warmMul; from = (long long)p0 - w > 0 ? (int)((long long)p0 - w) : 0; }
  }
  RunEnv X;
  X.C = &C; X.W = &W; X.S = &S0; X.T = T; X.tanhTab = tanhTab;
  X.lcg.valid = 0; X.lcg.idx = 0; X.lcg.state = 0; X.drawIdx = 0; X.amask = amask0;
  X.seq = seq; X.chainFirst = s; X.devPos = NQS_NOPOS; X.actIdx = 0; X.nslow = 0;
  X.ring = ring; X.ringPhase = 0u;
  X.fDitherMax = (float)C.ditherMax; X.fDitherMax1 = (float)(C.ditherMax - 1);
  X.divisor = (float)(1 + nqm::sqrt_((double)C.ditherMax));
  X.illusion0 = W.bn[0] > C.thresold;                      // yDiff == 1 in this mode: bn[(int)4096.0 & 4095] (GC:251-252)
  X.draws = 0;
  S0.nnotes = 0;
  S0.nreads = 0;
  S0.mispos = -1;
  if (from < p0) run_span<DM, DMI, NCH, false>(X, e, from, p0);    // warm-up: nothing is written, notes are not kept
  // a chain: the thread of an exact segment goes on through the following segments that hold error-dependent lookups
  // (stage 7 decides how many), handing each the exact state it needs
  int nchain = seq && S0.chain > 1 ? S0.chain : 1;
  if (s + nchain > C.nseg) nchain = C.nseg - s;
  X.actIdx = W.cdraw[p0];
  for (int c = 0; c < nchain; ++c) {
    SpecSeg& S = W.segs[s + c];
    const int q0 = (s + c) * C.seg, q1 = (q0 + C.seg < C.npix) ? q0 + C.seg : C.npix;
    X.S = &S;
    if (c > 0) {
      S.exact = 1; S.nnotes = 0; S.nreads = 0; S.mispos = -1;
#pragma unroll
      for (int k = 0; k < DM; ++k) { S.qstart[k][0] = e[k][0]; S.qstart[k][1] = e[k][1]; S.qstart[k][2] = e[k][2]; S.qstart[k][3] = NCH == 4 ? e[k][NCH - 1] : (float)((X.amask >> k) & 1u); }
    }
#pragma unroll
    for (int k = 0; k < DM; ++k) { S.qwarm[k][0] = e[k][0]; S.qwarm[k][1] = e[k][1]; S.qwarm[k][2] = e[k][2]; S.qwarm[k][3] = NCH == 4 ? e[k][NCH - 1] : (float)((X.amask >> k) & 1u); }
    X.draws = 0; X.nslow = 0;
    S.idx0 = X.actIdx;
    run_span<DM, DMI, NCH, true>(X, e, q0, q1);
#pragma unroll
    for (int k = 0; k < DM; ++k) { S.qout[k][0] = e[k][0]; S.qout[k][1] = e[k][1]; S.qout[k][2] = e[k][2]; S.qout[k][3] = NCH == 4 ? e[k][NCH - 1] : (float)((X.amask >> k) & 1u); }
    S.draws = X.draws;
    S.nslow = X.nslow;
    S.dev = seq ? X.devPos : NQS_NOPOS;
    S.dirty = 0;
  }
}
NQ_HD void stage_run(const SpecConst& C, const SpecWork& W, int s, const float* tanhTab) {
  const ScanTabs T = scan_tabs(C);
  if (C.opaque) {
    if (C.DM == 25) stage_run_t<25, 2, 3>(C, W, s, T, tanhTab);
    else if (C.DM == 16) stage_run_t<16, 1, 3>(C, W, s, T, tanhTab);
    else if (C.DM == 9) stage_run_t<9, 0, 3>(C, W, s, T, tanhTab);
  } else {
    if (C.DM == 25) stage_run_t<25, 2, 4>(C, W, s, T, tanhTab);
    else if (C.DM == 16) stage_run_t<16, 1, 4>(C, W, s, T, tanhTab);
    else if (C.DM == 9) stage_run_t<9, 0, 4>(C, W, s, T, tanhTab);
  }
}

// ---- stage 7: ordered validation of one image. Returns the number of segments still open. ------------------------
NQ_HD bool same_queue(const float (*a)[4], const float (*b)[4], int DM) {
  for (int k = 0; k < DM; ++k)
    for (int j = 0; j < 4; ++j)
      if (nqm::d2bits((double)a[k][j]) != nqm::d2bits((double)b[k][j])) return false;   // widening is exact and keeps the sign of zero
  return true;
}
// stage 6b, one call per segment (parallel): the comparison stage 7 needs, so that its sequential walk reads one flag
NQ_HD void stage_compare(const SpecConst& C, const SpecWork& W, int s) {
  SpecSeg& S = W.segs[s];
  if (S.done) return;
  S.qok = s == 0 || same_queue(S.exact ? S.qstart : S.qwarm, W.segs[s - 1].qout, C.DM);
  // A speculative segment whose warm-up did not reach its predecessor's state: do not wait for the ordered walk to get
  // here, try again at once with a four times longer warm-up (all such segments in parallel). The walk still decides.
  if (!S.qok && !S.exact && !S.dirty && S.warmMul < 64) { S.warmMul *= 4; S.dirty = 1; }
}
NQ_HD int stage_validate(const SpecConst& C, const SpecWork& W) {
  int s = W.state[0];
  if (W.state[1]) return 0;
  int delta = 0;                            // draws really made minus draws predicted, over the exact segments accepted in this call
  int minDev = NQS_NOPOS;                   // first draw against its prediction inside those segments
  for (; s < C.nseg; ++s) {
    SpecSeg& S = W.segs[s];
    const int p0 = s * C.seg, p1 = (p0 + C.seg < C.npix) ? p0 + C.seg : C.npix;
    if ((delta != 0 || minDev != NQS_NOPOS) && !S.exact) break;   // behind a shift of the draw indices only sequential truth counts: re-resolve first
    bool ok = S.nnotes <= NQS_NOTES && !S.dirty;            // (dirty: a patch touched it after its last run)
    if (ok && s > 0) ok = S.qok != 0;
    // An error-dependent lookup of a SPECULATIVE segment drew (or did not draw) against its prediction (PL:467: closest[2]
    // == 0 for the diffused colour but not for the pixel, or the reverse): behind that pixel the segment used wrong
    // draw indices. It is run again as sequential truth (below).
    if (ok && !S.exact && S.mispos >= 0) ok = false;
    // a sequential run is the truth only if it also started from the right draw index (a chain hands it on; the head of an
    // earlier chain may have been run again since)
    if (ok && S.exact && S.idx0 != W.cdraw[p0] + (unsigned)delta) ok = false;
    int predicted = 0;
    if (ok) {
      // the draws of the owned pixels against the prediction every later pre-lookup was computed with
      predicted = (int)(W.cdraw[p1] - W.cdraw[p0]);   // cdraw has npix + 1 entries
      if (S.draws != predicted && !S.exact) { W.state[1] = 1; W.state[11] = 3; return 0; }      // cannot happen without a mispos; kept as a guard
      for (int i = 0; i < S.nnotes; ++i) {
        const int key = S.noteKey[i], pos = S.notePos[i], val = S.noteVal[i];
        if (W.slowPos[key] < pos && W.slowVal[key] != val) { ok = false; break; }
      }
    }
#if defined(NQS_TRACE)
    if (!ok) fprintf(stderr, "  validate: segment %d fails (exact %d chained %d dirty %d qok %d mispos %d notes %d draws %d predicted %d)\n", s, S.exact, S.chained, S.dirty, S.qok, S.mispos, S.nnotes, S.draws, (int)(W.cdraw[p1] - W.cdraw[p0]));
#endif
    if (!ok) {
      if (S.exact && S.nnotes > NQS_NOTES) { W.state[1] = 1; W.state[11] = 4; return 0; }     // even the exact run overflows its notes
      // every failure costs a round in which one thread runs alone: past a quarter of the segments the serial kernel is cheaper
      if (++W.state[4] > (C.nseg >> 2) + 4) { W.state[1] = 1; W.state[11] = 5; return 0; }
      S.exact = 1; S.dirty = 1; S.chained = 0;
      if (s > 0) for (int k = 0; k < C.DM; ++k) for (int j = 0; j < 4; ++j) S.qstart[k][j] = W.segs[s - 1].qout[k][j];
      // its thread goes on through the following segments that hold error-dependent lookups: their draws are as uncertain
      int n = 1;
      while (n < NQS_MAXCHAIN && s + n < C.nseg && W.segs[s + n].nslow > 0 && !W.segs[s + n].done) {
        SpecSeg& N = W.segs[s + n];
        N.chained = 1; N.dirty = 1; N.exact = 1;
        ++n;
      }
      S.chain = n;
      break;
    }
    {
      // entries first created by an error-dependent lookup which the pre-lookups after it resolved differently: correct the
      // memo, ask for stage_patch (all of the segment's at once), and run the segment -- with its chain -- again (its own later
      // pixels read the entries too). Behind a draw that went against its prediction a sequential run decides the
      // pre-lookups itself and the re-resolve that follows drops what they had created (stage_rekey): nothing to patch there.
      int npatch = 0, first = NQS_NOPOS;
      for (int i = 0; i < S.nnotes && npatch < NQS_MAXPATCH; ++i) {
        const int key = S.noteKey[i], pos = S.notePos[i], val = S.noteVal[i];
        if (S.exact && S.dev != NQS_NOPOS && pos > S.dev) continue;
        if (W.slowPos[key] != NQS_NOPOS && W.slowPos[key] < pos) continue;      // agrees with an earlier entry (checked above)
        if (W.firstPos[key] != NQS_NOPOS && W.firstPos[key] > pos && W.memo[key] != (unsigned short)val) {
          W.memo[key] = (unsigned short)val; W.firstPos[key] = pos;
          W.patch[2 * npatch] = key; W.patch[2 * npatch + 1] = pos;
          ++npatch;
          if (pos < first) first = pos;
          for (int t = s + 1; t < C.nseg; ++t) {           // later segments whose error-dependent lookups read the old entry
            SpecSeg& T = W.segs[t];
            bool hit = T.nreads > NQS_READS;
            for (int r = 0; !hit && r < T.nreads; ++r) hit = T.readKey[r] == key;
            if (hit) { T.dirty = 1; if (!T.exact) { T.chained = 0; T.chain = 1; } }
          }
        }
      }
      if (npatch) {
        W.state[2] = npatch; W.state[3] = first;
        S.dirty = 1;
        if (S.exact && S.chain > 1) for (int t = 1; t < S.chain && s + t < C.nseg; ++t) { SpecSeg& N = W.segs[s + t]; if (!N.done) { N.chained = 1; N.dirty = 1; N.exact = 1; } }
        break;
      }
    }
    for (int i = 0; i < S.nnotes; ++i) {
      const int key = S.noteKey[i], pos = S.notePos[i], val = S.noteVal[i];
      if (W.slowPos[key] == NQS_NOPOS) { W.slowPos[key] = pos; W.slowVal[key] = (unsigned short)val; }
    }
    S.done = 1;
    S.chained = 0;
    delta += S.draws - predicted;
    if (S.exact && S.dev != NQS_NOPOS && S.dev < minDev) minDev = S.dev;
  }
  if (delta != 0 || minDev != NQS_NOPOS) {
    // The exact segments accepted above made another number of draws than predicted (stage 6 has corrected the flags of
    // their pixels): every draw index behind them moves. Ask for the prefix sum and stages 3-5 again behind position
    // s * seg - 1 (k_spec_redo_*) and run everything behind again.
    const int from = (s * C.seg < C.npix ? s * C.seg : C.npix) - 1;
    W.state[5] = from + 1;
    W.state[10] = minDev != NQS_NOPOS ? minDev + 1 : 0;
    for (int t = s; t < C.nseg; ++t) { SpecSeg& T = W.segs[t]; T.dirty = 1; T.chained = 0; T.chain = 1; if (T.exact && t > s) T.exact = 0; }
    if (++W.state[6] > NQS_MAXREDO) { W.state[1] = 1; W.state[11] = 6; return 0; }
  }
  W.state[0] = s;
  return C.nseg - s + (W.state[5] ? 1 : 0);   // a pending re-resolve keeps the image open even when every segment is done
}

#if defined(__CUDACC__) || defined(NQS_EMULATE)   // NQS_EMULATE: tests/spec_host_harness.cpp runs the kernels thread by thread on the CPU
// =====================================================================================================================
// Kernels: indexing only, every body is one of the stage functions above. One SpecImage per image of the batch. The
// per-pixel work arrays live in a pool of slots; an image is bound to a free slot when it is admitted (k_spec_admit)
// and gives it back when it is finished or handed back, so images of different ages share every launch ("rolling
// admission", spec_drive): grid.y indexes a LIST of images, not the batch.
// =====================================================================================================================
struct SpecImage {
  SpecConst C;
  SpecWork W;
  int eligible;
  int rounds;                    // validation rounds this image has been through
};
#define NQS_ACTIVE(P) ((P).eligible && !(P).W.state[1])
#define NQS_CHUNK 8192           // pixels per block of the draw-count prefix sum (stage 2)

// GilbertCurve / quantizer constants of every image, and which images this path takes (one thread per image).
// order: nullptr = every image walks its slot's own table (NqSlot::order); else one table for every image of the list (the
// CPU emulation of these kernels, tests/spec_host_harness.cpp, runs one size).
__global__ void k_spec_setup(NqImage* imgs, const NqSlot* slots, SpecImage* sp, const uint32_t* order, int nimg, int seg, int warm, int* eligOut) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nimg) return;
  NqImage& I = imgs[i];
  SpecImage& P = sp[i];
  SpecConst& C = P.C;
  const int plen = I.paletteLen;
  const int acceptedDiff = plen - I.gMargin > 2 ? plen - I.gMargin : 2;
  // PnnLABQuantizer, dither on, saliency map, ArrayDeque queue, opaque image (a transparent pixel leaves a constant alpha
  // error in the queue for ever: alpha is never shaped, GC:248), ditherPixel lookups independent of the diffused colour
  P.eligible = I.kind == NQ_KIND_LAB && I.dither && I.gUseSal && !I.gSorted && !I.gHasAlpha && !I.hasSemi && I.transIdx < 0 && !I.error &&
               plen > 64 && 2 * acceptedDiff > 101 && I.nmax > 2 && slots[i].cells != nullptr && I.npix >= 4 * seg;
  P.rounds = 0;
  // 1 = taken; 2 = not taken and k_dither_fifo runs its serial chain for it; 0 = another kernel's image
  eligOut[i] = P.eligible ? 1 : ((plen > 0 && !I.error && !I.gSorted) ? 2 : 0);
  I.specDone = P.eligible ? 2 : 0;                // 2 = pending here: k_dither_fifo leaves it alone until k_spec_finish has spoken
  if (!P.eligible) return;
  if (I.gDitherMaxQ != 9 && I.gDitherMaxQ != 16 && I.gDitherMaxQ != 25) { P.eligible = 0; eligOut[i] = 2; I.specDone = 0; return; }
  C.plen = plen; C.margin = I.gMargin; C.thresold = I.gThresold; C.DM = I.gDitherMaxQ; C.ditherMax = I.gDitherMax;
  C.width = I.width; C.npix = I.npix;
  C.isNano = I.isNano; C.hasTrans = I.transIdx >= 0; C.salReplaced = I.nmax < 128 && I.nmax > 2;
  C.seg = seg; C.warm = warm; C.nseg = (I.npix + seg - 1) / seg;
  C.transColor = I.transColor;
  C.gWeight = I.gWeight; C.PR = I.PR; C.PG = I.PG; C.PB = I.PB; C.ratio = I.ratioMerge;
  C.beta = I.gBeta;
  JRandom r; r.set_seed(I.seed);
  C.seed0 = r.seed;
  C.nrej = 0;
  for (int k = 0; k < NQ_MAXQ; ++k) C.w[k] = k < C.DM ? I.gWeights[k] : 0.f;
  int opaque = I.nonOpaque == 0;                  // ... and palette alphas of 254 or 255 (a mean of 255s can round to 254.99998, PL:301)
  for (int k = 0; k < plen; ++k) { C.pal[k] = I.palette[k]; opaque &= (I.palette[k] >> 24) >= 0xFEu; }
  C.opaque = opaque;
  // which instantiation of stage 6 runs this image: bits 8.. of the verdict (spec_drive groups the images by it)
  eligOut[i] |= (((C.DM == 25 ? 2 : (C.DM == 16 ? 1 : 0)) << 1) | (opaque ? 0 : 1)) << 8;
  P.W.order = order ? order : slots[i].order; P.W.in = slots[i].in; P.W.out = slots[i].out; P.W.cells = slots[i].cells;
  P.W.lut = g_gammaLut; P.W.bn = g_blueNoise;
  fill_tables(C, g_gammaLut);
}
// binds the images of `list` to their work-array slots: pool[slotOf[k]] holds the array pointers of that slot
__global__ void k_spec_admit(SpecImage* sp, const int* list, const int* slotOf, int cnt, const SpecWork* pool) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= cnt) return;
  SpecImage& P = sp[list[k]];
  const SpecWork& T = pool[slotOf[k]];
  SpecWork& W = P.W;
  W.cpx = T.cpx; W.ccol = T.ccol; W.ck0 = T.ck0; W.ck1 = T.ck1; W.cq = T.cq; W.cflag = T.cflag; W.rec = T.rec; W.cdraw = T.cdraw;
  W.firstPos = T.firstPos; W.memo = T.memo; W.slowPos = T.slowPos; W.slowVal = T.slowVal; W.segs = T.segs; W.state = T.state;
  W.chunkSum = T.chunkSum; W.patch = T.patch;
}
// The generator steps whose value Random.nextInt(32767) rejects, among the first npix + NQS_MAXREJ + 1 (every pixel draws at
// most once): 64 steps per thread from a jump to its first one. k_spec_rejsort orders the few that exist.
__global__ void __launch_bounds__(256) k_spec_rejects(SpecImage* sp, const int* list) {
  SpecImage& P = sp[list[blockIdx.y]];
  if (!P.eligible) return;
  const unsigned long long MASK = (1ULL << 48) - 1;
  const unsigned long long total = (unsigned long long)P.C.npix + NQS_MAXREJ + 1;
  for (unsigned long long base = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 64ULL; base < total;
       base += (unsigned long long)gridDim.x * blockDim.x * 64ULL) {
    unsigned long long st = lcg_jump(P.C.jmpA, P.C.jmpC, P.C.seed0, base);
    for (int k = 1; k <= 64 && base + (unsigned long long)k <= total; ++k) {
      st = (st * 0x5DEECE66DULL + 0xBULL) & MASK;
      if (lcg_rejects(st)) {
        const int at = atomicAdd(&P.C.nrej, 1);
        if (at < NQS_MAXREJ) P.C.rej[at] = (unsigned)(base + (unsigned long long)k);
      }
    }
  }
}
__global__ void k_spec_rejsort(SpecImage* sp, const int* list, int cnt) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= cnt) return;
  SpecImage& P = sp[list[k]];
  if (!P.eligible) return;
  if (P.C.nrej > NQS_MAXREJ) { P.C.nrej = 0; P.W.state[1] = 1; P.W.state[11] = 7; return; }   // (2 in 2^31 per step: never seen)
  for (int i = 1; i < P.C.nrej; ++i) {
    const unsigned v = P.C.rej[i];
    int j = i - 1;
    for (; j >= 0 && P.C.rej[j] > v; --j) P.C.rej[j + 1] = P.C.rej[j];
    P.C.rej[j + 1] = v;
  }
}
// memo tables, segment records, state (grid: x strides, y = list entry)
__global__ void __launch_bounds__(256) k_spec_init(SpecImage* sp, const int* list) {
  SpecImage& P = sp[list[blockIdx.y]];
  if (!P.eligible) return;
  const int t = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
  for (int k = t; k < 65536; k += nt) { P.W.firstPos[k] = NQS_NOPOS; P.W.slowPos[k] = NQS_NOPOS; P.W.memo[k] = 0xFFFF; P.W.slowVal[k] = 0; }
  for (int s = t; s < P.C.nseg; s += nt) { SpecSeg& S = P.W.segs[s]; S.exact = s == 0; S.dirty = 1; S.done = 0; S.draws = 0; S.nnotes = 0; S.nreads = 0; S.mispos = -1; S.warmMul = 1; S.nslow = 0; S.chain = 1; S.chained = 0; }
  if (t < 16) P.W.state[t] = 0;
}
#if defined(NQS_EMULATE)
__global__ void k_spec_pre(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!P.eligible) return;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) stage_pre(P.C, P.W, n);
}
#else
// the palette, the three cost tables, the gamma table and the blue-noise mask of the image in shared memory: stage 1 reads
// each of them several times per pixel
__global__ void __launch_bounds__(256) k_spec_pre(SpecImage* sp, const int* list) {
  __shared__ uint32_t sPal[NQ_MAXK];
  __shared__ double sT[3][256], sLut[256];
  __shared__ signed char sBn[4096];
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!P.eligible) return;
  for (int k = threadIdx.x; k < 256; k += blockDim.x) {
    sPal[k] = k < P.C.plen ? P.C.pal[k] : 0u;
    sT[0][k] = P.C.Tr[k]; sT[1][k] = P.C.Tg[k]; sT[2][k] = P.C.Tb[k];
    sLut[k] = P.W.lut[k];
  }
  for (int k = threadIdx.x; k < 4096; k += blockDim.x) sBn[k] = P.W.bn[k];
  __syncthreads();
  SpecWork W = P.W;
  W.lut = sLut; W.bn = sBn;
  ScanTabs T;
  T.pal = sPal; T.Tr = sT[0]; T.Tg = sT[1]; T.Tb = sT[2]; T.plen = P.C.plen;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) stage_pre(P.C, T, W, n);
}
#endif
// stage 2: exclusive prefix sum of the predicted draws in three steps: draws per NQS_CHUNK pixels (a), prefix of those per
// image (b), cdraw of every pixel (c). redo != 0: only images that asked for a re-resolve (state[5]).
#define NQS_SCAN_SKIP(P, redo) (!(P).eligible || ((redo) && (!(P).W.state[5] || (P).W.state[1])))
#if defined(NQS_EMULATE)
__global__ void k_spec_scan_a(SpecImage*, const int*, int) {}
__global__ void k_spec_scan_b(SpecImage*, const int*, int) {}
__global__ void k_spec_scan_c(SpecImage* sp, const int* list, int redo) {     // the block scan needs real warps: sequential stand-in
  const SpecImage& P = sp[list[blockIdx.y]];
  if (threadIdx.x || blockIdx.x || NQS_SCAN_SKIP(P, redo)) return;
  unsigned d = 0;
  for (int n = 0; n < P.C.npix; ++n) { P.W.cdraw[n] = d; d += (P.W.cflag[n] & NQS_F_DRAW) ? 1u : 0u; }
  P.W.cdraw[P.C.npix] = d;
}
#else
__global__ void __launch_bounds__(256) k_spec_scan_a(SpecImage* sp, const int* list, int redo) {
  __shared__ int sWarp[8];
  const SpecImage& P = sp[list[blockIdx.y]];
  if (NQS_SCAN_SKIP(P, redo)) return;
  const int npix = P.C.npix, nchunk = (npix + NQS_CHUNK - 1) / NQS_CHUNK;
  for (int c = blockIdx.x; c < nchunk; c += gridDim.x) {
    const int n0 = c * NQS_CHUNK, n1 = min(npix, n0 + NQS_CHUNK);
    int cnt = 0;
    for (int n = n0 + 4 * (int)threadIdx.x; n < n1; n += 1024) {
      if (n + 4 <= n1) {                                      // cflag + n0 is 4-byte aligned: NQS_CHUNK and the array base are
        const unsigned v = *reinterpret_cast<const unsigned*>(P.W.cflag + n) & (0x01010101u * NQS_F_DRAW);
        cnt += __popc(v);
      } else
        for (int k = n; k < n1; ++k) cnt += (P.W.cflag[k] & NQS_F_DRAW) ? 1 : 0;
    }
    cnt = __reduce_add_sync(0xffffffffu, cnt);
    if ((threadIdx.x & 31) == 0) sWarp[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) { int t = 0; for (int k = 0; k < 8; ++k) t += sWarp[k]; P.W.chunkSum[c] = (unsigned)t; }
    __syncthreads();
  }
}
__global__ void __launch_bounds__(1024) k_spec_scan_b(SpecImage* sp, const int* list, int redo) {
  __shared__ int sWarp[33];
  const SpecImage& P = sp[list[blockIdx.x]];
  if (NQS_SCAN_SKIP(P, redo)) return;
  const int npix = P.C.npix, nchunk = (npix + NQS_CHUNK - 1) / NQS_CHUNK;
  unsigned carry = 0;
  for (int base = 0; base < nchunk; base += 1024) {
    const int c = base + (int)threadIdx.x;
    const int v = c < nchunk ? (int)P.W.chunkSum[c] : 0;
    int total;
    const int excl = block_excl_scan_1024(v, &total, sWarp);
    if (c < nchunk) P.W.chunkSum[c] = carry + (unsigned)excl;
    carry += (unsigned)total;
  }
  if (threadIdx.x == 0) P.W.cdraw[npix] = carry;
}
__global__ void __launch_bounds__(256) k_spec_scan_c(SpecImage* sp, const int* list, int redo) {
  __shared__ int sWarp[8];
  const SpecImage& P = sp[list[blockIdx.y]];
  if (NQS_SCAN_SKIP(P, redo)) return;
  const int npix = P.C.npix, nchunk = (npix + NQS_CHUNK - 1) / NQS_CHUNK;
  const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int c = blockIdx.x; c < nchunk; c += gridDim.x) {
    const int n0 = c * NQS_CHUNK + (int)threadIdx.x * 32;     // 32 consecutive pixels per thread
    unsigned bits = 0;
    if (n0 + 32 <= npix) {
      const uint4* f = reinterpret_cast<const uint4*>(P.W.cflag + n0);
      const uint4 a = f[0], b = f[1];
      const unsigned wds[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
      for (int q = 0; q < 8; ++q)
#pragma unroll
        for (int j = 0; j < 4; ++j) bits |= ((wds[q] >> (8 * j)) & NQS_F_DRAW ? 1u : 0u) << (4 * q + j);
    } else
      for (int k = 0; k < 32; ++k) if (n0 + k < npix && (P.W.cflag[n0 + k] & NQS_F_DRAW)) bits |= 1u << k;
    const int mine = __popc(bits);
    int x = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= (unsigned)o) x += y; }
    if (lane == 31) sWarp[w] = x;
    __syncthreads();
    unsigned d = P.W.chunkSum[c] + (unsigned)(x - mine);
    for (unsigned k = 0; k < w; ++k) d += (unsigned)sWarp[k];
    if (n0 + 32 <= npix) {
      uint4* o = reinterpret_cast<uint4*>(P.W.cdraw + n0);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        uint4 v;
        v.x = d; d += (bits >> (4 * q)) & 1u;
        v.y = d; d += (bits >> (4 * q + 1)) & 1u;
        v.z = d; d += (bits >> (4 * q + 2)) & 1u;
        v.w = d; d += (bits >> (4 * q + 3)) & 1u;
        o[q] = v;
      }
    } else
      for (int k = 0; k < 32; ++k) if (n0 + k < npix) { P.W.cdraw[n0 + k] = d; d += (bits >> k) & 1u; }
    __syncthreads();
  }
}
#endif
#if defined(NQS_EMULATE)
__global__ void k_spec_resolve(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!P.eligible) return;
  int risk = 0, slow = 0;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) {
    int key;
    risk += (P.W.cflag[n] & NQS_F_RISK) ? 1 : 0;
    slow += (P.W.cflag[n] & NQS_F_PRE) ? 0 : 1;
    if (!stage_resolve(P.C, P.W, n, &key)) { P.W.state[1] = 1; P.W.state[11] = 7; }
    if (key >= 0) atomicMin(&P.W.firstPos[key], n);
  }
  if (risk) atomicAdd(&P.W.state[7], risk);
  if (slow) atomicAdd(&P.W.state[8], slow);
}
#else
// Stage 3 with the generator state carried along: every warp owns spans of NQS_RSPAN consecutive pixels, jumps to the state
// of the span's first draw once (O(log n)) and from there reaches the draw of each pixel with ONE multiply-add
// (state after k more steps = A^k state + C_k, k <= 48 from a shared table).
#define NQS_RSPAN 2048
__global__ void __launch_bounds__(256) k_spec_resolve(SpecImage* sp, const int* list) {
  __shared__ unsigned long long sA[64], sC[64];
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!P.eligible) return;
  const unsigned long long MASK = (1ULL << 48) - 1;
  if (threadIdx.x == 0) {
    unsigned long long a = 1ULL, c = 0ULL;
    for (int k = 0; k < 64; ++k) { sA[k] = a; sC[k] = c; a = (a * 0x5DEECE66DULL) & MASK; c = (c * 0x5DEECE66DULL + 0xBULL) & MASK; }
  }
  __syncthreads();
  const unsigned lane = threadIdx.x & 31;
  const int warpsPerGrid = (int)(gridDim.x * (blockDim.x >> 5)), warp = (int)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));
  const int npix = P.C.npix, nspan = (npix + NQS_RSPAN - 1) / NQS_RSPAN;
  int risk = 0, slow = 0;
  for (int sp_ = warp; sp_ < nspan; sp_ += warpsPerGrid) {
    const int n0 = sp_ * NQS_RSPAN, n1 = min(npix, n0 + NQS_RSPAN);
    unsigned long long curStep = lcg_step_of(P.C, (unsigned long long)P.W.cdraw[n0]);        // generator steps behind the draws in front of the span
    unsigned long long curState = lcg_jump(P.C.jmpA, P.C.jmpC, P.C.seed0, curStep);
    for (int base = n0; base < n1; base += 32) {
      const int n = base + (int)lane;
      const int nn = min(base + 32, npix);                                                    // cdraw has npix + 1 entries
      const unsigned long long nextStep = lcg_step_of(P.C, (unsigned long long)P.W.cdraw[nn]);
      if (n < n1) {
        const unsigned flag = P.W.cflag[n];
        risk += (flag & NQS_F_RISK) ? 1 : 0;
        slow += (flag & NQS_F_PRE) ? 0 : 1;
        unsigned long long st = 0ULL;
        const unsigned long long* stp = nullptr;
        if ((flag & NQS_F_PRE) && (flag & NQS_F_DRAW)) {
          const unsigned long long k = lcg_step_of(P.C, (unsigned long long)P.W.cdraw[n] + 1ULL) - curStep;
          if (k < 64ULL) { st = (sA[k] * curState + sC[k]) & MASK; stp = &st; }              // (else: the jump inside stage_resolve)
        }
        int key;
        if (!stage_resolve(P.C, P.W, n, &key, stp)) { P.W.state[1] = 1; P.W.state[11] = 7; }
        if (key >= 0) atomicMin(&P.W.firstPos[key], n);
      }
      const unsigned long long k2 = nextStep - curStep;
      curState = k2 < 64ULL ? (sA[k2] * curState + sC[k2]) & MASK : lcg_jump(P.C.jmpA, P.C.jmpC, P.C.seed0, nextStep);
      curStep = nextStep;
    }
  }
  risk = __reduce_add_sync(0xffffffffu, risk);
  slow = __reduce_add_sync(0xffffffffu, slow);
  if (lane == 0 && risk) atomicAdd(&P.W.state[7], risk);
  if (lane == 0 && slow) atomicAdd(&P.W.state[8], slow);
}
#endif
// re-resolve behind a draw misprediction (images with state[5] != 0): adopt = observed draws become the prediction (before the
// prefix sum), a = reset keys, b = stages 3, c = stage 4, d = stage 5
__global__ void __launch_bounds__(256) k_spec_adopt(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P) || !P.W.state[5]) return;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) stage_adopt(P.W, n);
}
__global__ void __launch_bounds__(256) k_spec_redo_a(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P) || !P.W.state[5]) return;
  const int from = P.W.state[5] - 1;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < 65536; k += gridDim.x * blockDim.x) stage_rekey(P.W, k, from);
}
__global__ void __launch_bounds__(256) k_spec_redo_b(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P) || !P.W.state[5]) return;
  const int from = P.W.state[5] - 1;
  for (int n = from + 1 + blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) {
    int key;
    if (!stage_resolve(P.C, P.W, n, &key)) { P.W.state[1] = 1; P.W.state[11] = 7; }
    if (key >= 0) atomicMin(&P.W.firstPos[key], n);
  }
}
__global__ void __launch_bounds__(256) k_spec_redo_c(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P) || !P.W.state[5]) return;
  const int from = P.W.state[5] - 1;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < 65536; k += gridDim.x * blockDim.x) stage_memo(P.C, P.W, k, from);
}
// d = stage 5 + 5b behind the misprediction (the records in front of it are unchanged)
__global__ void __launch_bounds__(256) k_spec_redo_d(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P) || !P.W.state[5]) return;
  const int from = P.W.state[5] - 1;
  for (int n = from + blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) { if (n > from) stage_fill(P.C, P.W, n); stage_pack(P.C, P.W, n); }
}
__global__ void __launch_bounds__(256) k_spec_memo(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P)) return;
  if (blockIdx.x == 0 && threadIdx.x == 0) stage_gate(P.C, P.W);   // seen by every later launch (NQS_ACTIVE)
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < 65536; k += gridDim.x * blockDim.x) stage_memo(P.C, P.W, k, -1);
}
#if defined(NQS_EMULATE)
__global__ void k_spec_fill(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P)) return;
  for (int n = blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) { stage_fill(P.C, P.W, n); stage_pack(P.C, P.W, n); }   // stages 5 and 5b
}
#else
// Stages 5 and 5b. The packed records are stored segment-interleaved (record of curve position n at (n % seg) * nseg + n / seg),
// i.e. TRANSPOSED against the curve order the work arrays are in: a tile of 32 segments x 32 offsets goes through shared
// memory so that both the reads (32 consecutive curve positions) and the writes (32 consecutive records) are coalesced.
__device__ __forceinline__ SpecRec make_rec(const SpecConst& C, const SpecWork& W, int n) {
  const uint32_t xy = W.order[n];
  const int bidx = (int)(xy & 0xFFFF) + (int)(xy >> 16) * C.width;
  SpecRec r;
  r.px = W.cpx[n];
  r.xy = xy;
  r.qf = (uint32_t)W.cq[n] | ((uint32_t)W.cflag[n] << 16) | (W.bn[bidx & 4095] > C.thresold ? 1u << 24 : 0u);
  r.sal = (W.cflag[n] & NQS_F_PRE) ? 0.f : saliency_of(C, W, r.px);
  return r;
}
__global__ void __launch_bounds__(256) k_spec_fill(SpecImage* sp, const int* list) {
  __shared__ uint4 tile[32][33];
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P)) return;
  const int seg = P.C.seg, nseg = P.C.nseg, npix = P.C.npix;
  const int tilesR = (seg + 31) >> 5, tilesC = (nseg + 31) >> 5;
  const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint4* const recs = reinterpret_cast<uint4*>(P.W.rec);
  for (int t = blockIdx.x; t < tilesR * tilesC; t += gridDim.x) {
    const int r0 = (t % tilesR) << 5, c0 = (t / tilesR) << 5;
    for (int k = (int)w; k < 32; k += 8) {                 // segment c0 + k, offsets r0 .. r0 + 31: consecutive curve positions
      const int c = c0 + k, r = r0 + (int)lane;
      const long long n = (long long)c * seg + r;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (c < nseg && r < seg && n < npix) {
        stage_fill(P.C, P.W, (int)n);
        const SpecRec rec = make_rec(P.C, P.W, (int)n);
        v = make_uint4(rec.px, rec.xy, rec.qf, __float_as_uint(rec.sal));
      }
      tile[k][lane] = v;
    }
    __syncthreads();
    for (int j = (int)w; j < 32; j += 8) {                 // offset r0 + j, segments c0 .. c0 + 31: consecutive records
      const int r = r0 + j, c = c0 + (int)lane;
      if (r < seg && c < nseg && (long long)c * seg + r < npix) recs[(size_t)r * (size_t)nseg + (size_t)c] = tile[lane][j];
    }
    __syncthreads();
  }
}
#endif
// stage 5b alone for the images with a pending patch (a patch may touch any pixel behind its position)
__global__ void __launch_bounds__(256) k_spec_pack(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P) || !P.W.state[2]) return;
  const int from = P.W.state[3];
  for (int n = from + blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) stage_pack(P.C, P.W, n);
}
// stage 6: one thread per segment; one instantiation per (DITHER_MAX, opaque or not), each with its own list of images
#define NQS_RUN_THREADS 128
#define NQS_VARIANTS 6
#if defined(NQS_EMULATE)
template <int DM, int DMI, int NCH>
__global__ void k_spec_run(SpecImage* sp, const int* list, const float* tanhTab) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P)) return;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < P.C.nseg) stage_run_t<DM, DMI, NCH>(P.C, P.W, s, scan_tabs(P.C), tanhTab);
}
#else
template <int DM, int DMI, int NCH>
__global__ void __launch_bounds__(NQS_RUN_THREADS, (DM + NQS_U) * NCH <= 96 ? 3 : 2) k_spec_run(SpecImage* sp, const int* list, const float* tanhTab) {
  __shared__ uint32_t sPal[NQ_MAXK];
  __shared__ float sTanh[512];
  __shared__ double sT[3][256];
  __shared__ WarpRing sRing[NQS_RUN_THREADS / 32];
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P)) return;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  // nothing to do for a whole block is the common case in the later rounds: look before loading the tables
  const bool work = s < P.C.nseg && !P.W.segs[s].done && P.W.segs[s].dirty;
  if (!__syncthreads_or(work)) return;
  const bool bulk = g_specBulk != 0;
  if (bulk && (threadIdx.x & 31) == 0) {
    mbar_init(&sRing[threadIdx.x >> 5].bar[0], 1u);
    mbar_init(&sRing[threadIdx.x >> 5].bar[1], 1u);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  for (int k = threadIdx.x; k < NQ_MAXK; k += blockDim.x) {
    sPal[k] = k < P.C.plen ? P.C.pal[k] : 0u;
    sT[0][k] = P.C.Tr[k]; sT[1][k] = P.C.Tg[k]; sT[2][k] = P.C.Tb[k];
  }
  for (int k = threadIdx.x; k < 511; k += blockDim.x) sTanh[k] = tanhTab[k];
  __syncthreads();
  ScanTabs T;
  T.pal = sPal; T.Tr = sT[0]; T.Tg = sT[1]; T.Tb = sT[2]; T.plen = P.C.plen;
  if (work) stage_run_t<DM, DMI, NCH>(P.C, P.W, s, T, sTanh, bulk ? &sRing[threadIdx.x >> 5] : nullptr);
}
#endif
template <class Backend>
void spec_launch_run(Backend& be, int variant, dim3 grid, SpecImage* sp, const int* list, const float* tanhTab) {
  switch (variant) {
    case 0: be.launch_run(k_spec_run<9, 0, 3>, grid, NQS_RUN_THREADS, sp, list, tanhTab); break;
    case 1: be.launch_run(k_spec_run<9, 0, 4>, grid, NQS_RUN_THREADS, sp, list, tanhTab); break;
    case 2: be.launch_run(k_spec_run<16, 1, 3>, grid, NQS_RUN_THREADS, sp, list, tanhTab); break;
    case 3: be.launch_run(k_spec_run<16, 1, 4>, grid, NQS_RUN_THREADS, sp, list, tanhTab); break;
    case 4: be.launch_run(k_spec_run<25, 2, 3>, grid, NQS_RUN_THREADS, sp, list, tanhTab); break;
    default: be.launch_run(k_spec_run<25, 2, 4>, grid, NQS_RUN_THREADS, sp, list, tanhTab); break;
  }
}
__global__ void __launch_bounds__(64) k_spec_compare(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P)) return;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < P.C.nseg) stage_compare(P.C, P.W, s);
}
// stage 7: one thread per listed image. status[k]: bit 0 = segments still open, 1 = patch requested, 2 = re-resolve
// requested, 3 = left to the serial kernel
__global__ void k_spec_validate(SpecImage* sp, const int* list, int cnt, int* status) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= cnt) return;
  SpecImage& P = sp[list[k]];
  int st = 0;
  if (P.eligible && !P.W.state[1]) {
    P.W.state[2] = 0;
    P.W.state[5] = 0;
    ++P.rounds;
    const int open = stage_validate(P.C, P.W);
    if (open > 0) st |= 1;
    if (P.W.state[2]) st |= 2;
    if (P.W.state[5]) st |= 4;
  }
  if (!P.eligible || P.W.state[1]) st = 8;
  status[k] = st;
}
__global__ void __launch_bounds__(256) k_spec_patch(SpecImage* sp, const int* list) {
  const SpecImage& P = sp[list[blockIdx.y]];
  if (!NQS_ACTIVE(P) || !P.W.state[2]) return;
  const int from = P.W.state[3];
  for (int n = from + 1 + blockIdx.x * blockDim.x + threadIdx.x; n < P.C.npix; n += gridDim.x * blockDim.x) stage_patch(P.C, P.W, n);
}
// images that leave the pool: completed ones are marked specDone = 1 (k_dither_fifo skips them), the others 3 (handed back)
__global__ void k_spec_finish(NqImage* imgs, SpecImage* sp, const int* list, int cnt) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= cnt) return;
  const int i = list[k];
  const SpecImage& P = sp[i];
  if (NQS_ACTIVE(P) && P.W.state[0] == P.C.nseg) {
    imgs[i].specDone = 1;
    imgs[i].rngDraws = P.W.cdraw[P.C.npix];
  } else {
    imgs[i].specDone = 3;
    // why (nq_get_spec_stats' fallbacks; NQ_SPEC_TIMING prints it): 1 risk gate, 2 too many error-dependent lookups, 3 draw guard,
    // 4 a sequential run overflowed its notes, 5 too many failed validations, 6 too many re-resolves, 7 a nextInt drew twice, 8 round cap
    imgs[i].pad1 = P.eligible ? (P.W.state[11] ? P.W.state[11] : 8) : 0;
  }
}

// ---- host side: layout of one slot of the pool, and the admission / round loop -------------------------------------
struct SpecLayout {
  size_t cpx, ccol, ck0, ck1, cdraw, cq, cflag, firstPos, slowPos, memo, slowVal, segs, state, rec, chunkSum, patch, perSlot;
  int nseg;
};
inline SpecLayout spec_layout(int npix, int seg) {
  SpecLayout L;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t r = o; o = (o + bytes + 255) / 256 * 256; return r; };
  L.nseg = (npix + seg - 1) / seg;
  L.cpx = take((size_t)npix * 4); L.ccol = take((size_t)npix * 4); L.ck0 = take((size_t)npix * 4); L.ck1 = take((size_t)npix * 4);
  L.cdraw = take(((size_t)npix + 1) * 4); L.cq = take((size_t)npix * 2); L.cflag = take((size_t)npix + 64);
  L.firstPos = take(65536 * 4); L.slowPos = take(65536 * 4); L.memo = take(65536 * 2); L.slowVal = take(65536 * 2);
  L.segs = take(sizeof(SpecSeg) * (size_t)L.nseg); L.state = take(64); L.rec = take(sizeof(SpecRec) * (size_t)L.nseg * (size_t)seg);
  L.chunkSum = take(((size_t)npix / NQS_CHUNK + 2) * 4);
  L.patch = take(sizeof(int) * 2 * NQS_MAXPATCH);
  L.perSlot = o;
  return L;
}
// array pointers of slot k of `buf` (host copy of the pool table that k_spec_admit reads)
inline void spec_bind_pool(SpecWork* pool, int nslots, unsigned char* buf, const SpecLayout& L) {
  for (int k = 0; k < nslots; ++k) {
    unsigned char* b = buf + L.perSlot * (size_t)k;
    SpecWork& W = pool[k];
    memset(&W, 0, sizeof(W));
    W.cpx = reinterpret_cast<uint32_t*>(b + L.cpx); W.ccol = reinterpret_cast<uint32_t*>(b + L.ccol);
    W.ck0 = reinterpret_cast<uint32_t*>(b + L.ck0); W.ck1 = reinterpret_cast<uint32_t*>(b + L.ck1);
    W.cdraw = reinterpret_cast<uint32_t*>(b + L.cdraw); W.cq = reinterpret_cast<unsigned short*>(b + L.cq); W.cflag = b + L.cflag;
    W.firstPos = reinterpret_cast<int*>(b + L.firstPos); W.slowPos = reinterpret_cast<int*>(b + L.slowPos);
    W.memo = reinterpret_cast<unsigned short*>(b + L.memo); W.slowVal = reinterpret_cast<unsigned short*>(b + L.slowVal);
    W.segs = reinterpret_cast<SpecSeg*>(b + L.segs); W.state = reinterpret_cast<int*>(b + L.state); W.rec = reinterpret_cast<SpecRec*>(b + L.rec);
    W.chunkSum = reinterpret_cast<unsigned*>(b + L.chunkSum);
    W.patch = reinterpret_cast<int*>(b + L.patch);
  }
}
struct SpecStats { unsigned long long done = 0, rounds = 0, handedBack = 0, patches = 0, redos = 0; };
// The admission / round loop. `be` launches kernels and moves a few ints: launch(kernel, grid, block, args...),
// write_ints(dev, host, n), read_ints(host, dev, n) (synchronises), lap(name), note(round, ...). Device scratch dInts:
// 4 lists of `nslots` ints (fresh images, their slots, active images, status). elig: host copy of k_spec_setup's verdicts.
// handedBack (optional): the images this path took and could not finish, for the serial kernel.
template <class Backend>
void spec_drive(Backend& be, NqImage* dImgs, SpecImage* dSpec, const SpecWork* dPool, const int* elig, int n, int npix, int seg, int nslots,
                int* dInts, const float* dTanh, int smCount, SpecStats* st, int* handedBack = nullptr) {
  const int nseg = (npix + seg - 1) / seg;
  const int roundCap = nseg / 4 + 96;
  int* dFresh = dInts; int* dFreshSlot = dInts + nslots; int* dActive = dInts + 2 * nslots; int* dStatus = dInts + 3 * nslots;
  // host mirrors
  int* active = new int[nslots]; int* slotOfActive = new int[nslots]; int* fresh = new int[nslots]; int* freshSlot = new int[nslots];
  int* status = new int[nslots]; int* freeSlots = new int[nslots]; int* rounds = new int[nslots]; int* leaving = new int[nslots];
  int nActive = 0, nFree = nslots, next = 0, nHanded = 0, prefix = 0;
  unsigned char* finished = new unsigned char[n];   // images this path will not touch again (not its own, completed, handed back)
  for (int i = 0; i < n; ++i) finished[i] = (elig[i] & 255) == 1 ? 0 : 2;
  for (int k = 0; k < nslots; ++k) freeSlots[k] = nslots - 1 - k;
  const int nchunk = (npix + NQS_CHUNK - 1) / NQS_CHUNK;
  auto pgrid = [&](int m) {
    int gx = (npix + 256 * 8 - 1) / (256 * 8);
    const int cap = (smCount * 8) / m > 1 ? (smCount * 8) / m : 1;
    return dim3((unsigned)(gx > cap ? cap : gx), (unsigned)m);
  };
  auto cgrid = [&](int m) {
    const int cap = (smCount * 16) / m > 1 ? (smCount * 16) / m : 1;
    return dim3((unsigned)(nchunk > cap ? cap : nchunk), (unsigned)m);
  };
  for (int round = 0;; ++round) {
    // ---- admit images into the free slots: stages 1-5 for them
    int nFresh = 0;
    while (nFree > 0 && next < n) {
      const int i = next++;
      if ((elig[i] & 255) != 1) continue;
      const int slot = freeSlots[--nFree];
      fresh[nFresh] = i; freshSlot[nFresh] = slot; ++nFresh;
      active[nActive] = i; slotOfActive[nActive] = slot; rounds[nActive] = 0; ++nActive;
    }
    if (nFresh) {
      be.write_ints(dFresh, fresh, nFresh); be.write_ints(dFreshSlot, freshSlot, nFresh);
      const dim3 pg = pgrid(nFresh), kg(8, (unsigned)nFresh), cg = cgrid(nFresh);
      be.launch(k_spec_admit, dim3((unsigned)((nFresh + 63) / 64)), 64, dSpec, (const int*)dFresh, (const int*)dFreshSlot, nFresh, dPool);
      be.launch(k_spec_init, kg, 256, dSpec, (const int*)dFresh);
      be.launch(k_spec_rejects, cg, 256, dSpec, (const int*)dFresh);
      be.launch(k_spec_rejsort, dim3((unsigned)((nFresh + 63) / 64)), 64, dSpec, (const int*)dFresh, nFresh); be.lap("init");
      be.launch(k_spec_pre, pg, 256, dSpec, (const int*)dFresh); be.lap("pre");
      be.launch(k_spec_scan_a, cg, 256, dSpec, (const int*)dFresh, 0);
      be.launch(k_spec_scan_b, dim3((unsigned)nFresh), 1024, dSpec, (const int*)dFresh, 0);
      be.launch(k_spec_scan_c, cg, 256, dSpec, (const int*)dFresh, 0); be.lap("scan");
      be.launch(k_spec_resolve, pg, 256, dSpec, (const int*)dFresh); be.lap("resolve");
      be.launch(k_spec_memo, kg, 256, dSpec, (const int*)dFresh); be.lap("memo");
      be.launch(k_spec_fill, dim3((unsigned)((smCount * 16) / nFresh > 1 ? (smCount * 16) / nFresh : 1), (unsigned)nFresh), 256, dSpec, (const int*)dFresh); be.lap("fill+pack");
    }
    if (!nActive) break;
    // ---- one round for everything in the pool: stages 6, 6b, 7. The list is kept grouped by stage-6 instantiation.
    {
      int at = 0;
      for (int v = 0; v < NQS_VARIANTS; ++v)
        for (int k = at; k < nActive; ++k)
          if (((elig[active[k]] >> 8) & 7) == v) {
            const int a = active[k], b = slotOfActive[k], r = rounds[k];
            active[k] = active[at]; slotOfActive[k] = slotOfActive[at]; rounds[k] = rounds[at];
            active[at] = a; slotOfActive[at] = b; rounds[at] = r; ++at;
          }
    }
    be.write_ints(dActive, active, nActive);
    const dim3 s64((unsigned)((nseg + 63) / 64), (unsigned)nActive);
    for (int k0 = 0; k0 < nActive;) {
      const int v = (elig[active[k0]] >> 8) & 7;
      int k1 = k0;
      while (k1 < nActive && ((elig[active[k1]] >> 8) & 7) == v) ++k1;
      spec_launch_run(be, v, dim3((unsigned)((nseg + NQS_RUN_THREADS - 1) / NQS_RUN_THREADS), (unsigned)(k1 - k0)), dSpec, (const int*)dActive + k0, dTanh);
      k0 = k1;
    }
    be.lap("run");
    be.launch(k_spec_compare, s64, 64, dSpec, (const int*)dActive); be.lap("compare");
    be.launch(k_spec_validate, dim3((unsigned)((nActive + 63) / 64)), 64, dSpec, (const int*)dActive, nActive, dStatus); be.lap("validate");
    be.read_ints(status, dStatus, nActive);
    ++st->rounds;
    int nOpen = 0, nPatch = 0, nRedo = 0, nLeave = 0;
    for (int k = 0; k < nActive; ++k) {
      ++rounds[k];
      if ((status[k] & 1) && rounds[k] >= roundCap) status[k] = 8;      // not converging: the serial kernel takes it
      nOpen += (status[k] & 1) && !(status[k] & 8); nPatch += (status[k] & 2) != 0; nRedo += (status[k] & 4) != 0;
    }
    st->patches += (unsigned long long)nPatch; st->redos += (unsigned long long)nRedo;
    be.note(round, nActive, nOpen, nPatch, nRedo);
    const dim3 pa = pgrid(nActive), ka(8, (unsigned)nActive), ca = cgrid(nActive);
    if (nPatch) { be.launch(k_spec_patch, pa, 256, dSpec, (const int*)dActive); be.launch(k_spec_pack, pa, 256, dSpec, (const int*)dActive); be.lap("patch"); }
    if (nRedo) {   // a draw misprediction: prefix sum again, then stages 3-5 behind it, for the images that asked
      be.launch(k_spec_adopt, pa, 256, dSpec, (const int*)dActive);
      be.launch(k_spec_scan_a, ca, 256, dSpec, (const int*)dActive, 1);
      be.launch(k_spec_scan_b, dim3((unsigned)nActive), 1024, dSpec, (const int*)dActive, 1);
      be.launch(k_spec_scan_c, ca, 256, dSpec, (const int*)dActive, 1);
      be.launch(k_spec_redo_a, ka, 256, dSpec, (const int*)dActive);
      be.launch(k_spec_redo_b, pa, 256, dSpec, (const int*)dActive);
      be.launch(k_spec_redo_c, ka, 256, dSpec, (const int*)dActive);
      be.launch(k_spec_redo_d, pa, 256, dSpec, (const int*)dActive); be.lap("re-resolve");
    }
    // ---- images that leave: completed (no segment open) or handed back; their slots are free for the next round
    int keep = 0;
    for (int k = 0; k < nActive; ++k) {
      const bool leave = (status[k] & 8) || !(status[k] & 1);
      if (leave) {
        leaving[nLeave++] = active[k];
        freeSlots[nFree++] = slotOfActive[k];
        if (status[k] & 8) { ++st->handedBack; if (handedBack) handedBack[nHanded] = active[k]; ++nHanded; finished[active[k]] = 2; }
        else { ++st->done; finished[active[k]] = 1; }
      } else { active[keep] = active[k]; slotOfActive[keep] = slotOfActive[k]; rounds[keep] = rounds[k]; ++keep; }
    }
    nActive = keep;
    if (nLeave) {
      be.write_ints(dFresh, leaving, nLeave);               // (dFresh is free again: stream order)
      be.launch(k_spec_finish, dim3((unsigned)((nLeave + 63) / 64)), 64, dImgs, dSpec, (const int*)dFresh, nLeave);
      // the leading run of images that are COMPLETE (a caller with host buffers starts copying them out while the rest is
      // still in the pool); it stops at the first image another kernel has to dither
      int p = prefix;
      while (p < n && finished[p] == 1) ++p;
      if (p > prefix) { prefix = p; be.done_prefix(prefix); }
    }
  }
  delete[] finished;
  delete[] active; delete[] slotOfActive; delete[] fresh; delete[] freshSlot; delete[] status; delete[] freeSlots; delete[] rounds; delete[] leaving;
}
#endif  // __CUDACC__ || NQS_EMULATE

}  // namespace spec
}  // namespace nq
