// nq_oracle.cpp -- TEST INFRASTRUCTURE ONLY. Single-threaded CPU restatement of the nQuant.android
// quantizer core, used as the parity checker for the CUDA path and as the reported CPU baseline.
// Nothing in the product (nquant_android_b200/) links or calls this file.
//
// PARITY UNPINNED: the reference ships no tests, golden vectors or fixtures for this path and no JVM
// exists in the build image, so this restatement could not be checked against the reference's own
// outputs. Its fidelity rests on line-by-line review against the cited Java sources plus the
// self-derived known answers in tests/test_oracle.py.
//
// Files followed (prefixes as in SURVEY.md):
//   PQ = nQuant.master/src/main/java/com/android/nQuant/PnnQuantizer.java
//   PL = .../PnnLABQuantizer.java   CL = .../CIELABConvertor.java   GC = .../GilbertCurve.java
//   BN = .../BlueNoise.java         BU = .../BitmapUtilities.java   DI = .../Ditherable.java
// Third-party arithmetic that is NOT under /root/reference and is restated from its published
// algorithm: androidx.core.graphics.ColorUtils {colorToLAB, LABToColor, setAlphaComponent}
// (androidx.core:core, resolved transitively from androidx.appcompat:appcompat:1.4.0-alpha03,
// nQuant.master/build.gradle:36 -- version not pinned by the reference); android.graphics.Color;
// java.util.{HashMap, ArrayDeque, PriorityQueue, Random}; java.lang.Math.
//
// Java numerics: strict IEEE-754, no FMA contraction (build with -ffp-contract=off), Java cast and
// promotion rules written out explicitly. Two math modes: 0 = shared nq_math.h kernels (bit-identical
// to the GPU), 1 = glibc libm (closest to what a JVM would call).
#include <cstdint>
#include <cstring>
#include <cmath>
#include <vector>
#include <deque>
#include <unordered_map>
#include <array>
#include <string>
#include <algorithm>
#include <stdexcept>

// study hook (tools/spec_dither_emul.cpp): sees every nearestMap key that is looked up; nothing by default
#ifndef NQ_ORACLE_PROBE
#define NQ_ORACLE_PROBE(key) ((void)0)
#endif

#include "../nquant_android_b200/csrc/nq_math.h"
#include "../nquant_android_b200/csrc/nq_bluenoise_table.h"

namespace {

// ---------------------------------------------------------------------------------------------
// java.lang.Math and cast rules
// ---------------------------------------------------------------------------------------------
struct JMath {
  int mode = 0;  // 0 shared, 1 libm
  double pow(double x, double y) const { return mode ? ::pow(x, y) : nqm::nq_pow(x, y); }
  double exp(double x) const { return mode ? ::exp(x) : nqm::nq_exp(x); }
  double tanh(double x) const { return mode ? ::tanh(x) : nqm::nq_tanh(x); }
  double cbrt(double x) const { return mode ? ::cbrt(x) : nqm::nq_cbrt(x); }
  double atan2(double y, double x) const { return mode ? ::atan2(y, x) : nqm::nq_atan2(y, x); }
  double sin(double x) const { return mode ? ::sin(x) : nqm::nq_sin(x); }
  double cos(double x) const { return mode ? ::cos(x) : nqm::nq_cos(x); }
  static double sqrt(double x) { return ::sqrt(x); }
};
static thread_local JMath M;

constexpr double JPI = 3.141592653589793;
constexpr double JE = 2.718281828459045;

// (int) of a double / float, JLS 5.1.3
inline int32_t j2i(double v) {
  if (v != v) return 0;
  if (v >= 2147483647.0) return INT32_MAX;
  if (v <= -2147483648.0) return INT32_MIN;
  return (int32_t)v;
}
inline int8_t j2b(double v) { return (int8_t)(uint8_t)(uint32_t)j2i(v); }
// Math.round(double): floor(x + 1/2) evaluated exactly
inline int64_t jround(double v) {
  if (v != v) return 0;
  double f = std::floor(v);
  double d = v - f;
  if (d >= 0.5) f += 1.0;
  if (f >= 9223372036854775807.0) return INT64_MAX;
  if (f <= -9223372036854775808.0) return INT64_MIN;
  return (int64_t)f;
}
inline int32_t iadd(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }

// ---------------------------------------------------------------------------------------------
// android.graphics.Color
// ---------------------------------------------------------------------------------------------
namespace Color {
inline int alpha(int32_t c) { return (int)((uint32_t)c >> 24); }
inline int red(int32_t c) { return (c >> 16) & 0xFF; }
inline int green(int32_t c) { return (c >> 8) & 0xFF; }
inline int blue(int32_t c) { return c & 0xFF; }
inline int32_t argb(int a, int r, int g, int b) {
  return (int32_t)(((uint32_t)a << 24) | ((uint32_t)r << 16) | ((uint32_t)g << 8) | (uint32_t)b);
}
constexpr int32_t BLACK = (int32_t)0xFF000000u;
constexpr int32_t WHITE = (int32_t)0xFFFFFFFFu;
}  // namespace Color

// ---------------------------------------------------------------------------------------------
// BitmapUtilities (BU:6-20)
// ---------------------------------------------------------------------------------------------
constexpr int BYTE_MAX = 255;  // BU:6
inline int getColorIndex(int32_t c, bool hasSemiTransparency, bool hasTransparency) {  // BU:8-15
  if (hasSemiTransparency)
    return (Color::alpha(c) & 0xF0) << 8 | (Color::red(c) & 0xF0) << 4 | (Color::green(c) & 0xF0) | (Color::blue(c) >> 4);
  if (hasTransparency)
    return (Color::alpha(c) & 0x80) << 8 | (Color::red(c) & 0xF8) << 7 | (Color::green(c) & 0xF8) << 2 | (Color::blue(c) >> 3);
  return (Color::red(c) & 0xF8) << 8 | (Color::green(c) & 0xFC) << 3 | (Color::blue(c) >> 3);
}
inline double sqr(double v) { return v * v; }  // BU:17

static const int8_t TELL_BLUE_NOISE[4096] = NQ_BLUE_NOISE_INIT;  // BN:13-178

// ---------------------------------------------------------------------------------------------
// androidx.core.graphics.ColorUtils (restated from the published algorithm; see header)
// ---------------------------------------------------------------------------------------------
namespace ColorUtils {
constexpr double XYZ_WHITE_REFERENCE_X = 95.047, XYZ_WHITE_REFERENCE_Y = 100, XYZ_WHITE_REFERENCE_Z = 108.883;
constexpr double XYZ_EPSILON = 0.008856, XYZ_KAPPA = 903.3;
inline double pivotXyzComponent(double component) {
  return component > XYZ_EPSILON ? M.pow(component, 1 / 3.0) : (XYZ_KAPPA * component + 16) / 116;
}
inline void colorToLAB(int32_t color, double out[3]) {
  double sr = Color::red(color) / 255.0;
  sr = sr < 0.04045 ? sr / 12.92 : M.pow((sr + 0.055) / 1.055, 2.4);
  double sg = Color::green(color) / 255.0;
  sg = sg < 0.04045 ? sg / 12.92 : M.pow((sg + 0.055) / 1.055, 2.4);
  double sb = Color::blue(color) / 255.0;
  sb = sb < 0.04045 ? sb / 12.92 : M.pow((sb + 0.055) / 1.055, 2.4);
  double x = 100 * (sr * 0.4124 + sg * 0.3576 + sb * 0.1805);
  double y = 100 * (sr * 0.2126 + sg * 0.7152 + sb * 0.0722);
  double z = 100 * (sr * 0.0193 + sg * 0.1192 + sb * 0.9505);
  x = pivotXyzComponent(x / XYZ_WHITE_REFERENCE_X);
  y = pivotXyzComponent(y / XYZ_WHITE_REFERENCE_Y);
  z = pivotXyzComponent(z / XYZ_WHITE_REFERENCE_Z);
  out[0] = std::max(0.0, 116 * y - 16);
  out[1] = 500 * (x - y);
  out[2] = 200 * (y - z);
}
inline int constrain(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
inline int32_t LABToColor(double l, double a, double b) {
  const double fy = (l + 16) / 116;
  const double fx = a / 500 + fy;
  const double fz = fy - b / 200;
  double tmp = M.pow(fx, 3);
  const double xr = tmp > XYZ_EPSILON ? tmp : (116 * fx - 16) / XYZ_KAPPA;
  const double yr = l > XYZ_KAPPA * XYZ_EPSILON ? M.pow(fy, 3) : l / XYZ_KAPPA;
  tmp = M.pow(fz, 3);
  const double zr = tmp > XYZ_EPSILON ? tmp : (116 * fz - 16) / XYZ_KAPPA;
  const double x = xr * XYZ_WHITE_REFERENCE_X, y = yr * XYZ_WHITE_REFERENCE_Y, z = zr * XYZ_WHITE_REFERENCE_Z;
  double r = (x * 3.2406 + y * -1.5372 + z * -0.4986) / 100;
  double g = (x * -0.9689 + y * 1.8758 + z * 0.0415) / 100;
  double bb = (x * 0.0557 + y * -0.2040 + z * 1.0570) / 100;
  r = r > 0.0031308 ? 1.055 * M.pow(r, 1 / 2.4) - 0.055 : 12.92 * r;
  g = g > 0.0031308 ? 1.055 * M.pow(g, 1 / 2.4) - 0.055 : 12.92 * g;
  bb = bb > 0.0031308 ? 1.055 * M.pow(bb, 1 / 2.4) - 0.055 : 12.92 * bb;
  int ri = constrain((int)jround(r * 255), 0, 255);
  int gi = constrain((int)jround(g * 255), 0, 255);
  int bi = constrain((int)jround(bb * 255), 0, 255);
  return Color::argb(255, ri, gi, bi);
}
inline int32_t setAlphaComponent(int32_t color, int alpha) {
  if (alpha < 0 || alpha > 255) throw std::invalid_argument("alpha must be between 0 and 255.");
  return (int32_t)(((uint32_t)color & 0x00ffffffu) | ((uint32_t)alpha << 24));
}
}  // namespace ColorUtils

// ---------------------------------------------------------------------------------------------
// CIELABConvertor (CL)
// ---------------------------------------------------------------------------------------------
struct Lab {  // CL:51-56
  float alpha = BYTE_MAX, A = 0.f, B = 0.f, L = 0.f;
};
namespace CIELAB {
inline Lab RGB2LAB(int32_t c1) {  // CL:58-69
  double labs[3];
  ColorUtils::colorToLAB(c1, labs);
  Lab lab;
  lab.alpha = (float)Color::alpha(c1);
  lab.L = (float)labs[0];
  lab.A = (float)labs[1];
  lab.B = (float)labs[2];
  return lab;
}
inline double gammaToLinear(int channel) {  // CL:71-75
  const double c = channel / 255.0;
  return c < 0.04045 ? c / 12.92 : M.pow((c + 0.055) / 1.055, 2.4);
}
inline int32_t LAB2RGB(const Lab& lab) {  // CL:77-80
  int32_t color = ColorUtils::LABToColor(lab.L, lab.A, lab.B);
  return ColorUtils::setAlphaComponent(color, j2i(lab.alpha));
}
inline float deg2Rad(double deg) { return (float)(deg * (JPI / 180.0)); }  // CL:86-89

inline float L_prime_div_k_L_S_L(const Lab& lab1, const Lab& lab2) {  // CL:91-98
  const float k_L = 1.0f;
  float deltaLPrime = lab2.L - lab1.L;
  float barLPrime = (lab1.L + lab2.L) / 2.f;
  float S_L = (float)(1 + ((0.015f * M.pow(barLPrime - 50.f, 2.f)) / JMath::sqrt(20 + M.pow(barLPrime - 50.f, 2.f))));
  return deltaLPrime / (k_L * S_L);
}
inline float C_prime_div_k_L_S_L(const Lab& lab1, const Lab& lab2, double& a1Prime, double& a2Prime, double& CPrime1, double& CPrime2) {  // CL:100-118
  const float k_C = 1.f;
  const float pow25To7 = 6103515625.f;
  float C1 = (float)(JMath::sqrt((double)((lab1.A * lab1.A) + (lab1.B * lab1.B))));
  float C2 = (float)(JMath::sqrt((double)((lab2.A * lab2.A) + (lab2.B * lab2.B))));
  float barC = (C1 + C2) / 2.f;
  float G = (float)(0.5f * (1 - JMath::sqrt(M.pow(barC, 7) / (M.pow(barC, 7) + pow25To7))));
  a1Prime = (1.0 + G) * lab1.A;
  a2Prime = (1.0 + G) * lab2.A;
  CPrime1 = JMath::sqrt((a1Prime * a1Prime) + (double)(lab1.B * lab1.B));
  CPrime2 = JMath::sqrt((a2Prime * a2Prime) + (double)(lab2.B * lab2.B));
  float deltaCPrime = (float)CPrime2 - (float)CPrime1;
  float barCPrime = ((float)CPrime1 + (float)CPrime2) / 2.f;
  float S_C = 1 + (0.045f * barCPrime);
  return deltaCPrime / (k_C * S_C);
}
// BigDecimal.ZERO.equals(new BigDecimal(x)) (CL:127,139,151,164): true only for +-0.0
inline bool isZero(double x) { return x == 0.0; }
inline float H_prime_div_k_L_S_L(const Lab& lab1, const Lab& lab2, double a1Prime, double a2Prime, double CPrime1, double CPrime2, double& barCPrime, double& barhPrime) {  // CL:120-185
  const float k_H = 1.f;
  const float deg360InRad = deg2Rad(360.f);
  const float deg180InRad = deg2Rad(180.f);
  double CPrimeProduct = CPrime1 * CPrime2;
  double hPrime1;
  if (isZero(lab1.B) && isZero(a1Prime)) hPrime1 = 0.0;
  else {
    hPrime1 = M.atan2(lab1.B, a1Prime);
    if (hPrime1 < 0) hPrime1 += deg360InRad;
  }
  double hPrime2;
  if (isZero(lab2.B) && isZero(a2Prime)) hPrime2 = 0.0;
  else {
    hPrime2 = M.atan2(lab2.B, a2Prime);
    if (hPrime2 < 0) hPrime2 += deg360InRad;
  }
  double deltahPrime;
  if (isZero(CPrimeProduct)) deltahPrime = 0;
  else {
    deltahPrime = hPrime2 - hPrime1;
    if (deltahPrime < -deg180InRad) deltahPrime += deg360InRad;
    else if (deltahPrime > deg180InRad) deltahPrime -= deg360InRad;
  }
  double deltaHPrime = 2.0 * JMath::sqrt(CPrimeProduct) * M.sin(deltahPrime / 2.0);
  double hPrimeSum = hPrime1 + hPrime2;
  if (isZero(CPrime1 * CPrime2)) barhPrime = hPrimeSum;
  else {
    if (std::fabs(hPrime1 - hPrime2) <= deg180InRad) barhPrime = hPrimeSum / 2.0;
    else {
      if (hPrimeSum < deg360InRad) barhPrime = (hPrimeSum + deg360InRad) / 2.0;
      else barhPrime = (hPrimeSum - deg360InRad) / 2.0;
    }
  }
  barCPrime = (CPrime1 + CPrime2) / 2.0;
  double T = 1.0 - (0.17 * M.cos(barhPrime - deg2Rad(30.f))) +
             (0.24 * M.cos(2.0 * barhPrime)) +
             (0.32 * M.cos((3.0 * barhPrime) + deg2Rad(6.f))) -
             (0.20 * M.cos((4.0 * barhPrime) - deg2Rad(63.f)));
  double S_H = 1 + (0.015f * barCPrime * T);
  return (float)(deltaHPrime / (k_H * S_H));
}
inline float R_T(double barCPrime, double barhPrime, float C_prime_div_k_L_S_L, float H_prime_div_k_L_S_L) {  // CL:187-194
  const double pow25To7 = 6103515625.0;
  double deltaTheta = deg2Rad(30.f) * M.exp(-M.pow((barhPrime - deg2Rad(275.f)) / deg2Rad(25.f), 2.0));
  double R_C = 2.0 * JMath::sqrt(M.pow(barCPrime, 7.0) / (M.pow(barCPrime, 7.0) + pow25To7));
  double R_T = (-M.sin(2.0 * deltaTheta)) * R_C;
  return (float)(R_T * C_prime_div_k_L_S_L * H_prime_div_k_L_S_L);
}
inline double color2Y(int32_t c) {  // CL:217-222
  double sr = gammaToLinear(Color::red(c));
  double sg = gammaToLinear(Color::green(c));
  double sb = gammaToLinear(Color::blue(c));
  return sr * 0.2126 + sg * 0.7152 + sb * 0.0722;
}
inline double Y_Diff(int32_t c1, int32_t c2) {  // CL:215-227
  double y = color2Y(c1);
  double y2 = color2Y(c2);
  return std::fabs(y2 - y) * 100;
}
inline double color2U(int32_t c) { return -0.09991 * Color::red(c) - 0.33609 * Color::green(c) + 0.436 * Color::blue(c); }  // CL:231-233
inline double U_Diff(int32_t c1, int32_t c2) {  // CL:229-238
  double u = color2U(c1);
  double u2 = color2U(c2);
  return std::fabs(u2 - u);
}
}  // namespace CIELAB

// ---------------------------------------------------------------------------------------------
// java.util.Random (48-bit LCG)
// ---------------------------------------------------------------------------------------------
struct JRandom {
  uint64_t seed;
  explicit JRandom(uint64_t s = 0) { setSeed(s); }
  void setSeed(uint64_t s) { seed = (s ^ 0x5DEECE66DULL) & ((1ULL << 48) - 1); }
  int32_t next(int bits) {
    seed = (seed * 0x5DEECE66DULL + 0xBULL) & ((1ULL << 48) - 1);
    return (int32_t)((int64_t)seed >> (48 - bits));
  }
  int32_t nextInt(int32_t bound) {
    int32_t r = next(31);
    int32_t m = bound - 1;
    if ((bound & m) == 0) r = (int32_t)(((int64_t)bound * (int64_t)r) >> 31);
    else {
      for (int32_t u = r; iadd(u - (r = u % bound), m) < 0; u = next(31)) {}
    }
    return r;
  }
};

// ---------------------------------------------------------------------------------------------
// java.util.HashMap<Integer,?> iteration order (only needed for PL:197)
// ---------------------------------------------------------------------------------------------
std::vector<int32_t> javaHashMapKeyOrder(const std::vector<int32_t>& insertionOrder) {
  struct Node { int32_t key; uint32_t hash; };
  std::vector<std::vector<Node>> table;
  size_t size = 0, threshold = 0;
  auto resize = [&]() {
    if (table.empty()) { table.assign(16, {}); threshold = 12; return; }
    size_t oldCap = table.size(), newCap = oldCap * 2;
    std::vector<std::vector<Node>> nt(newCap);
    for (size_t j = 0; j < oldCap; ++j)
      for (const Node& e : table[j]) nt[(e.hash & oldCap) ? j + oldCap : j].push_back(e);  // lo/hi split keeps order
    table.swap(nt);
    threshold = newCap * 3 / 4;
  };
  for (int32_t k : insertionOrder) {
    uint32_t h = (uint32_t)k;
    h ^= h >> 16;
    if (table.empty()) resize();
    auto& bucket = table[(table.size() - 1) & h];
    bool found = false;
    for (const Node& e : bucket) if (e.key == k) { found = true; break; }
    if (found) continue;
    bucket.push_back(Node{k, h});
    // treeifyBin on a 9th colliding node: with a table < 64 slots Java resizes instead; larger tables
    // would convert to a red-black bin whose iteration order is not emulated here (needs >= 9 colliding
    // keys among <= nMaxColors entries).
    if (bucket.size() >= 9 && table.size() < 64) resize();
    if (++size > threshold) resize();
  }
  std::vector<int32_t> out;
  for (auto& b : table) for (const Node& e : b) out.push_back(e.key);
  return out;
}

// ---------------------------------------------------------------------------------------------
// Ditherable (DI:3-7)
// ---------------------------------------------------------------------------------------------
struct Ditherable {
  virtual ~Ditherable() {}
  virtual int getColorIndex(int32_t c) = 0;
  virtual short nearestColorIndex(const std::vector<int32_t>& palette, int32_t c, int pos) = 0;
};

// ---------------------------------------------------------------------------------------------
// BlueNoise (BN:180-222)
// ---------------------------------------------------------------------------------------------
namespace BlueNoise {
inline int32_t diffuse(int32_t pixel, int32_t qPixel, float weight, float strength, int x, int y) {  // BN:180-197
  int r_pix = Color::red(pixel), g_pix = Color::green(pixel), b_pix = Color::blue(pixel), a_pix = Color::alpha(pixel);
  float adj = (TELL_BLUE_NOISE[(x & 63) | (y & 63) << 6] + 0.5f) / 127.5f;
  adj += (((x + y) & 1) - 0.5f) * strength / 8.f;
  adj *= weight;
  r_pix = j2i(std::min(255.0, std::max((double)(r_pix + (adj * (r_pix - Color::red(qPixel)))), 0.0)));
  g_pix = j2i(std::min(255.0, std::max((double)(g_pix + (adj * (g_pix - Color::green(qPixel)))), 0.0)));
  b_pix = j2i(std::min(255.0, std::max((double)(b_pix + (adj * (b_pix - Color::blue(qPixel)))), 0.0)));
  a_pix = j2i(std::min(255.0, std::max((double)(a_pix + (adj * (a_pix - Color::alpha(qPixel)))), 0.0)));
  return Color::argb(a_pix, r_pix, g_pix, b_pix);
}
inline void dither(int width, int height, const std::vector<int32_t>& pixels, const std::vector<int32_t>& palette, Ditherable& ditherable, std::vector<int32_t>& qPixels, float weight) {  // BN:207-222
  const float strength = 1 / 3.f;
  for (int y = 0; y < height; ++y)
    for (int x = 0; x < width; ++x) {
      const int bidx = x + y * width;
      int32_t pixel = pixels[bidx];
      int32_t qPixel = palette[qPixels[bidx]];
      int32_t c1 = diffuse(pixel, qPixel, weight, strength, x, y);
      qPixels[bidx] = palette[ditherable.nearestColorIndex(palette, c1, bidx)];
    }
}
}  // namespace BlueNoise

// ---------------------------------------------------------------------------------------------
// GilbertCurve (GC)
// ---------------------------------------------------------------------------------------------
struct GilbertParams {  // what the constructor derives (GC:50-112), exported for tests
  int margin, thresold, DITHER_MAX, ditherMax, sortedByYDiff, hasAlpha;
  float beta;
  double weight;
};

class GilbertCurve {
  struct ErrorBox {  // GC:16-32
    double yDiff = 0;
    float p[4] = {0, 0, 0, 0};
    ErrorBox() {}
    explicit ErrorBox(int32_t c) { p[0] = (float)Color::red(c); p[1] = (float)Color::green(c); p[2] = (float)Color::blue(c); p[3] = (float)Color::alpha(c); }
  };
  int8_t ditherMax, DITHER_MAX;
  float beta;
  std::vector<float> weights;
  const bool dither;
  bool hasAlpha, sortedByYDiff;
  const int width, height;
  double weight;
  const std::vector<int32_t>& pixels;
  const std::vector<int32_t>& palette;
  std::vector<int32_t>& qPixels;
  Ditherable& ditherable;
  const std::vector<float>* saliencies;
  // errorq: ArrayDeque (FIFO) or PriorityQueue (binary heap, array-order iteration), GC:87-94
  std::deque<ErrorBox> fifo;
  std::vector<ErrorBox> heap;
  int margin, thresold;
  static constexpr float BLOCK_SIZE = 343.f;

  // java.util.PriorityQueue with comparator Double.compare(o2.yDiff, o1.yDiff)
  static int cmp(const ErrorBox& o1, const ErrorBox& o2) {
    double a = o2.yDiff, b = o1.yDiff;
    return a < b ? -1 : (a > b ? 1 : 0);
  }
  void pqOffer(const ErrorBox& x) {
    size_t k = heap.size();
    heap.push_back(x);
    while (k > 0) {
      size_t parent = (k - 1) >> 1;
      if (cmp(x, heap[parent]) >= 0) break;
      heap[k] = heap[parent];
      k = parent;
    }
    heap[k] = x;
  }
  void pqPoll() {
    size_t n = heap.size() - 1;
    ErrorBox x = heap[n];
    heap.pop_back();
    if (n > 0) {
      size_t k = 0, half = n >> 1;
      while (k < half) {
        size_t child = (k << 1) + 1, right = child + 1;
        if (right < n && cmp(heap[child], heap[right]) > 0) child = right;
        if (cmp(x, heap[child]) <= 0) break;
        heap[k] = heap[child];
        k = child;
      }
      heap[k] = x;
    }
  }
  size_t qSize() const { return sortedByYDiff ? heap.size() : fifo.size(); }
  void qAdd(const ErrorBox& e) { if (sortedByYDiff) pqOffer(e); else fifo.push_back(e); }
  void qPoll() { if (sortedByYDiff) pqPoll(); else fifo.pop_front(); }
  const ErrorBox& qAt(size_t i) const { return sortedByYDiff ? heap[i] : fifo[i]; }

 public:
  GilbertCurve(int width_, int height_, const std::vector<int32_t>& image, const std::vector<int32_t>& palette_, std::vector<int32_t>& qPixels_, Ditherable& ditherable_, const std::vector<float>* saliencies_, double weight_, bool dither_)
      : dither(dither_), width(width_), height(height_), pixels(image), palette(palette_), qPixels(qPixels_), ditherable(ditherable_), saliencies(saliencies_) {  // GC:50-112
    const int plen = (int)palette.size();
    const double weight = weight_;  // the constructor body reads the signed PARAMETER (it shadows the field)
    this->hasAlpha = weight < 0;
    this->weight = std::fabs(weight);
    margin = weight < .0025 ? 12 : weight < .004 ? 8 : 6;
    sortedByYDiff = plen > 128 && weight >= .02 && (!hasAlpha || weight < .18);
    beta = plen > 4 ? (float)(.6f - .00625f * plen) : 1;
    if (plen > 4) {
      double boundary = .005 - .0000625 * plen;
      beta = (float)(weight > boundary ? .25 : std::min(1.5, beta + plen * weight));
      if (plen > 16 && plen <= 32 && weight < .003) beta += .075f;
      else if (weight < .0015 || (plen > 32 && plen < 256)) beta += .1f;
      if ((plen >= 64 && (weight > .012 && weight < .0125)) || (weight > .025 && weight < .03)) beta += .05f;
      else if (plen > 32 && plen < 64 && weight < .015) beta = .55f;
      else if (plen > 16 && plen <= 32 && weight <= .005) beta += (float)(.05 + weight * plen);
    } else
      beta *= .95f;

    if (plen > 64 || (plen > 4 && weight > .02)) beta *= .4f;
    if (plen > 64 && weight < .02) beta = .18f;

    DITHER_MAX = weight < .015 ? ((weight > .0025) ? (int8_t)25 : (int8_t)16) : (int8_t)9;
    if (weight > .99) {
      beta = (float)weight;
      DITHER_MAX = 25;
    }
    double edge = hasAlpha ? 1 : M.exp(weight) - .25;
    double deviation = weight > .002 ? -.25 : 1;
    ditherMax = (hasAlpha || DITHER_MAX > 9) ? j2b(sqr(JMath::sqrt(DITHER_MAX) + edge * deviation)) : j2b(DITHER_MAX * (saliencies != nullptr ? 2 : JE));
    const int density = plen > 16 ? 3200 : 1500;
    if (plen / weight > 5000 && (weight > .045 || (weight > .01 && plen < 64))) ditherMax = j2b(sqr(5 + edge));
    else if (weight < .03 && plen / weight < density && plen >= 16 && plen < 256) ditherMax = j2b(sqr(5 + edge));
    thresold = DITHER_MAX > 9 ? -112 : -64;
    weights.clear();
  }
  GilbertParams params() const { return GilbertParams{margin, thresold, DITHER_MAX, ditherMax, sortedByYDiff, hasAlpha, beta, weight}; }
  const std::vector<float>& getWeights() const { return weights; }

  static float normalDistribution(float x, float peak) {  // GC:114-123
    const float mean = .5f, stdDev = .1f;
    double exponent = -M.pow(x - mean, 2) / (2 * M.pow(stdDev, 2));
    double pdf = (1 / (stdDev * JMath::sqrt(2 * JPI))) * M.exp(exponent);
    double maxPdf = 1 / (stdDev * JMath::sqrt(2 * JPI));
    double scaledPdf = (pdf / maxPdf) * peak;
    return (float)std::max(0.0, std::min((double)peak, scaledPdf));
  }

  int ditherPixel(int x, int y, int32_t c2, float beta) {  // GC:125-185
    const int bidx = x + y * width;
    const int32_t pixel = pixels[bidx];
    const int plen = (int)palette.size();
    const std::vector<float>& sal = *saliencies;
    int r_pix = Color::red(c2), g_pix = Color::green(c2), b_pix = Color::blue(c2), a_pix = Color::alpha(c2);

    const float strength = 1 / 3.f;
    const int acceptedDiff = std::max(2, plen - margin);
    if (plen <= 4 && sal[bidx] > .2f && sal[bidx] < .25f)
      c2 = BlueNoise::diffuse(pixel, palette[qPixels[bidx]], beta * 2 / sal[bidx], strength, x, y);
    else if (plen <= 4 || CIELAB::Y_Diff(pixel, c2) < (2 * acceptedDiff)) {
      if (plen > 64) {
        float kappa = sal[bidx] < .6f ? beta * .15f / sal[bidx] : beta * .4f / sal[bidx];
        c2 = BlueNoise::diffuse(pixel, palette[qPixels[bidx]], kappa, strength, x, y);
      } else if (plen > 16 && weight < .005)
        c2 = BlueNoise::diffuse(pixel, palette[qPixels[bidx]], beta * normalDistribution(sal[bidx], .5f) + beta, strength, x, y);
      else
        c2 = BlueNoise::diffuse(pixel, palette[qPixels[bidx]], beta * .5f / sal[bidx], strength, x, y);
    }

    double gamma = (plen <= 32 && weight < .01 && weight > .007) ? (double)(1 - beta) : (double)beta;
    if (plen > 4 && CIELAB::Y_Diff(pixel, c2) > (gamma * acceptedDiff)) {
      if (margin > 6 || gamma > beta) {
        float kappa = sal[bidx] < .4f ? beta * .4f * sal[bidx] : beta * .4f / sal[bidx];
        int32_t c1 = Color::argb(a_pix, r_pix, g_pix, b_pix);
        if (plen > 32 && sal[bidx] < .9)
          kappa = beta * normalDistribution(sal[bidx], 2.f);
        else {
          if (weight >= .0015 && sal[bidx] < .6) c1 = pixel;
          if (weight >= .005 && sal[bidx] < .6)
            kappa = beta * normalDistribution(sal[bidx], weight < .0008 ? 2.5f : 1.75f);
          else if (plen >= 32 || CIELAB::Y_Diff(c1, c2) > (gamma * JPI * acceptedDiff)) {
            double ub = 1 - plen / 320.0;
            if (sal[bidx] > .15 && sal[bidx] < ub)
              kappa = beta * (!sortedByYDiff && weight < .0025 ? .55f : .5f) / sal[bidx];
            else
              kappa = beta * normalDistribution(sal[bidx], weight < .0025 ? 1.82f : 2.f);
          }
        }
        c2 = BlueNoise::diffuse(c1, palette[qPixels[bidx]], kappa, strength, x, y);
      } else if (plen <= 32 && weight >= .004)
        c2 = BlueNoise::diffuse(c2, palette[qPixels[bidx]], beta * normalDistribution(sal[bidx], .25f), strength, x, y);
      else
        c2 = Color::argb(a_pix, r_pix, g_pix, b_pix);
    }

    if (DITHER_MAX < 16 && plen > 4 && sal[bidx] < .6f && CIELAB::Y_Diff(pixel, c2) > margin - 1)
      c2 = Color::argb(a_pix, r_pix, g_pix, b_pix);
    if (plen > 32 && sal[bidx] > .95) {
      float kappa = beta * std::max(.05f, .75f - plen / 128.f) * sal[bidx];
      c2 = BlueNoise::diffuse(pixel, palette[qPixels[bidx]], kappa, strength, x, y);
    }
    return ditherable.nearestColorIndex(palette, c2, bidx);
  }

  void diffusePixel(int x, int y) {  // GC:187-280
    const int bidx = x + y * width;
    const int32_t pixel = pixels[bidx];
    const int plen = (int)palette.size();
    ErrorBox error(pixel);

    float maxErr = (float)(DITHER_MAX - 1);
    int i = sortedByYDiff ? (int)weights.size() - 1 : 0;
    for (size_t qi = 0, qn = qSize(); qi < qn; ++qi) {
      const ErrorBox& eb = qAt(qi);
      if (i < 0 || i >= (int)weights.size()) break;
      for (int j = 0; j < 4; ++j) {
        error.p[j] += eb.p[j] * weights[i];
        if (error.p[j] > maxErr) maxErr = error.p[j];
      }
      i += sortedByYDiff ? -1 : 1;
    }

    int r_pix = j2i(std::min(255.0, std::max((double)error.p[0], 0.0)));
    int g_pix = j2i(std::min(255.0, std::max((double)error.p[1], 0.0)));
    int b_pix = j2i(std::min(255.0, std::max((double)error.p[2], 0.0)));
    int a_pix = j2i(std::min(255.0, std::max((double)error.p[3], 0.0)));

    int32_t c2 = Color::argb(a_pix, r_pix, g_pix, b_pix);
    if (saliencies != nullptr && dither && !sortedByYDiff && (!hasAlpha || Color::alpha(pixel) < a_pix)) {
      if ((plen >= 256 && (*saliencies)[bidx] > .99f) || (hasAlpha && (Color::alpha(pixel) - a_pix) < (.5 * margin)))
        qPixels[bidx] = ditherable.nearestColorIndex(palette, c2, bidx);
      else
        qPixels[bidx] = ditherPixel(x, y, c2, beta);
    } else if (plen <= 32 && a_pix > 0xF0) {
      qPixels[bidx] = ditherable.nearestColorIndex(palette, c2, bidx);
      const int acceptedDiff = std::max(2, plen - margin);
      if (saliencies != nullptr && (CIELAB::Y_Diff(pixel, c2) > acceptedDiff || CIELAB::U_Diff(pixel, c2) > (2 * acceptedDiff))) {
        const float strength = 1 / 3.f;
        c2 = BlueNoise::diffuse(pixel, palette[qPixels[bidx]], 1 / (*saliencies)[bidx], strength, x, y);
        qPixels[bidx] = ditherable.nearestColorIndex(palette, c2, bidx);
      }
    } else
      qPixels[bidx] = ditherable.nearestColorIndex(palette, c2, bidx);

    if ((int)qSize() >= DITHER_MAX) qPoll();
    else if (qSize() != 0) initWeights((int)qSize());

    c2 = palette[qPixels[bidx]];
    error.p[0] = (float)(r_pix - Color::red(c2));
    error.p[1] = (float)(g_pix - Color::green(c2));
    error.p[2] = (float)(b_pix - Color::blue(c2));
    error.p[3] = (float)(a_pix - Color::alpha(c2));

    bool denoise = plen > 2;
    bool diffuse = TELL_BLUE_NOISE[bidx & 4095] > thresold;
    error.yDiff = sortedByYDiff ? CIELAB::Y_Diff(pixel, c2) : 1;
    bool illusion = !diffuse && TELL_BLUE_NOISE[j2i(error.yDiff * 4096) & 4095] > thresold;

    bool unaccepted = false;
    int errLength = denoise ? 4 - 1 : 0;
    for (int j = 0; j < errLength; ++j) {
      if (std::fabs(error.p[j]) >= ditherMax) {
        if (sortedByYDiff && saliencies != nullptr) unaccepted = true;
        if (diffuse)
          error.p[j] = (float)M.tanh(error.p[j] / maxErr * 20) * (ditherMax - 1);
        else if (illusion)
          error.p[j] = (float)(error.p[j] / maxErr * error.yDiff) * (ditherMax - 1);
        else
          error.p[j] /= (float)(1 + JMath::sqrt(ditherMax));
      }
      if (sortedByYDiff && saliencies == nullptr && std::fabs(error.p[j]) >= DITHER_MAX) unaccepted = true;
    }

    if (unaccepted) {
      if (saliencies != nullptr)
        qPixels[bidx] = ditherPixel(x, y, c2, beta);
      else if (CIELAB::Y_Diff(pixel, c2) > 3 && CIELAB::U_Diff(pixel, c2) > 3) {
        const float strength = 1 / 3.f;
        c2 = BlueNoise::diffuse(pixel, palette[qPixels[bidx]], strength, strength, x, y);
        qPixels[bidx] = ditherable.nearestColorIndex(palette, c2, bidx);
      }
    }

    qAdd(error);

    if (dither || plen <= 32) qPixels[bidx] = palette[qPixels[bidx]];
  }

  static int sgn(int v) { return (v > 0) - (v < 0); }
  void generate2d(int x, int y, int ax, int ay, int bx, int by) {  // GC:282-334
    int w = std::abs(ax + ay), h = std::abs(bx + by);
    int dax = sgn(ax), day = sgn(ay), dbx = sgn(bx), dby = sgn(by);
    if (h == 1) {
      for (int i = 0; i < w; ++i) { diffusePixel(x, y); x += dax; y += day; }
      return;
    }
    if (w == 1) {
      for (int i = 0; i < h; ++i) { diffusePixel(x, y); x += dbx; y += dby; }
      return;
    }
    int ax2 = ax / 2, ay2 = ay / 2, bx2 = bx / 2, by2 = by / 2;
    int w2 = std::abs(ax2 + ay2), h2 = std::abs(bx2 + by2);
    if (2 * w > 3 * h) {
      if ((w2 % 2) != 0 && w > 2) { ax2 += dax; ay2 += day; }
      generate2d(x, y, ax2, ay2, bx, by);
      generate2d(x + ax2, y + ay2, ax - ax2, ay - ay2, bx, by);
      return;
    }
    if ((h2 % 2) != 0 && h > 2) { bx2 += dbx; by2 += dby; }
    generate2d(x, y, bx2, by2, ax2, ay2);
    generate2d(x + bx2, y + by2, ax, ay, bx - bx2, by - by2);
    generate2d(x + (ax - dax) + (bx2 - dbx), y + (ay - day) + (by2 - dby), -bx2, -by2, -(ax - ax2), -(ay - ay2));
  }

  void initWeights(int size) {  // GC:336-354
    const float weightRatio = (float)M.pow(BLOCK_SIZE + 1.f, 1.f / (size - 1.f));
    float weight = 1.f, sumweight = 0.f;
    weights.assign(size, 0.f);
    for (int c = 0; c < size; ++c) {
      qAdd(ErrorBox());
      sumweight += (weights[size - c - 1] = weight);
      weight /= weightRatio;
    }
    weight = 0.f;
    for (int c = 0; c < size; ++c) weight += (weights[c] /= sumweight);
    weights[0] += 1.f - weight;
  }

  void run() {  // GC:356-365
    if (!sortedByYDiff) initWeights(DITHER_MAX);
    if (width >= height) generate2d(0, 0, width, 0, 0, height);
    else generate2d(0, 0, 0, height, width, 0);
  }
  void initWeightsPublic(int size) { initWeights(size); }
};

// Gilbert order only (GC:282-334, 356-365), for the known-answer tests
struct OrderOnly {
  std::vector<uint32_t> out;
  int width;
  static int sgn(int v) { return (v > 0) - (v < 0); }
  void gen(int x, int y, int ax, int ay, int bx, int by) {
    int w = std::abs(ax + ay), h = std::abs(bx + by);
    int dax = sgn(ax), day = sgn(ay), dbx = sgn(bx), dby = sgn(by);
    if (h == 1) { for (int i = 0; i < w; ++i) { out.push_back((uint32_t)(x + y * width)); x += dax; y += day; } return; }
    if (w == 1) { for (int i = 0; i < h; ++i) { out.push_back((uint32_t)(x + y * width)); x += dbx; y += dby; } return; }
    int ax2 = ax / 2, ay2 = ay / 2, bx2 = bx / 2, by2 = by / 2;
    int w2 = std::abs(ax2 + ay2), h2 = std::abs(bx2 + by2);
    if (2 * w > 3 * h) {
      if ((w2 % 2) != 0 && w > 2) { ax2 += dax; ay2 += day; }
      gen(x, y, ax2, ay2, bx, by);
      gen(x + ax2, y + ay2, ax - ax2, ay - ay2, bx, by);
      return;
    }
    if ((h2 % 2) != 0 && h > 2) { bx2 += dbx; by2 += dby; }
    gen(x, y, bx2, by2, ax2, ay2);
    gen(x + bx2, y + by2, ax, ay, bx - bx2, by - by2);
    gen(x + (ax - dax) + (bx2 - dbx), y + (ay - day) + (by2 - dby), -bx2, -by2, -(ax - ax2), -(ay - ay2));
  }
};

// ---------------------------------------------------------------------------------------------
// Trace of one convert() (what the parity tests compare stage by stage)
// ---------------------------------------------------------------------------------------------
struct Trace {
  int hasSemiTransparency = 0, transparentPixelIndex = -1, maxbins = 0, quan_rt = 0, texicab = 0, isNano = 0;
  int32_t transparentColor = 0;
  double weight = 0, ratio_init = 0, ratio_merge = 0, PR = 0, PG = 0, PB = 0, PA = 0, weight_final = 0;
  std::vector<double> bins;         // maxbins x 5: (ac, c1, c2, c3, cnt) after mean + quanFn, before merging
  std::vector<float> init_err;      // find_nn results of the initial sweep
  std::vector<int32_t> init_nn;
  std::vector<int32_t> merges;      // pairs (tb, nb) in merge order
  std::vector<float> saliencies;
  GilbertParams gp{};
  std::vector<float> gweights;
  int64_t rng_draws = 0, pixelMapSize = 0;
  int64_t n_rescans = 0, n_heap_pops = 0;  // merge loop: find_nn calls on a stale top, deleted tops replaced by the last entry
  bool keep_draws = false;          // debugging aid of tests/spec_host_harness.cpp: the pixel (bidx) of every draw, in order
  std::vector<int32_t> draw_bidx;
  float bn_weight = 0;
};

// ---------------------------------------------------------------------------------------------
// PnnQuantizer (PQ)
// ---------------------------------------------------------------------------------------------
class PnnQuantizer {
 protected:
  short alphaThreshold = 0xF;  // PQ:17
  bool hasSemiTransparency = false;
  int m_transparentPixelIndex = -1;
  int width, height;
  std::vector<int32_t> pixels;
  int32_t m_transparentColor = Color::argb(0, BYTE_MAX, BYTE_MAX, BYTE_MAX);  // PQ:22
  double PR = 0.299, PG = 0.587, PB = 0.114, PA = .3333;  // PQ:24
  double ratio = .5, weight = 1;                         // PQ:25
  static constexpr float coeffs[3][3] = {{0.299f, 0.587f, 0.114f}, {-0.14713f, -0.28886f, 0.436f}, {0.615f, -0.51499f, -0.10001f}};  // PQ:26-30
  std::unordered_map<int32_t, std::array<int32_t, 4>> closestMap;  // PQ:32
  std::unordered_map<int32_t, short> nearestMap;                   // PQ:33

  struct Pnnbin {  // PQ:51-55
    double ac = 0, rc = 0, gc = 0, bc = 0;
    float cnt = 0, err = 0;
    int nn = 0, fw = 0, bk = 0, tm = 0, mtm = 0;
  };

 public:
  Trace trace;
  uint64_t rngSeed = 0;

  PnnQuantizer(const uint32_t* argb, int w, int h) : width(w), height(h) {  // PQ:35-44 with int[] in place of a Bitmap
    pixels.resize((size_t)w * h);
    for (size_t i = 0; i < pixels.size(); ++i) pixels[i] = (int32_t)argb[i];
  }
  virtual ~PnnQuantizer() {}
  bool hasAlpha() const { return m_transparentPixelIndex > -1; }  // PQ:458-460

 private:
  void find_nn(std::vector<Pnnbin>& bins, int idx) {  // PQ:57-116
    int nn = 0;
    double err = 1e100;
    Pnnbin& bin1 = bins[idx];
    float n1 = bin1.cnt;
    double wa = bin1.ac, wr = bin1.rc, wg = bin1.gc, wb = bin1.bc;

    int start = 0;
    if (TELL_BLUE_NOISE[idx & 4095] > 0) start = (PG < coeffs[0][1]) ? 3 : 1;

    for (int i = bin1.fw; i != 0; i = bins[i].fw) {
      double n2 = bins[i].cnt, nerr2 = (n1 * n2) / (n1 + n2);
      if (nerr2 >= err) continue;

      double nerr = 0.0;
      if (hasSemiTransparency) {
        nerr += nerr2 * PA * sqr(bins[i].ac - wa);
        if (nerr >= err) continue;
      }
      nerr += nerr2 * (1 - ratio) * PR * sqr(bins[i].rc - wr);
      if (nerr >= err) continue;
      nerr += nerr2 * (1 - ratio) * PG * sqr(bins[i].gc - wg);
      if (nerr >= err) continue;
      nerr += nerr2 * (1 - ratio) * PB * sqr(bins[i].bc - wb);
      if (nerr >= err) continue;

      for (int j = start; j < 3; ++j) {
        nerr += nerr2 * ratio * sqr(coeffs[j][0] * (bins[i].rc - wr));
        if (nerr >= err) break;
        nerr += nerr2 * ratio * sqr(coeffs[j][1] * (bins[i].gc - wg));
        if (nerr >= err) break;
        nerr += nerr2 * ratio * sqr(coeffs[j][2] * (bins[i].bc - wb));
        if (nerr >= err) break;
      }
      err = nerr;  // reached after a break as well (PQ:97-112)
      nn = i;
    }
    bin1.err = (float)err;
    bin1.nn = nn;
  }

 protected:
  virtual float quanFn(int nMaxColors, short quan_rt, float cnt) {  // PQ:123-132
    if (quan_rt > 0) {
      if (nMaxColors < 64) return (float)JMath::sqrt(cnt);
      return (float)j2i(JMath::sqrt(cnt));
    }
    if (quan_rt < 0) return (float)j2i(M.cbrt(cnt));
    return cnt;
  }

  virtual std::vector<int32_t> pnnquan(const std::vector<int32_t>& pixels, int nMaxColors) {  // PQ:134-267
    short quan_rt = 1;
    std::vector<Pnnbin> storage;
    storage.reserve(65536);
    std::vector<int> slot(65536, -1);

    for (int32_t pixel : pixels) {  // PQ:140-154
      if (Color::alpha(pixel) <= alphaThreshold) pixel = m_transparentColor;
      int index = getColorIndex(pixel, hasSemiTransparency, nMaxColors < 64 || m_transparentPixelIndex >= 0);
      if (slot[index] < 0) { slot[index] = (int)storage.size(); storage.emplace_back(); }
      Pnnbin& tb = storage[slot[index]];
      tb.ac += Color::alpha(pixel);
      tb.rc += Color::red(pixel);
      tb.gc += Color::green(pixel);
      tb.bc += Color::blue(pixel);
      tb.cnt++;
    }

    int maxbins = 0;  // PQ:157-170
    std::vector<Pnnbin> bins(65536);
    for (int i = 0; i < 65536; ++i) {
      if (slot[i] < 0) continue;
      Pnnbin b = storage[slot[i]];
      float d = 1.f / b.cnt;
      b.ac *= d; b.rc *= d; b.gc *= d; b.bc *= d;
      bins[maxbins++] = b;
    }

    if (nMaxColors < 16) quan_rt = -1;
    weight = std::min(0.9, nMaxColors * 1.0 / maxbins);
    if (weight < .04 && PG >= coeffs[0][1]) {
      PR = PG = PB = PA = 1;
      if (nMaxColors >= 64) quan_rt = 0;
    }

    int j = 0;
    for (; j < maxbins - 1; ++j) {
      bins[j].fw = j + 1;
      bins[j + 1].bk = j;
      bins[j].cnt = quanFn(nMaxColors, quan_rt, bins[j].cnt);
    }
    bins[j].cnt = quanFn(nMaxColors, quan_rt, bins[j].cnt);

    trace.maxbins = maxbins; trace.quan_rt = quan_rt; trace.weight = weight; trace.ratio_init = trace.ratio_merge = ratio;
    trace.PR = PR; trace.PG = PG; trace.PB = PB; trace.PA = PA;
    trace.bins.resize((size_t)maxbins * 5);
    for (int i = 0; i < maxbins; ++i) {
      double* o = &trace.bins[(size_t)i * 5];
      o[0] = bins[i].ac; o[1] = bins[i].rc; o[2] = bins[i].gc; o[3] = bins[i].bc; o[4] = bins[i].cnt;
    }

    int h, l, l2;
    std::vector<int> heap(65537, 0);  // PQ:195
    for (int i = 0; i < maxbins; i++) {
      find_nn(bins, i);
      float err = bins[i].err;
      for (l = ++heap[0]; l > 1; l = l2) {
        l2 = l >> 1;
        if (bins[h = heap[l2]].err <= err) break;
        heap[l] = h;
      }
      heap[l] = i;
    }
    trace.init_err.resize(maxbins); trace.init_nn.resize(maxbins);
    for (int i = 0; i < maxbins; ++i) { trace.init_err[i] = bins[i].err; trace.init_nn[i] = bins[i].nn; }

    int extbins = maxbins - nMaxColors;  // PQ:210-255
    for (int i = 0; i < extbins;) {
      Pnnbin* tb;
      for (;;) {
        int b1 = heap[1];
        tb = &bins[b1];
        if ((tb->tm >= tb->mtm) && (bins[tb->nn].mtm <= tb->tm)) break;
        if (tb->mtm == 0xFFFF) {
          b1 = heap[1] = heap[heap[0]--];
          ++trace.n_heap_pops;
        } else {
          find_nn(bins, b1);
          tb->tm = i;
          ++trace.n_rescans;
        }
        float err = bins[b1].err;
        for (l = 1; (l2 = l + l) <= heap[0]; l = l2) {
          if ((l2 < heap[0]) && (bins[heap[l2]].err > bins[heap[l2 + 1]].err)) ++l2;
          if (err <= bins[h = heap[l2]].err) break;
          heap[l] = h;
        }
        heap[l] = b1;
      }

      Pnnbin& nb = bins[tb->nn];
      trace.merges.push_back((int32_t)(tb - &bins[0]));
      trace.merges.push_back(tb->nn);
      float n1 = tb->cnt, n2 = nb.cnt;
      float d = 1.f / (n1 + n2);
      tb->ac = d * (float)jround(n1 * tb->ac + n2 * nb.ac);  // float * long -> float (JLS 5.6.2), then widened
      tb->rc = d * (float)jround(n1 * tb->rc + n2 * nb.rc);  // float * long -> float (JLS 5.6.2), then widened
      tb->gc = d * (float)jround(n1 * tb->gc + n2 * nb.gc);  // float * long -> float (JLS 5.6.2), then widened
      tb->bc = d * (float)jround(n1 * tb->bc + n2 * nb.bc);  // float * long -> float (JLS 5.6.2), then widened
      tb->cnt += n2;
      tb->mtm = ++i;

      bins[nb.bk].fw = nb.fw;
      bins[nb.fw].bk = nb.bk;
      nb.mtm = 0xFFFF;
    }

    std::vector<int32_t> palette(extbins > 0 ? nMaxColors : maxbins);  // PQ:258-264
    short k = 0;
    for (int i = 0; k < (short)palette.size(); ++k) {
      palette[k] = Color::argb(j2i(bins[i].ac), j2i(bins[i].rc), j2i(bins[i].gc), j2i(bins[i].bc));
      i = bins[i].fw;
    }
    return palette;
  }

  virtual short nearestColorIndex(const std::vector<int32_t>& palette, int32_t c, int pos) {  // PQ:269-311
    const int32_t offset = weight > .015 ? c : getColorIndex(c, hasSemiTransparency, m_transparentPixelIndex >= 0);
    NQ_ORACLE_PROBE(offset);
    auto got = nearestMap.find(offset);
    if (got != nearestMap.end()) return got->second;

    short k = 0;
    const int plen = (int)palette.size();
    if (Color::alpha(c) <= alphaThreshold) c = m_transparentColor;
    if (plen > 2 && hasAlpha() && Color::alpha(c) > alphaThreshold) k = 1;

    double pr = PR, pg = PG, pb = PB, pa = PA;
    if (plen < 3) pr = pg = pb = pa = 1;

    double mindist = INT32_MAX;
    for (short i = k; i < plen; ++i) {
      int32_t c2 = palette[i];
      double curdist = pa * sqr(Color::alpha(c2) - Color::alpha(c));
      if (curdist > mindist) continue;
      curdist += pr * sqr(Color::red(c2) - Color::red(c));
      if (curdist > mindist) continue;
      curdist += pg * sqr(Color::green(c2) - Color::green(c));
      if (curdist > mindist) continue;
      curdist += pb * sqr(Color::blue(c2) - Color::blue(c));
      if (curdist > mindist) continue;
      mindist = curdist;
      k = i;
    }
    nearestMap[offset] = k;
    return k;
  }

  virtual short closestColorIndex(const std::vector<int32_t>& palette, int32_t c, int pos) {  // PQ:313-375
    short k = 0;
    const int plen = (int)palette.size();
    if (Color::alpha(c) <= alphaThreshold) return nearestColorIndex(palette, c, pos);

    const int32_t offset = weight > .015 ? c : getColorIndex(c, hasSemiTransparency, m_transparentPixelIndex >= 0);
    std::array<int32_t, 4> closest;
    auto it = closestMap.find(c);
    if (it == closestMap.end()) {
      closest = {0, 0, INT32_MAX, INT32_MAX};
      double pr = PR, pg = PG, pb = PB, pa = PA;
      if (plen < 3) pr = pg = pb = pa = 1;
      for (; k < plen; ++k) {
        int32_t c2 = palette[k];
        double err = pr * sqr(Color::red(c2) - Color::red(c));
        if (err >= closest[3]) continue;
        err += pg * sqr(Color::green(c2) - Color::green(c));
        if (err >= closest[3]) continue;
        err += pb * sqr(Color::blue(c2) - Color::blue(c));
        if (err >= closest[3]) continue;
        if (hasSemiTransparency) err += pa * sqr(Color::alpha(c2) - Color::alpha(c));
        if (err < closest[2]) {
          closest[1] = closest[0];
          closest[3] = closest[2];
          closest[0] = k;
          closest[2] = j2i(err);
        } else if (err < closest[3]) {
          closest[1] = k;
          closest[3] = j2i(err);
        }
      }
      if (closest[3] == INT32_MAX) closest[1] = closest[0];
      closestMap[offset] = closest;
    } else
      closest = it->second;

    int MAX_ERR = plen << 2;
    int idx = (pos + 1) % 2;
    if (closest[3] * .67 < (double)(closest[3] - closest[2])) idx = 0;
    else if (closest[0] > closest[1]) idx = pos % 2;

    if (closest[idx + 2] >= MAX_ERR || (hasAlpha() && closest[idx] == 0)) return nearestColorIndex(palette, c, pos);
    return (short)closest[idx];
  }

  // getDitherFn (PQ:377-391)
  struct RgbDitherable : Ditherable {
    PnnQuantizer& q; bool dither;
    RgbDitherable(PnnQuantizer& q_, bool d) : q(q_), dither(d) {}
    int getColorIndex(int32_t c) override { return ::getColorIndex(c, q.hasSemiTransparency, q.m_transparentPixelIndex >= 0); }
    short nearestColorIndex(const std::vector<int32_t>& palette, int32_t c, int pos) override {
      if (dither) return q.nearestColorIndex(palette, c, pos);
      return q.closestColorIndex(palette, c, pos);
    }
  };

  virtual std::vector<int32_t> ditherImage(const std::vector<int32_t>& cPixels, std::vector<int32_t>& palette, int width, int height, bool dither) {  // PQ:393-407
    RgbDitherable ditherable(*this, dither);
    if (hasSemiTransparency) weight *= -1;
    std::vector<int32_t> qPixels(cPixels.size(), 0);
    {
      GilbertCurve gc(width, height, cPixels, palette, qPixels, ditherable, nullptr, weight, dither);
      trace.gp = gc.params();
      gc.run();
      trace.gweights = gc.getWeights();
    }
    if (!dither && palette.size() > 32) {
      trace.bn_weight = 1.0f;
      BlueNoise::dither(width, height, cPixels, palette, ditherable, qPixels, 1.0f);
    }
    closestMap.clear();
    nearestMap.clear();
    return qPixels;
  }

 public:
  std::vector<int32_t> palette_out;

  std::vector<int32_t> convert(int nMaxColors, bool dither) {  // PQ:409-456
    int semiTransCount = 0;
    for (size_t i = 0; i < pixels.size(); ++i) {
      int32_t pixel = pixels[i];
      int alfa = (pixel >> 24) & 0xff, r = (pixel >> 16) & 0xff, g = (pixel >> 8) & 0xff, b = pixel & 0xff;
      pixels[i] = Color::argb(alfa, r, g, b);
      if (alfa < 0xE0) {
        if (alfa == 0) {
          m_transparentPixelIndex = (int)i;
          if (nMaxColors > 2) m_transparentColor = pixels[i];
          else pixels[i] = m_transparentColor;
        } else if (alfa > alphaThreshold)
          ++semiTransCount;
      }
    }

    hasSemiTransparency = semiTransCount > 0;
    if (nMaxColors <= 32) PR = PG = PB = PA = 1;
    else { PR = coeffs[0][0]; PG = coeffs[0][1]; PB = coeffs[0][2]; }

    std::vector<int32_t> palette;
    if (nMaxColors > 2) palette = pnnquan(pixels, nMaxColors);
    else {
      palette.resize(nMaxColors);
      weight = 1;
      if (m_transparentPixelIndex >= 0) {
        palette[0] = m_transparentColor;
        palette[1] = Color::BLACK;
      } else {
        palette[0] = Color::BLACK;
        palette[1] = Color::WHITE;
      }
    }
    trace.hasSemiTransparency = hasSemiTransparency;
    trace.transparentPixelIndex = m_transparentPixelIndex;
    trace.transparentColor = m_transparentColor;
    trace.weight = weight;
    palette_out = palette;

    std::vector<int32_t> qPixels = ditherImage(pixels, palette, width, height, dither);
    trace.weight_final = weight;
    return qPixels;
  }
};
constexpr float PnnQuantizer::coeffs[3][3];

// ---------------------------------------------------------------------------------------------
// PnnLABQuantizer (PL)
// ---------------------------------------------------------------------------------------------
class PnnLABQuantizer : public PnnQuantizer {
  bool isNano = false;  // PL:18
  std::vector<float> saliencies;  // PL:19 (empty + hasSaliencies=false stands for null)
  bool hasSaliencies = false;
  std::unordered_map<int32_t, Lab> pixelMap;  // PL:20
  std::vector<int32_t> pixelMapOrder;         // insertion order, for the HashMap iteration at PL:197
  JRandom random;                             // PL:22 (static, unseeded in the reference; seed injected here)

  struct Pnnbin {  // PL:28-32
    float ac = 0, Lc = 0, Ac = 0, Bc = 0, err = 0;
    float cnt = 0;
    int nn = 0, fw = 0, bk = 0, tm = 0, mtm = 0;
  };

  const Lab& getLab(int32_t c) {  // PL:34-42
    auto it = pixelMap.find(c);
    if (it == pixelMap.end()) {
      it = pixelMap.emplace(c, CIELAB::RGB2LAB(c)).first;
      pixelMapOrder.push_back(c);
    }
    return it->second;
  }

  void find_nn(std::vector<Pnnbin>& bins, int idx, bool texicab) {  // PL:44-115
    int nn = 0;
    double err = 1e100;
    Pnnbin& bin1 = bins[idx];
    float n1 = bin1.cnt;
    Lab lab1;
    lab1.alpha = bin1.ac; lab1.L = bin1.Lc; lab1.A = bin1.Ac; lab1.B = bin1.Bc;
    const double exp175 = M.exp(1.75);
    for (int i = bin1.fw; i != 0; i = bins[i].fw) {
      float n2 = bins[i].cnt;
      double nerr2 = (n1 * n2) / (n1 + n2);
      if (nerr2 >= err) continue;

      Lab lab2;
      lab2.alpha = bins[i].ac; lab2.L = bins[i].Lc; lab2.A = bins[i].Ac; lab2.B = bins[i].Bc;
      double alphaDiff = hasSemiTransparency ? sqr(lab2.alpha - lab1.alpha) / exp175 : 0;
      double nerr = nerr2 * alphaDiff;
      if (nerr >= err) continue;

      if (!texicab) {
        nerr += (1 - ratio) * nerr2 * sqr(lab2.L - lab1.L);
        if (nerr >= err) continue;
        nerr += (1 - ratio) * nerr2 * sqr(lab2.A - lab1.A);
        if (nerr >= err) continue;
        nerr += (1 - ratio) * nerr2 * sqr(lab2.B - lab1.B);
      } else {
        nerr += (1 - ratio) * nerr2 * std::fabs(lab2.L - lab1.L);
        if (nerr >= err) continue;
        nerr += (1 - ratio) * nerr2 * JMath::sqrt(sqr(lab2.A - lab1.A) + sqr(lab2.B - lab1.B));
      }
      if (nerr > err) continue;

      float deltaL_prime_div_k_L_S_L = CIELAB::L_prime_div_k_L_S_L(lab1, lab2);
      nerr += ratio * nerr2 * sqr(deltaL_prime_div_k_L_S_L);
      if (nerr > err) continue;

      double a1Prime = 0, a2Prime = 0, CPrime1 = 0, CPrime2 = 0;
      float deltaC_prime_div_k_L_S_L = CIELAB::C_prime_div_k_L_S_L(lab1, lab2, a1Prime, a2Prime, CPrime1, CPrime2);
      nerr += ratio * nerr2 * sqr(deltaC_prime_div_k_L_S_L);
      if (nerr > err) continue;

      double barCPrime = 0, barhPrime = 0;
      float deltaH_prime_div_k_L_S_L = CIELAB::H_prime_div_k_L_S_L(lab1, lab2, a1Prime, a2Prime, CPrime1, CPrime2, barCPrime, barhPrime);
      nerr += ratio * nerr2 * sqr(deltaH_prime_div_k_L_S_L);
      if (nerr > err) continue;

      nerr += ratio * nerr2 * CIELAB::R_T(barCPrime, barhPrime, deltaC_prime_div_k_L_S_L, deltaH_prime_div_k_L_S_L);
      if (nerr > err) continue;

      err = nerr;
      nn = i;
    }
    bin1.err = (float)err;
    bin1.nn = nn;
  }

 protected:
  float quanFn(int nMaxColors, short quan_rt, float cnt) override {  // PL:117-128
    if (quan_rt > 0) {
      if (quan_rt > 1) return (float)M.pow(cnt, 0.75);
      if (nMaxColors < 64) return (float)j2i(JMath::sqrt(cnt));
      return (float)JMath::sqrt(cnt);
    }
    return cnt;
  }

  std::vector<int32_t> pnnquan(const std::vector<int32_t>& pixels, int nMaxColors) override {  // PL:130-327
    short quan_rt = 1;
    std::vector<Pnnbin> storage;
    storage.reserve(65536);
    std::vector<int> slot(65536, -1);
    hasSaliencies = !(nMaxColors >= 128);
    saliencies.assign(hasSaliencies ? pixels.size() : 0, 0.f);
    float saliencyBase = .1f;

    for (size_t i = 0; i < pixels.size(); ++i) {  // PL:139-157
      int32_t pixel = pixels[i];
      if (Color::alpha(pixel) <= alphaThreshold) pixel = m_transparentColor;
      int index = getColorIndex(pixel, hasSemiTransparency, nMaxColors < 64 || m_transparentPixelIndex >= 0);
      const Lab& lab1 = getLab(pixel);
      if (slot[index] < 0) { slot[index] = (int)storage.size(); storage.emplace_back(); }
      Pnnbin& tb = storage[slot[index]];
      tb.ac += lab1.alpha;
      tb.Lc += lab1.L;
      tb.Ac += lab1.A;
      tb.Bc += lab1.B;
      tb.cnt += 1.0f;
      if (hasSaliencies) saliencies[i] = saliencyBase + (1 - saliencyBase) * lab1.L / 100.f * lab1.alpha / 255.f;
    }

    int maxbins = 0;  // PL:160-173
    std::vector<Pnnbin> bins(65536);
    for (int i = 0; i < 65536; ++i) {
      if (slot[i] < 0) continue;
      Pnnbin b = storage[slot[i]];
      float d = 1.f / b.cnt;
      b.ac *= d; b.Lc *= d; b.Ac *= d; b.Bc *= d;
      bins[maxbins++] = b;
    }

    double proportional = sqr(nMaxColors) / maxbins;
    if ((m_transparentPixelIndex >= 0 || hasSemiTransparency) && nMaxColors < 32) quan_rt = -1;

    weight = std::min(0.9, nMaxColors * 1.0 / maxbins);
    isNano = weight <= .015;
    if ((nMaxColors < 16 && weight < .0075) || weight < .001 || (weight > .0015 && weight < .0022)) quan_rt = 2;
    if (weight < .04 && PG < 1 && PG >= coeffs[0][1]) {
      if (nMaxColors >= 64) quan_rt = 0;
    }
    if (nMaxColors > 16 && nMaxColors < 64) {
      double weightB = nMaxColors / 8000.0;
      if (std::fabs(weightB - weight) < .001) quan_rt = 2;
    }
    trace.maxbins = maxbins; trace.weight = weight; trace.isNano = isNano;
    trace.PR = PR; trace.PG = PG; trace.PB = PB; trace.PA = PA;
    trace.pixelMapSize = (int64_t)pixelMap.size();

    if ((int)pixelMap.size() <= nMaxColors) {  // PL:193-206
      std::vector<int32_t> keys = javaHashMapKeyOrder(pixelMapOrder);
      std::vector<int32_t> palette(pixelMap.size());
      int k = 0;
      for (int32_t pixel : keys) {
        palette[k++] = pixel;
        if (k > 1 && Color::alpha(pixel) == 0) {
          palette[k - 1] = palette[0];
          palette[0] = pixel;
        }
      }
      trace.quan_rt = quan_rt;
      return palette;
    }

    int j = 0;
    for (; j < maxbins - 1; ++j) {
      bins[j].fw = j + 1;
      bins[j + 1].bk = j;
      bins[j].cnt = quanFn(nMaxColors, quan_rt, bins[j].cnt);
    }
    bins[j].cnt = quanFn(nMaxColors, quan_rt, bins[j].cnt);

    const bool texicab = proportional > .0225 && !hasSemiTransparency;

    if (hasSemiTransparency) ratio = .5;
    else if (quan_rt != 0 && nMaxColors < 64) {
      if (proportional > .018 && proportional < .022) ratio = std::min(1.0, proportional + weight * M.exp(3.13));
      else if (proportional > .1) ratio = std::min(1.0, 1.0 - weight);
      else if (proportional > .04) ratio = std::min(1.0, weight * M.exp(1.56));
      else if (proportional > .025 && (weight < .002 || weight > .0022)) ratio = std::min(1.0, proportional + weight * M.exp(3.66));
      else ratio = std::min(1.0, proportional + weight * M.exp(1.718));
    } else if (nMaxColors > 256) ratio = std::min(1.0, 1 - 1.0 / proportional);
    else ratio = std::min(1.0, 1 - weight * .7);

    if (!hasSemiTransparency && quan_rt < 0) ratio = std::min(1.0, weight * M.exp(3.13));

    trace.quan_rt = quan_rt; trace.texicab = texicab; trace.ratio_init = ratio;
    trace.bins.resize((size_t)maxbins * 5);
    for (int i = 0; i < maxbins; ++i) {
      double* o = &trace.bins[(size_t)i * 5];
      o[0] = bins[i].ac; o[1] = bins[i].Lc; o[2] = bins[i].Ac; o[3] = bins[i].Bc; o[4] = bins[i].cnt;
    }

    int h, l, l2;
    std::vector<int> heap(65537, 0);
    for (int i = 0; i < maxbins; ++i) {  // PL:246-257
      find_nn(bins, i, texicab);
      float err = bins[i].err;
      for (l = ++heap[0]; l > 1; l = l2) {
        l2 = l >> 1;
        if (bins[h = heap[l2]].err <= err) break;
        heap[l] = h;
      }
      heap[l] = i;
    }
    trace.init_err.resize(maxbins); trace.init_nn.resize(maxbins);
    for (int i = 0; i < maxbins; ++i) { trace.init_err[i] = bins[i].err; trace.init_nn[i] = bins[i].nn; }

    if (quan_rt > 0 && nMaxColors < 64 && proportional > .035 && proportional < .1) {  // PL:259-264
      const int dir = proportional > .04 ? 1 : -1;
      const double margin = dir > 0 ? .002 : .0025;
      const double delta = weight > margin && weight < .003 ? 1.872 : 1.632;
      ratio = std::min(1.0, proportional + dir * weight * M.exp(delta));
    }
    trace.ratio_merge = ratio;

    int extbins = maxbins - nMaxColors;  // PL:267-312
    for (int i = 0; i < extbins;) {
      Pnnbin* tb;
      for (;;) {
        int b1 = heap[1];
        tb = &bins[b1];
        if ((tb->tm >= tb->mtm) && (bins[tb->nn].mtm <= tb->tm)) break;
        if (tb->mtm == 0xFFFF) {
          b1 = heap[1] = heap[heap[0]--];
          ++trace.n_heap_pops;
        } else {
          find_nn(bins, b1, texicab);
          tb->tm = i;
          ++trace.n_rescans;
        }
        float err = bins[b1].err;
        for (l = 1; (l2 = l + l) <= heap[0]; l = l2) {
          if ((l2 < heap[0]) && (bins[heap[l2]].err > bins[heap[l2 + 1]].err)) ++l2;
          if (err <= bins[h = heap[l2]].err) break;
          heap[l] = h;
        }
        heap[l] = b1;
      }

      Pnnbin& nb = bins[tb->nn];
      trace.merges.push_back((int32_t)(tb - &bins[0]));
      trace.merges.push_back(tb->nn);
      float n1 = tb->cnt, n2 = nb.cnt;
      float d = 1.0f / (n1 + n2);
      tb->ac = d * (n1 * tb->ac + n2 * nb.ac);
      tb->Lc = d * (n1 * tb->Lc + n2 * nb.Lc);
      tb->Ac = d * (n1 * tb->Ac + n2 * nb.Ac);
      tb->Bc = d * (n1 * tb->Bc + n2 * nb.Bc);
      tb->cnt += n2;
      tb->mtm = ++i;

      bins[nb.bk].fw = nb.fw;
      bins[nb.fw].bk = nb.bk;
      nb.mtm = 0xFFFF;
    }

    std::vector<int32_t> palette(extbins > 0 ? nMaxColors : maxbins);  // PL:315-324
    short k = 0;
    for (int i = 0; k < (short)palette.size(); ++k) {
      Lab lab1;
      lab1.alpha = (float)j2i(bins[i].ac);
      lab1.L = bins[i].Lc; lab1.A = bins[i].Ac; lab1.B = bins[i].Bc;
      palette[k] = CIELAB::LAB2RGB(lab1);
      i = bins[i].fw;
    }
    return palette;
  }

  short nearestColorIndex(const std::vector<int32_t>& palette, int32_t c, int pos) override {  // PL:329-404
    const int32_t offset = !isNano ? c : getColorIndex(c, hasSemiTransparency, m_transparentPixelIndex >= 0);
    NQ_ORACLE_PROBE(offset);
    auto got = nearestMap.find(offset);
    if (got != nearestMap.end()) return got->second;

    short k = 0;
    const int plen = (int)palette.size();
    if (Color::alpha(c) <= alphaThreshold) c = m_transparentColor;
    if (plen > 2 && hasAlpha() && Color::alpha(c) > alphaThreshold) k = 1;

    double mindist = INT32_MAX;
    const Lab lab1 = getLab(c);
    const double exp15 = M.exp(1.5);
    for (short i = k; i < plen; ++i) {
      int32_t c2 = palette[i];
      double curdist = hasSemiTransparency ? sqr(Color::alpha(c2) - Color::alpha(c)) / exp15 : 0;
      if (curdist > mindist) continue;

      const Lab lab2 = getLab(c2);
      if (plen <= 4) {
        curdist = sqr(Color::red(c2) - Color::red(c)) + sqr(Color::green(c2) - Color::green(c)) + sqr(Color::blue(c2) - Color::blue(c));
        if (hasSemiTransparency) curdist += sqr(Color::alpha(c2) - Color::alpha(c));
      } else if (hasSemiTransparency || plen < 16) {
        curdist += sqr(lab2.L - lab1.L);
        if (curdist > mindist) continue;
        curdist += sqr(lab2.A - lab1.A);
        if (curdist > mindist) continue;
        curdist += sqr(lab2.B - lab1.B);
      } else if (plen > 32) {
        curdist += std::fabs(lab2.L - lab1.L);
        if (curdist > mindist) continue;
        curdist += JMath::sqrt(sqr(lab2.A - lab1.A) + sqr(lab2.B - lab1.B));
      } else {
        float deltaL_prime_div_k_L_S_L = CIELAB::L_prime_div_k_L_S_L(lab1, lab2);
        curdist += sqr(deltaL_prime_div_k_L_S_L);
        if (curdist > mindist) continue;

        double a1Prime = 0, a2Prime = 0, CPrime1 = 0, CPrime2 = 0;
        float deltaC_prime_div_k_L_S_L = CIELAB::C_prime_div_k_L_S_L(lab1, lab2, a1Prime, a2Prime, CPrime1, CPrime2);
        curdist += sqr(deltaC_prime_div_k_L_S_L);
        if (curdist > mindist) continue;

        double barCPrime = 0, barhPrime = 0;
        float deltaH_prime_div_k_L_S_L = CIELAB::H_prime_div_k_L_S_L(lab1, lab2, a1Prime, a2Prime, CPrime1, CPrime2, barCPrime, barhPrime);
        curdist += sqr(deltaH_prime_div_k_L_S_L);
        if (curdist > mindist) continue;

        curdist += CIELAB::R_T(barCPrime, barhPrime, deltaC_prime_div_k_L_S_L, deltaH_prime_div_k_L_S_L);
      }

      if (curdist > mindist) continue;
      mindist = curdist;
      k = i;
    }
    nearestMap[offset] = k;
    return k;
  }

  short closestColorIndex(const std::vector<int32_t>& palette, int32_t c, int pos) override {  // PL:406-474
    const int plen = (int)palette.size();
    if (Color::alpha(c) <= alphaThreshold) return nearestColorIndex(palette, c, pos);

    const int32_t offset = !isNano ? c : getColorIndex(c, hasSemiTransparency, m_transparentPixelIndex >= 0);
    std::array<int32_t, 4> closest;
    auto it = closestMap.find(c);
    if (it == closestMap.end()) {
      closest = {0, 0, INT32_MAX, INT32_MAX};
      for (short k = 0; k < plen; ++k) {
        int32_t c2 = palette[k];
        double err = PR * (1 - ratio) * sqr(Color::red(c2) - Color::red(c));
        if (err >= closest[3]) continue;
        err += PG * (1 - ratio) * sqr(Color::green(c2) - Color::green(c));
        if (err >= closest[3]) continue;
        err += PB * (1 - ratio) * sqr(Color::blue(c2) - Color::blue(c));
        if (err >= closest[3]) continue;
        if (hasSemiTransparency) err += PA * sqr(Color::alpha(c2) - Color::alpha(c));

        for (int i = 0; i < 3; ++i) {
          err += ratio * sqr(coeffs[i][0] * (Color::red(c2) - Color::red(c)));
          if (err >= closest[3]) break;
          err += ratio * sqr(coeffs[i][1] * (Color::green(c2) - Color::green(c)));
          if (err >= closest[3]) break;
          err += ratio * sqr(coeffs[i][2] * (Color::blue(c2) - Color::blue(c)));
          if (err >= closest[3]) break;
        }

        if (err < closest[2]) {
          closest[1] = closest[0];
          closest[3] = closest[2];
          closest[0] = k;
          closest[2] = j2i(err);
        } else if (err < closest[3]) {
          closest[1] = k;
          closest[3] = j2i(err);
        }
      }
      if (closest[3] == INT32_MAX) closest[1] = closest[0];
      closestMap[offset] = closest;
    } else
      closest = it->second;

    int idx = 1;
    if (closest[2] == 0) idx = 0;
    else {
      ++trace.rng_draws;
      if (trace.keep_draws) trace.draw_bidx.push_back(pos);
      if ((random.nextInt(32767) % iadd(closest[3], closest[2])) <= closest[3]) idx = 0;
    }

    int MAX_ERR = plen;
    if (closest[idx + 2] >= MAX_ERR || closest[idx] == 0 || Color::alpha(palette[closest[idx]]) < Color::alpha(c)) return nearestColorIndex(palette, c, pos);
    return (short)closest[idx];
  }

  struct LabDitherable : Ditherable {  // PL:476-490
    PnnLABQuantizer& q;
    explicit LabDitherable(PnnLABQuantizer& q_) : q(q_) {}
    int getColorIndex(int32_t c) override { return ::getColorIndex(c, q.hasSemiTransparency, q.m_transparentPixelIndex >= 0); }
    short nearestColorIndex(const std::vector<int32_t>& palette, int32_t c, int pos) override {
      if (palette.size() <= 4) return q.nearestColorIndex(palette, c, pos);
      return q.closestColorIndex(palette, c, pos);
    }
  };

  std::vector<int32_t> ditherImage(const std::vector<int32_t>& cPixels, std::vector<int32_t>& palette, int width, int height, bool dither) override {  // PL:492-522
    LabDitherable ditherable(*this);
    random.setSeed(rngSeed);
    if (hasSemiTransparency) weight *= -1;

    if (dither && !hasSaliencies && (palette.size() <= 256 || weight > .99)) {
      saliencies.assign(pixels.size(), 0.f);
      hasSaliencies = true;
      float saliencyBase = .1f;
      for (size_t i = 0; i < pixels.size(); ++i) {
        const Lab& lab1 = getLab(pixels[i]);
        saliencies[i] = saliencyBase + (1 - saliencyBase) * lab1.L / 100.f * lab1.alpha / 255.f;
      }
    }
    std::vector<int32_t> qPixels(cPixels.size(), 0);
    {
      GilbertCurve gc(width, height, cPixels, palette, qPixels, ditherable, hasSaliencies ? &saliencies : nullptr, weight, dither);
      trace.gp = gc.params();
      gc.run();
      trace.gweights = gc.getWeights();
    }
    if (!dither && palette.size() > 32) {
      double delta = sqr((double)palette.size()) / pixelMap.size();
      float weight = delta > 0.023 ? 1.0f : (float)(37.013 * delta + 0.906);
      trace.bn_weight = weight;
      trace.pixelMapSize = (int64_t)pixelMap.size();
      BlueNoise::dither(width, height, cPixels, palette, ditherable, qPixels, weight);
    }
    if (hasSaliencies) trace.saliencies = saliencies;
    closestMap.clear();
    nearestMap.clear();
    pixelMap.clear();
    return qPixels;
  }

 public:
  PnnLABQuantizer(const uint32_t* argb, int w, int h) : PnnQuantizer(argb, w, h) {}
};

}  // namespace

// ---------------------------------------------------------------------------------------------
// C entry points for the test harness (ctypes)
// ---------------------------------------------------------------------------------------------
struct nqo_handle {
  Trace trace;
  std::vector<int32_t> out, palette;
  std::string error;
};

extern "C" {

nqo_handle* nqo_create() { return new nqo_handle(); }
void nqo_destroy(nqo_handle* h) { delete h; }
const char* nqo_error(nqo_handle* h) { return h->error.c_str(); }

// kind: 0 = PnnQuantizer, 1 = PnnLABQuantizer. math_mode: 0 shared kernels, 1 libm.
int nqo_convert(nqo_handle* h, int kind, const uint32_t* argb, int w, int hgt, int nMaxColors, int dither, uint64_t seed, int math_mode, uint32_t* out, uint32_t* palette, int* palette_len) {
  try {
    M.mode = math_mode;
    std::vector<int32_t> q;
    if (kind == 0) {
      PnnQuantizer pq(argb, w, hgt);
      pq.rngSeed = seed;
      q = pq.convert(nMaxColors, dither != 0);
      h->trace = pq.trace; h->palette = pq.palette_out;
    } else {
      PnnLABQuantizer pq(argb, w, hgt);
      pq.rngSeed = seed;
      q = pq.convert(nMaxColors, dither != 0);
      h->trace = pq.trace; h->palette = pq.palette_out;
    }
    h->out = q;
    if (out) memcpy(out, q.data(), q.size() * 4);
    if (palette) memcpy(palette, h->palette.data(), h->palette.size() * 4);
    if (palette_len) *palette_len = (int)h->palette.size();
    return 0;
  } catch (const std::exception& e) {
    h->error = e.what();
    return -1;
  }
}

// trace accessors ---------------------------------------------------------------------------
struct nqo_scalars {
  int hasSemiTransparency, transparentPixelIndex, maxbins, quan_rt, texicab, isNano;
  int transparentColor;
  int margin, thresold, DITHER_MAX, ditherMax, sortedByYDiff, hasAlpha;
  float beta, bn_weight;
  double weight, weight_final, ratio_init, ratio_merge, PR, PG, PB, PA, gweight;
  long long rng_draws, pixelMapSize, n_merges, n_saliencies, n_gweights, n_bins, n_init;
  long long n_rescans, n_heap_pops;
};
void nqo_get_scalars(nqo_handle* h, nqo_scalars* s) {
  const Trace& t = h->trace;
  s->hasSemiTransparency = t.hasSemiTransparency; s->transparentPixelIndex = t.transparentPixelIndex;
  s->maxbins = t.maxbins; s->quan_rt = t.quan_rt; s->texicab = t.texicab; s->isNano = t.isNano;
  s->transparentColor = t.transparentColor;
  s->margin = t.gp.margin; s->thresold = t.gp.thresold; s->DITHER_MAX = t.gp.DITHER_MAX; s->ditherMax = t.gp.ditherMax;
  s->sortedByYDiff = t.gp.sortedByYDiff; s->hasAlpha = t.gp.hasAlpha; s->beta = t.gp.beta; s->bn_weight = t.bn_weight;
  s->weight = t.weight; s->weight_final = t.weight_final; s->ratio_init = t.ratio_init; s->ratio_merge = t.ratio_merge;
  s->PR = t.PR; s->PG = t.PG; s->PB = t.PB; s->PA = t.PA; s->gweight = t.gp.weight;
  s->rng_draws = t.rng_draws; s->pixelMapSize = t.pixelMapSize; s->n_merges = (long long)t.merges.size() / 2;
  s->n_saliencies = (long long)t.saliencies.size(); s->n_gweights = (long long)t.gweights.size();
  s->n_bins = (long long)t.bins.size() / 5; s->n_init = (long long)t.init_err.size();
  s->n_rescans = t.n_rescans; s->n_heap_pops = t.n_heap_pops;
}
void nqo_get_bins(nqo_handle* h, double* bins5) { memcpy(bins5, h->trace.bins.data(), h->trace.bins.size() * 8); }
void nqo_get_init_nn(nqo_handle* h, float* err, int* nn) {
  memcpy(err, h->trace.init_err.data(), h->trace.init_err.size() * 4);
  memcpy(nn, h->trace.init_nn.data(), h->trace.init_nn.size() * 4);
}
void nqo_get_merges(nqo_handle* h, int* pairs) { memcpy(pairs, h->trace.merges.data(), h->trace.merges.size() * 4); }
void nqo_get_saliencies(nqo_handle* h, float* s) { memcpy(s, h->trace.saliencies.data(), h->trace.saliencies.size() * 4); }
void nqo_get_gweights(nqo_handle* h, float* s) { memcpy(s, h->trace.gweights.data(), h->trace.gweights.size() * 4); }

// unit-level helpers for known-answer tests -----------------------------------------------------
void nqo_gilbert_order(int w, int hgt, uint32_t* out) {
  OrderOnly o; o.width = w; o.out.reserve((size_t)w * hgt);
  if (w >= hgt) o.gen(0, 0, w, 0, 0, hgt); else o.gen(0, 0, 0, hgt, w, 0);
  memcpy(out, o.out.data(), o.out.size() * 4);
}
namespace {
struct NullDitherable : Ditherable {
  int getColorIndex(int32_t) override { return 0; }
  short nearestColorIndex(const std::vector<int32_t>&, int32_t, int) override { return 0; }
};
}
// GilbertCurve constructor constants for (palette length, signed weight, saliencies present)
void nqo_gilbert_params(int palette_len, double weight, int has_saliencies, int math_mode, int* margin, int* thresold, int* DITHER_MAX, int* ditherMax, int* sorted, float* beta) {
  M.mode = math_mode;
  std::vector<int32_t> px(1, 0), pal(palette_len, 0), q(1, 0);
  std::vector<float> sal(1, 0.5f);
  NullDitherable d;
  GilbertCurve gc(1, 1, px, pal, q, d, has_saliencies ? &sal : nullptr, weight, true);
  GilbertParams p = gc.params();
  *margin = p.margin; *thresold = p.thresold; *DITHER_MAX = p.DITHER_MAX; *ditherMax = p.ditherMax; *sorted = p.sortedByYDiff; *beta = p.beta;
}
void nqo_init_weights(int size, int math_mode, float* out) {
  M.mode = math_mode;
  std::vector<int32_t> px(1, 0), pal(256, 0), q(1, 0);
  NullDitherable d;
  GilbertCurve gc(1, 1, px, pal, q, d, nullptr, 0.001, true);
  gc.initWeightsPublic(size);
  memcpy(out, gc.getWeights().data(), size * 4);
}
void nqo_rgb2lab(uint32_t c, int math_mode, float* out4) {
  M.mode = math_mode;
  Lab l = CIELAB::RGB2LAB((int32_t)c);
  out4[0] = l.alpha; out4[1] = l.L; out4[2] = l.A; out4[3] = l.B;
}
uint32_t nqo_lab2rgb(float alpha, float L, float A, float B, int math_mode) {
  M.mode = math_mode;
  Lab l; l.alpha = alpha; l.L = L; l.A = A; l.B = B;
  return (uint32_t)CIELAB::LAB2RGB(l);
}
// full CIEDE2000 pieces for a pair (CL:91-194), out = {L', C', H', R_T}
void nqo_ciede_parts(const float* lab1, const float* lab2, int math_mode, float* out4) {
  M.mode = math_mode;
  Lab a, b;
  a.L = lab1[0]; a.A = lab1[1]; a.B = lab1[2];
  b.L = lab2[0]; b.A = lab2[1]; b.B = lab2[2];
  double a1 = 0, a2 = 0, c1 = 0, c2 = 0, bc = 0, bh = 0;
  out4[0] = CIELAB::L_prime_div_k_L_S_L(a, b);
  out4[1] = CIELAB::C_prime_div_k_L_S_L(a, b, a1, a2, c1, c2);
  out4[2] = CIELAB::H_prime_div_k_L_S_L(a, b, a1, a2, c1, c2, bc, bh);
  out4[3] = CIELAB::R_T(bc, bh, out4[1], out4[2]);
}
// n pairs: lab1/lab2 hold n x (L, A, B), out n x 4 (L', C', H', R_T terms)
void nqo_ciede_parts_batch(const float* lab1, const float* lab2, int n, int math_mode, float* out) {
  for (int i = 0; i < n; ++i) nqo_ciede_parts(lab1 + 3 * (size_t)i, lab2 + 3 * (size_t)i, math_mode, out + 4 * (size_t)i);
}
int nqo_java_random_next_int(uint64_t seed, int bound, int n, int* out) {
  JRandom r(seed);
  for (int i = 0; i < n; ++i) out[i] = r.nextInt(bound);
  return 0;
}
int nqo_hashmap_order(const int* keys, int n, int* out) {
  std::vector<int32_t> k(keys, keys + n);
  std::vector<int32_t> o = javaHashMapKeyOrder(k);
  memcpy(out, o.data(), o.size() * 4);
  return (int)o.size();
}
double nqo_math(int fn, double x, double y, int math_mode) {
  M.mode = math_mode;
  switch (fn) {
    case 0: return M.pow(x, y);
    case 1: return M.exp(x);
    case 2: return M.tanh(x);
    case 3: return M.cbrt(x);
    case 4: return M.atan2(x, y);
    case 5: return M.sin(x);
    case 6: return M.cos(x);
    default: return 0;
  }
}
double nqo_y_diff(uint32_t c1, uint32_t c2, int math_mode) { M.mode = math_mode; return CIELAB::Y_Diff((int32_t)c1, (int32_t)c2); }

}  // extern "C"
