// nq_pnn.cuh -- pairwise-nearest-neighbour clustering of the compacted bins.
// Reference: find_nn (PQ:57-116, PL:44-115), heap build (PQ:195-207, PL:245-257), merge loop
// (PQ:210-255, PL:267-312), palette fill (PQ:258-264, PL:315-324).
//
// What must be preserved for the merge sequence (and therefore the palette) to be identical:
//  * find_nn is an ORDERED scan over the surviving bins after idx: whether candidate i is taken
//    depends on the running err left by earlier candidates. RGB: a candidate that passes the four
//    `continue` tests is always taken, with err := the first partial sum of the YUV loop that
//    reaches err (the `break` falls through, PQ:97-112) -- err can grow. LAB: err := full cost,
//    early exits use >= for the first tests and > later, and R_T may be negative (PL:57-108).
//    Candidates are pruned only by tests the reference itself would fail them on, evaluated against an
//    upper bound of the running err (block summaries, per-candidate bounds, exact prefixes), and the
//    survivors are resolved in list order with ballot rounds (one round per ACCEPTED candidate).
//  * the binary heap code, including its tie behaviour, is replayed verbatim by one thread; heap
//    slots carry a copy of the bin's err (a bin's err only changes while it sits at heap[1]).
//  * forward links only ever skip deleted bins, so "list order" == ascending index among live bins;
//    a periodically compacted live list replaces pointer chasing.
#pragma once
#include "nq_types.h"
#include "nq_color.h"
#include "nq_hist.cuh"
#include "nq_fastmath.cuh"

namespace nq {

__device__ const float c_coeffs[3][3] = {{0.299f, 0.587f, 0.114f}, {-0.14713f, -0.28886f, 0.436f}, {0.615f, -0.51499f, -0.10001f}};  // PQ:26-30

// -------------------------------------------------------------------------------------------------
// RGB candidate arithmetic (PQ:73-112)
// -------------------------------------------------------------------------------------------------
struct RgbProbe {
  float n1;
  double wa, wr, wg, wb;
  double PR, PG, PB, PA, ratio;
  int start;
  bool semi;
};

__device__ __forceinline__ RgbProbe rgb_probe(const NqImage& I, const NqSlot& S, int idx) {
  RgbProbe P;
  P.n1 = S.bCnt[idx];
  P.wa = S.bAc[idx]; P.wr = S.bC1[idx]; P.wg = S.bC2[idx]; P.wb = S.bC3[idx];
  P.PR = I.PR; P.PG = I.PG; P.PB = I.PB; P.PA = I.PA; P.ratio = I.ratio;
  P.semi = I.hasSemi != 0;
  P.start = 0;
  if (g_blueNoise[idx & 4095] > 0) P.start = (I.PG < (double)0.587f) ? 3 : 1;   // PQ:69-71
  return P;
}

struct RgbCand { double nerr2, q0, dr, dg, db; };

// gate: candidate is taken iff nerr2 < err and q0 < err (the partial sums before q0 are <= q0)
__device__ __forceinline__ double rgb_gate(const RgbProbe& P, const NqSlot& S, int i, RgbCand* c) {
  double n2 = (double)S.bCnt[i];
  double nerr2 = ((double)P.n1 * n2) / ((double)P.n1 + n2);
  double nerr = 0.0;
  if (P.semi) { double d = S.bAc[i] - P.wa; nerr += nerr2 * P.PA * (d * d); }
  double dr = S.bC1[i] - P.wr, dg = S.bC2[i] - P.wg, db = S.bC3[i] - P.wb;
  nerr += nerr2 * (1 - P.ratio) * P.PR * (dr * dr);
  nerr += nerr2 * (1 - P.ratio) * P.PG * (dg * dg);
  nerr += nerr2 * (1 - P.ratio) * P.PB * (db * db);
  c->nerr2 = nerr2; c->q0 = nerr; c->dr = dr; c->dg = dg; c->db = db;
  return nerr2 > nerr ? nerr2 : nerr;
}
// new err of a taken candidate (PQ:97-112)
__device__ __forceinline__ double rgb_take(const RgbProbe& P, const RgbCand& c, double err) {
  double nerr = c.q0;
  for (int j = P.start; j < 3; ++j) {
    double t = (double)c_coeffs[j][0] * c.dr;
    nerr += c.nerr2 * P.ratio * (t * t);
    if (nerr >= err) break;
    t = (double)c_coeffs[j][1] * c.dg;
    nerr += c.nerr2 * P.ratio * (t * t);
    if (nerr >= err) break;
    t = (double)c_coeffs[j][2] * c.db;
    nerr += c.nerr2 * P.ratio * (t * t);
    if (nerr >= err) break;
  }
  return nerr;
}

// -------------------------------------------------------------------------------------------------
// LAB candidate arithmetic (PL:54-112). err only ever decreases, so a candidate that fails a test
// against the err at the start of a chunk can be dropped for good. A survivor carries
// gs (must be < err), gw (must be <= err) and f (the new err).
// -------------------------------------------------------------------------------------------------
// upper bound of sqrt(A^2 + B^2) as a float
__device__ __forceinline__ float chroma_ub(float A, float B) {
  const float x = (A * A) + (B * B);
  // x * rsqrt(x) with the hardware estimate (relative error < 2^-22) and a margin: an upper bound is all that is needed
  return x > 1e-30f ? (x * __frsqrt_rn(x)) * 1.00001f : 1e-15f;
}

struct LabProbe {
  float n1, a1, L1, A1, B1, C1;   // C1: upper bound of the chroma sqrt(A1^2 + B1^2)
  float ratioLo;                  // ratio rounded down to float (lower bounds only)
  double ratio, exp175;
  bool semi, texicab;
};
__device__ __forceinline__ LabProbe lab_probe(const NqImage& I, const NqSlot& S, int idx, double ratio) {
  LabProbe P;
  P.n1 = S.bCnt[idx];
  P.a1 = S.fAc[idx]; P.L1 = S.fC1[idx]; P.A1 = S.fC2[idx]; P.B1 = S.fC3[idx];
  P.C1 = chroma_ub(P.A1, P.B1);
  P.ratio = ratio;
  P.ratioLo = __double2float_rd(ratio);
  P.semi = I.hasSemi != 0;
  P.exp175 = P.semi ? nqm::nq_exp(1.75) : 1.0;
  P.texicab = I.texicab != 0;
  return P;
}
struct LabCand { double gs, gw, f; };

// Candidate bins as position-indexed records plus one summary per 32 positions. For the
// initial sweep the position is the bin index; inside the merge loop it is the position in the
// compacted list of surviving bins (cnt < 0 marks a bin that died since the last compaction).
struct LabView {
  const float4* q;                      // {cnt, L, A, B} per position: one 16-byte load per candidate
  const float* al;                      // alpha per position (read only for semi-transparent images)
  const float4* bs;                     // per block of 32 positions, two float4: {min count, min L, max L, max chroma},
                                        // {min A, max A, min B, max B} (conservative: never tightened between compactions)
  int n;
};

// Lower bound of the cost of EVERY candidate of block `blk`, from the summary alone:
//   cost >= ratio * nerr2 * L'^2,  nerr2 = n1 n2 / (n1 + n2) increasing in n2,  |L'| = |dL| / S_L, S_L <= 1.7472
// (CL:91-98: S_L = 1 + .015 d^2 / sqrt(20 + d^2), |d| <= 50). The factors (1 - 1e-6) and (1 - 1e-5) cover
// the float roundings of the reference's own evaluation. A block may be skipped when even this bound
// fails the reference's tests against an upper bound U of the running err: nerr2 >= U (PL:57) or the
// prefix after the L' term > U (PL:88-90; every earlier term is >= 0).
__device__ float g_rtFac[256];   // see below (k_init_rtfac)
__device__ __forceinline__ float chroma_ub(float A, float B);
// s0 = {min count, min L, max L, max chroma}, s1 = {min A, max A, min B, max B} of the block. The bound is the
// per-candidate one of lab_cheap_keep_q with every quantity replaced by its most favourable value in the block.
__device__ __forceinline__ bool lab_block_skip_v(const LabProbe& P, const float4 s0, const float4 s1, double U) {
  const float cmin = s0.x;
  if (!(cmin >= 0.f)) return true;                        // block holds no live bin
  // float arithmetic throughout: a dozen roundings (6e-8 each) against the 1e-4 deflations; Uup >= U
  const float Uup = __double2float_ru(U);
  const float nerr2 = ((P.n1 * cmin) / (P.n1 + cmin)) * 0.9999f;
  if (nerr2 >= Uup) return true;
  const float dl = fmaxf(0.f, fmaxf(s0.y - P.L1, P.L1 - s0.z));
  const float da = fmaxf(0.f, fmaxf(s1.x - P.A1, P.A1 - s1.y));
  const float db = fmaxf(0.f, fmaxf(s1.z - P.B1, P.B1 - s1.w));
  const float cb = (0.75f * (P.C1 + s0.w)) * 1.00001f;
  const float sc = (1.f + (0.045f * cb)) * 1.00001f;
  const float rf = g_rtFac[min(255, (int)cb)];
  const float d2 = fmaxf(0.f, (((da * da) + (db * db)) * 0.9999f) - 1e-4f);
  const float t = dl * 0.57234f;                           // 1 / 1.7472 rounded down
  const float q = (t * t) + __fdividef(rf * d2, (sc * sc) * 1.00001f) * 0.99999f;
  const float lb = (P.ratioLo * nerr2) * q * 0.9999f;
  return lb > Uup;
}
__device__ __forceinline__ bool lab_block_skip(const LabProbe& P, const LabView& V, int blk, double U) {
  return lab_block_skip_v(P, V.bs[2 * blk], V.bs[2 * blk + 1], U);
}

// 1 - |R_T|max / 2 for barCPrime in [k, k + 1): R_T = -sin(2 dTheta) R_C with |sin(2 dTheta)| <= sin(60 deg) and
// R_C = 2 sqrt(c^7 / (c^7 + 25^7)) increasing in c (CL:187-194), so the table decreases.
__global__ void k_init_rtfac() {
  const int k = threadIdx.x;
  double f = 1.0 - 0.86603 * 1.000001;                    // barCPrime >= 255: R_C < 2
  if (k < 255) {
    const double c = (double)(k + 1) / 25.0, c2 = c * c, c7 = c2 * c2 * c2 * c;
    f = 1.0 - 0.5 * 0.86603 * (2.0 * nqm::sqrt_(c7 / (c7 + 1.0))) * 1.000001;
  }
  g_rtFac[k] = (float)f * 0.999999f;
}

// Per-candidate lower bound of the cost, from float arithmetic only:
//   L'^2 + C'^2 + H'^2 + R_T C' H' >= (dL / S_L)^2 + (1 - |R_T|/2) (C'^2 + H'^2),
//   (S_C C')^2 + (S_H H')^2 = dC'^2 + dH'^2 = (a1' - a2')^2 + (b1 - b2)^2 >= da^2 + db^2   (chord identity; a' = (1 + G) a),
//   S_H <= S_C = 1 + .045 barC', barC' <= .75 (C1 + C2)   (G <= .5).
// The slack terms cover the float roundings of the reference's own evaluation (the float difference of the two
// C' values is off by up to 1.3e-7 max(C')). Returns false only if the reference must reject i given err.
__device__ __forceinline__ bool lab_cheap_keep_q(const LabProbe& P, const float4 cq, double err);
__device__ __forceinline__ bool lab_cheap_keep(const LabProbe& P, const LabView& V, int i, double err) {
  return lab_cheap_keep_q(P, V.q[i], err);
}
__device__ __forceinline__ bool lab_cheap_keep_q(const LabProbe& P, const float4 cq, double err) {
  const float n2 = cq.x;
  if (!(n2 >= 0.f)) return false;
  const float nerr2 = (P.n1 * n2) / (P.n1 + n2);                  // the reference's own value and test (PL:56-57)
  if ((double)nerr2 >= err) return false;
  // the bound itself in float: a dozen roundings (6e-8 each) against the 1e-4 deflations; errUp >= err
  const float errUp = __double2float_ru(err);
  const float dl = cq.y - P.L1, da = cq.z - P.A1, db = cq.w - P.B1;
  const float cb = (0.75f * (P.C1 + chroma_ub(cq.z, cq.w))) * 1.00001f;
  const float sc = (1.f + (0.045f * cb)) * 1.00001f;
  const float rf = g_rtFac[min(255, (int)cb)];
  const float d2 = fmaxf(0.f, (((da * da) + (db * db)) * 0.9999f) - 1e-4f);
  const float tl = dl * 0.57234f;                                  // 1 / 1.7472 rounded down
  const float q = (tl * tl) + __fdividef(rf * d2, (sc * sc) * 1.00001f) * 0.99999f;
  const float lb = (P.ratioLo * nerr2) * q * 0.9999f;
  return !(lb > errUp);
}

// find_nn's tests for candidate i against err (PL:54-108). With STOP_AFTER_C the evaluation ends after
// the C' term (a cheap screen: two more square roots and a pow(.,7), no trigonometry); it then returns
// true iff the candidate is still alive there.
template <bool STOP_AFTER_C>
__device__ __forceinline__ bool lab_eval_t(const LabProbe& P, const LabView& V, int i, double err, LabCand* c) {
  const float4 cq = V.q[i];
  const float n2 = cq.x;
  if (!(n2 >= 0.f)) return false;                         // dead since the last compaction
  double nerr2 = (double)((P.n1 * n2) / (P.n1 + n2));
  if (nerr2 >= err) return false;
  const float L2 = cq.y, A2 = cq.z, B2 = cq.w;
  double alphaDiff = 0;
  if (P.semi) { double d = (double)(V.al[i] - P.a1); alphaDiff = (d * d) / P.exp175; }
  double nerr = nerr2 * alphaDiff;
  if (nerr >= err) return false;
  double gs = nerr2;
  if (!P.texicab) {
    double d = (double)(L2 - P.L1);
    nerr += (1 - P.ratio) * nerr2 * (d * d);
    if (nerr >= err) return false;
    d = (double)(A2 - P.A1);
    nerr += (1 - P.ratio) * nerr2 * (d * d);
    if (nerr >= err) return false;
    gs = nerr > gs ? nerr : gs;
    d = (double)(B2 - P.B1);
    nerr += (1 - P.ratio) * nerr2 * (d * d);
  } else {
    nerr += (1 - P.ratio) * nerr2 * (double)fabsf(L2 - P.L1);
    if (nerr >= err) return false;
    gs = nerr > gs ? nerr : gs;
    double da = (double)(A2 - P.A1), db = (double)(B2 - P.B1);
    nerr += (1 - P.ratio) * nerr2 * nqm::sqrt_((da * da) + (db * db));
  }
  if (nerr > err) return false;

  float tL = ciede_L(P.L1, L2);
  nerr += P.ratio * nerr2 * ((double)tL * (double)tL);
  if (nerr > err) return false;

  CiedeC cc;
  float tC = ciede_C(P.A1, P.B1, A2, B2, &cc);
  nerr += P.ratio * nerr2 * ((double)tC * (double)tC);
  if (nerr > err) return false;
  if (STOP_AFTER_C) return true;

  float tH, tRT;
  if (!nqf::ciede_HRT_fast(P.B1, B2, cc, tC, &tH, &tRT)) {   // the filter could not decide both floats
    double barC, barh;
    tH = ciede_H(P.B1, B2, cc, &barC, &barh);
    tRT = ciede_RT(barC, barh, tC, tH);
  }
  nerr += P.ratio * nerr2 * ((double)tH * (double)tH);
  if (nerr > err) return false;
  double gw = nerr;

  nerr += P.ratio * nerr2 * (double)tRT;
  if (nerr > err) return false;
  c->gs = gs; c->gw = nerr > gw ? nerr : gw; c->f = nerr;
  return true;
}

// ordered acceptance among up to 32 evaluated candidates held one per lane, in lane order: candidate
// i is taken iff gs < err and gw <= err with the err left by the candidates before it
__device__ __forceinline__ void lab_accept_in_order(bool alive, const LabCand& c, int id, double& err, int& nn) {
  unsigned remaining = 0xffffffffu;
  for (;;) {
    unsigned m = __ballot_sync(0xffffffffu, alive && c.gs < err && c.gw <= err) & remaining;
    if (!m) break;
    int L = __ffs(m) - 1;
    err = __shfl_sync(0xffffffffu, c.f, L);
    nn = __shfl_sync(0xffffffffu, id, L);
    remaining = (L == 31) ? 0u : ~((2u << L) - 1u);
  }
}

// find_nn for one bin by ONE warp, streaming over the candidates at positions >= first in order.
// The first 32 candidates are evaluated unconditionally (err is still infinite; they are the bins
// with the nearest histogram keys, so err is tight afterwards). From then on whole blocks are dropped
// by their summary, the candidates of the remaining blocks are screened through the C' term, and the
// survivors queue up (in order) until 32 of them can be evaluated in full together.
__device__ void warp_find_nn_lab(const LabProbe& P, const LabView& V, int first, int* sBufA /*[64]*/, int* sBufB /*[64], this warp's*/, double* errOut, int* nnOut) {
  const unsigned lane = lane_id();
  double err = 1e100;
  int nn = -1, nA = 0, nB = 0;
  const int n = V.n;
  auto shift = [&](int* buf, int& cnt, int take) {
    const int rest = cnt - take;
    const int v = ((int)lane < rest) ? buf[take + lane] : 0;
    __syncwarp();
    if ((int)lane < rest) buf[lane] = v;
    cnt = rest;
    __syncwarp();
  };
  auto flushB = [&](int take) {               // full evaluation + ordered acceptance
    int i = -1;
    LabCand c;
    bool alive = false;
    if ((int)lane < take) { i = sBufB[lane]; alive = lab_eval_t<false>(P, V, i, err, &c); }
    lab_accept_in_order(alive, c, i, err, nn);
    shift(sBufB, nB, take);
  };
  auto pushB = [&](bool keep, int i) {
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (keep) sBufB[nB + __popc(m & ((1u << lane) - 1u))] = i;
    nB += __popc(m);
    __syncwarp();
    if (nB >= 32) flushB(32);
  };
  auto flushA = [&](int take) {               // screen through the C' term
    int i = -1;
    bool keep = false;
    LabCand dummy;
    if ((int)lane < take) { i = sBufA[lane]; keep = lab_eval_t<true>(P, V, i, err, &dummy); }
    shift(sBufA, nA, take);
    pushB(keep, i);
  };
  auto pushA = [&](bool keep, int i) {
    const unsigned m = __ballot_sync(0xffffffffu, keep);
    if (!m) return;                           // most blocks that survive their summary hold no survivor
    if (keep) sBufA[nA + __popc(m & ((1u << lane) - 1u))] = i;
    nA += __popc(m);
    __syncwarp();
    if (nA >= 32) flushA(32);
  };
  int pos = first;
  if (pos < n) {
    const int i = pos + (int)lane;
    pushB(i < n && V.q[i].x >= 0.f, i);
    if (nB) flushB(nB);
    pos += 32;
  }
  const int stop = first + 32;     // positions below were handled by the unconditional tile
  // the summaries of the next 32 blocks are loaded while the current ones are processed (they come from L2)
  const int nblk = (n + 31) >> 5;
  int blk0 = pos >> 5;
  const float4 none = make_float4(-1.f, 0.f, 0.f, 0.f);
  float4 n0 = none, n1 = none;
  if (blk0 + (int)lane < nblk) { n0 = V.bs[2 * (blk0 + lane)]; n1 = V.bs[2 * (blk0 + lane) + 1]; }
  for (; blk0 < nblk; blk0 += 32) {
    const float4 s0 = n0, s1 = n1;
    const int nb = blk0 + 32 + (int)lane;
    n0 = none;
    if (nb < nblk) { n0 = V.bs[2 * nb]; n1 = V.bs[2 * nb + 1]; }
    unsigned bm = __ballot_sync(0xffffffffu, !lab_block_skip_v(P, s0, s1, err));
    // records of the next live block are requested before the current one is tested
    const float4 dead = make_float4(-1.f, 0.f, 0.f, 0.f);
    int b = bm ? __ffs(bm) - 1 : -1;
    int i = ((blk0 + b) << 5) + (int)lane;
    float4 rec = (b >= 0 && i >= stop && i < n) ? V.q[i] : dead;
    while (b >= 0) {
      bm &= bm - 1;
      const int b2 = bm ? __ffs(bm) - 1 : -1;
      const int i2 = ((blk0 + b2) << 5) + (int)lane;
      const float4 rec2 = (b2 >= 0 && i2 >= stop && i2 < n) ? V.q[i2] : dead;
      pushA(lab_cheap_keep_q(P, rec, err), i);
      b = b2; i = i2; rec = rec2;
    }
  }
  if (nA) flushA(nA);
  if (nB) flushB(nB);
  *errOut = err;
  *nnOut = nn;
}

// summaries of blocks [0, ceil(n/32)) over position-indexed arrays; one thread per block
__device__ __forceinline__ void lab_block_summary(const float4* q, int n, int blk, float4* bs) {
  float cm = -1.f, lo = 1e30f, hi = -1e30f, ch = 0.f, alo = 1e30f, ahi = -1e30f, blo = 1e30f, bhi = -1e30f;
  const int p0 = blk << 5, p1 = min(n, p0 + 32);
  for (int p = p0; p < p1; ++p) {
    const float4 v = q[p];
    if (!(v.x >= 0.f)) continue;
    cm = cm < 0.f ? v.x : fminf(cm, v.x);
    lo = fminf(lo, v.y); hi = fmaxf(hi, v.y);
    alo = fminf(alo, v.z); ahi = fmaxf(ahi, v.z);
    blo = fminf(blo, v.w); bhi = fmaxf(bhi, v.w);
    ch = fmaxf(ch, chroma_ub(v.z, v.w));
  }
  bs[2 * blk] = make_float4(cm, lo, hi, ch);
  bs[2 * blk + 1] = make_float4(alo, ahi, blo, bhi);
}

// scratch carved out of the histogram sum planes (free once the bins are compacted)
struct LabScratch { float4* q; float* al; float4* bs; };
__device__ __forceinline__ LabScratch lab_scratch(const NqSlot& S) {
  float* f = reinterpret_cast<float*>(S.hSum);
  LabScratch X;
  X.q = reinterpret_cast<float4*>(f); X.al = f + 4 * NQ_NBINS;
  X.bs = reinterpret_cast<float4*>(f + 5 * NQ_NBINS);
  return X;
}

__global__ void __launch_bounds__(256) k_lab_blocks(const NqImage* imgs, const NqSlot* slots) {
  const int img = blockIdx.y;
  const NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2 || I.skipPnn) return;
  const NqSlot& S = slots[img];
  const LabScratch X = lab_scratch(S);
  const int n = I.maxbins, nblk = (n + 31) >> 5;
  // one warp per block of 32 bins: pack the records and reduce the summary
  const unsigned lane = lane_id();
  for (int blk = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); blk < nblk; blk += gridDim.x * (blockDim.x >> 5)) {
    const int b = (blk << 5) + (int)lane;
    if (b < n) { X.q[b] = make_float4(S.bCnt[b], S.fC1[b], S.fC2[b], S.fC3[b]); X.al[b] = S.fAc[b]; }
    __syncwarp();
    if (lane == 0) lab_block_summary(X.q, n, blk, X.bs);
  }
}


// -------------------------------------------------------------------------------------------------
// initial sweep: find_nn for every bin (PQ:196-197, PL:246-247). One warp per bin.
// -------------------------------------------------------------------------------------------------
// CIELAB: one warp per bin, streaming with block summaries (warp_find_nn_lab). Bins are dealt out
// interleaved so that every warp gets a mix of long (small idx) and short candidate lists.
__global__ void __launch_bounds__(256, 3) k_find_nn_lab(NqImage* imgs, const NqSlot* slots, int nimg) {
  __shared__ int sBufA[8][64], sBufB[8][64];
  const unsigned lane = lane_id();
  const int w = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  for (int img = 0; img < nimg; ++img) {
    NqImage& I = imgs[img];
    if (I.kind != NQ_KIND_LAB || I.nmax <= 2 || I.skipPnn) continue;
    const NqSlot& S = slots[img];
    const LabScratch X = lab_scratch(S);
    const int maxbins = I.maxbins;
    const LabView V{X.q, X.al, X.bs, maxbins};
    unsigned long long pairs = 0;
    for (int idx = blockIdx.x * wpb + w; idx < maxbins; idx += gridDim.x * wpb) {
      const LabProbe P = lab_probe(I, S, idx, I.ratio);
      double err;
      int nn;
      warp_find_nn_lab(P, V, idx + 1, sBufA[w], sBufB[w], &err, &nn);
      pairs += (unsigned long long)(maxbins - idx - 1);
      if (lane == 0) { S.bErr[idx] = (float)err; S.bNn[idx] = nn < 0 ? 0 : nn; }
    }
    if (lane == 0 && pairs) atomicAdd(&I.statPairs, pairs);
  }
}

// -------------------------------------------------------------------------------------------------
// merge loops: one persistent 128-thread CTA per image, several images per SM (k_merge_lab, k_merge_rgb).
// -------------------------------------------------------------------------------------------------

// The heap of bin ids keyed by err (PQ:195-236). A slot also carries a copy of the bin's err (a bin's err only
// changes while it sits at heap[1]) and of its nn (likewise), so the top can be validated with ONE round trip
// to global memory: tm/mtm of the bin and mtm of its nn are loaded together.
template <int HS>
struct HeapView {
  static_assert((HS & 1) == 0, "children l2, l2 + 1 must fall on the same side of the split");
  float* sErr; unsigned* sIdNn;       // shared part, slots [0, HS): err, id | nn << 16
  uint2* gH;                          // global spill for the deepest levels: {err bits, id | nn << 16} per slot, so the
                                      // two children of a node (slots 2l, 2l + 1) arrive with ONE 16-byte load
  __device__ __forceinline__ float err(int l) const { return l < HS ? sErr[l] : __uint_as_float(gH[l].x); }
  __device__ __forceinline__ unsigned idnn(int l) const { return l < HS ? sIdNn[l] : gH[l].y; }
  __device__ __forceinline__ int id(int l) const { return (int)(idnn(l) & 0xFFFFu); }
  __device__ __forceinline__ void set(int l, unsigned idnn_, float e) {
    if (l < HS) { sErr[l] = e; sIdNn[l] = idnn_; } else gH[l] = make_uint2(__float_as_uint(e), idnn_);
  }
  // "push slot down" (PQ:228-236): sift (b1, e1) down from the root of a heap with heapN entries
  __device__ __forceinline__ void sift_down(unsigned idnn1, float e1, int heapN) {
    int l = 1, l2;
    for (; (l2 = l + l) <= heapN; l = l2) {
      float ea, eb = 0.f;
      unsigned ia, ib = 0u;
      if (l2 < HS) {
        ea = sErr[l2]; ia = sIdNn[l2];
        if (l2 < heapN) { eb = sErr[l2 + 1]; ib = sIdNn[l2 + 1]; }
      } else {
        const uint4 ch = *reinterpret_cast<const uint4*>(&gH[l2]);   // slot l2 + 1 exists in the allocation even past heapN
        ea = __uint_as_float(ch.x); ia = ch.y; eb = __uint_as_float(ch.z); ib = ch.w;
      }
      if (l2 < heapN && ea > eb) { ++l2; ea = eb; ia = ib; }
      if (e1 <= ea) break;
      set(l, ia, ea);
    }
    set(l, idnn1, e1);
  }
};
__device__ __forceinline__ unsigned pack_idnn(int id, int nn) { return (unsigned)id | ((unsigned)nn << 16); }

// -------------------------------------------------------------------------------------------------
// CIELAB merge loop. A full find_nn test costs a few thousand double-precision instructions
// (CIEDE2000 with correctly rounded atan2/sin/cos/exp/pow), so the kernel is organised around
// evaluating as FEW candidates in full as the reference's own early exits allow:
//   1. warp 0 evaluates the first 32 surviving bins after b1 in full (err is infinite there) and
//      resolves them in order -> err, the exact running error after 32 candidates;
//   2. all threads test the 32-bin block summaries of the rest against err (lab_block_skip);
//   3. the bins of the remaining blocks are screened through the C' term (lab_eval_t<true>);
//   4. the screened bins are evaluated in full, packed one per thread, and resolved in list order.
// Every test is the reference's test against an err that is >= the err the sequential scan would hold
// at that candidate, so nothing the reference would take is dropped, and step 4 replays its decisions.
//
// Rescans run in ROUNDS of up to NQ_LAB_ROUND bins. Between two merges the reference pops the heap top,
// rescans it if it is stale and pushes it down, until the top is valid (PL:271-293). A rescan of bin b is a
// pure function of b and the set of live bins, and it changes the validity of no other bin, so the bins it
// rescans before the next merge are the stale entries in the order the heap pops them, up to the first valid
// one. A round guesses them from the top levels of the heap (stale entries in ascending (err, slot), deleted
// ones skipped, none behind a valid one) and rescans them together: step 1 takes one warp per bin, and steps
// 2-4 run over all of them at once, batch g holding the g-th 32 live blocks of every bin, so that each bin is
// pruned on the schedule of a rescan of its own. Thread 0 then replays the reference's top loop verbatim: a stale top with a result from the current
// round takes it, one without starts the next round, and a merge discards the unused results. A wrong guess
// costs work, never a different result.
// 128 threads per CTA: several images share an SM and fill each other's serial gaps. The chain of one image is bound by
// latency, so more images per SM buy throughput, and each image's chain gets longer as they share the SM. Two instances:
// CTAS = 4 (128 registers, 44 KB of heap) has the shorter chain; CTAS = 8 (64 registers, a few spills at round boundaries,
// 16 KB of heap, one more heap level in global memory) runs twice the images at once. The host launches the first when the
// images in flight fit one wave of it and the second otherwise (lab_merge_ctas in nq_api.cu).
// -------------------------------------------------------------------------------------------------
#define NQ_LAB_THREADS 128
// heap slots kept in shared memory by the instance for `ctas` CTAs per SM (8 bytes each)
__host__ __device__ constexpr int lab_heap_smem(int ctas) { return ctas >= 8 ? 2048 : 5632; }
#define NQ_LAB_ROUND 4          // bins rescanned together in one round (8 would need 256-entry batches: more shared memory)

__device__ __forceinline__ int block_excl_scan_128(int v, int* total, int* sScan /*[8]*/) {
  const unsigned lane = lane_id(), w = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= (unsigned)o) x += y;
  }
  if (lane == 31) sScan[w] = x;
  __syncthreads();
  int base = 0, tot = 0;
#pragma unroll
  for (int k = 0; k < NQ_LAB_THREADS / 32; ++k) { const int c = sScan[k]; if (k < (int)w) base += c; tot += c; }
  *total = tot;
  __syncthreads();
  return base + x - v;
}

// rebuild the ascending list of live bins, their compacted records and the block summaries. Each warp
// owns a contiguous range of bins and walks it 32 at a time (coalesced), ranking survivors by ballot.
__device__ __forceinline__ int rebuild_live_lab(const NqSlot& S, const LabScratch& X, int maxbins, int* live, int* posOf, int* sScan) {
  const int t = threadIdx.x;
  const unsigned lane = lane_id(), w = t >> 5;
  const int W = NQ_LAB_THREADS / 32;
  const int per = (((maxbins + W - 1) / W) + 31) & ~31;
  const int b0 = min(maxbins, (int)w * per), b1 = min(maxbins, b0 + per);
  int c = 0;
  for (int b = b0 + (int)lane; b < b1; b += 32) c += S.bMtm[b] != NQ_DELETED;
  int total, j = block_excl_scan_128(c, &total, sScan);
  j = __shfl_sync(0xffffffffu, j, 0);          // this warp's first output slot
  for (int base = b0; base < b1; base += 32) {
    const int b = base + (int)lane;
    const bool alive = b < b1 && S.bMtm[b] != NQ_DELETED;
    const unsigned m = __ballot_sync(0xffffffffu, alive);
    if (alive) {
      const int p = j + __popc(m & ((1u << lane) - 1u));
      live[p] = b; posOf[b] = p;
      X.q[p] = make_float4(S.bCnt[b], S.fC1[b], S.fC2[b], S.fC3[b]);
      X.al[p] = S.fAc[b];
    }
    j += __popc(m);
  }
  __syncthreads();
  const int nblk = (total + 31) >> 5;
  for (int blk = t; blk < nblk; blk += NQ_LAB_THREADS) lab_block_summary(X.q, total, blk, X.bs);
  __syncthreads();
  return total;
}

template <int CTAS>
__global__ void __launch_bounds__(NQ_LAB_THREADS, CTAS) k_merge_lab(NqImage* imgs, const NqSlot* slots, int* liveBuf, int* posBuf, int logMerges) {
  constexpr int R = NQ_LAB_ROUND, HS = lab_heap_smem(CTAS);
  static_assert(R >= 1 && 32 * R <= NQ_LAB_THREADS, "a batch holds 32 blocks of each bin of the round, one per thread");
  extern __shared__ unsigned char smemRaw[];
  float* sErr = reinterpret_cast<float*>(smemRaw);
  unsigned* sId = reinterpret_cast<unsigned*>(smemRaw + (size_t)HS * 4);
  __shared__ int sScan[8];
  __shared__ unsigned sBits[R][64];          // live blocks of each bin of the round, one bit per block
  __shared__ unsigned short sPre[R][65];     // live blocks of the bin before each word of sBits; [64]: all of them
  __shared__ unsigned short sBat[NQ_LAB_THREADS];   // entries of the current batch: bin of the round << 11 | block, bin-major
  __shared__ unsigned sMaskA[NQ_LAB_THREADS];       // bins that passed the cheap bound, per entry of the batch
  __shared__ unsigned sMaskB[NQ_LAB_THREADS];       // ... of those, the ones that passed the screen, per 32 of them
  __shared__ int sOffA[NQ_LAB_THREADS + 1], sOffB[NQ_LAB_THREADS];
  __shared__ double sGs[NQ_LAB_THREADS], sGw[NQ_LAB_THREADS], sF[NQ_LAB_THREADS];
  __shared__ int sPos[NQ_LAB_THREADS];       // fully evaluated candidate: bin of the round << 17 | survived << 16 | position
  // the round: bin ids, probes, running err and nn of each (nn: position in the live list while the round runs, bin id
  // after it), first candidate position
  __shared__ LabProbe sProbe[R];
  __shared__ double sErrR[R];
  __shared__ int sBinR[R], sNnR[R], sFirstR[R];
  __shared__ int sAction, sB1, sHeapN, sIter, sNRound;

  const int img = blockIdx.x;
  NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2 || I.skipPnn) return;
  const NqSlot& S = slots[img];
  const LabScratch X = lab_scratch(S);
  const int t = threadIdx.x;
  const unsigned lane = lane_id(), w = t >> 5;
  const int W = NQ_LAB_THREADS / 32;
  const int maxbins = I.maxbins, extbins = I.extbins;
  int* live = liveBuf + (size_t)img * NQ_NBINS;
  int* posOf = posBuf + (size_t)img * NQ_NBINS;
  HeapView<HS> H{sErr, sId, S.heap};
  const float4 dead = make_float4(-1.f, 0.f, 0.f, 0.f);

  // ---- heap build: sequential pushes in bin order (PL:246-257), replayed by warp 0
  if (w == 0) {
    int heapN = 0;
    for (int base = 0; base < maxbins; base += 32) {
      float e = (base + (int)lane < maxbins) ? S.bErr[base + lane] : 0.f;
      const int nnv = (base + (int)lane < maxbins) ? S.bNn[base + lane] : 0;
      const int cnt = min(32, maxbins - base);
      for (int j = 0; j < cnt; ++j) {
        const float err = __shfl_sync(0xffffffffu, e, j);
        const int nnj = __shfl_sync(0xffffffffu, nnv, j);
        int l = ++heapN, l2;
        for (; l > 1; l = l2) {
          l2 = l >> 1;
          float pe = H.err(l2);
          if (pe <= err) break;
          unsigned pid = H.idnn(l2);
          if (lane == 0) H.set(l, pid, pe);
        }
        if (lane == 0) H.set(l, pack_idnn(base + j, nnj), err);
        __syncwarp();
      }
    }
    if (lane == 0) { sHeapN = heapN; sIter = 0; sNRound = 0; }
  }
  __syncthreads();
  int liveLen = rebuild_live_lab(S, X, maxbins, live, posOf, sScan);
  int liveAtRebuild = liveLen, iterAtRebuild = 0;
  unsigned long long rescans = 0, pairs = 0, fulls = 0, liveBlocks = 0, screened = 0, rounds = 0, discarded = 0;
  unsigned pops = 0;
  unsigned used = 0;                           // thread 0: results of the current round applied so far, one bit per bin
  const double ratioMerge = I.ratioMerge;
  long long cyc[6] = {0, 0, 0, 0, 0, 0};
  long long tk = clock64();
  auto tick = [&](int k) { const long long now = clock64(); cyc[k] += now - tk; tk = now; };

  for (;;) {
    if (w == 0) {
      // ---- thread 0: the reference's top loop (PL:271-293); a stale top takes its result from the current round
      if (lane == 0) {
        int action = 0;  // 0 = merge, 1 = new round, 2 = finished
        if (sIter >= extbins) action = 2;
        else {
          int heapN = sHeapN;
          const int nRound = sNRound;
          for (;;) {
            const unsigned top = H.idnn(1);
            const int b1 = (int)(top & 0xFFFFu);
            const int tm = S.bTm[b1], mtm = S.bMtm[b1], nmtm = S.bMtm[top >> 16];   // three independent loads
            if (tm >= mtm && nmtm <= tm) { action = 0; sB1 = b1; break; }
            if (mtm == NQ_DELETED) {
              const unsigned last = H.idnn(heapN);
              float e1 = H.err(heapN);
              --heapN;
              ++pops;
              H.sift_down(last, e1, heapN);
              continue;
            }
            int j = 0;
            while (j < nRound && sBinR[j] != b1) ++j;
            if (j == nRound) { action = 1; break; }
            // tb.tm = i; push slot down (PL:281-293)
            const float e1 = (float)sErrR[j];
            const int nnBin = sNnR[j];
            S.bErr[b1] = e1; S.bNn[b1] = nnBin; S.bTm[b1] = sIter;
            H.sift_down(pack_idnn(b1, nnBin), e1, heapN);
            ++rescans;
            used |= 1u << j;
            pairs += (unsigned long long)max(0, liveLen - sFirstR[j]);
          }
          sHeapN = heapN;
          if (action != 2) {                   // a merge or a new round: the results not applied are dropped
            discarded += (unsigned long long)__popc(~used & (nRound == 32 ? ~0u : (1u << nRound) - 1u));
            used = 0;
            sNRound = 0;
            rounds += action == 1;
          }
        }
        sAction = action;
      }
      __syncwarp();
      // ---- warp 0: choose the round from heap slots 1..32 (all in shared memory), one entry per lane. The stale
      // entries ahead of the first valid one in (err, slot) order, deleted ones skipped, at most R of them; the
      // stale top is the first. Deeper entries are never smaller than their ancestors, so the order is the heap's
      // own for the first entries of the window; beyond them it is a guess, which only costs work if wrong.
      if (sAction == 1) {
        const int l = 1 + (int)lane;
        float e = 0.f;
        int b = 0;
        bool valid = false, stale = false;
        if (l <= sHeapN) {
          const unsigned v = H.idnn(l);
          e = H.err(l); b = (int)(v & 0xFFFFu);
          const int tm = S.bTm[b], mtm = S.bMtm[b], nmtm = S.bMtm[v >> 16];
          valid = tm >= mtm && nmtm <= tm;
          stale = !valid && mtm != NQ_DELETED;
        }
        float ve = valid ? e : INFINITY;
#pragma unroll
        for (int o = 16; o; o >>= 1) ve = fminf(ve, __shfl_xor_sync(0xffffffffu, ve, o));
        const unsigned vm = __ballot_sync(0xffffffffu, valid && e == ve);
        const int lv = vm ? __ffs(vm) - 1 : 32;                  // the first valid entry
        const bool cand = stale && (e < ve || (e == ve && (int)lane < lv));
        const unsigned cm = __ballot_sync(0xffffffffu, cand);
        int rank = 0;
#pragma unroll
        for (int k = 0; k < 32; ++k) {
          const float ek = __shfl_sync(0xffffffffu, e, k);
          rank += ((cm >> k) & 1u) && (ek < e || (ek == e && k < (int)lane));
        }
        if (cand && rank < R) sBinR[rank] = b;
        if (lane == 0) sNRound = min(R, __popc(cm));
      }
    }
    __syncthreads();
    tick(0);
    const int action = sAction;
    if (action == 2) break;

    if (action == 1) {
      const int n = sNRound;
      const LabView V{X.q, X.al, X.bs, liveLen};
      for (int k = t; k < R * 64; k += NQ_LAB_THREADS) (&sBits[0][0])[k] = 0u;
      // -- 1. the first 32 candidates of each bin in full, one warp per bin
      for (int j = (int)w; j < n; j += W) {
        const int b = sBinR[j];
        const LabProbe P = lab_probe(I, S, b, ratioMerge);
        const int first = posOf[b] + 1;
        double err = 1e100;
        int nn = -1;                            // position in the live list
        const int i = first + (int)lane;
        LabCand c;
        const bool alive = i < liveLen && lab_eval_t<false>(P, V, i, err, &c);
        lab_accept_in_order(alive, c, i, err, nn);
        fulls += i < liveLen;
        if (lane == 0) { sProbe[j] = P; sErrR[j] = err; sNnR[j] = nn; sFirstR[j] = first; }
      }
      __syncthreads();
      tick(1);
      // -- 2. block summaries of everything behind them, the blocks of all bins of the round dealt out together
      const int nblk = (liveLen + 31) >> 5;
      {
        int j = -1, base = 0, beg = 0, cnt = 0;   // bin j owns the items [base, base + cnt): its blocks beg, beg + 1, ...
        for (int k = t;; k += NQ_LAB_THREADS) {
          while (k >= base + cnt) {
            if (++j == n) break;
            base += cnt;
            beg = (sFirstR[j] + 32) >> 5;
            cnt = max(0, nblk - beg);
          }
          if (j == n) break;
          const int blk = beg + (k - base);
          if (!lab_block_skip(sProbe[j], V, blk, sErrR[j])) atomicOr(&sBits[j][blk >> 5], 1u << (blk & 31));
        }
      }
      __syncthreads();
      for (int j = (int)w; j < n; j += W) {     // live blocks of each bin before each word of its bits
        const int c0 = __popc(sBits[j][2 * lane]), c = c0 + __popc(sBits[j][2 * lane + 1]);
        int x = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= (unsigned)o) x += y; }
        sPre[j][2 * lane] = (unsigned short)(x - c);
        sPre[j][2 * lane + 1] = (unsigned short)(x - c + c0);
        if (lane == 31) sPre[j][64] = (unsigned short)x;
      }
      __syncthreads();
      tick(2);
      // Batch g holds the live blocks 32 g .. 32 g + 31 of every bin of the round, bin-major: each bin is pruned and
      // resolved on the schedule of a rescan of its own, and the round takes as many batches as its longest bin.
      int nBatch = 0;
      for (int j = 0; j < n; ++j) nBatch = max(nBatch, (sPre[j][64] + 31) >> 5);
      for (int g = 0; g < nBatch; ++g) {
        int gn = 0;                               // entries of this batch; thread t < gn makes entry t
        {
          int jt = -1, rt = 0;
          for (int j = 0; j < n; ++j) {
            const int e = min(32, max(0, (int)sPre[j][64] - 32 * g));
            if (jt < 0 && t < gn + e) { jt = j; rt = 32 * g + t - gn; }
            gn += e;
          }
          if (jt >= 0) {
            int lo = 0, hi = 64;                  // the word of bin jt's rt-th live block
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sPre[jt][mid] <= rt) lo = mid; else hi = mid; }
            const int blk = (lo << 5) + (int)__fns(sBits[jt][lo], 0, rt - sPre[jt][lo] + 1);
            sBat[t] = (unsigned short)((jt << 11) | blk);
          }
        }
        liveBlocks += gn;
        // -- 3a. per-candidate lower bound (lab_cheap_keep): one warp per entry, one lane per bin
        sMaskA[t] = 0u;
        sMaskB[t] = 0u;
        __syncthreads();
        for (int r0 = (int)w; r0 < gn; r0 += 4 * W) {     // four records in flight per lane: the loads come from L2
          float4 v[4];
          int jr[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int r = r0 + u * W;
            const int e = r < gn ? (int)sBat[r] : 0;
            jr[u] = e >> 11;
            const int i = ((e & 2047) << 5) + (int)lane;
            v[u] = (r < gn && i >= sFirstR[jr[u]] + 32 && i < liveLen) ? X.q[i] : dead;
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int r = r0 + u * W;
            const unsigned m = __ballot_sync(0xffffffffu, lab_cheap_keep_q(sProbe[jr[u]], v[u], sErrR[jr[u]]));
            if (lane == 0 && r < gn) sMaskA[r] = m;
          }
        }
        __syncthreads();
        int totalA;
        sOffA[t] = block_excl_scan_128(__popc(sMaskA[t]), &totalA, sScan);
        if (t == 0) sOffA[NQ_LAB_THREADS] = totalA;
        __syncthreads();
        // the s-th candidate that passed 3a, in batch order, and its bin of the round
        auto posA = [&](int sIdx, int& j) {
          int lo = 0, hi = gn;                    // largest r with sOffA[r] <= sIdx
          while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sOffA[mid] <= sIdx) lo = mid; else hi = mid; }
          const int e = sBat[lo];
          j = e >> 11;
          return ((e & 2047) << 5) + (int)__fns(sMaskA[lo], 0, sIdx - sOffA[lo] + 1);
        };
        // -- 3b. screen through the C' term, packed one candidate per thread
        for (int base = 0; base < totalA; base += NQ_LAB_THREADS) {
          const int sIdx = base + t;
          bool keep = false;
          if (sIdx < totalA) {
            int j;
            const int i = posA(sIdx, j);
            LabCand dummy;
            keep = lab_eval_t<true>(sProbe[j], V, i, sErrR[j], &dummy);
          }
          const unsigned m = __ballot_sync(0xffffffffu, keep);
          if (lane == 0) sMaskB[(base >> 5) + w] = m;
        }
        __syncthreads();
        int total;
        sOffB[t] = block_excl_scan_128(__popc(sMaskB[t]), &total, sScan);
        __syncthreads();
        tick(3);
        screened += total;
        const int nW = (totalA + 31) >> 5;
        // -- 4. survivors in full, packed; then each bin's resolved in its own list order against its own err
        for (int base = 0; base < total; base += NQ_LAB_THREADS) {
          const int uIdx = base + t;
          int rec = 0;
          if (uIdx < total) {
            int lo = 0, hi = nW;                  // largest word with sOffB[word] <= uIdx
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sOffB[mid] <= uIdx) lo = mid; else hi = mid; }
            const int sIdx = (lo << 5) + (int)__fns(sMaskB[lo], 0, uIdx - sOffB[lo] + 1);   // index into the 3a list
            int j;
            const int i = posA(sIdx, j);
            LabCand c;
            rec = j << 17;
            if (lab_eval_t<false>(sProbe[j], V, i, sErrR[j], &c)) { rec |= (1 << 16) | i; sGs[t] = c.gs; sGw[t] = c.gw; sF[t] = c.f; }
          }
          sPos[t] = rec;
          fulls += uIdx < total;
          __syncthreads();
          if (w == 0) {                           // a bin's candidates are contiguous: the batch is bin-major
            const int cnt = min(NQ_LAB_THREADS, total - base);
            for (int q = 0; q < cnt; q += 32) {
              const int k = q + (int)lane;
              const int rk = k < cnt ? sPos[k] : 0;
              const bool alive = k < cnt && ((rk >> 16) & 1);
              const int jk = k < cnt ? rk >> 17 : -1;
              LabCand c{0, 0, 0};
              if (alive) { c.gs = sGs[k]; c.gw = sGw[k]; c.f = sF[k]; }
              const int j0 = __shfl_sync(0xffffffffu, jk, 0), j1 = __shfl_sync(0xffffffffu, jk, min(31, cnt - 1 - q));
              for (int j = j0; j <= j1; ++j) {
                double err = sErrR[j];
                int nn = sNnR[j];
                lab_accept_in_order(alive && jk == j, c, rk & 0xFFFF, err, nn);
                __syncwarp();
                if (lane == 0) { sErrR[j] = err; sNnR[j] = nn; }
              }
            }
          }
          __syncthreads();
          tick(4);
        }
      }
      if (t < n) { const int nn = sNnR[t]; sNnR[t] = nn < 0 ? 0 : live[nn]; }
      __syncthreads();
      continue;
    }

    // ---- merge tb <- tb + nb (PL:297-311)
    if (t == 0) {
      const int b1 = sB1;
      const int nbI = S.bNn[b1];
      const float n1 = S.bCnt[b1], n2 = S.bCnt[nbI];
      const float d = 1.0f / (n1 + n2);
      const float na = d * (n1 * S.fAc[b1] + n2 * S.fAc[nbI]);
      const float nL = d * (n1 * S.fC1[b1] + n2 * S.fC1[nbI]);
      const float nA = d * (n1 * S.fC2[b1] + n2 * S.fC2[nbI]);
      const float nB = d * (n1 * S.fC3[b1] + n2 * S.fC3[nbI]);
      S.fAc[b1] = na; S.fC1[b1] = nL; S.fC2[b1] = nA; S.fC3[b1] = nB;
      S.bCnt[b1] = n1 + n2;
      const int i = sIter + 1;
      S.bMtm[b1] = i;
      S.bMtm[nbI] = NQ_DELETED;
      // compacted copies and the summary of tb's block (the count only grows, L may leave the old range)
      const int pt = posOf[b1], pn = posOf[nbI];
      X.q[pt] = make_float4(n1 + n2, nL, nA, nB); X.al[pt] = na;
      X.q[pn].x = -1.f;
      {   // widen the summary of tb's block (the count only grows)
        float4 s0 = X.bs[2 * (pt >> 5)], s1 = X.bs[2 * (pt >> 5) + 1];
        s0.y = fminf(s0.y, nL); s0.z = fmaxf(s0.z, nL); s0.w = fmaxf(s0.w, chroma_ub(nA, nB));
        s1.x = fminf(s1.x, nA); s1.y = fmaxf(s1.y, nA); s1.z = fminf(s1.z, nB); s1.w = fmaxf(s1.w, nB);
        X.bs[2 * (pt >> 5)] = s0; X.bs[2 * (pt >> 5) + 1] = s1;
      }
      if (logMerges && S.mergeLog) { S.mergeLog[2 * (i - 1)] = b1; S.mergeLog[2 * (i - 1) + 1] = nbI; }
      sIter = i;
    }
    __syncthreads();
    const int it = sIter;
    if ((it - iterAtRebuild) * 4 > liveAtRebuild) {
      liveLen = rebuild_live_lab(S, X, maxbins, live, posOf, sScan);
      liveAtRebuild = liveLen; iterAtRebuild = it;
    }
    tick(5);
  }

  // ---- palette fill (PL:315-324): the k-th live bin in ascending order
  liveLen = rebuild_live_lab(S, X, maxbins, live, posOf, sScan);
  const int plen = extbins > 0 ? I.nmax : maxbins;
  for (int k = t; k < plen; k += NQ_LAB_THREADS) {
    const int b = live[k];
    uint32_t colr;
    if (!lab2rgb(j2i((double)S.fAc[b]), S.fC1[b], S.fC2[b], S.fC3[b], &colr)) { colr = 0; I.error = 3; }
    I.palette[k] = colr;
  }
  if (t == 0) {
    I.paletteLen = plen;
    I.statRescans = rescans; I.statPairs += pairs; I.statHeapPops = pops;
    for (int k = 0; k < 6; ++k) I.statCyc[k] = (unsigned long long)cyc[k];
    I.statLiveBlocks = liveBlocks; I.statScreened = screened;
    I.statRounds = rounds; I.statDiscarded = discarded;
  }
  if (fulls) atomicAdd(&I.statFullEvals, fulls);
}

// -------------------------------------------------------------------------------------------------
// RGB merge loop, same organisation as k_merge_lab: compacted records of the surviving bins, 32-bin
// block summaries, 128 threads per image and several images per SM.
// RGB's find_nn differs in one respect that matters here: a candidate that passes the four `continue`
// tests is taken with err := the first partial sum that reaches the old err (the `break` of PQ:97-108
// falls through to PQ:111), so the running err can GROW, and no candidate can be dismissed for good by
// comparing against the current err. The kernel therefore prunes against U = 4 x (err after the first
// 32 candidates): blocks and candidates whose gate max(nerr2, q0) is >= U cannot be taken while err < U.
// The survivors are replayed in list order with the exact err; if err ever reaches U the rescan is
// redone without pruning (U = infinity), which is the reference's own scan.
// -------------------------------------------------------------------------------------------------
#define NQ_RGB_THREADS 128
#define NQ_RGB_HEAP_SMEM 6144

struct RgbScratch {
  double2* rg;          // {r, g} per position
  double2* bc;          // {b, cnt} per position; cnt < 0 marks a bin that died since the last compaction
  double* al;           // alpha per position (semi-transparent images)
  double *cmin, *lo, *hi;   // per block of 32 positions: min count, and min / max of r, g, b (3 planes of 2048 each)
};
__device__ __forceinline__ RgbScratch rgb_scratch(const NqSlot& S) {
  RgbScratch X;
  X.rg = reinterpret_cast<double2*>(S.hSum);                       // 2 MiB of histogram sums, free after compaction
  X.bc = X.rg + NQ_NBINS;
  double* f = reinterpret_cast<double*>(S.fAc);                    // the CIELAB float planes (1 MiB), unused for RGB
  X.al = f;
  X.cmin = f + NQ_NBINS; X.lo = X.cmin + 2048; X.hi = X.lo + 3 * 2048;
  return X;
}

__device__ __forceinline__ double rgb_gate_rec(const RgbProbe& P, const double2 rg, const double2 bc, double al, RgbCand* c) {
  const double n2 = bc.y;
  double nerr2 = ((double)P.n1 * n2) / ((double)P.n1 + n2);
  double nerr = 0.0;
  if (P.semi) { double d = al - P.wa; nerr += nerr2 * P.PA * (d * d); }
  double dr = rg.x - P.wr, dg = rg.y - P.wg, db = bc.x - P.wb;
  nerr += nerr2 * (1 - P.ratio) * P.PR * (dr * dr);
  nerr += nerr2 * (1 - P.ratio) * P.PG * (dg * dg);
  nerr += nerr2 * (1 - P.ratio) * P.PB * (db * db);
  c->nerr2 = nerr2; c->q0 = nerr; c->dr = dr; c->dg = dg; c->db = db;
  return nerr2 > nerr ? nerr2 : nerr;
}

// true when no bin of the block can have a gate below U (the alpha term is >= 0 and left out)
__device__ __forceinline__ bool rgb_block_skip(const RgbProbe& P, const RgbScratch& X, int blk, double U) {
  const double cmin = X.cmin[blk];
  if (!(cmin >= 0.0)) return true;
  const double n1 = (double)P.n1;
  const double nerr2 = (n1 * cmin) / (n1 + cmin) * (1.0 - 1e-12);
  if (nerr2 >= U) return true;
  const double dr = fmax(0.0, fmax(X.lo[blk] - P.wr, P.wr - X.hi[blk]));
  const double dg = fmax(0.0, fmax(X.lo[2048 + blk] - P.wg, P.wg - X.hi[2048 + blk]));
  const double db = fmax(0.0, fmax(X.lo[4096 + blk] - P.wb, P.wb - X.hi[4096 + blk]));
  const double q0 = nerr2 * (1 - P.ratio) * (P.PR * (dr * dr) + P.PG * (dg * dg) + P.PB * (db * db)) * (1.0 - 1e-12);
  return q0 >= U;
}

__device__ __forceinline__ void rgb_block_summary(const RgbScratch& X, int n, int blk) {
  double cm = -1.0, lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
  const int p0 = blk << 5, p1 = min(n, p0 + 32);
  for (int p = p0; p < p1; ++p) {
    const double2 bc = X.bc[p];
    if (!(bc.y >= 0.0)) continue;
    const double2 rg = X.rg[p];
    cm = cm < 0.0 ? bc.y : fmin(cm, bc.y);
    lo[0] = fmin(lo[0], rg.x); hi[0] = fmax(hi[0], rg.x);
    lo[1] = fmin(lo[1], rg.y); hi[1] = fmax(hi[1], rg.y);
    lo[2] = fmin(lo[2], bc.x); hi[2] = fmax(hi[2], bc.x);
  }
  X.cmin[blk] = cm;
  for (int k = 0; k < 3; ++k) { X.lo[k * 2048 + blk] = lo[k]; X.hi[k * 2048 + blk] = hi[k]; }
}

__device__ __forceinline__ int rebuild_live_rgb(const NqSlot& S, const RgbScratch& X, int maxbins, int* live, int* posOf, int* sScan) {
  const int t = threadIdx.x;
  const unsigned lane = lane_id(), w = t >> 5;
  const int W = NQ_RGB_THREADS / 32;
  const int per = (((maxbins + W - 1) / W) + 31) & ~31;
  const int b0 = min(maxbins, (int)w * per), b1 = min(maxbins, b0 + per);
  int c = 0;
  for (int b = b0 + (int)lane; b < b1; b += 32) c += S.bMtm[b] != NQ_DELETED;
  int total, j = block_excl_scan_128(c, &total, sScan);
  j = __shfl_sync(0xffffffffu, j, 0);
  for (int base = b0; base < b1; base += 32) {
    const int b = base + (int)lane;
    const bool alive = b < b1 && S.bMtm[b] != NQ_DELETED;
    const unsigned m = __ballot_sync(0xffffffffu, alive);
    if (alive) {
      const int p = j + __popc(m & ((1u << lane) - 1u));
      live[p] = b; posOf[b] = p;
      X.rg[p] = make_double2(S.bC1[b], S.bC2[b]);
      X.bc[p] = make_double2(S.bC3[b], (double)S.bCnt[b]);
      X.al[p] = S.bAc[b];
    }
    j += __popc(m);
  }
  __syncthreads();
  const int nblk = (total + 31) >> 5;
  for (int blk = t; blk < nblk; blk += NQ_RGB_THREADS) rgb_block_summary(X, total, blk);
  __syncthreads();
  return total;
}

// replay of up to 32 candidates held one per lane, in lane order (PQ:73-112)
__device__ __forceinline__ void rgb_accept_in_order(const RgbProbe& P, double gate, const RgbCand& c, int id, double& err, int& nn, double& errMax) {
  const unsigned lane = lane_id();
  unsigned remaining = 0xffffffffu;
  for (;;) {
    const unsigned m = __ballot_sync(0xffffffffu, gate < err) & remaining;
    if (!m) break;
    const int L = __ffs(m) - 1;
    double e = 0;
    if ((int)lane == L) e = rgb_take(P, c, err);
    err = __shfl_sync(0xffffffffu, e, L);
    nn = __shfl_sync(0xffffffffu, id, L);
    errMax = err > errMax ? err : errMax;
    remaining = (L == 31) ? 0u : ~((2u << L) - 1u);
  }
}

static_assert(NQ_RGB_THREADS == NQ_LAB_THREADS, "block_excl_scan_128 is shared");

__global__ void __launch_bounds__(NQ_RGB_THREADS, 4) k_merge_rgb(NqImage* imgs, const NqSlot* slots, int* liveBuf, int* posBuf, int logMerges) {
  extern __shared__ unsigned char smemRaw[];
  float* sErr = reinterpret_cast<float*>(smemRaw);
  unsigned* sId = reinterpret_cast<unsigned*>(smemRaw + (size_t)NQ_RGB_HEAP_SMEM * 4);
  __shared__ int sScan[8];
  __shared__ unsigned sBits[64];
  __shared__ unsigned short sBlk[2048];
  __shared__ unsigned sMaskA[32];
  __shared__ int sOffA[33];
  __shared__ double sErrCur, sErrMax;
  __shared__ int sNnCur, sAction, sB1, sHeapN, sIter, sNLive;

  const int img = blockIdx.x;
  NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_RGB || I.nmax <= 2 || I.skipPnn) return;
  const NqSlot& S = slots[img];
  const RgbScratch X = rgb_scratch(S);
  const int t = threadIdx.x;
  const unsigned lane = lane_id(), w = t >> 5;
  const int W = NQ_RGB_THREADS / 32;
  const int maxbins = I.maxbins, extbins = I.extbins;
  int* live = liveBuf + (size_t)img * NQ_NBINS;
  int* posOf = posBuf + (size_t)img * NQ_NBINS;
  HeapView<NQ_RGB_HEAP_SMEM> H{sErr, sId, S.heap};

  // ---- heap build: sequential pushes in bin order (PQ:196-207), replayed by warp 0
  if (w == 0) {
    int heapN = 0;
    for (int base = 0; base < maxbins; base += 32) {
      float e = (base + (int)lane < maxbins) ? S.bErr[base + lane] : 0.f;
      const int nnv = (base + (int)lane < maxbins) ? S.bNn[base + lane] : 0;
      const int cnt = min(32, maxbins - base);
      for (int j = 0; j < cnt; ++j) {
        const float err = __shfl_sync(0xffffffffu, e, j);
        const int nnj = __shfl_sync(0xffffffffu, nnv, j);
        int l = ++heapN, l2;
        for (; l > 1; l = l2) {
          l2 = l >> 1;
          float pe = H.err(l2);
          if (pe <= err) break;
          unsigned pid = H.idnn(l2);
          if (lane == 0) H.set(l, pid, pe);
        }
        if (lane == 0) H.set(l, pack_idnn(base + j, nnj), err);
        __syncwarp();
      }
    }
    if (lane == 0) { sHeapN = heapN; sIter = 0; }
  }
  __syncthreads();
  int liveLen = rebuild_live_rgb(S, X, maxbins, live, posOf, sScan);
  int liveAtRebuild = liveLen, iterAtRebuild = 0;
  unsigned long long rescans = 0, pairs = 0, redone = 0;
  unsigned pops = 0;

  for (;;) {
    // ---- thread 0: look at the heap top (PQ:214-226)
    if (t == 0) {
      int action = 0;  // 0 = merge, 1 = rescan, 2 = finished
      if (sIter >= extbins) action = 2;
      else {
        int heapN = sHeapN;
        for (;;) {
          const unsigned top = H.idnn(1);
          int b1 = (int)(top & 0xFFFFu);
          const int tm = S.bTm[b1], mtm = S.bMtm[b1], nmtm = S.bMtm[top >> 16];   // three independent loads
          if (tm >= mtm && nmtm <= tm) { action = 0; sB1 = b1; break; }
          if (mtm == NQ_DELETED) {   // deleted node: b1 = heap[1] = heap[heap[0]--], then push down
            const unsigned last = H.idnn(heapN);
            float e1 = H.err(heapN);
            --heapN;
            ++pops;
            H.sift_down(last, e1, heapN);
            continue;
          }
          action = 1; sB1 = b1;
          break;
        }
        sHeapN = heapN;
      }
      sAction = action;
    }
    __syncthreads();
    const int action = sAction;
    if (action == 2) break;
    const int b1 = sB1;

    if (action == 1) {
      ++rescans;
      const int first = posOf[b1] + 1;
      const RgbProbe P = rgb_probe(I, S, b1);
      double err = 1e100, errMax = 0.0;
      int nn = -1;                              // position in the live list
      // -- 1. the first 32 candidates, exactly
      if (w == 0) {
        const int i = first + (int)lane;
        RgbCand c;
        double gate = 1e300;
        if (i < liveLen) { const double2 bc = X.bc[i]; if (bc.y >= 0.0) gate = rgb_gate_rec(P, X.rg[i], bc, P.semi ? X.al[i] : 0.0, &c); }
        rgb_accept_in_order(P, gate, c, i, err, nn, errMax);
        if (lane == 0) { sErrCur = err; sNnCur = nn; }
      }
      __syncthreads();
      const double err32 = sErrCur;
      const int nn32 = sNnCur;
      const int stop = first + 32;
      const int blkBeg = stop >> 5, nblk = (liveLen + 31) >> 5;
      for (int attempt = 0; attempt < 2; ++attempt) {
        // attempt 0 prunes against U = 4 err32; attempt 1 (only if err reached U) is the plain scan
        const double U = attempt == 0 ? (err32 < 1e99 ? 4.0 * err32 : 1e300) : 1e300;
        err = err32; nn = nn32; errMax = err32 < 1e99 ? err32 : 0.0;
        if (t < 64) sBits[t] = 0u;
        __syncthreads();
        for (int blk = blkBeg + t; blk < nblk; blk += NQ_RGB_THREADS)
          if (!rgb_block_skip(P, X, blk, U)) atomicOr(&sBits[blk >> 5], 1u << (blk & 31));
        __syncthreads();
        if (w == 0) {                             // bit set -> ordered list
          const unsigned m0 = sBits[2 * lane], m1 = sBits[2 * lane + 1];
          const int c = __popc(m0) + __popc(m1);
          int x = c;
#pragma unroll
          for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= (unsigned)o) x += y; }
          int at = x - c;
          for (unsigned m = m0; m; m &= m - 1) sBlk[at++] = (unsigned short)(64 * lane + (__ffs(m) - 1));
          for (unsigned m = m1; m; m &= m - 1) sBlk[at++] = (unsigned short)(64 * lane + 32 + (__ffs(m) - 1));
          if (lane == 31) sNLive = x;
        }
        __syncthreads();
        const int nLive = sNLive;
        for (int g0 = 0; g0 < nLive; g0 += 32) {  // batches of 32 live blocks, in list order
          const int gn = min(32, nLive - g0);
          if (t < 32) sMaskA[t] = 0u;
          __syncthreads();
          // -- 2. gates of the bins of the live blocks: one warp per block, one lane per bin
          for (int r = w; r < gn; r += W) {
            const int i = ((int)sBlk[g0 + r] << 5) + (int)lane;
            bool keep = false;
            if (i >= stop && i < liveLen) {
              const double2 bc = X.bc[i];
              RgbCand c;
              if (bc.y >= 0.0) keep = rgb_gate_rec(P, X.rg[i], bc, P.semi ? X.al[i] : 0.0, &c) < U;
            }
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (lane == 0) sMaskA[r] = m;
          }
          __syncthreads();
          // -- 3. warp 0 replays the kept bins in list order with the exact err
          if (w == 0) {
            const int c = __popc(sMaskA[lane]);
            int x = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= (unsigned)o) x += y; }
            sOffA[lane + 1] = x;
            if (lane == 0) sOffA[0] = 0;
            __syncwarp();
            const int totalA = sOffA[32];
            for (int base = 0; base < totalA; base += 32) {
              const int sIdx = base + (int)lane;
              RgbCand c;
              double gate = 1e300;
              int i = -1;
              if (sIdx < totalA) {
                int lo = 0, hi = 32;
                while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (sOffA[mid] <= sIdx) lo = mid; else hi = mid; }
                i = ((int)sBlk[g0 + lo] << 5) + (int)__fns(sMaskA[lo], 0, sIdx - sOffA[lo] + 1);
                gate = rgb_gate_rec(P, X.rg[i], X.bc[i], P.semi ? X.al[i] : 0.0, &c);
              }
              rgb_accept_in_order(P, gate, c, i, err, nn, errMax);
            }
          }
          __syncthreads();
        }
        if (w == 0 && lane == 0) { sErrCur = err; sNnCur = nn; sErrMax = errMax; }
        __syncthreads();
        if (!(sErrMax >= U)) break;               // err never reached U: the pruning was sound
        ++redone;
      }
      err = sErrCur; nn = sNnCur;
      pairs += (unsigned long long)max(0, liveLen - first);
      if (t == 0) {
        // tb.tm = i; push slot down (PQ:224-236)
        float e1 = (float)err;
        const int nnBin = nn < 0 ? 0 : live[nn];
        S.bErr[b1] = e1; S.bNn[b1] = nnBin; S.bTm[b1] = sIter;
        H.sift_down(pack_idnn(b1, nnBin), e1, sHeapN);
      }
      __syncthreads();
      continue;
    }

    // ---- merge tb <- tb + nb (PQ:240-254)
    if (t == 0) {
      const int nbI = S.bNn[b1];
      const float n1 = S.bCnt[b1], n2 = S.bCnt[nbI];
      const float d = 1.f / (n1 + n2);
      const double na = (double)(d * (float)jround((double)n1 * S.bAc[b1] + (double)n2 * S.bAc[nbI]));   // float * long -> float
      const double nr = (double)(d * (float)jround((double)n1 * S.bC1[b1] + (double)n2 * S.bC1[nbI]));
      const double ng = (double)(d * (float)jround((double)n1 * S.bC2[b1] + (double)n2 * S.bC2[nbI]));
      const double nb = (double)(d * (float)jround((double)n1 * S.bC3[b1] + (double)n2 * S.bC3[nbI]));
      S.bAc[b1] = na; S.bC1[b1] = nr; S.bC2[b1] = ng; S.bC3[b1] = nb;
      S.bCnt[b1] = n1 + n2;
      const int i = sIter + 1;
      S.bMtm[b1] = i;
      S.bMtm[nbI] = NQ_DELETED;
      const int pt = posOf[b1], pn = posOf[nbI], bt = pt >> 5;
      X.rg[pt] = make_double2(nr, ng); X.bc[pt] = make_double2(nb, (double)(n1 + n2)); X.al[pt] = na;
      X.bc[pn].y = -1.0;
      X.lo[bt] = fmin(X.lo[bt], nr); X.hi[bt] = fmax(X.hi[bt], nr);
      X.lo[2048 + bt] = fmin(X.lo[2048 + bt], ng); X.hi[2048 + bt] = fmax(X.hi[2048 + bt], ng);
      X.lo[4096 + bt] = fmin(X.lo[4096 + bt], nb); X.hi[4096 + bt] = fmax(X.hi[4096 + bt], nb);
      if (logMerges && S.mergeLog) { S.mergeLog[2 * (i - 1)] = b1; S.mergeLog[2 * (i - 1) + 1] = nbI; }
      sIter = i;
    }
    __syncthreads();
    const int it = sIter;
    if ((it - iterAtRebuild) * 4 > liveAtRebuild) {
      liveLen = rebuild_live_rgb(S, X, maxbins, live, posOf, sScan);
      liveAtRebuild = liveLen; iterAtRebuild = it;
    }
  }

  // ---- palette fill (PQ:258-264): the k-th live bin in ascending order
  liveLen = rebuild_live_rgb(S, X, maxbins, live, posOf, sScan);
  const int plen = extbins > 0 ? I.nmax : maxbins;
  for (int k = t; k < plen; k += NQ_RGB_THREADS) {
    const int b = live[k];
    I.palette[k] = c_argb(j2i(S.bAc[b]), j2i(S.bC1[b]), j2i(S.bC2[b]), j2i(S.bC3[b]));
  }
  if (t == 0) {
    I.paletteLen = plen;
    I.statRescans = rescans; I.statPairs += pairs; I.statHeapPops = pops; I.statFullEvals = redone;
  }
}


// -------------------------------------------------------------------------------------------------
// RGB initial sweep (PQ:196-197): one warp per bin over bin-indexed records (k_rgb_blocks), the first 32
// candidates exactly, then blocks pruned against U = 4 x that err and the rest replayed in order with the
// exact err; a bin whose err reached U is redone unpruned (see k_merge_rgb).
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_rgb_blocks(const NqImage* imgs, const NqSlot* slots) {
  const int img = blockIdx.y;
  const NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_RGB || I.nmax <= 2 || I.skipPnn) return;
  const NqSlot& S = slots[img];
  const RgbScratch X = rgb_scratch(S);
  const int n = I.maxbins, nblk = (n + 31) >> 5;
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < n; b += gridDim.x * blockDim.x) {
    X.rg[b] = make_double2(S.bC1[b], S.bC2[b]);
    X.bc[b] = make_double2(S.bC3[b], (double)S.bCnt[b]);
    X.al[b] = S.bAc[b];
  }
  // summaries straight from the bins (the records above are written by other threads)
  for (int blk = blockIdx.x * blockDim.x + threadIdx.x; blk < nblk; blk += gridDim.x * blockDim.x) {
    double cm = 1e300, lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    for (int b = blk << 5; b < min(n, (blk << 5) + 32); ++b) {
      cm = fmin(cm, (double)S.bCnt[b]);
      const double v[3] = {S.bC1[b], S.bC2[b], S.bC3[b]};
      for (int k = 0; k < 3; ++k) { lo[k] = fmin(lo[k], v[k]); hi[k] = fmax(hi[k], v[k]); }
    }
    X.cmin[blk] = cm;
    for (int k = 0; k < 3; ++k) { X.lo[k * 2048 + blk] = lo[k]; X.hi[k * 2048 + blk] = hi[k]; }
  }
}

__global__ void __launch_bounds__(256) k_find_nn_all(NqImage* imgs, const NqSlot* slots, int nimg) {
  const unsigned lane = lane_id();
  const int wpb = blockDim.x >> 5;
  for (int img = 0; img < nimg; ++img) {
    NqImage& I = imgs[img];
    if (I.kind != NQ_KIND_RGB || I.nmax <= 2 || I.skipPnn) continue;
    const NqSlot& S = slots[img];
    const RgbScratch X = rgb_scratch(S);
    const int maxbins = I.maxbins;
    unsigned long long pairs = 0;
    for (int idx = blockIdx.x * wpb + (threadIdx.x >> 5); idx < maxbins; idx += gridDim.x * wpb) {
      const RgbProbe P = rgb_probe(I, S, idx);
      double err = 1e100, errMax = 0.0;
      int nn = 0;
      {   // the first 32 candidates
        const int i = idx + 1 + (int)lane;
        RgbCand c;
        double gate = 1e300;
        if (i < maxbins) gate = rgb_gate_rec(P, X.rg[i], X.bc[i], P.semi ? X.al[i] : 0.0, &c);
        rgb_accept_in_order(P, gate, c, i, err, nn, errMax);
      }
      const double err32 = err;
      const int nn32 = nn, stop = idx + 33;
      for (int attempt = 0; attempt < 2; ++attempt) {
        const double U = attempt == 0 ? (err32 < 1e99 ? 4.0 * err32 : 1e300) : 1e300;
        err = err32; nn = nn32; errMax = err32 < 1e99 ? err32 : 0.0;
        for (int blk0 = stop >> 5; (blk0 << 5) < maxbins; blk0 += 32) {
          const int blk = blk0 + (int)lane;
          unsigned bm = __ballot_sync(0xffffffffu, (blk << 5) < maxbins && !rgb_block_skip(P, X, blk, U));
          while (bm) {
            const int b = __ffs(bm) - 1;
            bm &= bm - 1;
            const int i = ((blk0 + b) << 5) + (int)lane;
            RgbCand c;
            double gate = 1e300;
            if (i >= stop && i < maxbins) gate = rgb_gate_rec(P, X.rg[i], X.bc[i], P.semi ? X.al[i] : 0.0, &c);
            rgb_accept_in_order(P, gate, c, i, err, nn, errMax);
          }
        }
        if (!(errMax >= U)) break;
      }
      pairs += (unsigned long long)(maxbins - idx - 1);
      if (lane == 0) { S.bErr[idx] = (float)err; S.bNn[idx] = nn; }
    }
    if (lane == 0 && pairs) atomicAdd(&I.statPairs, pairs);
  }
}

}  // namespace nq
