// nq_hist.cuh -- pixel passes: alpha scan, RGB histogram, strict-order CIELAB histogram, saliency.
// Reference: PnnQuantizer.convert alpha scan (PQ:411-436), pnnquan histogram + compaction
// (PQ:137-191), PnnLABQuantizer.pnnquan (PL:134-241), getLab / RGB2LAB (PL:34-42, CL:58-69).
#pragma once
#include "nq_types.h"
#include "nq_color.h"

namespace nq {

__device__ double g_gammaLut[256];          // gammaToLinear(v), v = 0..255 (CL:71-75)
__device__ signed char g_blueNoise[4096];   // TELL_BLUE_NOISE (BN:13-178)

// RGB -> CIELAB for every 24-bit colour: (L, A, B, -) as float4. The reference memoizes getLab per colour
// in a HashMap (PL:34-42); with 180 GB of HBM the whole function fits in a 256 MiB table built once per
// device, so the pixel passes gather 16 bytes instead of evaluating three pow() per pixel.
__device__ const float4* g_labLut;

__global__ void __launch_bounds__(256) k_build_lab_lut(float4* lut) {
  const unsigned c = blockIdx.x * blockDim.x + threadIdx.x;   // 65536 blocks x 256
  Lab4 l = rgb2lab(0xFF000000u | c, g_gammaLut);
  lut[c] = make_float4(l.L, l.A, l.B, 0.f);
}
__device__ __forceinline__ Lab4 lab_of(uint32_t c) {
  const float4 v = __ldg(&g_labLut[c & 0xFFFFFFu]);
  Lab4 o;
  o.alpha = (float)(c >> 24); o.L = v.x; o.A = v.y; o.B = v.z;
  return o;
}

__global__ void k_init_tables(const signed char* bn) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < 256) g_gammaLut[t] = gamma_to_linear(t);
  for (int i = t; i < 4096; i += gridDim.x * blockDim.x) g_blueNoise[i] = bn[i];
}

__device__ __forceinline__ uint32_t eff_pixel(uint32_t p, int fixA0) {
  return (fixA0 && (p >> 24) == 0) ? 0x00FFFFFFu : p;
}
__device__ __forceinline__ uint4 ld_stream4(const uint32_t* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ unsigned lane_id() { return threadIdx.x & 31; }

// ---- alpha scan (PQ:411-429): count semi-transparent pixels, remember the LAST a==0 index --------
__global__ void __launch_bounds__(256) k_alpha_scan(NqImage* imgs, const NqSlot* slots) {
  const int img = blockIdx.y;
  const int n = imgs[img].npix;
  const uint32_t* in = slots[img].in;
  unsigned semi = 0, nonop = 0;
  int last = -1;
  const bool vec = ((uintptr_t)in & 15) == 0;
  const int n4 = vec ? (n >> 2) : 0;
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < n4; q += gridDim.x * blockDim.x) {
    uint4 v = ld_stream4(in + 4 * (size_t)q);
    uint32_t px[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      unsigned a = px[k] >> 24;
      if (a != 0xFF) {
        ++nonop;
        if (a < 0xE0) {
          if (a == 0) last = 4 * q + k;
          else if (a > 0xF) ++semi;
        }
      }
    }
  }
  for (int i = 4 * n4 + blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    unsigned a = in[i] >> 24;
    nonop += a != 0xFF;
    if (a < 0xE0) {
      if (a == 0) last = max(last, i);
      else if (a > 0xF) ++semi;
    }
  }
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    semi += __shfl_xor_sync(0xffffffffu, semi, o);
    nonop += __shfl_xor_sync(0xffffffffu, nonop, o);
    last = max(last, __shfl_xor_sync(0xffffffffu, last, o));
  }
  if (lane_id() == 0) {
    if (semi) atomicAdd(&imgs[img].semiCount, semi);
    if (nonop) atomicAdd(&imgs[img].nonOpaque, nonop);
    if (last >= 0) atomicMax(&imgs[img].transIdx, last);
  }
}

// ---- scalars that follow the scan (PQ:431-436, PQ:144) ------------------------------------------
__global__ void k_setup_scan(NqImage* imgs, const NqSlot* slots, int nimg) {
  int img = blockIdx.x * blockDim.x + threadIdx.x;
  if (img >= nimg) return;
  NqImage& I = imgs[img];
  I.hasSemi = I.semiCount > 0;
  I.fixA0 = I.nmax <= 2;
  I.transColor = 0x00FFFFFFu;                                  // PQ:22
  if (I.transIdx >= 0 && I.nmax > 2) I.transColor = slots[img].in[I.transIdx];   // PQ:421-422
  if (I.nmax <= 32) I.PR = I.PG = I.PB = I.PA = 1;             // PQ:432-433
  else { I.PR = (double)0.299f; I.PG = (double)0.587f; I.PB = (double)0.114f; I.PA = .3333; }   // PQ:435 (floats widened)
  I.ratio = I.ratioMerge = .5;
  I.weight = 1;
  I.keyTransp = (I.nmax < 64) || (I.transIdx >= 0);
}

// ---- RGB histogram (PQ:140-154): integer-exact sums -----------------------------------------------
// 65 536 bins x 5 accumulators do not fit in shared memory, but a stretch of neighbouring pixels only
// touches a few thousand of them. Each CTA walks NQ_HTW x NQ_HTW pixel tiles (128-bit loads, four
// pixels per thread per load) and combines them in a shared-memory hash table of NQ_HSLOTS entries
// (key tag + count + four channel sums, integer atomics); after every tile the occupied slots are
// flushed with global atomics. Pixels whose slot (and its neighbour) belongs to another key go to global
// memory directly. Sums are integers, so the result does not depend on any of this.
#define NQ_HSLOTS 2048
#define NQ_HTW 64           // tile side in pixels
struct HistTable { unsigned tag[NQ_HSLOTS], cnt[NQ_HSLOTS], sa[NQ_HSLOTS], sr[NQ_HSLOTS], sg[NQ_HSLOTS], sb[NQ_HSLOTS]; };

__device__ __forceinline__ void hist_rgb_add(HistTable& T, unsigned int* hc, unsigned long long* hs, uint32_t p, bool semi, bool tr) {
  const unsigned key = (unsigned)color_index(p, semi, tr);
  unsigned slot = (key ^ (key >> 7) ^ (key >> 12)) & (NQ_HSLOTS - 1);
  const unsigned tagv = key + 1u;
#pragma unroll
  for (int probe = 0; probe < 2; ++probe) {
    unsigned t = T.tag[slot];
    if (t == 0u) t = atomicCAS(&T.tag[slot], 0u, tagv), t = t == 0u ? tagv : t;
    if (t == tagv) {
      atomicAdd(&T.cnt[slot], 1u);
      atomicAdd(&T.sa[slot], p >> 24);
      atomicAdd(&T.sr[slot], (p >> 16) & 0xFFu);
      atomicAdd(&T.sg[slot], (p >> 8) & 0xFFu);
      atomicAdd(&T.sb[slot], p & 0xFFu);
      return;
    }
    slot = (slot + 1u) & (NQ_HSLOTS - 1);
  }
  atomicAdd(&hc[key], 1u);
  atomicAdd(&hs[key], (unsigned long long)(p >> 24));
  atomicAdd(&hs[NQ_NBINS + key], (unsigned long long)((p >> 16) & 0xFF));
  atomicAdd(&hs[2 * NQ_NBINS + key], (unsigned long long)((p >> 8) & 0xFF));
  atomicAdd(&hs[3 * NQ_NBINS + key], (unsigned long long)(p & 0xFF));
}

__global__ void __launch_bounds__(256) k_hist_rgb(const NqImage* imgs, const NqSlot* slots) {
  extern __shared__ unsigned char histSmem[];
  HistTable& T = *reinterpret_cast<HistTable*>(histSmem);
  const int img = blockIdx.y;
  const NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_RGB || I.nmax <= 2) return;
  const uint32_t* in = slots[img].in;
  unsigned int* hc = slots[img].hCnt;
  unsigned long long* hs = slots[img].hSum;
  const bool semi = I.hasSemi, tr = I.keyTransp;
  const uint32_t tc = I.transColor;
  const bool vec = ((uintptr_t)in & 15) == 0;
  const int t = threadIdx.x;
  for (int s = t; s < NQ_HSLOTS; s += 256) { T.tag[s] = 0u; T.cnt[s] = 0u; T.sa[s] = 0u; T.sr[s] = 0u; T.sg[s] = 0u; T.sb[s] = 0u; }
  __syncthreads();
  // square tiles: neighbouring pixels in BOTH directions share colours, a strip of full rows does not
  const int width = I.width, height = I.height;
  const int tx = (width + NQ_HTW - 1) / NQ_HTW, ty = (height + NQ_HTW - 1) / NQ_HTW;
  const bool vec4 = vec && (width & 3) == 0;
  for (int tile = blockIdx.x; tile < tx * ty; tile += gridDim.x) {
    const int x0 = (tile % tx) * NQ_HTW, y0 = (tile / tx) * NQ_HTW;
    const int x1 = min(width, x0 + NQ_HTW), y1 = min(height, y0 + NQ_HTW);
    if (vec4) {
      const int qw = (x1 - x0) >> 2;                 // quads per tile row (x0 and width are multiples of 4)
      const int total = qw * (y1 - y0);
      for (int e = t; e < total; e += 256) {
        const int ry = e / qw, rq = e - ry * qw;
        const uint4 v = ld_stream4(in + (size_t)(y0 + ry) * width + x0 + 4 * rq);
        uint32_t px[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          uint32_t p = px[k];
          if ((p >> 24) <= 0xF) p = tc;
          hist_rgb_add(T, hc, hs, p, semi, tr);
        }
      }
    } else {
      const int tw = x1 - x0, total = tw * (y1 - y0);
      for (int e = t; e < total; e += 256) {
        const int ry = e / tw, rx = e - ry * tw;
        uint32_t p = in[(size_t)(y0 + ry) * width + x0 + rx];
        if ((p >> 24) <= 0xF) p = tc;
        hist_rgb_add(T, hc, hs, p, semi, tr);
      }
    }
    __syncthreads();
    // flush the occupied slots and clear them for the next tile
    for (int s = t; s < NQ_HSLOTS; s += 256) {
      const unsigned tg = T.tag[s];
      if (tg) {
        const unsigned key = tg - 1u;
        atomicAdd(&hc[key], T.cnt[s]);
        atomicAdd(&hs[key], (unsigned long long)T.sa[s]);
        atomicAdd(&hs[NQ_NBINS + key], (unsigned long long)T.sr[s]);
        atomicAdd(&hs[2 * NQ_NBINS + key], (unsigned long long)T.sg[s]);
        atomicAdd(&hs[3 * NQ_NBINS + key], (unsigned long long)T.sb[s]);
        T.tag[s] = 0u; T.cnt[s] = 0u; T.sa[s] = 0u; T.sr[s] = 0u; T.sg[s] = 0u; T.sb[s] = 0u;
      }
    }
    __syncthreads();
  }
}

// block-wide exclusive scan of one int per thread (blockDim.x == 1024); returns the exclusive
// prefix, *total gets the block sum
__device__ __forceinline__ int block_excl_scan_1024(int v, int* total, int* sWarp /*[33]*/) {
  const unsigned lane = lane_id(), w = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= (unsigned)o) x += y;
  }
  if (lane == 31) sWarp[w] = x;
  __syncthreads();
  if (w == 0) {
    int s = sWarp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int y = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= (unsigned)o) s += y;
    }
    sWarp[lane] = s;
    if (lane == 31) sWarp[32] = s;
  }
  __syncthreads();
  int base = w ? sWarp[w - 1] : 0;
  *total = sWarp[32];
  int r = base + x - v;
  __syncthreads();
  return r;
}

// PnnQuantizer.getQuanFn (PQ:123-132)
__device__ __forceinline__ float quan_rgb(int nmax, int quan_rt, float cnt) {
  if (quan_rt > 0) {
    if (nmax < 64) return (float)nqm::sqrt_((double)cnt);
    return (float)j2i(nqm::sqrt_((double)cnt));
  }
  if (quan_rt < 0) return (float)j2i(nqm::nq_cbrt((double)cnt));
  return cnt;
}
// PnnLABQuantizer.getQuanFn (PL:117-128)
__device__ __forceinline__ float quan_lab(int nmax, int quan_rt, float cnt) {
  if (quan_rt > 0) {
    if (quan_rt > 1) return (float)nqm::nq_pow((double)cnt, 0.75);
    if (nmax < 64) return (float)j2i(nqm::sqrt_((double)cnt));
    return (float)nqm::sqrt_((double)cnt);
  }
  return cnt;
}

// ---- compaction + means + pnnquan scalars, RGB (PQ:157-191) --------------------------------------
__global__ void __launch_bounds__(1024) k_finalize_rgb(NqImage* imgs, const NqSlot* slots) {
  __shared__ int sWarp[33];
  const int img = blockIdx.x;
  NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_RGB || I.nmax <= 2) return;
  const NqSlot& S = slots[img];
  const int t = threadIdx.x, k0 = t * 64;
  int c = 0;
  for (int k = 0; k < 64; ++k) c += S.hCnt[k0 + k] != 0;
  int total, j = block_excl_scan_1024(c, &total, sWarp);
  for (int k = 0; k < 64; ++k) {
    unsigned cnt = S.hCnt[k0 + k];
    if (!cnt) continue;
    float fc = cnt > 16777216u ? 16777216.f : (float)cnt;   // float cnt++ saturates at 2^24 (PQ:153)
    float d = 1.f / fc;                                      // PQ:163
    S.bAc[j] = (double)S.hSum[k0 + k] * (double)d;
    S.bC1[j] = (double)S.hSum[NQ_NBINS + k0 + k] * (double)d;
    S.bC2[j] = (double)S.hSum[2 * NQ_NBINS + k0 + k] * (double)d;
    S.bC3[j] = (double)S.hSum[3 * NQ_NBINS + k0 + k] * (double)d;
    S.bCnt[j] = fc;
    S.bErr[j] = 0.f; S.bNn[j] = 0; S.bTm[j] = 0; S.bMtm[j] = 0;
    ++j;
  }
  if (t == 0) {
    int maxbins = total, quan_rt = 1;
    if (I.nmax < 16) quan_rt = -1;                                   // PQ:172-173
    I.weight = dmin(0.9, I.nmax * 1.0 / maxbins);                    // PQ:175
    if (I.weight < .04 && I.PG >= (double)0.587f) {                  // PQ:176-180
      I.PR = I.PG = I.PB = I.PA = 1;
      if (I.nmax >= 64) quan_rt = 0;
    }
    I.maxbins = maxbins; I.quan_rt = quan_rt; I.extbins = maxbins - I.nmax;
    I.isNano = !(I.weight > .015);                                   // reduced memo key (PQ:271)
  }
  __syncthreads();
  const int maxbins = I.maxbins, quan_rt = I.quan_rt, nmax = I.nmax;
  for (int b = t; b < maxbins; b += 1024) S.bCnt[b] = quan_rgb(nmax, quan_rt, S.bCnt[b]);   // PQ:185-191
}

// =================================================================================================
// CIELAB histogram, strict pixel order. The reference adds float Lab components per bin in pixel
// order (PL:150-154); float addition is not associative, so we stable-sort the (transparent-
// replaced) pixels by bin key with a two-pass LSD radix sort and let one warp per bin add its
// run sequentially. Counts come from integer atomics.
// =================================================================================================
#define NQ_RUN 8192   // pixels per warp run in the radix passes

__device__ __forceinline__ uint32_t lab_src_pixel(uint32_t p, uint32_t tc) { return ((p >> 24) <= 0xF) ? tc : p; }

// pixelMap.put(c, ...) (PL:34-42) as a bit set over all ARGB values; returns nothing, counts first insertions
__device__ __forceinline__ void pixelmap_add(unsigned int* bits, unsigned int* counter, uint32_t c, bool active) {
  bool fresh = false;
  if (active) {
    const unsigned m = 1u << (c & 31u);
    fresh = !(atomicOr(&bits[c >> 5], m) & m);
  }
  const unsigned f = __ballot_sync(__activemask(), fresh);
  if (f && (threadIdx.x & 31) == (unsigned)(__ffs(f) - 1)) atomicAdd(counter, (unsigned)__popc(f));
}

__global__ void __launch_bounds__(256) k_lab_count(NqImage* imgs, const NqSlot* slots) {
  const int img = blockIdx.y;
  NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2) return;
  const int n = I.npix;
  const uint32_t* in = slots[img].in;
  unsigned int* hc = slots[img].hCnt;
  const bool semi = I.hasSemi, tr = I.keyTransp;
  const uint32_t tc = I.transColor;
  unsigned int* bits = slots[img].bits;
  for (int i0 = blockIdx.x * blockDim.x; i0 < n; i0 += gridDim.x * blockDim.x) {
    const int i = i0 + (int)threadIdx.x;
    uint32_t p = 0;
    if (i < n) {
      p = lab_src_pixel(in[i], tc);
      atomicAdd(&hc[color_index(p, semi, tr)], 1u);
    }
    if (bits) pixelmap_add(bits, &I.distinctColors, p, i < n);     // getLab(pixel) in the histogram loop (PL:148)
  }
}

// exclusive scan of the 65536 key counts -> keyOff[0..65536]
__global__ void __launch_bounds__(1024) k_lab_scan_keys(const NqImage* imgs, const NqSlot* slots) {
  __shared__ int sWarp[33];
  const int img = blockIdx.x;
  const NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2) return;
  const NqSlot& S = slots[img];
  const int t = threadIdx.x, k0 = t * 64;
  int c = 0;
  for (int k = 0; k < 64; ++k) c += (int)S.hCnt[k0 + k];
  int total, base = block_excl_scan_1024(c, &total, sWarp);
  for (int k = 0; k < 64; ++k) { S.keyOff[k0 + k] = (unsigned)base; base += (int)S.hCnt[k0 + k]; }
  if (t == 1023) S.keyOff[NQ_NBINS] = (unsigned)base;
}

// radix pass, step 1: per-run digit counts. One warp per run of NQ_RUN consecutive pixels.
template <int PASS>
__global__ void __launch_bounds__(256) k_radix_count(const NqImage* imgs, const NqSlot* slots) {
  __shared__ unsigned sCnt[8][256];
  const int img = blockIdx.y;
  const NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2) return;
  const NqSlot& S = slots[img];
  const int n = I.npix, nruns = (n + NQ_RUN - 1) / NQ_RUN;
  const unsigned lane = lane_id(), w = threadIdx.x >> 5;
  const uint32_t* src = PASS == 0 ? S.in : S.sortA;
  const bool semi = I.hasSemi, tr = I.keyTransp;
  const uint32_t tc = I.transColor;
  for (int run = blockIdx.x * 8 + w; run < nruns; run += gridDim.x * 8) {
    for (int d = lane; d < 256; d += 32) sCnt[w][d] = 0;
    __syncwarp();
    const int beg = run * NQ_RUN, end = min(n, beg + NQ_RUN);
    for (int i = beg + lane; i - (int)lane < end; i += 32) {
      bool ok = i < end;
      uint32_t p = ok ? src[i] : 0;
      if (PASS == 0) p = lab_src_pixel(p, tc);
      int key = color_index(p, semi, tr);
      int dg = ok ? (PASS == 0 ? (key & 255) : (key >> 8)) : 256 + (int)lane;   // inactive lanes never match
      unsigned m = __match_any_sync(0xffffffffu, dg);
      if (ok && (m & ((1u << lane) - 1)) == 0) sCnt[w][dg] += __popc(m);
      __syncwarp();
    }
    for (int d = lane; d < 256; d += 32) S.warpHist[(size_t)run * 256 + d] = sCnt[w][d];
    __syncwarp();
  }
}

// radix pass, step 2: turn counts into global start offsets, digit-major then run-major.
__global__ void __launch_bounds__(256) k_radix_offsets(const NqImage* imgs, const NqSlot* slots) {
  __shared__ unsigned sTot[256];
  const int img = blockIdx.x;
  const NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2) return;
  const NqSlot& S = slots[img];
  const int nruns = (I.npix + NQ_RUN - 1) / NQ_RUN;
  const int d = threadIdx.x;
  unsigned acc = 0;
  for (int r0 = 0; r0 < nruns; r0 += 8) {      // eight loads in flight: the counters come from L2
    unsigned c[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) c[u] = r0 + u < nruns ? S.warpHist[(size_t)(r0 + u) * 256 + d] : 0u;
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (r0 + u < nruns) { S.warpHist[(size_t)(r0 + u) * 256 + d] = acc; acc += c[u]; }
  }
  sTot[d] = acc;
  __syncthreads();
  if (d == 0) {
    unsigned run = 0;
    for (int k = 0; k < 256; ++k) { unsigned c = sTot[k]; sTot[k] = run; run += c; }
  }
  __syncthreads();
  const unsigned base = sTot[d];
  for (int r0 = 0; r0 < nruns; r0 += 8) {
    unsigned c[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) c[u] = r0 + u < nruns ? S.warpHist[(size_t)(r0 + u) * 256 + d] : 0u;
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (r0 + u < nruns) S.warpHist[(size_t)(r0 + u) * 256 + d] = c[u] + base;
  }
}

// radix pass, step 3: stable scatter.
template <int PASS>
__global__ void __launch_bounds__(256) k_radix_scatter(const NqImage* imgs, const NqSlot* slots) {
  __shared__ unsigned sPos[8][256];
  const int img = blockIdx.y;
  const NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2) return;
  const NqSlot& S = slots[img];
  const int n = I.npix, nruns = (n + NQ_RUN - 1) / NQ_RUN;
  const unsigned lane = lane_id(), w = threadIdx.x >> 5;
  const uint32_t* src = PASS == 0 ? S.in : S.sortA;
  uint32_t* dst = PASS == 0 ? S.sortA : S.sortB;
  const bool semi = I.hasSemi, tr = I.keyTransp;
  const uint32_t tc = I.transColor;
  for (int run = blockIdx.x * 8 + w; run < nruns; run += gridDim.x * 8) {
    for (int d = lane; d < 256; d += 32) sPos[w][d] = S.warpHist[(size_t)run * 256 + d];
    __syncwarp();
    const int beg = run * NQ_RUN, end = min(n, beg + NQ_RUN);
    for (int i = beg + lane; i - (int)lane < end; i += 32) {
      bool ok = i < end;
      uint32_t p = ok ? src[i] : 0;
      if (PASS == 0) p = lab_src_pixel(p, tc);
      int key = color_index(p, semi, tr);
      int dg = ok ? (PASS == 0 ? (key & 255) : (key >> 8)) : 256 + (int)lane;
      unsigned m = __match_any_sync(0xffffffffu, dg);
      unsigned below = m & ((1u << lane) - 1);
      unsigned pos = ok ? sPos[w][dg] + __popc(below) : 0;
      __syncwarp();
      if (ok && below == 0) sPos[w][dg] += __popc(m);
      __syncwarp();
      if (ok) dst[pos] = p;
    }
  }
}

// one warp per histogram key: add the bin's pixels in pixel order (PL:150-154)
__global__ void __launch_bounds__(256) k_lab_bin_sum(const NqImage* imgs, const NqSlot* slots) {
  const int img = blockIdx.y;
  const NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2) return;
  const NqSlot& S = slots[img];
  const unsigned lane = lane_id();
  const int wpb = blockDim.x >> 5;
  for (int key = blockIdx.x * wpb + (threadIdx.x >> 5); key < NQ_NBINS; key += gridDim.x * wpb) {
    const unsigned beg = S.keyOff[key], end = S.keyOff[key + 1];
    if (beg == end) continue;
    float ac = 0.f, Lc = 0.f, Ac = 0.f, Bc = 0.f;
    for (unsigned base = beg; base < end; base += 32) {
      const unsigned i = base + lane;
      Lab4 v = {0.f, 0.f, 0.f, 0.f};
      if (i < end) v = lab_of(S.sortB[i]);
      const int cnt = (int)min(32u, end - base);
      for (int j = 0; j < cnt; ++j) {
        ac += __shfl_sync(0xffffffffu, v.alpha, j);
        Lc += __shfl_sync(0xffffffffu, v.L, j);
        Ac += __shfl_sync(0xffffffffu, v.A, j);
        Bc += __shfl_sync(0xffffffffu, v.B, j);
      }
    }
    if (lane == 0) {
      // reuse hSum storage as 4 float planes
      float* fs = reinterpret_cast<float*>(S.hSum);
      fs[key] = ac; fs[NQ_NBINS + key] = Lc; fs[2 * NQ_NBINS + key] = Ac; fs[3 * NQ_NBINS + key] = Bc;
    }
  }
}

// ---- compaction + means + pnnquan scalars, LAB (PL:160-241) --------------------------------------
// means == 0 (remap front): the scalars alone, which depend on the key counts only (maxbins), so neither the sorted float
// sums of k_lab_bin_sum nor the compacted bins are needed
__global__ void __launch_bounds__(1024) k_finalize_lab(NqImage* imgs, const NqSlot* slots, int means) {
  __shared__ int sWarp[33];
  const int img = blockIdx.x;
  NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2) return;
  const NqSlot& S = slots[img];
  const float* fs = reinterpret_cast<const float*>(S.hSum);
  const int t = threadIdx.x, k0 = t * 64;
  int c = 0;
  for (int k = 0; k < 64; ++k) c += S.hCnt[k0 + k] != 0;
  int total, j = block_excl_scan_1024(c, &total, sWarp);
  for (int k = 0; means && k < 64; ++k) {
    unsigned cnt = S.hCnt[k0 + k];
    if (!cnt) continue;
    float fc = cnt > 16777216u ? 16777216.f : (float)cnt;   // tb.cnt += 1.0f saturates at 2^24 (PL:154)
    float d = 1.f / fc;                                      // PL:166
    S.fAc[j] = fs[k0 + k] * d;
    S.fC1[j] = fs[NQ_NBINS + k0 + k] * d;
    S.fC2[j] = fs[2 * NQ_NBINS + k0 + k] * d;
    S.fC3[j] = fs[3 * NQ_NBINS + k0 + k] * d;
    S.bCnt[j] = fc;
    S.bErr[j] = 0.f; S.bNn[j] = 0; S.bTm[j] = 0; S.bMtm[j] = 0;
    ++j;
  }
  if (t == 0) {
    const int nmax = I.nmax, maxbins = total;
    int quan_rt = 1;
    double proportional = ((double)nmax * (double)nmax) / maxbins;                       // PL:175
    if ((I.transIdx >= 0 || I.hasSemi) && nmax < 32) quan_rt = -1;                       // PL:176-177
    double weight = dmin(0.9, nmax * 1.0 / maxbins);                                     // PL:179
    I.weight = weight;
    I.isNano = weight <= .015;                                                           // PL:180
    if ((nmax < 16 && weight < .0075) || weight < .001 || (weight > .0015 && weight < .0022)) quan_rt = 2;
    if (weight < .04 && I.PG < 1 && I.PG >= (double)0.587f) {
      if (nmax >= 64) quan_rt = 0;
    }
    if (nmax > 16 && nmax < 64) {
      double weightB = nmax / 8000.0;
      if (nqm::fabs_(weightB - weight) < .001) quan_rt = 2;
    }
    const bool texicab = proportional > .0225 && !I.hasSemi;                             // PL:219
    double ratio;
    if (I.hasSemi) ratio = .5;                                                           // PL:221-238
    else if (quan_rt != 0 && nmax < 64) {
      if (proportional > .018 && proportional < .022) ratio = dmin(1.0, proportional + weight * nqm::nq_exp(3.13));
      else if (proportional > .1) ratio = dmin(1.0, 1.0 - weight);
      else if (proportional > .04) ratio = dmin(1.0, weight * nqm::nq_exp(1.56));
      else if (proportional > .025 && (weight < .002 || weight > .0022)) ratio = dmin(1.0, proportional + weight * nqm::nq_exp(3.66));
      else ratio = dmin(1.0, proportional + weight * nqm::nq_exp(1.718));
    } else if (nmax > 256) ratio = dmin(1.0, 1 - 1.0 / proportional);
    else ratio = dmin(1.0, 1 - weight * .7);
    if (!I.hasSemi && quan_rt < 0) ratio = dmin(1.0, weight * nqm::nq_exp(3.13));        // PL:240-241
    double ratioMerge = ratio;
    if (quan_rt > 0 && nmax < 64 && proportional > .035 && proportional < .1) {         // PL:259-264
      const int dir = proportional > .04 ? 1 : -1;
      const double margin = dir > 0 ? .002 : .0025;
      const double delta = weight > margin && weight < .003 ? 1.872 : 1.632;
      ratioMerge = dmin(1.0, proportional + dir * weight * nqm::nq_exp(delta));
    }
    I.maxbins = maxbins; I.quan_rt = quan_rt; I.extbins = maxbins - nmax; I.texicab = texicab;
    I.ratio = ratio; I.ratioMerge = ratioMerge;
    // pixelMap.size() <= nMaxColors needs maxbins <= nMaxColors: leave the decision to k_lab_fewcolors (PL:193-206)
    I.skipPnn = maxbins <= nmax ? 2 : 0;
  }
  if (!means) return;
  __syncthreads();
  const int maxbins = I.maxbins, quan_rt = I.quan_rt, nmax = I.nmax;
  for (int b = t; b < maxbins; b += 1024) S.bCnt[b] = quan_lab(nmax, quan_rt, S.bCnt[b]);   // PL:210-217
}

// ---- few-colours shortcut (PL:193-206): when the image holds at most nMaxColors distinct colours the palette is
//      pixelMap.keySet() in java.util.HashMap iteration order, a fully transparent colour swapped to slot 0.
//      One CTA per candidate image (skipPnn == 2, i.e. at most nMaxColors occupied bins): a 1024-slot shared hash
//      set collects the distinct colours with the index of their first pixel (= insertion order of pixelMap).
__global__ void __launch_bounds__(256) k_lab_fewcolors(NqImage* imgs, const NqSlot* slots) {
  __shared__ unsigned long long sKey[1024];
  __shared__ int sFirst[1024];
  __shared__ int sCount, sOverflow;
  __shared__ uint32_t sCol[NQ_MAXK];
  __shared__ int sIdx[NQ_MAXK];
  const int img = blockIdx.x;
  NqImage& I = imgs[img];
  if (I.kind != NQ_KIND_LAB || I.nmax <= 2 || I.skipPnn != 2) return;
  const int t = threadIdx.x, n = I.npix, nmax = I.nmax;
  const uint32_t* in = slots[img].in;
  const uint32_t tc = I.transColor;
  for (int s = t; s < 1024; s += 256) { sKey[s] = ~0ULL; sFirst[s] = 0x7fffffff; }
  if (t == 0) { sCount = 0; sOverflow = 0; }
  __syncthreads();
  for (int i0 = 0; i0 < n; i0 += 256) {
    const int i = i0 + t;
    if (i < n) {
      const uint32_t p = lab_src_pixel(in[i], tc);
      unsigned slot = (p ^ (p >> 11) ^ (p >> 22)) & 1023u;
      for (int probe = 0; probe < 1024; ++probe) {
        unsigned long long k = sKey[slot];
        if (k == ~0ULL) {
          k = atomicCAS(&sKey[slot], ~0ULL, (unsigned long long)p);
          if (k == ~0ULL) { k = p; if (atomicAdd(&sCount, 1) >= nmax) sOverflow = 1; }
        }
        if (k == (unsigned long long)p) { atomicMin(&sFirst[slot], i); break; }
        slot = (slot + 1) & 1023u;
      }
    }
    if ((i0 & 0xFFFF) == 0) {          // every 256 rounds: stop early once there are too many colours
      __syncthreads();
      if (sOverflow) break;
    }
  }
  __syncthreads();
  if (sOverflow || sCount > nmax) { if (t == 0) I.skipPnn = 0; return; }
  if (t == 0) {
    // insertion order = order of first occurrence
    int cnt = 0;
    for (int s = 0; s < 1024; ++s)
      if (sKey[s] != ~0ULL) {
        const uint32_t col = (uint32_t)sKey[s];
        const int fi = sFirst[s];
        int j = cnt++;
        while (j > 0 && sIdx[j - 1] > fi) { sCol[j] = sCol[j - 1]; sIdx[j] = sIdx[j - 1]; --j; }
        sCol[j] = col; sIdx[j] = fi;
      }
    // java.util.HashMap<Integer, ...>: table of 16, doubled when size exceeds 3/4 of it, or when a 9th node lands
    // in one bucket of a table smaller than 64 (treeifyBin resizes instead); buckets keep insertion order and
    // a resize splits them in order, so the final order is (bucket under the final capacity, insertion order)
    int cap = 16, thr = 12, size = 0;
    for (int i = 0; i < cnt; ++i) {
      const uint32_t h = sCol[i] ^ (sCol[i] >> 16);
      int chain = 1;
      for (int j = 0; j < i; ++j) chain += ((sCol[j] ^ (sCol[j] >> 16)) & (unsigned)(cap - 1)) == (h & (unsigned)(cap - 1));
      if (chain >= 9 && cap < 64) { cap *= 2; thr = cap * 3 / 4; }
      if (++size > thr) { cap *= 2; thr = cap * 3 / 4; }
    }
    int k = 0;
    for (int b = 0; b < cap; ++b)
      for (int i = 0; i < cnt; ++i)
        if (((sCol[i] ^ (sCol[i] >> 16)) & (unsigned)(cap - 1)) == (unsigned)b) {
          const uint32_t pixel = sCol[i];
          I.palette[k++] = pixel;
          if (k > 1 && (pixel >> 24) == 0) { I.palette[k - 1] = I.palette[0]; I.palette[0] = pixel; }   // PL:200-202
        }
    I.paletteLen = cnt;
    I.skipPnn = 1;
    I.ratio = I.ratioMerge = .5;      // pnnquan returns before PL:219-241: `ratio` keeps its field default (PQ:25)
  }
}

// ---- saliency map (PL:155-156 inside pnnquan for nMaxColors < 128; PL:499-508 inside dither) ------
__global__ void __launch_bounds__(256) k_saliency(const NqImage* imgs, const NqSlot* slots) {
  const int img = blockIdx.y;
  const NqImage& I = imgs[img];
  if (!I.gUseSal || !slots[img].sal) return;
  const int n = I.npix;
  const uint32_t* in = slots[img].in;
  float* sal = slots[img].sal;
  const bool replaced = I.nmax < 128 && I.nmax > 2;   // which source pixel feeds getLab (Q21)
  const uint32_t tc = I.transColor;
  const int fixA0 = I.fixA0;
  const float saliencyBase = .1f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    uint32_t p = eff_pixel(in[i], fixA0);
    if (replaced) p = lab_src_pixel(p, tc);
    Lab4 l = lab_of(p);
    sal[i] = saliencyBase + (1 - saliencyBase) * l.L / 100.f * l.alpha / 255.f;
  }
}

}  // namespace nq
